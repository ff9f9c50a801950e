"""GPU (-m gpu): the drop-in INTEGRATION.md tells a maintainer to use -- `patch_reference_model(model)` on a LIVE, UNMODIFIED
reference `LayoutDM` (imported from the packaged archive oracle/_ref/trainer_ref.zip, or /root/reference where that exists).
After patching, the reference's own `model.sample(...)` / `model.model.sample(get_intermediate_results=True)` /
`_sample_single_step(...)` run on the sm_100a library and are compared with the golden trajectories the same reference
produced on the CPU (tests/golden) under the shared noise key."""
import copy

import pytest
import torch

from fixtures import Fixture
from oracle import layoutdm_oracle as O
from oracle import ref_harness as rh

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not rh.reference_available(), reason="reference archive missing: run python oracle/make_ref.py")]


def patched(fx):
    from layoutdm_b200 import patch_reference_model
    model, tok = rh.build_reference(fx.meta["dataset"], T=fx.meta["T"], q_type=fx.meta["q_type"], state_dict=fx.weights())
    return patch_reference_model(model), tok


def ref_cfg(fx):
    kw = dict(num_timesteps=fx.meta["T_eval"])
    if fx.meta["time_difference"]:
        kw["time_difference"] = fx.meta["time_difference"]
    if fx.meta.get("refine"):
        kw.update(fx.meta["refine"])
    return rh.sampling_cfg(fx.meta["sampling"], **kw)


@pytest.mark.parametrize("name", ["rico25_uncond_T50", "publaynet_c_top_p", "rico25_refinement_T200", "rico25_vanilla_random"])
def test_patched_reference_model_sample(name):
    fx = Fixture(name)
    model, tok = patched(fx)
    core = model.model.module
    assert hasattr(core, "_ldm_b200")
    cond = copy.deepcopy(fx.cond)
    if cond is not None and "refine_table" in cond:
        del cond["refine_table"]                 # the reference's get_cond output has no table: the patched sample() builds it from sampling_cfg
    seed = fx.meta["noise_seed"]
    # 1. LayoutDM.sample (layoutdm.py:77-88): decoded layouts on the CPU, the reference's own tokenizer.decode
    out = model.sample(batch_size=fx.B, cond=copy.deepcopy(cond), sampling_cfg=ref_cfg(fx), cond_type=fx.meta["cond"], seed=seed)
    assert set(out) >= {"bbox", "label", "mask"} and out["bbox"].shape == (fx.B, 25, 4) and not out["bbox"].is_cuda
    # 2. the core's sample with the intermediate results (notebooks/demo.ipynb)
    res = model.model.sample(batch_size=fx.B, cond=copy.deepcopy(cond), sampling_cfg=ref_cfg(fx), get_intermediate_results=True, seed=seed)
    assert isinstance(res, list) and len(res) == len(fx.plan) and res[0].shape == (fx.B, 125) and res[0].dtype == torch.int64
    ids = res[-1]
    want = tok.decode(ids)
    for k in ("bbox", "label", "mask"):
        assert torch.equal(out[k], want[k]), k   # same key -> same trajectory -> same layouts
    # 3. against the golden trajectory of the reference on the CPU (same noise key): the first steps are the reference's ids
    #    except where 16-bit operand rounding flips a near-tie (after a flip the trajectories drift apart)
    first = (res[0] == fx.x_out[0]).float().mean().item()
    final = (ids == fx.ids_final).float().mean().item()
    print(f"{name}: identical tokens after step 0: {first:.4f}, after the last step: {final:.4f}")
    assert first > 0.99
    assert final > 0.5
    if cond is not None:
        m = fx.cond["mask"]
        assert torch.equal(ids[m], fx.cond["seq"][m])          # strong mask reproduced exactly
    if fx.plan[-1][1] == 0:
        assert (ids != fx.vocab.mask_id).all()
    # 4. torch.manual_seed controls the run when no key is passed, as in the reference
    torch.manual_seed(5)
    a = model.model.sample(batch_size=fx.B, cond=copy.deepcopy(cond), sampling_cfg=ref_cfg(fx))
    torch.manual_seed(5)
    b = model.model.sample(batch_size=fx.B, cond=copy.deepcopy(cond), sampling_cfg=ref_cfg(fx))
    assert torch.equal(a, b)


def test_patched_single_step_matches_reference_step():
    """`_sample_single_step` (base.py:205-291) on (B,C,S) log one-hots: step-wise on the reference's own x_t the ids equal the
    golden ones up to 16-bit near-ties; the pinned noise key makes the call reproducible."""
    fx = Fixture("rico25_uncond_random")
    model, tok = patched(fx)
    core = model.model.module
    fused = core._ldm_b200
    cfg = ref_cfg(fx)
    mism = tot = 0
    for i in (0, 1, 50, 99):
        t_model, _ = fx.plan[i]
        skip = (fx.plan[i - 1][0] - t_model - 1) if i else (fx.meta["T"] - t_model - 1)
        log_z = torch.log(torch.nn.functional.one_hot(fx.x_in[i], fx.vocab.C).permute(0, 2, 1).float().clamp(min=1e-30))
        fused.reset_noise(fx.meta["noise_seed"]); fused._step_ctr = i
        out = core._sample_single_step(log_z=log_z.cuda(), model_t=torch.full((fx.B,), t_model, device="cuda"), skip_step=skip, sampling_cfg=cfg, cond=None)
        assert out.shape == (fx.B, fx.vocab.C, 125)
        got = out.argmax(1).cpu()
        mism += int((got != fx.x_out[i]).sum()); tot += got.numel()
    assert mism / tot < 0.01, f"{mism}/{tot}"
    fused.reset_noise(None)


def test_single_condition_many_outputs_refinement():
    """duplicate_cond (task.py:235-248): ONE refinement condition, batch_size > 1 -- the (C, C) band table must not be repeated"""
    fx = Fixture("rico25_refinement_T200")
    model, tok = patched(fx)
    cond = {k: (v[:1].clone() if isinstance(v, torch.Tensor) and k != "refine_table" else v) for k, v in fx.cond.items()}
    cond.pop("refine_table")
    cfg = rh.sampling_cfg("random", num_timesteps=20, **fx.meta["refine"])
    ids = model.model.sample(batch_size=6, cond=cond, sampling_cfg=cfg, seed=1)
    assert ids.shape == (6, 125)
    m = fx.cond["mask"][0]
    assert (ids[:, m] == fx.cond["seq"][0][m]).all()
    assert not all(torch.equal(ids[0], ids[i]) for i in range(1, 6))     # distinct noise per output


def test_patched_model_relation_device_vs_reference_autograd_update():
    """cond = "relation" end to end on a live reference model: the device update kernel (default) against the reference's own
    autograd `update` running through the log-prob taps (relation_on_device = False), same noise key"""
    import random
    fx = Fixture("rico25_uncond_random")
    model, tok = patched(fx)
    fused = model.model.module._ldm_b200
    rh._setup_path()
    from trainer.helpers.task import get_cond
    random.seed(0); torch.manual_seed(0)
    B = 6
    batch = rh.make_relation_batch(B, fx.vocab.n_cat, 21)
    cond = get_cond(batch, tok, "relation", model_type="LayoutDM")
    cfg = rh.sampling_cfg("random", num_timesteps=25, relation_lambda=3e6, relation_mode="average", relation_tau=1.0, relation_num_update=3)
    res = {}
    for on_device in (True, False):
        fused.relation_on_device = on_device
        res[on_device] = model.model.sample(batch_size=B, cond=copy.copy(cond), sampling_cfg=cfg, seed=77, get_intermediate_results=True)
    fused.relation_on_device = True
    first = (res[True][0] == res[False][0]).float().mean().item()
    final = (res[True][-1] == res[False][-1]).float().mean().item()
    print(f"relation: device update vs reference autograd update: identical tokens after step 0 {first:.4f}, after the last step {final:.4f}")
    assert first > 0.995 and final > 0.9
    m = cond["mask"]
    assert torch.equal(res[True][-1][m], cond["seq"][m])
    out = model.sample(batch_size=B, cond=copy.copy(cond), sampling_cfg=cfg, cond_type="relation", seed=77)
    assert torch.equal(out["label"], tok.decode(res[True][-1])["label"])
