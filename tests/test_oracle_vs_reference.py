"""CPU: pieces of the oracle against what the UNMODIFIED reference computed on the same inputs (tests/golden/ref_checks,
written by tests/golden/make_ref_checks.py), beyond what tests/golden/make_golden.py already asserts while generating the
fixtures.  (B, S, C) reference results are stored as a fixed sample of token rows (all C classes each)."""
import os

import numpy as np
import pytest
import torch

from oracle import layoutdm_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_checks", "oracle_vs_reference.npz")


@pytest.fixture(scope="module")
def ref():
    return np.load(GOLDEN)


def tensor(z, key, dtype=None):
    t = torch.from_numpy(z[key])
    return t.to(dtype) if dtype is not None else t


def checksum(x):
    x = x.double()
    return np.array([float(x.sum()), float(x.abs().sum())])


def random_x0(vocab, B, g):
    x0 = torch.empty(B, vocab.S, dtype=torch.long)
    for a in range(5):
        ids = torch.tensor(vocab.group_full_ids(a)[:-1])               # normal classes + PAD (no MASK in x0)
        x0[:, a::5] = ids[torch.randint(0, len(ids), (B, 25), generator=g)]
    return x0


def test_q_sample_ids_matches_reference_q_sample(ref):
    """forward (corruption) process: oracle.q_sample_ids == reference q_sample per attribute (constrained.py:223-230),
    with the Gumbel uniforms injected through torch.rand_like"""
    vocab = O.RICO25
    B, S, C, T = 6, vocab.S, vocab.C, 100
    x0 = random_x0(vocab, B, torch.Generator().manual_seed(3))
    assert torch.equal(x0, tensor(ref, "q_sample_x0", torch.long)), "torch generator drifted from the stored inputs"
    t = torch.tensor([0, 1, 37, 64, 98, 99])
    u = O.uniforms(77, 0, 2, 0, B, S, C)
    want = O.q_sample_ids(x0, t, T, vocab, O.group_schedules(T, vocab), u)
    assert torch.equal(tensor(ref, "q_sample_ids", torch.long), want)
    # sanity: late timesteps are mostly MASK, early ones mostly unchanged
    assert (want[5] == vocab.mask_id).float().mean() > 0.9 and (want[0] == x0[0]).float().mean() > 0.9


def test_decode_matches_reference_tokenizer(ref):
    vocab = O.RICO25
    ids = torch.randint(0, vocab.C, (32, vocab.S), generator=torch.Generator().manual_seed(0))
    assert torch.equal(ids, tensor(ref, "decode_ids", torch.long)), "torch generator drifted from the stored inputs"
    b = O.decode_ids(ids, vocab)
    for k in ("bbox", "label", "mask"):
        assert torch.equal(tensor(ref, f"decode_{k}").to(b[k].dtype), b[k]), k


@pytest.mark.parametrize("cond_type", ["c", "cwh", "gt", "refinement"])
def test_make_cond_matches_reference_get_cond(ref, cond_type):
    """cond construction: oracle.make_cond == the reference's get_cond (task.py:27-151) on a dense fake batch, incl.
    boxes outside [0, 1] and on the rounding boundaries of the linear quantisation"""
    vocab = O.RICO25
    bbox = tensor(ref, "cond_refinement_bbox" if cond_type == "refinement" else "cond_bbox")   # refinement: with the noise of task.py:127
    got = O.make_cond(tensor(ref, "cond_label", torch.long), bbox, tensor(ref, "cond_mask_in"), vocab, cond_type)
    p = f"cond_{cond_type}_"
    for k in ("seq", "mask") + (("seq_orig",) if cond_type == "refinement" else ()):
        assert torch.equal(tensor(ref, p + k).to(got[k].dtype), got[k]), k
    if cond_type != "gt":
        assert torch.equal(tensor(ref, p + "num_element").to(got["num_element"].dtype), got["num_element"])


@pytest.mark.parametrize("q_type", ["constrained", "vanilla"])
def test_training_side_api_matches_reference(ref, q_type):
    """q_posterior with ANY log p(x0) and per-layout timesteps, q_pred, and the loss terms of `forward` (constrained.py:232-333 /
    vanilla.py) -- oracle restatement vs the unmodified reference, which saw the same x_t and (t, pt)"""
    vocab, spec = O.RICO25, O.ModelSpec()
    sd = O.make_weights(vocab, spec, seed=7, scale=2.0)
    scheds = O.group_schedules(100, vocab, q_type)
    p = f"train_{q_type}_"
    B, S, C = 7, vocab.S, vocab.C
    g = torch.Generator().manual_seed(0)
    x0 = random_x0(vocab, B, g)
    t = torch.tensor([0, 1, 50, 99, 37, 0, 98])
    xt = O.q_sample_ids(x0, t, 100, vocab, O.group_schedules(100, vocab), O.uniforms(3, 0, 2, 0, B, S, C))
    lx = torch.log_softmax(torch.randn(B, S, C, generator=g) * 2.0, dim=-1).clamp(-70.0, 0.0)
    assert torch.equal(x0, tensor(ref, p + "x0", torch.long)), "torch generator drifted from the stored inputs"
    assert np.allclose(checksum(lx), ref[p + "lx_checksum"], rtol=1e-9), "torch generator drifted from the stored inputs"
    assert torch.equal(xt, tensor(ref, p + "xt", torch.long))
    rows = (tensor(ref, p + "rows_b", torch.long), tensor(ref, p + "rows_s", torch.long))

    def max_err(got_full, key):
        want = tensor(ref, p + key)
        defined = ~torch.isnan(want)
        assert defined.any(dim=-1).all()
        return (got_full[rows][defined] - want[defined]).abs().max().item()

    # 1. q_posterior, arbitrary log p(x0)
    assert max_err(O.q_posterior(lx, xt, t, 100, vocab, scheds, q_type), "q_posterior") < 1e-5
    # 2. q_pred (t = -1 wraps to T, constrained.py:115); the constrained reference defines each attribute's group only
    tq = torch.tensor([-1, 0, 50, 99, 37, 5, 98])
    assert max_err(O.q_pred_full(lx, tq, 100, vocab, scheds, q_type), "q_pred") < 1e-5
    # 2b. q_pred_one_timestep and log_sample_categorical (gumbel) with the reference's noise drawn by torch.rand_like
    t1 = torch.tensor([0, 1, 50, 99, 37, 5, 98])
    assert max_err(O.q_pred_one_timestep_full(lx, t1, 100, vocab, scheds, q_type), "q_pred_one_timestep") < 1e-5
    if q_type == "constrained":
        u_all = O.uniforms(9, 0, 2, 0, B, S, C)
        for a in range(5):
            idx = torch.tensor(vocab.group_full_ids(a))
            part = lx[:, a::5][..., idx]
            u_part = torch.from_numpy(u_all)[:, a::5][..., idx].contiguous()
            assert torch.equal(tensor(ref, p + "gumbel_argmax", torch.long)[a], O.gumbel_argmax(part, u_part.numpy()))
    # 3. forward: the reference's loss terms at (t, pt = 1 / T) on this x_t
    logits = O.denoiser_forward(sd, xt, t, vocab, spec)
    pt = torch.full((B,), 1.0 / 100)
    r = O.vb_terms(logits, x0, xt, t, 100, vocab, scheds, q_type)
    assert max_err(r["log_model_prob"].exp(), "probs") < 1e-5
    kl_want, aux_want = ref[p + "losses"]
    mask = (t == 0).float()
    kl_loss = mask * r["decoder_nll"] + (1 - mask) * r["kl"]
    assert abs((kl_loss / pt).mean().item() - kl_want) < 1e-4 * abs(kl_want)
    aux = mask * r["decoder_nll"] + (1 - mask) * r["kl_aux"]
    assert abs((((1 - t / 100) + 1.0) * 0.1 * aux / pt).mean().item() - aux_want) < 1e-4 * abs(aux_want)
    # the oracle's denoiser at per-layout timesteps == the reference's transformer
    assert max_err(logits, "logits") < 2e-5
