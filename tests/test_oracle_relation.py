"""The oracle's hand-derived restatement of the cond=relation logit adjustment (oracle.relation_update) against what the
UNMODIFIED reference `update()` (logit_adjustment.py:88-126: autograd through _stochastic_convert and the 14 costs of
models/clg/const.py) computed on synthetic relation batches built with the reference's own transforms (AddCanvasElement,
AddRelationConstraints, data/util.py:106-170).  Batches, conditions and results are stored in tests/golden/ref_checks
(tests/golden/make_ref_checks.py); the updated log-probs as the rows the update moved most plus a seeded sample."""
import os

import numpy as np
import pytest
import torch

from oracle import layoutdm_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_checks", "oracle_relation.npz")


@pytest.fixture(scope="module")
def ref():
    return np.load(GOLDEN)


def tensor(z, key, dtype=torch.long):
    return torch.from_numpy(z[key]).to(dtype)


def adjacency(z, p, B):
    return O.relation_adjacency(tensor(z, p + "edge_index"), tensor(z, p + "edge_attr"), tensor(z, p + "batch"), B, O.RICO25.n_elem + 1)


@pytest.mark.parametrize("seed,t,lam,n_up", [(0, 50, 3e6, 3), (1, 10, 1e6, 1), (2, 9, 3e6, 3), (3, 99, 3e7, 5)])
def test_relation_update_matches_reference_autograd(ref, seed, t, lam, n_up):
    vo = O.RICO25
    B = 5
    p = f"update_{seed}_"
    seq = tensor(ref, p + "seq")
    assert seq.shape == (B, vo.S)
    # a log-prob tensor like the one the posterior hands over: log-softmax inside each attribute's group, log(1e-30) outside
    g = torch.Generator().manual_seed(seed + 7)
    lp = torch.full((B, vo.S, vo.C), O.LOG_EPS)
    for s in range(vo.S):
        a = s % 5
        lo, n = vo.group_start(a), vo.group_n(a)
        lp[:, s, lo:lo + n] = torch.log_softmax(torch.randn(B, n, generator=g) * 2.0, dim=-1)
    x = lp.double()
    assert np.allclose([float(x.sum()), float(x.abs().sum())], ref[p + "lp_checksum"], rtol=1e-9), "torch generator drifted from the stored inputs"
    centers = torch.stack([torch.as_tensor(c, dtype=torch.float32) for c in O.linear_centers(vo.n_bins)])
    adj = adjacency(ref, p, B)
    # expected boxes first (the forward half)
    _, bbox, valid = O.relation_bbox(lp, seq, centers, vo)
    assert torch.allclose(bbox[valid], tensor(ref, p + "bbox", torch.float32), atol=1e-6)
    got = O.relation_update(lp, seq, adj, centers, vo, t, lam, n_up)
    rows = (tensor(ref, p + "rows_b"), tensor(ref, p + "rows_s"))
    want = tensor(ref, p + "want", torch.float32)
    moved = float(ref[p + "moved"])
    err = (got[rows] - want).abs().max().item()
    print(f"seed {seed} t={t}: edges {ref[p + 'edge_index'].shape[1]}, update moved log-probs by up to {moved:.3e}, |oracle - reference| {err:.3e}")
    if t >= 10:
        assert moved > 1e-3, "test inputs do not exercise the update"
        assert (got - lp).abs().max().item() > 1e-3
    assert err <= 2e-5 * max(1.0, moved)


def test_relation_step_order_matches_reference_single_step(ref):
    """whole `_sample_single_step` (base.py:205-291) with cond=relation: strong mask -> update() -> PAD-disable -> draw, the
    reference (autograd update) against the oracle step with the hand-derived update; ids equal under the shared noise."""
    vo, spec = O.RICO25, O.ModelSpec()
    sd = O.make_weights(vo, spec, seed=7, scale=2.0)
    B = 4
    seq, mask = tensor(ref, "step_seq"), tensor(ref, "step_mask", torch.bool)
    lam, n_up = 3e6, 3
    ocond = dict(seq=seq.clone(), mask=mask.clone(), type="relation", rel_lambda=lam, rel_num_update=n_up, rel_adj=adjacency(ref, "step_", B))
    orc = O.Oracle(vo, spec, sd)
    g = torch.Generator().manual_seed(3)
    for t in (60, 9):
        x_t = torch.where(torch.rand(B, vo.S, generator=g) < 0.5, seq, torch.full_like(seq, vo.mask_id))
        x_t = torch.where(mask, seq, x_t)
        assert torch.equal(x_t, tensor(ref, f"step_{t}_x_t")), "torch generator drifted from the stored inputs"
        u = O.uniforms(5, t, 0, 0, B, vo.S, vo.C)
        want = tensor(ref, f"step_{t}_ids")
        lp, _ = orc.step_logprob(x_t, t, t, ocond)
        got = O.draw(lp, O.SamplingCfg(name="random"), u)
        assert torch.equal(got, want), f"t={t}: {(got != want).sum().item()} ids differ"
