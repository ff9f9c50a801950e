"""
TEST / BENCH INFRASTRUCTURE.  Builds the UNMODIFIED reference LayoutDM for oracle validation, golden-vector generation,
the reference arm of bench.py and the drop-in test of `patch_reference_model`.  The reference package is imported from
/root/reference when that exists (the build container) and otherwise from the archive oracle/make_ref.py packaged
(oracle/_ref/trainer_ref.zip, zipimport: it travels to the GPU box, /root/reference does not), in both cases through the
import stand-ins of oracle/ref_shims.

Recipe = SURVEY.md Appendix B.
"""
from __future__ import annotations

import os
import sys
from contextlib import contextmanager

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
REF_SRC = "/root/reference/src/trainer"
REF_ZIP = os.path.join(HERE, "_ref", "trainer_ref.zip")


def reference_source() -> str | None:
    """where the reference's `trainer` package is imported from: the read-only checkout, else the packaged archive"""
    if os.path.isdir(os.path.join(REF_SRC, "trainer")):
        return REF_SRC
    return REF_ZIP if os.path.exists(REF_ZIP) else None


def reference_available() -> bool:
    return reference_source() is not None


def _setup_path():
    src = reference_source()
    assert src is not None, "reference not available: run `python oracle/make_ref.py` in the build container"
    for p in (src, os.path.join(HERE, "ref_shims")):
        if p not in sys.path:
            sys.path.insert(0, p)
    if REPO not in sys.path:
        sys.path.insert(0, REPO)


def build_reference(dataset: str = "rico25", T: int = 100, q_type: str = "constrained", state_dict=None):
    """returns (model, tokenizer); model is the reference LayoutDM in eval mode on CPU."""
    _setup_path()
    from omegaconf import OmegaConf
    from trainer.helpers.layout_tokenizer import LayoutSequenceTokenizer
    from trainer.models.layoutdm import LayoutDM

    data_cfg = OmegaConf.create(dict(
        batch_size=64, bbox_quantization="linear", num_bin_bboxes=32, num_workers=1, pad_until_max=True,
        shared_bbox_vocab="x-y-w-h", special_tokens=["pad", "mask"], transforms=["RandomOrder"], var_order="c-x-y-w-h"))
    target = {"rico25": "trainer.datasets.rico.Rico25Dataset", "publaynet": "trainer.datasets.publaynet.PubLayNetDataset"}[dataset]
    dataset_cfg = OmegaConf.create(dict(_target_=target, _partial_=True, dir="x", max_seq_length=25))
    backbone_cfg = OmegaConf.create(dict(
        _target_="trainer.models.transformer_utils.TransformerEncoder", num_layers=4,
        encoder_layer=dict(_target_="trainer.models.transformer_utils.Block", d_model=512, nhead=8,
                           dim_feedforward=2048, dropout=0.0, batch_first=True, norm_first=True,
                           timestep_type="adalayernorm", diffusion_step=T)))
    tok = LayoutSequenceTokenizer(data_cfg, dataset_cfg)
    torch.manual_seed(0)
    model = LayoutDM(backbone_cfg=backbone_cfg, tokenizer=tok, q_type=q_type, num_timesteps=T).eval()
    if state_dict is not None:
        missing, unexpected = model.load_state_dict(state_dict, strict=False)
        # only the schedule buffers / Lt_* may be missing from a weights-only dict
        assert all(("_log_" in k) or k.split(".")[-1].startswith(("Lt_", "log_")) for k in missing), missing
        assert not unexpected, unexpected
    return model, tok


def sampling_cfg(name="random", **kw):
    _setup_path()
    from omegaconf import OmegaConf
    d = {"name": name}
    if name != "deterministic":
        d["temperature"] = 1.0
    if name == "top_p":
        d["top_p"] = 0.9
    if name == "top_k":
        d["top_k"] = 5
    d.update(kw)
    return OmegaConf.create(d)


class FakeBatch:
    """stand-in for a torch_geometric DataBatch (x: bbox xywh, y: label, batch: layout index)"""

    def __init__(self, x, y, batch):
        self.x, self.y, self.batch = x, y, batch
        self.attr = {"has_canvas_element": False}

    def to(self, device):
        """like torch_geometric's Batch.to: every tensor attribute moves"""
        out = FakeBatch.__new__(FakeBatch)
        for k, v in self.__dict__.items():
            setattr(out, k, v.to(device) if isinstance(v, torch.Tensor) else v)
        return out


def synthetic_layouts(B: int, n_cat: int, seed: int = 0, max_elem: int = 25) -> FakeBatch:
    g = torch.Generator().manual_seed(seed)
    n = torch.randint(1, max_elem + 1, (B,), generator=g)
    batch = torch.repeat_interleave(torch.arange(B), n)
    N = int(n.sum())
    y = torch.randint(0, n_cat, (N,), generator=g)
    x = torch.rand(N, 4, generator=g)
    return FakeBatch(x, y, batch)


def make_relation_batch(B, n_cat, seed, edge_ratio=0.3) -> FakeBatch:
    """synthetic cond=relation batch built with the reference's own transforms (AddCanvasElement, AddRelationConstraints,
    data/util.py:106-170): element 0 of every layout is the canvas, edges carry the relation labels"""
    _setup_path()
    from trainer.data.util import AddCanvasElement, AddRelationConstraints
    g = torch.Generator().manual_seed(seed)
    add_c, add_r = AddCanvasElement(), AddRelationConstraints(seed=seed, edge_ratio=edge_ratio)
    xs, ys, bs, ei, ea = [], [], [], [], []
    off = 0
    for b in range(B):
        n = int(torch.randint(1, 26, (1,), generator=g)) if b else 25
        class D:
            pass
        d = D()
        d.x = torch.rand(n, 4, generator=g) * torch.tensor([1.0, 1.0, 0.6, 0.6]) + torch.tensor([0.0, 0.0, 0.02, 0.02])
        d.y = torch.randint(0, n_cat, (n,), generator=g)
        d.attr = {"has_canvas_element": torch.tensor(False)}
        d = add_c(d)
        d.attr["has_canvas_element"] = True
        d = add_r(d)
        xs.append(d.x); ys.append(d.y); bs.append(torch.full((n + 1,), b))
        if d.edge_index.numel():
            ei.append(d.edge_index + off); ea.append(d.edge_attr)
        off += n + 1
    batch = FakeBatch(torch.cat(xs), torch.cat(ys), torch.cat(bs))
    batch.edge_index = torch.cat(ei, dim=1) if ei else torch.zeros(2, 0, dtype=torch.long)
    batch.edge_attr = torch.cat(ea) if ea else torch.zeros(0, dtype=torch.long)
    batch.attr = {"has_canvas_element": True}
    return batch


@contextmanager
def injected_multinomial(uniform_fn):
    """Replace torch.multinomial(probs, 1) by argmax(probs / -log(u)) with u supplied by the caller
    (this is ATen's own single-sample algorithm with the RNG swapped out; SURVEY.md §7.2-6).
    uniform_fn(call_index, n_rows, n_classes) -> float32 ndarray (n_rows, n_classes)."""
    orig = torch.multinomial
    state = {"i": 0}

    def fake(probs, num_samples, replacement=False, *, generator=None):
        assert num_samples == 1 and probs.dim() == 2
        u = torch.from_numpy(np.ascontiguousarray(uniform_fn(state["i"], probs.shape[0], probs.shape[1])))
        state["i"] += 1
        e = -torch.log(u)
        return torch.argmax(probs / e, dim=-1, keepdim=True)

    torch.multinomial = fake
    try:
        yield state
    finally:
        torch.multinomial = orig
