#!/usr/bin/env python
"""bench.py -- layouts/sec of the LayoutDM denoising loop (BASELINE.json metric) on N GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one full pass of the hot path over one batch: `sample()` of B=1024 layouts per GPU through all T=100
denoising iterations (BASELINE.json configs[1]: rico25 unconditional, T=100, batch 1024, random sampling).
Prints ONE JSON line (rank 0).  `value` = layouts/s with everything device-resident; `e2e` = the same metric through
the host-buffer C-ABI entry (ldm_sample_host: pinned-host inputs -> H2D -> loop -> D2H of the ids);
`roofline` = the dominant kernel against the measured bf16 tensor peak; `cpu_baseline` = the unmodified reference's
`LayoutDM.sample` on the host cores (bounded sample; packaged by oracle/make_ref.py), `gpu_eager_baseline` = the same
reference run eagerly on the GPU.  `--impl reference` times the CPU reference alone.
`--dump-outputs DIR` writes what the last timed step returned (the final token ids, as float32) to DIR/ids.npy; weights
and noise keys are fixed by the arguments, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

# stdout carries exactly ONE JSON line: everything else that writes to fd 1 (NCCL's version banner, library chatter from C code)
# is sent to stderr; the line itself goes to the saved descriptor
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: str):
    os.write(_REAL_STDOUT, (line + "\n").encode())


METRIC = "layouts_per_sec_T100_batch1024_N25"
UNIT = "layouts/s"
T = 100
# algorithmic FLOPs per layout per launch (unpadded shapes, SURVEY.md 8d / BASELINE.md 3)
FLOPS = {"qkv_gemm": 161_472_000, "outproj_gemm": 53_824_000, "ff1_gemm": 215_296_000, "ff2_gemm": 215_296_000,
         "attention": 29_000_000, "head_gemm": 17_980_000}
FLOPS_PER_LAYOUT_STEP = 2_717_532_000
# algorithmic HBM bytes per layout per launch (DESIGN.md 3: rows of 128 tokens; x16/z16 119 KB, x32/y32 237 KB, qkv16 393 KB, att16 131 KB,
# hid16 475 KB, logits 82 KB): what each kernel must read + write when every intermediate makes one round trip through HBM
BYTES = {"embed_adaln": 237_568 + 118_784, "qkv_gemm": 118_784 + 393_216, "attention": 393_216 + 131_072,
         "outproj_gemm": 131_072 + 2 * 237_568 + 118_784, "ff1_gemm": 118_784 + 475_136, "ff2_gemm": 475_136 + 2 * 237_568 + 118_784,
         "head_gemm": 118_784 + 81_920, "posterior_sample": 81_920 + 2_000}


def load_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/ncu_traffic.json)"""
    try:
        d = json.load(open(os.path.join(REPO, "profiles", "ncu_traffic.json")))
        return float(d["dram_bytes_per_launch"][kernel]), d["source"]
    except Exception:
        return None, None


def kernel_record(k, v, B, tot_ms, peaks):
    """per-kernel line of the roofline table: achieved tensor rate (algorithmic FLOPs) and HBM rate (algorithmic bytes when every
    intermediate makes one round trip) against the measured peaks; the kernel's own roofline is the larger of the two fractions"""
    us = v[0] / v[1] * 1e3
    r = {"ms_per_pass": round(v[0], 3), "launches": v[1], "us_per_launch": round(us, 1), "share": round(v[0] / tot_ms, 4)}
    fr = []
    if k in FLOPS:
        tf = FLOPS[k] * B / (us * 1e-6) / 1e12
        r["tflops"] = round(tf, 1); r["tensor_frac"] = round(tf / peaks["sustained"], 3); fr.append(("tensor", r["tensor_frac"]))
    if k in BYTES:
        gb = BYTES[k] * B / (us * 1e-6) / 1e9
        r["hbm_gbs"] = round(gb, 0); r["hbm_frac"] = round(gb / peaks["hbm"], 3); fr.append(("hbm", r["hbm_frac"]))
    if fr:
        r["bound"], r["frac"] = max(fr, key=lambda x: x[1])
    return r


def load_precision():
    """logit error of the 16-bit operand path vs the fp32 oracle at weight scales 1 / 2 / 3, measured on the GPU box by
    tools/precision_report.py and committed under profiles/ (bench.py itself must not run the oracle outside the CPU legs)"""
    try:
        d = json.load(open(os.path.join(REPO, "profiles", "r02c_precision.json")))
        return {"source": "profiles/r02c_precision.json (tools/precision_report.py: max-abs logit error vs the fp32 oracle, B=32, t in {0, 42, 99})",
                "rows": [{k: r[k] for k in ("operand_dtype", "weight_scale", "max_abs_logit", "logit_err_vs_fp32", "logit_err_vs_same_rounding", "fp16_headroom_x", "nonfinite")}
                         for r in d["rows"]]}
    except Exception:
        return None


def load_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(burst=d["bf16_tflops"], sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), hbm=d["hbm_gbs"], src="measured (MEASURED_PEAKS.json)")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons while the timed region runs"""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        # under load = samples at or above the median of the upper half
        busy = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"      # NCCL_DEBUG=VERSION prints a banner on stdout: keep stdout to the one JSON line
        dist.init_process_group("nccl" if torch.cuda.is_available() else "gloo", rank=rank, world_size=world,
                                device_id=torch.device("cuda", local) if torch.cuda.is_available() else None)
    return world, rank, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


def max_over_ranks(x: float, world, device):
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


# --------------------------------------------------------------------------------------------------------------
# Reference arm: the UNMODIFIED reference `LayoutDM.sample` (layoutdm.py:77-88 -> base.py:293-371) from the archive
# oracle/make_ref.py packaged (oracle/_ref/trainer_ref.zip; /root/reference does not exist on the GPU box), on the host
# cores.  Falls back to the oracle port (kind "port") only if the archive is missing.
# --------------------------------------------------------------------------------------------------------------
REF_B, REF_NT = 64, 100      # fixed bounded sample: one step = sample() of 64 layouts through the FULL T=100 loop (no extrapolation in T;
                             # B=64 is the reference's most efficient CPU batch per layout: measured 64 / 256 / 512 -> 1.96 / 1.28 / 1.12
                             # layouts/s on 8 cores).  ~3.6 s per step on the 64 physical cores of the GPU box (r02b: 17.7 layouts/s)


def physical_cores(cap=64):
    """physical cores this process may run on (SMT siblings counted once), capped"""
    aff = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else set(range(os.cpu_count() or 1))
    cores = set()
    try:
        cpu = phys = core = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("processor"):
                cpu = int(line.split(":")[1])
            elif line.startswith("physical id"):
                phys = int(line.split(":")[1])
            elif line.startswith("core id"):
                core = int(line.split(":")[1])
            elif not line.strip():
                if cpu in aff and phys is not None and core is not None:
                    cores.add((phys, core))
                cpu = phys = core = None
    except Exception:
        pass
    n = len(cores) if cores else len(aff)
    return max(1, min(n, cap))


class CpuArm:
    """one `step` = sample() of REF_B layouts through REF_NT denoising iterations on the host cores"""

    def __init__(self):
        from oracle import ref_harness as rh         # allowed here: cpu_baseline / --impl reference legs only
        from layoutdm_b200 import Vocab
        from layoutdm_b200.synthetic import random_state_dict
        self.sd = random_state_dict(Vocab.for_dataset("rico25"), num_timesteps=T, seed=0)
        self.rh = rh
        if rh.reference_available():
            self.kind = "reference"
            self.model, _ = rh.build_reference("rico25", T=T, state_dict=self.sd)
            self.cfg = rh.sampling_cfg("random", num_timesteps=REF_NT)
            self.what = "unmodified reference LayoutDM.sample (fp32 PyTorch eager, CPU)"
        else:
            from oracle import layoutdm_oracle as O
            self.kind = "port"
            self.O = O
            self.orc = O.Oracle(O.RICO25, O.ModelSpec(T=T), self.sd)
            self.what = "fp32 torch-CPU port of the reference path (oracle)"

    def step(self, seed):
        torch.manual_seed(seed)
        t0 = time.perf_counter()
        with torch.no_grad():
            if self.kind == "reference":
                out = self.model.sample(batch_size=REF_B, cond=None, sampling_cfg=self.cfg)
                assert out["bbox"].shape[0] == REF_B
            else:
                O, vo = self.O, self.orc.vocab
                x = torch.full((REF_B, vo.S), vo.mask_id, dtype=torch.long)
                for i, (tm, tp) in enumerate(O.timestep_plan(T, REF_NT)):
                    lp, _ = self.orc.step_logprob(x, tm, tp)
                    x = O.draw(lp, O.SamplingCfg(name="random"), O.uniforms(seed, i, 0, 0, REF_B, vo.S, vo.C))
        return time.perf_counter() - t0

    def layouts_per_s(self, dt):
        return REF_B / (dt * T / REF_NT)             # per-iteration cost does not depend on t: scale to the full T-step loop

    def sample_desc(self, dt):
        scaled = "" if REF_NT == T else f", scaled x{T / REF_NT:.1f} to T={T}"
        return f"{REF_B} layouts x {REF_NT} of {T} denoising iterations per step ({dt:.1f} s of CPU work per step){scaled}; {self.what}"


def run_reference_arm(args, world, rank):
    if rank != 0:
        return
    cores = physical_cores()
    torch.set_num_threads(cores)                     # torchrun exports OMP_NUM_THREADS=1: use the physical cores (no SMT oversubscription)
    arm = CpuArm()
    for w in range(max(1, args.warmup)):
        arm.step(w)
    dts = [arm.step(100 + k) for k in range(args.steps)]
    dt = sum(dts) / len(dts)
    lps = arm.layouts_per_s(dt)
    line = {"impl": "reference", "metric": METRIC, "value": lps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": max(1, args.warmup),
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "rico25 unconditional, T=100, random sampling, N=25 (S=125, C=155); bounded CPU sample of the batch-1024 workload"},
            "cpu_baseline": {"value": lps, "unit": UNIT, "cores": cores, "kind": arm.kind, "sample": arm.sample_desc(dt),
                             "best_step_value": arm.layouts_per_s(min(dts)), "step_seconds": [round(x, 3) for x in dts]},
            "e2e": {"value": lps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit(json.dumps(line))


def gpu_eager_reference(B, dev):
    """the north star's denominator: the unmodified reference `LayoutDM.sample` run eagerly (fp32) on the same GPU, full
    T=100 loop, chunks of <= 512 layouts (Converter limit, layout_tokenizer.py:530), synchronize-bracketed like test.py:194-203"""
    from oracle import ref_harness as rh
    if not rh.reference_available():
        return None
    from layoutdm_b200 import Vocab
    from layoutdm_b200.synthetic import random_state_dict
    model, _ = rh.build_reference("rico25", T=T, state_dict=random_state_dict(Vocab.for_dataset("rico25"), num_timesteps=T, seed=0))
    model = model.to(dev)
    cfg = rh.sampling_cfg("random", num_timesteps=T)
    chunks = [min(512, B - i) for i in range(0, B, 512)]
    with torch.no_grad():
        model.sample(batch_size=min(64, B), cond=None, sampling_cfg=rh.sampling_cfg("random", num_timesteps=5))   # warm-up (cuBLAS handles, allocator)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for b in chunks:
            model.sample(batch_size=b, cond=None, sampling_cfg=cfg)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
    del model
    torch.cuda.empty_cache()
    return {"value": B / dt, "unit": UNIT, "seconds": dt, "kind": "reference",
            "what": f"unmodified reference LayoutDM.sample, fp32 PyTorch eager on the same GPU, batch {B} in chunks of <= 512, T={T}, one pass"}


def other_configs(local):
    """device-resident sample() at BASELINE.json configs 0 / 2 / 3 (synthetic weights and conditions); config 1 is the main line,
    config 4 (8 x 1024) is what the N-GPU runs of this script measure"""
    from layoutdm_b200 import Engine, Vocab, timestep_plan
    from layoutdm_b200.synthetic import random_state_dict, synthetic_cond
    cases = [("configs[0] rico25 unconditional, T_eval=50, batch=8", "rico25", 100, 50, 8, {"name": "random", "temperature": 1.0}, None, 5),
             ("configs[2] publaynet cond=c, T=100, batch=1024, top_p=0.9", "publaynet", 100, 100, 1024, {"name": "top_p", "temperature": 1.0, "top_p": 0.9}, "c", 2),
             ("configs[3] rico25 cond=refinement (logit masking), T=200, batch=4096", "rico25", 200, 200, 4096, {"name": "random", "temperature": 1.0}, "refinement", 2)]
    out = []
    for name, ds, Tm, T_eval, B, cfg, ctype, n in cases:
        vocab = Vocab.for_dataset(ds)
        eng = Engine.from_state_dict(random_state_dict(vocab, num_timesteps=Tm), vocab, num_timesteps=Tm, device=local)
        cond = None
        if ctype:
            cond = {k: (v.cuda(local) if isinstance(v, torch.Tensor) else v) for k, v in synthetic_cond(vocab, B, ctype).items()}
        plan = timestep_plan(Tm, T_eval)
        ids0 = cond["seq"] if cond else None
        for w in range(3 if B < 1024 else 1):
            eng.sample_loop(B, plan, cfg, cond=cond, seed=1 + w, ids_init=ids0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            ids = eng.sample_loop(B, plan, cfg, cond=cond, seed=10 + i, ids_init=ids0)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        if cond is not None:
            assert torch.equal(ids[cond["mask"]], cond["seq"][cond["mask"]])      # strong conditioning reproduced exactly
        assert int(ids.max()) < vocab.C - 1                                       # no MASK left
        out.append({"config": name, "ms_per_step": round(ms, 3), "layouts_per_s": round(B / (ms * 1e-3), 1),
                    "ms_per_denoising_iteration": round(ms / T_eval, 4), "passes_timed": n})
        eng.close()
        del eng
        torch.cuda.empty_cache()
    return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, ids):
    """ids (layouts, S) -> path/ids.npy as float32 (token ids are exact there); above DUMP_LIMIT_BYTES a fixed, seeded
    sample of layouts (rows kept in order) is written instead"""
    os.makedirs(path, exist_ok=True)
    a = ids.cpu().numpy().astype(np.float32)
    max_rows = DUMP_LIMIT_BYTES // (a.shape[1] * a.itemsize)
    if a.shape[0] > max_rows:
        a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], max_rows, replace=False))]
    np.save(os.path.join(path, "ids.npy"), a)


# --------------------------------------------------------------------------------------------------------------
def run_b200_arm(args, world, rank, local):
    from layoutdm_b200 import Engine, Vocab, timestep_plan
    from layoutdm_b200.parallel import all_gather_ids
    from layoutdm_b200.synthetic import random_state_dict

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    vocab = Vocab.for_dataset("rico25")
    eng = Engine.from_state_dict(random_state_dict(vocab, num_timesteps=T, seed=0), vocab, num_timesteps=T, operand_dtype=args.dtype, device=local)
    B = args.batch                                    # per GPU (weak scaling: configs[4] = 8 x 1024)
    strong = args.total_batch > 0
    if strong:
        assert args.total_batch % world == 0
        B = args.total_batch // world
    total = B * world
    plan = timestep_plan(T, T)
    cfg = {"name": "random", "temperature": 1.0}
    b0 = rank * B

    def device_pass(seed):
        ids = eng.sample_loop(B, plan, cfg, seed=seed, b_global0=b0)
        return all_gather_ids(ids, total) if world > 1 else ids

    for w in range(max(args.warmup, 3)):
        device_pass(100 + w)
    torch.cuda.synchronize()
    barrier(world)

    # ---- device-resident timing (CUDA events on the launching stream) ----
    l0 = eng.launch_count
    with ClockSampler(local) as cs:
        torch.cuda.synchronize(); barrier(world)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(args.steps):
            out = device_pass(1000 + k)
        e1.record()
        torch.cuda.synchronize(); barrier(world)
        ms_total = e0.elapsed_time(e1)
    launches = eng.launch_count - l0
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    ms_total = max_over_ranks(ms_total, world, dev)
    ms_step = ms_total / args.steps
    value = total / (ms_step * 1e-3)
    clocks = cs.summary()
    assert int(out.max()) < vocab.mask_id, "MASK token survived the loop"

    # ---- end to end through the host-buffer entry (pinned host buffers, H2D + D2H inside the timed region) ----
    init = torch.full((B, vocab.S), vocab.mask_id, dtype=torch.int64).pin_memory()
    host_out = torch.empty(B, vocab.S, dtype=torch.int64).pin_memory()
    eng.sample_host(B, plan, cfg, seed=7, b_global0=b0, ids_init=init, out=host_out)
    torch.cuda.synchronize(); barrier(world)
    t0 = time.perf_counter()
    for k in range(args.steps):
        _, h2d, d2h = eng.sample_host(B, plan, cfg, seed=2000 + k, b_global0=b0, ids_init=init, out=host_out)
    torch.cuda.synchronize(); barrier(world)
    e2e_s = max_over_ranks((time.perf_counter() - t0) / args.steps, world, dev)
    e2e = {"value": total / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d + 2 * 4 * len(plan)), "d2h_bytes_per_step": int(d2h),
           "path": "ldm_sample_host (pinned host ids_init -> H2D, 100-step loop, D2H of final ids); per-rank shard, max over ranks"}

    # ---- per-kernel timing for the roofline (one extra profiled pass; CUDA events around every launch) ----
    eng.profile_begin()
    eng.sample_loop(B, plan, cfg, seed=5, b_global0=b0)
    prof = eng.profile_end()
    peaks = load_peaks()
    gemm = {k: v for k, v in prof.items() if k in FLOPS and v[1] > 0}
    dom = max(gemm, key=lambda k: gemm[k][0])
    dom_ms, dom_n = gemm[dom]
    achieved = FLOPS[dom] * B / (dom_ms / dom_n * 1e-3) / 1e12
    tot_prof = sum(v[0] for v in prof.values())
    traffic, traffic_src = load_traffic(dom) if B == 1024 else (None, None)
    roofline = {"bound": "tensor", "kernel": dom, "achieved": achieved, "peak": peaks["sustained"], "unit": "TFLOP/s",
                "frac": achieved / peaks["sustained"], "traffic": traffic, "traffic_unit": "bytes/launch", "traffic_source": traffic_src,
                "algorithmic_flops_per_launch": FLOPS[dom] * B, "peak_source": peaks["src"] + ", sustained bf16 (kernel timed inside a long step)",
                "share_of_step": dom_ms / tot_prof,
                "kernels": {k: kernel_record(k, v, B, tot_prof, peaks) for k, v in prof.items() if v[1]},
                "hbm_peak_gbs": peaks["hbm"],
                "path_tflops": value / world * T * FLOPS_PER_LAYOUT_STEP / 1e12,
                "path_frac": value / world * T * FLOPS_PER_LAYOUT_STEP / 1e12 / peaks["sustained"]}

    # ---- the other single-GPU BASELINE.json configs (rank 0, N=1 only): parity-test cases, reported as sub-records ----
    configs = None
    if rank == 0 and world == 1 and not args.no_configs:
        configs = other_configs(local)

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload on the host cores; reference on the same GPU ----
    cpu = gpu_eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = physical_cores()
        torch.set_num_threads(cores)
        arm = CpuArm()
        arm.step(0)
        dts = [arm.step(1 + k) for k in range(3)]                 # ~15 s of CPU work in total
        dt = sum(dts) / len(dts)
        cpu = {"value": arm.layouts_per_s(dt), "unit": UNIT, "cores": cores, "kind": arm.kind, "sample": arm.sample_desc(dt) + f"; mean of {len(dts)} steps after 1 warm-up"}
        gpu_eager = gpu_eager_reference(B, dev)
        if gpu_eager:
            gpu_eager["speedup_e2e"] = e2e["value"] / gpu_eager["value"]

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
                "dtype": args.dtype, "data": "synthetic",
                "config": {"workload": f"rico25 unconditional, T=100, batch={B} per GPU, N=25 (S=125 tokens, C=155), sampling=random, random-init weights",
                           "global_batch": total, "parallelism": f"dp{world} (batch-sharded replicas, one all-gather of ids)" if world > 1 else "single GPU",
                           "l2": "per-step activation working set (1.9 GB at B=1024) >> 126 MB L2, no explicit flush needed",
                           "operands": f"{args.dtype} tensor-core operands, fp32 accumulate / LayerNorm / softmax / posterior"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "gpu_eager_baseline": gpu_eager, "configs": configs, "precision": load_precision()}
        emit(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the sub-records of BASELINE.json configs 0 / 2 / 3")
    ap.add_argument("--total-batch", type=int, default=0, help="strong scaling: this many layouts in total, split over the ranks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the ids of the last timed step to DIR/ids.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the output of --impl b200")
    if args.impl == "reference":
        world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
        run_reference_arm(args, world, rank)
        return
    world, rank, local = dist_setup(args.gpus)
    try:
        run_b200_arm(args, world, rank, local)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
