#!/usr/bin/env python
"""bench.py — block-sparse attention at HunyuanVideo 720p (BASELINE.json metric / configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes the output of the last timed step, sampled at fixed token rows, to DIR/out.npy
(see dump_outputs), so that two builds run with the same arguments can be compared output for output.

One step = one pass of the SVG1 sparse attention core over synthetic Q/K/V of the HunyuanVideo 720p
shape (B=1, H=24, S=119056 = 33 frames x 3600 tokens + 256 text, D=128, bf16) under the executed SVG1
band mask at 30 % density (W = 19072, hyvideo/utils.py:20-44,142-151): online profiling (sample_mse ->
best_mask_idx), head placement of Q/K/V, element-exact block-sparse attention, inverse placement of O —
the sparse branch of attention_core_logic (svg/models/hyvideo/attention.py:506-524).  Heads are sharded
across ranks (strong scaling: total work fixed), the output all-gathered once.

Printed JSON (one line, rank 0): the contract keys plus `roofline` (dominant kernel = the tcgen05
attention kernel, CUDA-event timed on its stream), `cpu_baseline` (oracle naive attention on the host
cores, bounded sample), `e2e` (same step through the public API from pinned host buffers, H2D + D2H in
the timed region), `clocks`, `gpu_launches`, and `svg2` (variable-block kernel at rho = 0.30,
QC=400/KC=1000, the SVG2 shape of the same model — reported, not the headline).

--impl reference: times the reference's own CPU formulation of this path (naive masked
torch attention, svg/kernels/test/test_sparse_attn.py:109-157, restated in oracle/attention.py) on all
host cores, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "sparse-videogen_b200"))
sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ for the modules imported from it

import torch  # noqa: E402

# ---- workload constants (SURVEY Appendix A, HunyuanVideo T2V 720p) --------------------------------
H_TOTAL, D, CTX, F, P, PROMPT_LEN = 24, 128, 256, 33, 3600, 60
S = CTX + F * P
SPARSITY = 0.30
N_SAMPLED_ROWS, SAMPLE_MAX_ROW = 64, 10000
DUMP_ROWS = 2048  # token rows kept by --dump-outputs: 24 heads x 2048 x 128 fp32 = 25 MB instead of 1.5 GB


def dump_outputs(out_dir, o):
    """Write the attention output o [1, H, S, D] at DUMP_ROWS token rows drawn once from a fixed seed (sorted) as
    <out_dir>/out.npy, float32 [H, DUMP_ROWS, D]."""
    import numpy as np

    rows = torch.randperm(S, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    sample = o[0].index_select(1, rows.to(o.device)).float().cpu().numpy()
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "out.npy", sample)


def band_width(sparsity=SPARSITY):
    """sparsity_to_width (hyvideo/utils.py:142-151) then floor to 128 (:24-25)."""
    seq = S
    s2 = (sparsity * seq * seq - 2 * seq * CTX) / (seq * seq)
    mul = seq * (1 - math.sqrt(1 - s2)) / P
    return math.floor(mul * P / 128) * 128, mul


def band_pairs(W):
    """number of allowed (q, kv) pairs per head under the HY mask_mod (exact, closed form per row)."""
    V, R = F * P, F * P + PROMPT_LEN
    q = torch.arange(S, dtype=torch.int64)
    lo = torch.clamp(q - (W - 1), min=0)
    hi = torch.clamp(q + (W - 1), max=V - 1)
    band = torch.clamp(hi - lo + 1, min=0)
    per_row = torch.where(q < V, band + PROMPT_LEN, torch.where(q < R, torch.tensor(R), torch.tensor(S - R)))
    return int(per_row.sum().item())


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"burst": d.get("bf16_tflops"), "sustained": d.get("bf16_tflops_sustained"), "hbm": d.get("hbm_gbs"),
                "src": "measured (MEASURED_PEAKS.json)"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm": 6650.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.proc, self.lines, self.index = None, [], index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
                pw.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        # under-load median: drop idle samples (below 60 % of the max seen)
        loaded = [x for x in sm if sm and x >= 0.6 * sm[-1]] or sm
        return {"sm_mhz": loaded[len(loaded) // 2] if loaded else None, "sm_max_mhz": mx,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: naive masked attention on the host cores, bounded sample
# ---------------------------------------------------------------------------------------------------
def usable_cores():
    """Host threads this process may really use: cpu_count capped by the affinity mask and the cgroup CPU quota
    (a container can report 128 CPUs and be allowed 16; oversubscribing makes the CPU arm look worse than it is)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        quota, period = (Path("/sys/fs/cgroup/cpu.max").read_text().split() + ["100000"])[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def cpu_naive_sample(rows=1024, seconds=10.0):
    """One head, up to `rows` query rows spread over the sequence (256 at a time, until `seconds` of work are
    done), full S keys, HY band mask, fp32.  Returns (tflops, seconds, sample description, threads).  Same
    arithmetic as ref_torch_attn_impl (svg/kernels/test/test_sparse_attn.py:109-157)."""
    from oracle.attention import hy_mask_mod

    cores = usable_cores()
    torch.set_num_threads(cores)
    W, mul = band_width()
    g = torch.Generator().manual_seed(0)
    k = torch.randn(S, D, generator=g)
    v = torch.randn(S, D, generator=g)
    qrows = torch.linspace(0, S - 1, rows).long()
    qrows = qrows[torch.randperm(rows, generator=g)]  # any prefix of the sample covers the whole sequence
    q = torch.randn(rows, D, generator=g)
    mod = hy_mask_mod(CTX, PROMPT_LEN, F, P, mul)
    kv_idx = torch.arange(S).view(1, S)
    t0 = time.perf_counter()
    pairs, done = 0, 0
    for r0 in range(0, rows, 256):
        qi = qrows[r0:r0 + 256].view(-1, 1)
        s = (q[r0:r0 + 256] @ k.T) / math.sqrt(D)
        m = mod(qi, kv_idx)
        s = s.masked_fill(~m, float("-inf"))
        w = torch.softmax(s, dim=-1)
        _ = w @ v
        pairs += int(m.sum().item())
        done += qi.numel()
        if time.perf_counter() - t0 >= seconds:
            break
    dt = time.perf_counter() - t0
    # the naive formulation computes every (q, kv) pair and masks afterwards; credit only the
    # algorithmic (allowed) pairs so the unit matches the GPU arm
    flops = 4.0 * D * pairs
    return (flops / dt / 1e12, dt,
            f"1 head, {done} query rows spread over S={S}, all keys, HY band W={W}, {cores} threads", cores)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals, secs = [], []
    for i in range(args.warmup + args.steps):
        tf, dt, sample, cores = cpu_naive_sample(rows=4096, seconds=10.0)
        if i >= args.warmup:
            vals.append(tf)
            secs.append(dt)
    value = sum(vals) / len(vals)
    W, _ = band_width()
    pairs = band_pairs(W)
    ms_call = 4.0 * D * pairs * H_TOTAL / (value * 1e12) * 1e3
    line = {
        "impl": "reference", "metric": "block-sparse attention TFLOP/s (density-adjusted)", "value": value,
        "unit": "TFLOP/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": sum(secs) / len(secs) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "HunyuanVideo-720p SVG1 sparse attention core (sample_mse + placement + band attention "
                               "+ inverse placement), rho=0.30", "S": S, "heads": H_TOTAL, "head_dim": D,
                   "band_W": W, "density": pairs / S / S,
                   "note": "the reference's naive torch attention on the host cores, bounded sample per step; "
                           "ms per call extrapolated", "extrapolated_ms_per_call": ms_call},
        "cpu_baseline": {"value": value, "unit": "TFLOP/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def svg2_map(heads, seed=7, rho=0.30, QC=400, KC=1000, ctx=CTX, plen=PROMPT_LEN, video=F * P):
    """The SVG2 shape of the same model: QC x KC Bernoulli(rho) map over uniform cluster sizes plus HunyuanVideo's prompt
    / padding blocks (hyvideo/attention.py:681-697).  Returns (map [H,QC+t,KC+t] bool, row_sz, col_sz, flops)."""
    gm = torch.Generator().manual_seed(seed)

    def sizes(n):
        b = torch.full((heads, n), video // n, dtype=torch.int32)
        b[:, : video - (video // n) * n] += 1
        return b

    t = 2 if ctx else 0
    row, col = sizes(QC), sizes(KC)
    bm = torch.zeros(heads, QC + t, KC + t, dtype=torch.bool)
    bm[:, :QC, :KC] = torch.rand(heads, QC, KC, generator=gm) < rho
    if ctx:
        extra = torch.tensor([[plen, ctx - plen]] * heads, dtype=torch.int32)
        row, col = torch.cat([row, extra], 1), torch.cat([col, extra], 1)
        bm[:, -2, :-1] = True   # prompt block <-> everything but the padding
        bm[:, :-1, -2] = True
        bm[:, -1, -1] = True
    fl = 4.0 * D * (row.double()[:, :, None] * col.double()[:, None, :] * bm).sum().item()
    return bm, row, col, fl


def _time(fn, warm=2, iters=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def svg2_pipeline_probe(dev, model):
    """Whole SVG2 core (k-means x2, which also returns the cluster-sorted token order -> dynamic map -> permute x3 ->
    plan -> attention with fused inverse permutation) at a model's full shape, on tokens with cluster structure: per-stage CUDA-event times + the total of
    a warm-started step call (2 Lloyd iterations, the reference's steady state)."""
    from svgb200 import core, kmeans_utils as ku
    from svgb200.models import hyvideo as hy, wan

    if model == "hy":
        Hh, ctx, Fm, Pm, QC, KC = 24, CTX, F, P, 400, 1000
        sap = hy.HunyuanSAPCore(ctx, Fm, Pm, num_q_centroids=QC, num_k_centroids=KC, top_p_kmeans=0.9, min_kc_ratio=0.1,
                                kmeans_iter_init=10, kmeans_iter_step=2, prompt_length=PROMPT_LEN)
    else:
        Hh, ctx, Fm, Pm, QC, KC = 40, 0, 21, 3600, 300, 1000
        sap = wan.WanSAPCore(Fm, Pm, num_q_centroids=QC, num_k_centroids=KC, top_p_kmeans=0.9, min_kc_ratio=0.1,
                             kmeans_iter_init=10, kmeans_iter_step=2)
    V, Sm = Fm * Pm, ctx + Fm * Pm
    g = torch.Generator(device=dev).manual_seed(11)
    q, k, v = (torch.randn(1, Hh, Sm, D, device=dev, generator=g).to(torch.bfloat16) for _ in range(3))
    base = torch.randn(1, Hh, 96, D, device=dev, generator=g) * 1.5
    which = torch.randint(0, 96, (Sm,), device=dev, generator=g)
    q = (q.float() * 0.7 + base[:, :, which]).to(torch.bfloat16)
    k = (k.float() * 0.7 + base[:, :, which]).to(torch.bfloat16)
    del base
    sap.sparse_core(q, k, v)  # first call: k-means init
    total = _time(lambda: sap.sparse_core(q, k, v), warm=1, iters=3)
    last = sap.last
    dyn, row_sz, col_sz, q_perm, k_perm = (last[x] for x in ("dynamic_map", "q_sizes", "k_sizes", "q_sorted_indices",
                                                               "k_sorted_indices"))
    qv, kv = q[0, :, :V], k[0, :, :V]  # strided views of the video part, clustered in place like sparse_core does
    qc0, kc0 = sap.state.q_centroids[sap.layer_idx], sap.state.k_centroids[sap.layer_idx]
    st = {}
    st["kmeans_q_2it"] = _time(lambda: ku.batch_kmeans_Euclid_sorted(qv, QC, max_iters=2, init_centroids=qc0), 1, 3)
    st["kmeans_k_2it"] = _time(lambda: ku.batch_kmeans_Euclid_sorted(kv, KC, max_iters=2, init_centroids=kc0), 1, 3)
    ql, qc, qs, _, _ = ku.batch_kmeans_Euclid_sorted(qv, QC, max_iters=2, init_centroids=qc0)
    kl, kc, ks, _, _ = ku.batch_kmeans_Euclid_sorted(kv, KC, max_iters=2, init_centroids=kc0)
    st["dynamic_map"] = _time(lambda: ku.identify_dynamic_map(qc[None], kc[None], qs[None], ks[None], 0.9, 0.1), 1, 3)
    st["permute_x3"] = _time(lambda: (core.permute_gather(q, q_perm), core.permute_gather(k, k_perm),
                                      core.permute_gather(v, k_perm)), 1, 3)
    qp, kp, vp = core.permute_gather(q, q_perm), core.permute_gather(k, k_perm), core.permute_gather(v, k_perm)
    st["plan"] = _time(lambda: core.plan_varblock(dyn, row_sz, col_sz, Sm), 1, 3)
    plan = core.plan_varblock(dyn, row_sz, col_sz, Sm)
    st["attention"] = _time(lambda: core.attn_fwd(qp, kp, vp, plan, o_rows=q_perm), 1, 3)
    fl = 4.0 * D * (row_sz.double()[:, :, None] * col_sz.double()[:, None, :] * dyn).sum().item()
    return {"shape": f"H={Hh} S={Sm} QC={QC} KC={KC} top_p=0.9 (k-means on clustered synthetic tokens)",
            "density": fl / (4.0 * D * Hh * Sm * Sm), "step_call_ms": total, "stages_ms": st,
            "front_half_ms": total - st["attention"], "glue_ms": total - sum(st.values()),
            "attention_tflops": fl / st["attention"] / 1e9,
            "step_tflops": fl / total / 1e9}


def fp8_density_sweep(dev, world, rank, dist):
    """BASELINE configs[4]: Wan 2.1 720p SVG2 shape (S = 75 600, 40 heads, QC = 300 / KC = 1000), bf16 vs FP8 (e4m3)
    variable-block attention at block densities 10-50 %.  Heads are sharded over the ranks (5 per GPU at N = 8); times
    are the max over ranks, TFLOP/s whole-job."""
    from svgb200 import core

    Hw, Fw, Pw = 40, 21, 3600
    Sw = Fw * Pw
    if Hw % world:
        return {"skipped": f"{Hw} heads do not divide over {world} ranks"}
    Hl = Hw // world
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    q, k, v = (torch.randn(1, Hl, Sw, D, device=dev, generator=g).to(torch.bfloat16) for _ in range(3))
    (q8, sq), (k8, sk), (v8, sv) = (core.quantize_e4m3(x) for x in (q, k, v))
    rows = []
    for rho in (0.1, 0.2, 0.3, 0.4, 0.5):
        bm, row, col, fl = svg2_map(Hl, seed=int(rho * 100) + rank, rho=rho, QC=300, KC=1000, ctx=0, plen=0, video=Sw)
        plan = core.plan_varblock(bm.to(dev), row.to(dev), col.to(dev), Sw)
        ms16 = _time(lambda: core.attn_fwd(q, k, v, plan), 1, 3)
        ms8 = _time(lambda: core.attn_fwd_fp8(q8, k8, v8, sq, sk, sv, plan), 1, 3)
        t = torch.tensor([ms16, ms8, fl], device=dev, dtype=torch.float64)
        if world > 1:
            tm = t.clone()
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            ms16, ms8, fl = tm[0].item(), tm[1].item(), t[2].item()
        rows.append({"density": rho, "bf16_ms": ms16, "fp8_ms": ms8, "bf16_tflops": fl / ms16 / 1e9,
                     "fp8_tflops": fl / ms8 / 1e9, "fp8_speedup": ms16 / ms8})
    return {"shape": f"Wan 2.1 720p SVG2: S={Sw}, {Hw} heads ({Hl}/GPU), QC=300 KC=1000 Bernoulli maps, uniform sizes",
            "n_gpus": world, "sweep": rows}


def run_ours(args):
    import torch.distributed as dist

    from svgb200 import core
    from svgb200.models import hyvideo as hy

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    core.device_check()
    assert H_TOTAL % world == 0, "heads must divide across ranks"
    Hl = H_TOTAL // world
    t_wall0 = time.time()

    # synthetic inputs: head h is generated from seed + h so results are identical for any N
    def make(seed_off):
        t = torch.empty(1, Hl, S, D, dtype=torch.bfloat16, device=dev)
        for i in range(Hl):
            g = torch.Generator(device=dev).manual_seed(1000 * seed_off + i * world + rank)  # global head id
            t[0, i] = torch.randn(S, D, generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)
        return t

    q, k, v = make(1), make(2), make(3)
    W, mul = band_width()
    pairs = band_pairs(W)
    flops_total = 4.0 * D * pairs * H_TOTAL
    flops_local = 4.0 * D * pairs * Hl

    proc = hy.HunyuanSVG1Core(context_length=CTX, prompt_length=PROMPT_LEN, num_frame=F, frame_size=P,
                              num_heads=Hl, head_dim=D, sparsity=SPARSITY, num_sampled_rows=N_SAMPLED_ROWS,
                              sample_mse_max_row=SAMPLE_MAX_ROW, device=dev)
    gen = torch.Generator().manual_seed(1234)  # CPU generator like the reference's torch.randint (attention.py:381)
    from svgb200.parallel import HeadParallel

    hp = HeadParallel() if world > 1 else None
    gathered = torch.empty(1, H_TOTAL, S, D, dtype=torch.bfloat16, device=dev) if world > 1 else None
    attn_ev = []

    def step(timed=False, rows=None, trace=None):
        if rows is None:
            rows = torch.randint(0, SAMPLE_MAX_ROW, (N_SAMPLED_ROWS,), generator=gen)
        if world > 1:
            # per-head attention, each head's output all-gather overlapped with the next head's compute
            return proc.sparse_core_head_parallel(q, k, v, hp, sampled_rows=rows, out=gathered,
                                                  attn_events=attn_ev if timed else None, trace=trace)
        return proc.sparse_core(q, k, v, sampled_rows=rows, attn_events=attn_ev if timed else None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = core.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        out = None  # release the previous step's output before this step allocates, as in the warmup steps
        out = step(timed=True)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = core.launch_count - launches0
    clocks = sampler.stop() if rank == 0 else None
    if world == 1:
        attn_ms = sum(a.elapsed_time(b) for a, b in attn_ev) / max(1, args.steps)
    else:
        # per-head launches overlap across streams in the step, so time the dominant kernel on its own:
        # one launch over all local heads (same plan, same inputs), CUDA events on its stream
        attn_ms = _time(lambda: core.attn_fwd(q, k, v, proc.block_mask.plan), 1, 3)
    t = torch.tensor([ms_total, attn_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = t[0].item() / args.steps
    attn_ms = t[1].item()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    del out

    # ---- output checksum on FIXED sampled rows: must be identical for every N (heads are generated per global id,
    # per-head computation does not depend on the sharding) -> compare across the lines of a scaling run
    fixed_rows = torch.randint(0, SAMPLE_MAX_ROW, (N_SAMPLED_ROWS,), generator=torch.Generator().manual_seed(4321))
    o_full = step(rows=fixed_rows)
    torch.cuda.synchronize()
    if world == 1:
        o_all = o_full
    else:
        o_all = gathered
    cs = o_all.double()
    checksum = {"sum": cs.sum().item(), "abs_sum": cs.abs().sum().item(),
                "per_head_sum_first3": [cs[0, h].sum().item() for h in range(3)],
                "note": "fixed sampled rows (seed 4321); equal across N => the gathered [1,24,S,D] output is the same"}
    del cs, o_full

    # ---- N > 1: per-rank stage timeline of one step (event stamps), gathered to rank 0
    timeline = None
    if world > 1:
        tr = {}
        step(rows=fixed_rows, trace=tr)
        torch.cuda.synchronize()
        mine = {"rank": rank, "prologue_ms(sample_mse+placement)": tr["t0"].elapsed_time(tr["start"]),
                "head_compute_done_ms": [tr["t0"].elapsed_time(e) for e in tr["compute_done"]],
                "head_allgather_done_ms": [tr["t0"].elapsed_time(e) for e in tr["comm_done"]],
                "end_ms": tr["t0"].elapsed_time(tr["end"])}
        allr = [None] * world
        dist.all_gather_object(allr, mine)
        if rank == 0:
            ends = [r["end_ms"] for r in allr]
            last_c = [r["head_compute_done_ms"][-1] for r in allr]
            timeline = {"per_rank": allr, "end_ms_max": max(ends), "end_ms_min": min(ends),
                        "last_head_compute_done_ms_max": max(last_c),
                        "exposed_allgather_ms(max end - max last compute)": max(ends) - max(last_c),
                        "attention_alone_ms(one launch, all local heads)": attn_ms,
                        "note": "ms since the step began on each rank; heads alternate over two compute streams, each "
                                "head's ncclAllGather follows on the communication stream"}

    # ---- e2e: pinned host buffers -> H2D -> step -> D2H of the result, through the public API.  N > 1: every head
    # group's output is also all-gathered on the device (same pipeline as `value`); D2H returns the local heads.
    hq, hk, hv = (x.cpu().pin_memory() for x in (q, k, v))
    ho = torch.empty(1, Hl, S, D, dtype=torch.bfloat16).pin_memory()
    hps = 2 if Hl >= 12 else 1

    def e2e_step():
        rows = torch.randint(0, SAMPLE_MAX_ROW, (N_SAMPLED_ROWS,), generator=gen)
        proc.sparse_core_from_host(hq, hk, hv, ho, sampled_rows=rows, heads_per_stage=hps, hp=hp, gathered=gathered)

    e2e_steps = max(2, min(args.steps, 5))
    e2e_step()
    barrier()
    e0.record()
    for _ in range(e2e_steps):
        e2e_step()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1) / e2e_steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = t.item()
    del hq, hk, hv, ho

    # ---- SVG2 variable-block kernel at rho = 0.30 (reported beside the headline)
    svg2 = None
    if rank == 0:
        bm, row, col, fl = svg2_map(Hl)
        plan = core.plan_varblock(bm.to(dev), row.to(dev), col.to(dev), S)
        ms = _time(lambda: core.attn_fwd(q, k, v, plan), 2, 3)
        pk_ = peaks()
        svg2 = {"workload": f"variable-block map QC=400+2 KC=1000+2 Bernoulli(0.30), uniform cluster sizes, {Hl} heads",
                "ms_per_call": ms, "tflops": fl / ms / 1e9, "density": fl / (4.0 * D * Hl * S * S),
                "frac_of_sustained": fl / ms / 1e9 / pk_["sustained"] if pk_["sustained"] else None,
                "dense_equiv_tflops": 4.0 * D * Hl * S * S / ms / 1e9}
        del plan

    # ---- FP8 (e4m3) variant of the same band-mask attention (BASELINE config 5 flavour), reported beside it
    fp8 = None
    if rank == 0:
        try:
            (q8, sq), (k8, sk), (v8, sv) = (core.quantize_e4m3(x) for x in (q, k, v))
            ms8 = _time(lambda: core.attn_fwd_fp8(q8, k8, v8, sq, sk, sv, proc.block_mask.plan), 2, 3)
            msq = _time(lambda: core.quantize_e4m3(q), 1, 2)
            fp8 = {"workload": f"same band mask, e4m3 Q/K/V (per-head scales), bf16 out, {Hl} heads", "ms_per_call": ms8,
                   "tflops": flops_local / ms8 / 1e9, "quantize_ms_per_tensor": msq}
            del q8, k8, v8
        except Exception as e:  # noqa: BLE001
            fp8 = {"error": repr(e)[:200]}

    # ---- pre-attention chain (SURVEY 8f-1): fused transpose + QK-RMSNorm + RoPE, HBM-bound
    prep = None
    if rank == 0:
        try:
            qi, ki, vi = (torch.randn(1, S, Hl * D, device=dev).bfloat16() for _ in range(3))
            gq, gk = (torch.randn(D, device=dev).bfloat16() for _ in range(2))
            cos, sin = (torch.randn(S - CTX, D, device=dev) for _ in range(2))
            outs = tuple(torch.empty(1, Hl, S, D, device=dev, dtype=torch.bfloat16) for _ in range(3))

            def prep_call():
                core.qkv_prep(qi, ki, vi, Hl, out=outs, norm=core.NORM_RMS_HEAD, gamma_q=gq, gamma_k=gk, eps=1e-6, rope=1,
                              cos=cos, sin=sin, rope_lo=0, rope_n=S - CTX)
            msp = _time(prep_call, 2, 5)
            nbytes = 6 * Hl * S * D * 2
            hbm = peaks()["hbm"]
            prep = {"workload": f"[1,S,{Hl}x{D}] q,k,v -> [1,{Hl},S,{D}]: transpose + per-head RMSNorm(q,k) + RoPE (text last)",
                    "ms_per_call": msp, "algorithmic_bytes": nbytes, "gbs": nbytes / msp / 1e6,
                    "hbm_peak_gbs": hbm, "frac": (nbytes / msp / 1e6 / hbm) if hbm else None}
            del qi, ki, vi, outs
        except Exception as e:  # noqa: BLE001
            prep = {"error": repr(e)[:200]}

    del q, k, v, gathered
    torch.cuda.empty_cache()

    # ---- BASELINE configs[4]: FP8 density sweep at the Wan shape (all ranks: heads sharded)
    fp8_sweep = None
    if not args.no_extras:
        try:
            fp8_sweep = fp8_density_sweep(dev, world, rank, dist)
        except Exception as e:  # noqa: BLE001
            fp8_sweep = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- BASELINE configs[2] + the SVG2 front half: whole SAP core per stage at the HY and Wan shapes (N = 1 only)
    svg2_pipeline = None
    if world == 1 and not args.no_extras:
        svg2_pipeline = {}
        for model in ("hy", "wan"):
            try:
                svg2_pipeline[model] = svg2_pipeline_probe(dev, model)
            except Exception as e:  # noqa: BLE001
                svg2_pipeline[model] = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()

    # ---- the reference's own GPU paths on this box (north_star: >= 1.5x), as a subprocess under a timeout
    ref_gpu = None
    if world == 1 and not args.no_ref_gpu and not args.no_extras:
        try:
            r = subprocess.run([sys.executable, str(ROOT / "tools" / "ref_gpu_paths.py"), "--heads", str(H_TOTAL)],
                               capture_output=True, text=True, timeout=args.ref_gpu_timeout,
                               env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
            for ln in r.stdout.splitlines():
                if ln.startswith("REF_GPU_JSON "):
                    ref_gpu = json.loads(ln[len("REF_GPU_JSON "):])
            if ref_gpu is None:
                ref_gpu = {"error": "no result", "rc": r.returncode, "stderr_tail": r.stderr[-400:]}
        except subprocess.TimeoutExpired:
            ref_gpu = {"error": f"timed out after {args.ref_gpu_timeout} s"}
        except Exception as e:  # noqa: BLE001
            ref_gpu = {"error": repr(e)[:300]}

    pk = peaks()
    achieved = flops_local / attn_ms / 1e9 if attn_ms > 0 else None
    traffic, traffic_src = None, None
    tj = ROOT / "profiles" / "attn_traffic.json"
    if tj.exists():
        try:
            tjd = json.loads(tj.read_text())
            traffic = tjd.get("dram_bytes_per_launch")
            traffic_src = "profiles/attn_traffic.json (" + str(tjd.get("source", "ncu --set full capture")) + "); not measured in this run"
        except Exception:
            traffic = None
    tf_cpu, dt_cpu, sample, cores = cpu_naive_sample(rows=4096, seconds=12.0)
    value = flops_total / ms_step / 1e9
    bytes_in = 3 * Hl * S * D * 2
    bytes_out = Hl * S * D * 2
    line = {
        "metric": "block-sparse attention TFLOP/s (density-adjusted)", "value": value, "unit": "TFLOP/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "HunyuanVideo-720p SVG1 sparse attention core (sample_mse + placement + band attention "
                               "+ inverse placement), rho=0.30", "S": S, "heads": H_TOTAL, "head_dim": D,
                   "band_W": W, "density": pairs / S / S, "heads_per_gpu": Hl, "parallelism": f"head-parallel x{world}",
                   "l2": "inputs (2.2 GB/GPU-set) larger than L2; no flush needed",
                   "attn_ms_per_call": attn_ms, "flops_per_call": flops_total},
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": pk["sustained"], "unit": "TFLOP/s",
                     "frac": (achieved / pk["sustained"]) if achieved and pk["sustained"] else None,
                     "frac_of_burst": (achieved / pk["burst"]) if achieved and pk["burst"] else None,
                     "peak_src": pk["src"] + ", sustained (kernel runs ~50 ms back to back)",
                     "kernel": "svgb::attn_fwd_kernel<128,DT_BF16>", "traffic": traffic, "traffic_src": traffic_src},
        "cpu_baseline": {"value": tf_cpu, "unit": "TFLOP/s", "cores": cores, "kind": "port", "sample": sample,
                         "seconds": dt_cpu,
                         "bound_by": "the naive formulation itself: it computes all S keys for every sampled query row, "
                                     "builds the boolean mask and masked_fill's a [256, 119056] fp32 score block before "
                                     "the softmax; only the allowed pairs are credited as FLOPs"},
        "e2e": {"value": flops_total / e2e_ms / 1e9, "unit": "TFLOP/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": bytes_in, "d2h_bytes_per_step": bytes_out,
                "note": "per rank: H2D of its heads' Q,K,V, compute, (N>1: device all-gather of every head's output, as in "
                        "`value`), D2H of its heads' output; 3-stream pipeline, heads_per_stage=%d" % hps},
        "clocks": clocks, "gpu_launches": launches, "output_checksum": checksum, "scaling_timeline": timeline,
        "svg2": svg2, "svg2_pipeline": svg2_pipeline, "fp8": fp8, "fp8_sweep": fp8_sweep, "prep": prep,
        "ref_gpu": ref_gpu, "wall_s": time.time() - t_wall0,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="headline + roofline + e2e only (skip SVG2 pipeline, FP8 sweep, ref_gpu)")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip timing the reference's own GPU paths")
    ap.add_argument("--ref-gpu-timeout", type=float, default=420.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's output, sampled at fixed token rows, to DIR/out.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
