#!/usr/bin/env python
"""Benchmark of the decoder-block hot path (fused residual Add-RMSNorm -> SwiGLU feed-forward).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload 11b|90b] [--mode prefill|train]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic activations: norm2(attn_out, residual) ->
ff(normed) (reference Model/model.py:271-272) at BASELINE.json configs[1] (Llama-3.2-11B text block, hidden 4096,
hidden_dim 14336, bf16 prefill, 4 x 2048 tokens).  Prints ONE JSON line on rank 0 (contract in the task statement):
  value   : whole-job tokens/s with inputs resident in HBM (CUDA events, barrier + synchronize on both sides,
            max over ranks);
  e2e     : the same metric through the public module API with HOST (pinned) input buffers and a host copy of
            the result, host<->device copies inside the timed region (double-buffered on copy streams);
  roofline: dominant kernel = the fused gate/up tcgen05 GEMM, achieved TFLOP/s from CUDA events recorded around
            that launch inside the timed region, against MEASURED_PEAKS.json;
  cpu_baseline: the reference's own CPU path (PyTorch fp32 expressions, oracle port) on this box's host cores, full
            4 x 2048-token steps;
  extra   : the other quantities BASELINE.json's metric names, measured in the same process -- Add-RMSNorm GB/s, KV-decode
            FFN us/step, training steps, a >= 3 s sustained loop, what the reference executes on a GPU today (cuBLAS
            F.linear x 3 + eager SiLU*mul + eager norm) and the reference's own fp16 CUDA RMSNorm kernel (oracle/_ref) at
            the same shapes, and `config5_90b_strong`: BASELINE.json configs[4] (90B text block, 4 x 2048 tokens IN
            TOTAL, tensor-parallel over the N GPUs of this run) with its efficiency against one GPU measured in the run.
--impl reference times the CPU path alone (rank 0 only) and prints the same line with "impl": "reference".
N > 1: tensor-parallel FFN (column-sharded gate/up, row-sharded down), sequence-parallel Add-RMSNorm.  Default
--scaling weak: every GPU keeps config 2's 4 x 2048 tokens (global batch = N x 8192; per-GPU flops fixed, the exchanged
bytes per GPU grow with N); --scaling strong keeps the global batch at 8192 tokens.  Default --tp-impl fused: the all-gather
is pulled over NVLink inside the gate/up tcgen05 GEMM and the reduce-scatter is pushed from the down-GEMM epilogue (peer
memory, no NCCL on the data path); --tp-impl nccl is the NCCL reduce-scatter / all-gather baseline with the same sharding.
Before anything is timed at N > 1, every rank checks 64 of its output rows against the CPU oracle (`tp_parity_rel_l2`, exit
code 3 above 1e-2).  --mode train times forward + backward (all FFN weights and gamma trainable), tensor-parallel at N > 1.
"""
from __future__ import annotations

import argparse
import glob
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (hidden, inter, batch, seq, label)
    "11b": (4096, 14336, 4, 2048, "llama-3.2-11b-vision text block: add-rmsnorm + swiglu ffn, bf16 prefill 4x2048 tokens"),
    "90b": (8192, 28672, 4, 2048, "llama-3.2-90b-vision text block: add-rmsnorm + swiglu ffn, bf16 prefill 4x2048 tokens"),
}
METRIC = "ffn_block_tokens_per_sec"
UNIT = "tokens/s"
EPS = 1e-5
PARITY_TOL = 1e-2


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"],
                    bf16_tflops_sustained=p.get("bf16_tflops_sustained"), source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0,
                source="fallback (B200_PROFILING.md)")


def config_for(args, world):
    """The `config` object of the JSON line: a pure function of the command line, so both arms print the same one."""
    hidden, inter, batch, seq, label = WORKLOADS[args.workload]
    weak = world > 1 and args.scaling == "weak"
    tokens = batch * seq * (world if weak else 1)
    train = args.mode == "train"
    return {"workload": label + (" fwd+bwd (all weights trainable)" if train else " forward"),
            "hidden": hidden, "hidden_dim": inter, "global_batch_tokens": tokens, "tokens_per_gpu": tokens // world,
            "parallelism": (f"tp{world} ({args.tp_impl}), sequence-parallel norm" if world > 1 else "single-gpu"),
            "l2_policy": "inputs larger than L2: ~0.85 GB touched per step, 2 rotating activation buffers"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()

        def parse(rows):
            sm, mx, pw, reasons = [], [], [], set()
            for _, line in rows:
                f = [v.strip() for v in line.split(",")]
                if len(f) < 8:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, pw, reasons

        inside = [r for r in self.rows if t0 is None or (t0 <= r[0] <= t1 + 0.15)]
        note = None
        sm, mx, pw, reasons = parse(inside)
        if not sm:
            sm, mx, pw, reasons = parse(self.rows)
            note = "timed region shorter than one 100 ms sample; all samples of the run used"
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
               "reasons": sorted(reasons)}
        if note:
            out["note"] = note
        return out


# ------------------------------------------------------------------------------------------------ CPU reference
def cpu_reference(hidden, inter, tokens, steps, warmup, min_seconds=0.0, max_seconds=60.0):
    """The reference's live CPU path for this hot path (PyTorch fp32: Model/model.py:166-171 +
    Tools/swiglu/FusedSwiglu.py:18-20 + model.py:217), restated in oracle/ffn_oracle.py, on all host cores.
    Each step processes `tokens` tokens.  Returns (tokens_per_s, ms_per_step, cores, steps)."""
    from oracle import ffn_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(tokens, hidden, generator=g)
    res = torch.randn(tokens, hidden, generator=g)
    gamma = 1 + 0.1 * torch.randn(hidden, generator=g)
    wg = (torch.rand(inter, hidden, generator=g) * 2 - 1) / hidden ** 0.5
    wu = (torch.rand(inter, hidden, generator=g) * 2 - 1) / hidden ** 0.5
    wd = (torch.rand(hidden, inter, generator=g) * 2 - 1) / inter ** 0.5

    def step():
        with torch.no_grad():
            return O.feedforward(O.add_rmsnorm(x, gamma, EPS, res), wg, wu, wd)

    for _ in range(warmup):
        step()
    done, t0 = 0, time.perf_counter()
    while True:
        step()
        done += 1
        el = time.perf_counter() - t0
        if (done >= steps and el >= min_seconds) or el >= max_seconds:
            break
    return tokens * done / el, el / done * 1e3, torch.get_num_threads(), done


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path, on this box's host cores, at OUR arm's config
    (full 4 x 2048-token steps), exactly --steps timed steps."""
    hidden, inter, batch, seq, label = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    tokens = batch * seq
    tps, ms, cores, done = cpu_reference(hidden, inter, tokens, args.steps, min(args.warmup, 2), max_seconds=float("inf"))
    sample_txt = (f"{done} full steps of {tokens} tokens (one GPU's share of the workload), fp32, torch CPU (MKL) with {cores} "
                  "threads; oracle port of reference Model/model.py:166-171,217 + Tools/swiglu/FusedSwiglu.py:18-20")
    line = {
        "impl": "reference", "metric": METRIC, "value": tps, "unit": UNIT, "n_gpus": args.gpus, "steps": done,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak" if (world == 1 or args.scaling == "weak") else "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_for(args, world),
        "note": "reference CPU path on host cores (the reference has no working accelerated FFN); rank 0 only",
        "cpu_baseline": {"value": tps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample_txt},
        "e2e": {"value": tps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ helpers
def _time_cuda(fn, iters, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3   # seconds


def _time_cuda_graph(fn, iters, warm=3):
    """Device time per call: `iters` calls captured into ONE CUDA graph, one warm replay, one timed replay.  For kernels of
    ~0.1 ms the Python + ctypes + tensor-map-encode cost of an eager call can exceed the kernel; a serving loop replays graphs."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    try:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(iters):
                fn()
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters * 1e-3   # seconds
    except RuntimeError:                             # a capture this torch build refuses: time the eager launches instead
        torch.cuda.synchronize()
        return _time_cuda(fn, iters, warm=1)


def _gpu_weights(hidden, inter, dev, seed, dt=torch.bfloat16):
    """gamma, w_gate, w_up, w_down drawn on the device exactly as the modules initialise them (U(+-1/sqrt(fan_in)),
    gamma = 1 + 0.1 N(0,1)); the same seed gives the same tensors on every rank."""
    gen = torch.Generator(device=dev).manual_seed(seed)
    uni = lambda r, c: ((torch.rand(r, c, device=dev, generator=gen) * 2 - 1) / c ** 0.5).to(dt)
    gamma = (1 + 0.1 * torch.randn(hidden, device=dev, generator=gen)).to(dt)
    return gamma, uni(inter, hidden), uni(inter, hidden), uni(hidden, inter)


def oracle_rows_rel_l2(y_rows, x_rows, r_rows, gamma, wg, wu, wd):
    """CHECKER (not timed, not shipped): rel-L2 of `y_rows` against the CPU oracle on the same rows, fp32."""
    from oracle import ffn_oracle as O
    f = lambda t: t.detach().float().cpu()
    ref = O.feedforward(O.add_rmsnorm(f(x_rows), f(gamma), EPS, f(r_rows)), f(wg), f(wu), f(wd))
    return float(O.rel_l2(f(y_rows), ref))


def _max_over_ranks(v, dev, world):
    if world == 1:
        return v
    import torch.distributed as dist
    t = torch.tensor([v], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _gather_floats(v, dev, world):
    if world == 1:
        return [v]
    import torch.distributed as dist
    t = torch.tensor([v], device=dev, dtype=torch.float64)
    out = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [float(o.item()) for o in out]


def _timed_steps(fn, steps, warm, dev, world):
    """barrier + synchronize, K steps between CUDA events, barrier + synchronize; max over ranks.  Seconds per step."""
    import torch.distributed as dist
    for i in range(warm):
        fn(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    return _max_over_ranks(e0.elapsed_time(e1), dev, world) / steps * 1e-3


DUMP_BUDGET_BYTES = 60 << 20     # all arrays together, headers included, stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Write every tensor of `arrays` as out_dir/<name>.npy in float32, so that two builds run with the same arguments can be
    compared output for output.  Smallest first, each array gets an equal share of what is left of DUMP_BUDGET_BYTES, so the
    room small arrays do not use goes to the large ones.  An array larger than its share is stored as a 2-D sample of its rows
    (last dimension kept whole), drawn from a fixed seed and sorted, so every run stores the same rows."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BUDGET_BYTES
    for n, (name, t) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].numel())):
        t = t.detach()
        share = left // (len(arrays) - n)
        if t.numel() * 4 > share:
            rows = t.reshape(-1, t.shape[-1])
            keep = share // (rows.shape[1] * 4)
            idx = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = rows[idx.to(rows.device)]
        left -= t.numel() * 4
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


# ------------------------------------------------------------------------------------------------ secondary numbers
def torch_eager_block(x, r, gamma, wg, wu, wd):
    """What the REFERENCE executes on a GPU today for this path with 16-bit CUDA tensors when its extensions are absent
    (they are: swiglu_fused cannot be imported, rmsnorm is fp16-only): the eager PyTorch expressions of
    Model/model.py:166-171 and Tools/swiglu/FusedSwiglu.py:18-20 + model.py:217 -- cuBLAS F.linear x 3 + elementwise kernels."""
    F = torch.nn.functional
    h = x + r
    variance = h.pow(2).mean(-1, keepdim=True)
    normed = h * torch.rsqrt(variance + EPS) * gamma
    return F.linear(F.silu(F.linear(normed, wg)) * F.linear(normed, wu), wd)


def load_ref_cuda_rmsnorm():
    """The reference's own CUDA RMSNorm extension built by oracle/build_ref.sh (checker / baseline only); None if absent."""
    import importlib.util
    so = glob.glob(os.path.join(ROOT, "oracle", "_ref", "rmsnorm_ref*.so"))
    if not so:
        return None
    try:
        spec = importlib.util.spec_from_file_location("rmsnorm_ref", so[0])
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    except Exception:   # noqa: BLE001 -- a baseline that does not load is reported as absent, never fatal
        return None


def extra_numbers(dev, peaks):
    """The other headline quantities of BASELINE.json's metric, measured in the same process (single GPU).  Every
    HBM-bound kernel rotates >= 3 buffer sets larger than the 126 MB L2."""
    from llama32_b200 import ops
    import llama32_b200 as L
    dt = torch.bfloat16
    out = {}
    gen = torch.Generator(device=dev).manual_seed(7)
    rnd = lambda *s, d=dt: torch.randn(*s, device=dev, generator=gen).to(d)
    hbm = peaks["hbm_gbs"]
    st = {"i": 0}

    def nx():
        st["i"] += 1
        return st["i"]

    # ---- Add-RMSNorm at the config-2 (8192 x 4096) and config-5 (8192 x 8192) activation shapes, bf16; and in fp16 beside the
    #      reference's own CUDA kernel (Tools/rmsnorm/rmsnorm.cu:7-61 compiled into oracle/_ref; fp16 is all it supports)
    ref_ext = load_ref_cuda_rmsnorm()
    ref_cmp = {}
    for T, H in ((8192, 4096), (8192, 8192)):
        nb = 6 if H == 4096 else 4
        b = T * H * 2
        gamma = (1 + 0.1 * torch.randn(H, device=dev, generator=gen)).to(dt)
        rms = torch.rand(T, device=dev, generator=gen) + 0.5
        xs, rs, dys = ([rnd(T, H) for _ in range(nb)] for _ in range(3))
        t = _time_cuda(lambda: ops.add_rmsnorm_forward(xs[nx() % nb], gamma, rs[nx() % nb], EPS, want_rms=False), 100)
        out[f"add_rmsnorm_fwd_{T}x{H}"] = {"us": t * 1e6, "GBps": 3 * b / t / 1e9, "frac_of_measured_hbm": 3 * b / t / 1e9 / hbm,
                                           "algorithmic_bytes": 3 * b,
                                           "note": "above 1.0 = part of the output is absorbed by the 126 MB L2 (ncu: DRAM writes "
                                                   "< output bytes), not > 100 % DRAM"}
        t = _time_cuda(lambda: ops.rmsnorm_backward(dys[nx() % nb], xs[nx() % nb], gamma, rms), 100)
        out[f"rmsnorm_bwd_{T}x{H}"] = {"us": t * 1e6, "GBps": 3 * b / t / 1e9, "frac_of_measured_hbm": 3 * b / t / 1e9 / hbm,
                                       "algorithmic_bytes": 3 * b}
        if ref_ext is not None:
            xh, rh, dyh = ([v.half() for v in vs] for vs in (xs, rs, dys))
            gh = gamma.half()
            ours_f = _time_cuda(lambda: ops.add_rmsnorm_forward(xh[nx() % nb], gh, rh[nx() % nb], EPS, want_h=True), 50)
            # the reference kernel updates `residual` in place (residual := input + residual): the same 4 streams as want_h
            ref_f = _time_cuda(lambda: ref_ext.forward(xh[nx() % nb], gh, rh[nx() % nb], EPS), 50)
            ours_b = _time_cuda(lambda: ops.rmsnorm_backward(dyh[nx() % nb], xh[nx() % nb], gh, rms), 50)
            ref_b = _time_cuda(lambda: ref_ext.backward(dyh[nx() % nb], xh[nx() % nb], gh, rms), 50)
            ref_cmp[f"{T}x{H}"] = {"fwd_us_reference_kernel": ref_f * 1e6, "fwd_us_ours": ours_f * 1e6, "fwd_speedup": ref_f / ours_f,
                                   "bwd_us_reference_kernel": ref_b * 1e6, "bwd_us_ours": ours_b * 1e6, "bwd_speedup": ref_b / ours_b}
            del xh, rh, dyh
        del xs, rs, dys
    out["ref_cuda_rmsnorm_fp16"] = ref_cmp if ref_cmp else {"unavailable": "oracle/_ref/rmsnorm_ref*.so not built / not loadable"}
    if ref_cmp:
        out["ref_cuda_rmsnorm_fp16"]["what"] = ("the reference's own fp16 CUDA kernels (Tools/rmsnorm/rmsnorm.cu:7-61, rmsnorm.cuh:13-154) "
                                                "compiled for sm_100a from the reference sources (oracle/build_ref.sh), timed beside "
                                                "ours in fp16 on the same rotating buffers; forward = 4 streams (h written) on both sides")
    torch.cuda.empty_cache()

    # ---- KV-cached decode FFN (config 3), 11B shape, 3 rotating weight sets (1.06 GB)
    H, I = 4096, 14336
    ws = [_gpu_weights(H, I, dev, 100 + k) for k in range(3)]
    gamma = ws[0][0]
    wbytes = 3.0 * H * I * 2
    for B in (1, 16, 32, 64):
        x = rnd(B, 1, H)
        r = rnd(B, 1, H)

        def dec():
            _, wg, wu, wd = ws[nx() % 3]
            ops.ffn_forward(ops.add_rmsnorm_forward(x, gamma, r, EPS, want_rms=False)[0], wg, wu, wd)
        t = _time_cuda(dec, 150, warm=10)
        out[f"decode_11b_batch{B}"] = {"us_per_step": t * 1e6, "tokens_per_s": B / t, "GBps": wbytes / t / 1e9,
                                       "frac_of_measured_hbm": wbytes / t / 1e9 / hbm, "algorithmic_bytes": wbytes,
                                       "what": "add-rmsnorm + FFN per decode step, weights streamed from HBM"}

    # ---- what the reference executes on a GPU today at config 2 (cuBLAS F.linear x 3 + eager elementwise), same buffers
    T = 8192
    _, wg, wu, wd = ws[0]
    xs2, rs2 = [rnd(T, H) for _ in range(2)], [rnd(T, H) for _ in range(2)]

    def ours_step():
        i = nx() % 2
        ops.ffn_forward(ops.add_rmsnorm_forward(xs2[i], gamma, rs2[i], EPS, want_rms=False)[0], wg, wu, wd)

    def eager_step():
        i = nx() % 2
        with torch.no_grad():
            torch_eager_block(xs2[i], rs2[i], gamma, wg, wu, wd)
    t_ours = _time_cuda(ours_step, 20, warm=5)
    t_eager = _time_cuda(eager_step, 20, warm=5)
    out["gpu_fallback_ffn_11b"] = {"ms_per_step_torch_eager": t_eager * 1e3, "tokens_per_s_torch_eager": T / t_eager,
                                   "ms_per_step_ours": t_ours * 1e3, "tokens_per_s_ours": T / t_ours, "speedup_ours": t_eager / t_ours,
                                   "what": "same GPU, same shape (8192 x 4096 -> 14336), dtype bf16 and buffers: the reference's eager "
                                           "PyTorch path (Model/model.py:166-171 + FusedSwiglu.py:18-20 + model.py:217 = cuBLAS "
                                           "F.linear x 3 + elementwise kernels) vs this repository's three kernels"}

    # ---- sustained: >= 3 s of back-to-back steps (the GPU settles under its power cap), clocks sampled inside the loop
    n_sus = max(200, int(3.2 / t_ours))
    for _ in range(20):
        ours_step()
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    time.sleep(0.2)
    k_ev = []
    tw0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for it in range(n_sus):
        i = it % 2
        normed = ops.add_rmsnorm_forward(xs2[i], gamma, rs2[i], EPS, want_rms=False)[0]
        if it % 25 == 24:
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            act, _, _ = ops.swiglu_forward(normed, wg, wu)
            b_.record()
            k_ev.append((a, b_))
        else:
            act, _, _ = ops.swiglu_forward(normed, wg, wu)
        ops.linear_forward(act, wd)
    e1.record()
    torch.cuda.synchronize()
    tw1 = time.time()
    clocks = sampler.stop(tw0, tw1)
    t_sus = e0.elapsed_time(e1) / n_sus * 1e-3
    k_ms = statistics.mean(a.elapsed_time(b_) for a, b_ in k_ev[len(k_ev) // 2:])   # second half: settled clocks
    k_tf = 4.0 * T * H * I / (k_ms * 1e-3) / 1e12
    sus_peak = peaks["bf16_tflops_sustained"] or peaks["bf16_tflops"]
    out["sustained_prefill_11b"] = {
        "seconds": e0.elapsed_time(e1) * 1e-3, "steps": n_sus, "ms_per_step": t_sus * 1e3, "tokens_per_s": T / t_sus,
        "step_TFLOPs": 6.0 * T * H * I / t_sus / 1e12, "gate_up_kernel_ms": k_ms, "gate_up_TFLOPs": k_tf,
        "gate_up_frac_of_bf16_burst_peak": k_tf / peaks["bf16_tflops"], "gate_up_frac_of_bf16_sustained_peak": k_tf / sus_peak,
        "clocks": clocks,
        "what": "the config-2 step repeated back to back for >= 3 s; gate/up kernel timed by CUDA events around every 25th launch "
                "(second half of the loop); peaks = cuBLAS bf16 burst / 4-s sustained figures of MEASURED_PEAKS.json"}
    del xs2, rs2

    # ---- 11B training step (config 4 without the LoRA side path: all FFN weights trainable), fwd + bwd
    norm = L.LLAMARMSNorm(H, eps=EPS).to(dev, dt)
    ffn = L.FusedFeedforward(H, I).to(dev, dt)
    with torch.no_grad():
        ffn.swiglu.w_gate.copy_(wg); ffn.swiglu.w_up.copy_(wu); ffn.w_down.weight.copy_(wd)
    del ws, wg, wu, wd
    x, r, dy = rnd(T, H), rnd(T, H), rnd(T, H)

    def train_step():
        xx = x.detach().requires_grad_(True)
        ffn(norm(xx, residual=r)).backward(dy)
    t = _time_cuda(train_step, 10, warm=3)
    fl = 18.0 * T * H * I
    out["train_11b_fwd_bwd_8192tok"] = {"ms": t * 1e3, "tokens_per_s": T / t, "TFLOPs": fl / t / 1e12,
                                        "frac_of_bf16_burst_peak": fl / t / 1e12 / peaks["bf16_tflops"]}
    # ---- config 4 proper: LoRA (rank 16, alpha 32) on a frozen w_down, gate / up trainable; adapter fused into the GEMMs
    lo = L.Linear_LORA(I, H, rank=16, alpha=32.0, dropout=0.0).to(dev, dt)
    with torch.no_grad():
        lo.linear.weight.copy_(ffn.w_down.weight)
        lo.lora_b.weight.normal_(0, 0.02)
    ffn.w_down = lo
    t = _time_cuda(train_step, 10, warm=3)
    fl = 16.0 * T * H * I                                # 6 fwd + d_act 2 + dX 4 + dWg/dWu 4 (no dW_down); O(rank) terms ignored
    out["train_11b_lora_r16_fwd_bwd_8192tok"] = {"ms": t * 1e3, "tokens_per_s": T / t, "TFLOPs": fl / t / 1e12,
                                                 "frac_of_bf16_burst_peak": fl / t / 1e12 / peaks["bf16_tflops"]}
    del norm, ffn, lo, x, r, dy
    torch.cuda.empty_cache()

    # ---- lm_head + shifted cross entropy (SURVEY.md 8f rank 4) at the 11B sizes: 8192 tokens, hidden 4096, vocab 128 256
    V = 128256
    head = torch.nn.Linear(H, V, bias=False).to(dev, dt)
    hs = rnd(4, 2048, H)
    labels = torch.randint(0, V, (4, 2048), device=dev, generator=gen)
    fl = 2.0 * T * H * V

    def ours_fwd():
        with torch.no_grad():
            L.lm_head_loss(head, hs, labels)

    def eager_fwd():
        with torch.no_grad():
            logits = head(hs)
            torch.nn.functional.cross_entropy(logits[..., :-1, :].reshape(-1, V), labels[..., 1:].reshape(-1), ignore_index=-100)

    def ours_train():
        x_ = hs.detach().requires_grad_(True)
        head.weight.grad = None
        L.lm_head_loss(head, x_, labels)[1].backward()
    t_f = _time_cuda(ours_fwd, 5, warm=2)
    t_e = _time_cuda(eager_fwd, 5, warm=2)
    t_t = _time_cuda(ours_train, 5, warm=2)
    out["lm_head_ce_11b_8192tok"] = {"fwd_ms": t_f * 1e3, "fwd_TFLOPs": fl / t_f / 1e12, "fwd_frac_of_bf16_burst_peak": fl / t_f / 1e12 / peaks["bf16_tflops"],
                                     "fwd_ms_torch_eager": t_e * 1e3, "fwd_speedup_vs_torch_eager": t_e / t_f,
                                     "fwd_bwd_ms": t_t * 1e3, "fwd_bwd_TFLOPs": 3 * fl / t_t / 1e12,
                                     "what": "logits (bf16, stored) + mean shifted cross entropy in one tcgen05 GEMM whose epilogue gathers "
                                             "the softmax statistics (Model/model.py:429-438); eager = nn.Linear + F.cross_entropy in bf16"}
    del head, hs, labels
    torch.cuda.empty_cache()

    # ---- attention (SURVEY.md 8f rank 3) at the 11B geometry: 32 query / 8 KV heads of 128, 4 x 2048 tokens, causal prefill;
    #      then KV-cached decode steps at batch 64 with 2048 cached tokens.  Baselines on the same GPU: the reference's own
    #      expressions (materialised scores + repeat_kv, Model/model.py:238-253) and torch's fused SDPA.
    from llama32_b200 import ops as _ops
    Bq, Tq, NH, NKV, D = 4, 2048, 32, 8, 128
    q = rnd(Bq, Tq, NH * D)
    ck, cv = torch.zeros(Bq, NKV, Tq, D, device=dev, dtype=dt), torch.zeros(Bq, NKV, Tq, D, device=dev, dtype=dt)
    ck.copy_(rnd(Bq, NKV, Tq, D)); cv.copy_(rnd(Bq, NKV, Tq, D))
    fl_att = 4.0 * Bq * NH * Tq * Tq * D / 2                          # causal: half of the score matrix
    t_ours_eager = _time_cuda(lambda: _ops.gqa_attention_forward(q, ck, cv, Tq, 0, causal=True), 20, warm=3)
    t_ours = _time_cuda_graph(lambda: _ops.gqa_attention_forward(q, ck, cv, Tq, 0, causal=True), 20)
    q4 = q.view(Bq, Tq, NH, D).transpose(1, 2)

    def sdpa():
        with torch.no_grad():
            torch.nn.functional.scaled_dot_product_attention(q4, ck, cv, is_causal=True, enable_gqa=True)

    def eager_ref():
        with torch.no_grad():
            kk = ck[:, :, None].expand(Bq, NKV, NH // NKV, Tq, D).reshape(Bq, NH, Tq, D)
            vv = cv[:, :, None].expand(Bq, NKV, NH // NKV, Tq, D).reshape(Bq, NH, Tq, D)
            sc = q4 @ kk.transpose(2, 3) + causal_mask
            (torch.softmax(sc / D ** 0.5, dim=-1) @ vv).transpose(1, 2).contiguous()
    causal_mask = torch.triu(torch.full((Tq, Tq), float("-inf"), device=dev, dtype=dt), diagonal=1)[None, None]
    try:
        t_sdpa = _time_cuda_graph(sdpa, 20)
    except Exception:   # noqa: BLE001 -- a baseline that this torch build cannot run is reported as absent
        try:
            t_sdpa = _time_cuda(sdpa, 20, warm=3)
        except Exception:   # noqa: BLE001
            t_sdpa = None
    t_eager = _time_cuda(eager_ref, 5, warm=2)
    out["attention_prefill_11b_4x2048"] = {"ms": t_ours * 1e3, "TFLOPs": fl_att / t_ours / 1e12, "ms_reference_expressions": t_eager * 1e3,
                                           "speedup_vs_reference_expressions": t_eager / t_ours,
                                           "ms_torch_sdpa": (t_sdpa * 1e3 if t_sdpa else None),
                                           "ms_eager_launch_from_python": t_ours_eager * 1e3,
                                           "timing": "device time: 20 calls captured in one CUDA graph, timed replay (ours and SDPA alike)",
                                           "what": "causal GQA forward, 32/8 heads x 128, bf16: flash-style tcgen05 kernel vs the reference's "
                                                   "materialised-score expressions (Model/model.py:244-252) and torch SDPA (library flash kernel)"}
    del q, q4, ck, cv, causal_mask
    Bd, Lk = 64, 2048
    qd = rnd(Bd, 1, NH * D)
    ck, cv = rnd(Bd, NKV, Lk + 64, D), rnd(Bd, NKV, Lk + 64, D)
    kv_bytes = 2.0 * Bd * NKV * Lk * D * 2
    t_dec = _time_cuda_graph(lambda: _ops.gqa_attention_forward(qd, ck, cv, Lk, Lk - 1, causal=True), 50, warm=5)
    out["attention_decode_11b_b64_kv2048"] = {"us": t_dec * 1e6, "GBps_kv_read": kv_bytes / t_dec / 1e9,
                                              "frac_of_measured_hbm": kv_bytes / t_dec / 1e9 / hbm, "algorithmic_bytes": kv_bytes,
                                              "what": "one decode step of attention for 64 sequences with 2048 cached tokens each "
                                                      "(K and V of the 8 KV heads read once: HBM-bound)"}
    del qd, ck, cv
    torch.cuda.empty_cache()

    # ---- one WHOLE decoder layer at the 11B geometry (norm1 -> GQA attention with RoPE + KV cache -> norm2 -> SwiGLU FFN ->
    #      residual; reference Model/model.py:257-273) from the drop-in modules, against the same layer evaluated with the
    #      reference's own expressions on the same GPU (what the reference executes when its extensions are unusable)
    class _C:
        hidden_size, n_heads, n_kv_groups, rope_base = H, NH, NKV, 500000.0

    class _Layer(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.att = L.GroupQueryAttention(_C, layer_idx=0)
            self.norm1, self.norm2 = L.LLAMARMSNorm(H, EPS), L.LLAMARMSNorm(H, EPS)
            self.ff = L.FusedFeedforward(H, I)

        def forward(self, hs, mask, pos, cache):
            a = self.att(self.norm1(hs), attention_mask=mask, position_ids=pos, kv_cache=cache)
            return L.block_tail(self.norm2, self.ff, a, hs)

        def reference(self, hs, mask, pos, cache):           # the reference's expressions, op for op
            n1 = torch_rms(hs, None, self.norm1.weight)
            a = self.att._reference_forward(n1, mask, pos, cache)
            n2 = torch_rms(a, hs, self.norm2.weight)
            F = torch.nn.functional
            return a + F.linear(F.silu(F.linear(n2, self.ff.swiglu.w_gate)) * F.linear(n2, self.ff.swiglu.w_up), self.ff.w_down.weight)

    def torch_rms(x_, r_, w_):
        h_ = x_ if r_ is None else x_ + r_
        return h_ * torch.rsqrt(h_.pow(2).mean(-1, keepdim=True) + EPS) * w_

    layer = _Layer().to(dev, dt).eval()
    Bp, Tp = 4, 2048
    hs = rnd(Bp, Tp, H)
    pos = torch.arange(Tp, device=dev)[None].expand(Bp, -1).contiguous()
    mask = torch.triu(torch.full((Tp, Tp), float("-inf"), device=dev, dtype=dt), diagonal=1)[None, None].expand(Bp, 1, Tp, Tp)

    def ours_prefill():
        with torch.no_grad():
            layer(hs, mask, pos, L.KVCache(capacity=Tp))

    def ref_prefill():
        with torch.no_grad():
            layer.reference(hs, mask, pos, None)
    t_o = _time_cuda(ours_prefill, 10, warm=3)
    t_r = _time_cuda(ref_prefill, 5, warm=2)
    res = {"prefill_4x2048_ms": t_o * 1e3, "prefill_tokens_per_s": Bp * Tp / t_o, "prefill_ms_reference_expressions": t_r * 1e3,
           "prefill_speedup": t_r / t_o}
    # decode: batch 64, 2048 cached tokens, one step replayed from a CUDA graph (preallocated cache: stable addresses)
    Bd, Lk = 64, 2048
    cache = L.KVCache(capacity=Lk + 64)
    with torch.no_grad():
        for i in range(0, Lk, 512):                          # fill the cache with 2048 positions
            chunk = rnd(Bd, 512, H)
            cpos = torch.arange(i, i + 512, device=dev)[None].expand(Bd, -1).contiguous()
            layer.att(layer.norm1(chunk), attention_mask=None, position_ids=cpos, kv_cache=cache)
    x1 = rnd(Bd, 1, H)
    p1 = torch.full((Bd, 1), Lk, device=dev, dtype=torch.long)
    zmask = torch.zeros(Bd, 1, 1, 1, device=dev, dtype=dt)

    def dec_step():
        with torch.no_grad():
            cache._len[0] = Lk
            cache.advance(0, 0)
            return layer(x1, zmask, p1, cache)
    for _ in range(3):
        dec_step()
    torch.cuda.synchronize()
    t_eager = _time_cuda(dec_step, 30, warm=3)
    gph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gph):
        dec_step()
    t_graph = _time_cuda(gph.replay, 50, warm=5)
    res.update({"decode_b64_kv2048_us_graph": t_graph * 1e6, "decode_b64_kv2048_us_eager_launch": t_eager * 1e6,
                "decode_tokens_per_s_graph": Bd / t_graph,
                "what": "one decoder layer (32/8 heads x 128, hidden 4096, FFN 14336), bf16: drop-in modules (tcgen05 GEMMs, flash-style "
                        "attention, preallocated KV cache, fused block tail) vs the same layer through the reference's own expressions "
                        "(materialised scores, repeat_kv, eager norm / SwiGLU) on the same GPU; decode = 64 sequences x 2048 cached "
                        "tokens, the step replayed from a CUDA graph and launched eagerly from Python"})
    out["decoder_layer_11b"] = res
    del layer, hs, mask, cache
    torch.cuda.empty_cache()
    return out


def config5_90b(dev, rank, world, peaks, steps, train_too=True):
    """BASELINE.json configs[4]: the 90B text block (hidden 8192, hidden_dim 28672), 4 x 2048 tokens IN TOTAL (strong
    scaling), tensor-parallel over the `world` GPUs of this run with the collectives fused into the GEMMs.  Also measures the
    same step on ONE GPU in this run (every rank runs the unsharded block at the same time) so the efficiency is
    self-contained, and checks 64 rows per rank against the CPU oracle before timing.  Collective: every rank calls it."""
    import torch.distributed as dist
    from llama32_b200 import ops
    from llama32_b200.tp import FusedTensorParallelBlock, TpRankBuffers
    H, I, T = 8192, 28672, 8192
    dt = torch.bfloat16
    gamma, wg, wu, wd = _gpu_weights(H, I, dev, 5)
    gen = torch.Generator(device=dev).manual_seed(50)               # same activations on every rank (each uses its rows)
    xs = [torch.randn(T, H, device=dev, generator=gen).to(dt) for _ in range(2)]
    rs = [torch.randn(T, H, device=dev, generator=gen).to(dt) for _ in range(2)]
    res = {"shape": {"hidden": H, "hidden_dim": I, "tokens_total": T, "tp": world}}
    fl = 6.0 * T * H * I

    # one GPU, unsharded (what N = 1 runs): forward, and forward + backward
    cnt = {"i": 0}

    def single():
        cnt["i"] += 1
        i = cnt["i"] % 2
        ops.ffn_forward(ops.add_rmsnorm_forward(xs[i], gamma, rs[i], EPS, want_rms=False)[0], wg, wu, wd)
    t1 = _time_cuda(single, max(5, steps // 2), warm=3)
    t1_all = _gather_floats(t1, dev, world)
    t1_med = statistics.median(t1_all)
    res["single_gpu"] = {"ms_per_step": t1_med * 1e3, "tokens_per_s": T / t1_med, "TFLOPs": fl / t1_med / 1e12,
                         "frac_of_bf16_burst_peak": fl / t1_med / 1e12 / peaks["bf16_tflops"],
                         "ms_per_step_every_rank": [v * 1e3 for v in t1_all],
                         "what": "the unsharded 90B block on one GPU, measured on every GPU of this run at the same time; median"}
    t1_train = None
    if train_too:
        import llama32_b200 as L
        norm = L.LLAMARMSNorm(H, eps=EPS).to(dev, dt)
        ffn = L.FusedFeedforward(H, I).to(dev, dt)
        with torch.no_grad():
            norm.weight.copy_(gamma)
        ffn.swiglu.w_gate.data, ffn.swiglu.w_up.data, ffn.w_down.weight.data = wg, wu, wd   # no second copy of 1.4 GB
        dy1 = torch.randn(T, H, device=dev, generator=gen).to(dt)

        def single_train():
            xx = xs[0].detach().requires_grad_(True)
            ffn(norm(xx, residual=rs[0])).backward(dy1)
        t1_train = statistics.median(_gather_floats(_time_cuda(single_train, max(3, steps // 4), warm=2), dev, world))
        res["single_gpu_train"] = {"ms_per_step": t1_train * 1e3, "tokens_per_s": T / t1_train, "TFLOPs": 3 * fl / t1_train / 1e12}
        del norm, ffn, dy1
    if world == 1:
        res.update({"tokens_per_s": T / t1_med, "ms_per_step": t1_med * 1e3, "efficiency_vs_1gpu_90b": 1.0,
                    "tp_parity_rel_l2": None})
        sub = torch.arange(0, T, T // 64, device=dev)
        y = ops.ffn_forward(ops.add_rmsnorm_forward(xs[0], gamma, rs[0], EPS, want_rms=False)[0], wg, wu, wd)[0]
        res["parity_rel_l2"] = oracle_rows_rel_l2(y[sub], xs[0][sub], rs[0][sub], gamma, wg, wu, wd)
        if train_too:
            res["train"] = {"tokens_per_s": T / t1_train, "ms_per_step": t1_train * 1e3, "efficiency_vs_1gpu_90b": 1.0}
        return res

    bufs = TpRankBuffers.symmetric(T, H, dt, dev)
    blk = FusedTensorParallelBlock(gamma, EPS, wg, wu, wd, bufs)
    lo, hi, _ = blk.rows_of(T)
    # parity first: 64 of this rank's rows against the CPU oracle (needs the full weights, so before they are dropped)
    y = blk.forward(xs[0][lo:hi], rs[0][lo:hi], T)
    sub = torch.arange(0, hi - lo, max(1, (hi - lo) // 64), device=dev)[:64]
    err = oracle_rows_rel_l2(y[sub], xs[0][lo:hi][sub], rs[0][lo:hi][sub], gamma, wg, wu, wd)
    errs = _gather_floats(err, dev, world)
    res["tp_parity_rel_l2"] = max(errs)
    res["tp_parity_rel_l2_every_rank"] = errs
    del wg, wu, wd
    torch.cuda.empty_cache()
    xl = [v[lo:hi].contiguous() for v in xs]
    rl = [v[lo:hi].contiguous() for v in rs]
    del xs, rs
    t = _timed_steps(lambda i: blk.forward(xl[i % 2], rl[i % 2], T), steps, 5, dev, world)
    res.update({"tokens_per_s": T / t, "ms_per_step": t * 1e3, "TFLOPs_per_gpu": fl / t / 1e12 / world,
                "efficiency_vs_1gpu_90b": (T / t) / (world * T / t1_med)})
    if train_too:
        for w in (blk.gamma, blk.w_gate, blk.w_up, blk.w_down):
            w.requires_grad_(True)
        dyl = torch.randn(hi - lo, H, device=dev, generator=gen).to(dt)

        def tp_train(i):
            xx = xl[i % 2].detach().requires_grad_(True)
            blk.apply(xx, rl[i % 2], T).backward(dyl)
            for w in (blk.gamma, blk.w_gate, blk.w_up, blk.w_down):
                w.grad = None
        tt = _timed_steps(tp_train, max(3, steps // 2), 3, dev, world)
        res["train"] = {"tokens_per_s": T / tt, "ms_per_step": tt * 1e3, "TFLOPs_per_gpu": 3 * fl / tt / 1e12 / world,
                        "efficiency_vs_1gpu_90b": (T / tt) / (world * T / t1_train)}
    del blk, bufs
    torch.cuda.empty_cache()
    return res


def host_copy_ceiling(dev, world, h_x, h_r, h_y, d_x, d_r, d_y, steps):
    """The e2e step's copies alone (H2D of x and residual, D2H of y; every rank at once, no compute): the floor PCIe and the
    host's memory system put under `e2e.ms_per_step` on this box."""
    s_h2d, s_d2h = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    cur = torch.cuda.current_stream(dev)

    def copies(i):
        b = i % len(h_x)
        if i == 0:                                    # the side streams start behind the start event
            s_h2d.wait_stream(cur)
            s_d2h.wait_stream(cur)
        with torch.cuda.stream(s_h2d):
            d_x[b].copy_(h_x[b], non_blocking=True)
            d_r[b].copy_(h_r[b], non_blocking=True)
        with torch.cuda.stream(s_d2h):
            h_y[b].copy_(d_y, non_blocking=True)
        if i == steps - 1:                            # ... and the end event behind the last copies
            cur.wait_stream(s_h2d)
            cur.wait_stream(s_d2h)
    return _timed_steps(copies, steps, 0, dev, world)


# ------------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import torch.distributed as dist
    import llama32_b200 as L
    from llama32_b200 import _lib, ops
    from llama32_b200.tp import FusedTensorParallelBlock, TensorParallelFFN, TpRankBuffers

    hidden, inter, batch, seq, label = WORKLOADS[args.workload]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    weak = world > 1 and args.scaling == "weak"
    if weak:
        batch *= world                                 # 4 x 2048 tokens PER GPU
    tokens = batch * seq
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    dt = torch.bfloat16
    train = args.mode == "train"
    if train and world > 1 and args.tp_impl != "fused":
        raise SystemExit("--mode train at N > 1 needs --tp-impl fused (the NCCL baseline path is forward only)")

    # synthetic inputs and random-init weights exactly as the modules initialise them (SURVEY.md 8d); same seed
    # on every rank so the replicated tensors agree
    torch.manual_seed(0)
    norm = L.LLAMARMSNorm(hidden, eps=EPS)
    ffn = L.FusedFeedforward(hidden, inter)           # kaiming_uniform(a=sqrt 5) == U(+-1/sqrt(fan_in))
    with torch.no_grad():
        norm.weight.copy_(1 + 0.1 * torch.randn(hidden))
    norm = norm.to(dev, dt)
    ffn = ffn.to(dev, dt)
    nbuf = 2                                           # rotate input buffers; footprint per step >> 126 MB L2
    gen = torch.Generator(device=dev).manual_seed(1)
    tp = fused = None
    xs = rs = dys = None
    tp_parity = None
    if world > 1 and args.tp_impl == "fused":
        bufs = TpRankBuffers.symmetric(tokens, hidden, dt, dev)
        fused = FusedTensorParallelBlock(norm.weight.detach(), EPS, ffn.swiglu.w_gate.detach(), ffn.swiglu.w_up.detach(),
                                         ffn.w_down.weight.detach(), bufs, one_kernel=args.tp_one_kernel)
        lo, hi, _ = fused.rows_of(tokens)
        gen = torch.Generator(device=dev).manual_seed(1 + rank)
        # sequence-parallel: every rank holds (and generates) only its own rows
        xs_loc = [torch.randn(hi - lo, hidden, device=dev, generator=gen).to(dt) for _ in range(nbuf)]
        rs_loc = [torch.randn(hi - lo, hidden, device=dev, generator=gen).to(dt) for _ in range(nbuf)]
        dys_loc = [torch.randn(hi - lo, hidden, device=dev, generator=gen).to(dt) for _ in range(nbuf)] if train else None
        # ---- parity BEFORE anything is timed: 64 of this rank's output rows against the CPU oracle (checker only)
        with torch.no_grad():
            y = fused.forward(xs_loc[0], rs_loc[0], tokens)
        sub = torch.arange(0, hi - lo, max(1, (hi - lo) // 64), device=dev)[:64]
        err = oracle_rows_rel_l2(y[sub], xs_loc[0][sub], rs_loc[0][sub], norm.weight, ffn.swiglu.w_gate, ffn.swiglu.w_up,
                                 ffn.w_down.weight)
        errs = _gather_floats(err, dev, world)
        tp_parity = {"tp_parity_rel_l2": max(errs), "every_rank": errs, "rows_per_rank": int(sub.numel()), "tolerance": PARITY_TOL}
        if max(errs) > PARITY_TOL:
            if rank == 0:
                print(json.dumps({"error": "tensor-parallel output differs from the oracle", **tp_parity}), flush=True)
            dist.destroy_process_group()
            sys.exit(3)
        del y
        if train:
            for w in (fused.gamma, fused.w_gate, fused.w_up, fused.w_down):
                w.requires_grad_(True)
    else:
        xs = [torch.randn(batch, seq, hidden, device=dev, generator=gen).to(dt) for _ in range(nbuf)]
        rs = [torch.randn(batch, seq, hidden, device=dev, generator=gen).to(dt) for _ in range(nbuf)]
        dys = [torch.randn(batch, seq, hidden, device=dev, generator=gen).to(dt) for _ in range(nbuf)] if train else None
        if world > 1:
            tp = TensorParallelFFN(ffn, chunks=args.tp_chunks)
    if world > 1:
        ffn = None                                     # the unsharded copy is not needed any more
        torch.cuda.empty_cache()
    if train and world == 1:
        for p in list(norm.parameters()) + list(ffn.parameters()):
            p.requires_grad_(True)

    k_ev = []                                          # (start, end) events around the dominant kernel

    def step(i, instrument=False):
        if fused is None:
            x, r = xs[i % nbuf], rs[i % nbuf]
        if train:
            if fused is not None:
                xx = xs_loc[i % nbuf].detach().requires_grad_(True)
                y = fused.apply(xx, rs_loc[i % nbuf], tokens)
                y.backward(dys_loc[i % nbuf])
                for w in (fused.gamma, fused.w_gate, fused.w_up, fused.w_down):
                    w.grad = None
                return y, xx.grad
            x = x.detach().requires_grad_(True)
            normed = norm(x, residual=r)
            y = ffn(normed)
            y.backward(dys[i % nbuf])
            return y, x.grad
        with torch.no_grad():
            if fused is not None:
                if instrument:
                    fused.phase_norm(xs_loc[i % nbuf], rs_loc[i % nbuf], tokens)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    if fused.one_kernel:
                        fused.phase_ffn(tokens)
                        fused.phase_reduce(tokens)
                        return None
                    fused.phase_gate_up(tokens)
                    e1.record()
                    k_ev.append((e0, e1))
                    fused.phase_down(tokens)
                    return fused.phase_reduce(tokens)
                return fused.forward(xs_loc[i % nbuf], rs_loc[i % nbuf], tokens)
            normed = norm(x, residual=r)
            if tp is not None:
                return tp(normed)
            if instrument:
                # same three launches as ffn(normed), with events around the fused gate/up GEMM
                n2 = normed.view(-1, hidden)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                act, _, _ = ops.swiglu_forward(n2, ffn.swiglu.w_gate, ffn.swiglu.w_up)
                e1.record()
                k_ev.append((e0, e1))
                return ops.linear_forward(act, ffn.w_down.weight).view(batch, seq, hidden)
            return ffn(normed)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(3, args.warmup)
    for i in range(warm):
        last = step(i)      # held like the timed loop holds it, so the allocator reaches the same steady state
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    # ---- timed region 1: device-resident inputs
    launches0 = _lib.lib().l32_kernel_launch_count()
    barrier()
    t_wall0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        if train and fused is None and i == args.steps - 1:   # the last step's gradients alone, not a sum over all steps
            norm.zero_grad(set_to_none=True)
            ffn.zero_grad(set_to_none=True)
        last = step(i, instrument=((world == 1 or fused is not None) and not train))
    e1.record()
    barrier()
    t_wall1 = time.time()
    launches = _lib.lib().l32_kernel_launch_count() - launches0
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    if args.dump_outputs:
        if train:
            outs = {"y": last[0], "dx": last[1], "grad_gamma": norm.weight.grad, "grad_w_gate": ffn.swiglu.w_gate.grad,
                    "grad_w_up": ffn.swiglu.w_up.grad, "grad_w_down": ffn.w_down.weight.grad}
        else:
            outs = {"y": last}
        dump_outputs(args.dump_outputs, outs)
    del last
    ms_total = _max_over_ranks(ms_total, dev, world)
    ms_step = ms_total / args.steps
    value = tokens / (ms_step * 1e-3)

    # ---- timed region 2: end to end through the module API with pinned host buffers
    if fused is not None:
        lo, hi, _ = fused.rows_of(tokens)
        io_shape = (hi - lo, hidden)                   # every rank moves only its own rows over PCIe
    else:
        io_shape = (batch, seq, hidden)
    e2e = None
    if not train:
        h_x = [torch.randn(*io_shape).to(dt).pin_memory() for _ in range(nbuf)]
        h_r = [torch.randn(*io_shape).to(dt).pin_memory() for _ in range(nbuf)]
        h_y = [torch.empty(*io_shape, dtype=dt).pin_memory() for _ in range(nbuf)]
        d_x = [torch.empty(*io_shape, device=dev, dtype=dt) for _ in range(nbuf)]
        d_r = [torch.empty(*io_shape, device=dev, dtype=dt) for _ in range(nbuf)]
        s_h2d, s_d2h, s_cmp = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.current_stream(dev)
        ev_in = [torch.cuda.Event() for _ in range(nbuf)]
        ev_cmp = [torch.cuda.Event() for _ in range(nbuf)]
        ev_out = [torch.cuda.Event() for _ in range(nbuf)]

        y_keep = [None] * nbuf                             # the step's result stays referenced until its D2H copy has been
                                                           # ordered before later compute (no record_stream: the caching
                                                           # allocator then only ever reuses blocks on the compute stream)

        def e2e_steps(n):
            for i in range(n):
                b = i % nbuf
                with torch.cuda.stream(s_h2d):
                    s_h2d.wait_event(ev_cmp[b])            # the compute that last read d_x[b] / d_r[b] is done
                    d_x[b].copy_(h_x[b], non_blocking=True)
                    d_r[b].copy_(h_r[b], non_blocking=True)
                    ev_in[b].record(s_h2d)
                s_cmp.wait_event(ev_in[b])
                s_cmp.wait_event(ev_out[b])                # the D2H copy of the result held in this slot (nbuf steps ago) is
                y_keep[b] = None                           # done: its memory may be reused by the compute below
                with torch.no_grad():
                    if fused is not None:
                        y = fused.forward(d_x[b], d_r[b], tokens)
                    else:
                        normed = norm(d_x[b], residual=d_r[b])
                        y = tp(normed) if tp is not None else ffn(normed)
                ev_cmp[b].record(s_cmp)
                y_keep[b] = y
                with torch.cuda.stream(s_d2h):
                    s_d2h.wait_event(ev_cmp[b])
                    h_y[b].copy_(y, non_blocking=True)
                    ev_out[b].record(s_d2h)

        e2e_steps(max(warm, 8))
        barrier()
        e0.record()
        e2e_steps(args.steps)
        s_cmp.wait_stream(s_d2h)
        s_cmp.wait_stream(s_h2d)
        e1.record()
        barrier()
        ms_e2e = _max_over_ranks(e0.elapsed_time(e1), dev, world)
        per_tensor = h_x[0].numel() * 2
        # the copies alone, every rank at once: what the host side of this box allows
        d_y = torch.empty(*io_shape, device=dev, dtype=dt)
        t_copy = host_copy_ceiling(dev, world, h_x, h_r, h_y, d_x, d_r, d_y, max(5, args.steps))
        api = ("llama32_b200.LLAMARMSNorm + FusedFeedforward modules" if world == 1 else
               ("llama32_b200.tp.FusedTensorParallelBlock.forward (bytes are per rank: each rank moves its own rows)"
                if fused is not None else "llama32_b200.LLAMARMSNorm + tp.TensorParallelFFN"))
        e2e = {"value": tokens / (ms_e2e / args.steps * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
               "h2d_bytes_per_step": 2 * per_tensor, "d2h_bytes_per_step": per_tensor,
               "copies_only_ms_per_step": t_copy * 1e3,
               "copies_only_GBps_all_ranks": 3 * per_tensor * world / t_copy / 1e9,
               "copies_note": "copies_only = the same H2D + D2H traffic with no compute, every rank at once: the floor set by "
                              "PCIe and the host's memory system (all ranks share one host; the container's CPU set and the "
                              "pinned buffers sit on one NUMA node)",
               "api": api + "; pinned host buffers, copies on side streams double-buffered against compute"}
        y_keep = None
        del h_x, h_r, h_y, d_x, d_r, d_y

    # ---- BASELINE.json configs[4] in every line: 90B, 4 x 2048 tokens in total, tensor-parallel over this run's GPUs
    cfg5 = None
    if not args.no_extra and not train:
        xs = rs = xs_loc = rs_loc = None               # the main workload's activations are not needed any more
        torch.cuda.empty_cache()
        cfg5 = config5_90b(dev, rank, world, load_peaks(), steps=max(10, min(args.steps, 40)))
        if cfg5.get("tp_parity_rel_l2") is not None and cfg5["tp_parity_rel_l2"] > PARITY_TOL:
            if rank == 0:
                print(json.dumps({"error": "config 5 tensor-parallel output differs from the oracle", **cfg5}), flush=True)
            dist.destroy_process_group()
            sys.exit(3)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    flops_step = 6.0 * tokens * hidden * inter * (3.0 if train else 1.0)
    roofline = None
    if k_ev:
        torch.cuda.synchronize()
        k_ms = statistics.mean(a.elapsed_time(b) for a, b in k_ev)
        alg_flops = 4.0 * tokens * hidden * inter / world  # gate + up GEMMs: 4*H*I flop per token (SURVEY.md 8d), per rank
        achieved = alg_flops / (k_ms * 1e-3) / 1e12
        kname = "gemm_kernel<cta_group 2, EPI_SWIGLU, bf16> (fused gate/up + SiLU*mul)"
        if world > 1:
            kname += f", all-gather of {(world - 1) * tokens // world} rows pulled over NVLink inside the kernel (rank 0's timing)"
        roofline = {"bound": "tensor", "kernel": kname,
                    "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                    "frac": achieved / peaks["bf16_tflops"], "peak_source": peaks["source"] + ", burst figure",
                    "kernel_ms": k_ms, "kernel_share_of_step": k_ms / ms_step,
                    "frac_of_sustained_peak": (achieved / peaks["bf16_tflops_sustained"]) if peaks["bf16_tflops_sustained"] else None,
                    "traffic": None, "traffic_note": "see profiles/ for dram__bytes of this kernel from ncu --set full"}
        if world == 1 and args.workload == "11b":
            try:   # DRAM bytes of this kernel at this shape from the committed ncu --set full capture (per launch)
                with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                    tr = json.load(f)["gemm_swiglu_11b_8192tok"]
                roofline["traffic"] = tr["dram_bytes_read"] + tr["dram_bytes_write"]
                roofline["traffic_note"] = (f"dram__bytes_read.sum + dram__bytes_write.sum of one launch, {tr['source']}; "
                                            f"algorithmic bytes {tr['algorithmic_bytes']} (x, both weight matrices, act)")
            except (OSError, KeyError, ValueError):
                pass
    step_tflops = flops_step / (ms_step * 1e-3) / 1e12

    extra = {}
    if world == 1 and not train and not args.no_extra:
        torch.cuda.empty_cache()
        extra.update(extra_numbers(dev, peaks))
    if cfg5 is not None:
        extra["config5_90b_strong"] = cfg5
    if tp_parity is not None:
        extra["tp_parity"] = tp_parity

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        tps, ms, cores, done = cpu_reference(hidden, inter, batch * seq, steps=3, warmup=1, min_seconds=10.0, max_seconds=30.0)
        cpu = {"value": tps, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{done} full steps x {batch * seq} tokens (the whole config-2 batch), fp32 torch CPU path of the reference "
                         f"(oracle port), {ms:.1f} ms/step"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak" if (weak or world == 1) else "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config_for(args, world),
        "step_tflops": step_tflops, "step_frac_of_bf16_peak": step_tflops / world / peaks["bf16_tflops"],
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
    }
    if tp_parity is not None:
        line["tp_parity_rel_l2"] = tp_parity["tp_parity_rel_l2"]
    if extra:
        line["extra"] = extra
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 400; 20 for --impl reference, whose steps take seconds each on the CPU)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="11b")
    ap.add_argument("--mode", choices=["prefill", "train"], default="prefill")
    ap.add_argument("--tp-chunks", type=int, default=4)
    ap.add_argument("--tp-impl", choices=["fused", "nccl"], default="fused")
    ap.add_argument("--tp-one-kernel", action="store_true",
                    help="N > 1, fused: gate/up and down as ONE persistent kernel (l32_tp_ffn_forward_fused)")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak",
                    help="N > 1: weak = 4x2048 tokens per GPU (global batch grows with N), strong = 4x2048 tokens in total")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the secondary measurements (RMSNorm GB/s, decode, sustained, baselines, train, config 5)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="one GPU: after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32; "
                         "at most 64 MB in all, larger outputs as the same seeded sample of rows in every run)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.impl == "reference" else 400
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.gpus != 1):
        ap.error("--dump-outputs is implemented for the GPU arm on one GPU")
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (the CUDA path has no CPU fallback); "
                             "use --impl reference for the CPU reference arm")
        run_ours(args)


if __name__ == "__main__":
    main()
