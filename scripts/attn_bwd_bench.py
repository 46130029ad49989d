"""Attention backward for training calls: timing, rates and memory.  python scripts/attn_bwd_bench.py [--parent-root DIR]

1. Backward (delta + dK/dV + dQ kernels, one l32_gqa_attention_backward call) at 4 x 2048 and 1 x 8192 tokens, causal,
   32 / 8 heads, head_dim 128 and 64.  Rates over the seven GEMMs the kernels run (3.5 x the causal forward's
   4 B H T^2 d / 2) and in the FA2 convention (2.5 x).  Next to it, on the same GPU: torch SDPA backward (enable_gqa) and the
   reference's expressions (repeat_kv + materialised softmax) under autograd.  Every working set here is larger than the
   126 MB L2 (q, dO, ctx alone are 3 x 64 MB at 4 x 2048), so nothing is served from a warm cache.
2. The inference forward (lse == nullptr) of this tree against a built checkout of another commit (--parent-root: its package
   and, through L32_LIB_PATH, its libl32ffn.so, in a subprocess), alternated so that drift on the shared machine shows up as
   spread.
3. One decoder layer LoRA training step at the 11B geometry (4 x 2048 tokens, r = 16 on q/k/v/o and w_down, gate/up
   trainable): time and peak memory, GQAAttentionFunction against the same layer with the reference's attention expressions.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.environ.get("ATTN_BENCH_ROOT") or os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

dev, dt = "cuda", torch.bfloat16


def timeit(fn, iters=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return f"{name}, power limit / max SM clock: {pl}"


def forward_only(iters):
    """Child process: time the inference forward of whichever library L32_LIB_PATH names (or the in-tree one)."""
    from llama32_b200 import ops
    g = torch.Generator(device=dev).manual_seed(0)
    out = {}
    for B, T, NH, NKV, D in ((4, 2048, 32, 8, 128), (4, 2048, 32, 8, 64)):
        q = torch.randn(B, T, NH * D, device=dev, generator=g).to(dt)
        ck = torch.randn(B, NKV, T, D, device=dev, generator=g).to(dt)
        cv = torch.randn(B, NKV, T, D, device=dev, generator=g).to(dt)
        out[f"{B}x{T} d{D}"] = timeit(lambda: ops.gqa_attention_forward(q, ck, cv, T, 0, causal=True), iters=iters, warm=5)
    print(json.dumps(out))


def backward_section():
    from llama32_b200 import ops
    g = torch.Generator(device=dev).manual_seed(1)
    rnd = lambda *s: torch.randn(*s, device=dev, generator=g).to(dt)
    for B, T, D in ((4, 2048, 128), (1, 8192, 128), (4, 2048, 64), (1, 8192, 64)):
        NH, NKV = 32, 8
        q, k, v, gy = rnd(B, T, NH * D), rnd(B, T, NKV * D), rnd(B, T, NKV * D), rnd(B, T, NH * D)
        pos = torch.arange(T, device=dev)[None].expand(B, -1).contiguous()
        qr = q.clone()
        ck, cv = torch.empty(B, NKV, T, D, device=dev, dtype=dt), torch.empty(B, NKV, T, D, device=dev, dtype=dt)
        ops.rope_kv_append(qr, k, v, pos, ck, cv, 0)
        ctx, lse = ops.gqa_attention_forward_train(qr, ck, cv, True, None)
        ms_fwd = timeit(lambda: ops.gqa_attention_forward_train(qr, ck, cv, True, None))
        ms = timeit(lambda: ops.gqa_attention_backward(gy, qr, ck, cv, ctx, lse, pos, True, None))
        f_fwd = 4.0 * B * NH * T * T * D / 2
        # torch SDPA backward (flash / cuDNN, whichever torch picks) on the same rotated tensors
        q4 = qr.view(B, T, NH, D).transpose(1, 2).detach().requires_grad_(True)
        k4, v4 = ck.detach().requires_grad_(True), cv.detach().requires_grad_(True)
        o4 = torch.nn.functional.scaled_dot_product_attention(q4, k4, v4, is_causal=True, enable_gqa=True)
        g4 = gy.view(B, T, NH, D).transpose(1, 2)
        ms_sdpa = timeit(lambda: torch.autograd.grad(o4, (q4, k4, v4), g4, retain_graph=True))
        # the reference's expressions (Model/model.py:244-252) under autograd: repeat_kv, scores + mask, softmax, P V
        mask = torch.triu(torch.full((T, T), float("-inf"), device=dev, dtype=dt), 1)
        kr, vr = k4.repeat_interleave(NH // NKV, 1), v4.repeat_interleave(NH // NKV, 1)
        o_ref = torch.softmax((q4 @ kr.transpose(2, 3) + mask) / D ** 0.5, dim=-1) @ vr
        ms_ref = timeit(lambda: torch.autograd.grad(o_ref, (q4, k4, v4), g4, retain_graph=True), iters=5, warm=1)
        print(f"backward B={B} T={T} heads {NH}/{NKV} d={D}: {ms:.3f} ms  {3.5 * f_fwd / ms / 1e9:.0f} TFLOP/s over the 7 GEMMs run, "
              f"{2.5 * f_fwd / ms / 1e9:.0f} TFLOP/s FA2 convention | torch SDPA bwd {ms_sdpa:.3f} ms | reference exprs bwd "
              f"{ms_ref:.3f} ms | forward_train {ms_fwd:.3f} ms", flush=True)
        del o4, o_ref, kr, vr, mask
        torch.cuda.empty_cache()


def forward_ab(parent_root):
    cmd = [sys.executable, os.path.abspath(__file__), "--forward-only"]
    runs = {"this": [], "parent": []}
    for rep in range(4):
        for tag in ("parent", "this") if rep % 2 else ("this", "parent"):
            env = dict(os.environ)
            env.pop("L32_LIB_PATH", None)
            env.pop("ATTN_BENCH_ROOT", None)
            if tag == "parent":
                env["ATTN_BENCH_ROOT"] = os.path.abspath(parent_root)
                env["L32_LIB_PATH"] = os.path.join(os.path.abspath(parent_root), "llama-3.2-multimodal_b200", "libl32ffn.so")
            r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
            if r.returncode != 0:
                raise RuntimeError(r.stderr[-2000:])
            runs[tag].append(json.loads(r.stdout.strip().splitlines()[-1]))
    for key in runs["this"][0]:
        a = [x[key] for x in runs["this"]]
        b = [x[key] for x in runs["parent"]]
        print(f"inference forward {key}: this build {min(a):.4f}..{max(a):.4f} ms, parent build {min(b):.4f}..{max(b):.4f} ms",
              flush=True)


def layer_section():
    import llama32_b200 as L

    class Cfg:
        hidden_size, n_heads, n_kv_groups, rope_base = 4096, 32, 8, 500000.0

    B, T, H, I, r = 4, 2048, 4096, 14336, 16
    torch.manual_seed(0)
    norm1, norm2 = L.LLAMARMSNorm(H, 1e-5), L.LLAMARMSNorm(H, 1e-5)
    att = L.GroupQueryAttention(Cfg())
    for name in ("W_query", "W_key", "W_value", "out_proj"):
        old = getattr(att, name)
        setattr(att, name, L.Linear_LORA(old.in_features, old.out_features, r, 2 * r, 0.0))
    ff = L.FusedFeedforward(H, I)
    ff.w_down = L.Linear_LORA(I, H, r, 2 * r, 0.0)
    mods = torch.nn.ModuleList([norm1, norm2, att, ff]).to(dev, dt)
    for p in norm1.parameters():
        p.requires_grad_(False)
    for p in norm2.parameters():
        p.requires_grad_(False)
    x = (torch.randn(B, T, H, device=dev) * 0.5).to(dt)
    gy = torch.randn(B, T, H, device=dev).to(dt)
    mask = torch.triu(torch.full((T, T), float("-inf"), device=dev, dtype=dt), 1)[None, None].expand(B, 1, T, T)
    pos = torch.arange(T, device=dev)[None].expand(B, -1).contiguous()

    def step(reference):
        for p in mods.parameters():
            p.grad = None
        xi = x.detach().requires_grad_(True)
        h = norm1(xi)
        a = att._reference_forward(h, mask, pos, None) if reference else att(h, attention_mask=mask, position_ids=pos)
        y = L.block_tail(norm2, ff, a, xi)
        y.backward(gy)

    for reference in (False, True):
        step(reference)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        ms = timeit(lambda: step(reference), iters=10, warm=2)
        peak = (torch.cuda.max_memory_allocated() - base) / 2 ** 30
        print(f"decoder layer LoRA training step 4x2048 (11B geometry), attention = "
              f"{'reference expressions' if reference else 'GQAAttentionFunction'}: {ms:.2f} ms, peak {peak:.2f} GiB above weights "
              f"and inputs", flush=True)
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--forward-only", action="store_true")
    ap.add_argument("--parent-root", default=None, help="a built checkout of another commit for the forward A/B")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    if args.forward_only:
        forward_only(iters=50)
        return
    print(gpu_info(), flush=True)
    backward_section()
    if args.parent_root:
        forward_ab(args.parent_root)
    layer_section()
    print(gpu_info(), flush=True)


if __name__ == "__main__":
    main()
