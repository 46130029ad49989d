"""Whole decoder layer under tensor parallelism: attention sharded by KV group (FusedTensorParallelAttention) + the fused
tensor-parallel feed-forward, on one buffer set.  One JSON line per configuration.

Multi-GPU:  python -m torch.distributed.run --nproc-per-node P scripts/tp_layer_bench.py
  11B (32 / 8 heads, hidden 4096, inter 14336) and 90B (64 / 8, 8192, 28672) geometry at this P:
    * prefill forward and training forward + backward at 4 x 2048 tokens, decode at b = 64 with 2048 cached tokens;
    * the same layer with attention REPLICATED (the single-GPU GroupQueryAttention on every rank) and only the
      feed-forward tensor-parallel, at the same P;
    * the one-GPU layer (GroupQueryAttention + block_tail) on rank 0, and the strong-scaling efficiency against it;
    * per-rank parity of the TP output against the one-GPU layer on the same weights (rel-L2, bf16 vs bf16).
  Times: CUDA events around `--iters` steps after `--warmup`, the maximum over ranks.
Single GPU: python scripts/tp_layer_bench.py
  per-rank phase times at the P = 8 shard shapes, from the single-GPU emulation (all ranks' buffers on one device, the
  ranks' phases one after another).  The pulls and pushes are then local copies, not NVLink: these are per-rank kernel
  times at the shard shapes, not a scaling figure.  The one-GPU layer is timed as well.
Decode under tensor parallelism launches eagerly (the epochs are host values, so a step cannot be graph-captured).
Every line carries the GPU name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import llama32_b200 as L  # noqa: E402
from llama32_b200.modules import KVCache, block_tail  # noqa: E402
from llama32_b200.tp import (FusedTensorParallelAttention, FusedTensorParallelBlock, TensorParallelDecoderLayer,  # noqa: E402
                             TpRankBuffers, rows_of)

GEOMETRY = {"11B": dict(n_heads=32, n_kv=8, hidden=4096, inter=14336), "90B": dict(n_heads=64, n_kv=8, hidden=8192, inter=28672)}
EPS = 1e-5


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return dict(gpu=name, power_limit=power)


class Cfg:
    def __init__(self, g):
        self.hidden_size, self.n_heads, self.n_kv_groups, self.rope_base = g["hidden"], g["n_heads"], g["n_kv"], 500000.0


def one_gpu_layer(g, dev, seed=0):
    """The single-GPU layer modules (norm1, GroupQueryAttention, norm2, FusedFeedforward) with seeded bf16 weights."""
    torch.manual_seed(seed)
    m = torch.nn.ModuleDict(dict(norm1=L.LLAMARMSNorm(g["hidden"], eps=EPS), att=L.GroupQueryAttention(Cfg(g), layer_idx=0),
                                 norm2=L.LLAMARMSNorm(g["hidden"], eps=EPS), ff=L.FusedFeedforward(g["hidden"], g["inter"])))
    with torch.no_grad():
        for p in m.parameters():
            if p.dim() == 2:
                p.uniform_(-1, 1).mul_(p.shape[1] ** -0.5)
            else:
                p.normal_(1.0, 0.1)
    return m.to(dev, torch.bfloat16)


def one_gpu_forward(m, x, pos, mask, cache=None):
    a = m.att(m.norm1(x), attention_mask=mask, position_ids=pos, kv_cache=cache)
    return block_tail(m.norm2, m.ff, a, x)


def tp_layer(m, g, bufs):
    a, f = m.att, m.ff
    attn = FusedTensorParallelAttention(m.norm1.weight.detach(), EPS, a.W_query.weight.detach(), a.W_key.weight.detach(),
                                        a.W_value.weight.detach(), a.out_proj.weight.detach(), g["n_heads"], g["n_kv"], bufs)
    ffn = FusedTensorParallelBlock(m.norm2.weight.detach(), EPS, f.swiglu.w_gate.detach(), f.swiglu.w_up.detach(),
                                   f.w_down.weight.detach(), bufs)
    return TensorParallelDecoderLayer(attn, ffn)


def causal_mask(b, t, dev):
    m = torch.triu(torch.full((t, t), float("-inf"), device=dev), diagonal=1)
    return m[None, None].expand(b, 1, t, t).to(torch.bfloat16)


def time_ms(fn, warmup, iters, group=None):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if group is not None:
        dist.barrier(group)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / iters], device="cuda")
    if group is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX, group=group)
    return float(ms)


def rel_l2(a, b):
    a, b = a.float(), b.float()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def multi_gpu(args):
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    info = gpu_info()
    b, t = 4, 2048
    for name in args.configs:
        g = GEOMETRY[name]
        m = one_gpu_layer(g, dev)
        tokens = b * t
        x = torch.randn(b, t, g["hidden"], device=dev, generator=torch.Generator(device=dev).manual_seed(1)).bfloat16()
        pos, mask = torch.arange(t, device=dev)[None].expand(b, t), causal_mask(b, t, dev)
        lo, hi, _ = rows_of(tokens, world, rank)
        x2 = x.reshape(tokens, -1)
        res = dict(config=name, world=world, tokens=tokens, **info)
        with torch.no_grad():
            ref = one_gpu_forward(m, x, pos, mask).reshape(tokens, -1)
            res["one_gpu_prefill_ms"] = time_ms(lambda: one_gpu_forward(m, x, pos, mask), args.warmup, args.iters)
        bufs = TpRankBuffers.symmetric(tokens, g["hidden"], torch.bfloat16, dev)
        layer = tp_layer(m, g, bufs)
        with torch.no_grad():
            y = layer.forward(x2[lo:hi], pos, mask)
            res["parity_rel_l2_max"] = rel_l2(y, ref[lo:hi])
            res["tp_prefill_ms"] = time_ms(lambda: layer.forward(x2[lo:hi], pos, mask), args.warmup, args.iters, bufs.group)

            def replicated():                      # attention on every rank, only the feed-forward tensor-parallel
                a = m.att(m.norm1(x), attention_mask=mask, position_ids=pos).reshape(tokens, -1)
                return layer.ffn.forward(a[lo:hi], x2[lo:hi], tokens, addend=a[lo:hi])
            res["replicated_attention_prefill_ms"] = time_ms(replicated, args.warmup, args.iters, bufs.group)
        res["prefill_efficiency"] = res["one_gpu_prefill_ms"] / (world * res["tp_prefill_ms"])
        # training forward + backward
        params = (layer.attn.gamma, layer.attn.wq, layer.attn.wk, layer.attn.wv, layer.attn.wo, layer.ffn.gamma, layer.ffn.w_gate,
                  layer.ffn.w_up, layer.ffn.w_down)
        for p in params:
            p.requires_grad_(True)
        dy = torch.randn(hi - lo, g["hidden"], device=dev).bfloat16()

        def train_step():
            xl = x2[lo:hi].detach().requires_grad_(True)
            layer.apply(xl, pos, mask).backward(dy)
        res["tp_train_ms"] = time_ms(train_step, args.warmup, args.iters, bufs.group)
        for p in m.parameters():
            p.requires_grad_(True)
        dy_full = torch.randn(b, t, g["hidden"], device=dev).bfloat16()

        def one_gpu_train():
            xf = x.detach().requires_grad_(True)
            one_gpu_forward(m, xf, pos, mask).backward(dy_full)
        res["one_gpu_train_ms"] = time_ms(one_gpu_train, args.warmup, args.iters)
        res["train_efficiency"] = res["one_gpu_train_ms"] / (world * res["tp_train_ms"])
        for p in list(params) + list(m.parameters()):
            p.requires_grad_(False)
            p.grad = None
        del bufs, layer
        # decode: b = 64, 2048 cached tokens, one token per step
        db, past = 64, 2048
        bufs = TpRankBuffers.symmetric(db * 64, g["hidden"], torch.bfloat16, dev)
        layer = tp_layer(m, g, bufs)
        with torch.no_grad():
            cache, cache1 = KVCache(capacity=past + 64), KVCache(capacity=past + 64)
            xp = torch.randn(db, 64, g["hidden"], device=dev).bfloat16()
            for c0 in range(0, past, 64):     # fill the caches chunk by chunk (the buffers hold 64 x 64 token rows)
                p = torch.arange(c0, c0 + 64, device=dev)[None].expand(db, 64)
                lo_, hi_, _ = rows_of(db * 64, world, rank)
                layer.forward(xp.reshape(db * 64, -1)[lo_:hi_], p, causal_mask(db, 64, dev), cache, 0)
                one_gpu_forward(m, xp, p, causal_mask(db, 64, dev), cache1)
            xd = torch.randn(db, 1, g["hidden"], device=dev).bfloat16()
            lo_, hi_, _ = rows_of(db, world, rank)

            def tp_decode():
                n = cache.length(0)
                layer.forward(xd.reshape(db, -1)[lo_:hi_], torch.full((db, 1), n, device=dev), None, cache, 0)
                cache._len[0] = n                  # keep the cache at `past` tokens: every step is the same step

            def one_decode():
                n = cache1.length(0)
                one_gpu_forward(m, xd, torch.full((db, 1), n, device=dev), None, cache1)
                cache1._len[0] = n
            res["tp_decode_ms"] = time_ms(tp_decode, args.warmup, args.iters, bufs.group)
            res["one_gpu_decode_ms"] = time_ms(one_decode, args.warmup, args.iters)
        res["decode_efficiency"] = res["one_gpu_decode_ms"] / (world * res["tp_decode_ms"])
        del bufs, layer, m
        torch.cuda.empty_cache()
        if rank == 0:
            print(json.dumps(res), flush=True)
    dist.destroy_process_group()


def emulation(args):
    """Per-rank phase times at the P-way shard shapes with every rank on this one GPU."""
    dev = torch.device("cuda")
    info = gpu_info()
    p = args.emulate
    b, t = 4, 2048
    tokens = b * t
    for name in args.configs:
        g = GEOMETRY[name]
        m = one_gpu_layer(g, dev)
        x = torch.randn(b, t, g["hidden"], device=dev, generator=torch.Generator(device=dev).manual_seed(1)).bfloat16()
        pos, mask = torch.arange(t, device=dev)[None].expand(b, t), causal_mask(b, t, dev)
        x2 = x.reshape(tokens, -1)
        res = dict(config=name, mode=f"single-GPU emulation of {p} ranks (pulls / pushes are local copies, not NVLink)",
                   tokens=tokens, **info)
        with torch.no_grad():
            ref = one_gpu_forward(m, x, pos, mask).reshape(tokens, -1)
            res["one_gpu_prefill_ms"] = time_ms(lambda: one_gpu_forward(m, x, pos, mask), args.warmup, args.iters)
            bufs = TpRankBuffers.local_world(p, tokens, g["hidden"], torch.bfloat16, dev)
            layers = [tp_layer(m, g, bb) for bb in bufs]
            phases = {}
            ev = lambda: torch.cuda.Event(enable_timing=True)

            def run(rep):
                rows = [rows_of(tokens, p, r) for r in range(p)]
                marks = []

                def each(tag, fn):
                    for r, lay in enumerate(layers):
                        e0, e1 = ev(), ev()
                        e0.record()
                        out = fn(r, lay)
                        e1.record()
                        marks.append((tag, e0, e1))
                        yield out
                list(each("attn.norm", lambda r, lay: lay.attn.phase_norm(x2[rows[r][0]:rows[r][1]], tokens)))
                list(each("attn.qkv", lambda r, lay: lay.attn.phase_qkv(tokens)))
                list(each("attn.attention", lambda r, lay: lay.attn.phase_attention(pos, mask)))
                list(each("attn.out", lambda r, lay: lay.attn.phase_out(tokens)))
                a = list(each("attn.reduce", lambda r, lay: lay.attn.phase_reduce(tokens)))
                list(each("ffn.norm", lambda r, lay: lay.ffn.phase_norm(a[r], x2[rows[r][0]:rows[r][1]], tokens)))
                list(each("ffn.gate_up", lambda r, lay: lay.ffn.phase_gate_up(tokens)))
                list(each("ffn.down", lambda r, lay: lay.ffn.phase_down(tokens)))
                y = list(each("ffn.reduce", lambda r, lay: lay.ffn.phase_reduce(tokens, addend=a[r])))
                torch.cuda.synchronize()
                if rep >= args.warmup:
                    for tag, e0, e1 in marks:
                        phases.setdefault(tag, []).append(e0.elapsed_time(e1))
                return torch.cat(y)
            for rep in range(args.warmup + args.iters):
                y = run(rep)
            res["parity_rel_l2"] = rel_l2(y, ref)
            # every phase: mean over repetitions of the slowest rank (the critical path of a real run is per phase max)
            per_phase = {}
            for tag, vals in phases.items():
                reps = [max(vals[i * p:(i + 1) * p]) for i in range(len(vals) // p)]
                per_phase[tag] = sum(reps) / len(reps)
            res["phase_ms_max_over_ranks"] = {k: round(v, 4) for k, v in per_phase.items()}
            res["sum_of_phases_ms"] = round(sum(per_phase.values()), 4)
            res["scaling"] = "not measured (one GPU)"
        print(json.dumps(res), flush=True)
        del bufs, layers, m
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--configs", nargs="+", default=["11B", "90B"], choices=sorted(GEOMETRY))
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--emulate", type=int, default=8, help="ranks emulated on one GPU when run without torch.distributed")
    args = ap.parse_args()
    if "RANK" in os.environ and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        multi_gpu(args)
    else:
        emulation(args)


if __name__ == "__main__":
    main()
