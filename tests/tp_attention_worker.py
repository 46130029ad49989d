"""torchrun worker: tensor-parallel attention and the whole tensor-parallel decoder layer on real GPUs (one process per
GPU, symmetric memory) against the CPU oracle.  Launched by tests/test_tp_attention_gpu.py::test_tp_attention_multi_process
(and runnable by hand: python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tests/tp_attention_worker.py).
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from llama32_b200.modules import KVCache  # noqa: E402
from llama32_b200.tp import (FusedTensorParallelAttention, FusedTensorParallelBlock, TensorParallelDecoderLayer,  # noqa: E402
                             TpRankBuffers, shard_attention_weights, shard_range)
from oracle import ffn_oracle as O  # noqa: E402

EPS = 1e-5


def _check(got, ref, what, rtol=1e-2, mtol=2.0 ** -6):
    got, ref = got.float().cpu(), ref.float().cpu()
    r, m = O.rel_l2(got, ref), O.max_abs_over_max_ref(got, ref)
    assert r <= rtol and m <= mtol, f"{what}: rel-L2 {r:.3e}, max-abs/max|ref| {m:.3e}"


def _synthetic(b, t, hidden, n_heads, n_kv, d, inter, seed):
    g = torch.Generator().manual_seed(seed)       # same seed -> same tensors on every rank
    r = O.bf16_representable
    u = lambda rows, cols: r((torch.rand(rows, cols, generator=g) * 2 - 1) / cols ** 0.5)
    s = dict(x=r(torch.randn(b, t, hidden, generator=g)), gamma=r(1 + 0.1 * torch.randn(hidden, generator=g)),
             wq=u(n_heads * d, hidden), wk=u(n_kv * d, hidden), wv=u(n_kv * d, hidden), wo=u(hidden, n_heads * d),
             dy=r(torch.randn(b * t, hidden, generator=g)))
    f = O.synthetic_ffn(b * t, hidden, inter, seed=seed + 1)
    return s, f


def _layer_ref(s, f, n_heads, n_kv, pos, mask):
    attn, _, _ = O.gqa_attention(O.add_rmsnorm(s["x"], s["gamma"], EPS), s["wq"], s["wk"], s["wv"], s["wo"], n_heads, n_kv, pos, mask)
    return O.block_hot_path(attn, s["x"], f["gamma"], EPS, f["w_gate"], f["w_up"], f["w_down"])[2]


def _layer(s, f, n_heads, n_kv, bufs, dev):
    bf = lambda v: v.to(dev, torch.bfloat16)
    attn = FusedTensorParallelAttention(bf(s["gamma"]), EPS, bf(s["wq"]), bf(s["wk"]), bf(s["wv"]), bf(s["wo"]), n_heads, n_kv, bufs)
    ffn = FusedTensorParallelBlock(bf(f["gamma"]), EPS, bf(f["w_gate"]), bf(f["w_up"]), bf(f["w_down"]), bufs)
    return TensorParallelDecoderLayer(attn, ffn)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    bf = lambda t: t.to(dev, torch.bfloat16)
    kv = 8
    # ---- whole layer forward, full oracle (causal + left padding: rows that see no key left out)
    for b, t, n_heads, d, inter in [(2, 300, 16, 64, 2048), (3, 257, 32, 128, 4096)]:
        hidden = n_heads * d
        s, f = _synthetic(b, t, hidden, n_heads, kv, d, inter, seed=3)
        keep = torch.ones(b, t)
        keep[1, :37] = 0
        mask, pos = O.causal_padding_mask(keep, t), torch.arange(t)[None].expand(b, t)
        ref = _layer_ref(s, f, n_heads, kv, pos, mask).reshape(b * t, hidden)
        bufs = TpRankBuffers.symmetric(b * t, hidden, torch.bfloat16, dev)
        layer = _layer(s, f, n_heads, kv, bufs, dev)
        lo, hi, _ = layer.attn.rows_of(b * t)
        rows = keep.bool().reshape(-1)[lo:hi]
        for step in range(2):
            y = layer.forward(bf(s["x"].reshape(b * t, hidden)[lo:hi]), pos.to(dev), mask.to(dev))
            torch.cuda.synchronize()
            _check(y[rows.to(dev)], ref[lo:hi][rows], f"rank {rank} layer {(b, t, n_heads, d)} step {step}")
        del bufs, layer
        dist.barrier()
    if rank == 0:
        print("tp attention layer ok", flush=True)
    # ---- whole layer forward + backward through autograd, every gradient against autograd over the oracle
    b, t, n_heads, d, inter = 2, 384, 16, 128, 4096
    hidden = n_heads * d
    s, f = _synthetic(b, t, hidden, n_heads, kv, d, inter, seed=9)
    mask, pos = O.causal_padding_mask(torch.ones(b, t), t), torch.arange(t)[None].expand(b, t)
    leaves = {k: s[k].clone().requires_grad_(True) for k in ("x", "gamma", "wq", "wk", "wv", "wo")}
    fl = {k: f[k].clone().requires_grad_(True) for k in ("gamma", "w_gate", "w_up", "w_down")}
    yr = _layer_ref(leaves, fl, n_heads, kv, pos, mask)
    yr.backward(s["dy"].reshape(b, t, hidden))
    bufs = TpRankBuffers.symmetric(b * t, hidden, torch.bfloat16, dev)
    layer = _layer(s, f, n_heads, kv, bufs, dev)
    params = (layer.attn.gamma, layer.attn.wq, layer.attn.wk, layer.attn.wv, layer.attn.wo, layer.ffn.gamma, layer.ffn.w_gate,
              layer.ffn.w_up, layer.ffn.w_down)
    for p in params:
        p.requires_grad_(True)
    lo, hi, _ = layer.attn.rows_of(b * t)
    rq, rk, rv, ro = shard_attention_weights(*(leaves[k].grad for k in ("wq", "wk", "wv", "wo")), n_heads, kv, world, rank)
    slo, shi = shard_range(inter, world, rank)
    g = dict(rtol=1.5e-2, mtol=2.0 ** -5)
    for step in range(2):
        for p in params:
            p.grad = None
        xl = bf(s["x"].reshape(b * t, hidden)[lo:hi]).requires_grad_(True)
        y = layer.apply(xl, pos.to(dev), mask.to(dev))
        y.backward(bf(s["dy"][lo:hi]))
        torch.cuda.synchronize()
        what = f"rank {rank} train step {step}"
        _check(y, yr.detach().reshape(b * t, hidden)[lo:hi], what + " y")
        _check(xl.grad, leaves["x"].grad.reshape(b * t, hidden)[lo:hi], what + " dx", **g)
        for got, ref, name in ((layer.attn.gamma, leaves["gamma"].grad, "dgamma1"), (layer.attn.wq, rq, "dwq"),
                               (layer.attn.wk, rk, "dwk"), (layer.attn.wv, rv, "dwv"), (layer.attn.wo, ro, "dwo"),
                               (layer.ffn.gamma, fl["gamma"].grad, "dgamma2"), (layer.ffn.w_gate, fl["w_gate"].grad[slo:shi], "dw_gate"),
                               (layer.ffn.w_up, fl["w_up"].grad[slo:shi], "dw_up"), (layer.ffn.w_down, fl["w_down"].grad[:, slo:shi], "dw_down")):
            _check(got.grad, ref, f"{what} {name}", **g)
    del bufs, layer
    dist.barrier()
    if rank == 0:
        print("tp attention backward ok", flush=True)
    # ---- KV-cached decode loop of the whole layer (b = 1 and b = 3: at world 8 some ranks own no rows of a step)
    for b in (1, 3):
        t0, steps, n_heads, d, inter = 64, 6, 16, 128, 2048
        hidden = n_heads * d
        s, f = _synthetic(b, t0 + steps, hidden, n_heads, kv, d, inter, seed=20 + b)
        f = O.synthetic_ffn(b * t0, hidden, inter, seed=21 + b)
        bufs = TpRankBuffers.symmetric(b * t0, hidden, torch.bfloat16, dev)
        layer = _layer(s, f, n_heads, kv, bufs, dev)
        cache = KVCache()
        normed = O.add_rmsnorm(s["x"], s["gamma"], EPS)
        past_k = past_v = None
        for i in range(1 + steps):
            sl = slice(0, t0) if i == 0 else slice(t0 + i - 1, t0 + i)
            tt = sl.stop - sl.start
            pos = torch.arange(sl.start, sl.stop)[None].expand(b, tt)
            mask = O.causal_padding_mask(torch.ones(b, tt), tt) if i == 0 else None
            attn, past_k, past_v = O.gqa_attention(normed[:, sl], s["wq"], s["wk"], s["wv"], s["wo"], n_heads, kv, pos, mask,
                                                   past_k=past_k, past_v=past_v)
            ref = O.block_hot_path(attn, s["x"][:, sl], f["gamma"], EPS, f["w_gate"], f["w_up"], f["w_down"])[2].reshape(b * tt, hidden)
            lo, hi, _ = layer.attn.rows_of(b * tt)
            y = layer.forward(bf(s["x"][:, sl].reshape(b * tt, hidden)[lo:hi]), pos.to(dev), None if mask is None else mask.to(dev),
                              cache, 0)
            torch.cuda.synchronize()
            _check(y, ref[lo:hi], f"rank {rank} decode b={b} step {i}")
        del bufs, layer
        dist.barrier()
    if rank == 0:
        print("tp attention decode ok", flush=True)
    # ---- shard shapes of the real models at this world size: 11B (32 / 8 heads of 128, hidden 4096) and 90B (64 / 8,
    #      hidden 8192); oracle on 32 rows of every rank
    for n_heads, hidden in ((32, 4096), (64, 8192)):
        b, t, d = 1, 1024, 128
        s, f = _synthetic(b, t, hidden, n_heads, kv, d, 256, seed=30)
        bufs = TpRankBuffers.symmetric(b * t, hidden, torch.bfloat16, dev)
        attn = FusedTensorParallelAttention(bf(s["gamma"]), EPS, bf(s["wq"]), bf(s["wk"]), bf(s["wv"]), bf(s["wo"]), n_heads, kv, bufs)
        assert attn.heads == n_heads // world and attn.kv_heads == kv // world
        mask, pos = O.causal_padding_mask(torch.ones(b, t), t), torch.arange(t)[None].expand(b, t)
        ref, _, _ = O.gqa_attention(O.add_rmsnorm(s["x"], s["gamma"], EPS), s["wq"], s["wk"], s["wv"], s["wo"], n_heads, kv, pos, mask)
        ref = ref.reshape(t, hidden)
        lo, hi, _ = attn.rows_of(t)
        rows = torch.arange(lo, hi)[torch.linspace(0, hi - lo - 1, 32).long()]
        y = attn.forward(bf(s["x"].reshape(t, hidden)[lo:hi]), pos.to(dev), mask.to(dev))
        torch.cuda.synchronize()
        _check(y[(rows - lo).to(dev)], ref[rows], f"rank {rank} model shard {n_heads} heads hidden {hidden}")
        del bufs, attn
        dist.barrier()
    if rank == 0:
        print("tp attention model shards ok", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
