"""Tensor-parallel attention (heads sharded by KV group, collectives inside the tcgen05 GEMMs): parity against the oracle.

* single-GPU emulation: all ranks' buffers on one device, the ranks' phases run one after another, every phase of every
  rank before the next phase -- so every flag a launch waits on was raised by an earlier launch;
* real processes (torchrun, one per GPU, symmetric memory) at every power of two up to the visible GPU count.
Tolerances of tests/test_tp_fused_gpu.py: forward rel-L2 <= 1e-2 and max-abs <= 2^-6 max|ref|; gradients rel-L2 <= 1.5e-2 and
max-abs <= 2^-5 max|ref|.  Query rows that see no key at all (inside a left padding) are left out: the kernels give them
zeros, the reference a uniform softmax over padded keys (GroupQueryAttention documents this).
"""
import os
import subprocess
import sys

import pytest
import torch

from llama32_b200 import ops
from llama32_b200.modules import KVCache
from llama32_b200.tp import (FLAG_READY, FLAG_RS_DONE, FusedTensorParallelAttention, FusedTensorParallelBlock,
                             TensorParallelDecoderLayer, TpAttnSaved, TpRankBuffers, shard_attention_weights)
from oracle import ffn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 1e-5


def _close(got, ref, what, rtol=1e-2, mtol=2.0 ** -6):
    got, ref = got.float().cpu(), ref.float().cpu()
    r, m = O.rel_l2(got, ref), O.max_abs_over_max_ref(got, ref)
    assert r <= rtol and m <= mtol, f"{what}: rel-L2 {r:.3e}, max-abs/max|ref| {m:.3e}"


def _grad_close(got, ref, what):
    _close(got, ref, what, 1.5e-2, 2.0 ** -5)


def _synthetic(b, t, hidden, n_heads, n_kv, d, seed):
    """bf16-representable fp32 inputs: x ~ N(0,1), gamma1 = 1 + 0.1 N(0,1), weights ~ U(+-1/sqrt(fan_in))."""
    g = torch.Generator().manual_seed(seed)
    r = O.bf16_representable
    u = lambda rows, cols: r((torch.rand(rows, cols, generator=g) * 2 - 1) / cols ** 0.5)
    return dict(x=r(torch.randn(b, t, hidden, generator=g)), gamma=r(1 + 0.1 * torch.randn(hidden, generator=g)),
                wq=u(n_heads * d, hidden), wk=u(n_kv * d, hidden), wv=u(n_kv * d, hidden), wo=u(hidden, n_heads * d),
                dy=r(torch.randn(b, t, hidden, generator=g)))


def _mask(b, t, pad):
    """(4-D reference mask | None, [b, t] bool of the query rows that see at least one key).  pad None: no masking; else
    causal + a left padding of `pad` keys on every second sequence."""
    if pad is None:
        return None, torch.ones(b, t, dtype=torch.bool)
    keep = torch.ones(b, t)
    keep[1::2, :pad] = 0
    return O.causal_padding_mask(keep, t), keep.bool()


def _blocks(s, bufs, n_heads, n_kv):
    bf = lambda v: v.to(DEV, torch.bfloat16)
    return [FusedTensorParallelAttention(bf(s["gamma"]), EPS, bf(s["wq"]), bf(s["wk"]), bf(s["wv"]), bf(s["wo"]), n_heads, n_kv, bb)
            for bb in bufs]


def _attn_forward_emulated(blocks, x2, pos, mask_dev, caches=None, layer_idx=0):
    """Every forward phase of every rank before the next phase; returns the concatenated rows of all ranks."""
    tokens = pos.numel()
    for blk in blocks:
        lo, hi, _ = blk.rows_of(tokens)
        blk.phase_norm(x2[lo:hi], tokens)
    for blk in blocks:
        blk.phase_qkv(tokens)
    for r, blk in enumerate(blocks):
        blk.phase_attention(pos, mask_dev, None if caches is None else caches[r], layer_idx)
    for blk in blocks:
        blk.phase_out(tokens)
    return torch.cat([blk.phase_reduce(tokens) for blk in blocks])


@pytest.mark.parametrize("world,n_heads,n_kv,d,b,t,pad", [
    (1, 8, 2, 64, 2, 77, 5), (2, 8, 2, 128, 3, 100, 5), (3, 6, 3, 64, 2, 333, 200), (3, 12, 6, 128, 1, 250, None),
    (4, 16, 8, 64, 4, 300, 140), (8, 16, 8, 128, 2, 300, 7), (8, 32, 8, 64, 3, 129, None), (2, 4, 2, 128, 2, 1000, 300)])
def test_attention_forward_emulation(world, n_heads, n_kv, d, b, t, pad):
    hidden = n_heads * d
    s = _synthetic(b, t, hidden, n_heads, n_kv, d, seed=world * 31 + d)
    mask, valid = _mask(b, t, pad)
    pos = torch.arange(t)[None].expand(b, t)
    ref, _, _ = O.gqa_attention(O.add_rmsnorm(s["x"], s["gamma"], EPS), s["wq"], s["wk"], s["wv"], s["wo"], n_heads, n_kv, pos, mask)
    tokens = b * t
    bufs = TpRankBuffers.local_world(world, tokens, hidden, torch.bfloat16, DEV)
    blocks = _blocks(s, bufs, n_heads, n_kv)
    assert all(blk.heads == n_heads // world and blk.kv_heads == n_kv // world for blk in blocks)
    x2 = s["x"].reshape(tokens, hidden).to(DEV, torch.bfloat16)
    mask_dev = None if mask is None else mask.to(DEV)
    pos_dev = pos.to(DEV)
    keep_rows = valid.reshape(-1)
    for step in range(2):   # the second step re-uses buffers and flags (epoch 2)
        y = _attn_forward_emulated(blocks, x2, pos_dev, mask_dev)
        torch.cuda.synchronize()
        assert y.shape == (tokens, hidden)
        _close(y[keep_rows.to(DEV)], ref.reshape(tokens, hidden)[keep_rows], f"TP attention world={world} d={d} step={step}")


@pytest.mark.parametrize("world,n_heads,n_kv,d,b", [(8, 16, 8, 64, 1), (8, 32, 8, 128, 3), (2, 8, 2, 128, 4), (4, 8, 4, 64, 2)])
def test_attention_prefill_then_decode_with_rank_caches(world, n_heads, n_kv, d, b):
    """Prefill then several decode steps through one KVCache per rank (local KV heads only); at b < world some ranks own
    no rows of a decode step."""
    hidden, t0, steps = n_heads * d, 40, 4
    s = _synthetic(b, t0 + steps, hidden, n_heads, n_kv, d, seed=world + 7 * b)
    bf = lambda v: v.to(DEV, torch.bfloat16)
    bufs = TpRankBuffers.local_world(world, b * t0, hidden, torch.bfloat16, DEV)
    blocks = _blocks(s, bufs, n_heads, n_kv)
    caches = [KVCache() for _ in range(world)]
    normed = O.add_rmsnorm(s["x"], s["gamma"], EPS)
    mask, _ = _mask(b, t0, 0)                       # causal, no padding
    pos = torch.arange(t0)[None].expand(b, t0)
    ref, k_all, v_all = O.gqa_attention(normed[:, :t0], s["wq"], s["wk"], s["wv"], s["wo"], n_heads, n_kv, pos, mask)
    y = _attn_forward_emulated(blocks, bf(s["x"][:, :t0].reshape(b * t0, hidden)), pos.to(DEV), mask.to(DEV), caches)
    torch.cuda.synchronize()
    _close(y, ref.reshape(-1, hidden), f"prefill world={world} b={b}")
    for i in range(steps):
        p = torch.full((b, 1), t0 + i, dtype=torch.int64)
        ref, k_all, v_all = O.gqa_attention(normed[:, t0 + i:t0 + i + 1], s["wq"], s["wk"], s["wv"], s["wo"], n_heads, n_kv, p, None,
                                            past_k=k_all, past_v=v_all)
        y = _attn_forward_emulated(blocks, bf(s["x"][:, t0 + i]), p.to(DEV), None, caches)
        torch.cuda.synchronize()
        _close(y, ref.reshape(b, hidden), f"decode step {i} world={world} b={b}")
    kv_per = n_kv // world
    for r, c in enumerate(caches):
        assert c.length(0) == t0 + steps and c.key_cache[0].shape[1] == kv_per
        _close(c.key_cache[0], k_all[:, r * kv_per:(r + 1) * kv_per], f"rank {r} cached keys")


def _oracle_attention_grads(s, n_heads, n_kv, pos, mask, dy):
    leaves = {k: s[k].clone().requires_grad_(True) for k in ("x", "gamma", "wq", "wk", "wv", "wo")}
    y, _, _ = O.gqa_attention(O.add_rmsnorm(leaves["x"], leaves["gamma"], EPS), leaves["wq"], leaves["wk"], leaves["wv"], leaves["wo"],
                              n_heads, n_kv, pos, mask)
    y.backward(dy)
    return y.detach(), {k: v.grad for k, v in leaves.items()}


@pytest.mark.parametrize("world,n_heads,n_kv,d,b,t,pad", [
    (1, 8, 2, 128, 2, 200, None), (2, 8, 2, 128, 2, 300, 37), (3, 6, 3, 64, 3, 150, 0), (4, 16, 8, 64, 2, 257, 0),
    (8, 16, 8, 128, 1, 512, 0)])
def test_attention_forward_backward_phases_emulation(world, n_heads, n_kv, d, b, t, pad):
    """Training forward + backward phase by phase against fp32 autograd: dx, dgamma1 and every rank's weight shards."""
    hidden, tokens = n_heads * d, b * t
    s = _synthetic(b, t, hidden, n_heads, n_kv, d, seed=world * 5 + t)
    mask, valid = _mask(b, t, pad)
    dy = s["dy"] * valid[..., None]                 # rows that see no key carry no gradient (see the module docstring)
    pos = torch.arange(t)[None].expand(b, t)
    yref, gref = _oracle_attention_grads(s, n_heads, n_kv, pos, mask, dy)
    bufs = TpRankBuffers.local_world(world, tokens, hidden, torch.bfloat16, DEV)
    blocks = _blocks(s, bufs, n_heads, n_kv)
    bf = lambda v: v.to(DEV, torch.bfloat16)
    x2, dy2 = bf(s["x"].reshape(tokens, hidden)), bf(dy.reshape(tokens, hidden))
    mask_dev, pos_dev = (None if mask is None else mask.to(DEV)), pos.to(DEV)
    for step in range(2):
        saved = [TpAttnSaved() for _ in blocks]
        for blk, sv in zip(blocks, saved):
            lo, hi, _ = blk.rows_of(tokens)
            blk.phase_norm(x2[lo:hi], tokens, sv)
        for blk, sv in zip(blocks, saved):
            blk.phase_qkv(tokens, sv)
        for blk, sv in zip(blocks, saved):
            blk.phase_attention(pos_dev, mask_dev, saved=sv)
        for blk in blocks:
            blk.phase_out(tokens)
        y = torch.cat([blk.phase_reduce(tokens) for blk in blocks])
        rows = valid.reshape(-1)
        _close(y[rows.to(DEV)], yref.reshape(tokens, hidden)[rows], f"train forward world={world} step={step}")
        for blk, sv in zip(blocks, saved):
            lo, hi, _ = blk.rows_of(tokens)
            blk.bwd_phase_publish(dy2[lo:hi], sv)
        for blk, sv in zip(blocks, saved):
            blk.bwd_phase_dctx(sv)
        for blk, sv in zip(blocks, saved):
            blk.bwd_phase_attention(sv)
        for blk, sv in zip(blocks, saved):
            blk.bwd_phase_dx(sv)
        wgr = [blk.bwd_phase_wgrads(sv) for blk, sv in zip(blocks, saved)]
        outs = [blk.bwd_phase_reduce_norm(sv) for blk, sv in zip(blocks, saved)]
        torch.cuda.synchronize()
        _grad_close(torch.cat([o[0] for o in outs]), gref["x"].reshape(tokens, hidden), f"dx world={world} step={step}")
        _grad_close(sum(o[1].float() for o in outs), gref["gamma"], "dgamma1")
        for r, (dwq, dwk, dwv, dwo) in enumerate(wgr):
            rq, rk, rv, ro = shard_attention_weights(gref["wq"], gref["wk"], gref["wv"], gref["wo"], n_heads, n_kv, world, r)
            _grad_close(dwq, rq, f"dwq shard {r}")
            _grad_close(dwk, rk, f"dwk shard {r}")
            _grad_close(dwv, rv, f"dwv shard {r}")
            _grad_close(dwo, ro, f"dwo shard {r}")


def _layer_ref(s, f, n_heads, n_kv, pos, mask):
    attn, _, _ = O.gqa_attention(O.add_rmsnorm(s["x"], s["gamma"], EPS), s["wq"], s["wk"], s["wv"], s["wo"], n_heads, n_kv, pos, mask)
    return O.block_hot_path(attn, s["x"], f["gamma"], EPS, f["w_gate"], f["w_up"], f["w_down"])[2]


@pytest.mark.parametrize("world,n_heads,n_kv,d,b,t,inter", [(2, 8, 2, 64, 2, 300, 1024), (4, 8, 4, 128, 3, 128, 2048),
                                                             (8, 16, 8, 64, 1, 700, 2048)])
def test_decoder_layer_emulation(world, n_heads, n_kv, d, b, t, inter):
    """Attention + feed-forward blocks on ONE buffer set, two steps (epochs 1..4), against the oracle layer."""
    hidden, tokens = n_heads * d, b * t
    s = _synthetic(b, t, hidden, n_heads, n_kv, d, seed=world + 100)
    f = O.synthetic_ffn(tokens, hidden, inter, seed=world + 200)
    mask, _ = _mask(b, t, 0)
    pos = torch.arange(t)[None].expand(b, t)
    ref = _layer_ref(s, f, n_heads, n_kv, pos, mask).reshape(tokens, hidden)
    bf = lambda v: v.to(DEV, torch.bfloat16)
    bufs = TpRankBuffers.local_world(world, tokens, hidden, torch.bfloat16, DEV)
    attn = _blocks(s, bufs, n_heads, n_kv)
    ffn = [FusedTensorParallelBlock(bf(f["gamma"]), EPS, bf(f["w_gate"]), bf(f["w_up"]), bf(f["w_down"]), bb) for bb in bufs]
    x2 = bf(s["x"].reshape(tokens, hidden))
    for step in range(2):
        a_out = _attn_forward_emulated(attn, x2, pos.to(DEV), mask.to(DEV))
        parts = []
        for blk in ffn:
            lo, hi, _ = blk.rows_of(tokens)
            parts.append((lo, hi))
            blk.phase_norm(a_out[lo:hi], x2[lo:hi], tokens)
        for blk in ffn:
            blk.phase_gate_up(tokens)
        for blk in ffn:
            blk.phase_down(tokens)
        y = torch.cat([blk.phase_reduce(tokens, addend=a_out[lo:hi]) for blk, (lo, hi) in zip(ffn, parts)])
        torch.cuda.synchronize()
        _close(y, ref, f"decoder layer world={world} step={step}")
    assert all(bb.epoch == 4 for bb in bufs)


def test_decoder_layer_world1_forward_and_autograd():
    """At world 1 nothing waits on another rank, so the composed module calls run as they are: forward() with a cache and
    apply() through autograd, every gradient against fp32 autograd over the oracle layer."""
    n_heads, n_kv, d, b, t, inter = 8, 2, 128, 2, 192, 1024
    hidden, tokens = n_heads * d, b * t
    s = _synthetic(b, t, hidden, n_heads, n_kv, d, seed=41)
    f = O.synthetic_ffn(tokens, hidden, inter, seed=42)
    mask, _ = _mask(b, t, 0)
    pos = torch.arange(t)[None].expand(b, t)
    bf = lambda v: v.to(DEV, torch.bfloat16)
    bufs = TpRankBuffers.local_world(1, tokens, hidden, torch.bfloat16, DEV)[0]
    attn = FusedTensorParallelAttention(bf(s["gamma"]), EPS, bf(s["wq"]), bf(s["wk"]), bf(s["wv"]), bf(s["wo"]), n_heads, n_kv, bufs)
    ffn = FusedTensorParallelBlock(bf(f["gamma"]), EPS, bf(f["w_gate"]), bf(f["w_up"]), bf(f["w_down"]), bufs)
    layer = TensorParallelDecoderLayer(attn, ffn)
    ref = _layer_ref(s, f, n_heads, n_kv, pos, mask).reshape(tokens, hidden)
    y = layer.forward(bf(s["x"].reshape(tokens, hidden)), pos.to(DEV), mask.to(DEV), KVCache(), 0)
    _close(y, ref, "layer forward with a cache")

    leaves = {k: s[k].clone().requires_grad_(True) for k in ("x", "gamma", "wq", "wk", "wv", "wo")}
    fl = {k: f[k].clone().requires_grad_(True) for k in ("gamma", "w_gate", "w_up", "w_down")}
    yr = _layer_ref(leaves, fl, n_heads, n_kv, pos, mask)
    yr.backward(f["dy"].reshape(b, t, hidden))
    for tns in (attn.gamma, attn.wq, attn.wk, attn.wv, attn.wo, ffn.gamma, ffn.w_gate, ffn.w_up, ffn.w_down):
        tns.requires_grad_(True)
    for step in range(2):
        for tns in (attn.gamma, attn.wq, attn.wk, attn.wv, attn.wo, ffn.gamma, ffn.w_gate, ffn.w_up, ffn.w_down):
            tns.grad = None
        xl = bf(s["x"].reshape(tokens, hidden)).requires_grad_(True)
        y = layer.apply(xl, pos.to(DEV), mask.to(DEV))
        y.backward(bf(f["dy"]))
        torch.cuda.synchronize()
        _close(y, yr.detach().reshape(tokens, hidden), f"layer apply step {step}")
        _grad_close(xl.grad, leaves["x"].grad.reshape(tokens, hidden), "dx")
        for got, name in ((attn.gamma, "gamma"), (attn.wq, "wq"), (attn.wk, "wk"), (attn.wv, "wv"), (attn.wo, "wo")):
            _grad_close(got.grad, leaves[name].grad, f"attention d{name}")
        for got, name in ((ffn.gamma, "gamma"), (ffn.w_gate, "w_gate"), (ffn.w_up, "w_up"), (ffn.w_down, "w_down")):
            _grad_close(got.grad, fl[name].grad, f"ffn d{name}")


# ---------------------------------------------------------------------------------------------- the new GEMM entries
def _publish(bufs, x):
    """Every rank writes its own rows of x into its exchange buffer and raises its ready flag (a new epoch)."""
    tokens = x.shape[0]
    for bb in bufs:
        ep = bb.next_epoch()
        per = -(-tokens // bb.world)
        lo, hi = min(bb.rank * per, tokens), min((bb.rank + 1) * per, tokens)
        bb.normed[lo:hi].copy_(x[lo:hi])
        ops.tp_signal(bb.peer_flags, FLAG_READY + bb.rank, ep, x.device, zero8=bb.done)
    return -(-tokens // bufs[0].world)


@pytest.mark.parametrize("world,tokens,hidden,outs", [(1, 300, 256, (512, 128, 128)), (2, 1000, 512, (256,)),
                                                      (3, 777, 384, (512, 128)), (2, 4096, 1024, (512, 128, 128)),
                                                      (8, 64, 256, (256, 64, 64))])
def test_group_forward_allgather_matches_gemm(world, tokens, hidden, outs):
    """Grouped q/k/v GEMM with the all-gather pulled in, gathering in place and into a caller-owned tensor."""
    g = torch.Generator(device=DEV).manual_seed(tokens)
    x = torch.randn(tokens, hidden, device=DEV, generator=g).bfloat16()
    ws = [(torch.randn(o, hidden, device=DEV, generator=g) / hidden ** 0.5).bfloat16() for o in outs]
    refs = [ops.gemm(x, w) for w in ws]
    bufs = TpRankBuffers.local_world(world, tokens, hidden, torch.bfloat16, DEV)
    for step in range(2):
        own = step == 1 and world > 1
        per = _publish(bufs, x)
        dsts = [torch.empty_like(x) if own else bb.normed[:tokens] for bb in bufs]
        ys = [ops.tp_linear_group_forward_allgather(d_, bb.peer_normed, bb.flags[FLAG_READY:FLAG_READY + 8], bb.done, bb.epoch,
                                                    bb.rank, per, ws) for d_, bb in zip(dsts, bufs)]
        torch.cuda.synchronize()
        for r, (rank_ys, d_) in enumerate(zip(ys, dsts)):
            assert torch.equal(d_, x), f"gathered rows of rank {r}"
            for i, (y, ref) in enumerate(zip(rank_ys, refs)):
                _close(y, ref, f"world={world} rank {r} problem {i} step {step}", rtol=2e-3, mtol=2.0 ** -8)
    if world == 1:   # the tiled path of linear_group_forward, bit for bit
        for y, yr in zip(ys[0], ops.linear_group_forward(x, ws)):
            assert torch.equal(y, yr)


@pytest.mark.parametrize("world,tokens,hidden,out_f", [(2, 1000, 512, 256), (4, 2048, 2048, 512), (1, 130, 256, 128)])
def test_forward_allgather_mn_major_matches_gemm(world, tokens, hidden, out_f):
    g = torch.Generator(device=DEV).manual_seed(out_f)
    dy = torch.randn(tokens, hidden, device=DEV, generator=g).bfloat16()
    wo = (torch.randn(hidden, out_f, device=DEV, generator=g) / hidden ** 0.5).bfloat16()   # [hidden, heads_local * d]
    bufs = TpRankBuffers.local_world(world, tokens, hidden, torch.bfloat16, DEV)
    per = _publish(bufs, dy)
    dsts = [torch.empty_like(dy) if world > 1 else bb.normed[:tokens] for bb in bufs]
    ys = [ops.tp_linear_forward_allgather(d_, bb.peer_normed, bb.flags[FLAG_READY:FLAG_READY + 8], bb.done, bb.epoch, bb.rank, per, wo,
                                          w_mn_major=True) for d_, bb in zip(dsts, bufs)]
    torch.cuda.synchronize()
    ref = ops.gemm(dy, wo, b_mn_major=True)
    for y, d_ in zip(ys, dsts):
        _close(y, ref, f"d_ctx world={world}", rtol=2e-3, mtol=2.0 ** -8)
        assert torch.equal(d_, dy)


@pytest.mark.parametrize("world,tokens,hidden,ks", [(1, 300, 256, (256, 64, 64)), (2, 1000, 512, (512, 128, 128)),
                                                    (3, 777, 384, (128, 128)), (8, 2048, 1024, (512, 128, 128)),
                                                    (4, 64, 256, (128,))])
def test_group_backward_dx_reduce_scatter(world, tokens, hidden, ks):
    """Three-phase partial dX with the reduce-scatter pushed out: the owners' sums equal sum over ranks of the partials."""
    g = torch.Generator(device=DEV).manual_seed(tokens + len(ks))
    bufs = TpRankBuffers.local_world(world, tokens, hidden, torch.bfloat16, DEV)
    per = -(-tokens // world)
    total = torch.zeros(tokens, hidden, device=DEV)
    for step in range(2):
        ref = torch.zeros(tokens, hidden, device=DEV)
        for bb in bufs:
            ep = bb.next_epoch()
            dys = [torch.randn(tokens, k, device=DEV, generator=g).bfloat16() for k in ks]
            ws = [(torch.randn(k, hidden, device=DEV, generator=g) / k ** 0.5).bfloat16() for k in ks]
            ref += sum(dy_.float() @ w.float() for dy_, w in zip(dys, ws))
            ops.tp_linear_group_backward_dx_reduce_scatter(dys, ws, bb.peer_slots, bb.rank, per)
            ops.tp_signal(bb.peer_flags, FLAG_RS_DONE + bb.rank, ep, DEV)
        out = torch.cat([ops.tp_reduce_partials(bb.slots, bb.flags[FLAG_RS_DONE:FLAG_RS_DONE + 8], bb.epoch, bb.rank,
                                                max(min(per, tokens - bb.rank * per), 0)) for bb in bufs])
        torch.cuda.synchronize()
        assert out.shape == (tokens, hidden)
        _close(out, ref, f"three-phase dX world={world} step={step}")


# ---------------------------------------------------------------------------------------------- real processes
def _pow2_upto_device_count():
    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    out, p = [], 2
    while p <= max(n, 2):
        out.append(p)
        p *= 2
    return out


@pytest.mark.parametrize("nproc", _pow2_upto_device_count() or [2])
def test_tp_attention_multi_process(nproc):
    """One process per GPU on symmetric memory: layer forward, autograd forward + backward of the whole layer, a KV-cached
    decode loop and the shard shapes of the 11B / 90B models."""
    if torch.cuda.device_count() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr",
           "127.0.0.1", "--master-port", str(29611 + nproc), os.path.join(ROOT, "tests", "tp_attention_worker.py")]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1200, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-4000:]
    for tag in ("tp attention layer ok", "tp attention backward ok", "tp attention decode ok", "tp attention model shards ok"):
        assert tag in r.stdout, r.stdout[-4000:]
