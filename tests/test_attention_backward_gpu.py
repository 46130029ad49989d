"""GPU: attention backward for training calls (GQAAttentionFunction, l32_gqa_attention_forward_train / _backward).

Gradients are compared with the project's gradient tolerances (rel-L2 <= 1e-2, max-abs <= 2^-5 * max|ref|) against fp32
autograd on the CPU: of the softmax written out at kernel level, and of the reference's own expressions at module level.
"""
import copy
import math

import pytest
import torch

import llama32_b200 as L
from llama32_b200 import ops
from oracle import ffn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
FWD = (1e-2, 2.0 ** -6)
BWD = (1e-2, 2.0 ** -5)
BASE = 500000.0


def close(got, ref, tol, what=""):
    got = got.detach().float().cpu()
    ref = ref.detach().float().cpu()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    assert torch.isfinite(got).all(), what
    r, m = O.rel_l2(got, ref), O.max_abs_over_max_ref(got, ref)
    assert r <= tol[0] and m <= tol[1], f"{what}: rel-L2 {r:.3e} (<= {tol[0]}), max-abs/max|ref| {m:.3e} (<= {tol[1]:.3e})"


def _rope(x, pos, d):
    """RoPE of x [b, h, t, d] at positions pos [b, t] in fp32 (angles as the kernels compute them)."""
    i = torch.arange(d // 2, dtype=torch.float32)
    inv = torch.exp2(-math.log2(BASE) * (2.0 * i / d))
    ang = pos.float()[:, None, :, None] * inv
    cs, sn = ang.cos(), ang.sin()
    x1, x2 = x[..., : d // 2], x[..., d // 2:]
    return torch.cat((x1 * cs - x2 * sn, x2 * cs + x1 * sn), -1)


def _attention_ref(q, k, v, pos, causal, keep, heads, kv, d):
    """fp32 softmax attention over pre-RoPE q [b, t, heads*d], k / v [b, t, kv*d]; rows without a visible key give zeros."""
    b, t, _ = q.shape
    q4 = _rope(q.view(b, t, heads, d).transpose(1, 2), pos, d)
    k4 = _rope(k.view(b, t, kv, d).transpose(1, 2), pos, d).repeat_interleave(heads // kv, 1)
    v4 = v.view(b, t, kv, d).transpose(1, 2).repeat_interleave(heads // kv, 1)
    sc = q4 @ k4.transpose(-1, -2) / d ** 0.5
    m = torch.ones(t, t, dtype=torch.bool)
    if causal:
        m &= torch.arange(t)[None] <= torch.arange(t)[:, None]
    m = m[None, None] & keep[:, None, None, :].bool()
    alive = m.any(-1, keepdim=True)
    pr = torch.softmax(sc.masked_fill(~m, -1e30), -1) * alive
    return (pr @ v4).transpose(1, 2).reshape(b, t, heads * d), alive[:, 0, :, 0]


def _inputs(b, t, heads, kv, d, pad, seed):
    gen = torch.Generator().manual_seed(seed)
    rep = lambda x: x.to(torch.bfloat16).float()
    q = rep(torch.randn(b, t, heads * d, generator=gen))
    k = rep(torch.randn(b, t, kv * d, generator=gen))
    v = rep(torch.randn(b, t, kv * d, generator=gen))
    g = rep(torch.randn(b, t, heads * d, generator=gen))
    keep = torch.ones(b, t, dtype=torch.uint8)
    keep[0, :pad] = 0
    pos = (7 + 3 * torch.arange(b)[:, None] + torch.arange(t)[None]).to(torch.int64)   # positions that do not start at 0
    return q, k, v, g, keep, pos


def _gpu_fwd_bwd(q, k, v, g, keep, pos, causal, heads, kv, d, dtype):
    b, t, _ = q.shape
    qr = q.to(DEV, dtype).contiguous()
    ck = torch.empty(b, kv, t, d, device=DEV, dtype=dtype)
    cv = torch.empty_like(ck)
    ops.rope_kv_append(qr, k.to(DEV, dtype), v.to(DEV, dtype), pos.to(DEV), ck, cv, 0, BASE)
    keep_d = keep.to(DEV)
    ctx, lse = ops.gqa_attention_forward_train(qr, ck, cv, causal, keep_d)
    grads = ops.gqa_attention_backward(g.to(DEV, dtype), qr, ck, cv, ctx, lse, pos.to(DEV), causal, keep_d, BASE)
    return ctx, lse, grads, (qr, ck, cv, keep_d)


GRID = [  # (b, t, heads, kv, d, causal, pad, dtype): the forward key-padding test's grid, then t in {1, 63, 129, 300, 2048}
    (1, 128, 1, 1, 128, True, 0, torch.bfloat16), (1, 128, 1, 1, 128, True, 5, torch.bfloat16),
    (1, 128, 1, 1, 128, True, 37, torch.bfloat16), (1, 128, 1, 1, 128, True, 64, torch.bfloat16),
    (1, 128, 1, 1, 128, True, 70, torch.bfloat16), (2, 300, 4, 2, 128, True, 37, torch.bfloat16),
    (2, 300, 4, 2, 64, True, 37, torch.bfloat16), (2, 512, 8, 2, 128, False, 0, torch.bfloat16),
    (1, 2048, 8, 2, 128, True, 100, torch.bfloat16),
    (2, 1, 4, 1, 128, True, 0, torch.bfloat16), (3, 63, 4, 4, 64, True, 3, torch.float16),
    (1, 129, 8, 2, 128, False, 0, torch.float16), (2, 129, 4, 1, 64, True, 17, torch.bfloat16),
    (2, 300, 8, 2, 128, True, 0, torch.float16), (1, 2048, 4, 1, 64, True, 0, torch.float16),
    (1, 300, 2, 1, 128, False, 40, torch.float16),
]


@pytest.mark.parametrize("b,t,heads,kv,d,causal,pad,dtype", GRID)
def test_attention_backward_kernels_vs_fp32_autograd(b, t, heads, kv, d, causal, pad, dtype):
    """dq, dk, dv of the pre-RoPE projections (inverse RoPE included) against fp32 autograd of the softmax written out.
    Rows that see no key must give dq == 0 exactly and lse == +inf; padded keys dk == dv == 0 exactly."""
    q, k, v, g, keep, pos = _inputs(b, t, heads, kv, d, pad, seed=b * 131 + t + pad + d)
    ctx, lse, (dq, dk, dv), _ = _gpu_fwd_bwd(q, k, v, g, keep, pos, causal, heads, kv, d, dtype)
    qs, ks, vs = (x.clone().requires_grad_(True) for x in (q, k, v))
    ref, alive = _attention_ref(qs, ks, vs, pos, causal, keep, heads, kv, d)
    (ref * g).sum().backward()
    close(ctx, ref, FWD, "ctx")
    if t == 1:   # one key: the softmax is constant, dq and dk are zero up to the rounding of delta (from the 16-bit ctx)
        for got, ref in ((dq, qs.grad), (dk, ks.grad)):
            assert ref.abs().max() == 0 and got.float().abs().max().item() < 1e-4 * g.abs().max().item()
    else:
        close(dq, qs.grad, BWD, "dq")
        close(dk, ks.grad, BWD, "dk")
    close(dv, vs.grad, BWD, "dv")
    lse_c = lse.cpu()
    assert torch.isfinite(lse_c.transpose(1, 2)[alive]).all()
    dead = ~alive
    if dead.any():
        assert torch.isinf(lse_c.transpose(1, 2)[dead]).all()
        assert (dq.float().cpu()[dead] == 0).all(), "rows without any visible key must give dq == 0 exactly"
    padded = keep == 0
    if padded.any():
        assert (dk.float().cpu()[padded] == 0).all() and (dv.float().cpu()[padded] == 0).all(), "padded keys: dk = dv = 0"


def test_attention_backward_is_deterministic():
    """Two backward calls on the same inputs give the same bits (no floating-point atomics; the GQA reduction is in TMEM)."""
    b, t, heads, kv, d = 2, 700, 8, 2, 128
    q, k, v, g, keep, pos = _inputs(b, t, heads, kv, d, 13, seed=5)
    ctx, lse, first, (qr, ck, cv, keep_d) = _gpu_fwd_bwd(q, k, v, g, keep, pos, True, heads, kv, d, torch.bfloat16)
    gd = g.to(DEV, torch.bfloat16)
    for _ in range(2):
        again = ops.gqa_attention_backward(gd, qr, ck, cv, ctx, lse, pos.to(DEV), True, keep_d, BASE)
        for a, bb, what in zip(first, again, ("dq", "dk", "dv")):
            assert torch.equal(a, bb), what


class _Cfg:
    def __init__(self, hidden, heads, kv, rope_base=BASE):
        self.hidden_size, self.n_heads, self.n_kv_groups, self.rope_base = hidden, heads, kv, rope_base


def _alive_rows(mask2d):
    """[b, t]: causal rows that see at least one unpadded key."""
    return mask2d.bool().cumsum(-1) > 0


def _trainable(m):
    return [(n, p) for n, p in m.named_parameters() if p.requires_grad]


@pytest.mark.parametrize("lora", [False, True])
def test_group_query_attention_training_vs_reference_module(lora):
    """GroupQueryAttention in bf16 under autograd (projections on LinearFunction / LinearLoRAFunction, attention on
    GQAAttentionFunction) against a CPU fp32 copy of the same module, which evaluates the reference's expressions.  4-D causal
    + padding mask; the loss is weighted to zero on rows that see no key."""
    torch.manual_seed(11)
    b, t, hidden, heads, kv = 2, 300, 512, 4, 2
    att = L.GroupQueryAttention(_Cfg(hidden, heads, kv))
    if lora:
        for name in ("W_query", "W_key", "W_value", "out_proj"):
            old = getattr(att, name)
            setattr(att, name, L.Linear_LORA(old.in_features, old.out_features, 16, 32, 0.0))
    with torch.no_grad():
        for p in att.parameters():
            p.copy_(O.bf16_representable(p))
    ref = copy.deepcopy(att).float()
    gpu = att.to(DEV, torch.bfloat16).train()
    assert not lora or not gpu.W_query.linear.weight.requires_grad
    mask2d = torch.ones(b, t)
    mask2d[0, :9] = 0                      # left padding: the first rows of sequence 0 see no key
    mask2d[1, t - 5:] = 0
    mask4 = O.causal_padding_mask(mask2d, t)
    pos = torch.arange(t)[None].expand(b, -1).contiguous()
    x = O.bf16_representable(torch.randn(b, t, hidden))
    w = O.bf16_representable(torch.randn(b, t, hidden)) * _alive_rows(mask2d)[..., None]
    xg = x.to(DEV, torch.bfloat16).requires_grad_(True)
    y = gpu(xg, attention_mask=mask4.to(DEV, torch.bfloat16), position_ids=pos.to(DEV))
    assert y.grad_fn is not None
    (y.float() * w.to(DEV)).sum().backward()
    xr = x.clone().requires_grad_(True)
    yr = ref(xr, attention_mask=mask4, position_ids=pos)
    (yr * w).sum().backward()
    alive = _alive_rows(mask2d)
    close(y.float().cpu()[alive], yr.detach()[alive], FWD, "y")
    close(xg.grad, xr.grad, BWD, "dx")
    got, want = dict(_trainable(gpu)), dict(_trainable(ref))
    assert sorted(got) == sorted(want) and got
    for n in want:
        close(got[n].grad, want[n].grad, BWD, f"d {n}")


def test_decoder_layer_forward_backward_vs_fp32_cpu():
    """norm1 -> attention -> block_tail (the reference's TransformerBlock, Model/model.py:265-273) forward + backward in bf16
    on the kernels against the same layer in fp32 on the CPU."""
    torch.manual_seed(5)
    b, t, hidden, heads, kv, inter = 2, 200, 256, 4, 2, 688

    class Layer(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.norm1, self.norm2 = L.LLAMARMSNorm(hidden, 1e-5), L.LLAMARMSNorm(hidden, 1e-5)
            self.att = L.GroupQueryAttention(_Cfg(hidden, heads, kv))
            self.ff = L.FusedFeedforward(hidden, inter)

        def forward(self, x, mask, pos):
            a = self.att(self.norm1(x), attention_mask=mask, position_ids=pos)
            return L.block_tail(self.norm2, self.ff, a, x)

    layer = Layer()
    with torch.no_grad():
        for p in layer.parameters():
            p.copy_(O.bf16_representable(p + (0.1 * torch.randn_like(p) if p.dim() == 1 else 0.0)))
    ref = copy.deepcopy(layer).float()
    gpu = layer.to(DEV, torch.bfloat16)
    mask4 = O.causal_padding_mask(torch.ones(b, t), t)
    pos = torch.arange(t)[None].expand(b, -1).contiguous()
    x = O.bf16_representable(torch.randn(b, t, hidden))
    gy = O.bf16_representable(torch.randn(b, t, hidden))
    xg = x.to(DEV, torch.bfloat16).requires_grad_(True)
    y = gpu(xg, mask4.to(DEV, torch.bfloat16), pos.to(DEV))
    y.backward(gy.to(DEV, torch.bfloat16))
    xr = x.clone().requires_grad_(True)
    yr = ref(xr, mask4, pos)
    yr.backward(gy)
    close(y, yr, FWD, "y")
    close(xg.grad, xr.grad, BWD, "dx")
    got, want = dict(gpu.named_parameters()), dict(ref.named_parameters())
    for n, p in want.items():
        close(got[n].grad, p.grad, BWD, f"d {n}")


def test_attention_training_memory_is_linear_in_tokens():
    """1 x 8192 tokens, 32 / 8 heads of 128: forward + backward of GQAAttentionFunction allocate under 512 MiB above their
    inputs (the reference's saved probabilities alone are 4.3 GB at this size)."""
    b, t, heads, kv, d = 1, 8192, 32, 8, 128
    q = torch.randn(b, t, heads * d, device=DEV, dtype=torch.bfloat16, requires_grad=True)
    k = torch.randn(b, t, kv * d, device=DEV, dtype=torch.bfloat16, requires_grad=True)
    v = torch.randn(b, t, kv * d, device=DEV, dtype=torch.bfloat16, requires_grad=True)
    g = torch.randn(b, t, heads * d, device=DEV, dtype=torch.bfloat16)
    pos = torch.arange(t, device=DEV)[None].contiguous()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = L.GQAAttentionFunction.apply(q, k, v, pos, True, None, BASE, kv)
    out.backward(g)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < 512 * 2 ** 20, f"peak {peak / 2 ** 20:.0f} MiB above the inputs"
    assert torch.isfinite(q.grad.float()).all() and torch.isfinite(k.grad.float()).all() and torch.isfinite(v.grad.float()).all()


def test_attention_train_forward_backward_graph_replay():
    """forward_train + backward captured once in a CUDA graph and replayed give the same bits as eager execution (nothing
    allocates outside torch's allocator, nothing synchronises)."""
    b, t, heads, kv, d = 2, 320, 8, 2, 64
    q, k, v, g, keep, pos = _inputs(b, t, heads, kv, d, 20, seed=9)
    qr = q.to(DEV, torch.bfloat16).contiguous()
    ck = torch.empty(b, kv, t, d, device=DEV, dtype=torch.bfloat16)
    cv = torch.empty_like(ck)
    ops.rope_kv_append(qr, k.to(DEV, torch.bfloat16), v.to(DEV, torch.bfloat16), pos.to(DEV), ck, cv, 0, BASE)
    gd, keep_d, pos_d = g.to(DEV, torch.bfloat16), keep.to(DEV), pos.to(DEV)

    def step():
        ctx, lse = ops.gqa_attention_forward_train(qr, ck, cv, True, keep_d)
        return (ctx, lse) + ops.gqa_attention_backward(gd, qr, ck, cv, ctx, lse, pos_d, True, keep_d, BASE)

    eager = step()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()                                       # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = step()
    graph.replay()
    torch.cuda.synchronize()
    for a, bb, what in zip(eager, captured, ("ctx", "lse", "dq", "dk", "dv")):
        assert torch.equal(a, bb), what
