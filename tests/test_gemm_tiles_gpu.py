"""The persistent tcgen05 GEMM (csrc/gemm_sm100.cu) where it branches: every SwiGLU act-tile width, cta_group 1 and 2, the
persistent loop wrapping over many tiles per CTA, ragged tile edges (checked with sentinel canaries), the two cache-load
paths of the SwiGLU backward epilogue, grouped launches, and the cross-entropy epilogue's label and tile edges.

Every output is compared element by element with a float64 reference computed from the same 16-bit inputs, against a
bound that follows from the arithmetic: the storage rounding (2^-8 for bf16, 2^-11 for fp16, times |ref|) plus
K * 2^-22 * sum_k |a_k b_k| for the fp32 accumulation.  A rel-L2 check would barely move if one 16-column chunk of one
tile were wrong; this bound does not let it pass.  The launch plan (gemm_plan.py, checked against the library on the CPU)
picks the shapes, and each test asserts through l32_debug_gemm_plan that the regime it targets was taken."""
import math

import pytest
import torch

import gemm_plan as P
from llama32_b200 import ops
from llama32_b200._lib import check, lib

pytestmark = pytest.mark.gpu
DEV = "cuda"
DTYPES = [torch.bfloat16, torch.float16]
STORE = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
ACC = 2.0 ** -22
TINY = 2.0 ** -24          # fp16 subnormal spacing
SENTINEL = -12345          # int16 bit pattern of untouched canary elements
N_ACTS = [16, 32, 48, 64, 80, 96, 112, 128]


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def rnd(g, *shape, dtype, scale=1.0):
    return (torch.randn(*shape, device=DEV, generator=g) * scale).to(dtype)


def num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def dev_plan(epilogue, m, n, cta_group=0, max_ctas=0):
    return P.library_plan(lib(), epilogue, m, n, 0, cta_group, max_ctas)


def within(got, ref, bound, what):
    """|got - ref| <= bound everywhere (NaN fails); reports the first offending element."""
    got = got.double()
    bad = ~((got - ref).abs() <= bound)
    if bool(bad.any()):
        idx = tuple(bad.nonzero()[0].tolist())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements out of bound, first at {idx}: "
                             f"got {float(got[idx]):.6g}, ref {float(ref[idx]):.6g}, bound {float(bound[idx]):.3g}")


def mm(a, b):
    """float64 a b^T and |a| |b|^T of 16-bit [m, k] x [n, k]."""
    a64, b64 = a.double(), b.double()
    return a64 @ b64.T, a64.abs() @ b64.abs().T


def check_gemm(got, ref, absum, k, dtype, what, extra=0.0):
    within(got, ref, STORE[dtype] * ref.abs() + (k + 1) * ACC * absum + extra + TINY, what)


def same_bits(a, b, what):
    assert a.shape == b.shape, (what, a.shape, b.shape)
    diff = a.contiguous().view(torch.int16) != b.contiguous().view(torch.int16)
    assert not bool(diff.any()), f"{what}: {int(diff.sum())} elements differ in their bits, first at {diff.nonzero()[0].tolist()}"


def canvas(rows, cols, dtype):
    return torch.full((rows, cols), SENTINEL, dtype=torch.int16, device=DEV).view(dtype)


def untouched(buf, mask, what):
    bits = buf.view(torch.int16)
    bad = (bits != SENTINEL) & ~mask
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} elements outside the output were written, first at {bad.nonzero()[0].tolist()}"


def stream():
    return torch.cuda.current_stream().cuda_stream


# ---------------------------------------------------------------------------------------------------- EPI_SWIGLU
def silu64(g):
    return g * torch.sigmoid(g)


def check_swiglu(x, wg, wu, bg, bu, act, gate, up, what):
    dt, k = x.dtype, x.shape[1]
    g, ga = mm(x, wg)
    u, ua = mm(x, wu)
    if bg is not None:
        g, ga = g + bg.double(), ga + bg.double().abs()
    if bu is not None:
        u, ua = u + bu.double(), ua + bu.double().abs()
    dg, du = (k + 1) * ACC * ga, (k + 1) * ACC * ua
    if gate is not None:
        within(gate, g, STORE[dt] * g.abs() + dg + TINY, f"{what} gate cache")
        within(up, u, STORE[dt] * u.abs() + du + TINY, f"{what} up cache")
    a = silu64(g) * u
    # |d silu / dg| <= 1.1; silu_f32 uses __expf and a reciprocal: (4 + 1.2 |g|) fp32 ulps relative
    bound = (STORE[dt] * a.abs() + 1.1 * u.abs() * dg + silu64(g).abs() * du + 1.1 * dg * du +
             2.0 ** -23 * (4 + 1.2 * g.abs()) * a.abs() + TINY)
    within(act, a, bound, f"{what} act")


BIASES = ["none", "gate", "up", "both"]
HIDDENS = [72, 200, 328]      # ragged last k-block: 8, 8 and 8 columns of 64


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("m,cta_group", [(257, 2), (383, 2), (1, 1), (77, 1), (128, 1)])
@pytest.mark.parametrize("n_act", N_ACTS)
def test_swiglu_every_tile_width(n_act, m, cta_group, dtype, monkeypatch):
    """Every legal act-tile width forced through L32_SWIGLU_TILE_N, both CTA groupings (the 1-CTA kernel loads gate and up
    through two maps), an inter whose last tile has 8 valid columns, one exactly one tile wide and one narrower than a
    tile, ragged k-blocks and every bias combination; act must not depend on whether the caches are written."""
    monkeypatch.setenv("L32_SWIGLU_TILE_N", str(n_act))
    monkeypatch.setenv("L32_DECODE_MAX_TOKENS", "0")     # tokens <= 128 go to the tiled kernel too
    salt = N_ACTS.index(n_act) + m + DTYPES.index(dtype)
    for i, inter in enumerate([2 * n_act + 8, n_act, max(n_act - 8, 8)]):
        hidden, bias = HIDDENS[(salt + i) % 3], BIASES[(salt + 2 * i) % 4]
        plan = dev_plan(P.EPI_SWIGLU, m, inter)
        assert (plan["n_act"], plan["cta_group"]) == (n_act, cta_group), plan
        g = gen(1000 * n_act + m + i)
        x = rnd(g, m, hidden, dtype=dtype)
        wg = rnd(g, inter, hidden, dtype=dtype, scale=hidden ** -0.5)
        wu = rnd(g, inter, hidden, dtype=dtype, scale=hidden ** -0.5)
        bg = rnd(g, inter, dtype=dtype, scale=0.5) if bias in ("gate", "both") else None
        bu = rnd(g, inter, dtype=dtype, scale=0.5) if bias in ("up", "both") else None
        act, gate, up = ops.swiglu_forward(x, wg, wu, bg, bu, want_cache=True)
        act_nc, _, _ = ops.swiglu_forward(x, wg, wu, bg, bu)
        what = f"n_act {n_act} m {m} inter {inter} hidden {hidden} bias {bias}"
        check_swiglu(x, wg, wu, bg, bu, act, gate, up, what)
        same_bits(act_nc, act, f"{what}: act with and without the caches")


# tokens x inter -> n_act the wave-cost model picks on 148 SMs (cta_group 2)
AUTO_SHAPES = [((256, 4744), 80), ((256, 5928), 96), ((256, 7112), 112), ((256, 8296), 128), ((1024, 14336), 112),
               ((512, 14336), 80)]


@pytest.mark.parametrize("shape,n_act_148", AUTO_SHAPES)
def test_swiglu_auto_planned_widths(shape, n_act_148, monkeypatch):
    monkeypatch.delenv("L32_SWIGLU_TILE_N", raising=False)
    m, inter = shape
    hidden = 128
    plan = dev_plan(P.EPI_SWIGLU, m, inter)
    assert plan == P.plan(P.EPI_SWIGLU, m, inter, num_sms())
    if num_sms() == 148:
        assert plan["n_act"] == n_act_148, plan
    g = gen(inter + m)
    x = rnd(g, m, hidden, dtype=torch.bfloat16)
    wg = rnd(g, inter, hidden, dtype=torch.bfloat16, scale=hidden ** -0.5)
    wu = rnd(g, inter, hidden, dtype=torch.bfloat16, scale=hidden ** -0.5)
    act, gate, up = ops.swiglu_forward(x, wg, wu, want_cache=True)
    check_swiglu(x, wg, wu, None, None, act, gate, up, f"{m} x {inter}, plan {plan}")


# ---------------------------------------------------------------------------------------------------- persistent loop
# k-blocks of 64: one block (8, 64), ragged (72), below / equal to / not a multiple of the 4 (cta_group 1) and 6 (cta_group
# 2) ring stages (192 = 3, 256 = 4, 384 = 6, 400 = 7, 840 = 14 blocks)
K_CASES = [(8, None), (64, None), (72, None), (192, None), (256, None), (384, None), (400, None), (840, None), (72, 8),
           (200, 328), (384, 64)]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("cta_group", [1, 2])
@pytest.mark.parametrize("k,k1", K_CASES)
def test_gemm_persistent_wrap_and_raster(k, k1, cta_group, dtype, monkeypatch):
    """Each CTA runs many tiles: the smem ring and both TMEM accumulator stages wrap mid-sequence (three clusters give
    CTAs different stage parities).  A tile computes the same bits on any CTA and in any raster order."""
    monkeypatch.delenv("L32_RASTER_GROUP", raising=False)
    m, n = 1000, 1032
    g = gen(k * 7 + (k1 or 0) + cta_group)
    a, b = rnd(g, m, k, dtype=dtype), rnd(g, n, k, dtype=dtype, scale=k ** -0.5)
    a1 = b1 = None
    ref, absum = mm(a, b)
    kk = k
    if k1 is not None:
        a1, b1 = rnd(g, m, k1, dtype=dtype), rnd(g, n, k1, dtype=dtype, scale=k1 ** -0.5)
        r1, s1 = mm(a1, b1)
        ref, absum, kk = ref + r1, absum + s1, k + k1
    d0 = ops.gemm(a, b, a1=a1, b1=b1, cta_group=cta_group)
    check_gemm(d0, ref, absum, kk, dtype, f"k {k} k1 {k1} default grid")
    for clusters in (1, 2, 3):
        plan = dev_plan(P.EPI_STORE, m, n, cta_group, clusters * cta_group)
        assert plan["ctas"] == clusters * cta_group and plan["num_tiles"] >= 3 * clusters, plan
        d = ops.gemm(a, b, a1=a1, b1=b1, cta_group=cta_group, max_ctas=clusters * cta_group)
        same_bits(d, d0, f"k {k} k1 {k1}: {clusters} cluster(s) vs the default grid")
    tiles_m = dev_plan(P.EPI_STORE, m, n, cta_group)["tiles_m"]
    for group in (1, 3, tiles_m + 2):
        monkeypatch.setenv("L32_RASTER_GROUP", str(group))
        assert dev_plan(P.EPI_STORE, m, n, cta_group)["raster_group"] == group
        d = ops.gemm(a, b, a1=a1, b1=b1, cta_group=cta_group, max_ctas=3 * cta_group)
        same_bits(d, d0, f"k {k} k1 {k1}: raster group {group}")


@pytest.mark.parametrize("a_mn,b_mn", [(True, True), (False, True), (True, False)])
@pytest.mark.parametrize("cta_group", [1, 2])
def test_gemm_mn_major_operands_wrap(a_mn, b_mn, cta_group):
    """The MN-major operand loads of the backward GEMMs, over a wrapping persistent loop."""
    m, n, k = 1000, 1032, 400
    g = gen(11 + 2 * a_mn + b_mn + cta_group)
    a, b = rnd(g, m, k, dtype=torch.bfloat16), rnd(g, n, k, dtype=torch.bfloat16, scale=k ** -0.5)
    ref, absum = mm(a, b)
    aa = a.t().contiguous() if a_mn else a
    bb = b.t().contiguous() if b_mn else b
    d0 = ops.gemm(aa, bb, a_mn_major=a_mn, b_mn_major=b_mn, cta_group=cta_group)
    check_gemm(d0, ref, absum, k, torch.bfloat16, f"mn-major a {a_mn} b {b_mn}")
    d1 = ops.gemm(aa, bb, a_mn_major=a_mn, b_mn_major=b_mn, cta_group=cta_group, max_ctas=cta_group)
    same_bits(d1, d0, "one cluster vs the default grid")


# ---------------------------------------------------------------------------------------------------- edges and canaries
EDGE_M = [1, 127, 128, 129, 255, 256, 257]
EDGE_N = [8, 120, 248, 256, 264]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("cta_group", [1, 2])
def test_gemm_store_stays_inside_the_output(cta_group, dtype):
    """D written with a row pitch ldd > n into a buffer with spare rows, all pre-filled with a sentinel: every element
    outside [m, n] keeps it."""
    L = lib()
    k = 72
    for m in EDGE_M:
        for n in EDGE_N:
            g = gen(m * 1000 + n)
            a, b = rnd(g, m, k, dtype=dtype), rnd(g, n, k, dtype=dtype, scale=k ** -0.5)
            ldd = n + 40
            buf = canvas(m + 129, ldd, dtype)
            check(L.l32_gemm(a.data_ptr(), k, 0, b.data_ptr(), k, 0, None, 0, None, 0, buf.data_ptr(), ldd, m, n, k, 0,
                             ops._dtype_code(a), cta_group, 0, stream()), "l32_gemm")
            ref, absum = mm(a, b)
            check_gemm(buf[:m, :n], ref, absum, k, dtype, f"m {m} n {n}")
            mask = torch.zeros(buf.shape, dtype=torch.bool, device=DEV)
            mask[:m, :n] = True
            untouched(buf, mask, f"cta_group {cta_group} m {m} n {n} ldd {ldd}")


@pytest.mark.parametrize("dtype", DTYPES)
def test_linear_bias_and_block_tail_addend_edges(dtype, monkeypatch):
    """The bias and the fused addend of the EPI_STORE epilogue on every 32-column part of a row, n not a multiple of 32,
    and no store past the last row."""
    monkeypatch.setenv("L32_DECODE_MAX_TOKENS", "0")
    L = lib()
    code = ops._dtype_code(torch.empty(0, dtype=dtype))
    for m in (1, 77, 129, 257):
        for n, k in ((40, 72), (120, 200), (264, 64), (1000, 136)):
            g = gen(m + n)
            a, w = rnd(g, m, k, dtype=dtype), rnd(g, n, k, dtype=dtype, scale=k ** -0.5)
            bias = rnd(g, n, dtype=dtype)
            buf = canvas(m + 3, n, dtype)
            check(L.l32_linear_forward(a.data_ptr(), w.data_ptr(), bias.data_ptr(), buf.data_ptr(), m, k, n, code, stream()),
                  "l32_linear_forward")
            ref, absum = mm(a, w)
            check_gemm(buf[:m], ref + bias.double(), absum + bias.double().abs(), k, dtype, f"linear+bias m {m} n {n}")
            mask = torch.zeros(buf.shape, dtype=torch.bool, device=DEV)
            mask[:m] = True
            untouched(buf, mask, f"linear+bias m {m} n {n}")
    # block tail: out = attn_out + act w_down^T, the addend fused into the down GEMM's epilogue
    for m, hidden, inter in ((129, 264, 200), (300, 120, 328), (77, 40, 72)):
        g = gen(m + hidden)
        attn = rnd(g, m, hidden, dtype=dtype)
        nw = (1 + 0.1 * rnd(g, hidden, dtype=torch.float32)).to(dtype)
        wg = rnd(g, inter, hidden, dtype=dtype, scale=hidden ** -0.5)
        wu = rnd(g, inter, hidden, dtype=dtype, scale=hidden ** -0.5)
        wd = rnd(g, hidden, inter, dtype=dtype, scale=inter ** -0.5)
        normed, act = torch.empty_like(attn), torch.empty(m, inter, dtype=dtype, device=DEV)
        out = canvas(m + 3, hidden, dtype)
        check(L.l32_block_tail_forward_ex(attn.data_ptr(), None, nw.data_ptr(), 1e-5, wg.data_ptr(), wu.data_ptr(), wd.data_ptr(),
                                          out.data_ptr(), normed.data_ptr(), act.data_ptr(), None, None, None, None, None, 0.0,
                                          None, None, m, hidden, inter, code, stream()), "l32_block_tail_forward_ex")
        acc, absum = mm(act, wd)
        add = attn.double()
        # two roundings: the product to 16 bit, then the sum
        within(out[:m], acc + add, STORE[dtype] * (acc.abs() + (acc + add).abs()) + (inter + 1) * ACC * absum + TINY,
               f"block tail m {m} hidden {hidden}")
        mask = torch.zeros(out.shape, dtype=torch.bool, device=DEV)
        mask[:m] = True
        untouched(out, mask, f"block tail m {m}")


# ---------------------------------------------------------------------------------------------------- EPI_SWIGLU_BWD
def align256(v):
    return (v + 255) // 256 * 256


def swiglu_bwd_call(dy, wd, gate, up, want_act):
    """l32_ffn_backward with only the d_act GEMM (and dw_down when want_act) into a sentinel-filled workspace.
    Returns (d_gate, d_up, act, workspace bytes, part size)."""
    m, hidden = dy.shape
    inter = gate.shape[1]
    L = lib()
    ws_bytes = L.l32_ffn_backward_workspace_bytes(m, inter)
    part = align256(m * inter * 2)
    assert ws_bytes == 3 * part
    ws = torch.full((ws_bytes // 2,), SENTINEL, dtype=torch.int16, device=DEV)
    dwd = torch.empty(hidden, inter, dtype=dy.dtype, device=DEV) if want_act else None
    check(L.l32_ffn_backward(dy.data_ptr(), dy.data_ptr(), wd.data_ptr(), wd.data_ptr(), wd.data_ptr(), gate.data_ptr(),
                             up.data_ptr(), None, None, None, None if dwd is None else dwd.data_ptr(), ws.data_ptr(), ws_bytes,
                             m, hidden, inter, ops._dtype_code(dy), stream()), "l32_ffn_backward")
    n = m * inter
    parts = [ws[i * part // 2:i * part // 2 + n].view(dy.dtype).view(m, inter) for i in range(3)]
    return parts[0], parts[1], parts[2], ws, part


def check_swiglu_bwd(dy, wd, gate, up, d_gate, d_up, act, what):
    dt, k = dy.dtype, dy.shape[1]
    da, dabs = mm(dy, wd.t().contiguous())          # d_act = dy w_down, w_down [hidden, inter]
    dd = (k + 1) * ACC * dabs
    g, u = gate.double(), up.double()
    s = torch.sigmoid(g)
    coef_g = u * s * (1 + g * (1 - s))
    silu = g * s
    fast = 2.0 ** -23 * (8 + 2.4 * g.abs())        # __expf + reciprocal + the products, relative
    ref_dg, ref_du = da * coef_g, da * silu
    within(d_gate, ref_dg, STORE[dt] * ref_dg.abs() + coef_g.abs() * dd + fast * ref_dg.abs() + TINY, f"{what} d_gate")
    within(d_up, ref_du, STORE[dt] * ref_du.abs() + silu.abs() * dd + fast * ref_du.abs() + TINY, f"{what} d_up")
    if act is not None:
        a = silu * u
        within(act, a, STORE[dt] * a.abs() + fast * a.abs() + TINY, f"{what} act")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("m,hidden,inter", [(129, 200, 1040), (300, 256, 1032), (77, 136, 1040), (1000, 72, 264),
                                            (257, 128, 2056)])
def test_swiglu_backward_wide_and_narrow_loads(m, hidden, inter, dtype):
    """d_gate, d_up and act against the float64 formula on the stored caches; the 32-byte streaming cache loads and the
    16-byte loads (caches at a 16- but not 32-byte aligned address) give the same bits; the slack between the workspace
    parts and, without dw_down, the act part keep their sentinel."""
    g = gen(m + inter + hidden)
    dy = rnd(g, m, hidden, dtype=dtype)
    wd = rnd(g, hidden, inter, dtype=dtype, scale=hidden ** -0.5)
    gate, up = rnd(g, m, inter, dtype=dtype, scale=2.0), rnd(g, m, inter, dtype=dtype)
    # the same caches 16 bytes into a fresh allocation: a 16- but not 32-byte aligned address
    shifted = []
    for c in (gate, up):
        raw = torch.empty(m * inter + 8, dtype=dtype, device=DEV)
        v = raw[8:].view(m, inter)
        v.copy_(c)
        assert v.data_ptr() % 32 == 16
        shifted.append(v)
    d_gate, d_up, act, ws, part = swiglu_bwd_call(dy, wd, gate, up, want_act=True)
    what = f"m {m} hidden {hidden} inter {inter} ({'wide' if inter % 16 == 0 else 'narrow'} loads)"
    check_swiglu_bwd(dy, wd, gate, up, d_gate, d_up, act, what)
    n = m * inter
    mask = torch.zeros(ws.shape, dtype=torch.bool, device=DEV)
    for i in range(3):
        mask[i * part // 2:i * part // 2 + n] = True
    untouched(ws, mask, f"{what}: workspace slack")
    d_gate2, d_up2, act2, ws2, _ = swiglu_bwd_call(dy, wd, shifted[0], shifted[1], want_act=True)
    for x, y, name in ((d_gate, d_gate2, "d_gate"), (d_up, d_up2, "d_up"), (act, act2, "act")):
        same_bits(y, x, f"{what}: {name} from 16-byte aligned caches vs aligned caches")
    d_gate3, d_up3, _, ws3, _ = swiglu_bwd_call(dy, wd, gate, up, want_act=False)
    same_bits(d_gate3, d_gate, f"{what}: d_gate without act")
    same_bits(d_up3, d_up, f"{what}: d_up without act")
    mask[2 * part // 2:] = False
    untouched(ws3, mask, f"{what}: act part without dw_down")


# ---------------------------------------------------------------------------------------------------- fp16 training
def ffn64(x, wg, wu, wd, la=None, lbs=None):
    act = silu64(x @ wg.T) * (x @ wu.T)
    y = act @ wd.T
    if la is not None:
        y = y + (act @ la.T) @ lbs.T
    return y


def rel_close(got, ref, what, rel=1e-2, mx=2.0 ** -5):
    got, ref = got.detach().double(), ref.detach().double()
    assert torch.isfinite(got).all(), f"{what}: non-finite"
    r = float((got - ref).norm() / ref.norm().clamp_min(1e-30))
    a = float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
    assert r <= rel and a <= mx, f"{what}: rel-L2 {r:.3e} (<= {rel}), max-abs/max|ref| {a:.3e} (<= {mx:.3e})"


@pytest.mark.parametrize("tokens,hidden,inter", [(300, 256, 688), (1000, 200, 1032), (129, 328, 264)])
def test_fp16_ffn_and_lora_training(tokens, hidden, inter):
    dt = torch.float16
    g = gen(tokens + hidden + inter)
    x = rnd(g, tokens, hidden, dtype=dt)
    wg = rnd(g, inter, hidden, dtype=dt, scale=hidden ** -0.5)
    wu = rnd(g, inter, hidden, dtype=dt, scale=hidden ** -0.5)
    wd = rnd(g, hidden, inter, dtype=dt, scale=inter ** -0.5)
    dy = rnd(g, tokens, hidden, dtype=dt)
    y, gate, up = ops.ffn_forward(x, wg, wu, wd, want_cache=True)
    dx, dwg, dwu, dwd, _, _ = ops.ffn_backward(dy, x, wg, wu, wd, gate, up)
    leaves = [t.double().requires_grad_(True) for t in (x, wg, wu, wd)]
    yr = ffn64(*leaves)
    yr.backward(dy.double())
    rel_close(y, yr, "fp16 ffn y")
    for got, ref, name in zip((dx, dwg, dwu, dwd), leaves, ("dx", "dw_gate", "dw_up", "dw_down")):
        rel_close(got, ref.grad, f"fp16 ffn {name}", rel=1.5e-2)
    rank = 16
    la = rnd(g, rank, inter, dtype=dt, scale=inter ** -0.5)
    lbs = rnd(g, hidden, rank, dtype=dt, scale=0.5)
    y, t, gate, up = ops.ffn_lora_forward(x, wg, wu, wd, la, lbs, want_cache=True)
    dx, dwg, dwu, dla, dlb = ops.ffn_lora_backward(dy, x, wg, wu, wd, la, lbs, t, gate, up)
    leaves = [t_.double().requires_grad_(True) for t_ in (x, wg, wu, wd, la, lbs)]
    yr = ffn64(*leaves)
    yr.backward(dy.double())
    rel_close(y, yr, "fp16 lora y")
    for got, ref, name in zip((dx, dwg, dwu, dla, dlb), [leaves[i] for i in (0, 1, 2, 4, 5)],
                              ("dx", "dw_gate", "dw_up", "dlora_a", "dlora_b")):
        rel_close(got, ref.grad, f"fp16 lora {name}", rel=1.5e-2)


# ---------------------------------------------------------------------------------------------------- grouped launches
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("tokens", [129, 300, 1000])
def test_grouped_weight_gradients_match_single_launches(tokens, dtype):
    """The 3-problem (ffn_backward) and 2-problem (swiglu_backward) grouped weight-gradient launches give the bits of the
    single-problem launches they replace."""
    hidden, inter = 264, 1032
    g = gen(tokens)
    x = rnd(g, tokens, hidden, dtype=dtype)
    wg = rnd(g, inter, hidden, dtype=dtype, scale=hidden ** -0.5)
    wu = rnd(g, inter, hidden, dtype=dtype, scale=hidden ** -0.5)
    wd = rnd(g, hidden, inter, dtype=dtype, scale=inter ** -0.5)
    dy = rnd(g, tokens, hidden, dtype=dtype)
    gate, up = rnd(g, tokens, inter, dtype=dtype, scale=2.0), rnd(g, tokens, inter, dtype=dtype)
    _, dwg, dwu, dwd, d_gate, d_up = ops.ffn_backward(dy, x, wg, wu, wd, gate, up)
    _, _, _, dwd1, _, _ = ops.ffn_backward(dy, x, wg, wu, wd, gate, up, want_dx=False, want_dw_gate_up=False)
    same_bits(dwd1, dwd, "dw_down: single launch vs the 3-problem group")
    for got, d, name in ((dwg, d_gate, "dw_gate"), (dwu, d_up, "dw_up")):
        single = ops.gemm(d, x, a_mn_major=True, b_mn_major=True)
        same_bits(got, single, f"{name}: 3-problem group vs single launch")
        ref, absum = mm(d.t().contiguous(), x.t().contiguous())
        check_gemm(got, ref, absum, tokens, dtype, name)
    d_act = rnd(g, tokens, inter, dtype=dtype)
    _, dwg2, dwu2, d_gate2, d_up2 = ops.swiglu_backward(d_act, x, wg, wu, gate, up, want_dx=False)
    for got, d, name in ((dwg2, d_gate2, "dw_gate"), (dwu2, d_up2, "dw_up")):
        same_bits(got, ops.gemm(d, x, a_mn_major=True, b_mn_major=True), f"{name}: 2-problem group vs single launch")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("tokens", [129, 300, 1000])
def test_linear_group_uneven_problems(tokens, dtype):
    """Three problems of very different widths in one tile loop: one of them a single partial tile."""
    hidden = 200
    g = gen(tokens + 5)
    a = rnd(g, tokens, hidden, dtype=dtype)
    ws = [rnd(g, n, hidden, dtype=dtype, scale=hidden ** -0.5) for n in (4096, 8, 1032)]
    ys = ops.linear_group_forward(a, ws)
    for y, w in zip(ys, ws):
        ref, absum = mm(a, w)
        check_gemm(y, ref, absum, hidden, dtype, f"group problem n {w.shape[0]}")
        same_bits(y, ops.linear_forward(a, w), f"group problem n {w.shape[0]} vs single launch")


# ---------------------------------------------------------------------------------------------------- EPI_CE
def ce_labels(m, vocab, ignore, g):
    special = [c for c in (0, 31, 32, 127, 128, 255, 256, vocab - 8, vocab - 1) if 0 <= c < vocab]
    invalid = [vocab, -1, -100, ignore]
    lab = torch.randint(0, vocab, (m,), device=DEV, generator=g)
    seq = special + invalid
    for r in range(min(m, len(seq))):
        lab[r] = seq[r]
    for r in range(len(seq), m, 7):            # more label hits all over the rows
        lab[r] = special[r % len(special)]
    return lab


def check_ce(h, w, lab, ignore, out, what):
    dt, (m, k), vocab = h.dtype, h.shape, w.shape[0]
    logits = out["logits"]
    ref, absum = mm(h, w)
    check_gemm(logits, ref, absum, k, dt, f"{what} logits")
    stored = logits.double()
    valid = (lab >= 0) & (lab < vocab) & (lab != ignore)
    lse, loss_rows, lc = out["lse"], out["loss_rows"], out["loss_and_count"]
    # lse against the stored logits: __expf errs by (2 + 1.16 |x|) ulps, weighted by exp(x) that is < (2 + 0.43) ulps per
    # term of the shifted sum; the chunk / tile rescales and sums add a few ulps per 32-column chunk level
    mx = stored.max(dim=1, keepdim=True).values
    e = torch.exp(stored - mx)
    s = e.sum(1)
    xe = ((stored - mx).abs() * e).sum(1)
    lse_ref = (mx.squeeze(1) + torch.log(s))
    tiles_n = P.cdiv(vocab, 256)
    # (plus the fp32 rounding of logit - max in every exponent, and of the final m + log(s))
    tol = 2.0 ** -23 * (4 + 2.4 * xe / s + 24 * tiles_n + 96) + 2.0 ** -22 * (lse_ref.abs() + mx.squeeze(1).abs())
    within(lse, lse_ref, tol, f"{what} lse")
    total = torch.exp(stored - lse.double()[:, None]).sum(1)
    within(total, torch.ones_like(total), 1.01 * tol, f"{what} sum of softmax")
    rows = valid.nonzero().squeeze(1)
    tgt = logits[rows, lab[rows]].float()
    want = lse[rows] - tgt                       # the same fp32 subtraction the kernel does
    bad = loss_rows[rows] != want
    assert not bool(bad.any()), (f"{what}: loss_rows != lse - logits[label] at rows {rows[bad][:8].tolist()} (labels "
                                 f"{lab[rows[bad]][:8].tolist()}): {loss_rows[rows[bad]][:4].tolist()} vs {want[bad][:4].tolist()}")
    assert bool((loss_rows[~valid] == 0).all()), f"{what}: an ignored row has a loss"
    cnt = int(valid.sum())
    assert float(lc[1]) == cnt, (what, float(lc[1]), cnt)
    if cnt == 0:
        assert math.isnan(float(lc[0])), f"{what}: loss of an all-ignored batch must be NaN"
    else:
        mean = float(loss_rows.double()[valid].mean())
        # an fp32 sum of m non-negative losses, then one division
        assert abs(float(lc[0]) - mean) <= 2.0 ** -24 * (m + 4) * abs(mean) + 1e-7, (what, float(lc[0]), mean)
    return valid, cnt


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("vocab", [8, 136, 256, 264, 1000, 128256])
@pytest.mark.parametrize("m", [77, 255, 256, 257])
def test_lm_head_ce_edges(m, vocab, dtype):
    """Labels on 32-column chunk and 256-column tile boundaries and in the last partial tile; labels that must not count
    (vocab, -1, -100, a custom ignore_index that is a real column); logits of magnitude ~80 where an unshifted exp
    overflows; a row whose maximum lies in the last tile; m <= 128, where the pair's second CTA has no rows."""
    hidden = 64
    g = gen(m * 7 + vocab)
    h = rnd(g, m, hidden, dtype=dtype)
    w = rnd(g, vocab, hidden, dtype=dtype, scale=24.0 / math.sqrt(hidden))
    h[1] = (w[vocab - 1].float() * (4.0 / w[vocab - 1].float().norm())).to(dtype)   # row 1: its maximum in the last column
    plan = dev_plan(P.EPI_CE, m, vocab, 2)
    assert plan["cta_group"] == 2 and plan["tiles_n"] == P.cdiv(vocab, 256)
    for ignore in (-100, 3):
        lab = ce_labels(m, vocab, ignore, g)
        out = ops.lm_head_ce_forward(h, w, lab, ignore_index=ignore)
        what = f"m {m} vocab {vocab} ignore {ignore}"
        if ignore == -100:
            assert int(out["logits"][1].float().argmax()) == vocab - 1, f"{what}: row 1 does not peak in the last column"
            assert float(out["logits"].float().abs().max()) > 60, what
        valid, cnt = check_ce(h, w, lab, ignore, out, what)
        dh, dw, dlogits = ops.lm_head_ce_backward(out["logits"], out["lse"], lab, ignore, out["loss_and_count"], None, h, w)
        p = torch.exp(out["logits"].double() - out["lse"].double()[:, None])
        onehot = torch.zeros_like(p)
        vr = valid.nonzero().squeeze(1)
        onehot[vr, lab[vr]] = 1.0
        ref = (p - onehot) / cnt * valid.double()[:, None]
        x = (out["logits"].double() - out["lse"].double()[:, None]).abs()
        # __expf of (logit - lse), that difference rounded in fp32, then scaled by 1 / count and stored
        fast = 2.0 ** -23 * (4 + 1.2 * x) + 2.0 ** -22 * out["lse"].double().abs()[:, None]
        within(dlogits, ref, STORE[dtype] * ref.abs() + fast * p / max(cnt, 1) + TINY, f"{what} dlogits")
        assert bool((dlogits[~valid] == 0).all()), f"{what}: an ignored row has a gradient"
        rd, ad = mm(dlogits, w.t().contiguous())
        check_gemm(dh, rd, ad, vocab, dtype, f"{what} d_hidden")
        rw, aw = mm(dlogits.t().contiguous(), h.t().contiguous())
        check_gemm(dw, rw, aw, m, dtype, f"{what} d_weight")


@pytest.mark.parametrize("dtype", DTYPES)
def test_lm_head_ce_all_ignored(dtype):
    m, hidden, vocab = 300, 64, 1000
    g = gen(5)
    h, w = rnd(g, m, hidden, dtype=dtype), rnd(g, vocab, hidden, dtype=dtype, scale=0.2)
    lab = torch.tensor([-100, -1, vocab, 7] * (m // 4), device=DEV)
    out = ops.lm_head_ce_forward(h, w, lab, ignore_index=7)
    check_ce(h, w, lab, 7, out, "all ignored")
    _, _, dlogits = ops.lm_head_ce_backward(out["logits"], out["lse"], lab, 7, out["loss_and_count"], None, h, w)
    assert bool((dlogits == 0).all()), "all-ignored batch: dlogits must be zero"


# ---------------------------------------------------------------------------------------------------- determinism
def test_tiled_path_is_deterministic_and_graph_replayable():
    dt = torch.bfloat16
    tokens, hidden, inter, vocab = 300, 256, 1032, 1000
    g = gen(77)
    x = rnd(g, tokens, hidden, dtype=dt)
    wg = rnd(g, inter, hidden, dtype=dt, scale=hidden ** -0.5)
    wu = rnd(g, inter, hidden, dtype=dt, scale=hidden ** -0.5)
    wd = rnd(g, hidden, inter, dtype=dt, scale=inter ** -0.5)
    dy = rnd(g, tokens, hidden, dtype=dt)
    wl = rnd(g, vocab, hidden, dtype=dt, scale=0.3)
    lab = torch.randint(0, vocab, (tokens,), device=DEV, generator=g)

    def step():
        y, gate, up = ops.ffn_forward(x, wg, wu, wd, want_cache=True)
        dx, dwg, dwu, dwd, _, _ = ops.ffn_backward(dy, x, wg, wu, wd, gate, up)
        ce = ops.lm_head_ce_forward(y, wl, lab)
        dh, dw, _ = ops.lm_head_ce_backward(ce["logits"], ce["lse"], lab, -100, ce["loss_and_count"], None, y, wl)
        return [y, gate, up, dx, dwg, dwu, dwd, ce["logits"], ce["lse"], ce["loss_rows"], ce["loss_and_count"], dh, dw]

    first = [t.clone() for t in step()]
    second = step()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()                                     # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = step()
    graph.replay()
    torch.cuda.synchronize()
    names = ["y", "gate", "up", "dx", "dw_gate", "dw_up", "dw_down", "logits", "lse", "loss_rows", "loss", "d_hidden", "d_lm_head"]
    for name, a, b, c in zip(names, first, second, captured):
        assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), f"{name}: two eager runs differ"
        assert torch.equal(a.view(torch.uint8), c.view(torch.uint8)), f"{name}: graph replay differs from eager"
