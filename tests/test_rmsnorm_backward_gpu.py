"""RMSNorm backward (l32_rmsnorm_backward_add) at the row counts where its loops wrap.

The fast kernel (C % 8 == 0, C <= 16384, 16-byte-aligned pointers) is persistent, grid = min(rows, SMs): a producer warp
streams rows into a ring of `stages` shared-memory slots and G = consumers / RT row groups take them in turn.  d_gamma is
summed in registers per group, folded through the idle ring, and leaves as one fp32 partial row per CTA, which
rmsnorm_dw_reduce_kernel sums.  The generic kernel runs 2 * min(rows, SMs) CTAs, so from 129 rows on a device with more than
128 SMs the reduce takes its loop over partial rows beyond 256.

Each case is a hidden size and a row count derived from the SM count and `bwd_plan`, and asserts the branch it is meant to
reach: a changed plan fails here instead of moving a case off its branch.  The GPU tests are marked one by one, so the plan
table is checked without a device as well.
"""
import pytest
import torch

from llama32_b200 import ops

DEV = "cuda"
BWD = (1e-2, 2.0 ** -5)
# One dropped or doubled row of 8192 moves d_gamma by about 1 / sqrt(8192) = 1.1 % rel-L2, which BWD cannot see; the 16-bit
# output rounding is 2^-9 and the fp32 sum over the rows adds little to it.
DGAMMA = (4e-3, 2.0 ** -8)
DW_REDUCE_ROWS = 8 * 32        # partial rows rmsnorm_dw_reduce_kernel covers without its tail loop


def bwd_plan(C):
    """(RT, G, stages) of the fast backward for hidden size C (rmsnorm_bwd_t / launch_bwd_fast), or None for the generic
    kernel.  RT threads per row, G row groups per CTA, `stages` ring slots of one dy row and one h row each."""
    if C % 8 or C > 16384:
        return None
    if C <= 1024:
        rt, consumers = 64, 512
    elif C <= 2048:
        rt, consumers = 128, 512
    elif C <= 4096:
        rt, consumers = 128, 384
    else:
        rt, consumers = 512, 512
    g = consumers // rt
    stages = (200 * 1024 - 2 * C) // (4 * C)
    stages = min(stages, -(-12 // g) * g)   # at least 12 where they fit, a multiple of G: each slot has one consumer group
    return rt, g, stages - stages % g


def test_bwd_plan_table():
    assert [bwd_plan(c) for c in (8, 1000, 1024, 1032, 2048, 2056, 4096, 4104, 8192, 16384)] == [
        (64, 8, 16), (64, 8, 16), (64, 8, 16), (128, 4, 12), (128, 4, 12), (128, 3, 12), (128, 3, 12), (512, 1, 11),
        (512, 1, 5), (512, 1, 2)]
    assert bwd_plan(1004) is None and bwd_plan(20000) is None and bwd_plan(16392) is None
    for c in range(8, 16385, 8):
        rt, g, stages = bwd_plan(c)
        assert stages % g == 0 and stages >= 2 and stages >= g - 1, c          # the d_gamma fold of G - 1 rows fits the ring
        assert stages * 4 * c + 2 * c + 2 * 16 * 8 + 2 * 16 * 16 * 4 * 2 <= 227 * 1024, c


FAST = (8, 1000, 2048, 4096, 4104, 8192, 16384)   # 1000: 125 vectors, not a multiple of RT; 4104: 513 vectors
GENERIC = ((1004, False), (20000, False), (4096, True))   # C % 8 != 0, C > 16384, a view 2 bytes past an aligned base


def _cases():
    out = []
    for c in FAST:
        for spec in ("1", "S-1", "S+1", "SG+5", "wrap") + (("8192",) if c in (4096, 8192) else ()):
            out.append((c, False, spec, torch.bfloat16))
        out.append((c, False, "wrap", torch.float16))
    for c, misaligned in GENERIC:
        for spec in ("1", "S-1", "S+1", "wrap"):
            out.append((c, misaligned, spec, torch.bfloat16))
        out.append((c, misaligned, "wrap", torch.float16))
    return out


CASES = _cases()
IDS = [f"C{c}{'-misaligned' if m else ''}-{spec}-{str(dt)[6:]}" for c, m, spec, dt in CASES]


def _rows(C, misaligned, spec):
    """Row count of a case on this device, with what the case exercises asserted."""
    S = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    plan = None if misaligned else bwd_plan(C)
    if plan is None:
        rows = {"1": 1, "S-1": S - 1, "S+1": S + 1, "wrap": 3 * S + 37}[spec]
        if spec == "wrap":
            assert 2 * min(rows, S) > DW_REDUCE_ROWS, "the d_gamma reduce must sum more than 256 partial rows"
        return rows
    _, g, stages = plan
    rows = {"1": 1, "S-1": S - 1, "S+1": S + 1, "SG+5": S * g + 5, "wrap": 3 * S * stages + 37, "8192": 8192}[spec]
    if spec == "SG+5":
        assert rows // S >= g and rows % S, "every row group of every CTA has a row, some CTAs one more"
    if spec == "wrap":
        assert rows // S >= 3 * stages and rows % S, "each CTA passes its ring at least 3 times, plus a remainder"
    return rows


def _place(x, misaligned):
    """x itself, or a contiguous copy of it that starts 2 bytes past a 16-byte boundary."""
    if not misaligned:
        return x
    flat = torch.empty(x.numel() + 8, dtype=x.dtype, device=x.device)
    v = flat[1:1 + x.numel()].view(x.shape)
    v.copy_(x)
    assert v.is_contiguous() and v.data_ptr() % 16 != 0
    return v


def _close(got, ref, tol, what):
    """rel-L2 and max-abs / max|ref| in fp64 on the device."""
    got, ref = got.double(), ref.double()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    assert torch.isfinite(got).all(), what
    r = ((got - ref).norm() / ref.norm().clamp_min(1e-300)).item()
    m = ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-300)).item()
    assert r <= tol[0] and m <= tol[1], f"{what}: rel-L2 {r:.3e} (<= {tol[0]}), max-abs/max|ref| {m:.3e} (<= {tol[1]:.3e})"


def _reference(dy, h, w, rms):
    """Closed form in fp64 with the rms the kernel is given: dx = rstd dy w - h rstd^3 mean(dy w h), dgamma = sum dy h rstd."""
    dy, h, w = dy.double(), h.double(), w.double()
    rstd = 1.0 / rms.double()[:, None]
    dyw = dy * w
    dx = rstd * dyw - h * rstd ** 3 * (dyw * h).mean(1, keepdim=True)
    return dx, (dy * h * rstd).sum(0)


def _mismatch(got, want):
    bad = got != want
    return f"{int(bad.sum())} of {bad.numel()} differ, first at {tuple(bad.nonzero()[0].tolist()) if bad.any() else None}"


@pytest.mark.gpu
@pytest.mark.parametrize("C,misaligned,spec,dtype", CASES, ids=IDS)
def test_backward_bookkeeping_is_exact(C, misaligned, spec, dtype):
    """h = +-1, dy in {0, +-1}, gamma = 1, rms in {1/2, 1} (so rstd in {1, 2}): every product and partial sum is an integer
    that fp32 holds exactly, so d_gamma must equal the fp64 reference bit for bit.  A row that lands in the wrong stage, is
    dropped, read twice, scaled by another row's rms or folded from the wrong group changes a column by at least 1.  dx is
    exact too when 1 / C is (C a power of two), else within one 16-bit ulp."""
    rows = _rows(C, misaligned, spec)
    gen = torch.Generator(device=DEV).manual_seed(C * 7919 + rows)
    sign = lambda: torch.randint(0, 2, (rows, C), generator=gen, device=DEV, dtype=torch.int8) * 2 - 1
    h = sign()
    p = min(0.5, 800.0 / rows)                      # column sums of dy h rstd stay far inside +-256
    dy = sign() * (torch.rand(rows, C, generator=gen, device=DEV) < p)
    rms = torch.where(torch.rand(rows, generator=gen, device=DEV) < 0.5, 0.5, 1.0).float()
    gamma = torch.ones(C, device=DEV, dtype=dtype)
    dx_ref, dg_ref = _reference(dy, h, gamma, rms)
    assert dg_ref.abs().max().item() <= 256, "d_gamma must be exact in the 16-bit type"
    dx, dg = ops.rmsnorm_backward(_place(dy.to(dtype), misaligned), _place(h.to(dtype), misaligned), gamma, rms)
    want = dg_ref.to(dtype)
    assert torch.equal(dg, want), f"d_gamma: {_mismatch(dg, want)}"
    if C & (C - 1) == 0:
        want = dx_ref.to(dtype)
        assert torch.equal(dx, want), f"dx: {_mismatch(dx, want)}"
    else:
        fi = torch.finfo(dtype)
        _, e = torch.frexp(dx_ref)
        ulp = torch.ldexp(torch.full_like(dx_ref, fi.eps), e - 1)          # |x| in [2^(e-1), 2^e)
        ulp = torch.where(dx_ref == 0, 0.0, ulp).clamp_min(fi.tiny * fi.eps)  # below: the subnormal step
        err = (dx.double() - dx_ref).abs() / ulp
        assert err.max().item() <= 1.0, f"dx: {int((err > 1).sum())} elements more than one ulp off, max {err.max().item():.2f}"


@pytest.mark.gpu
@pytest.mark.parametrize("C", [8, 1000, 8192, 20000])
def test_backward_zero_rows(C):
    dx, dg = ops.rmsnorm_backward(torch.empty(0, C, device=DEV, dtype=torch.bfloat16),
                                  torch.empty(0, C, device=DEV, dtype=torch.bfloat16),
                                  torch.ones(C, device=DEV, dtype=torch.bfloat16), torch.empty(0, device=DEV))
    assert dx.shape == (0, C) and dg.shape == (C,) and (dg == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("C,misaligned,spec,dtype", CASES, ids=IDS)
def test_backward_vs_fp64(C, misaligned, spec, dtype):
    """Gaussian h with a per-row scale in [1/4, 4], gaussian dy, gamma = 1 + 0.1 N, rms from the forward on the same h,
    against the closed form in fp64; then the same call with an addend (l32_rmsnorm_backward_add, the block tail's path),
    whose dx_plain must match the plain reference and dx the reference plus the addend."""
    rows = _rows(C, misaligned, spec)
    gen = torch.Generator(device=DEV).manual_seed(C * 104729 + rows)
    rn = lambda *shape: torch.randn(*shape, generator=gen, device=DEV)
    h = (rn(rows, C) * torch.exp2(4 * torch.rand(rows, 1, generator=gen, device=DEV) - 2)).to(dtype)
    dy = rn(rows, C).to(dtype)
    gamma = (1 + 0.1 * rn(C)).to(dtype)
    _, rms, _ = ops.add_rmsnorm_forward(h, gamma, None, 1e-5)
    dx_ref, dg_ref = _reference(dy, h, gamma, rms)
    dyp, hp = _place(dy, misaligned), _place(h, misaligned)
    dx, dg = ops.rmsnorm_backward(dyp, hp, gamma, rms)
    _close(dx, dx_ref, BWD, "dx")
    _close(dg, dg_ref, DGAMMA, "d_gamma")
    addend = rn(rows, C).to(dtype)
    dx, dg, dx_plain = ops.rmsnorm_backward(dyp, hp, gamma, rms, addend=addend, want_plain=True)
    _close(dx_plain, dx_ref, BWD, "dx_plain")
    _close(dx, dx_ref + addend.double(), BWD, "dx + addend")
    _close(dg, dg_ref, DGAMMA, "d_gamma (addend call)")


@pytest.mark.gpu
@pytest.mark.parametrize("C,misaligned,spec", [(8192, False, "8192"), (16384, False, "wrap"), (20000, False, "wrap"),
                                               (4096, True, "wrap")])
def test_backward_is_deterministic(C, misaligned, spec):
    """Two calls give the same bits: fixed summation order, no atomics."""
    rows = _rows(C, misaligned, spec)
    gen = torch.Generator(device=DEV).manual_seed(C + rows)
    h = _place(torch.randn(rows, C, generator=gen, device=DEV).bfloat16(), misaligned)
    dy = _place(torch.randn(rows, C, generator=gen, device=DEV).bfloat16(), misaligned)
    gamma = (1 + 0.1 * torch.randn(C, generator=gen, device=DEV)).bfloat16()
    rms = 0.5 + torch.rand(rows, generator=gen, device=DEV)
    first = ops.rmsnorm_backward(dy, h, gamma, rms)
    again = ops.rmsnorm_backward(dy, h, gamma, rms)
    assert torch.equal(first[0], again[0]), "dx"
    assert torch.equal(first[1], again[1]), "d_gamma"
