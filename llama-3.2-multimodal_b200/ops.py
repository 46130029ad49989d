"""Tensor-level wrappers over the C-ABI: torch is used only for device memory and the current stream.

Every function takes CUDA bf16/fp16 tensors, allocates outputs with torch, and enqueues the kernels on
torch's current stream of the tensor's device.
"""
from __future__ import annotations

import ctypes
import weakref

import torch

from ._lib import L32Error, check, lib

_DT = {torch.bfloat16: 0, torch.float16: 1}
KV_PAGE = 64   # tokens per page of a paged KV cache (L32_KV_PAGE, include/l32_ffn.h): one key tile of the attention kernel


def _dtype_code(t: torch.Tensor) -> int:
    try:
        return _DT[t.dtype]
    except KeyError:
        raise L32Error(f"unsupported dtype {t.dtype}: the sm_100a kernels take bfloat16 or float16") from None


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _check_cuda(*ts):
    dev = None
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise L32Error("expected CUDA tensors (the CUDA path has no CPU fallback)")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise L32Error(f"tensors on different devices: {dev} vs {t.device}")
    return dev


# Cast / contiguous copies of WEIGHTS are cached per source tensor (and its version counter): a norm weight kept in fp32
# next to bf16 activations, or a non-contiguous view, would otherwise cost a cast kernel on every call -- a visible tax on
# a 60 us decode step -- and, worse, that cast would be a producer launched directly in front of a kernel that prefetches
# its weights before it waits for the previous kernel (include/l32_ffn.h, "weights must be final").  On a miss the new
# copy is made and the stream is synchronised once (skipped while a CUDA graph is being captured: capture follows a
# warm-up run, which has filled the cache).
_weight_cache: dict[int, tuple] = {}


def _weight(w: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    if w.dtype == dtype and w.is_contiguous():
        return w
    key = id(w)
    ent = _weight_cache.get(key)
    if ent is not None and ent[0]() is w and ent[1] == w._version and ent[2].dtype == dtype and ent[3] == w.data_ptr():
        return ent[2]
    cast = w.detach().contiguous().to(dtype)
    if w.is_cuda and not torch.cuda.is_current_stream_capturing():
        torch.cuda.current_stream(w.device).synchronize()
    _weight_cache[key] = (weakref.ref(w, lambda _r, k=key: _weight_cache.pop(k, None)), w._version, cast, w.data_ptr())
    return cast


def supported(x: torch.Tensor) -> bool:
    """The reference's gate for its CUDA path (Model/model.py:165): CUDA tensor of a 16-bit float type."""
    return x.is_cuda and x.dtype in _DT


# --------------------------------------------------------------------------------------------- RMSNorm
def add_rmsnorm_forward(x, weight, residual=None, eps=1e-5, *, want_h=False, want_rms=True, h_out=None, out=None):
    """y = rmsnorm(x + residual) * weight.  Returns (y, rms|None, h|None).

    h (= x + residual rounded to x.dtype) is produced only when `want_h` and a residual is given (without a
    residual h is x itself).  `h_out` lets the raw reference ABI alias h onto `residual`.
    """
    _check_cuda(x, weight, residual)
    hidden = x.shape[-1]
    xc = x.contiguous()
    rows = xc.numel() // hidden if hidden else 0
    rc = None if residual is None else residual.contiguous()
    if rc is not None and rc.shape != xc.shape:
        raise L32Error(f"residual shape {tuple(rc.shape)} != input shape {tuple(xc.shape)}")
    w = _weight(weight, xc.dtype)
    if w.numel() != hidden:
        raise L32Error(f"weight has {w.numel()} elements, expected {hidden}")
    if out is not None:
        if out.shape != xc.shape or out.dtype != xc.dtype or not out.is_contiguous():
            raise L32Error("add_rmsnorm_forward: `out` must be a contiguous tensor shaped and typed like the input")
        y = out
    else:
        y = torch.empty_like(xc)
    rms = torch.empty(rows, dtype=torch.float32, device=xc.device) if want_rms else None
    h = h_out
    if h is None and want_h and rc is not None:
        h = torch.empty_like(xc)
    with torch.cuda.device(xc.device):
        check(lib().l32_add_rmsnorm_forward(_ptr(xc), _ptr(rc), _ptr(w), _ptr(y), _ptr(h), _ptr(rms), rows, hidden,
                                            float(eps), _dtype_code(xc), _stream(xc)), "l32_add_rmsnorm_forward")
    return y.view(x.shape), rms, (h.view(x.shape) if h is not None else None)


def rmsnorm_backward(grad_out, h, weight, rms, *, want_dweight=True, addend=None, want_plain=False):
    """(dx, dweight|None) for y = rmsnorm(h) * weight, given rms = sqrt(mean(h^2) + eps) from the forward.
    `addend` (shaped like h): dx = (norm backward) + addend, added in the kernel's store pass; with `want_plain` the
    return value is (dx, dweight|None, dx_plain) where dx_plain is the norm backward without the addend."""
    _check_cuda(grad_out, h, weight, rms, addend)
    hidden = h.shape[-1]
    hc = h.contiguous()
    gc = grad_out.contiguous()
    if gc.dtype != hc.dtype:
        gc = gc.to(hc.dtype)
    rows = hc.numel() // hidden if hidden else 0
    w = _weight(weight, hc.dtype)
    dx = torch.empty_like(hc)
    dw = torch.empty(hidden, dtype=hc.dtype, device=hc.device) if want_dweight else None
    L = lib()
    ws_bytes = L.l32_rmsnorm_backward_workspace_bytes(rows, hidden)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=hc.device)
    ad = None
    if addend is not None:
        ad = addend.contiguous()
        if ad.shape != hc.shape or ad.dtype != hc.dtype:
            raise L32Error("rmsnorm_backward: `addend` must be shaped and typed like h")
    dxp = torch.empty_like(hc) if (want_plain and ad is not None) else None
    with torch.cuda.device(hc.device):
        check(L.l32_rmsnorm_backward_add(_ptr(gc), _ptr(hc), _ptr(w), _ptr(rms.contiguous()), _ptr(ad), _ptr(dx), _ptr(dxp),
                                         _ptr(dw), _ptr(ws), ws_bytes, rows, hidden, _dtype_code(hc), _stream(hc)),
              "l32_rmsnorm_backward_add")
    if want_plain:
        return dx.view(h.shape), dw, (dxp.view(h.shape) if dxp is not None else dx.view(h.shape))
    return dx.view(h.shape), dw


# --------------------------------------------------------------------------------------------- SwiGLU / FFN
def _flat_tokens(x):
    hidden = x.shape[-1]
    xc = x.contiguous()
    return xc.view(-1, hidden), xc.numel() // hidden if hidden else 0


def _check_ffn_weights(x2, w_gate, w_up, w_down=None):
    inter, hidden = w_gate.shape
    if x2.shape[1] != hidden or tuple(w_up.shape) != (inter, hidden):
        raise L32Error(f"shape mismatch: x[..., {x2.shape[1]}], w_gate{tuple(w_gate.shape)}, w_up{tuple(w_up.shape)}")
    if w_down is not None and tuple(w_down.shape) != (hidden, inter):
        raise L32Error(f"w_down{tuple(w_down.shape)} is not [hidden={hidden}, inter={inter}]")
    for w in (w_gate, w_up, w_down):
        if w is not None and w.dtype != x2.dtype:
            raise L32Error(f"weight dtype {w.dtype} != activation dtype {x2.dtype}")
    return hidden, inter


def swiglu_forward(x, w_gate, w_up, b_gate=None, b_up=None, *, want_cache=False):
    """act = silu(x w_gate^T + b_gate) * (x w_up^T + b_up).  Returns (act, gate_cache|None, up_cache|None)."""
    _check_cuda(x, w_gate, w_up, b_gate, b_up)
    x2, tokens = _flat_tokens(x)
    wg, wu = _weight(w_gate, w_gate.dtype), _weight(w_up, w_up.dtype)
    hidden, inter = _check_ffn_weights(x2, wg, wu)
    out_shape = (*x.shape[:-1], inter)
    act = torch.empty(tokens, inter, dtype=x2.dtype, device=x2.device)
    gate = torch.empty_like(act) if want_cache else None
    up = torch.empty_like(act) if want_cache else None
    bg = None if b_gate is None else _weight(b_gate, x2.dtype)
    bu = None if b_up is None else _weight(b_up, x2.dtype)
    with torch.cuda.device(x2.device):
        check(lib().l32_swiglu_forward(_ptr(x2), _ptr(wg), _ptr(wu), _ptr(bg), _ptr(bu), _ptr(act), _ptr(gate), _ptr(up),
                                       tokens, hidden, inter, _dtype_code(x2), _stream(x2)), "l32_swiglu_forward")
    if want_cache:
        return act.view(out_shape), gate.view(out_shape), up.view(out_shape)
    return act.view(out_shape), None, None


def swiglu_backward(grad_act, x, w_gate, w_up, gate_cache, up_cache, *, want_dx=True, want_dw=True):
    """(dx|None, dw_gate|None, dw_up|None, d_gate, d_up); d_gate/d_up are views into the workspace."""
    _check_cuda(grad_act, x, w_gate, w_up, gate_cache, up_cache)
    x2, tokens = _flat_tokens(x)
    wg, wu = _weight(w_gate, w_gate.dtype), _weight(w_up, w_up.dtype)
    hidden, inter = _check_ffn_weights(x2, wg, wu)
    ga = grad_act.contiguous().view(-1, inter)
    if ga.dtype != x2.dtype:
        ga = ga.to(x2.dtype)
    dx = torch.empty_like(x2) if want_dx else None
    dwg = torch.empty_like(wg) if want_dw else None
    dwu = torch.empty_like(wu) if want_dw else None
    L = lib()
    ws_bytes = L.l32_swiglu_backward_workspace_bytes(tokens, inter)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=x2.device)
    with torch.cuda.device(x2.device):
        check(L.l32_swiglu_backward(_ptr(ga), _ptr(x2), _ptr(wg), _ptr(wu), _ptr(gate_cache.contiguous()),
                                    _ptr(up_cache.contiguous()), _ptr(dx), _ptr(dwg), _ptr(dwu), _ptr(ws), ws_bytes,
                                    tokens, hidden, inter, _dtype_code(x2), _stream(x2)), "l32_swiglu_backward")
    part = ws_bytes // 2
    n = tokens * inter
    d_gate = ws[:n * 2].view(x2.dtype).view(tokens, inter)
    d_up = ws[part:part + n * 2].view(x2.dtype).view(tokens, inter)
    return (dx.view(x.shape) if dx is not None else None), dwg, dwu, d_gate, d_up


def linear_forward(a, weight, bias=None):
    """y = a weight^T + bias with weight [out_features, in_features] (nn.Linear layout)."""
    _check_cuda(a, weight, bias)
    a2, tokens = _flat_tokens(a)
    w = _weight(weight, weight.dtype)
    out_f, in_f = w.shape
    if a2.shape[1] != in_f or w.dtype != a2.dtype:
        raise L32Error(f"linear: a[..., {a2.shape[1]}] {a2.dtype} vs weight{tuple(w.shape)} {w.dtype}")
    y = torch.empty(tokens, out_f, dtype=a2.dtype, device=a2.device)
    b = None if bias is None else _weight(bias, a2.dtype)
    with torch.cuda.device(a2.device):
        check(lib().l32_linear_forward(_ptr(a2), _ptr(w), _ptr(b), _ptr(y), tokens, in_f, out_f, _dtype_code(a2),
                                       _stream(a2)), "l32_linear_forward")
    return y.view(*a.shape[:-1], out_f)


def linear_group_forward(a, weights):
    """[a w^T for w in weights] (1..3 bias-free nn.Linear weights over the same activations) in one launch."""
    _check_cuda(a, *weights)
    if not 1 <= len(weights) <= 3:
        raise L32Error("linear_group_forward takes one to three weights")
    a2, tokens = _flat_tokens(a)
    ws = [_weight(w, w.dtype) for w in weights]
    in_f = a2.shape[1]
    for w in ws:
        if w.shape[1] != in_f or w.dtype != a2.dtype:
            raise L32Error(f"linear group: a[..., {in_f}] {a2.dtype} vs weight{tuple(w.shape)} {w.dtype}")
    ys = [torch.empty(tokens, w.shape[0], dtype=a2.dtype, device=a2.device) for w in ws]
    n = len(ws)
    w_arr = (ctypes.c_void_p * n)(*[_ptr(w) for w in ws])
    y_arr = (ctypes.c_void_p * n)(*[_ptr(y) for y in ys])
    o_arr = (ctypes.c_int * n)(*[w.shape[0] for w in ws])
    with torch.cuda.device(a2.device):
        check(lib().l32_linear_group_forward(_ptr(a2), w_arr, y_arr, o_arr, n, tokens, in_f, _dtype_code(a2), _stream(a2)),
              "l32_linear_group_forward")
    return [y.view(*a.shape[:-1], y.shape[1]) for y in ys]


def ffn_forward(x, w_gate, w_up, w_down, b_gate=None, b_up=None, b_down=None, *, want_cache=False):
    """y = (silu(x w_gate^T) * (x w_up^T)) w_down^T.  Returns (y, gate_cache|None, up_cache|None)."""
    _check_cuda(x, w_gate, w_up, w_down, b_gate, b_up, b_down)
    x2, tokens = _flat_tokens(x)
    wg, wu, wd = _weight(w_gate, w_gate.dtype), _weight(w_up, w_up.dtype), _weight(w_down, w_down.dtype)
    hidden, inter = _check_ffn_weights(x2, wg, wu, wd)
    y = torch.empty(tokens, hidden, dtype=x2.dtype, device=x2.device)
    act = torch.empty(tokens, inter, dtype=x2.dtype, device=x2.device)
    gate = torch.empty_like(act) if want_cache else None
    up = torch.empty_like(act) if want_cache else None
    cast = lambda b: None if b is None else _weight(b, x2.dtype)
    bg, bu, bd = cast(b_gate), cast(b_up), cast(b_down)
    with torch.cuda.device(x2.device):
        check(lib().l32_ffn_forward(_ptr(x2), _ptr(wg), _ptr(wu), _ptr(wd), _ptr(bg), _ptr(bu), _ptr(bd), _ptr(y),
                                    _ptr(act), _ptr(gate), _ptr(up), tokens, hidden, inter, _dtype_code(x2), _stream(x2)),
              "l32_ffn_forward")
    return y.view(x.shape), gate, up


def block_tail_forward(attn_out, residual, norm_weight, eps, w_gate, w_up, w_down, *, train=False, next_norm_weight=None,
                       next_eps=1e-5):
    """out = attn_out + ff(rmsnorm(attn_out + residual) * norm_weight): the decoder-block tail in one C call
    (reference Model/model.py:270-273), the final add fused into the down-GEMM epilogue.
    train: also return what the backward needs.  next_norm_weight: also return rmsnorm(out) * next_norm_weight -- the next
    block's norm1 / final_norm (Model/model.py:267, :346) -- computed in the same call.
    Returns out, or a dict(out, normed, h, rms, gate, up, next_normed, next_rms) when train or next_norm_weight is given."""
    _check_cuda(attn_out, residual, norm_weight, w_gate, w_up, w_down, next_norm_weight)
    a2, tokens = _flat_tokens(attn_out)
    wg, wu, wd = _weight(w_gate, w_gate.dtype), _weight(w_up, w_up.dtype), _weight(w_down, w_down.dtype)
    hidden, inter = _check_ffn_weights(a2, wg, wu, wd)
    r2 = None if residual is None else residual.contiguous().view(-1, hidden)
    if r2 is not None and r2.shape != a2.shape:
        raise L32Error(f"residual shape {tuple(residual.shape)} != attn_out shape {tuple(attn_out.shape)}")
    w = _weight(norm_weight, a2.dtype)
    nw = None if next_norm_weight is None else _weight(next_norm_weight, a2.dtype)
    new = lambda *shape, dt=a2.dtype: torch.empty(*shape, dtype=dt, device=a2.device)
    out, normed, act = torch.empty_like(a2), torch.empty_like(a2), new(tokens, inter)
    h = torch.empty_like(a2) if (train and r2 is not None) else None
    rms = new(tokens, dt=torch.float32) if train else None
    gate = new(tokens, inter) if train else None
    up = new(tokens, inter) if train else None
    nn = torch.empty_like(a2) if nw is not None else None
    nrms = new(tokens, dt=torch.float32) if (nw is not None and train) else None
    with torch.cuda.device(a2.device):
        check(lib().l32_block_tail_forward_ex(_ptr(a2), _ptr(r2), _ptr(w), float(eps), _ptr(wg), _ptr(wu), _ptr(wd), _ptr(out),
                                              _ptr(normed), _ptr(act), _ptr(h), _ptr(rms), _ptr(gate), _ptr(up), _ptr(nw),
                                              float(next_eps), _ptr(nn), _ptr(nrms), tokens, hidden, inter, _dtype_code(a2),
                                              _stream(a2)), "l32_block_tail_forward_ex")
    if not train and nw is None:
        return out.view(attn_out.shape)
    shp = attn_out.shape
    return dict(out=out.view(shp), normed=normed.view(shp), h=(h.view(shp) if h is not None else (attn_out if train else None)),
                rms=rms, gate=gate, up=up, next_normed=(nn.view(shp) if nn is not None else None), next_rms=nrms)


def linear_lora_forward(x, weight, lora_a, lora_bs, bias=None, x_lora=None):
    """y = x weight^T + bias + (x_lora lora_a^T) lora_bs^T, adapter fused into the base GEMM (lora_bs pre-scaled by
    alpha / rank; x_lora = dropout(x) or None for x).  Returns (y, t [tokens, rank])."""
    _check_cuda(x, weight, lora_a, lora_bs, bias, x_lora)
    x2, tokens = _flat_tokens(x)
    w = _weight(weight, weight.dtype)
    out_f, in_f = w.shape
    la, lb = lora_a.contiguous(), lora_bs.contiguous()
    rank = la.shape[0]
    if (x2.shape[1] != in_f or tuple(la.shape) != (rank, in_f) or tuple(lb.shape) != (out_f, rank) or
            any(t.dtype != x2.dtype for t in (w, la, lb))):
        raise L32Error(f"linear_lora: x[..., {x2.shape[1]}] {x2.dtype}, weight{tuple(w.shape)} {w.dtype}, lora_a{tuple(la.shape)} "
                       f"{la.dtype}, lora_b{tuple(lb.shape)} {lb.dtype}")
    xl = None
    if x_lora is not None:
        xl = x_lora.contiguous().view(-1, in_f)
        if xl.shape != x2.shape or xl.dtype != x2.dtype:
            raise L32Error("linear_lora: x_lora must be shaped and typed like x")
    y = torch.empty(tokens, out_f, dtype=x2.dtype, device=x2.device)
    t = torch.empty(tokens, rank, dtype=x2.dtype, device=x2.device)
    b = None if bias is None else _weight(bias, x2.dtype)
    with torch.cuda.device(x2.device):
        check(lib().l32_linear_lora_forward(_ptr(x2), _ptr(xl), _ptr(w), _ptr(b), _ptr(la), _ptr(lb), _ptr(y), _ptr(t), tokens,
                                            in_f, out_f, rank, _dtype_code(x2), _stream(x2)), "l32_linear_lora_forward")
    return y.view(*x.shape[:-1], out_f), t


def linear_lora_backward(grad_y, x_lora, weight, lora_a, lora_bs, t, *, want_dx=True, want_dlora=True, dx_addend_fn=None):
    """(dx|None, dlora_a|None, dlora_bs|None) for linear_lora_forward with a frozen base weight.
    dx_addend_fn(u) -> [tokens, in]: LoRA dropout -- the caller turns u = dy lora_bs into the masked adapter gradient
    mask * (u lora_a) / (1 - p), which the base GEMM's epilogue adds; None = no dropout (adapter fused as a second phase)."""
    _check_cuda(grad_y, x_lora, weight, lora_a, lora_bs, t)
    w = _weight(weight, weight.dtype)
    out_f, in_f = w.shape
    la, lb = lora_a.contiguous(), lora_bs.contiguous()
    rank = la.shape[0]
    gy = grad_y.contiguous().view(-1, out_f)
    if gy.dtype != w.dtype:
        gy = gy.to(w.dtype)
    tokens = gy.shape[0]
    xl = x_lora.contiguous().view(-1, in_f)
    new = lambda *shape: torch.empty(*shape, dtype=w.dtype, device=w.device)
    u = new(tokens, rank)
    dla = torch.empty_like(la) if want_dlora else None
    dlb = torch.empty_like(lb) if want_dlora else None
    L = lib()
    args = (tokens, in_f, out_f, rank, _dtype_code(gy), _stream(gy))
    with torch.cuda.device(gy.device):
        if dx_addend_fn is None or not want_dx:
            dx = new(tokens, in_f) if want_dx else None
            check(L.l32_linear_lora_backward(_ptr(gy), _ptr(xl), _ptr(w), _ptr(la), _ptr(lb), _ptr(t.contiguous()), None, _ptr(dx),
                                             _ptr(dla), _ptr(dlb), _ptr(u), *args), "l32_linear_lora_backward")
        else:
            # pass 1: u and the adapter gradients; the caller masks u lora_a; pass 2: dx = dy w + addend
            check(L.l32_linear_lora_backward(_ptr(gy), _ptr(xl), _ptr(w), _ptr(la), _ptr(lb), _ptr(t.contiguous()), None, None,
                                             _ptr(dla), _ptr(dlb), _ptr(u), *args), "l32_linear_lora_backward")
            addend = dx_addend_fn(u).contiguous().view(tokens, in_f)
            dx = new(tokens, in_f)
            check(L.l32_linear_lora_backward(_ptr(gy), None, _ptr(w), _ptr(la), _ptr(lb), None, _ptr(addend), _ptr(dx), None, None,
                                             None, *args), "l32_linear_lora_backward")
    return dx, dla, dlb


def ffn_backward(grad_y, x, w_gate, w_up, w_down, gate_cache, up_cache, *, want_dx=True, want_dw_gate_up=True,
                 want_dw_down=True):
    """(dx|None, dw_gate|None, dw_up|None, dw_down|None, d_gate, d_up) for the whole feed-forward."""
    _check_cuda(grad_y, x, w_gate, w_up, w_down, gate_cache, up_cache)
    x2, tokens = _flat_tokens(x)
    wg, wu, wd = _weight(w_gate, w_gate.dtype), _weight(w_up, w_up.dtype), _weight(w_down, w_down.dtype)
    hidden, inter = _check_ffn_weights(x2, wg, wu, wd)
    gy = grad_y.contiguous().view(-1, hidden)
    if gy.dtype != x2.dtype:
        gy = gy.to(x2.dtype)
    dx = torch.empty_like(x2) if want_dx else None
    dwg = torch.empty_like(wg) if want_dw_gate_up else None
    dwu = torch.empty_like(wu) if want_dw_gate_up else None
    dwd = torch.empty_like(wd) if want_dw_down else None
    L = lib()
    ws_bytes = L.l32_ffn_backward_workspace_bytes(tokens, inter)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=x2.device)
    with torch.cuda.device(x2.device):
        check(L.l32_ffn_backward(_ptr(gy), _ptr(x2), _ptr(wg), _ptr(wu), _ptr(wd), _ptr(gate_cache.contiguous()),
                                 _ptr(up_cache.contiguous()), _ptr(dx), _ptr(dwg), _ptr(dwu), _ptr(dwd), _ptr(ws), ws_bytes,
                                 tokens, hidden, inter, _dtype_code(x2), _stream(x2)), "l32_ffn_backward")
    part = ws_bytes // 3
    n = tokens * inter
    d_gate = ws[:n * 2].view(x2.dtype).view(tokens, inter)
    d_up = ws[part:part + n * 2].view(x2.dtype).view(tokens, inter)
    return (dx.view(x.shape) if dx is not None else None), dwg, dwu, dwd, d_gate, d_up


def ffn_lora_forward(x, w_gate, w_up, w_down, lora_a, lora_bs, *, want_cache=False):
    """y = act w_down^T + (act lora_a^T) lora_bs^T with the adapter fused into the down GEMM (lora_bs pre-scaled by
    alpha / rank).  Returns (y, t [tokens, rank], gate_cache|None, up_cache|None)."""
    _check_cuda(x, w_gate, w_up, w_down, lora_a, lora_bs)
    x2, tokens = _flat_tokens(x)
    wg, wu, wd = _weight(w_gate, w_gate.dtype), _weight(w_up, w_up.dtype), _weight(w_down, w_down.dtype)
    hidden, inter = _check_ffn_weights(x2, wg, wu, wd)
    la, lb = lora_a.contiguous(), lora_bs.contiguous()
    rank = la.shape[0]
    if tuple(la.shape) != (rank, inter) or tuple(lb.shape) != (hidden, rank) or la.dtype != x2.dtype or lb.dtype != x2.dtype:
        raise L32Error(f"lora shapes/dtypes: lora_a{tuple(la.shape)} {la.dtype}, lora_b{tuple(lb.shape)} {lb.dtype}")
    y = torch.empty(tokens, hidden, dtype=x2.dtype, device=x2.device)
    act = torch.empty(tokens, inter, dtype=x2.dtype, device=x2.device)
    t = torch.empty(tokens, rank, dtype=x2.dtype, device=x2.device)
    gate = torch.empty_like(act) if want_cache else None
    up = torch.empty_like(act) if want_cache else None
    with torch.cuda.device(x2.device):
        check(lib().l32_ffn_lora_forward(_ptr(x2), _ptr(wg), _ptr(wu), _ptr(wd), _ptr(la), _ptr(lb), _ptr(y), _ptr(act), _ptr(t),
                                         _ptr(gate), _ptr(up), tokens, hidden, inter, rank, _dtype_code(x2), _stream(x2)),
              "l32_ffn_lora_forward")
    return y.view(x.shape), t, gate, up


def ffn_lora_backward(grad_y, x, w_gate, w_up, w_down, lora_a, lora_bs, t, gate_cache, up_cache, *, want_dx=True,
                      want_dw_gate_up=True, want_dlora=True):
    """(dx|None, dw_gate|None, dw_up|None, dlora_a|None, dlora_bs|None) for ffn_lora_forward (frozen w_down)."""
    _check_cuda(grad_y, x, w_gate, w_up, w_down, lora_a, lora_bs, t, gate_cache, up_cache)
    x2, tokens = _flat_tokens(x)
    wg, wu, wd = _weight(w_gate, w_gate.dtype), _weight(w_up, w_up.dtype), _weight(w_down, w_down.dtype)
    hidden, inter = _check_ffn_weights(x2, wg, wu, wd)
    la, lb = lora_a.contiguous(), lora_bs.contiguous()
    rank = la.shape[0]
    gy = grad_y.contiguous().view(-1, hidden)
    if gy.dtype != x2.dtype:
        gy = gy.to(x2.dtype)
    dx = torch.empty_like(x2) if want_dx else None
    dwg = torch.empty_like(wg) if want_dw_gate_up else None
    dwu = torch.empty_like(wu) if want_dw_gate_up else None
    dla = torch.empty_like(la) if want_dlora else None
    dlb = torch.empty_like(lb) if want_dlora else None
    L = lib()
    ws_bytes = L.l32_ffn_lora_backward_workspace_bytes(tokens, inter, rank)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=x2.device)
    with torch.cuda.device(x2.device):
        check(L.l32_ffn_lora_backward(_ptr(gy), _ptr(x2), _ptr(wg), _ptr(wu), _ptr(wd), _ptr(la), _ptr(lb), _ptr(t.contiguous()),
                                      _ptr(gate_cache.contiguous()), _ptr(up_cache.contiguous()), _ptr(dx), _ptr(dwg), _ptr(dwu),
                                      _ptr(dla), _ptr(dlb), _ptr(ws), ws_bytes, tokens, hidden, inter, rank, _dtype_code(x2),
                                      _stream(x2)), "l32_ffn_lora_backward")
    return (dx.view(x.shape) if dx is not None else None), dwg, dwu, dla, dlb


# --------------------------------------------------------------------------------------------- attention
def rope_kv_append(q, k_new, v_new, position_ids, cache_k, cache_v, past_len, rope_base=500000.0):
    """RoPE on q [b, t, heads*d] IN PLACE and on k_new while it is stored into cache_k [b, kv_heads, max_len, d] at
    past_len; v_new stored next to it.  position_ids [b, t] int64."""
    _check_cuda(q, k_new, v_new, position_ids, cache_k, cache_v)
    b, t = q.shape[0], q.shape[1]
    _, kvh, max_len, d = cache_k.shape
    heads = q.shape[-1] // d
    for ten in (q, k_new, v_new, cache_k, cache_v):
        if not ten.is_contiguous():
            raise L32Error("rope_kv_append: tensors must be contiguous")
    pos = position_ids.contiguous()
    if pos.dtype != torch.int64 or pos.numel() != b * t:
        raise L32Error("rope_kv_append: position_ids must be int64 [batch, q_len]")
    with torch.cuda.device(q.device):
        check(lib().l32_rope_kv_append(_ptr(q), _ptr(k_new), _ptr(v_new), _ptr(pos), _ptr(cache_k), _ptr(cache_v), b, t, heads, kvh,
                                       d, max_len, int(past_len), float(rope_base), _dtype_code(q), _stream(q)),
              "l32_rope_kv_append")


def gqa_attention_forward(q, cache_k, cache_v, kv_len, past_len, *, causal=True, key_keep=None):
    """ctx [b, t, heads*d] = softmax(q k^T / sqrt(d) + mask) v over cache[:, :, :kv_len]; q [b, t, heads*d] (RoPE applied)."""
    _check_cuda(q, cache_k, cache_v, key_keep)
    b, t = q.shape[0], q.shape[1]
    _, kvh, max_len, d = cache_k.shape
    heads = q.shape[-1] // d
    qc = q.contiguous()
    keep = None
    if key_keep is not None:
        keep = key_keep.to(torch.uint8).contiguous()
        if tuple(keep.shape) != (b, kv_len):
            raise L32Error(f"key_keep must be [batch, kv_len] = {(b, kv_len)}, got {tuple(keep.shape)}")
    ctx = torch.empty_like(qc)
    L = lib()
    ws_bytes = L.l32_gqa_attention_workspace_bytes(b, t, heads, kvh, d, int(kv_len)) if keep is None else 0
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=q.device) if ws_bytes else None
    with torch.cuda.device(q.device):
        check(L.l32_gqa_attention_forward(_ptr(qc), _ptr(cache_k), _ptr(cache_v), _ptr(keep), _ptr(ctx), _ptr(ws), ws_bytes, b, t,
                                          heads, kvh, d, max_len, int(kv_len), int(past_len), int(bool(causal)), _dtype_code(qc),
                                          _stream(qc)), "l32_gqa_attention_forward")
    return ctx


def _paged_args(q, pool_k, pool_v, block_table, past_lens, new_lens, what):
    """Shapes of a paged-cache call, checked: (b, t, heads, kv_heads, d, num_pages, max_pages_per_seq)."""
    b, t = q.shape[0], q.shape[1]
    num_pages, kvh, page, d = pool_k.shape
    if page != KV_PAGE or tuple(pool_v.shape) != tuple(pool_k.shape) or pool_v.dtype != pool_k.dtype:
        raise L32Error(f"{what}: pools must both be [num_pages, kv_heads, {KV_PAGE}, head_dim], got {tuple(pool_k.shape)} / "
                       f"{tuple(pool_v.shape)}")
    if q.dim() != 3 or q.shape[-1] % d != 0 or q.dtype != pool_k.dtype:
        raise L32Error(f"{what}: q must be [batch, q_len, heads * {d}] {pool_k.dtype}, got {tuple(q.shape)} {q.dtype}")
    for ten in (q, pool_k, pool_v, block_table, past_lens, new_lens):
        if ten is not None and not ten.is_contiguous():
            raise L32Error(f"{what}: tensors must be contiguous")
    for name, ten in (("block_table", block_table), ("past_lens", past_lens), ("new_lens", new_lens)):
        if ten is not None and ten.dtype != torch.int32:
            raise L32Error(f"{what}: {name} must be int32")
    if block_table.dim() != 2 or block_table.shape[0] < b or past_lens.numel() < b or (new_lens is not None and new_lens.numel() < b):
        raise L32Error(f"{what}: block_table [>= {b}, max_pages], past_lens / new_lens [>= {b}] expected")
    return b, t, q.shape[-1] // d, kvh, d, num_pages, block_table.shape[1]


def rope_kv_append_paged(q, k_new, v_new, position_ids, pool_k, pool_v, block_table, past_lens, new_lens=None, rope_base=500000.0):
    """RoPE on q [b, t, heads*d] IN PLACE and on k_new while it is stored into the paged pool_k [num_pages, kv_heads, 64, d]:
    token i of sequence b goes to position past_lens[b] + i, row pos % 64 of page block_table[b][pos // 64]; v_new is stored
    next to it.  Tokens i >= new_lens[b] write nothing.  block_table int32 [>= b, max_pages], past_lens / new_lens int32
    [>= b] in device memory: their values are trusted (PagedKVCache checks them when it builds them)."""
    _check_cuda(q, k_new, v_new, position_ids, pool_k, pool_v, block_table, past_lens, new_lens)
    b, t, heads, kvh, d, num_pages, max_pages = _paged_args(q, pool_k, pool_v, block_table, past_lens, new_lens,
                                                            "rope_kv_append_paged")
    for ten in (k_new, v_new):
        if not ten.is_contiguous() or ten.shape[:2] != q.shape[:2] or ten.shape[-1] != kvh * d:
            raise L32Error(f"rope_kv_append_paged: k_new / v_new must be contiguous [{b}, {t}, {kvh * d}]")
    pos = position_ids.contiguous()
    if pos.dtype != torch.int64 or pos.numel() != b * t:
        raise L32Error("rope_kv_append_paged: position_ids must be int64 [batch, q_len]")
    with torch.cuda.device(q.device):
        check(lib().l32_rope_kv_append_paged(_ptr(q), _ptr(k_new), _ptr(v_new), _ptr(pos), _ptr(pool_k), _ptr(pool_v),
                                             _ptr(block_table), _ptr(past_lens), _ptr(new_lens), b, t, heads, kvh, d, num_pages,
                                             max_pages, float(rope_base), _dtype_code(q), _stream(q)),
              "l32_rope_kv_append_paged")


def gqa_attention_forward_paged(q, pool_k, pool_v, block_table, past_lens, new_lens=None, *, max_kv_len=None):
    """ctx [b, t, heads*d]: causal attention of each sequence's queries (positions past_lens[b] + i, RoPE applied) over its own
    keys [0, past_lens[b] + new_lens[b]) in the paged pools; padded query rows (i >= new_lens[b]) give zeros.  max_kv_len: a
    bound on every sequence's length that sizes the split-KV plan (default: the table's capacity, max_pages * 64)."""
    _check_cuda(q, pool_k, pool_v, block_table, past_lens, new_lens)
    b, t, heads, kvh, d, num_pages, max_pages = _paged_args(q, pool_k, pool_v, block_table, past_lens, new_lens,
                                                            "gqa_attention_forward_paged")
    max_kv_len = max_pages * KV_PAGE if max_kv_len is None else int(max_kv_len)
    ctx = torch.empty_like(q)
    L = lib()
    ws_bytes = L.l32_gqa_attention_workspace_bytes(b, t, heads, kvh, d, max_kv_len)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=q.device) if ws_bytes else None
    with torch.cuda.device(q.device):
        check(L.l32_gqa_attention_forward_paged(_ptr(q), _ptr(pool_k), _ptr(pool_v), _ptr(block_table), _ptr(past_lens),
                                                _ptr(new_lens), _ptr(ctx), _ptr(ws), ws_bytes, b, t, heads, kvh, d, num_pages,
                                                max_pages, max_kv_len, _dtype_code(q), _stream(q)),
              "l32_gqa_attention_forward_paged")
    return ctx


def _attention_train_args(q_rot, cache_k, cache_v, key_keep):
    """Shapes of a training call (keys = queries, no past) and the key_keep bytes, checked as gqa_attention_forward does."""
    b, t = q_rot.shape[0], q_rot.shape[1]
    _, kvh, max_len, d = cache_k.shape
    heads = q_rot.shape[-1] // d
    for ten in (cache_k, cache_v):
        if not ten.is_contiguous():
            raise L32Error("attention: cache_k / cache_v must be contiguous")
    keep = None
    if key_keep is not None:
        keep = key_keep.to(torch.uint8).contiguous()
        if tuple(keep.shape) != (b, t):
            raise L32Error(f"key_keep must be [batch, kv_len] = {(b, t)}, got {tuple(keep.shape)}")
    return b, t, heads, kvh, d, max_len, keep


def gqa_attention_forward_train(q_rot, cache_k, cache_v, causal=True, key_keep=None):
    """Training forward over keys [0, t) of the K / V buffers: (ctx [b, t, heads*d], lse [b, heads, t] fp32, log2 domain, +inf
    for a row that sees no key).  q_rot [b, t, heads*d] with RoPE applied."""
    _check_cuda(q_rot, cache_k, cache_v, key_keep)
    b, t, heads, kvh, d, max_len, keep = _attention_train_args(q_rot, cache_k, cache_v, key_keep)
    qc = q_rot.contiguous()
    ctx = torch.empty_like(qc)
    lse = torch.empty(b, heads, t, dtype=torch.float32, device=q_rot.device)
    with torch.cuda.device(q_rot.device):
        check(lib().l32_gqa_attention_forward_train(_ptr(qc), _ptr(cache_k), _ptr(cache_v), _ptr(keep), _ptr(ctx), _ptr(lse), b, t,
                                                    heads, kvh, d, max_len, int(bool(causal)), _dtype_code(qc), _stream(qc)),
              "l32_gqa_attention_forward_train")
    return ctx, lse


def gqa_attention_backward(d_ctx, q_rot, cache_k, cache_v, ctx, lse, position_ids, causal=True, key_keep=None, rope_base=500000.0):
    """Gradients of gqa_attention_forward_train with respect to the PRE-RoPE q [b, t, heads*d], k and v [b, t, kv_heads*d]:
    (dq, dk, dv).  position_ids [b, t] int64: the positions RoPE was applied at."""
    _check_cuda(d_ctx, q_rot, cache_k, cache_v, ctx, lse, position_ids, key_keep)
    b, t, heads, kvh, d, max_len, keep = _attention_train_args(q_rot, cache_k, cache_v, key_keep)
    qc, gc, oc = q_rot.contiguous(), d_ctx.contiguous(), ctx.contiguous()
    if gc.dtype != qc.dtype:
        gc = gc.to(qc.dtype)
    pos = position_ids.contiguous()
    if pos.dtype != torch.int64 or pos.numel() != b * t:
        raise L32Error("gqa_attention_backward: position_ids must be int64 [batch, q_len]")
    if lse.dtype != torch.float32 or lse.numel() != b * heads * t:
        raise L32Error("gqa_attention_backward: lse must be the fp32 [batch, heads, q_len] of gqa_attention_forward_train")
    lse = lse.contiguous()
    dq = torch.empty_like(qc)
    dk = torch.empty(b, t, kvh * d, dtype=qc.dtype, device=qc.device)
    dv = torch.empty_like(dk)
    L = lib()
    ws_bytes = L.l32_gqa_attention_backward_workspace_bytes(b, t, heads)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=qc.device)
    with torch.cuda.device(qc.device):
        check(L.l32_gqa_attention_backward(_ptr(gc), _ptr(qc), _ptr(cache_k), _ptr(cache_v), _ptr(oc), _ptr(lse), _ptr(keep), _ptr(pos),
                                           _ptr(dq), _ptr(dk), _ptr(dv), _ptr(ws), ws_bytes, b, t, heads, kvh, d, max_len,
                                           int(bool(causal)), float(rope_base), _dtype_code(qc), _stream(qc)),
              "l32_gqa_attention_backward")
    return dq, dk, dv


# --------------------------------------------------------------------------------------------- lm_head + cross entropy
def lm_head_ce_forward(hidden_states, weight, labels_shifted, ignore_index=-100):
    """logits = hidden_states weight^T and the mean cross entropy against `labels_shifted` (int64, one per token row, already
    shifted; ignore_index rows do not count) in one GEMM + two tiny reductions.
    Returns dict(logits [.., vocab], loss (0-dim fp32), lse [tokens], loss_rows [tokens], loss_and_count [2])."""
    _check_cuda(hidden_states, weight, labels_shifted)
    h2, tokens = _flat_tokens(hidden_states)
    w = _weight(weight, weight.dtype)
    vocab, hidden = w.shape
    if h2.shape[1] != hidden or w.dtype != h2.dtype:
        raise L32Error(f"lm_head: hidden_states[..., {h2.shape[1]}] {h2.dtype} vs weight{tuple(w.shape)} {w.dtype}")
    lab = labels_shifted.contiguous().view(-1)
    if lab.dtype != torch.int64 or lab.numel() != tokens:
        raise L32Error(f"lm_head: labels must be int64 with one entry per token row ({lab.dtype}, {lab.numel()} vs {tokens})")
    dev = h2.device
    logits = torch.empty(tokens, vocab, dtype=h2.dtype, device=dev)
    lse = torch.empty(tokens, dtype=torch.float32, device=dev)
    loss_rows = torch.empty(tokens, dtype=torch.float32, device=dev)
    lc = torch.empty(2, dtype=torch.float32, device=dev)
    L = lib()
    ws_bytes = L.l32_lm_head_ce_workspace_bytes(tokens, vocab)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(L.l32_lm_head_ce_forward(_ptr(h2), _ptr(w), _ptr(lab), int(ignore_index), _ptr(logits), _ptr(lse), _ptr(loss_rows),
                                       _ptr(lc), _ptr(ws), ws_bytes, tokens, hidden, vocab, _dtype_code(h2), _stream(h2)),
              "l32_lm_head_ce_forward")
    return dict(logits=logits.view(*hidden_states.shape[:-1], vocab), loss=lc[0], lse=lse, loss_rows=loss_rows, loss_and_count=lc)


def lm_head_ce_backward(logits, lse, labels_shifted, ignore_index, loss_and_count, grad_loss, hidden_states, weight, *,
                        want_dhidden=True, want_dweight=True, in_place=False):
    """(d_hidden|None, d_weight|None, dlogits) of the mean cross entropy scaled by `grad_loss` (fp32 device scalar or None)."""
    _check_cuda(logits, lse, labels_shifted, hidden_states, weight)
    h2, tokens = _flat_tokens(hidden_states)
    w = _weight(weight, weight.dtype)
    vocab, hidden = w.shape
    lg = logits.contiguous().view(tokens, vocab)
    lab = labels_shifted.contiguous().view(-1)
    dlogits = lg if in_place else torch.empty_like(lg)
    dh = torch.empty_like(h2) if want_dhidden else None
    dw = torch.empty_like(w) if want_dweight else None
    gl = None
    if grad_loss is not None:
        gl = grad_loss.detach().to(device=h2.device, dtype=torch.float32).reshape(1).contiguous()
    with torch.cuda.device(h2.device):
        check(lib().l32_lm_head_ce_backward(_ptr(lg), _ptr(lse), _ptr(lab), int(ignore_index), _ptr(loss_and_count), _ptr(gl),
                                            _ptr(h2), _ptr(w), _ptr(dlogits), _ptr(dh), _ptr(dw), tokens, hidden, vocab,
                                            _dtype_code(h2), _stream(h2)), "l32_lm_head_ce_backward")
    return (dh.view(hidden_states.shape) if dh is not None else None), dw, dlogits


def gemm(a, b, *, a_mn_major=False, b_mn_major=False, a1=None, b1=None, cta_group=0, max_ctas=0):
    """D[m,n] = A B^T (+ A1 B1^T).  K-major operand: tensor [rows, k]; MN-major operand: tensor [k, rows]."""
    _check_cuda(a, b, a1, b1)
    m, k = (a.shape[1], a.shape[0]) if a_mn_major else (a.shape[0], a.shape[1])
    n, kb = (b.shape[1], b.shape[0]) if b_mn_major else (b.shape[0], b.shape[1])
    if k != kb:
        raise L32Error(f"gemm: reduction lengths differ ({k} vs {kb})")
    k1 = 0
    if a1 is not None:
        k1 = a1.shape[0] if a_mn_major else a1.shape[1]
    for t in (a, b, a1, b1):
        if t is not None and (t.stride(-1) != 1 or t.dtype != a.dtype):
            raise L32Error("gemm operands must share a dtype and be contiguous along the last dimension")
    d = torch.empty(m, n, dtype=a.dtype, device=a.device)
    with torch.cuda.device(a.device):
        check(lib().l32_gemm(_ptr(a), a.stride(0), int(a_mn_major), _ptr(b), b.stride(0), int(b_mn_major), _ptr(a1),
                             0 if a1 is None else a1.stride(0), _ptr(b1), 0 if b1 is None else b1.stride(0), _ptr(d), n,
                             m, n, k, k1, _dtype_code(a), cta_group, max_ctas, _stream(a)), "l32_gemm")
    return d


def swiglu_act(gate, up):
    """Unfused act = silu(gate) * up (benchmark reference point for the fusion saving)."""
    _check_cuda(gate, up)
    g, u = gate.contiguous(), up.contiguous()
    act = torch.empty_like(g)
    with torch.cuda.device(g.device):
        check(lib().l32_swiglu_act(_ptr(g), _ptr(u), _ptr(act), g.numel(), _dtype_code(g), _stream(g)), "l32_swiglu_act")
    return act


# --------------------------------------------------------------------------------------------- tensor parallel
def _ptr_array(ptrs):
    import ctypes
    arr = (ctypes.c_void_p * len(ptrs))(*[int(p) for p in ptrs])
    return arr


def tp_signal(peer_flag_ptrs, index, value, device, zero8=None):
    """flag[index] := value on every rank (host list of `world` device pointers to each rank's uint32 flag array);
    optionally clears 8 uint32 counters (`zero8`) in the same kernel."""
    arr = _ptr_array(peer_flag_ptrs)
    with torch.cuda.device(device):
        check(lib().l32_tp_signal(arr, len(peer_flag_ptrs), int(index), int(value), _ptr(zero8),
                                  torch.cuda.current_stream(device).cuda_stream), "l32_tp_signal")


def tp_swiglu_forward_allgather(x_full, peer_x_ptrs, ready, done, epoch, rank, rows_per_rank, w_gate, w_up, out=None,
                                want_cache=False):
    """Fused all-gather (pulled over NVLink inside the GEMM) + gate/up projection + SiLU*mul on this rank's shard.
    x_full may be the published buffer itself (gather in place) or a fresh [tokens, hidden] tensor (own rows copied too).
    Returns act, or (act, gate_cache, up_cache) with want_cache."""
    _check_cuda(x_full, ready, done, w_gate, w_up)
    tokens, hidden = x_full.shape
    inter = w_gate.shape[0]
    act = out if out is not None else torch.empty(tokens, inter, dtype=x_full.dtype, device=x_full.device)
    gate = torch.empty_like(act) if want_cache else None
    up = torch.empty_like(act) if want_cache else None
    world = len(peer_x_ptrs)
    arr = _ptr_array(peer_x_ptrs)
    with torch.cuda.device(x_full.device):
        check(lib().l32_tp_swiglu_forward_allgather(_ptr(x_full), arr, _ptr(ready), _ptr(done), int(epoch), int(rank), world,
                                                    int(rows_per_rank), _ptr(w_gate), _ptr(w_up), None, None, _ptr(act),
                                                    _ptr(gate), _ptr(up), tokens, hidden, inter, _dtype_code(x_full),
                                                    _stream(x_full)),
              "l32_tp_swiglu_forward_allgather")
    return (act, gate, up) if want_cache else act


def tp_ffn_backward_dact_allgather(dy_full, peer_dy_ptrs, ready, done, epoch, rank, rows_per_rank, w_down, gate_cache,
                                   up_cache, want_act=True):
    """Fused all-gather of dY (pulled inside the GEMM) + d_act = dY w_down_shard + SiLU' epilogue.
    Returns (d_gate, d_up, act|None), all [tokens, inter_local]."""
    _check_cuda(dy_full, ready, done, w_down, gate_cache, up_cache)
    tokens, hidden = dy_full.shape
    inter = w_down.shape[1]
    d_gate = torch.empty(tokens, inter, dtype=dy_full.dtype, device=dy_full.device)
    d_up = torch.empty_like(d_gate)
    act = torch.empty_like(d_gate) if want_act else None
    arr = _ptr_array(peer_dy_ptrs)
    with torch.cuda.device(dy_full.device):
        check(lib().l32_tp_ffn_backward_dact_allgather(_ptr(dy_full), arr, _ptr(ready), _ptr(done), int(epoch), int(rank),
                                                       len(peer_dy_ptrs), int(rows_per_rank), _ptr(w_down), _ptr(gate_cache),
                                                       _ptr(up_cache), _ptr(d_gate), _ptr(d_up), _ptr(act), tokens, hidden,
                                                       inter, _dtype_code(dy_full), _stream(dy_full)),
              "l32_tp_ffn_backward_dact_allgather")
    return d_gate, d_up, act


def tp_ffn_backward_dx_reduce_scatter(d_gate, d_up, w_gate, w_up, peer_slot_ptrs, rank, rows_per_rank):
    """Partial dX = d_gate w_gate_shard + d_up w_up_shard (two-phase GEMM) + reduce-scatter pushed from the epilogue."""
    _check_cuda(d_gate, d_up, w_gate, w_up)
    tokens, inter = d_gate.shape
    hidden = w_gate.shape[1]
    arr = _ptr_array(peer_slot_ptrs)
    with torch.cuda.device(d_gate.device):
        check(lib().l32_tp_ffn_backward_dx_reduce_scatter(_ptr(d_gate), _ptr(d_up), _ptr(w_gate), _ptr(w_up), arr, int(rank),
                                                          len(peer_slot_ptrs), int(rows_per_rank), tokens, hidden, inter,
                                                          _dtype_code(d_gate), _stream(d_gate)),
              "l32_tp_ffn_backward_dx_reduce_scatter")


def tp_linear_forward_reduce_scatter(a, weight, peer_slot_ptrs, rank, rows_per_rank):
    """Fused down projection + reduce-scatter: every output row is stored into its owner's slot for this rank."""
    _check_cuda(a, weight)
    tokens, in_f = a.shape
    out_f = weight.shape[0]
    arr = _ptr_array(peer_slot_ptrs)
    with torch.cuda.device(a.device):
        check(lib().l32_tp_linear_forward_reduce_scatter(_ptr(a), _ptr(weight), arr, int(rank), len(peer_slot_ptrs),
                                                         int(rows_per_rank), tokens, in_f, out_f, _dtype_code(a), _stream(a)),
              "l32_tp_linear_forward_reduce_scatter")


def tp_ffn_forward_fused(x_full, peer_x_ptrs, ready, done, epoch, rank, rows_per_rank, w_gate, w_up, w_down, peer_slot_ptrs,
                         act=None, act_done=None):
    """Gate/up (+ pulled all-gather) and down (+ pushed reduce-scatter) of this rank's shard in ONE persistent kernel."""
    _check_cuda(x_full, ready, done, w_gate, w_up, w_down)
    tokens, hidden = x_full.shape
    inter = w_gate.shape[0]
    if act is None:
        act = torch.empty(tokens, inter, dtype=x_full.dtype, device=x_full.device)
    if act_done is None:
        act_done = torch.empty((tokens + 255) // 256, dtype=torch.int32, device=x_full.device)
    world = len(peer_x_ptrs)
    px, ps = _ptr_array(peer_x_ptrs), _ptr_array(peer_slot_ptrs)
    with torch.cuda.device(x_full.device):
        check(lib().l32_tp_ffn_forward_fused(_ptr(x_full), px, _ptr(ready), _ptr(done), int(epoch), int(rank), world,
                                             int(rows_per_rank), _ptr(w_gate), _ptr(w_up), _ptr(w_down), _ptr(act),
                                             _ptr(act_done), ps, tokens, hidden, inter, _dtype_code(x_full), _stream(x_full)),
              "l32_tp_ffn_forward_fused")
    return act


def tp_reduce_partials(slots, flags, epoch, rank, rows, addend=None, out=None):
    """y = sum over ranks of the partial slots [world, slot_rows, hidden] (+ addend), after every peer signalled."""
    _check_cuda(slots, flags, addend)
    world, slot_rows, hidden = slots.shape
    y = out if out is not None else torch.empty(rows, hidden, dtype=slots.dtype, device=slots.device)
    with torch.cuda.device(slots.device):
        check(lib().l32_tp_reduce_partials(_ptr(slots), _ptr(flags), int(epoch), world, int(rank), _ptr(addend), _ptr(y),
                                           int(rows), slot_rows, hidden, _dtype_code(slots), _stream(slots)),
              "l32_tp_reduce_partials")
    return y


def tp_linear_group_forward_allgather(x_full, peer_x_ptrs, ready, done, epoch, rank, rows_per_rank, weights):
    """[x_full w^T for w in weights] (1..3 K-major [out_i, hidden] weights, e.g. the q / k / v rows of a rank's heads) in one
    persistent launch with the all-gather of x_full pulled in, as in tp_swiglu_forward_allgather."""
    _check_cuda(x_full, ready, done, *weights)
    if not 1 <= len(weights) <= 3:
        raise L32Error("tp_linear_group_forward_allgather takes one to three weights")
    tokens, hidden = x_full.shape
    for w in weights:
        if w.dim() != 2 or w.shape[1] != hidden or not w.is_contiguous() or w.dtype != x_full.dtype:
            raise L32Error(f"tp linear group: x_full[..., {hidden}] {x_full.dtype} vs weight{tuple(w.shape)} {w.dtype}")
    ys = [torch.empty(tokens, w.shape[0], dtype=x_full.dtype, device=x_full.device) for w in weights]
    n = len(weights)
    w_arr = (ctypes.c_void_p * n)(*[_ptr(w) for w in weights])
    y_arr = (ctypes.c_void_p * n)(*[_ptr(y) for y in ys])
    o_arr = (ctypes.c_int * n)(*[w.shape[0] for w in weights])
    with torch.cuda.device(x_full.device):
        check(lib().l32_tp_linear_group_forward_allgather(_ptr(x_full), _ptr_array(peer_x_ptrs), _ptr(ready), _ptr(done), int(epoch),
                                                          int(rank), len(peer_x_ptrs), int(rows_per_rank), w_arr, y_arr, o_arr, n,
                                                          tokens, hidden, _dtype_code(x_full), _stream(x_full)),
              "l32_tp_linear_group_forward_allgather")
    return ys


def tp_linear_forward_allgather(a_full, peer_a_ptrs, ready, done, epoch, rank, rows_per_rank, weight, w_mn_major=False):
    """y = a_full W with the all-gather of a_full pulled in.  weight [out, in] (w_mn_major=False, y = a w^T) or [in, out]
    (w_mn_major=True, y = a w: e.g. the out_proj shard [hidden, heads_local*d] in the backward)."""
    _check_cuda(a_full, ready, done, weight)
    tokens, in_f = a_full.shape
    out_f = weight.shape[1] if w_mn_major else weight.shape[0]
    if (weight.shape[0] if w_mn_major else weight.shape[1]) != in_f or not weight.is_contiguous() or weight.dtype != a_full.dtype:
        raise L32Error(f"tp linear: a_full[..., {in_f}] {a_full.dtype} vs weight{tuple(weight.shape)} {weight.dtype}")
    y = torch.empty(tokens, out_f, dtype=a_full.dtype, device=a_full.device)
    with torch.cuda.device(a_full.device):
        check(lib().l32_tp_linear_forward_allgather(_ptr(a_full), _ptr_array(peer_a_ptrs), _ptr(ready), _ptr(done), int(epoch),
                                                    int(rank), len(peer_a_ptrs), int(rows_per_rank), _ptr(weight), int(bool(w_mn_major)),
                                                    _ptr(y), tokens, in_f, out_f, _dtype_code(a_full), _stream(a_full)),
              "l32_tp_linear_forward_allgather")
    return y


def tp_linear_group_backward_dx_reduce_scatter(dys, weights, peer_slot_ptrs, rank, rows_per_rank):
    """Partial dX = sum_i dys[i] weights[i] (dys[i] [tokens, k_i], weights[i] [k_i, hidden]; one GEMM of up to three
    accumulation phases) with every row pushed into its owner's slot, as in tp_ffn_backward_dx_reduce_scatter."""
    _check_cuda(*dys, *weights)
    n = len(dys)
    if not 1 <= n <= 3 or len(weights) != n:
        raise L32Error("tp_linear_group_backward_dx_reduce_scatter takes one to three (dy, weight) pairs")
    tokens = dys[0].shape[0]
    hidden = weights[0].shape[1]
    for dy, w in zip(dys, weights):
        if (dy.dim() != 2 or dy.shape[0] != tokens or w.shape != (dy.shape[1], hidden) or not dy.is_contiguous() or
                not w.is_contiguous() or dy.dtype != w.dtype or dy.dtype != dys[0].dtype):
            raise L32Error(f"tp dx: dy{tuple(dy.shape)} {dy.dtype} vs weight{tuple(w.shape)} {w.dtype}")
    dy_arr = (ctypes.c_void_p * n)(*[_ptr(t) for t in dys])
    w_arr = (ctypes.c_void_p * n)(*[_ptr(w) for w in weights])
    k_arr = (ctypes.c_int * n)(*[dy.shape[1] for dy in dys])
    with torch.cuda.device(dys[0].device):
        check(lib().l32_tp_linear_group_backward_dx_reduce_scatter(dy_arr, w_arr, k_arr, n, _ptr_array(peer_slot_ptrs), int(rank),
                                                                   len(peer_slot_ptrs), int(rows_per_rank), tokens, hidden,
                                                                   _dtype_code(dys[0]), _stream(dys[0])),
              "l32_tp_linear_group_backward_dx_reduce_scatter")
