"""Host-side mirror of the reference's operator interface for the decoder-block hot path.

Same class names, constructor arguments, attribute names and state_dict keys as the reference:
  LLAMARMSNorm / RMSNormFunction            reference Model/model.py:135-171
  SwiGLUFunction / FusedSwiGLU              reference Tools/swiglu/FusedSwiglu.py:14-91
  FusedFeedforward (+ FusedFeedForward)     reference Model/model.py:210-217, Tools/swiglu/FusedSwiglu.py:94-131
  Linear_LORA                               reference Model/model.py:107-121
  convert_feedforward_to_fused              reference Tools/swiglu/FusedSwiglu.py:134-166

Dispatch follows the reference's gate (Model/model.py:165): CUDA tensors of a 16-bit float type run the
sm_100a kernels through the C-ABI; everything else (fp32, CPU) evaluates the reference's own PyTorch
expressions, which is what the reference does for those inputs.  The autograd wrappers are the *fixed*
versions described in SURVEY.md section 8(b): they save what backward needs, honour needs_input_grad,
never return a gradient for a None input and never mutate caller tensors.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops

__all__ = [
    "RMSNormFunction", "LLAMARMSNorm", "SwiGLUFunction", "FusedSwiGLU", "LinearFunction", "Linear_LORA", "FFNFunction", "FFNLoRAFunction",
    "FusedFeedforward", "FusedFeedForward", "convert_feedforward_to_fused", "patch_reference", "convert_instances", "block_tail",
    "BlockTailFunction", "LinearLoRAFunction", "chain_block_norms", "LMHeadCEFunction", "lm_head_loss", "shift_labels", "GroupQueryAttention", "KVCache",
    "GQAAttentionFunction", "PagedKVCache",
]


def _dims8(*dims) -> bool:
    """The tcgen05 / TMA kernels want every matrix dimension to be a multiple of 8 elements (16-byte rows).  Shapes that are
    not take the reference's own F.linear expressions, which accept anything (the reference's live path does too)."""
    return all(int(d) % 8 == 0 and int(d) > 0 for d in dims)


def _wants_grad(*tensors) -> bool:
    """True when autograd will record this call.  Function.forward always runs with grad mode off and
    ctx.needs_input_grad ignores an enclosing torch.no_grad(), so the decision is taken in `apply`."""
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


# ------------------------------------------------------------------------------------------------ RMSNorm
class RMSNormFunction(torch.autograd.Function):
    """y = rmsnorm(x + residual) * weight on the sm_100a kernels (reference Model/model.py:135-155)."""

    @classmethod
    def apply(cls, x, weight, eps, residual=None):
        if not _wants_grad(x, weight, residual):
            # inference: 3 streams (x, residual, y) -- no h, no rms
            return ops.add_rmsnorm_forward(x, weight, residual, eps, want_h=False, want_rms=False)[0]
        return super().apply(x, weight, eps, residual)

    @staticmethod
    def forward(ctx, x, weight, eps, residual=None):
        y, rms, h = ops.add_rmsnorm_forward(x, weight, residual, eps, want_h=True, want_rms=True)
        # without a residual the normalised input is x itself: nothing extra is written
        ctx.save_for_backward(h if h is not None else x, weight, rms)
        ctx.has_residual = residual is not None
        return y

    @staticmethod
    def backward(ctx, grad_output):
        h, weight, rms = ctx.saved_tensors
        dx, dw = ops.rmsnorm_backward(grad_output, h, weight, rms, want_dweight=ctx.needs_input_grad[1])
        if dw is not None and dw.dtype != weight.dtype:
            dw = dw.to(weight.dtype)
        d_res = dx if (ctx.has_residual and ctx.needs_input_grad[3]) else None
        return (dx if ctx.needs_input_grad[0] else None), dw, None, d_res


class LLAMARMSNorm(nn.Module):
    """Drop-in for reference Model/model.py:158-171 (same ctor, `.weight`, forward(x, residual=None))."""

    def __init__(self, dim: int, eps: float = 1e-6):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(dim))

    def forward(self, x, residual=None):
        if residual is None:
            # the previous block's tail may already have normalised this very tensor with this very module
            # (block_tail(..., next_norm=self) attaches the result): nothing left to do
            pre = getattr(x, "_l32_prenormed", None)
            if pre is not None and pre[0] is self and pre[2] == x._version:   # ... and nobody has written to x since
                return pre[1]
        if ops.supported(x):
            return RMSNormFunction.apply(x, self.weight, self.eps, residual)
        # reference semantics for fp32 / CPU inputs (Model/model.py:166-171)
        if residual is not None:
            x = x + residual
        variance = x.pow(2).mean(-1, keepdim=True)
        x = x * torch.rsqrt(variance + self.eps)
        return x * self.weight


# ------------------------------------------------------------------------------------------------ SwiGLU
def _silu_bwd(d_act, gate, up):
    s = torch.sigmoid(gate)
    return d_act * up * (s * (1 + gate * (1 - s))), d_act * (gate * s)


class SwiGLUFunction(torch.autograd.Function):
    """act = silu(x w_gate^T + b_gate) * (x w_up^T + b_up) (reference Tools/swiglu/FusedSwiglu.py:14-40).

    Differentiable on every path (the reference's fallback branch saved nothing and its CUDA backward was
    never defined); bias gradients are returned when biases exist.
    """

    @staticmethod
    def _cuda_path(x, w_gate, w_up):
        # sm_100a kernels only when activations AND weights share a 16-bit CUDA dtype; anything else (fp32 master weights
        # under bf16 activations, CPU, fp32) evaluates the reference's F.linear expressions (FusedSwiglu.py:17-20)
        return (ops.supported(x) and w_gate.dtype == x.dtype and w_up.dtype == x.dtype and w_gate.is_cuda and w_up.is_cuda and
                _dims8(*w_gate.shape))

    @classmethod
    def apply(cls, x, w_gate, w_up, b_gate=None, b_up=None):
        if cls._cuda_path(x, w_gate, w_up) and not _wants_grad(x, w_gate, w_up, b_gate, b_up):
            return ops.swiglu_forward(x, w_gate, w_up, b_gate, b_up, want_cache=False)[0]
        return super().apply(x, w_gate, w_up, b_gate, b_up)

    @staticmethod
    def forward(ctx, x, w_gate, w_up, b_gate=None, b_up=None):
        need_grad = any(ctx.needs_input_grad)
        ctx.cuda_path = SwiGLUFunction._cuda_path(x, w_gate, w_up)
        if not ctx.cuda_path:
            gate = F.linear(x, w_gate, b_gate)
            up = F.linear(x, w_up, b_up)
            if need_grad:
                ctx.save_for_backward(x, w_gate, w_up, gate, up)
            return F.silu(gate) * up
        act, gate, up = ops.swiglu_forward(x, w_gate, w_up, b_gate, b_up, want_cache=need_grad)
        if need_grad:
            ctx.save_for_backward(x, w_gate, w_up, gate, up)
        return act

    @staticmethod
    def backward(ctx, grad_output):
        x, w_gate, w_up, gate, up = ctx.saved_tensors
        nx, ng, nu, nbg, nbu = ctx.needs_input_grad
        if not ctx.cuda_path:
            d_gate, d_up = _silu_bwd(grad_output, gate, up)
            dg2, du2 = d_gate.reshape(-1, d_gate.shape[-1]), d_up.reshape(-1, d_up.shape[-1])
            x2 = x.reshape(-1, x.shape[-1])
            dx = (d_gate @ w_gate + d_up @ w_up) if nx else None
            return (dx, dg2.t() @ x2 if ng else None, du2.t() @ x2 if nu else None,
                    dg2.sum(0) if nbg else None, du2.sum(0) if nbu else None)
        dx, dwg, dwu, d_gate, d_up = ops.swiglu_backward(grad_output, x, w_gate, w_up, gate, up, want_dx=nx,
                                                         want_dw=(ng or nu))
        dbg = d_gate.float().sum(0).to(gate.dtype) if nbg else None
        dbu = d_up.float().sum(0).to(up.dtype) if nbu else None
        return dx, (dwg if ng else None), (dwu if nu else None), dbg, dbu


class FusedSwiGLU(nn.Module):
    """Drop-in for reference Tools/swiglu/FusedSwiglu.py:43-91 (params w_gate, w_up [I, H]; b_gate, b_up)."""

    def __init__(self, hidden_size, intermediate_size, bias=False):
        super().__init__()
        self.hidden_size = hidden_size
        self.intermediate_size = intermediate_size
        self.w_gate = nn.Parameter(torch.empty(intermediate_size, hidden_size))
        self.w_up = nn.Parameter(torch.empty(intermediate_size, hidden_size))
        if bias:
            self.b_gate = nn.Parameter(torch.zeros(intermediate_size))
            self.b_up = nn.Parameter(torch.zeros(intermediate_size))
        else:
            self.register_parameter("b_gate", None)
            self.register_parameter("b_up", None)
        self.reset_parameters()

    def reset_parameters(self):
        nn.init.kaiming_uniform_(self.w_gate, a=5 ** 0.5)
        nn.init.kaiming_uniform_(self.w_up, a=5 ** 0.5)

    def forward(self, x):
        return SwiGLUFunction.apply(x, self.w_gate, self.w_up, self.b_gate, self.b_up)

    def extra_repr(self):
        return (f"hidden_size={self.hidden_size}, intermediate_size={self.intermediate_size}, "
                f"bias={self.b_gate is not None}")


# ------------------------------------------------------------------------------------------------ Linear / LoRA
class LinearFunction(torch.autograd.Function):
    """y = a w^T + b on the tcgen05 GEMM; backward = two more GEMMs with MN-major operands (no transposes)."""

    @classmethod
    def apply(cls, a, weight, bias=None):
        if not _wants_grad(a, weight, bias):
            return ops.linear_forward(a, weight, bias)
        return super().apply(a, weight, bias)

    @staticmethod
    def forward(ctx, a, weight, bias=None):
        ctx.save_for_backward(a, weight)
        ctx.has_bias = bias is not None
        return ops.linear_forward(a, weight, bias)

    @staticmethod
    def backward(ctx, grad_y):
        a, weight = ctx.saved_tensors
        out_f, in_f = weight.shape
        gy = grad_y.contiguous().view(-1, out_f)
        if gy.dtype != a.dtype:
            gy = gy.to(a.dtype)
        a2 = a.contiguous().view(-1, in_f)
        da = dw = db = None
        if ctx.needs_input_grad[0]:
            da = ops.gemm(gy, weight.contiguous(), b_mn_major=True).view(a.shape)      # gy [T,out] x W[out,in]
        if ctx.needs_input_grad[1]:
            dw = ops.gemm(gy, a2, a_mn_major=True, b_mn_major=True)                     # gy^T a
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = gy.float().sum(0).to(weight.dtype)
        return da, dw, db


def _linear(x, weight, bias=None):
    if ops.supported(x) and weight.dtype == x.dtype and weight.is_cuda and _dims8(*weight.shape):
        return LinearFunction.apply(x, weight, bias)
    return F.linear(x, weight, bias)


class LinearLoRAFunction(torch.autograd.Function):
    """y = x W^T + bias + scale * (dropout(x) A^T) B^T for a frozen base W (reference Model/model.py:107-121): the adapter is
    a second accumulation phase (K = rank) of the base GEMM, forward and backward; with LoRA dropout the mask is drawn here
    (nn.Dropout semantics: Bernoulli(1 - p) keep mask, kept values scaled by 1 / (1 - p)) and stays fused -- forward feeds
    dropout(x) to the rank-r GEMM only, backward adds the masked adapter gradient in the base GEMM's epilogue."""

    @classmethod
    def apply(cls, x, weight, bias, lora_a, lora_b, scale, p_drop):
        if not _wants_grad(x, lora_a, lora_b):
            xl = F.dropout(x, p_drop, True) if p_drop > 0.0 else None
            return ops.linear_lora_forward(x, weight, lora_a, lora_b * scale, bias, xl)[0]
        return super().apply(x, weight, bias, lora_a, lora_b, scale, p_drop)

    @staticmethod
    def forward(ctx, x, weight, bias, lora_a, lora_b, scale, p_drop):
        lora_bs = lora_b * scale
        mask = xl = None
        if p_drop > 0.0:
            mask = torch.empty_like(x).bernoulli_(1.0 - p_drop).mul_(1.0 / (1.0 - p_drop))   # keep mask, pre-scaled
            xl = x * mask
        y, t = ops.linear_lora_forward(x, weight, lora_a, lora_bs, bias, xl)
        ctx.save_for_backward(xl if xl is not None else x, weight, lora_a, lora_bs, t, mask)
        ctx.scale, ctx.x_shape = scale, x.shape
        return y

    @staticmethod
    def backward(ctx, grad_y):
        xl, weight, lora_a, lora_bs, t, mask = ctx.saved_tensors
        nx, nw, nb, na, nlb, _, _ = ctx.needs_input_grad
        if nw:
            raise RuntimeError("LinearLoRAFunction: the base weight is frozen under LoRA (Model/model.py:117)")
        fn = None
        if mask is not None:
            in_f = weight.shape[1]
            fn = lambda u: ops.gemm(u, lora_a, b_mn_major=True).view(-1, in_f) * mask.reshape(-1, in_f)   # mask * (u A)
        dx, dla, dlbs = ops.linear_lora_backward(grad_y, xl, weight, lora_a, lora_bs, t, want_dx=nx, want_dlora=(na or nlb),
                                                 dx_addend_fn=fn)
        db = grad_y.reshape(-1, grad_y.shape[-1]).float().sum(0).to(weight.dtype) if nb else None
        dlb = (dlbs * ctx.scale) if (dlbs is not None and nlb) else None
        return (dx.view(ctx.x_shape) if dx is not None else None), None, db, (dla if na else None), dlb, None, None


class Linear_LORA(nn.Module):
    """Drop-in for reference Model/model.py:107-121: frozen base + (alpha/rank) * B(A(dropout(x))).

    16-bit CUDA tensors with a frozen base: base projection and the rank-r adapter run as ONE tcgen05 GEMM with two
    accumulation phases (LinearLoRAFunction), dropout included.  Anything else evaluates the reference's expression."""

    def __init__(self, in_dim: int, out_dim: int, rank: int, alpha: float, dropout: float):
        super().__init__()
        self.linear = nn.Linear(in_dim, out_dim, bias=False)
        self.lora_a = nn.Linear(in_dim, rank, bias=False)
        self.lora_b = nn.Linear(rank, out_dim, bias=False)
        self.rank = rank
        self.alpha = alpha
        self.dropout = nn.Dropout(p=dropout)
        self.linear.weight.requires_grad = False
        self.lora_a.weight.requires_grad = True
        self.lora_b.weight.requires_grad = True

    def _fusable(self, x):
        w = self.linear.weight
        return (ops.supported(x) and w.is_cuda and not w.requires_grad and w.dtype == x.dtype and
                self.lora_a.weight.dtype == x.dtype and self.lora_b.weight.dtype == x.dtype and
                self.rank % 8 == 0 and self.rank <= 64 and w.shape[0] % 8 == 0 and w.shape[1] % 8 == 0 and
                x.numel() // max(1, x.shape[-1]) > 0)

    def forward(self, x):
        if self._fusable(x):
            p = self.dropout.p if (self.training and isinstance(self.dropout, nn.Dropout)) else 0.0
            if p < 1.0:
                return LinearLoRAFunction.apply(x, self.linear.weight, self.linear.bias, self.lora_a.weight, self.lora_b.weight,
                                                self.alpha / self.rank, float(p))
        base = _linear(x, self.linear.weight, self.linear.bias)
        return base + (self.alpha / self.rank) * self.lora_b(self.lora_a(self.dropout(x)))


# ------------------------------------------------------------------------------------------------ feed-forward
class FFNFunction(torch.autograd.Function):
    """Whole feed-forward y = w_down(silu(x w_gate^T) * (x w_up^T)) with a hand-written backward:
    d_act GEMM whose epilogue recomputes SiLU' in registers, two-phase dX GEMM, three wgrad GEMMs."""

    @classmethod
    def apply(cls, x, w_gate, w_up, w_down, b_gate=None, b_up=None, b_down=None):
        if not _wants_grad(x, w_gate, w_up, w_down, b_gate, b_up, b_down):
            return ops.ffn_forward(x, w_gate, w_up, w_down, b_gate, b_up, b_down, want_cache=False)[0]
        return super().apply(x, w_gate, w_up, w_down, b_gate, b_up, b_down)

    @staticmethod
    def forward(ctx, x, w_gate, w_up, w_down, b_gate=None, b_up=None, b_down=None):
        need_grad = any(ctx.needs_input_grad)
        y, gate, up = ops.ffn_forward(x, w_gate, w_up, w_down, b_gate, b_up, b_down, want_cache=need_grad)
        if need_grad:
            ctx.save_for_backward(x, w_gate, w_up, w_down, gate, up)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        x, w_gate, w_up, w_down, gate, up = ctx.saved_tensors
        nx, ng, nu, nd, nbg, nbu, nbd = ctx.needs_input_grad
        dx, dwg, dwu, dwd, d_gate, d_up = ops.ffn_backward(grad_y, x, w_gate, w_up, w_down, gate, up, want_dx=nx,
                                                           want_dw_gate_up=(ng or nu), want_dw_down=nd)
        dbg = d_gate.float().sum(0).to(gate.dtype) if nbg else None
        dbu = d_up.float().sum(0).to(up.dtype) if nbu else None
        dbd = grad_y.reshape(-1, grad_y.shape[-1]).float().sum(0).to(w_down.dtype) if nbd else None
        return dx, (dwg if ng else None), (dwu if nu else None), dwd, dbg, dbu, dbd


class FFNLoRAFunction(torch.autograd.Function):
    """Feed-forward with a LoRA adapter on a frozen w_down (reference README.md:179-188 swaps Linear_LORA,
    Model/model.py:107-121, into FusedFeedforward.w_down): the adapter is a second accumulation phase (K = rank) of the
    down GEMM in forward and of the d_act GEMM in backward, so neither [tokens, hidden] nor [tokens, inter] LoRA
    terms are materialised.  `scale` = alpha / rank."""

    @classmethod
    def apply(cls, x, w_gate, w_up, w_down, lora_a, lora_b, scale):
        if not _wants_grad(x, w_gate, w_up, lora_a, lora_b):
            return ops.ffn_lora_forward(x, w_gate, w_up, w_down, lora_a, lora_b * scale, want_cache=False)[0]
        return super().apply(x, w_gate, w_up, w_down, lora_a, lora_b, scale)

    @staticmethod
    def forward(ctx, x, w_gate, w_up, w_down, lora_a, lora_b, scale):
        lora_bs = lora_b * scale
        y, t, gate, up = ops.ffn_lora_forward(x, w_gate, w_up, w_down, lora_a, lora_bs, want_cache=True)
        ctx.save_for_backward(x, w_gate, w_up, w_down, lora_a, lora_bs, t, gate, up)
        ctx.scale = scale
        return y

    @staticmethod
    def backward(ctx, grad_y):
        x, w_gate, w_up, w_down, lora_a, lora_bs, t, gate, up = ctx.saved_tensors
        nx, ng, nu, nd, na, nb, _ = ctx.needs_input_grad
        if nd:
            raise RuntimeError("FFNLoRAFunction: the base w_down is frozen under LoRA (Model/model.py:117); "
                               "set requires_grad=False on it or use FusedFeedforward without an adapter")
        dx, dwg, dwu, dla, dlbs = ops.ffn_lora_backward(grad_y, x, w_gate, w_up, w_down, lora_a, lora_bs, t, gate, up,
                                                        want_dx=nx, want_dw_gate_up=(ng or nu), want_dlora=(na or nb))
        dlb = (dlbs * ctx.scale) if (dlbs is not None and nb) else None
        return dx, (dwg if ng else None), (dwu if nu else None), None, (dla if na else None), dlb, None


def _is_lora(m) -> bool:
    return all(hasattr(m, a) for a in ("linear", "lora_a", "lora_b", "rank", "alpha"))


class FusedFeedforward(nn.Module):
    """Drop-in for reference Model/model.py:210-217 (`.swiglu`, `.w_down`; state_dict keys unchanged).

    `w_down` may be swapped for a Linear_LORA (ours or the reference's) by the README's LoRA surgery
    (reference README.md:179-188); its frozen base then still runs on the tcgen05 GEMM.
    """

    def __init__(self, hidden_size: int, intermediate_size: int, bias: bool = False):
        super().__init__()
        self.hidden_size = hidden_size
        self.intermediate_size = intermediate_size
        self.swiglu = FusedSwiGLU(hidden_size, intermediate_size, bias=bias)
        self.w_down = nn.Linear(intermediate_size, hidden_size, bias=bias)

    def forward(self, x):
        sw, wd = self.swiglu, self.w_down
        if ops.supported(x) and sw.w_gate.dtype == x.dtype and _dims8(*sw.w_gate.shape):
            if isinstance(wd, nn.Linear) and wd.weight.dtype == x.dtype:
                return FFNFunction.apply(x, sw.w_gate, sw.w_up, wd.weight, sw.b_gate, sw.b_up, wd.bias)
            if _is_lora(wd) and wd.linear.weight.dtype == x.dtype:
                drop = getattr(wd, "dropout", None)
                no_dropout = drop is None or not (self.training and getattr(drop, "p", 0.0) > 0.0)
                if (no_dropout and sw.b_gate is None and wd.linear.bias is None and not wd.linear.weight.requires_grad and
                        wd.lora_a.weight.dtype == x.dtype and wd.lora_b.weight.dtype == x.dtype and
                        wd.rank % 8 == 0 and wd.rank <= 64 and x.numel() // x.shape[-1] > 0):
                    return FFNLoRAFunction.apply(x, sw.w_gate, sw.w_up, wd.linear.weight, wd.lora_a.weight,
                                                 wd.lora_b.weight, wd.alpha / wd.rank)
                act = sw(x)
                base = LinearFunction.apply(act, wd.linear.weight, wd.linear.bias)
                return base + (wd.alpha / wd.rank) * wd.lora_b(wd.lora_a(wd.dropout(act)))
        return wd(sw(x))


class BlockTailFunction(torch.autograd.Function):
    """out = attn_out + ff(norm2(attn_out, residual))  [, next_normed = next_norm(out)] -- the tail of the reference's
    TransformerBlock.forward (Model/model.py:270-273) and, optionally, the next block's norm1 / final_norm (:267, :346) --
    as one differentiable op: forward is ONE C call (l32_block_tail_forward_ex), backward is the FFN backward (d_act GEMM
    with the SiLU' epilogue, two-phase dX, wgrads) between two RMSNorm backwards whose store passes absorb the two
    "gradient around the norm" additions (d_out into the next norm's dx, d_out into norm2's dx for attn_out)."""

    @staticmethod
    def forward(ctx, attn_out, residual, norm_w, eps, w_gate, w_up, w_down, next_w, next_eps):
        r = ops.block_tail_forward(attn_out, residual, norm_w, eps, w_gate, w_up, w_down, train=True, next_norm_weight=next_w,
                                   next_eps=next_eps)
        ctx.save_for_backward(r["h"], r["rms"], r["normed"], r["gate"], r["up"], norm_w, w_gate, w_up, w_down,
                              r["out"] if next_w is not None else None, next_w, r["next_rms"])
        ctx.has_residual = residual is not None
        if next_w is None:
            return r["out"]
        return r["out"], r["next_normed"]

    @staticmethod
    def backward(ctx, d_out, d_next=None):
        h, rms, normed, gate, up, norm_w, w_gate, w_up, w_down, out, next_w, next_rms = ctx.saved_tensors
        na, nr, nnw, _, ng, nu, nd, nnext, _ = ctx.needs_input_grad
        d_next_w = None
        if next_w is not None:
            # gradient of the chained norm, with the gradient that reaches `out` directly added in its store pass
            d_out, d_next_w = ops.rmsnorm_backward(d_next, out, next_w, next_rms, want_dweight=nnext, addend=d_out)
            if d_next_w is not None and d_next_w.dtype != next_w.dtype:
                d_next_w = d_next_w.to(next_w.dtype)
        d_out = d_out.contiguous()
        d_normed, dwg, dwu, dwd, _, _ = ops.ffn_backward(d_out, normed, w_gate, w_up, w_down, gate, up, want_dx=True,
                                                         want_dw_gate_up=(ng or nu), want_dw_down=nd)
        # d_attn_out = d_out + norm2 backward; d_residual = norm2 backward alone
        want_res = bool(ctx.has_residual and nr)
        res = ops.rmsnorm_backward(d_normed, h, norm_w, rms, want_dweight=nnw, addend=d_out, want_plain=want_res)
        d_attn, d_norm_w, d_h = res if want_res else (res[0], res[1], None)
        if d_norm_w is not None and d_norm_w.dtype != norm_w.dtype:
            d_norm_w = d_norm_w.to(norm_w.dtype)
        return ((d_attn if na else None), (d_h if (ctx.has_residual and nr) else None), d_norm_w, None,
                (dwg if ng else None), (dwu if nu else None), dwd, d_next_w, None)


def block_tail(norm2, ff, attn_out, residual, next_norm=None):
    """`attn_out + ff(norm2(attn_out, residual=residual))` -- the tail of the reference's TransformerBlock.forward
    (Model/model.py:270-273).  On 16-bit CUDA tensors with a plain `w_down` it is one C call (Add-RMSNorm, fused gate/up
    GEMM, down GEMM whose epilogue adds attn_out), with or without autograd (BlockTailFunction).  `next_norm`: the
    LLAMARMSNorm that will consume the result next (the following block's norm1, or final_norm): its output is computed in
    the same call and attached to the returned tensor, where LLAMARMSNorm.forward picks it up.  Otherwise (fp32, CPU,
    LoRA / biases) the modules are composed exactly as the reference does."""
    sw, wd = ff.swiglu, ff.w_down
    fusable = (ops.supported(attn_out) and isinstance(wd, nn.Linear) and wd.bias is None and sw.b_gate is None and
               _dims8(*sw.w_gate.shape) and
               sw.w_gate.dtype == attn_out.dtype and wd.weight.dtype == attn_out.dtype and
               (residual is None or (residual.shape == attn_out.shape and residual.dtype == attn_out.dtype)) and
               attn_out.numel() > 0)
    if not fusable:
        return attn_out + ff(norm2(attn_out, residual=residual))
    nw = next_norm.weight if isinstance(next_norm, LLAMARMSNorm) else None
    neps = next_norm.eps if nw is not None else 0.0
    if _wants_grad(attn_out, residual, norm2.weight, sw.w_gate, sw.w_up, wd.weight, nw):
        res = BlockTailFunction.apply(attn_out, residual, norm2.weight, norm2.eps, sw.w_gate, sw.w_up, wd.weight, nw, neps)
        out, nn_ = res if nw is not None else (res, None)
    else:
        res = ops.block_tail_forward(attn_out, residual, norm2.weight, norm2.eps, sw.w_gate, sw.w_up, wd.weight,
                                     next_norm_weight=nw, next_eps=neps)
        out, nn_ = (res["out"], res["next_normed"]) if nw is not None else (res, None)
    if nn_ is not None:
        out._l32_prenormed = (next_norm, nn_, out._version)
    return out


def _transformer_block_forward(self, hidden_states, attention_mask=None, position_ids=None, kv_cache=None):
    """Same computation as the reference's TransformerBlock.forward (Model/model.py:265-273) with the tail fused and
    chained into the norm that consumes the block's output (`_l32_next_norm`, wired by `chain_block_norms`)."""
    normed = self.norm1(hidden_states)          # picks up the previous block's chained result when there is one
    attn_out = self.att(normed, attention_mask=attention_mask, position_ids=position_ids, kv_cache=kv_cache)
    return block_tail(self.norm2, self.ff, attn_out, hidden_states, next_norm=getattr(self, "_l32_next_norm", None))


def chain_block_norms(blocks, final_norm=None):
    """Tell every decoder block which norm consumes its output: the next block's norm1, and `final_norm` after the last
    one (reference Model/model.py:341-346 runs `for layer in self.layers` then `self.final_norm`).  Stored outside the module
    tree (no new state_dict keys, no parameter sharing)."""
    blocks = list(blocks)
    for i, blk in enumerate(blocks):
        nxt = blocks[i + 1].norm1 if i + 1 < len(blocks) else final_norm
        object.__setattr__(blk, "_l32_next_norm", nxt if isinstance(nxt, LLAMARMSNorm) else None)


# ------------------------------------------------------------------------------------------------ attention + KV cache
class KVCache:
    """Drop-in for reference Model/model.py:12-29 with PREALLOCATED storage: per layer one zero-initialised
    [batch, kv_heads, capacity, head_dim] buffer for keys and one for values; appending is a store at the current length
    (capacity doubles when it runs out) instead of the reference's torch.cat per layer per step.
    Same surface (`key_cache`, `value_cache`, `num_items()`, `update()`); `update` returns views of the filled part, so code
    written against the reference's cache keeps working."""

    def __init__(self, capacity: int = 0):
        self.key_cache: list = []        # per layer: the FILLED view [B, kv, len, d] (what the reference keeps)
        self.value_cache: list = []
        self._k: list = []               # per layer: preallocated storage
        self._v: list = []
        self._len: list = []
        self._capacity = int(capacity)

    def num_items(self) -> int:
        return self._len[0] if self._len else 0

    def length(self, layer_idx: int) -> int:
        return self._len[layer_idx] if layer_idx < len(self._len) else 0

    def reserve(self, layer_idx, batch, kv_heads, head_dim, need, dtype, device):
        """Storage of layer `layer_idx` with room for `need` tokens; returns (cache_k, cache_v, current length)."""
        while len(self._k) <= layer_idx:
            self._k.append(None); self._v.append(None); self._len.append(0)
            self.key_cache.append(None); self.value_cache.append(None)
        k = self._k[layer_idx]
        if k is not None and (k.shape[0] != batch or k.shape[1] != kv_heads or k.shape[3] != head_dim or k.dtype != dtype or
                              k.device != torch.device(device)):
            k = None                                  # a different batch / geometry starts a fresh cache for this layer
            self._k[layer_idx] = self._v[layer_idx] = None
            self._len[layer_idx] = 0
        if k is None or k.shape[2] < need:
            cap = max(need, self._capacity, 2 * (k.shape[2] if k is not None else 0), 64)
            cap = -(-cap // 64) * 64
            nk = torch.zeros(batch, kv_heads, cap, head_dim, dtype=dtype, device=device)
            nv = torch.zeros_like(nk)
            if k is not None and self._len[layer_idx] > 0:
                n = self._len[layer_idx]
                nk[:, :, :n].copy_(k[:, :, :n]); nv[:, :, :n].copy_(self._v[layer_idx][:, :, :n])
            self._k[layer_idx], self._v[layer_idx] = nk, nv
        return self._k[layer_idx], self._v[layer_idx], self._len[layer_idx]

    def advance(self, layer_idx, n):
        self._len[layer_idx] += n
        ln = self._len[layer_idx]
        self.key_cache[layer_idx] = self._k[layer_idx][:, :, :ln]
        self.value_cache[layer_idx] = self._v[layer_idx][:, :, :ln]

    def update(self, key_states, value_states, layer_idx: int):
        """Reference-compatible append of [B, kv, t, d] keys / values (already rotated); returns the filled views."""
        b, kvh, t, d = key_states.shape
        ck, cv, ln = self.reserve(layer_idx, b, kvh, d, self.length(layer_idx) + t, key_states.dtype, key_states.device)
        ck[:, :, ln:ln + t].copy_(key_states)
        cv[:, :, ln:ln + t].copy_(value_states)
        self.advance(layer_idx, t)
        return self.key_cache[layer_idx], self.value_cache[layer_idx]


class PagedKVCache:
    """KV cache for serving several sequences at once (inference only): keys / values live in pages of 64 tokens
    (ops.KV_PAGE, one key tile of the attention kernel) named by a block table, and every sequence has its own length.
    A finished sequence hands its pages back (`free_sequence`) and a new one can join in the same step (`add_sequence`).

    Per layer one pool for K and one for V, [num_pages, kv_heads, 64, head_dim], zero-initialised on the layer's first
    forward; page index p names the same slot in every layer, so one allocator serves all layers.  The host keeps the
    bookkeeping (free list, each sequence's pages and length) and is the source of truth: nothing is ever read back from
    the device.  The block table and the lengths of the current batch live in static device buffers sized for `max_batch`,
    so a CUDA graph captured over a forward stays valid while `set_batch` changes their contents between replays.

    One step:  set_batch(ids, new_lens) -> every layer's forward -> advance().
    Rows of the device buffers past len(ids) hold zero lengths: a forward over more rows than the batch (a graph captured
    at a larger batch) leaves those rows' output zero and writes no page.
    Pages handed out again keep what the previous sequence wrote: finite values, which is all the kernels require of rows
    past a sequence's length (include/l32_ffn.h)."""

    def __init__(self, num_pages: int, max_batch: int, max_pages_per_seq: int, device=None):
        if num_pages <= 0 or max_batch <= 0 or max_pages_per_seq <= 0:
            raise ValueError("PagedKVCache: num_pages, max_batch and max_pages_per_seq must be positive")
        self.num_pages, self.max_batch, self.max_pages_per_seq = int(num_pages), int(max_batch), int(max_pages_per_seq)
        self.page_size = ops.KV_PAGE
        self._free = list(range(self.num_pages - 1, -1, -1))   # pop() hands out the lowest free page first
        self._pages: dict = {}                                   # sequence id -> its pages, in logical order
        self._len: dict = {}                                     # sequence id -> tokens cached
        self._next_id = 0
        self.batch_ids: list = []
        self.batch_new_lens: list = []
        self._pool_k: list = []                                  # per layer
        self._pool_v: list = []
        if device is None and torch.cuda.is_available():
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = None if device is None else torch.device(device)
        # one device buffer: the block table [max_batch, max_pages_per_seq], then past_lens [max_batch], new_lens [max_batch]
        n = self.max_batch * (self.max_pages_per_seq + 2)
        self._dev = torch.zeros(n, dtype=torch.int32, device=self.device) if self.device is not None else None
        self.block_table = self.past_lens = self.new_lens = None
        if self._dev is not None:
            t = self.max_batch * self.max_pages_per_seq
            self.block_table = self._dev[:t].view(self.max_batch, self.max_pages_per_seq)
            self.past_lens = self._dev[t:t + self.max_batch]
            self.new_lens = self._dev[t + self.max_batch:]

    # -- allocator
    @property
    def free_pages(self) -> int:
        return len(self._free)

    @property
    def max_kv_len(self) -> int:
        """The bound on every sequence's length the attention's split plan is sized for."""
        return self.max_pages_per_seq * self.page_size

    def add_sequence(self) -> int:
        sid = self._next_id
        self._next_id += 1
        self._pages[sid] = []
        self._len[sid] = 0
        return sid

    def free_sequence(self, sid: int) -> None:
        """Hand the sequence's pages back.  If it is part of the current batch, that batch is dropped: call set_batch again
        before the next forward."""
        pages = self._pages.pop(sid)
        del self._len[sid]
        self._free.extend(reversed(pages))
        if sid in self.batch_ids:
            self.batch_ids, self.batch_new_lens = [], []

    def length(self, sid: int) -> int:
        return self._len[sid]

    def pages(self, sid: int) -> list:
        return list(self._pages[sid])

    def set_batch(self, ids, new_lens) -> None:
        """Choose the sequences (rows, in this order) of the next forward calls and the number of tokens each appends, reserve
        the pages those tokens need and upload the block table and lengths (stream-ordered copies from pinned host memory on
        the current stream).  Raises before anything is reserved or enqueued when the pages run out or a sequence would
        outgrow max_pages_per_seq."""
        ids, new_lens = [int(i) for i in ids], [int(n) for n in new_lens]
        if len(ids) != len(new_lens) or not 0 < len(ids) <= self.max_batch:
            raise ValueError(f"set_batch: {len(ids)} ids / {len(new_lens)} lengths for a cache of max_batch {self.max_batch}")
        if len(set(ids)) != len(ids) or any(i not in self._pages for i in ids):
            raise ValueError(f"set_batch: ids must be distinct live sequences, got {ids}")
        if any(n < 0 for n in new_lens):
            raise ValueError(f"set_batch: negative new length in {new_lens}")
        want = []
        for sid, n in zip(ids, new_lens):
            need = -(-(self._len[sid] + n) // self.page_size)
            if need > self.max_pages_per_seq:
                raise ValueError(f"set_batch: sequence {sid} would hold {self._len[sid] + n} tokens, more than max_pages_per_seq "
                                 f"* {self.page_size} = {self.max_kv_len}")
            want.append(max(0, need - len(self._pages[sid])))
        if sum(want) > len(self._free):
            raise RuntimeError(f"PagedKVCache out of pages: this step needs {sum(want)} more, {len(self._free)} free of "
                               f"{self.num_pages}")
        for sid, w in zip(ids, want):
            self._pages[sid].extend(self._free.pop() for _ in range(w))
        self.batch_ids, self.batch_new_lens = ids, new_lens
        host = torch.zeros(self.max_batch * (self.max_pages_per_seq + 2), dtype=torch.int32,
                           pin_memory=self._dev is not None)
        t = self.max_batch * self.max_pages_per_seq
        table = host[:t].view(self.max_batch, self.max_pages_per_seq)
        for r, sid in enumerate(ids):
            pages = self._pages[sid]
            if any(not 0 <= p < self.num_pages for p in pages):
                raise RuntimeError(f"PagedKVCache: page index out of range in sequence {sid}: {pages}")
            if pages:
                table[r, :len(pages)] = torch.tensor(pages, dtype=torch.int32)
            host[t + r] = self._len[sid]
            host[t + self.max_batch + r] = new_lens[r]
        self._host = host                                   # (the last upload's contents, for inspection)
        if self._dev is not None:
            # torch's pinned-memory allocator keeps `host` from being reused until this copy has run, so no host-side wait
            self._dev.copy_(host, non_blocking=True)

    def advance(self) -> None:
        """After the step's last layer: every sequence of the batch now holds its new tokens."""
        for sid, n in zip(self.batch_ids, self.batch_new_lens):
            self._len[sid] += n

    # -- per-layer pools
    def pools(self, layer_idx, kv_heads, head_dim, dtype, device):
        """(pool_k, pool_v) of layer `layer_idx`, created zeroed on first use with this geometry."""
        while len(self._pool_k) <= layer_idx:
            self._pool_k.append(None)
            self._pool_v.append(None)
        k = self._pool_k[layer_idx]
        shape = (self.num_pages, kv_heads, self.page_size, head_dim)
        if k is None:
            k = torch.zeros(shape, dtype=dtype, device=device)
            self._pool_k[layer_idx], self._pool_v[layer_idx] = k, torch.zeros_like(k)
        elif tuple(k.shape) != shape or k.dtype != dtype or k.device != torch.device(device):
            raise ValueError(f"PagedKVCache layer {layer_idx}: pool is {tuple(k.shape)} {k.dtype} on {k.device}, this call "
                             f"needs {shape} {dtype} on {device}")
        return self._pool_k[layer_idx], self._pool_v[layer_idx]


def _rotate_half(x):
    x1, x2 = x[..., : x.shape[-1] // 2], x[..., x.shape[-1] // 2:]
    return torch.cat((-x2, x1), dim=-1)


class GQAAttentionFunction(torch.autograd.Function):
    """ctx [b, t, heads*d] = attention over the PRE-RoPE projection outputs q [b, t, heads*d], k, v [b, t, kv_heads*d] of a
    training call (no KV cache, query i at position_ids[:, i], keys = queries), on the tcgen05 kernels in both directions.
    Saves O(t) tensors (the rotated q / k, v, ctx and the per-row log-sum-exp): no [B, heads, S, S] tensor exists.  The
    backward is one C-ABI call (deterministic) that returns the gradients of q, k, v with the inverse RoPE applied."""

    @staticmethod
    def forward(ctx, q, k, v, position_ids, causal, key_keep, rope_base, kv_heads):
        b, t, _ = q.shape
        d = k.shape[-1] // kv_heads
        q_rot = q.contiguous().clone()                  # rotated in place below: the caller's q stays as it was
        ck = torch.empty(b, kv_heads, t, d, dtype=q.dtype, device=q.device)
        cv = torch.empty_like(ck)
        if key_keep is not None:
            key_keep = key_keep.to(torch.uint8).contiguous()
        ops.rope_kv_append(q_rot, k.contiguous(), v.contiguous(), position_ids, ck, cv, 0, rope_base)
        out, lse = ops.gqa_attention_forward_train(q_rot, ck, cv, causal, key_keep)
        ctx.save_for_backward(q_rot, ck, cv, out, lse, key_keep, position_ids)
        ctx.causal, ctx.rope_base = causal, rope_base
        return out

    @staticmethod
    def backward(ctx, grad_out):
        q_rot, ck, cv, out, lse, keep, position_ids = ctx.saved_tensors
        dq, dk, dv = ops.gqa_attention_backward(grad_out, q_rot, ck, cv, out, lse, position_ids, ctx.causal, keep, ctx.rope_base)
        return dq, dk, dv, None, None, None, None, None


def _mask_causal_keep(attention_mask, b, t, kv_len):
    """The reference's Llama3Model mask (Model/model.py:304-319: causal + key padding) as (causal, key_keep [b, kv_len] | None).
    None means no masking at all; the key-padding row is read from the last query row, which sees every key the causal part
    allows.  A decode step (t = 1) reads it too: a [b, 1, 1, kv_len] mask pads keys of the cache like a prefill mask does."""
    if attention_mask is None:
        return False, None
    keep = None
    if attention_mask.dim() == 4 and attention_mask.shape[-1] == kv_len and attention_mask.shape[-2] == t:
        keep = attention_mask[:, 0, -1, :] > (torch.finfo(attention_mask.dtype).min / 2)
        if keep.shape[0] != b:
            keep = keep.expand(b, -1)
    return True, keep


class GroupQueryAttention(nn.Module):
    """Drop-in for reference Model/model.py:220-254 (same ctor, submodule names and state_dict keys: W_query, W_key, W_value,
    out_proj).  16-bit CUDA inference with head_dim 64 / 128: the three projections and out_proj run on the tcgen05 GEMM
    (fused with their adapter when they are Linear_LORA), RoPE + cache append is one kernel writing straight into the
    preallocated KVCache, and the attention itself is the flash-style tcgen05 kernel -- no [B, heads, S, S] scores, no
    repeat_kv copies, no torch.cat.  `attention_mask` is interpreted as the mask the reference's Llama3Model builds
    (Model/model.py:304-319: causal + key padding); None means no masking at all, as in the reference.
    Under autograd without a cache (training) the same holds in both directions: the projections run as LinearFunction /
    LinearLoRAFunction and the attention as GQAAttentionFunction (tcgen05 forward + backward, O(t) saved memory).  A query row
    that sees no key gets zeros and no gradient (the reference gives it a uniform softmax; a model ignores its loss).
    Anything else (fp32, CPU, other head sizes, a cache under autograd, a foreign cache object) evaluates the reference's own
    expressions."""

    def __init__(self, config, layer_idx=None, dtype=None):
        super().__init__()
        assert config.hidden_size % config.n_heads == 0
        assert config.n_heads % config.n_kv_groups == 0
        self.config = config
        self.layer_idx = layer_idx
        self.num_heads = config.n_heads
        self.head_dim = config.hidden_size // config.n_heads
        self.num_kv_groups = config.n_kv_groups
        self.group_size = config.n_heads // config.n_kv_groups
        self.W_query = nn.Linear(config.hidden_size, config.n_heads * self.head_dim, bias=False, dtype=dtype)
        self.W_key = nn.Linear(config.hidden_size, config.n_kv_groups * self.head_dim, bias=False, dtype=dtype)
        self.W_value = nn.Linear(config.hidden_size, config.n_kv_groups * self.head_dim, bias=False, dtype=dtype)
        self.out_proj = nn.Linear(config.n_heads * self.head_dim, config.hidden_size, bias=False, dtype=dtype)
        self.rope_base = float(getattr(config, "rope_base", 500000.0))
        self.is_causal = True

    # -- reference expressions (Model/model.py:176-198, 238-253)
    def _cos_sin(self, x, position_ids):
        inv_freq = 1.0 / (self.rope_base ** (torch.arange(0, self.head_dim, 2, dtype=torch.int64).float() / self.head_dim))
        inv_freq = inv_freq.to(x.device)
        freqs = (inv_freq[None, :, None].float().expand(position_ids.shape[0], -1, 1) @ position_ids[:, None, :].float()).transpose(1, 2)
        emb = torch.cat((freqs, freqs), dim=-1)
        return emb.cos().to(x.dtype), emb.sin().to(x.dtype)

    def _reference_forward(self, hidden_states, attention_mask, position_ids, kv_cache):
        b, t, _ = hidden_states.shape
        q = self.W_query(hidden_states).view(b, t, self.num_heads, self.head_dim).transpose(1, 2)
        k = self.W_key(hidden_states).view(b, t, self.num_kv_groups, self.head_dim).transpose(1, 2)
        v = self.W_value(hidden_states).view(b, t, self.num_kv_groups, self.head_dim).transpose(1, 2)
        cos, sin = self._cos_sin(v, position_ids)
        cos, sin = cos.unsqueeze(1), sin.unsqueeze(1)
        q, k = (q * cos) + (_rotate_half(q) * sin), (k * cos) + (_rotate_half(k) * sin)
        if kv_cache is not None:
            k, v = kv_cache.update(k, v, self.layer_idx)
        g = self.group_size
        if g > 1:
            k = k[:, :, None].expand(b, self.num_kv_groups, g, k.shape[-2], self.head_dim).reshape(b, self.num_heads, k.shape[-2], self.head_dim)
            v = v[:, :, None].expand(b, self.num_kv_groups, g, v.shape[-2], self.head_dim).reshape(b, self.num_heads, v.shape[-2], self.head_dim)
        score = q @ k.transpose(2, 3)
        if attention_mask is not None:
            score = score + attention_mask[:, :, :, : k.shape[-2]]
        w = torch.softmax(score / (k.shape[-1] ** 0.5), dim=-1)
        ctx = (w @ v).transpose(1, 2).contiguous().reshape(b, t, -1)
        return self.out_proj(ctx)

    def _kernel_ok(self, x):
        ws = [m.linear.weight if _is_lora(m) else m.weight for m in (self.W_query, self.W_key, self.W_value, self.out_proj)]
        return (ops.supported(x) and self.head_dim in (64, 128) and x.dim() == 3 and x.numel() > 0 and
                all(w.is_cuda and w.dtype == x.dtype for w in ws))

    def _records_grad(self, x):
        mods = (self.W_query, self.W_key, self.W_value, self.out_proj)
        return _wants_grad(x, *[p for m in mods for p in m.parameters()])

    def _fast_ok(self, x, kv_cache):
        return (self._kernel_ok(x) and (kv_cache is None or isinstance(kv_cache, KVCache)) and not self._records_grad(x))

    def _train_ok(self, x, kv_cache):
        return kv_cache is None and self._kernel_ok(x) and self._records_grad(x)

    @staticmethod
    def _project(mod, x):
        return mod(x) if _is_lora(mod) else _linear(x, mod.weight, mod.bias)

    def _qkv(self, hidden_states):
        projs = (self.W_query, self.W_key, self.W_value)
        if (not torch.is_grad_enabled() or not _wants_grad(hidden_states, *[m.weight for m in projs])) and all(
                not _is_lora(m) and m.bias is None and m.weight.dtype == hidden_states.dtype and _dims8(*m.weight.shape) for m in projs):
            # inference: the three projections of the same activations in ONE launch (reference Model/model.py:231-233)
            return ops.linear_group_forward(hidden_states, [m.weight for m in projs])
        q = self._project(self.W_query, hidden_states)           # [b, t, heads * d]: the kernels read this layout as it is
        k = self._project(self.W_key, hidden_states)
        v = self._project(self.W_value, hidden_states)
        return q, k, v

    def _paged_forward(self, hidden_states, attention_mask, position_ids, cache):
        """Inference over a PagedKVCache: row r of hidden_states [len(batch), t, hidden] (right-padded, t >= every new length)
        is sequence cache.batch_ids[r]; attention is causal over that sequence's own keys.  There are no reference expressions
        for a paged cache, so inputs the kernels do not take are an error."""
        if attention_mask is not None:
            raise ValueError("GroupQueryAttention with a PagedKVCache takes no attention_mask: the cache's lengths are the mask")
        if position_ids is None:
            raise ValueError("GroupQueryAttention with a PagedKVCache needs position_ids")
        if self._records_grad(hidden_states):
            raise ValueError("a PagedKVCache is inference-only: run the forward under torch.no_grad()")
        if not self._kernel_ok(hidden_states):
            raise ValueError("GroupQueryAttention with a PagedKVCache runs on the sm_100a kernels only: CUDA bf16 / fp16 "
                             "[batch, t, hidden] inputs and weights, head_dim 64 or 128")
        b, t, _ = hidden_states.shape
        if not cache.batch_ids or b != len(cache.batch_ids) or t < max(cache.batch_new_lens):
            raise ValueError(f"hidden_states [{b}, {t}, ...] does not fit the cache's batch: {len(cache.batch_ids)} sequences "
                             f"appending {cache.batch_new_lens} tokens (call set_batch first)")
        if cache.device is None or hidden_states.device != cache.device:
            raise ValueError(f"PagedKVCache on {cache.device}, hidden_states on {hidden_states.device}")
        if position_ids.dim() == 1:
            position_ids = position_ids[None]
        pos = position_ids.to(device=hidden_states.device, dtype=torch.int64).expand(b, t).contiguous()
        q, k, v = self._qkv(hidden_states)
        pk, pv = cache.pools(self.layer_idx or 0, self.num_kv_groups, self.head_dim, q.dtype, q.device)
        ops.rope_kv_append_paged(q, k, v, pos, pk, pv, cache.block_table, cache.past_lens, cache.new_lens, self.rope_base)
        ctx = ops.gqa_attention_forward_paged(q, pk, pv, cache.block_table, cache.past_lens, cache.new_lens,
                                              max_kv_len=cache.max_kv_len)
        return self._project(self.out_proj, ctx)

    def forward(self, hidden_states, attention_mask=None, position_ids=None, kv_cache=None):
        if isinstance(kv_cache, PagedKVCache):
            return self._paged_forward(hidden_states, attention_mask, position_ids, kv_cache)
        if (position_ids is None or (attention_mask is not None and not attention_mask.is_floating_point())):
            return self._reference_forward(hidden_states, attention_mask, position_ids, kv_cache)
        train = self._train_ok(hidden_states, kv_cache)
        if not train and not self._fast_ok(hidden_states, kv_cache):
            return self._reference_forward(hidden_states, attention_mask, position_ids, kv_cache)
        b, t, _ = hidden_states.shape
        if position_ids.dim() == 1:
            position_ids = position_ids[None]
        if position_ids.shape[0] != b:
            position_ids = position_ids.expand(b, -1)
        if train:
            q = self._project(self.W_query, hidden_states)
            k = self._project(self.W_key, hidden_states)
            v = self._project(self.W_value, hidden_states)
            causal, keep = _mask_causal_keep(attention_mask, b, t, t)
            pos = position_ids.to(device=q.device, dtype=torch.int64).contiguous()
            ctx = GQAAttentionFunction.apply(q, k, v, pos, causal, keep, self.rope_base, self.num_kv_groups)
            return self._project(self.out_proj, ctx)
        q, k, v = self._qkv(hidden_states)
        cache = kv_cache if kv_cache is not None else KVCache()
        layer = self.layer_idx if kv_cache is not None else 0
        past = cache.length(layer)
        ck, cv, _ = cache.reserve(layer, b, self.num_kv_groups, self.head_dim, past + t, q.dtype, q.device)
        ops.rope_kv_append(q, k, v, position_ids.to(device=q.device, dtype=torch.int64), ck, cv, past, self.rope_base)
        cache.advance(layer, t)
        kv_len = past + t
        causal, keep = _mask_causal_keep(attention_mask, b, t, kv_len)
        ctx = ops.gqa_attention_forward(q, ck, cv, kv_len, past, causal=causal, key_keep=keep)
        return self._project(self.out_proj, ctx)


# ------------------------------------------------------------------------------------------------ lm_head + loss
def shift_labels(labels, ignore_index=-100):
    """Row-aligned targets for `shift_logits = logits[..., :-1, :]` / `shift_labels = labels[..., 1:]` (reference
    Model/model.py:432-433): position (b, s) is scored against labels[b, s + 1]; the last position of every sequence has no
    target.  Same shape as `labels`."""
    out = torch.full_like(labels, ignore_index)
    out[..., :-1] = labels[..., 1:]
    return out


class LMHeadCEFunction(torch.autograd.Function):
    """(loss, logits) = lm_head + mean cross entropy over the non-ignored rows (reference Model/model.py:429-438) on the
    tcgen05 GEMM whose epilogue gathers the softmax statistics.  `logits` is returned for the caller's output dict and is
    not differentiable here (the reference's training recipe back-propagates the loss only)."""

    @staticmethod
    def forward(ctx, hidden_states, weight, labels_shifted, ignore_index):
        r = ops.lm_head_ce_forward(hidden_states, weight, labels_shifted, ignore_index)
        ctx.save_for_backward(hidden_states, weight, labels_shifted, r["logits"], r["lse"], r["loss_and_count"])
        ctx.ignore_index = ignore_index
        ctx.mark_non_differentiable(r["logits"])
        return r["loss"], r["logits"]

    @staticmethod
    def backward(ctx, grad_loss, _grad_logits):
        hidden_states, weight, labels_shifted, logits, lse, lc = ctx.saved_tensors
        nh, nw, _, _ = ctx.needs_input_grad
        # the upstream gradient of the scalar loss stays on the device (no host synchronisation): the dlogits kernel reads it
        dh, dw, _ = ops.lm_head_ce_backward(logits, lse, labels_shifted, ctx.ignore_index, lc, grad_loss, hidden_states, weight,
                                            want_dhidden=nh, want_dweight=nw)
        return dh, dw, None, None


def lm_head_loss(lm_head, hidden_states, labels=None, ignore_index=-100):
    """`logits = lm_head(hidden_states)` and, with labels, the shifted cross entropy of the reference's
    MllamaForConditionalGeneration.forward (Model/model.py:429-438).  Returns (logits, loss|None).
    16-bit CUDA tensors with a bias-free head run the fused GEMM + CE kernels; anything else evaluates the reference's own
    expressions."""
    w = lm_head.weight
    fused = (labels is not None and ops.supported(hidden_states) and w.is_cuda and w.dtype == hidden_states.dtype and
             getattr(lm_head, "bias", None) is None and w.shape[0] % 8 == 0 and w.shape[1] % 8 == 0 and hidden_states.numel() > 0)
    if not fused:
        logits = lm_head(hidden_states)
        loss = None
        if labels is not None:
            sl = logits[..., :-1, :].contiguous()
            tl = labels[..., 1:].contiguous()
            loss = nn.CrossEntropyLoss(ignore_index=ignore_index)(sl.view(-1, sl.size(-1)), tl.view(-1))
        return logits, loss
    loss, logits = LMHeadCEFunction.apply(hidden_states, w, shift_labels(labels, ignore_index), ignore_index)
    return logits, loss


def _mllama_forward(self, input_ids=None, pixel_values=None, attention_mask=None, position_ids=None, image_mask=None,
                    labels=None, kv_cache=None, **kwargs):
    """The reference's MllamaForConditionalGeneration.forward (Model/model.py:398-440) with its last eight lines -- lm_head and
    the shifted CrossEntropyLoss -- replaced by `lm_head_loss`; everything before is the reference's own code path."""
    image_features = None
    if pixel_values is not None:
        image_features = self.multi_modal_projector(self.vision_model(pixel_values))
    inputs_embeds = None
    if input_ids is not None:
        inputs_embeds = self.language_model.model.get_input_embeddings()(input_ids)
    if image_features is not None and inputs_embeds is not None:
        inputs_embeds, attention_mask = self._merge_input_ids_with_image_features(image_features, inputs_embeds, input_ids,
                                                                                  attention_mask)
    hidden_states = self.language_model.model(input_embeds=inputs_embeds, attention_mask=attention_mask,
                                              position_ids=position_ids, kv_cache=kv_cache)
    logits, loss = lm_head_loss(self.language_model.lm_head, hidden_states, labels, getattr(self, "ignore_index", -100))
    return {"logits": logits, "loss": loss, "hidden_states": hidden_states, "kv_cache": kv_cache}


FusedFeedForward = FusedFeedforward   # the reference spells it both ways (FusedSwiglu.py:94 vs model.py:210)


def convert_feedforward_to_fused(feedforward_module):
    """w1 = gate, w3 = up, w2 = down (reference Tools/swiglu/FusedSwiglu.py:134-166)."""
    hidden_size = feedforward_module.w2.out_features
    intermediate_size = feedforward_module.w1.out_features
    has_bias = feedforward_module.w1.bias is not None
    fused = FusedFeedforward(hidden_size, intermediate_size, bias=has_bias)
    fused = fused.to(device=feedforward_module.w1.weight.device, dtype=feedforward_module.w1.weight.dtype)
    with torch.no_grad():
        fused.swiglu.w_gate.copy_(feedforward_module.w1.weight)
        fused.swiglu.w_up.copy_(feedforward_module.w3.weight)
        fused.w_down.weight.copy_(feedforward_module.w2.weight)
        if has_bias:
            fused.swiglu.b_gate.copy_(feedforward_module.w1.bias)
            fused.swiglu.b_up.copy_(feedforward_module.w3.bias)
            fused.w_down.bias.copy_(feedforward_module.w2.bias)
    return fused


def patch_reference(model_module, swiglu_module=None, fuse_block_tail=True):
    """Point an imported reference `Model.model` (and `Tools.swiglu.FusedSwiglu`) at this implementation.

    After the call, models built from the reference's own classes (MllamaForConditionalGeneration,
    TransformerBlock, ...) construct our LLAMARMSNorm / FusedFeedforward / Linear_LORA; existing instances
    can be converted with `convert_instances`.
    """
    model_module.LLAMARMSNorm = LLAMARMSNorm
    model_module.RMSNormFunction = RMSNormFunction
    model_module.FusedFeedforward = FusedFeedforward
    model_module.FusedSwiGLU = FusedSwiGLU
    model_module.Linear_LORA = Linear_LORA
    model_module.GroupQueryAttention = GroupQueryAttention
    model_module.KVCache = KVCache
    model_module.HAS_RMSNORM_EXT = True
    if fuse_block_tail and hasattr(model_module, "TransformerBlock"):
        model_module.TransformerBlock.forward = _transformer_block_forward
    if fuse_block_tail and hasattr(model_module, "MllamaForConditionalGeneration"):
        model_module.MllamaForConditionalGeneration.forward = _mllama_forward
    if swiglu_module is not None:
        swiglu_module.SwiGLUFunction = SwiGLUFunction
        swiglu_module.FusedSwiGLU = FusedSwiGLU
        swiglu_module.FusedFeedForward = FusedFeedforward
        swiglu_module.CUDA_AVAILABLE = True


def convert_instances(root: nn.Module) -> nn.Module:
    """Re-class existing reference module instances in place (parameters and state_dict keys untouched)."""
    for m in root.modules():
        name = type(m).__name__
        if name == "LLAMARMSNorm" and not isinstance(m, LLAMARMSNorm):
            m.__class__ = LLAMARMSNorm
        elif name == "FusedSwiGLU" and not isinstance(m, FusedSwiGLU):
            m.__class__ = FusedSwiGLU
        elif name in ("FusedFeedforward", "FusedFeedForward") and not isinstance(m, FusedFeedforward):
            m.__class__ = FusedFeedforward
            if not hasattr(m, "hidden_size"):
                m.hidden_size = m.swiglu.hidden_size
                m.intermediate_size = m.swiglu.intermediate_size
        elif name == "Linear_LORA" and not isinstance(m, Linear_LORA):
            m.__class__ = Linear_LORA
        elif name == "GroupQueryAttention" and not isinstance(m, GroupQueryAttention):
            m.__class__ = GroupQueryAttention
            if not hasattr(m, "rope_base"):
                m.rope_base = float(getattr(getattr(m, "config", None), "rope_base", 500000.0))
    # chain every stack of decoder blocks into the norm that follows it (a `layers` ModuleList next to a `final_norm`)
    # (the reference's Llama3Model keeps them in `trf_blocks`, Model/model.py:296-299)
    for m in root.modules():
        for child in m.children():
            if (isinstance(child, nn.ModuleList) and len(child) and
                    all(hasattr(b, "norm1") and hasattr(b, "norm2") and hasattr(b, "ff") for b in child)):
                chain_block_norms(child, getattr(m, "final_norm", None))
    return root
