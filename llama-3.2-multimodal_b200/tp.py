"""Tensor-parallel SwiGLU feed-forward across the GPUs of one node (one process per GPU, torch.distributed).

The reference has no distributed code at all (SURVEY.md section 2: grep for nccl / all_reduce / world_size finds
nothing); this is the sharding BASELINE.json's north_star asks for:
  * w_gate / w_up are column-parallel: rank r owns rows [r*I/p, (r+1)*I/p) of the [I, H] matrices
    (reference layout Tools/swiglu/FusedSwiglu.py:63-64), a contiguous slice -- no copy;
  * w_down is row-parallel: rank r owns columns [r*I/p, (r+1)*I/p) of the [H, I] matrix (reference
    Model/model.py:214), copied once to a contiguous [H, I/p] shard;
  * forward: x [M, H] replicated -> local fused gate/up+SiLU*mul GEMM -> local down GEMM gives a PARTIAL
    y_r [M, H]; the one real exchange step is reduce-scatter(y_r) over rows followed by all-gather
    (= all-reduce split in two so a sequence-parallel RMSNorm can sit in between).
The token dimension is processed in chunks: the NCCL reduce-scatter / all-gather of chunk c runs on NCCL's
stream while the tcgen05 GEMMs of chunk c+1 run on the compute stream, so the exchange over NVLink overlaps
the math.

Works on CPU tensors with the gloo backend too (tests/test_tp_gloo.py): the per-rank math then goes through the
same modules' fp32 expressions, and reduce-scatter is emulated with all_reduce + slice because gloo has no
reduce_scatter.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import ops
from .modules import FusedFeedforward, KVCache, _mask_causal_keep


def shard_range(inter: int, world: int, rank: int, granule: int = 128) -> tuple[int, int]:
    """Contiguous slice of the intermediate dimension owned by `rank`; multiples of `granule` (one act tile of
    the tcgen05 kernel) wherever possible so no rank gets a ragged tile."""
    units = inter // granule
    if units >= world:
        base, extra = divmod(units, world)
        lo = (rank * base + min(rank, extra)) * granule
        hi = lo + (base + (1 if rank < extra else 0)) * granule
        if rank == world - 1:
            hi = inter
        return lo, hi
    per = -(-inter // world)
    per = -(-per // 8) * 8
    lo = min(rank * per, inter)
    hi = min(lo + per, inter)
    if hi <= lo:
        raise ValueError(f"intermediate size {inter} is too small to shard over {world} ranks: rank {rank} would own "
                         "no columns (every rank needs at least 8)")
    return lo, hi


def shard_ffn_weights(w_gate, w_up, w_down, world: int, rank: int):
    """(w_gate_r [I/p, H] view, w_up_r view, w_down_r [H, I/p] contiguous copy)."""
    lo, hi = shard_range(w_gate.shape[0], world, rank)
    return w_gate[lo:hi], w_up[lo:hi], w_down[:, lo:hi].contiguous()


def attention_head_range(n_heads: int, n_kv: int, world: int, rank: int) -> tuple[tuple[int, int], tuple[int, int]]:
    """((q_lo, q_hi), (kv_lo, kv_hi)): the query heads and KV heads rank `rank` owns.  Heads are sharded by KV group, so
    every query head h of the rank uses a KV head h // (n_heads / n_kv) of the same rank and attention needs no exchange."""
    if n_kv <= 0 or n_heads % n_kv != 0:
        raise ValueError(f"{n_heads} query heads do not split into {n_kv} KV groups")
    if world < 1 or n_kv % world != 0:
        raise ValueError(f"{n_kv} KV heads do not shard over {world} ranks (tensor-parallel attention needs kv_heads % world == 0)")
    if not 0 <= rank < world:
        raise ValueError(f"rank {rank} outside a world of {world}")
    kv_per, q_per = n_kv // world, n_heads // world
    return (rank * q_per, (rank + 1) * q_per), (rank * kv_per, (rank + 1) * kv_per)


def shard_attention_weights(wq, wk, wv, wo, n_heads: int, n_kv: int, world: int, rank: int):
    """(wq_r [Hl*d, hidden] view, wk_r [KVl*d, hidden] view, wv_r view, wo_r [hidden, Hl*d] contiguous copy) of rank `rank`:
    the rows of W_query / W_key / W_value and the columns of out_proj (nn.Linear layouts, reference Model/model.py:231-234)
    of the heads attention_head_range gives it."""
    (qlo, qhi), (klo, khi) = attention_head_range(n_heads, n_kv, world, rank)
    d = wq.shape[0] // n_heads
    return wq[qlo * d:qhi * d], wk[klo * d:khi * d], wv[klo * d:khi * d], wo[:, qlo * d:qhi * d].contiguous()


def shard_state_dict_for_rank(state, world: int, rank: int, *, n_heads: int | None = None, n_kv: int | None = None):
    """Load-time packing (SURVEY.md 8f rank 4): the reference's loader builds a full `converted_state` and hands it to
    load_state_dict (Model/utils.py:149-166); under tensor parallelism a rank only needs its slice of every feed-forward
    weight.  This cuts `*.swiglu.w_gate` / `*.swiglu.w_up` (row slices) and `*.w_down.weight` (column slice, made contiguous)
    down to rank `rank`'s shard while the tensors are still on the host (or memory-mapped safetensors slices), so the full
    matrices never reach the device and FusedTensorParallelBlock(..., presharded=True) takes them as they are.
    Given the head counts `n_heads` / `n_kv`, the attention weights are cut as well (`*.W_query.weight`, `*.W_key.weight`,
    `*.W_value.weight`: rows of the rank's heads; `*.out_proj.weight`: their columns), for
    FusedTensorParallelAttention(..., presharded=True).
    Every other entry is passed through untouched.  Returns a new dict."""
    attn = n_heads is not None and n_kv is not None
    if attn:
        (qlo, qhi), (klo, khi) = attention_head_range(n_heads, n_kv, world, rank)
    out = {}
    for name, t in state.items():
        if attn and name.endswith("W_query.weight"):
            d = t.shape[0] // n_heads
            out[name] = t[qlo * d:qhi * d].contiguous()
        elif attn and (name.endswith("W_key.weight") or name.endswith("W_value.weight")):
            d = t.shape[0] // n_kv
            out[name] = t[klo * d:khi * d].contiguous()
        elif attn and name.endswith("out_proj.weight"):
            d = t.shape[1] // n_heads
            out[name] = t[:, qlo * d:qhi * d].contiguous()
        elif name.endswith("swiglu.w_gate") or name.endswith("swiglu.w_up"):
            lo, hi = shard_range(t.shape[0], world, rank)
            out[name] = t[lo:hi].contiguous()
        elif name.endswith("w_down.weight") or name.endswith("w_down.linear.weight"):
            lo, hi = shard_range(t.shape[1], world, rank)
            out[name] = t[:, lo:hi].contiguous()
        else:
            out[name] = t
    return out


class TensorParallelFFN(torch.nn.Module):
    """Drop-in for FusedFeedforward.forward on `group`: same input, same (replicated) output."""

    def __init__(self, ffn: FusedFeedforward, group=None, chunks: int = 4):
        super().__init__()
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.chunks = chunks
        wg, wu, wd = shard_ffn_weights(ffn.swiglu.w_gate.detach(), ffn.swiglu.w_up.detach(), ffn.w_down.weight.detach(),
                                       self.world, self.rank)
        self.w_gate = torch.nn.Parameter(wg.contiguous(), requires_grad=False)
        self.w_up = torch.nn.Parameter(wu.contiguous(), requires_grad=False)
        self.w_down = torch.nn.Parameter(wd, requires_grad=False)
        self.hidden_size = self.w_gate.shape[1]

    # -- local math: sm_100a kernels for CUDA 16-bit tensors, the reference's fp32 expressions otherwise
    def _partial(self, x2):
        if ops.supported(x2):
            y, _, _ = ops.ffn_forward(x2, self.w_gate, self.w_up, self.w_down)
            return y
        act = torch.nn.functional.silu(torch.nn.functional.linear(x2, self.w_gate)) * torch.nn.functional.linear(x2, self.w_up)
        return torch.nn.functional.linear(act, self.w_down)

    def _reduce_scatter(self, part, out):
        if part.is_cuda:
            return dist.reduce_scatter_tensor(out, part, group=self.group, async_op=True)
        dist.all_reduce(part, group=self.group)          # gloo: no reduce_scatter
        rows = out.shape[0]
        out.copy_(part[self.rank * rows:(self.rank + 1) * rows])
        return None

    def forward_scattered(self, x):
        """Returns the list of (row_offset, rows, y_slice [rows/p, H]) per chunk: this rank's rows after the
        reduce-scatter -- the hand-off point for a sequence-parallel Add-RMSNorm."""
        x2 = x.reshape(-1, x.shape[-1])
        m = x2.shape[0]
        p = self.world
        step = -(-m // self.chunks)
        step = max(p, -(-step // p) * p)
        out, works = [], []
        for lo in range(0, m, step):
            hi = min(lo + step, m)
            rows = hi - lo
            part = self._partial(x2[lo:hi])
            if rows % p:                                   # ragged last chunk: pad rows so they split evenly
                pad = p - rows % p
                part = torch.cat([part, part.new_zeros(pad, part.shape[1])])
            piece = torch.empty(part.shape[0] // p, part.shape[1], dtype=part.dtype, device=part.device)
            works.append(self._reduce_scatter(part, piece))
            out.append((lo, rows, piece))
        for w in works:
            if w is not None:
                w.wait()
        return out

    def forward(self, x):
        x2 = x.reshape(-1, x.shape[-1])
        m, p = x2.shape[0], self.world
        y = torch.empty(m, self.hidden_size, dtype=x2.dtype, device=x2.device)
        works = []
        for lo, rows, piece in self.forward_scattered(x):
            padded = piece.shape[0] * p
            if padded == rows:
                works.append(dist.all_gather_into_tensor(y[lo:lo + rows], piece, group=self.group, async_op=True))
            else:
                full = torch.empty(padded, piece.shape[1], dtype=piece.dtype, device=piece.device)
                dist.all_gather_into_tensor(full, piece, group=self.group)
                y[lo:lo + rows].copy_(full[:rows])
        for w in works:
            w.wait()
        return y.view(x.shape)


# ======================================================================================================================
# Fused path: the collectives live INSIDE the tcgen05 GEMM kernels (peer memory over NVLink 5 / NVSwitch), no NCCL on
# the data path.  Sequence-parallel in, sequence-parallel out:
#
#   rank r holds rows [r*R, (r+1)*R) of x / residual (R = ceil(tokens / world))
#   1. Add-RMSNorm of the own rows, written into the own full-size `normed` buffer      (K1, local)
#      -> signal ready[r] = epoch on every rank
#   2. gate/up GEMM + SiLU*mul on the weight shard; the other ranks' normed rows are PULLED out of peer memory by the
#      spare warps of the GEMM CTAs while the tensor cores work on the rows already there (fused all-gather)
#   3. down GEMM on the shard; the epilogue stores every output row straight into the slot of the rank that owns the
#      row (fused reduce-scatter, peer stores)  -> signal rs_done[r] = epoch on every rank
#   4. the owner sums the `world` slots (fp32, rank order) once every peer has signalled -> y rows [r*R, (r+1)*R)
#
# Backward mirrors it: the own rows of dY are published in the same exchange buffer, the d_act GEMM (SiLU' epilogue) pulls
# the other ranks' dY rows, the two-phase dX GEMM pushes its partial rows to their owners, the weight gradients are local
# GEMMs on the shard, and the owner sums the dX partials and runs the RMSNorm backward on its own rows.
#
# Buffer reuse across steps is safe without extra barriers: a rank can only start step i+1's publish after its own step-i
# reduce, which waited for every peer's rs_done flag, which each peer raises after its step-i GEMMs (the pulls included).
# The step counter ("epoch") belongs to the BUFFERS, not to a block: any number of blocks (one per layer) may share one
# buffer set, every forward or backward pass through any of them is one more epoch.
# ======================================================================================================================
FLAG_READY, FLAG_RS_DONE, NUM_FLAGS = 0, 8, 64


class TpRankBuffers:
    """Buffers of one rank of the fused path plus the addresses of every rank's buffers (entry [rank] = own).
    `normed` is the exchange buffer (normalised activations in forward, dY in backward); `epoch` counts the passes."""

    def __init__(self, rank, world, max_tokens, hidden, normed, slots, flags, peer_normed, peer_slots_base, peer_flags,
                 group=None):
        self.rank, self.world, self.max_tokens, self.hidden = rank, world, max_tokens, hidden
        self.slot_rows = slots.shape[1]
        self.normed, self.slots, self.flags = normed, slots, flags
        self.done = torch.zeros(8, dtype=torch.int32, device=normed.device)
        self.peer_normed = list(peer_normed)
        self.peer_flags = list(peer_flags)
        self.group = group
        self.epoch = 0
        slot_bytes = self.slot_rows * hidden * normed.element_size()
        # where THIS rank's partial for owner o lands: slot [rank] of rank o's slots buffer
        self.peer_slots = [int(base) + rank * slot_bytes for base in peer_slots_base]

    def next_epoch(self) -> int:
        """One more pass (forward or backward, of whichever block) through these buffers.  Every rank calls this the same
        number of times in the same order, so the counters agree without communication."""
        self.epoch += 1
        return self.epoch

    @staticmethod
    def slot_rows_for(max_tokens, world):
        return -(-max_tokens // world)

    @classmethod
    def symmetric(cls, max_tokens, hidden, dtype, device, group=None):
        """Allocate the three buffers as symmetric memory and exchange the peer mappings (one process per GPU)."""
        import torch.distributed._symmetric_memory as symm
        group = group if group is not None else dist.group.WORLD
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        rows = cls.slot_rows_for(max_tokens, world)
        normed = symm.empty(max_tokens, hidden, dtype=dtype, device=device)
        slots = symm.empty(world, rows, hidden, dtype=dtype, device=device)
        flags = symm.empty(NUM_FLAGS, dtype=torch.int32, device=device)
        flags.zero_()
        hn, hs, hf = (symm.rendezvous(t, group) for t in (normed, slots, flags))
        torch.cuda.synchronize(device)
        dist.barrier(group)   # every rank's flags are zero before anybody can signal
        bufs = cls(rank, world, max_tokens, hidden, normed, slots, flags, hn.buffer_ptrs, hs.buffer_ptrs, hf.buffer_ptrs,
                   group=group)
        bufs._handles = (hn, hs, hf)   # keep the mappings alive
        return bufs

    @classmethod
    def local_world(cls, world, max_tokens, hidden, dtype, device):
        """All ranks' buffers on ONE device, cross-wired with plain pointers: the single-GPU emulation used by the
        tests (the ranks' phases are then run one after another, never concurrently)."""
        rows = cls.slot_rows_for(max_tokens, world)
        normed = [torch.zeros(max_tokens, hidden, dtype=dtype, device=device) for _ in range(world)]
        slots = [torch.zeros(world, rows, hidden, dtype=dtype, device=device) for _ in range(world)]
        flags = [torch.zeros(NUM_FLAGS, dtype=torch.int32, device=device) for _ in range(world)]
        return [cls(r, world, max_tokens, hidden, normed[r], slots[r], flags[r], [t.data_ptr() for t in normed],
                    [t.data_ptr() for t in slots], [t.data_ptr() for t in flags]) for r in range(world)]


class TpSaved:
    """What one training forward of a rank leaves for its backward."""
    __slots__ = ("tokens", "h", "rms", "x_full", "gate", "up", "dy_full", "d_gate", "d_up", "act", "has_residual")


class FusedTensorParallelBlock:
    """norm2(x, residual) -> feed-forward of one rank, collectives fused into the GEMM kernels (see above).
    Inference: forward().  Training: forward_train() / backward(), or `apply()` which wires both into autograd."""

    def __init__(self, gamma, eps, w_gate, w_up, w_down, bufs: TpRankBuffers, one_kernel: bool = False, presharded: bool = False):
        """gamma [H]; w_gate / w_up / w_down are the FULL matrices ([I,H], [I,H], [H,I]); the shard is taken here -- unless
        `presharded`: then they already are this rank's shard ([I/p,H], [I/p,H], [H,I/p], see shard_state_dict_for_rank).
        one_kernel: run gate/up and down as ONE persistent kernel (l32_tp_ffn_forward_fused) instead of two.  Measured
        at 8 GPUs (DESIGN.md section 6): equal within 2-5 % either way -- the two-kernel path already hides both
        collectives -- so the simpler two-kernel path is the default."""
        self.bufs = bufs
        self.one_kernel = one_kernel
        self.eps = eps
        self.gamma = gamma
        if presharded:
            wg, wu, wd = w_gate, w_up, w_down.contiguous()
        else:
            wg, wu, wd = shard_ffn_weights(w_gate, w_up, w_down, bufs.world, bufs.rank)
        self.w_gate, self.w_up, self.w_down = wg.contiguous(), wu.contiguous(), wd
        self._epoch = 0
        self._act = None

    @property
    def epoch(self):
        """Epoch of the pass this block is currently in (the counter itself lives in the shared buffers)."""
        return self._epoch

    def rows_of(self, tokens, rank=None):
        rank = self.bufs.rank if rank is None else rank
        per = -(-tokens // self.bufs.world)
        lo = min(rank * per, tokens)
        return lo, min(lo + per, tokens), per

    def _check_tokens(self, tokens):
        if tokens > self.bufs.max_tokens:
            raise ValueError(f"tokens {tokens} exceeds the buffers' capacity {self.bufs.max_tokens}")

    # -- the four forward phases (run back to back by forward(); the single-GPU emulation interleaves them across ranks)
    def phase_norm(self, x_local, residual_local, tokens, saved: TpSaved | None = None):
        b = self.bufs
        self._epoch = b.next_epoch()
        lo, hi, _ = self.rows_of(tokens)
        if hi > lo:
            train = saved is not None
            _, rms, h = ops.add_rmsnorm_forward(x_local, self.gamma, residual_local, self.eps, want_h=train, want_rms=train,
                                                out=b.normed[lo:hi])
            if train:
                saved.h, saved.rms = (h if h is not None else x_local), rms
        if saved is not None:
            saved.tokens, saved.has_residual = tokens, residual_local is not None
        ops.tp_signal(b.peer_flags, FLAG_READY + b.rank, self._epoch, b.normed.device, zero8=b.done)

    def phase_gate_up(self, tokens, saved: TpSaved | None = None):
        b = self.bufs
        _, _, per = self.rows_of(tokens)
        ready = b.flags[FLAG_READY:FLAG_READY + 8]
        if saved is None:
            self._act = ops.tp_swiglu_forward_allgather(b.normed[:tokens], b.peer_normed, ready, b.done, self._epoch, b.rank,
                                                        per, self.w_gate, self.w_up)
            return
        # training: gather into a tensor of its own (the exchange buffer is recycled by the next pass) and keep the caches
        if b.world > 1:
            saved.x_full = torch.empty(tokens, b.hidden, dtype=b.normed.dtype, device=b.normed.device)
        else:
            saved.x_full = b.normed[:tokens].clone()
        x_arg = saved.x_full if b.world > 1 else b.normed[:tokens]
        self._act, saved.gate, saved.up = ops.tp_swiglu_forward_allgather(x_arg, b.peer_normed, ready, b.done, self._epoch,
                                                                          b.rank, per, self.w_gate, self.w_up, want_cache=True)

    def phase_down(self, tokens):
        b = self.bufs
        _, _, per = self.rows_of(tokens)
        ops.tp_linear_forward_reduce_scatter(self._act, self.w_down, b.peer_slots, b.rank, per)
        self._act = None
        ops.tp_signal(b.peer_flags, FLAG_RS_DONE + b.rank, self._epoch, b.normed.device)

    def phase_ffn(self, tokens):
        """phase_gate_up + phase_down as one persistent kernel, then the rs_done signal."""
        b = self.bufs
        _, _, per = self.rows_of(tokens)
        ops.tp_ffn_forward_fused(b.normed[:tokens], b.peer_normed, b.flags[FLAG_READY:FLAG_READY + 8], b.done, self._epoch,
                                 b.rank, per, self.w_gate, self.w_up, self.w_down, b.peer_slots)
        ops.tp_signal(b.peer_flags, FLAG_RS_DONE + b.rank, self._epoch, b.normed.device)

    def phase_reduce(self, tokens, addend=None):
        b = self.bufs
        lo, hi, _ = self.rows_of(tokens)
        return ops.tp_reduce_partials(b.slots, b.flags[FLAG_RS_DONE:FLAG_RS_DONE + 8], self._epoch, b.rank, hi - lo, addend=addend)

    def forward(self, x_local, residual_local, tokens, addend=None):
        """x_local / residual_local: this rank's rows [rows_local, H]; returns this rank's rows of the FFN output."""
        self._check_tokens(tokens)
        self.phase_norm(x_local, residual_local, tokens)
        if self.one_kernel:
            self.phase_ffn(tokens)
        else:
            self.phase_gate_up(tokens)
            self.phase_down(tokens)
        return self.phase_reduce(tokens, addend)

    # -- training: forward that keeps what the backward needs, and the backward phases
    def forward_train(self, x_local, residual_local, tokens):
        """Like forward(); also returns the TpSaved record for backward()."""
        self._check_tokens(tokens)
        saved = TpSaved()
        self.phase_norm(x_local, residual_local, tokens, saved)
        self.phase_gate_up(tokens, saved)
        self.phase_down(tokens)
        return self.phase_reduce(tokens), saved

    def bwd_phase_publish(self, dy_local, saved: TpSaved):
        """Own rows of dY into the exchange buffer + ready signal (a new epoch)."""
        b = self.bufs
        self._epoch = b.next_epoch()
        lo, hi, _ = self.rows_of(saved.tokens)
        if hi > lo:
            b.normed[lo:hi].copy_(dy_local.reshape(hi - lo, b.hidden))
        ops.tp_signal(b.peer_flags, FLAG_READY + b.rank, self._epoch, b.normed.device, zero8=b.done)

    def bwd_phase_dact(self, saved: TpSaved, want_dw_down=True):
        """d_act = dY w_down_shard with the all-gather of dY pulled in; SiLU' recomputed in the epilogue."""
        b = self.bufs
        tokens = saved.tokens
        _, _, per = self.rows_of(tokens)
        if b.world > 1:
            saved.dy_full = torch.empty(tokens, b.hidden, dtype=b.normed.dtype, device=b.normed.device)
            dy_arg = saved.dy_full
        else:
            dy_arg = b.normed[:tokens]
            saved.dy_full = dy_arg
        saved.d_gate, saved.d_up, saved.act = ops.tp_ffn_backward_dact_allgather(
            dy_arg, b.peer_normed, b.flags[FLAG_READY:FLAG_READY + 8], b.done, self._epoch, b.rank, per, self.w_down,
            saved.gate, saved.up, want_act=want_dw_down)

    def bwd_phase_dx(self, saved: TpSaved):
        """Partial dX = d_gate Wg_shard + d_up Wu_shard, rows pushed to their owners; then the rs_done signal."""
        b = self.bufs
        _, _, per = self.rows_of(saved.tokens)
        ops.tp_ffn_backward_dx_reduce_scatter(saved.d_gate, saved.d_up, self.w_gate, self.w_up, b.peer_slots, b.rank, per)
        ops.tp_signal(b.peer_flags, FLAG_RS_DONE + b.rank, self._epoch, b.normed.device)

    def bwd_phase_wgrads(self, saved: TpSaved, want_gate_up=True, want_down=True):
        """Weight gradients of the shard: local MN-major x MN-major GEMMs (they run while the peers' partial dX rows are
        still in flight).  Returns (dw_gate [I/p,H], dw_up [I/p,H], dw_down [H,I/p])."""
        dwg = dwu = dwd = None
        if want_gate_up:
            dwg = ops.gemm(saved.d_gate, saved.x_full, a_mn_major=True, b_mn_major=True)
            dwu = ops.gemm(saved.d_up, saved.x_full, a_mn_major=True, b_mn_major=True)
        if want_down:
            dwd = ops.gemm(saved.dy_full, saved.act, a_mn_major=True, b_mn_major=True)
        return dwg, dwu, dwd

    def bwd_phase_reduce_norm(self, saved: TpSaved, want_dgamma=True):
        """Sum of the dX partials of the own rows, then the RMSNorm backward on them.  Returns (dx_local, dgamma) where
        dgamma covers the OWN rows only (sum it over the ranks: `allreduce_dgamma`); d_residual == dx_local."""
        b = self.bufs
        lo, hi, _ = self.rows_of(saved.tokens)
        d_normed = ops.tp_reduce_partials(b.slots, b.flags[FLAG_RS_DONE:FLAG_RS_DONE + 8], self._epoch, b.rank, hi - lo)
        if hi <= lo:
            return d_normed, (torch.zeros_like(self.gamma) if want_dgamma else None)
        return ops.rmsnorm_backward(d_normed, saved.h, self.gamma, saved.rms, want_dweight=want_dgamma)

    def allreduce_dgamma(self, dgamma):
        """gamma is replicated, its gradient is the sum over the ranks' rows (fp32 on the wire; [H] elements)."""
        b = self.bufs
        if b.world > 1 and b.group is not None:
            g32 = dgamma.float()
            dist.all_reduce(g32, group=b.group)
            return g32.to(dgamma.dtype)
        return dgamma

    def backward(self, dy_local, saved: TpSaved, want_dw_gate_up=True, want_dw_down=True, want_dgamma=True):
        """Returns (dx_local, dgamma, dw_gate_shard, dw_up_shard, dw_down_shard)."""
        self.bwd_phase_publish(dy_local, saved)
        self.bwd_phase_dact(saved, want_dw_down)
        self.bwd_phase_dx(saved)
        dwg, dwu, dwd = self.bwd_phase_wgrads(saved, want_dw_gate_up, want_dw_down)
        dx, dgamma = self.bwd_phase_reduce_norm(saved, want_dgamma)
        if dgamma is not None:
            dgamma = self.allreduce_dgamma(dgamma)
        return dx, dgamma, dwg, dwu, dwd

    def apply(self, x_local, residual_local, tokens):
        """Autograd-aware call: y_local = block(x_local, residual_local).  Gradients flow to x_local, residual_local and to
        self.gamma / self.w_gate / self.w_up / self.w_down when they require grad (make them leaf tensors or Parameters)."""
        tensors = (x_local, residual_local, self.gamma, self.w_gate, self.w_up, self.w_down)
        if not (torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)):
            return self.forward(x_local, residual_local, tokens)
        return _TpBlockFunction.apply(self, tokens, x_local, residual_local, self.gamma, self.w_gate, self.w_up, self.w_down)


class _TpBlockFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, block, tokens, x_local, residual_local, gamma, w_gate, w_up, w_down):
        y, saved = block.forward_train(x_local.detach(), None if residual_local is None else residual_local.detach(), tokens)
        ctx.block, ctx.saved_rec = block, saved
        return y

    @staticmethod
    def backward(ctx, dy_local):
        blk, saved = ctx.block, ctx.saved_rec
        _, _, nx, nr, ng, nwg, nwu, nwd = ctx.needs_input_grad
        dx, dgamma, dwg, dwu, dwd = blk.backward(dy_local.contiguous(), saved, want_dw_gate_up=(nwg or nwu), want_dw_down=nwd,
                                                 want_dgamma=ng)
        ctx.saved_rec = None
        d_res = dx if (nr and saved.has_residual) else None
        return None, None, (dx if nx else None), d_res, dgamma, (dwg if nwg else None), (dwu if nwu else None), dwd


# ======================================================================================================================
# Tensor-parallel attention: norm1 + GroupQueryAttention (reference Model/model.py:238-253, 267-268) with the heads sharded
# by KV group, on the same buffers and flags as the feed-forward block above.  Rank r owns query heads [r H/p, (r+1) H/p)
# and KV heads [r kv/p, (r+1) kv/p), so the GQA group never crosses ranks and the attention itself is local:
#
#   1. RMSNorm of the own rows into the own `normed` buffer                                 -> ready[r] = epoch everywhere
#   2. q / k / v of the rank's heads: ONE grouped GEMM (three problems, one tile loop) that pulls the other ranks' normed
#      rows out of peer memory while it works on the rows already there (fused all-gather)
#   3. RoPE + K/V store (the rank's own KVCache, local KV heads only) and the flash attention kernel on the local heads
#   4. out_proj on the rank's columns: a PARTIAL [tokens, hidden]; the epilogue pushes every row to its owner's slot
#                                                                                            -> rs_done[r] = epoch everywhere
#   5. the owner sums the slots of its rows                                                  -> attn_out rows of rank r
#
# Backward: dY rows published (new epoch); d_ctx = dY_full out_proj_r with the all-gather of dY pulled in; the attention
# backward on the local heads gives dq, dk, dv before RoPE; ONE three-phase GEMM forms the partial dX = dq Wq_r + dk Wk_r +
# dv Wv_r and pushes its rows to their owners; the weight gradients of the shard are local GEMMs; the owner sums the
# partials and runs the RMSNorm backward of its rows.
# ======================================================================================================================
def rows_of(tokens, world, rank):
    """(lo, hi, rows_per_rank): the token rows rank `rank` owns in the sequence-parallel layout (possibly none)."""
    per = -(-tokens // world)
    lo = min(rank * per, tokens)
    return lo, min(lo + per, tokens), per


class TpAttnSaved:
    """What one training forward of a rank's attention block leaves for its backward."""
    __slots__ = ("tokens", "batch", "h", "rms", "x_full", "q_rot", "ck", "cv", "ctx", "lse", "pos", "causal", "keep", "dy_full",
                 "d_ctx", "dq", "dk", "dv")


class FusedTensorParallelAttention:
    """norm1(x) -> GroupQueryAttention of one rank's heads, collectives fused into the GEMM kernels (see above).  The
    attention core is the single-GPU module's: tcgen05 flash forward / backward, RoPE at absolute positions, masks as
    `_mask_causal_keep` reads the reference's 4-D mask (causal + key padding; None = no masking).
    Inference: forward().  Training: forward_train() / backward(), or `apply()` which wires both into autograd."""

    def __init__(self, gamma1, eps, wq, wk, wv, wo, n_heads, n_kv, bufs: TpRankBuffers, rope_base=500000.0,
                 presharded: bool = False):
        """gamma1 [hidden]; wq / wk / wv / wo are the FULL nn.Linear weights ([H d, hidden], [kv d, hidden] x 2, [hidden, H d]);
        the shard is taken here -- unless `presharded`: then they already are this rank's (shard_state_dict_for_rank with
        the head counts).  Raises ValueError unless n_kv % world == 0."""
        (qlo, qhi), (klo, khi) = attention_head_range(n_heads, n_kv, bufs.world, bufs.rank)
        self.bufs, self.eps, self.gamma, self.rope_base = bufs, eps, gamma1, float(rope_base)
        self.heads, self.kv_heads = qhi - qlo, khi - klo
        if presharded:
            wq_r, wk_r, wv_r, wo_r = wq, wk, wv, wo.contiguous()
        else:
            wq_r, wk_r, wv_r, wo_r = shard_attention_weights(wq, wk, wv, wo, n_heads, n_kv, bufs.world, bufs.rank)
        self.wq, self.wk, self.wv, self.wo = wq_r.contiguous(), wk_r.contiguous(), wv_r.contiguous(), wo_r
        self.head_dim = self.wq.shape[0] // self.heads
        if self.wk.shape[0] != self.kv_heads * self.head_dim or self.wo.shape != (bufs.hidden, self.heads * self.head_dim):
            raise ValueError(f"attention shard shapes do not match {self.heads} query / {self.kv_heads} KV heads of "
                             f"{self.head_dim}: wk {tuple(self.wk.shape)}, wo {tuple(self.wo.shape)}")
        self._epoch = 0
        self._qkv = None
        self._ctx = None

    @property
    def epoch(self):
        """Epoch of the pass this block is currently in (the counter itself lives in the shared buffers)."""
        return self._epoch

    def rows_of(self, tokens, rank=None):
        return rows_of(tokens, self.bufs.world, self.bufs.rank if rank is None else rank)

    @staticmethod
    def _positions(position_ids, device):
        if position_ids.dim() != 2:
            raise ValueError("position_ids must be [batch, q_len]: the batch shape is what splits the token rows into sequences")
        return position_ids.to(device=device, dtype=torch.int64).contiguous()

    # -- forward phases (run back to back by forward(); the single-GPU emulation interleaves them across ranks)
    def phase_norm(self, x_local, tokens, saved: TpAttnSaved | None = None):
        b = self.bufs
        if tokens > b.max_tokens:
            raise ValueError(f"tokens {tokens} exceeds the buffers' capacity {b.max_tokens}")
        self._epoch = b.next_epoch()
        lo, hi, _ = self.rows_of(tokens)
        if hi > lo:
            train = saved is not None
            _, rms, _ = ops.add_rmsnorm_forward(x_local, self.gamma, None, self.eps, want_rms=train, out=b.normed[lo:hi])
            if train:
                saved.h, saved.rms = x_local, rms
        if saved is not None:
            saved.tokens = tokens
        ops.tp_signal(b.peer_flags, FLAG_READY + b.rank, self._epoch, b.normed.device, zero8=b.done)

    def phase_qkv(self, tokens, saved: TpAttnSaved | None = None):
        b = self.bufs
        _, _, per = self.rows_of(tokens)
        x_arg = b.normed[:tokens]
        if saved is not None:
            # training: gather into a tensor of its own (the exchange buffer is recycled by the next pass), the input of dW
            saved.x_full = torch.empty_like(x_arg) if b.world > 1 else x_arg.clone()
            if b.world > 1:
                x_arg = saved.x_full
        self._qkv = ops.tp_linear_group_forward_allgather(x_arg, b.peer_normed, b.flags[FLAG_READY:FLAG_READY + 8], b.done,
                                                          self._epoch, b.rank, per, [self.wq, self.wk, self.wv])

    def phase_attention(self, position_ids, attention_mask=None, kv_cache: KVCache | None = None, layer_idx: int = 0,
                        saved: TpAttnSaved | None = None):
        q, k, v = self._qkv
        self._qkv = None
        pos = self._positions(position_ids, q.device)
        bsz, t = pos.shape
        q, k, v = q.view(bsz, t, -1), k.view(bsz, t, -1), v.view(bsz, t, -1)
        d = self.head_dim
        if saved is None:
            cache = kv_cache if kv_cache is not None else KVCache()
            layer = layer_idx if kv_cache is not None else 0
            past = cache.length(layer)
            ck, cv, _ = cache.reserve(layer, bsz, self.kv_heads, d, past + t, q.dtype, q.device)
            ops.rope_kv_append(q, k, v, pos, ck, cv, past, self.rope_base)
            cache.advance(layer, t)
            causal, keep = _mask_causal_keep(attention_mask, bsz, t, past + t)
            ctx = ops.gqa_attention_forward(q, ck, cv, past + t, past, causal=causal, key_keep=keep)
        else:
            if kv_cache is not None:
                raise ValueError("tensor-parallel attention trains without a KV cache")
            ck = torch.empty(bsz, self.kv_heads, t, d, dtype=q.dtype, device=q.device)
            cv = torch.empty_like(ck)
            ops.rope_kv_append(q, k, v, pos, ck, cv, 0, self.rope_base)     # q is this call's own tensor: rotated in place
            causal, keep = _mask_causal_keep(attention_mask, bsz, t, t)
            if keep is not None:
                keep = keep.to(torch.uint8).contiguous()
            ctx, lse = ops.gqa_attention_forward_train(q, ck, cv, causal, keep)
            saved.batch, saved.q_rot, saved.ck, saved.cv, saved.ctx, saved.lse = bsz, q, ck, cv, ctx, lse
            saved.pos, saved.causal, saved.keep = pos, causal, keep
        self._ctx = ctx.view(bsz * t, -1)

    def phase_out(self, tokens):
        b = self.bufs
        _, _, per = self.rows_of(tokens)
        ops.tp_linear_forward_reduce_scatter(self._ctx, self.wo, b.peer_slots, b.rank, per)
        self._ctx = None
        ops.tp_signal(b.peer_flags, FLAG_RS_DONE + b.rank, self._epoch, b.normed.device)

    def phase_reduce(self, tokens, addend=None):
        b = self.bufs
        lo, hi, _ = self.rows_of(tokens)
        return ops.tp_reduce_partials(b.slots, b.flags[FLAG_RS_DONE:FLAG_RS_DONE + 8], self._epoch, b.rank, hi - lo, addend=addend)

    def forward(self, x_local, position_ids, attention_mask=None, kv_cache: KVCache | None = None, layer_idx: int = 0):
        """x_local: this rank's rows [rows_local, hidden] of the [batch * q_len] token rows; position_ids [batch, q_len]
        (absolute positions); kv_cache: this rank's own cache (it holds the local KV heads only).  Returns this rank's rows
        of the attention output (out_proj summed over all ranks' heads)."""
        tokens = position_ids.numel()
        self.phase_norm(x_local, tokens)
        self.phase_qkv(tokens)
        self.phase_attention(position_ids, attention_mask, kv_cache, layer_idx)
        self.phase_out(tokens)
        return self.phase_reduce(tokens)

    # -- training
    def forward_train(self, x_local, position_ids, attention_mask=None):
        """Like forward() without a cache; also returns the TpAttnSaved record for backward()."""
        tokens = position_ids.numel()
        saved = TpAttnSaved()
        self.phase_norm(x_local, tokens, saved)
        self.phase_qkv(tokens, saved)
        self.phase_attention(position_ids, attention_mask, saved=saved)
        self.phase_out(tokens)
        return self.phase_reduce(tokens), saved

    def bwd_phase_publish(self, dy_local, saved: TpAttnSaved):
        """Own rows of d(attn_out) into the exchange buffer + ready signal (a new epoch)."""
        b = self.bufs
        self._epoch = b.next_epoch()
        lo, hi, _ = self.rows_of(saved.tokens)
        if hi > lo:
            b.normed[lo:hi].copy_(dy_local.reshape(hi - lo, b.hidden))
        ops.tp_signal(b.peer_flags, FLAG_READY + b.rank, self._epoch, b.normed.device, zero8=b.done)

    def bwd_phase_dctx(self, saved: TpAttnSaved):
        """d_ctx = dY_full out_proj_r with the all-gather of dY pulled in (dY_full is kept for dW_out)."""
        b = self.bufs
        tokens = saved.tokens
        _, _, per = self.rows_of(tokens)
        saved.dy_full = torch.empty(tokens, b.hidden, dtype=b.normed.dtype, device=b.normed.device) if b.world > 1 else \
            b.normed[:tokens]
        saved.d_ctx = ops.tp_linear_forward_allgather(saved.dy_full, b.peer_normed, b.flags[FLAG_READY:FLAG_READY + 8], b.done,
                                                      self._epoch, b.rank, per, self.wo, w_mn_major=True)

    def bwd_phase_attention(self, saved: TpAttnSaved):
        """Attention backward of the local heads: dq, dk, dv of the projections (before RoPE)."""
        bsz = saved.batch
        t = saved.tokens // bsz
        dq, dk, dv = ops.gqa_attention_backward(saved.d_ctx.view(bsz, t, -1), saved.q_rot, saved.ck, saved.cv, saved.ctx, saved.lse,
                                                saved.pos, saved.causal, saved.keep, self.rope_base)
        saved.dq, saved.dk, saved.dv = dq.view(saved.tokens, -1), dk.view(saved.tokens, -1), dv.view(saved.tokens, -1)
        saved.d_ctx = saved.q_rot = saved.ck = saved.cv = saved.lse = None

    def bwd_phase_dx(self, saved: TpAttnSaved):
        """Partial dX = dq Wq_r + dk Wk_r + dv Wv_r (one three-phase GEMM), rows pushed to their owners; rs_done signal."""
        b = self.bufs
        _, _, per = self.rows_of(saved.tokens)
        ops.tp_linear_group_backward_dx_reduce_scatter([saved.dq, saved.dk, saved.dv], [self.wq, self.wk, self.wv], b.peer_slots,
                                                       b.rank, per)
        ops.tp_signal(b.peer_flags, FLAG_RS_DONE + b.rank, self._epoch, b.normed.device)

    def bwd_phase_wgrads(self, saved: TpAttnSaved, want_qkv=True, want_out=True):
        """Weight gradients of the shard (local MN-major x MN-major GEMMs, while the peers' partial dX rows are in flight).
        Returns (dwq [Hl d, hidden], dwk [KVl d, hidden], dwv, dwo [hidden, Hl d])."""
        dwq = dwk = dwv = dwo = None
        if want_qkv:
            dwq, dwk, dwv = (ops.gemm(g, saved.x_full, a_mn_major=True, b_mn_major=True) for g in (saved.dq, saved.dk, saved.dv))
        if want_out:
            dwo = ops.gemm(saved.dy_full, saved.ctx.view(saved.tokens, -1), a_mn_major=True, b_mn_major=True)
        return dwq, dwk, dwv, dwo

    def bwd_phase_reduce_norm(self, saved: TpAttnSaved, want_dgamma=True):
        """Sum of the dX partials of the own rows, then the RMSNorm backward on them.  Returns (dx_local, dgamma of the OWN
        rows -- sum it over the ranks: `allreduce_dgamma`)."""
        b = self.bufs
        lo, hi, _ = self.rows_of(saved.tokens)
        d_normed = ops.tp_reduce_partials(b.slots, b.flags[FLAG_RS_DONE:FLAG_RS_DONE + 8], self._epoch, b.rank, hi - lo)
        if hi <= lo:
            return d_normed, (torch.zeros_like(self.gamma) if want_dgamma else None)
        return ops.rmsnorm_backward(d_normed, saved.h, self.gamma, saved.rms, want_dweight=want_dgamma)

    allreduce_dgamma = FusedTensorParallelBlock.allreduce_dgamma

    def backward(self, dy_local, saved: TpAttnSaved, want_dw_qkv=True, want_dw_out=True, want_dgamma=True):
        """Returns (dx_local, dgamma, dwq_shard, dwk_shard, dwv_shard, dwo_shard)."""
        self.bwd_phase_publish(dy_local, saved)
        self.bwd_phase_dctx(saved)
        self.bwd_phase_attention(saved)
        self.bwd_phase_dx(saved)
        dwq, dwk, dwv, dwo = self.bwd_phase_wgrads(saved, want_dw_qkv, want_dw_out)
        dx, dgamma = self.bwd_phase_reduce_norm(saved, want_dgamma)
        if dgamma is not None:
            dgamma = self.allreduce_dgamma(dgamma)
        return dx, dgamma, dwq, dwk, dwv, dwo

    def apply(self, x_local, position_ids, attention_mask=None):
        """Autograd-aware call without a cache: attn_out_local = block(x_local).  Gradients flow to x_local and to
        self.gamma / self.wq / self.wk / self.wv / self.wo when they require grad (make them leaf tensors or Parameters)."""
        tensors = (x_local, self.gamma, self.wq, self.wk, self.wv, self.wo)
        if not (torch.is_grad_enabled() and any(t.requires_grad for t in tensors)):
            return self.forward(x_local, position_ids, attention_mask)
        return _TpAttentionFunction.apply(self, position_ids, attention_mask, *tensors)


class _TpAttentionFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, block, position_ids, attention_mask, x_local, gamma, wq, wk, wv, wo):
        y, saved = block.forward_train(x_local.detach(), position_ids, attention_mask)
        ctx.block, ctx.saved_rec = block, saved
        return y

    @staticmethod
    def backward(ctx, dy_local):
        blk, saved = ctx.block, ctx.saved_rec
        _, _, _, nx, ng, nq, nk, nv, no = ctx.needs_input_grad
        dx, dgamma, dwq, dwk, dwv, dwo = blk.backward(dy_local.contiguous(), saved, want_dw_qkv=(nq or nk or nv), want_dw_out=no,
                                                      want_dgamma=ng)
        ctx.saved_rec = None
        return (None, None, None, (dx if nx else None), dgamma, (dwq if nq else None), (dwk if nk else None),
                (dwv if nv else None), dwo)


class TensorParallelDecoderLayer:
    """One decoder layer of the reference (TransformerBlock.forward, Model/model.py:265-273) fully tensor-parallel on ONE
    TpRankBuffers: attn_out = attention block(x); out = attn_out + ff(norm2(attn_out + x)) on this rank's rows (the residual
    is dropped from the output as in the reference, SURVEY.md section 0.6)."""

    def __init__(self, attn_block: FusedTensorParallelAttention, ffn_block: FusedTensorParallelBlock):
        if attn_block.bufs is not ffn_block.bufs:
            raise ValueError("the attention and feed-forward blocks of a layer must share one buffer set")
        self.attn, self.ffn = attn_block, ffn_block

    def forward(self, x_local, position_ids, attention_mask=None, kv_cache: KVCache | None = None, layer_idx: int = 0):
        """x_local: this rank's rows of the layer input; returns this rank's rows of the layer output."""
        attn_out = self.attn.forward(x_local, position_ids, attention_mask, kv_cache, layer_idx)
        return self.ffn.forward(attn_out, x_local, position_ids.numel(), addend=attn_out)

    def apply(self, x_local, position_ids, attention_mask=None):
        """Autograd-aware call (no cache) through both blocks' apply()."""
        attn_out = self.attn.apply(x_local, position_ids, attention_mask)
        return attn_out + self.ffn.apply(attn_out, x_local, position_ids.numel())
