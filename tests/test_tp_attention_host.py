"""CPU: sharding logic of the tensor-parallel attention (head ranges, weight shards, the state-dict cutter), an fp32
restatement of the sharded computation against the oracle, and argument validation of the new C entry points (every
call here fails validation or is empty, so nothing touches a device)."""
import ctypes
import os

import pytest
import torch

from llama32_b200 import _lib
from llama32_b200.tp import attention_head_range, shard_attention_weights, shard_state_dict_for_rank
from oracle import ffn_oracle as O

BF16 = 0


@pytest.mark.parametrize("n_heads,n_kv", [(32, 8), (64, 8)])
@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_head_ranges_keep_gqa_groups_on_one_rank(n_heads, n_kv, world):
    group = n_heads // n_kv
    q_seen, kv_seen = [], []
    for rank in range(world):
        (qlo, qhi), (klo, khi) = attention_head_range(n_heads, n_kv, world, rank)
        assert qhi - qlo == n_heads // world and khi - klo == n_kv // world
        assert {h // group for h in range(qlo, qhi)} == set(range(klo, khi))
        q_seen += range(qlo, qhi)
        kv_seen += range(klo, khi)
    assert q_seen == list(range(n_heads)) and kv_seen == list(range(n_kv))


@pytest.mark.parametrize("n_heads,n_kv,world", [(32, 8, 3), (64, 8, 16), (24, 6, 4), (12, 3, 2)])
def test_kv_heads_not_divisible_by_world_raise(n_heads, n_kv, world):
    with pytest.raises(ValueError):
        attention_head_range(n_heads, n_kv, world, 0)
    w = torch.zeros(n_heads * 8, 16)
    with pytest.raises(ValueError):
        shard_attention_weights(w, w[: n_kv * 8], w[: n_kv * 8], w.t(), n_heads, n_kv, world, 0)


@pytest.mark.parametrize("n_heads,n_kv,world", [(8, 4, 4), (6, 3, 3), (8, 2, 2), (4, 4, 1)])
def test_sharded_attention_sums_to_the_oracle(n_heads, n_kv, world):
    """sum over ranks of (attention over the rank's heads) . out_proj shard^T == the full attention (fp32)."""
    b, t, d = 2, 11, 16
    hidden = n_heads * d
    g = torch.Generator().manual_seed(n_heads * 10 + world)
    x = torch.randn(b, t, hidden, generator=g)
    wq = torch.randn(n_heads * d, hidden, generator=g) / hidden ** 0.5
    wk = torch.randn(n_kv * d, hidden, generator=g) / hidden ** 0.5
    wv = torch.randn(n_kv * d, hidden, generator=g) / hidden ** 0.5
    wo = torch.randn(hidden, n_heads * d, generator=g) / hidden ** 0.5
    pos = torch.arange(t)[None].expand(b, t)
    keep = torch.ones(b, t)
    keep[1, :4] = 0                                    # left padding of the second sequence
    mask = O.causal_padding_mask(keep, t)
    ref, _, _ = O.gqa_attention(x, wq, wk, wv, wo, n_heads, n_kv, pos, mask)
    total = torch.zeros_like(ref)
    for rank in range(world):
        wq_r, wk_r, wv_r, wo_r = shard_attention_weights(wq, wk, wv, wo, n_heads, n_kv, world, rank)
        part, _, _ = O.gqa_attention(x, wq_r, wk_r, wv_r, wo_r, n_heads // world, n_kv // world, pos, mask)
        total += part
    torch.testing.assert_close(total, ref, rtol=1e-5, atol=1e-5)


def test_state_dict_cutter_with_and_without_head_counts():
    n_heads, n_kv, d, hidden, inter, world = 8, 4, 4, 32, 256, 2
    g = torch.Generator().manual_seed(1)
    state = {
        "layers.0.att.W_query.weight": torch.randn(n_heads * d, hidden, generator=g),
        "layers.0.att.W_key.weight": torch.randn(n_kv * d, hidden, generator=g),
        "layers.0.att.W_value.weight": torch.randn(n_kv * d, hidden, generator=g),
        "layers.0.att.out_proj.weight": torch.randn(hidden, n_heads * d, generator=g),
        "layers.0.ff.swiglu.w_gate": torch.randn(inter, hidden, generator=g),
        "layers.0.ff.w_down.weight": torch.randn(hidden, inter, generator=g),
        "layers.0.norm1.weight": torch.randn(hidden, generator=g),
    }
    plain = shard_state_dict_for_rank(state, world, 1)
    for k in ("W_query", "W_key", "W_value", "out_proj"):
        name = f"layers.0.att.{k}.weight"
        assert plain[name] is state[name]              # without the head counts the attention passes through
    assert plain["layers.0.ff.swiglu.w_gate"].shape == (inter // world, hidden)
    for rank in range(world):
        cut = shard_state_dict_for_rank(state, world, rank, n_heads=n_heads, n_kv=n_kv)
        ref = shard_attention_weights(*(state[f"layers.0.att.{k}.weight"] for k in ("W_query", "W_key", "W_value", "out_proj")),
                                      n_heads, n_kv, world, rank)
        for k, r in zip(("W_query", "W_key", "W_value", "out_proj"), ref):
            got = cut[f"layers.0.att.{k}.weight"]
            assert got.is_contiguous() and torch.equal(got, r)
        assert torch.equal(cut["layers.0.ff.swiglu.w_gate"], plain["layers.0.ff.swiglu.w_gate"]) or rank != 1
        assert cut["layers.0.norm1.weight"] is state["layers.0.norm1.weight"]
    with pytest.raises(ValueError):
        shard_state_dict_for_rank(state, 8, 0, n_heads=n_heads, n_kv=n_kv)


# ---------------------------------------------------------------------------------------------- C-ABI validation
@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _lib.lib()


P = ctypes.c_void_p


def _arr(ctype, vals):
    return (ctype * len(vals))(*vals)


def _group_fwd(lib, x=256, w=(256, 256, 256), y=(256, 256, 256), outs=(128, 64, 64), count=3, rank=0, world=2, rpr=32, tokens=64,
               hidden=128, dtype=BF16, peers=(256, 512)):
    return lib.l32_tp_linear_group_forward_allgather(P(x), _arr(P, peers) if peers else None, P(256), P(256), 1, rank, world, rpr,
                                                     _arr(P, w) if w else None, _arr(P, y), _arr(ctypes.c_int, outs), count,
                                                     tokens, hidden, dtype, P(0))


def test_group_forward_allgather_validation(lib):
    assert _group_fwd(lib, dtype=7) == -1
    assert _group_fwd(lib, world=0) == -2
    assert _group_fwd(lib, world=9, rpr=8) == -2
    assert _group_fwd(lib, rank=2) == -2
    assert _group_fwd(lib, rank=-1) == -2
    assert _group_fwd(lib, rpr=16) == -2                 # rows_per_rank * world < tokens
    assert _group_fwd(lib, count=0) == -2
    assert _group_fwd(lib, count=4, w=(256,) * 4, y=(256,) * 4, outs=(64,) * 4) == -2
    assert _group_fwd(lib, outs=(128, 60, 64)) == -2      # output width not a multiple of 8
    assert _group_fwd(lib, w=None) == -4
    assert _group_fwd(lib, w=(256, 0, 256)) == -4
    assert _group_fwd(lib, y=(256, 256, 0)) == -4
    assert _group_fwd(lib, x=0) == -4
    assert _group_fwd(lib, x=0, tokens=0) == 0


def _fwd(lib, a=256, w=256, y=256, mn=1, rank=1, world=2, rpr=32, tokens=64, dtype=BF16):
    return lib.l32_tp_linear_forward_allgather(P(a), _arr(P, (256, 512)), P(256), P(256), 1, rank, world, rpr, P(w), mn, P(y),
                                               tokens, 128, 64, dtype, P(0))


def test_forward_allgather_validation(lib):
    assert _fwd(lib, dtype=2) == -1
    assert _fwd(lib, mn=2) == -2
    assert _fwd(lib, rank=2) == -2
    assert _fwd(lib, world=9) == -2
    assert _fwd(lib, w=0) == -4
    assert _fwd(lib, y=0) == -4
    assert _fwd(lib, a=0) == -4
    assert _fwd(lib, a=0, w=0, y=0, tokens=0) == 0


def _dx(lib, dy=(256, 256, 256), w=(256, 256, 256), k=(128, 64, 64), phases=3, slots=(256, 512), rank=0, world=2, rpr=32,
        tokens=64, hidden=128, dtype=BF16):
    return lib.l32_tp_linear_group_backward_dx_reduce_scatter(_arr(P, dy), _arr(P, w) if w else None, _arr(ctypes.c_int, k), phases,
                                                              _arr(P, slots) if slots else None, rank, world, rpr, tokens, hidden,
                                                              dtype, P(0))


def test_group_backward_dx_reduce_scatter_validation(lib):
    assert _dx(lib, dtype=9) == -1
    assert _dx(lib, phases=0) == -2
    assert _dx(lib, phases=4, dy=(256,) * 4, w=(256,) * 4, k=(64,) * 4) == -2
    assert _dx(lib, rank=3) == -2
    assert _dx(lib, world=0) == -2
    assert _dx(lib, k=(128, 0, 64)) == -2
    assert _dx(lib, hidden=100) == -2
    assert _dx(lib, w=None) == -4
    assert _dx(lib, dy=(256, 256, 0)) == -4
    assert _dx(lib, w=(0, 256, 256)) == -4
    assert _dx(lib, slots=None) == -4
    assert _dx(lib, slots=(256, 0)) == -4
    assert _dx(lib, dy=(0, 0, 0), tokens=0) == 0
