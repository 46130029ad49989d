"""CPU: speculative decoding's host side -- the restatement of the n-gram draft rule on hand-built histories, commit()'s
page accounting, fork with a token pool, SpeculativeDecoder's validation and the C argument checks of the new entry points
(no compute calls without a GPU)."""
import ctypes
import os
from types import SimpleNamespace

import pytest
import torch

import llama32_b200 as L
from llama32_b200 import _lib, ops
from spec_ref import accept, ngram_draft

PAGE = 64


# ------------------------------------------------------------------------------------------------ the draft rule
def test_draft_overlapping_match():
    # S = 1 2 1 2 1 | pending 2: suffix "1 2" (n=2) last occurs at j=2, proposal S[4:] = 1 2 (runs into the suffix)
    ids, n = ngram_draft([1, 2, 1, 2, 1], 2, 4, 1, 2)
    assert ids == [2, 1, 2, 2, 2] and n == 2


def test_draft_prefers_longest_n_then_latest_j():
    h = [5, 6, 7, 9, 6, 7, 8, 3, 6]
    # S = h + [7]: the suffix "6 7" occurs at j = 1 and j = 4; the latest, j = 4, proposes 8 3 6
    ids, n = ngram_draft(h, 7, 3, 1, 2)
    assert ids == [7, 8, 3, 6] and n == 3
    # n_max = 3: the suffix "3 6 7" never occurred before, so n = 2 decides
    assert ngram_draft(h, 7, 3, 1, 3) == ngram_draft(h, 7, 3, 1, 2)


def test_draft_cut_at_end_and_padded():
    ids, n = ngram_draft([4, 8, 4], 8, 5, 1, 3)        # S = 4 8 4 8: "4 8" at j=0 proposes S[2:4] = 4 8 (cut), pad 8
    assert ids == [8, 4, 8, 8, 8, 8] and n == 2


def test_draft_no_match_pads_with_pending():
    assert ngram_draft([1, 2, 3], 4, 3, 1, 3) == ([4, 4, 4, 4], 0)
    assert ngram_draft([], 9, 2, 1, 3) == ([9, 9, 9], 0)


@pytest.mark.parametrize("n_min", [1, 2, 3])
@pytest.mark.parametrize("n_max", [3, 4])
def test_draft_every_n_range(n_min, n_max):
    h = [1, 2, 3, 4, 0, 3, 4, 7, 2, 3, 4]
    ids, n = ngram_draft(h, 5, 2, n_min, n_max)        # S ends "3 4 5": 5 never occurred, so no n matches
    assert (ids, n) == ([5, 5, 5], 0)
    ids, n = ngram_draft(h, 0, 2, n_min, n_max)        # S ends "3 4 0", which occurred at j = 2: the proposal is 3 4
    assert ids == [0, 3, 4] and n == 2


def test_accept_rule():
    assert accept([7, 1, 2, 3], [1, 2, 9, 4], 4) == (3, [1, 2, 9])
    assert accept([7, 1, 2, 3], [5, 2, 3, 4], 4) == (1, [5])
    assert accept([7, 1, 2, 3], [1, 2, 3, 4], 4) == (4, [1, 2, 3, 4])
    assert accept([7, 1, 2, 3], [1, 2, 3, 4], 2) == (2, [1, 2])


# ------------------------------------------------------------------------------------------------ commit
@pytest.mark.parametrize("past", [0, 1, 60, 63, 64, 127])
def test_commit_page_accounting(past):
    new = 8
    for keep in range(new + 1):
        c = L.PagedKVCache(16, 4, 8)
        a = c.add_sequence()
        if past:
            c.set_batch([a], [past])
            c.advance()
        held = list(c.pages(a))
        free0 = c.free_pages
        c.set_batch([a], [new], verify=True)
        assert c.verify and not c.cascade
        assert len(c.pages(a)) == -(-(past + new) // PAGE)
        c.commit([keep])
        assert c.length(a) == past + keep
        want = max(len(held), -(-(past + keep) // PAGE))
        assert c.pages(a)[:len(held)] == held and len(c.pages(a)) == want
        assert c.free_pages == free0 - (want - len(held))
        assert all(c.refcount(p) == 1 for p in c.pages(a))
        assert sum(r == 0 for r in c._refs) == c.free_pages and len(set(c._free)) == c.free_pages
        assert c.batch_ids == []
        with pytest.raises(ValueError):
            c.commit([0])                                # the batch was dropped


def test_commit_rows_and_validation():
    c = L.PagedKVCache(16, 4, 8)
    a, b = c.add_sequence(), c.add_sequence()
    c.set_batch([a, b], [60, 70])
    c.advance()
    c.set_batch([a, b], [5, 0], verify=True)
    with pytest.raises(ValueError):
        c.commit([6, 0])
    with pytest.raises(ValueError):
        c.commit([1])
    c.commit([5, 0])
    assert (c.length(a), c.length(b)) == (65, 70)
    c.set_batch([a], [1])
    assert not c.verify                                 # a plain step again


# ------------------------------------------------------------------------------------------------ fork with a token pool
@pytest.mark.parametrize("n", [0, 63, 64, 65])
def test_fork_copies_the_partial_token_page(n):
    c = L.PagedKVCache(8, 4, 4)
    c._tokens = torch.arange(8 * PAGE, dtype=torch.int32).view(8, PAGE)   # the pool a CUDA cache creates in token_pool()
    a = c.add_sequence()
    if n:
        c.set_batch([a], [n])
        c.advance()
    before = c._tokens.clone()
    k = c.fork(a)
    full = n // PAGE
    assert c.pages(k)[:full] == c.pages(a)[:full]
    if n % PAGE:
        src, dst = c.pages(a)[full], c.pages(k)[full]
        assert src != dst and torch.equal(c._tokens[dst], before[src])
        others = [p for p in range(8) if p != dst]
        assert torch.equal(c._tokens[others], before[others])
    else:
        assert len(c.pages(k)) == full and torch.equal(c._tokens, before)


# ------------------------------------------------------------------------------------------------ decoder validation
def gqa_model(heads, kv):
    cfg = SimpleNamespace(hidden_size=heads * 64, n_heads=heads, n_kv_groups=kv)
    return torch.nn.ModuleList([L.GroupQueryAttention(cfg, 0)])


def test_decoder_validation():
    c = L.PagedKVCache(8, 4, 4)
    head = torch.nn.Linear(8, 16, bias=False)
    m = gqa_model(32, 8)                                 # group 4
    for k in (0, -1, 1.5, True, 32):                     # group * (k + 1) <= 128: k <= 31
        with pytest.raises(ValueError):
            L.SpeculativeDecoder(m, head, c, 4, k)
    for ng in ((0, 3), (3, 2), (1, ops.NGRAM_MAX + 1)):
        with pytest.raises(ValueError):
            L.SpeculativeDecoder(m, head, c, 4, 3, ngram=ng)
    for mb in (0, 5):
        with pytest.raises(ValueError):
            L.SpeculativeDecoder(m, head, c, mb, 3)
    with pytest.raises(ValueError):
        L.SpeculativeDecoder(gqa_model(64, 8), head, c, 4, 16)   # group 8: 8 * 17 > 128
    with pytest.raises(ValueError):
        L.SpeculativeDecoder(m, head, object(), 4, 3)
    if c.device is None:                                 # valid geometry, but this cache has no device
        with pytest.raises(ValueError, match="no CUDA device"):
            L.SpeculativeDecoder(m, head, c, 4, 31)
    assert ops.verify_fits(4, 32) and not ops.verify_fits(4, 33) and not ops.verify_fits(1, 2)


# ------------------------------------------------------------------------------------------------ C argument checks
@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _lib.lib()


def test_symbols_in_header_and_signatures():
    for n in ("l32_gqa_attention_forward_paged_verify", "l32_gqa_attention_verify_workspace_bytes", "l32_ngram_draft_paged",
              "l32_speculative_accept"):
        assert n in _lib.header_symbols() and n in _lib.SIGNATURES
    text = open(_lib.HEADER_PATH).read()
    assert "#define L32_VERIFY_TILE_ROWS 128" in text and f"#define L32_NGRAM_MAX {ops.NGRAM_MAX}" in text


def test_verify_argument_validation_without_device(lib):
    null, one = ctypes.c_void_p(0), ctypes.c_void_p(256)
    f = lambda ptrs, b, t, h, kv, d, pages=8, mp=4, mkv=256, dt=0, ws=0: lib.l32_gqa_attention_forward_paged_verify(
        *ptrs, ws, b, t, h, kv, d, pages, mp, mkv, dt, null)
    p8 = [one] * 8
    assert f(p8, 2, 4, 32, 8, 128, dt=2) == -1            # dtype
    assert f(p8, 2, 4, 8, 8, 128) == -2                   # group 1
    assert f(p8, 2, 33, 32, 8, 128) == -2                 # 4 * 33 > 128
    assert f(p8, 2, 17, 64, 8, 128) == -2                 # 8 * 17 > 128
    assert f(p8, 2, 4, 32, 8, 96) == -2                   # head_dim
    assert f(p8, 2, 4, 30, 8, 128) == -2                  # heads % kv_heads
    assert f(p8, -1, 4, 32, 8, 128) == -2
    assert f(p8, 2, 4, 32, 8, 128, mkv=257) == -2         # max_kv_len > max_pages * 64
    assert f(p8, 2, 4, 32, 8, 128, pages=0) == -2
    for i in (0, 1, 2, 3, 4, 6):                          # new_lens (5) and the workspace (7) may be null
        args = list(p8)
        args[i] = null
        assert f(args, 2, 4, 32, 8, 128) == -4, i
    args = list(p8)
    args[0] = ctypes.c_void_p(8)
    assert f(args, 2, 4, 32, 8, 128) == -3                # q not 16-byte aligned
    args = list(p8)
    args[7] = ctypes.c_void_p(8)
    assert f(args, 2, 4, 32, 8, 128) == -6                # workspace not 16-byte aligned
    assert f([null] * 8, 0, 4, 32, 8, 128) == 0           # empty batch
    assert f(p8, 2, 4, 32, 8, 128, mkv=-1) == -2
    assert f(p8, 2, 4, 32, 8, 128, mp=0) == -2            # no table columns
    args = list(p8)
    args[6] = ctypes.c_void_p(8)
    assert f(args, 2, 4, 32, 8, 128) == -3                # ctx not 16-byte aligned
    # a call with several faults gets the code of the first check: dtype, shape, empty batch, nulls, alignment, workspace
    assert f([null] * 8, 0, 4, 32, 8, 128, dt=2) == -1
    assert f([null] * 8, 2, 4, 32, 8, 128, mkv=257) == -2
    assert f([null] * 8, 2, 33, 32, 8, 128) == -2
    assert f([ctypes.c_void_p(8), one, one, null, one, one, one, one], 2, 4, 32, 8, 128) == -4
    assert f([ctypes.c_void_p(8)] + p8[1:7] + [ctypes.c_void_p(8)], 2, 4, 32, 8, 128) == -3
    assert lib.l32_gqa_attention_verify_workspace_bytes(2, 33, 32, 8, 128, 4096) == 0


def test_draft_and_accept_argument_validation_without_device(lib):
    null, one = ctypes.c_void_p(0), ctypes.c_void_p(256)
    d = lambda ptrs, b=2, k=4, n0=1, n1=3, pages=8, mp=4: lib.l32_ngram_draft_paged(*ptrs, b, k, n0, n1, pages, mp, null)
    p6 = [one] * 6
    for kw in (dict(k=0), dict(n0=0), dict(n0=3, n1=2), dict(n1=ops.NGRAM_MAX + 1), dict(b=-1), dict(pages=0), dict(mp=0)):
        assert d(p6, **kw) == -2, kw
    for i in range(5):                                    # draft_len (5) may be null
        args = list(p6)
        args[i] = null
        assert d(args) == -4, i
    assert d([null] * 6, b=0) == 0
    a = lambda ptrs, b=2, w=5, pages=8, mp=4: lib.l32_speculative_accept(*ptrs, b, w, pages, mp, null)
    p7 = [one] * 7
    for kw in (dict(w=0), dict(b=-1), dict(pages=0), dict(mp=0)):
        assert a(p7, **kw) == -2, kw
    for i in (0, 2, 3, 4, 5):                             # sampled (1) and out (6) may be null
        args = list(p7)
        args[i] = null
        assert a(args) == -4, i
    assert a([null] * 7, b=0) == 0
