"""CPU: shared prefixes on the PagedKVCache -- reference-counted pages through fork / free_sequence, the copy-on-write
invariant (a shared page is full and never written), the cascade plan builder, and the cascade entry point's argument
checks (no compute calls without a GPU)."""
import ctypes
import os

import pytest

import llama32_b200 as L
from llama32_b200 import _lib
from llama32_b200.modules import cascade_items_capacity, cascade_plan

PAGE = 64


def grow(c, sid, n):
    c.set_batch([sid], [n])
    c.advance()


def written_pages(c, ids, news):
    """Pages the append kernel writes in a step: rows [past, past + new) of each sequence, through its table."""
    out = set()
    for sid, n in zip(ids, news):
        pages, past = c.pages(sid), c.length(sid)
        out |= {pages[pos // PAGE] for pos in range(past, past + n)}
    return out


def test_counts_through_fork_and_free_in_any_order():
    c = L.PagedKVCache(20, 8, 8)
    a = c.add_sequence()
    grow(c, a, 130)                                   # pages: 2 full + 1 partial
    assert c.free_pages == 17
    kids = [c.fork(a) for _ in range(3)]              # each: the 2 full pages shared, its own copy of the tail
    assert c.free_pages == 14
    full = c.pages(a)[:2]
    assert all(c.refcount(p) == 4 for p in full)
    assert all(c.refcount(c.pages(k)[2]) == 1 for k in kids)
    c.free_sequence(a)                                # the children keep the shared pages
    assert c.free_pages == 15 and all(c.refcount(p) == 3 for p in full)
    for k in kids[:2]:
        assert c.pages(k)[:2] == full and c.length(k) == 130
    c.free_sequence(kids[1])
    grand = c.fork(kids[0])
    c.free_sequence(kids[0])
    assert all(c.refcount(p) == 2 for p in full)
    c.free_sequence(grand)
    c.free_sequence(kids[2])
    assert c.free_pages == 20 and all(r == 0 for r in c._refs)


@pytest.mark.parametrize("n", [0, 63, 64, 65, 130])
def test_fork_shares_exactly_the_full_pages(n):
    c = L.PagedKVCache(16, 4, 8)
    a = c.add_sequence()
    if n:
        grow(c, a, n)
    before = c.free_pages
    k = c.fork(a)
    full = n // PAGE
    assert c.length(k) == n
    assert c.pages(k)[:full] == c.pages(a)[:full]
    own = c.pages(k)[full:]
    assert len(own) == (1 if n % PAGE else 0) and not set(own) & set(c.pages(a))
    assert c.free_pages == before - len(own)


def test_fork_out_of_pages_changes_nothing():
    c = L.PagedKVCache(3, 4, 8)
    a = c.add_sequence()
    grow(c, a, 130)                                   # all 3 pages in use
    state = (c.free_pages, list(c._refs), c.pages(a), c._next_id)
    with pytest.raises(RuntimeError, match="out of pages"):
        c.fork(a)
    assert (c.free_pages, list(c._refs), c.pages(a), c._next_id) == state
    c2 = L.PagedKVCache(4, 4, 2)                      # a parent at max_pages_per_seq: the child shares it, cannot grow
    p = c2.add_sequence()
    grow(c2, p, 128)
    k = c2.fork(p)
    assert c2.free_pages == 2 and c2.pages(k) == c2.pages(p)
    free = c2.free_pages
    with pytest.raises(ValueError, match="max_pages_per_seq"):
        c2.set_batch([k], [1])
    assert c2.free_pages == free


def test_no_shared_page_is_ever_written():
    c = L.PagedKVCache(64, 8, 8)
    root = c.add_sequence()
    grow(c, root, 150)
    ids = [root] + [c.fork(root) for _ in range(3)]
    ids.append(c.fork(ids[1]))
    for step, news in enumerate([[1] * 5, [40, 1, 1, 64, 1], [1] * 5, [0, 70, 1, 1, 2]]):
        c.set_batch(ids, news)
        shared = {p for p in range(c.num_pages) if c.refcount(p) > 1}
        assert not written_pages(c, ids, news) & shared, f"step {step}"
        c.advance()
        if step == 1:
            ids.append(c.fork(ids[3]))
            ids[0:1] = []
            c.free_sequence(root)


# --------------------------------------------------------------------------------------------- the plan builder
def rows_of(tables_and_lens):
    return [t for t, _ in tables_and_lens], [n for _, n in tables_and_lens]


def test_plan_groups_by_first_page_and_longest_common_prefix():
    pre = list(range(10))
    tables = [pre + [100], [50, 51, 52, 53, 54], pre[:6] + [101, 102], pre + [103], [60, 61], pre[:8] + [104]]
    lens = [10 * 64 + 5, 5 * 64, 8 * 64, 10 * 64 + 1, 2 * 64, 8 * 64 + 3]
    items, members, seq = cascade_plan(tables, lens, [1] * 6, group=4, max_items=37, min_shared_pages=4)
    assert members == [0, 2, 3, 5]
    assert all(seq[r][0] == 6 for r in members)      # the common prefix of the whole group: pages 0..5
    assert seq[1] == seq[4] == (0, 0, 0, 0)           # unshared rows
    assert [seq[r][3] for r in members] == [0, 4, 8, 12]
    assert sum(it[2] for it in items) == 6 and all(it[0] == 0 and it[3] == 0 and it[4] == 4 for it in items)
    # the prefix stops below a member's past length: the page it appends to this step is not shared
    tables2 = [pre, pre[:3] + [200]]
    plan = cascade_plan(tables2, [10 * 64, 3 * 64 + 10], [1, 1], group=2, max_items=37, min_shared_pages=1)
    assert plan[2][0][0] == 3 and plan[2][1][0] == 3


@pytest.mark.parametrize("group,members_n", [(4, 33), (8, 17), (2, 70), (128, 3)])
def test_plan_chunks_at_one_query_tile(group, members_n):
    tables = [list(range(12)) + [1000 + r] for r in range(members_n)]
    items, members, seq = cascade_plan(tables, [12 * 64 + 3] * members_n, [1] * members_n, group, max_items=200,
                                       min_shared_pages=4)
    per = 128 // group
    chunks = {}
    for it in items:
        chunks.setdefault(it[3], []).append(it)
    sizes = [v[0][4] for _, v in sorted(chunks.items())]
    assert sizes == [min(per, members_n - c0) for c0 in range(0, members_n, per)]
    for r in range(members_n):
        tiles, first, n, row0 = seq[r]
        assert tiles == 12 and row0 == (r % per) * group
        cov = [(items[k][1], items[k][2]) for k in range(first, first + n)]
        assert sum(t for _, t in cov) == 12 and cov[0][0] == 0
        assert all(members[items[k][3] + row0 // group] == r for k in range(first, first + n))


def test_plan_none_for_non_decode_or_below_threshold():
    pre = list(range(8))
    tables = [pre + [90], pre + [91]]
    assert cascade_plan(tables, [8 * 64 + 1] * 2, [1, 2], 4, 37) is None             # not a decode step
    assert cascade_plan(tables, [8 * 64 + 1] * 2, [1, 1], 1, 37) is None             # group 1: the existing path
    assert cascade_plan(tables, [8 * 64 + 1] * 2, [1, 1], 4, 37, min_shared_pages=9) is None
    assert cascade_plan([pre, [77] + pre[1:]], [8 * 64] * 2, [1, 1], 4, 37, min_shared_pages=1) is None
    assert cascade_plan([pre], [8 * 64], [1], 4, 37, min_shared_pages=1) is None      # one member is no group
    assert cascade_plan(tables, [8 * 64 + 1] * 2, [1, 1], 4, 37, min_shared_pages=8) is not None


@pytest.mark.parametrize("kv_heads,group", [(8, 4), (8, 8), (1, 2), (16, 128)])
def test_plan_capacity_never_exceeded_and_deterministic(kv_heads, group):
    max_batch, sms = 256, 148
    cap = cascade_items_capacity(sms, kv_heads)
    for n_groups, pages in [(1, 128), (4, 32), (max_batch // 2, 5), (max_batch // 2, 200)]:
        tables, lens = [], []
        for r in range(max_batch):
            g = r % n_groups
            tables.append([10000 * g + j for j in range(pages)] + [900000 + r])
            lens.append(pages * 64 + 7)
        plan = cascade_plan(tables, lens, [1] * max_batch, group, cap)
        assert plan == cascade_plan(tables, lens, [1] * max_batch, group, cap)
        items, members, seq = plan
        assert 1 <= len(items) <= cap and len(members) <= max_batch and len(set(members)) == len(members)
        assert all(it[2] >= 1 and it[4] * group <= 128 for it in items)


# --------------------------------------------------------------------------------------------- the C entry point
def test_cascade_symbols_in_the_abi_tables():
    names = _lib.header_symbols()
    for n in ("l32_gqa_attention_forward_paged_cascade", "l32_gqa_attention_cascade_workspace_bytes"):
        assert n in names and n in _lib.SIGNATURES
    assert "#define L32_CASCADE_TILE_ROWS 128" in open(_lib.HEADER_PATH).read()


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _lib.lib()


def test_cascade_argument_validation_without_device(lib):
    null = ctypes.c_void_p(0)
    one = ctypes.c_void_p(256)   # never dereferenced: validation fails first
    ws = lambda *a: lib.l32_gqa_attention_cascade_workspace_bytes(*a)
    att = lambda *a: lib.l32_gqa_attention_forward_paged_cascade(*a)
    assert ws(64, 32, 8, 128, 2048, 37) > 64 * 37 * 8 * 128 * 130 * 4 // 64
    assert ws(64, 8, 8, 128, 2048, 37) == 0                                            # group 1
    # (q, pool_k, pool_v, table, past, new, items, members, seq, ctx, ws, ws_bytes, batch, heads, kv, d, pages, max_pages,
    #  max_kv_len, max_items, dtype, stream)
    p11 = [one] * 11
    need = ws(2, 32, 8, 128, 256, 37)
    assert att(*p11, need, 2, 32, 8, 128, 16, 4, 256, 37, 7, null) == -1               # dtype
    assert att(*p11, need, 2, 8, 8, 128, 16, 4, 256, 37, 0, null) == -2                 # group 1
    assert att(*p11, need, 2, 32, 8, 96, 16, 4, 256, 37, 0, null) == -2                 # head_dim
    assert att(*p11, need, 2, 32, 8, 128, 16, 4, 257, 37, 0, null) == -2                # max_kv_len > max_pages * 64
    assert att(*p11, need, 2, 32, 8, 128, 16, 4, 256, 0, 0, null) == -2                 # no items
    assert att(*p11, need, 2, 512, 2, 128, 16, 4, 256, 37, 0, null) == -2               # group 256 > one query tile
    for i in (0, 1, 2, 3, 4, 6, 7, 8, 9, 10):                                          # new_lens (5) may be null
        args = list(p11)
        args[i] = null
        assert att(*args, need, 2, 32, 8, 128, 16, 4, 256, 37, 0, null) == -4, i
    assert att(ctypes.c_void_p(8), *p11[1:], need, 2, 32, 8, 128, 16, 4, 256, 37, 0, null) == -3
    assert att(*p11, need - 1, 2, 32, 8, 128, 16, 4, 256, 37, 0, null) == -6           # workspace short
    assert att(*p11[:10], ctypes.c_void_p(8), need, 2, 32, 8, 128, 16, 4, 256, 37, 0, null) == -6
    assert att(*([null] * 11), 0, 0, 32, 8, 128, 16, 4, 256, 37, 0, null) == 0          # empty batch
    assert att(*p11, need, 2, 32, 8, 128, 16, 4, -1, 37, 0, null) == -2
    assert att(*p11, need, 2, 32, 8, 128, 0, 4, 256, 37, 0, null) == -2                 # no pages
    assert att(*p11[:9], ctypes.c_void_p(8), one, need, 2, 32, 8, 128, 16, 4, 256, 37, 0, null) == -3   # ctx
    assert att(one, one, ctypes.c_void_p(8), *p11[3:], need, 2, 32, 8, 128, 16, 4, 256, 37, 0, null) == -3   # pool_v
    # a call with several faults gets the code of the first check: dtype, shape, empty batch, nulls, alignment, workspace
    assert att(*([null] * 11), 0, 0, 32, 8, 128, 16, 4, 256, 37, 7, null) == -1
    assert att(*([null] * 11), 0, 2, 32, 8, 128, 16, 4, 257, 37, 0, null) == -2
    assert att(ctypes.c_void_p(8), *p11[1:6], null, *p11[7:], need, 2, 32, 8, 128, 16, 4, 256, 37, 0, null) == -4
    assert att(ctypes.c_void_p(8), *p11[1:10], ctypes.c_void_p(8), need - 1, 2, 32, 8, 128, 16, 4, 256, 37, 0, null) == -3
