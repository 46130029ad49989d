"""CPU: PagedKVCache's host bookkeeping (allocator, block table, lengths), the module's refusals with a paged cache, and the
paged C-ABI entry points' argument checks (no compute calls without a GPU)."""
import ctypes
import os

import pytest
import torch

import llama32_b200 as L
from llama32_b200 import _lib

PAGE = 64


def host_cache(num_pages, max_batch, max_pages):
    return L.PagedKVCache(num_pages, max_batch, max_pages)     # device buffers only when a GPU is present


def uploaded(cache):
    """(table, past_lens, new_lens) of the last upload, from the host staging copy."""
    t = cache.max_batch * cache.max_pages_per_seq
    h = cache._host
    return h[:t].view(cache.max_batch, cache.max_pages_per_seq), h[t:t + cache.max_batch], h[t + cache.max_batch:]


def test_allocator_accounting_and_reuse():
    c = host_cache(10, 4, 8)
    a, b = c.add_sequence(), c.add_sequence()
    assert a != b and c.free_pages == 10
    c.set_batch([a, b], [130, 64])                  # 3 pages + 1 page
    assert len(c.pages(a)) == 3 and len(c.pages(b)) == 1 and c.free_pages == 6
    assert len(set(c.pages(a)) | set(c.pages(b))) == 4
    c.advance()
    assert (c.length(a), c.length(b)) == (130, 64)
    freed = set(c.pages(a))
    c.free_sequence(a)
    assert c.free_pages == 9 and c.batch_ids == []        # the batch that held `a` is dropped
    d = c.add_sequence()
    c.set_batch([b, d], [1, 190])                    # b crosses into its second page, d needs 3: the freed pages go first
    assert len(c.pages(b)) == 2 and len(c.pages(d)) == 3
    assert freed <= {c.pages(b)[1], *c.pages(d)}
    assert c.free_pages == 5


def test_table_contents_across_page_boundaries():
    c = host_cache(16, 3, 6)
    ids = [c.add_sequence() for _ in range(3)]
    steps = [[63, 64, 65], [1, 1, 1], [0, 64, 127]]
    for news in steps:
        c.set_batch(ids, news)
        table, past, new = uploaded(c)
        for r, sid in enumerate(ids):
            pages = c.pages(sid)
            need = -(-(c.length(sid) + news[r]) // PAGE)
            assert len(pages) == need
            assert table[r, :need].tolist() == pages
            assert (table[r, need:] == 0).all()
            assert past[r].item() == c.length(sid) and new[r].item() == news[r]
        assert (past[3:] == 0).all() and (new[3:] == 0).all()       # rows past the batch are inert
        c.advance()
    assert [c.length(s) for s in ids] == [64, 129, 193]
    all_pages = sum((c.pages(s) for s in ids), [])
    assert len(all_pages) == len(set(all_pages)) and all(0 <= p < 16 for p in all_pages)


def test_out_of_pages_raises_before_reserving():
    c = host_cache(4, 2, 8)
    a, b = c.add_sequence(), c.add_sequence()
    c.set_batch([a], [192])
    c.advance()
    before = (c.free_pages, c.pages(a), c.pages(b), c.batch_ids)
    with pytest.raises(RuntimeError, match="out of pages"):
        c.set_batch([a, b], [1, 65])                 # a needs a 4th page, b two: 3 > 1 free
    assert (c.free_pages, c.pages(a), c.pages(b), c.batch_ids) == before
    d = host_cache(64, 1, 2)
    s = d.add_sequence()
    with pytest.raises(ValueError, match="max_pages_per_seq"):
        d.set_batch([s], [129])
    with pytest.raises(ValueError):
        d.set_batch([s, s], [1, 1])
    with pytest.raises(ValueError):
        d.set_batch([s + 1], [1])


def _att(dtype=torch.bfloat16, head_dim=64):
    heads, kv = 4, 2
    cfg = type("Cfg", (), dict(hidden_size=heads * head_dim, n_heads=heads, n_kv_groups=kv, rope_base=500000.0))()
    return L.GroupQueryAttention(cfg, layer_idx=0).to(dtype).eval()


def test_module_refuses_what_the_kernels_do_not_take():
    c = host_cache(8, 2, 4)
    s = c.add_sequence()
    c.set_batch([s], [3])
    pos = torch.arange(3)[None]
    att = _att()
    x = torch.randn(1, 3, att.num_heads * att.head_dim, dtype=torch.bfloat16)
    with torch.no_grad():
        with pytest.raises(ValueError, match="attention_mask"):
            att(x, attention_mask=torch.zeros(1, 1, 3, 3, dtype=torch.bfloat16), position_ids=pos, kv_cache=c)
        with pytest.raises(ValueError, match="position_ids"):
            att(x, position_ids=None, kv_cache=c)
        with pytest.raises(ValueError, match="sm_100a kernels"):            # CPU tensors
            att(x, position_ids=pos, kv_cache=c)
        with pytest.raises(ValueError, match="sm_100a kernels"):            # fp32
            _att(torch.float32)(x.float(), position_ids=pos, kv_cache=c)
    with pytest.raises(ValueError, match="inference-only"):                  # autograd would record the call
        att(x, position_ids=pos, kv_cache=c)


def test_paged_symbols_in_the_abi_tables():
    names = _lib.header_symbols()
    for n in ("l32_rope_kv_append_paged", "l32_gqa_attention_forward_paged"):
        assert n in names and n in _lib.SIGNATURES
    assert "#define L32_KV_PAGE 64" in open(_lib.HEADER_PATH).read()


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _lib.lib()


def test_paged_argument_validation_without_device(lib):
    null = ctypes.c_void_p(0)
    one = ctypes.c_void_p(256)   # never dereferenced: validation fails first
    rope = lambda *a: lib.l32_rope_kv_append_paged(*a)
    att = lambda *a: lib.l32_gqa_attention_forward_paged(*a)
    p9 = [one] * 9
    # rope: (ptrs x9, batch, q_len, heads, kv_heads, head_dim, num_pages, max_pages, rope_base, dtype, stream)
    assert rope(*p9, 2, 3, 8, 2, 64, 16, 4, 500000.0, 5, null) == -1                    # dtype
    assert rope(*p9, 2, 3, 8, 3, 64, 16, 4, 500000.0, 0, null) == -2                    # heads % kv_heads
    assert rope(*p9, 2, 3, 8, 2, 96, 16, 4, 500000.0, 0, null) == -2                    # head_dim
    assert rope(*p9, 2, 3, 8, 2, 64, 0, 4, 500000.0, 0, null) == -2                     # no pages
    assert rope(*p9, 2, 3, 8, 2, 64, 16, 0, 500000.0, 0, null) == -2                    # no table columns
    assert rope(*p9[:6], null, one, one, 2, 3, 8, 2, 64, 16, 4, 500000.0, 0, null) == -4   # block_table
    assert rope(*p9[:7], null, one, 2, 3, 8, 2, 64, 16, 4, 500000.0, 0, null) == -4     # past_lens
    assert rope(*p9[:8], null, 0, 3, 8, 2, 64, 16, 4, 500000.0, 0, null) == 0           # empty batch: nothing to do
    # attention: (q, pool_k, pool_v, table, past, new, ctx, ws, ws_bytes, batch, q_len, heads, kv, d, pages, max_pages,
    #             max_kv_len, dtype, stream)
    p8 = [one] * 8
    assert att(*p8, 0, 2, 1, 32, 8, 128, 16, 4, 256, 9, null) == -1
    assert att(*p8, 0, 2, 1, 32, 8, 128, 16, 4, 257, 0, null) == -2                     # max_kv_len > max_pages * 64
    assert att(*p8, 0, 2, 1, 32, 8, 128, 16, 4, -1, 0, null) == -2
    assert att(*p8, 0, 2, 1, 32, 8, 80, 16, 4, 256, 0, null) == -2
    assert att(one, one, one, null, one, one, one, null, 0, 2, 1, 32, 8, 128, 16, 4, 256, 0, null) == -4
    assert att(one, one, one, one, one, one, null, null, 0, 2, 1, 32, 8, 128, 16, 4, 256, 0, null) == -4
    assert att(one, null, one, one, one, one, one, null, 0, 2, 1, 32, 8, 128, 16, 4, 256, 0, null) == -4
    assert att(ctypes.c_void_p(8), one, one, one, one, one, one, null, 0, 2, 1, 32, 8, 128, 16, 4, 256, 0, null) == -3
    assert att(*p8[:7], ctypes.c_void_p(8), 1 << 20, 2, 1, 32, 8, 128, 16, 4, 256, 0, null) == -6
    assert att(null, null, null, null, null, null, null, null, 0, 0, 1, 32, 8, 128, 16, 4, 256, 0, null) == 0
    assert att(*p8, 0, -1, 1, 32, 8, 128, 16, 4, 256, 0, null) == -2
    assert att(*p8, 0, 2, 1, 32, 8, 128, 0, 4, 256, 0, null) == -2                      # no pages
    assert att(one, one, null, one, one, one, one, null, 0, 2, 1, 32, 8, 128, 16, 4, 256, 0, null) == -4   # pool_v
    assert att(one, one, one, one, null, one, one, null, 0, 2, 1, 32, 8, 128, 16, 4, 256, 0, null) == -4   # past_lens
    assert att(*p8[:6], ctypes.c_void_p(8), null, 0, 2, 1, 32, 8, 128, 16, 4, 256, 0, null) == -3          # ctx
    # a call with several faults gets the code of the first check: dtype, shape, empty batch, nulls, alignment, workspace
    assert att(*[null] * 8, 0, 0, 1, 32, 8, 128, 16, 4, 256, 9, null) == -1
    assert att(*[null] * 8, 0, 2, 1, 32, 8, 128, 16, 4, 257, 0, null) == -2
    assert att(ctypes.c_void_p(8), one, one, null, one, one, one, null, 0, 2, 1, 32, 8, 128, 16, 4, 256, 0, null) == -4
    assert att(ctypes.c_void_p(8), *p8[1:7], ctypes.c_void_p(8), 1 << 20, 2, 1, 32, 8, 128, 16, 4, 256, 0, null) == -3
