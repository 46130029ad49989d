"""CPU: the attention forward's split plan and workspace layout (the three *_workspace_bytes entry points against a restatement),
and the form a PagedKVCache step takes (plain paged, cascade or verify), with the ops entry points recording their calls."""
import os

import pytest
import torch

import llama32_b200 as L
from llama32_b200 import _lib, ops

PAGE, Q_TILE = 64, 128


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _lib.lib()


def num_sms():
    # the library plans for the current device, and for 148 SMs when it cannot ask one
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count if torch.cuda.is_available() else 148


def decode_splits(sms, batch, heads, kv_heads, kv_len):
    group = heads // kv_heads
    if batch <= 0 or group < 2 or group > Q_TILE:
        return 1
    ctas = batch * kv_heads
    splits = min((2 * sms + ctas - 1) // ctas, (kv_len + PAGE - 1) // PAGE // 2)
    return 1 if splits < 2 else splits


def split_bytes(rows, splits, d):
    """part_o (rows * splits rows of d fp32) and part_ml (rows * splits float2), with 256 bytes for part_ml's alignment."""
    return rows * splits * (d + 2) * 4 + 256


def up(x):
    return (x + 255) // 256 * 256


def workspace_bytes(sms, b, t, h, kv, d, kv_len):
    if b <= 0 or t <= 0 or kv_len <= 0 or t != 1:
        return 0
    s = decode_splits(sms, b, h, kv, kv_len)
    return split_bytes(b * h, s, d) if s >= 2 else 0


def verify_workspace_bytes(sms, b, t, h, kv, d, max_kv_len):
    if b <= 0 or t <= 0 or h // kv < 2 or (h // kv) * t > 128:
        return 0
    s = decode_splits(sms, b, h, kv, max_kv_len)
    return split_bytes(b * h * t, s, d) if s >= 2 else 0


def cascade_workspace_bytes(sms, b, h, kv, d, max_kv_len, max_items):
    if b <= 0 or not 2 <= h // kv <= 128:
        return 0
    own = b * h * decode_splits(sms, b, h, kv, max_kv_len)           # at least one split's partials
    pfx = max_items * kv * Q_TILE
    return up(own * d * 4) + up(own * 8) + up(pfx * d * 4) + up(pfx * 8)


HEADS = [(8, 8), (32, 8), (64, 8), (8, 2), (16, 1), (128, 1), (256, 1)]    # groups 1, 4, 8, 4, 16, 128, 256
KV_LENS = [0, 1, 63, 64, 127, 128, 129, 1000, 2048, 8191, 65536]


@pytest.mark.parametrize("d", [64, 128])
def test_workspace_bytes_match_the_split_plan(lib, d):
    sms = num_sms()
    for b in range(1, 301):
        for h, kv in HEADS:
            for n in KV_LENS:
                for t in (1, 2):
                    assert lib.l32_gqa_attention_workspace_bytes(b, t, h, kv, d, n) == workspace_bytes(sms, b, t, h, kv, d, n), \
                        (b, t, h, kv, d, n)
                for t in (1, 2, 4, 8, 16, 33):
                    assert lib.l32_gqa_attention_verify_workspace_bytes(b, t, h, kv, d, n) == \
                        verify_workspace_bytes(sms, b, t, h, kv, d, n), (b, t, h, kv, d, n)
                for items in (1, 37, 296, 65535):
                    assert lib.l32_gqa_attention_cascade_workspace_bytes(b, h, kv, d, n, items) == \
                        cascade_workspace_bytes(sms, b, h, kv, d, n, items), (b, h, kv, d, n, items)


@pytest.fixture
def calls(monkeypatch):
    """The three paged attention entry points of ops, replaced by recorders: [(form, q, kwargs)]."""
    log = []
    for form, name in (("plain", "gqa_attention_forward_paged"), ("cascade", "gqa_attention_forward_paged_cascade"),
                       ("verify", "gqa_attention_forward_paged_verify")):
        monkeypatch.setattr(ops, name, lambda q, *a, _form=form, **kw: log.append((_form, a, kw)) or _form)
    return log


def step(cache, t, heads=32, kv_heads=8, d=128):
    """One layer's attention call of a step with t tokens per row, on stand-in tensors of the kernels' shapes."""
    q = torch.zeros(len(cache.batch_ids), t, heads * d)
    pool = torch.zeros(cache.num_pages, kv_heads, PAGE, d)
    return cache.attention(q, pool, pool)


def cache_with_batch(new_lens, verify=False):
    cache = L.PagedKVCache(64, 4, 8)
    ids = [cache.add_sequence() for _ in new_lens]
    cache.set_batch(ids, new_lens, verify=verify)
    return cache


def test_form_choice_of_a_paged_step(calls):
    # first use records the geometry (group 4, 8 kv heads); a prefill step takes the plain form
    cache = cache_with_batch([3, 5])
    assert cache.cascade_geometry is None
    assert step(cache, 5) == "plain" and cache.cascade_geometry == (4, 8)
    assert calls[-1][2] == {"max_kv_len": cache.max_kv_len}
    # a verify step that fits one query tile (4 * 32 = 128 rows) takes the verify form
    cache = cache_with_batch([32, 32], verify=True)
    assert step(cache, 32) == "verify" and calls[-1][2] == {"max_kv_len": cache.max_kv_len}
    assert cache.cascade_geometry == (4, 8)
    # ... one that does not (4 * 33 rows) the plain form, as does a verify step of a group-1 attention
    cache = cache_with_batch([33, 33], verify=True)
    assert step(cache, 33) == "plain"
    cache = cache_with_batch([2, 2], verify=True)
    assert step(cache, 2, heads=8) == "plain"
    # a decode step with a cascade plan for this geometry takes the cascade form, with the cache's plan buffers
    cache = cache_with_batch([1, 1])
    cache.cascade_geometry, cache.cascade, cache.cascade_max_items = (4, 8), True, 37
    assert step(cache, 1) == "cascade"
    assert calls[-1][1][-4:] == (cache.plan_items, cache.plan_members, cache.plan_seq, 37)
    assert calls[-1][2] == {"max_kv_len": cache.max_kv_len}
    # ... the plain form for another attention geometry, or for a step of more than one token
    assert step(cache, 1, heads=64) == "plain"
    assert step(cache, 1, kv_heads=4, heads=16) == "plain"
    assert step(cache, 2) == "plain"
    # a decode step without a plan takes the plain form
    cache.cascade = False
    assert step(cache, 1) == "plain"
    # a verify step that fits takes the verify form even when a plan is present
    cache = cache_with_batch([1, 1], verify=True)
    cache.cascade_geometry, cache.cascade = (4, 8), True
    assert step(cache, 1) == "verify"
