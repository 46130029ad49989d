"""The inference attention kernels (csrc/attention.cu) where they branch: split-KV decode and its combine, the packed GQA
decode, chunked prefill onto a cache, the lazy online-softmax rescale, the cache rows beyond kv_len and rope_kv_append.

Every comparison is against a float64 restatement of the same operation.  Random-input parity alone cannot see a dropped
or duplicated key at kv_len 2048 (it moves the output by ~1/2048 of |v|), so the "needle" tests give one key a dominant
score: the output is then that key's value row, exactly, or visibly not."""
import math

import pytest
import torch

import llama32_b200 as L
from llama32_b200 import ops
from llama32_b200._lib import lib
from oracle import ffn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
FWD = (1e-2, 2.0 ** -6)
KV_TILE, Q_TILE = 64, 128
DTYPES = [torch.bfloat16, torch.float16]
DIMS = [64, 128]
# decode geometries: group 1 (not packed), 2, 4 (11B: 32 / 8) and 8 (90B: 64 / 8)
HEADS = {1: (8, 8), 2: (16, 8), 4: (32, 8), 8: (64, 8)}


def close(got, ref, tol, what=""):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    assert torch.isfinite(got).all(), f"{what}: non-finite output"
    r, m = O.rel_l2(got, ref), O.max_abs_over_max_ref(got, ref)
    assert r <= tol[0] and m <= tol[1], f"{what}: rel-L2 {r:.3e} (<= {tol[0]}), max-abs/max|ref| {m:.3e} (<= {tol[1]:.3e})"


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def rnd(g, *shape, dtype, scale=1.0):
    return (torch.randn(*shape, device=DEV, generator=g) * scale).to(dtype)


def ref_attention(q, cache_k, cache_v, kv_len, past_len, causal, keep=None):
    """float64 attention over cache[:, :, :kv_len] (cache layout [b, kv, max_len, d]); q [b, t, heads*d] holds the queries at
    positions past_len .. past_len + t - 1.  keep [b, kv_len]: 0 = padded key.  A row with no visible key gives exact zeros.
    Returns (out [b, t, heads*d], lse [b, heads, t] in log2 units, +inf for such a row)."""
    b, t, hd = q.shape
    _, kv, _, d = cache_k.shape
    heads = hd // d
    g = heads // kv
    q5 = q.double().view(b, t, kv, g, d).permute(0, 2, 3, 1, 4).reshape(b, kv, g * t, d)
    k, v = cache_k[:, :, :kv_len].double(), cache_v[:, :, :kv_len].double()
    s = (q5 @ k.transpose(-1, -2)) / math.sqrt(d)                                   # [b, kv, g*t, kv_len]
    vis = torch.ones(t, kv_len, dtype=torch.bool, device=q.device)
    if causal:
        vis &= torch.arange(kv_len, device=q.device)[None] <= (past_len + torch.arange(t, device=q.device))[:, None]
    vis = vis.repeat(g, 1)[None, None]
    if keep is not None:
        vis = vis & keep.bool()[:, None, None, :]
    s = s.masked_fill(~vis, float("-inf"))
    m = s.amax(-1, keepdim=True)
    m = torch.where(torch.isfinite(m), m, torch.zeros_like(m))
    p = torch.exp(s - m)
    l = p.sum(-1, keepdim=True)
    o = (p @ v) / torch.where(l > 0, l, torch.ones_like(l))
    lse = ((m + torch.log(l)) / math.log(2.0)).squeeze(-1)                          # log(0) = -inf ...
    lse = torch.where(l.squeeze(-1) > 0, lse, torch.full_like(lse, float("inf")))    # ... but a dead row reports +inf
    out = o.view(b, kv, g, t, d).permute(0, 3, 1, 2, 4).reshape(b, t, hd)
    return out, lse.view(b, kv, g, t).reshape(b, heads, t)


# ------------------------------------------------------------------------------------------------------- the split plan
def num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def wanted_splits(batch, kv, sms):
    """Splits the plan aims at before the clamp: two CTAs per SM over the batch * kv_heads packed decode CTAs."""
    return -(-2 * sms // (batch * kv))


def split_plan(batch, heads, kv, kv_len, sms):
    """Restatement of decode_splits() in csrc/attention.cu: (splits, key tiles per split, empty trailing splits).  Only the
    packed decode (2 <= group <= 128) splits; a split covers at least two key tiles."""
    group = heads // kv
    tiles = -(-kv_len // KV_TILE)
    if group < 2 or group > Q_TILE:
        return 1, tiles, 0
    splits = min(wanted_splits(batch, kv, sms), tiles // 2)
    if splits < 2:
        return 1, tiles, 0
    per = -(-tiles // splits)
    return splits, per, splits - (-(-tiles // per))


def first_empty_trailing(batch, heads, kv, sms, limit=16384):
    for kv_len in range(128, limit):
        if split_plan(batch, heads, kv, kv_len, sms)[2] > 0:
            return kv_len
    return None


def regime_of(batch, heads, kv, kv_len, sms):
    splits, per, empty = split_plan(batch, heads, kv, kv_len, sms)
    tags = set()
    if splits == 1:
        tags.add("no_split")
    else:
        if splits == 2:
            tags.add("two_splits")
        if empty > 0:
            tags.add("empty_trailing")
        if kv_len % KV_TILE != 0:
            tags.add("partial_last_tile")
        if wanted_splits(batch, kv, sms) > (-(-kv_len // KV_TILE)) // 2:
            tags.add("clamp")
    return tags


def regime_shapes(regime, sms, count=2):
    """The first `count` decode shapes (group, batch, kv_len) of the axes that take `regime` on this GPU, of distinct groups
    (no split: largest batch and length first; a partial last tile: longest length first)."""
    found, groups = [], set()
    for group in (2, 4, 8, 1):
        for batch in ((64, 37, 3, 1) if regime == "no_split" else (1, 3, 37, 64)):
            heads, kv = HEADS[group]
            # 300 keys = 5 tiles: two splits whenever the plan wants two or more
            lens = [1, 63, 64, 65, 127, 128, 129, first_empty_trailing(batch, heads, kv, sms), 300, 2047, 2048, 8193]
            for kv_len in (lens[::-1] if regime in ("no_split", "partial_last_tile") else lens):
                if kv_len is None or group in groups or regime not in regime_of(batch, heads, kv, kv_len, sms):
                    continue
                found.append((group, batch, kv_len))
                groups.add(group)
    return found[:count]


def decode_inputs(batch, heads, kv, kv_len, d, dtype, seed, tail=0):
    g = gen(seed)
    max_len = kv_len + tail
    q = rnd(g, batch, 1, heads * d, dtype=dtype)
    ck, cv = rnd(g, batch, kv, max_len, d, dtype=dtype), rnd(g, batch, kv, max_len, d, dtype=dtype)
    return q, ck, cv


def run_decode(q, ck, cv, kv_len):
    """One decode call through ops; returns (out, kernel launches it took)."""
    n0 = lib().l32_kernel_launch_count()
    y = ops.gqa_attention_forward(q, ck, cv, kv_len, kv_len - 1, causal=True)
    return y, lib().l32_kernel_launch_count() - n0


def assert_plan_taken(batch, heads, kv, d, kv_len, launches):
    splits = split_plan(batch, heads, kv, kv_len, num_sms())[0]
    ws = lib().l32_gqa_attention_workspace_bytes(batch, 1, heads, kv, d, kv_len)
    assert (ws > 0) == (splits > 1), f"workspace {ws} B but the plan has {splits} split(s)"
    assert launches == (2 if splits > 1 else 1), f"{launches} launches for {splits} split(s)"


REGIMES = ["empty_trailing", "partial_last_tile", "clamp", "two_splits", "no_split"]


@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("regime", REGIMES)
def test_decode_regimes_vs_fp64(regime, dtype, d):
    """q_len = 1 against the float64 reference, at shapes the split plan sends into `regime` on this GPU; asserts the regime
    was taken (workspace > 0 exactly when split, two launches with a split: kernel + combine)."""
    sms = num_sms()
    shapes = regime_shapes(regime, sms)
    assert shapes, f"no decode shape of the axes takes {regime} with {sms} SMs"
    for group, batch, kv_len in shapes:
        heads, kv = HEADS[group]
        q, ck, cv = decode_inputs(batch, heads, kv, kv_len, d, dtype, seed=kv_len * 7 + batch + group, tail=5)
        y, launches = run_decode(q, ck, cv, kv_len)
        assert_plan_taken(batch, heads, kv, d, kv_len, launches)
        close(y, ref_attention(q, ck, cv, kv_len, kv_len - 1, True)[0], FWD,
              f"{regime}: group {group} batch {batch} kv_len {kv_len} plan {split_plan(batch, heads, kv, kv_len, sms)}")


@pytest.mark.parametrize("group", [1, 2, 4, 8])
@pytest.mark.parametrize("kv_len", [1, 63, 64, 65, 127, 128, 129, 2047, 2048, 8193])
def test_decode_grid_vs_fp64(group, kv_len):
    """The group x kv_len axes at batch 3 (bf16 d128 / fp16 d64 alternating), whatever the plan makes of them."""
    heads, kv = HEADS[group]
    dtype, d = (torch.bfloat16, 128) if (group + kv_len) % 2 else (torch.float16, 64)
    q, ck, cv = decode_inputs(3, heads, kv, kv_len, d, dtype, seed=kv_len + 31 * group, tail=3)
    y, launches = run_decode(q, ck, cv, kv_len)
    assert_plan_taken(3, heads, kv, d, kv_len, launches)
    close(y, ref_attention(q, ck, cv, kv_len, kv_len - 1, True)[0], FWD, f"group {group} kv_len {kv_len}")


def raw_forward(q, ck, cv, out, kv_len, past_len, ws, ws_bytes, causal=True):
    b, t = q.shape[0], q.shape[1]
    _, kv, max_len, d = ck.shape
    ops.check(lib().l32_gqa_attention_forward(q.data_ptr(), ck.data_ptr(), cv.data_ptr(), None, out.data_ptr(),
                                              None if ws is None else ws.data_ptr(), ws_bytes, b, t, q.shape[-1] // d, kv, d,
                                              max_len, kv_len, past_len, int(causal), ops._dtype_code(q), ops._stream(q)),
              "l32_gqa_attention_forward")


@pytest.mark.parametrize("dtype", DTYPES)
def test_decode_short_workspace_determinism_and_graph_replay(dtype):
    """A workspace one byte short of what the plan needs takes the one-pass path (one launch) and agrees with the split result;
    two runs give the same bits; a CUDA-graph replay gives the eager bits."""
    batch, (heads, kv), kv_len, d = 1, HEADS[4], 2047, 128
    assert split_plan(batch, heads, kv, kv_len, num_sms())[0] > 1
    q, ck, cv = decode_inputs(batch, heads, kv, kv_len, d, dtype, seed=5, tail=1)
    need = lib().l32_gqa_attention_workspace_bytes(batch, 1, heads, kv, d, kv_len)
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    split_out, short_out = torch.empty_like(q), torch.empty_like(q)
    n0 = lib().l32_kernel_launch_count()
    raw_forward(q, ck, cv, split_out, kv_len, kv_len - 1, ws, need)
    n1 = lib().l32_kernel_launch_count()
    raw_forward(q, ck, cv, short_out, kv_len, kv_len - 1, ws, need - 1)
    n2 = lib().l32_kernel_launch_count()
    assert (n1 - n0, n2 - n1) == (2, 1)
    ref = ref_attention(q, ck, cv, kv_len, kv_len - 1, True)[0]
    close(split_out, ref, FWD, "split")
    close(short_out, ref, FWD, "workspace too short: one pass")
    close(short_out, split_out, (4e-3, 2.0 ** -8), "one pass vs split")
    a, b = run_decode(q, ck, cv, kv_len)[0], run_decode(q, ck, cv, kv_len)[0]
    assert torch.equal(a, b), "split decode is not deterministic"
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        yg = ops.gqa_attention_forward(q, ck, cv, kv_len, kv_len - 1, causal=True)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(yg, a), "graph replay differs from eager"


# ---------------------------------------------------------------------------------------------------- needle tests
def needle_inputs(batch, heads, kv, t, max_len, d, dtype, seed):
    """q rows of +-1 (the same per KV group); keys small, so their scores are ~0; values N(0, 1)."""
    g = gen(seed)
    u = (torch.randint(0, 2, (batch, kv, 1, d), device=DEV, generator=g) * 2 - 1).float()
    q = u[:, :, None].expand(batch, kv, heads // kv, t, d).permute(0, 3, 1, 2, 4).reshape(batch, t, heads * d).to(dtype)
    ck = (torch.rand(batch, kv, max_len, d, device=DEV, generator=g) * 0.1 - 0.05).to(dtype)
    cv = rnd(g, batch, kv, max_len, d, dtype=dtype)
    return q, ck, cv, u


def plant(ck, cv, u, pos, d):
    """Key `pos` of every (batch, KV head) gets score 4 sqrt(d) (>= 32) against its group's queries: the output is its v row."""
    k, v = ck.clone(), cv.clone()
    k[:, :, pos] = (u[:, :, 0] * 4).to(k.dtype)
    return k, v


def expected_rows(cv, pos, heads, t):
    """[b, t, heads*d]: value row `pos` of each query head's KV group."""
    b, kv, _, d = cv.shape
    vrow = cv[:, :, pos].float()                                                       # [b, kv, d]
    return vrow[:, :, None, None].expand(b, kv, heads // kv, t, d).permute(0, 3, 1, 2, 4).reshape(b, t, heads * d)


def assert_is_needle(y, want, what):
    err = (y.float() - want).abs().max().item()
    assert err <= 2.0 ** -7 * want.abs().max().item(), f"{what}: max |y - v_needle| = {err:.3e}"


def assert_not_needle(y, want, what):
    assert (y.float() - want).abs().amax(-1).min().item() > 0.5, f"{what}: a row is the needle's value"


@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("group,batch,kv_len", [(4, 1, 8193), (4, 1, 2047), (8, 3, 1000), (4, 64, 2048), (1, 2, 300)])
def test_decode_needle(group, batch, kv_len, dtype, d):
    """Decode with one dominant key: at 0, 63, 64, both sides of every split boundary and kv_len - 1 the output is its value
    row; at kv_len .. tile end - 1 (beyond the sequence) it is ignored."""
    heads, kv = HEADS[group]
    splits, per, _ = split_plan(batch, heads, kv, kv_len, num_sms())
    tile_end = -(-kv_len // KV_TILE) * KV_TILE
    q, ck, cv, u = needle_inputs(batch, heads, kv, 1, tile_end + 8, d, dtype, seed=kv_len + group)
    seen = {0, 63, 64, kv_len - 1}
    for s in range(1, splits):
        seen |= {s * per * KV_TILE - 1, s * per * KV_TILE}
    for pos in sorted(p for p in seen if 0 <= p < kv_len):
        k, v = plant(ck, cv, u, pos, d)
        y, launches = run_decode(q, k, v, kv_len)
        assert launches == (2 if splits > 1 else 1)
        assert_is_needle(y, expected_rows(v, pos, heads, 1), f"needle at {pos} of {kv_len} ({splits} splits of {per} tiles)")
    for pos in sorted({kv_len, tile_end - 1}):
        if not kv_len <= pos < tile_end:
            continue
        k, v = plant(ck, cv, u, pos, d)
        y = run_decode(q, k, v, kv_len)[0]
        assert_not_needle(y, expected_rows(v, pos, heads, 1), f"needle at {pos} beyond kv_len {kv_len}")
        close(y, ref_attention(q, k, v, kv_len, kv_len - 1, True)[0], FWD, f"needle at {pos} beyond kv_len {kv_len}")


@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("past,t", [(0, 300), (200, 129), (1000, 64)])
def test_prefill_needle_causal_edge(past, t, dtype, d):
    """Prefill (past 0) and chunked prefill: a needle at key past + i is seen by query i and every later one, never by query
    i - 1; a key-padding byte over it hides it from every query."""
    b, heads, kv = 2, 8, 2
    kv_len = past + t
    q, ck, cv, u = needle_inputs(b, heads, kv, t, kv_len + 16, d, dtype, seed=past + t)
    for i in sorted({0, 1, 63, 64, 127, 128, t // 2, t - 1}):
        if i >= t:
            continue
        pos = past + i
        k, v = plant(ck, cv, u, pos, d)
        y = ops.gqa_attention_forward(q, k, v, kv_len, past, causal=True)
        want = expected_rows(v, pos, heads, t)
        assert_is_needle(y[:, i:], want[:, i:], f"needle at key {pos}: queries {i}..")
        if i > 0:
            assert_not_needle(y[:, :i], want[:, :i], f"needle at key {pos}: queries ..{i - 1}")
            close(y[:, :i], ref_attention(q, k, v, kv_len, past, True)[0][:, :i], FWD, f"needle at key {pos}: queries ..{i - 1}")
        keep = torch.ones(b, kv_len, dtype=torch.uint8, device=DEV)
        keep[:, pos] = 0
        yk = ops.gqa_attention_forward(q, k, v, kv_len, past, causal=True, key_keep=keep)
        assert_not_needle(yk[:, max(i, 1):], want[:, max(i, 1):], f"padded needle at key {pos}")
        close(yk, ref_attention(q, k, v, kv_len, past, True, keep)[0], FWD, f"padded needle at key {pos}")


# ------------------------------------------------------------------------------------------------- chunked prefill
CHUNKED = [(c, p) for c in (2, 17, 64, 127, 128, 129, 300) for p in (1, 63, 64, 200, 1000)]


@pytest.mark.parametrize("chunk,past", CHUNKED)
def test_chunked_prefill_kernels(chunk, past):
    """rope_kv_append + gqa_attention_forward with past_len > 0 (a chunk appended to a cache that holds `past` tokens), causal,
    with and without key padding: against float64 and against the one-shot prefill of the whole sequence."""
    i = CHUNKED.index((chunk, past))
    dtype, d = DTYPES[i % 2], DIMS[(i // 2) % 2]
    b, heads, kv = 2, 8, 2
    total = past + chunk
    g = gen(i)
    max_len = total + 40
    q_all = rnd(g, b, total, heads * d, dtype=dtype)
    k_all, v_all = rnd(g, b, total, kv * d, dtype=dtype), rnd(g, b, total, kv * d, dtype=dtype)
    pos = torch.arange(total, device=DEV)[None].expand(b, -1).contiguous()
    ck = torch.zeros(b, kv, max_len, d, device=DEV, dtype=dtype)
    cv = torch.zeros_like(ck)
    q_past, q_new = q_all[:, :past].contiguous(), q_all[:, past:].contiguous()
    ops.rope_kv_append(q_past, k_all[:, :past].contiguous(), v_all[:, :past].contiguous(), pos[:, :past].contiguous(), ck, cv, 0)
    ops.rope_kv_append(q_new, k_all[:, past:].contiguous(), v_all[:, past:].contiguous(), pos[:, past:].contiguous(), ck, cv, past)
    keep = torch.ones(b, total, dtype=torch.uint8, device=DEV)
    keep[1, : min(70, total - 1)] = 0                                       # left padding longer than a tile
    keep[0, past + chunk // 2] = 0                                          # a padded key inside the chunk
    one_shot_q = torch.cat([q_past, q_new], 1).contiguous()
    for kk in (None, keep):
        y = ops.gqa_attention_forward(q_new, ck, cv, total, past, causal=True, key_keep=kk)
        ref = ref_attention(q_new, ck, cv, total, past, True, kk)[0]
        close(y, ref, FWD, f"chunk {chunk} on {past} ({'padded' if kk is not None else 'no padding'})")
        full = ops.gqa_attention_forward(one_shot_q, ck, cv, total, 0, causal=True, key_keep=kk)[:, past:]
        close(y, full, (1e-3, 2.0 ** -9), "chunk vs one-shot prefill")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("d", DIMS)
def test_module_chunked_prefill_through_one_cache(dtype, d):
    """GroupQueryAttention fills one KVCache chunk by chunk with the model's mask [b, 1, t, past + t] (causal offset plus key
    padding); every chunk against the oracle with the cache contents so far."""
    b, heads, kv = 2, 8, 2
    hidden = heads * d
    torch.manual_seed(d)
    rep = O.bf16_representable if dtype == torch.bfloat16 else O.fp16_representable
    mk = lambda o, i: rep((torch.rand(o, i) * 2 - 1) / i ** 0.5)
    wq, wk, wv, wo = mk(heads * d, hidden), mk(kv * d, hidden), mk(kv * d, hidden), mk(hidden, heads * d)
    att = L.GroupQueryAttention(type("Cfg", (), dict(hidden_size=hidden, n_heads=heads, n_kv_groups=kv, rope_base=500000.0))(),
                                layer_idx=0).to(DEV, dtype).eval()
    with torch.no_grad():
        for m, w in ((att.W_query, wq), (att.W_key, wk), (att.W_value, wv), (att.out_proj, wo)):
            m.weight.copy_(w.to(DEV, dtype))
    chunks = [70, 17, 1, 129, 64, 1]
    total = sum(chunks)
    mask2d = torch.ones(b, total)
    mask2d[1, :5] = 0                                                       # left padding
    mask2d[0, 80:83] = 0                                                    # padded keys inside the second chunk
    cache = L.KVCache(capacity=96)                                          # grows (and copies) once on the way
    pk = pv = None
    past = 0
    for ci, t in enumerate(chunks):
        x = rep(torch.randn(b, t, hidden))
        pos = torch.arange(past, past + t)[None].expand(b, -1).contiguous()
        qpos, kpos = torch.arange(past, past + t), torch.arange(past + t)
        m4 = torch.zeros(b, 1, t, past + t)
        m4 = m4.masked_fill((kpos[None, :] > qpos[:, None])[None, None], float("-inf"))
        m4 = m4 + ((1.0 - mask2d[:, : past + t]) * torch.finfo(torch.float32).min)[:, None, None, :]
        with torch.no_grad():
            y = att(x.to(DEV, dtype), attention_mask=m4.to(DEV, dtype), position_ids=pos.to(DEV), kv_cache=cache)
        yr, pk, pv = O.gqa_attention(x, wq, wk, wv, wo, heads, kv, pos, m4, past_k=pk, past_v=pv)
        live = (mask2d[:, : past + t][:, None, :].bool() & (kpos[None, None, :] <= qpos[None, :, None])).any(-1)   # [b, t]
        close(y.float().cpu()[live], yr[live], FWD, f"chunk {ci} ({t} tokens on {past})")
        past += t
    assert cache.num_items() == total


# ------------------------------------------------------------------------------------------ online-softmax rescale
def rescale_inputs(b, heads, kv, t, kv_len, d, dtype, seed, max_len=None):
    """Scores that grow along the key axis: by ~7.9 log2 units a tile over the first half (no new reference every tile, so P
    reaches ~2^8) and by ~10 a tile over the second (a new reference with a tiny alpha every tile), up to a few hundred;
    the query rows alternate in sign, so in every warp some rows rescale and the others keep their reference."""
    g = gen(seed)
    max_len = max_len or kv_len
    u = (torch.randint(0, 2, (b, kv, 1, d), device=DEV, generator=g) * 2 - 1).float()
    tiles = -(-kv_len // KV_TILE)
    steps = torch.tensor([5.5 if i < tiles // 2 else 7.0 for i in range(tiles)], device=DEV)      # natural units per tile
    base = torch.cumsum(steps, 0) - steps[0]
    j = torch.arange(max_len, device=DEV)
    score = base[(j // KV_TILE).clamp(max=tiles - 1)] - 3.0 * torch.rand(max_len, device=DEV, generator=g)  # q.k / sqrt(d)
    ck = (score[None, None, :, None] / math.sqrt(d) * u).to(dtype)                # [b, kv, max_len, d]
    cv = rnd(g, b, kv, max_len, d, dtype=dtype)
    sign = torch.where(torch.arange(heads // kv * t, device=DEV) % 2 == 0, 1.0, -1.0).view(heads // kv, t)
    qh = u[:, :, None] * sign[None, None, :, :, None]                               # [b, kv, g, t, d]
    q = qh.permute(0, 3, 1, 2, 4).reshape(b, t, heads * d).to(dtype)
    return q, ck.contiguous(), cv


@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("dtype", DTYPES)
def test_online_softmax_rescale(dtype, d):
    """Prefill (with left padding longer than a tile), split decode (splits whose maxima differ by ~10 log2 units each) and the
    training forward with its lse, on scores that force the lazy rescale with 0 < alpha < 1."""
    b, heads, kv, kv_len = 2, 8, 2, 2048
    # prefill: 256 queries at the end of the sequence, key padding over the first 70 keys of sequence 1
    t = 256
    q, ck, cv = rescale_inputs(b, heads, kv, t, kv_len, d, dtype, seed=d)
    keep = torch.ones(b, kv_len, dtype=torch.uint8, device=DEV)
    keep[1, :70] = 0
    for kk in (None, keep):
        y = ops.gqa_attention_forward(q, ck, cv, kv_len, kv_len - t, causal=True, key_keep=kk)
        close(y, ref_attention(q, ck, cv, kv_len, kv_len - t, True, kk)[0], FWD, f"prefill rescale (padding: {kk is not None})")
    # split decode: group 4 at batch 1
    heads_d, kv_d = HEADS[4]
    q1, ck1, cv1 = rescale_inputs(1, heads_d, kv_d, 1, kv_len, d, dtype, seed=d + 1, max_len=kv_len + 3)
    y1, launches = run_decode(q1, ck1, cv1, kv_len)
    assert_plan_taken(1, heads_d, kv_d, d, kv_len, launches)
    assert launches == 2
    close(y1, ref_attention(q1, ck1, cv1, kv_len, kv_len - 1, True)[0], FWD, "split decode rescale")
    # training forward over keys = queries (K / V buffers exactly t rows), causal, left padding
    tt = 1024
    qt, ckt, cvt = rescale_inputs(b, heads, kv, tt, tt, d, dtype, seed=d + 2)
    keep_t = torch.ones(b, tt, dtype=torch.uint8, device=DEV)
    keep_t[1, :70] = 0
    ctx, lse = ops.gqa_attention_forward_train(qt, ckt, cvt, causal=True, key_keep=keep_t)
    ref, ref_lse = ref_attention(qt, ckt, cvt, tt, 0, True, keep_t)
    close(ctx, ref, FWD, "training forward rescale")
    dead = torch.isinf(ref_lse)
    assert dead.any() and torch.isinf(lse[dead]).all() and (lse[dead] > 0).all(), "rows without a key must report +inf"
    err = (lse[~dead].double() - ref_lse[~dead]).abs().max().item()
    assert err <= 2e-3, f"lse (log2 units, up to {ref_lse[~dead].abs().max().item():.0f}) off by {err:.3e}"


# ------------------------------------------------------------------------------------------------ cache tail
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", ["decode_split", "decode_one_pass", "prefill", "chunked_prefill"])
def test_cache_tail_is_never_read(case, dtype, d):
    """Cache rows [kv_len, max_len) hold NaN, then +-Inf, then large finite values: the output must be finite and bit-identical
    to the same call with a zero tail (masked keys get P = 0, and 0 * NaN would still be NaN in P V)."""
    if case.startswith("decode"):
        batch, (heads, kv), t = (1, HEADS[4], 1) if case == "decode_split" else (64, HEADS[4], 1)
    else:
        batch, heads, kv, t = 2, 8, 2, 200
    kv_len = 1000 + 37                                                       # the last tile holds 27 rows of tail
    past = kv_len - t if case != "prefill" else 0
    if case == "prefill":
        kv_len = t
    g = gen(len(case) + d)
    max_len = kv_len + 100
    q = rnd(g, batch, t, heads * d, dtype=dtype)
    ck, cv = rnd(g, batch, kv, max_len, d, dtype=dtype), rnd(g, batch, kv, max_len, d, dtype=dtype)
    ck[:, :, kv_len:] = 0
    cv[:, :, kv_len:] = 0
    if case.startswith("decode"):
        splits = split_plan(batch, heads, kv, kv_len, num_sms())[0]
        assert (splits > 1) == (case == "decode_split"), splits
    base = ops.gqa_attention_forward(q, ck, cv, kv_len, past, causal=True)
    close(base, ref_attention(q, ck, cv, kv_len, past, True)[0], FWD, f"{case} zero tail")
    big = torch.finfo(dtype).max
    tails = {"nan": float("nan"), "inf": None, "finite": big / 2}
    for name, val in tails.items():
        k2, v2 = ck.clone(), cv.clone()
        for x in (k2, v2):
            if val is None:
                x[:, :, kv_len:] = torch.where(torch.rand(x[:, :, kv_len:].shape, device=DEV, generator=g) < 0.5,
                                               float("inf"), float("-inf")).to(dtype)
            else:
                x[:, :, kv_len:] = val
        y = ops.gqa_attention_forward(q, k2, v2, kv_len, past, causal=True)
        assert torch.isfinite(y).all(), f"{case}: {name} in the cache tail reached the output"
        assert torch.equal(y, base), f"{case}: {name} in the cache tail changed the output"


# ------------------------------------------------------------------------------------------------ RoPE + append
def rope_ref(x, pos, d, base=500000.0):
    """float64 rotate_half RoPE of x [b, t, h, d] at positions pos [b, t]; also returns the angles [b, t, d/2]."""
    i = torch.arange(d // 2, device=x.device, dtype=torch.float64)
    inv = base ** (-2.0 * i / d)
    ang = pos.double()[..., None] * inv                                             # [b, t, d/2]
    c, s = torch.cos(ang)[:, :, None], torch.sin(ang)[:, :, None]
    x1, x2 = x.double()[..., : d // 2], x.double()[..., d // 2:]
    return torch.cat([x1 * c - x2 * s, x2 * c + x1 * s], -1), ang


def ulp16(x, dtype):
    """One unit in the last place of |x| in the 16-bit type (its subnormal spacing below the normal range)."""
    mant, tiny = (7, torch.finfo(torch.bfloat16).tiny) if dtype == torch.bfloat16 else (10, torch.finfo(torch.float16).tiny)
    e = torch.floor(torch.log2(x.abs().clamp(min=tiny)))
    return torch.exp2(e - mant)


def rope_tolerance(x, ref, ang, d, dtype, base=500000.0):
    """One 16-bit ulp of the result plus what the kernel's fp32 angle costs.  The kernel forms inv_freq_i = exp2f(-e_i),
    e_i = log2f(base) * 2i/d (the rounding of log2f(base) and of the product is e_i 2^-23 in absolute terms, so inv_freq_i
    is off by ln2 e_i 2^-23 relative, plus exp2f's own few ulp), then the fp32 product pos * inv_freq_i (2^-24 relative)
    and sincosf of it (2 ulp).  The angle error is therefore |angle_i| (ln2 e_i + 3) 2^-23 plus 2^-22 for sincosf, and it
    moves each output element by at most (|x_i| + |x_{i+d/2}|) times that."""
    i = torch.arange(d // 2, device=x.device, dtype=torch.float64)
    e = math.log2(base) * 2.0 * i / d
    dang = ang * (math.log(2.0) * e + 3.0) * 2.0 ** -23 + 2.0 ** -22               # [b, t, d/2]
    xa = x.double().abs()
    mag = (xa[..., : d // 2] + xa[..., d // 2:])                                     # [b, t, h, d/2]
    extra = (mag * dang[:, :, None]).repeat(1, 1, 1, 2)
    return ulp16(ref, dtype) + extra


@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("heads,kv", [(32, 8), (64, 8)])
@pytest.mark.parametrize("past", [0, 37])
def test_rope_kv_append(heads, kv, past, dtype, d):
    """q rotated in place and k rotated into the cache at past_len against a float64 rotation, at positions up to 131071 with
    per-sequence offsets and a non-monotone (padded) row; v copied bit for bit; nothing else of the cache written; k_new and
    v_new untouched."""
    b, t = 4, 33
    g = gen(heads + past + d)
    max_len = past + t + 19
    q = rnd(g, b, t, heads * d, dtype=dtype)
    kn, vn = rnd(g, b, t, kv * d, dtype=dtype), rnd(g, b, t, kv * d, dtype=dtype)
    pos = torch.stack([torch.arange(t), torch.arange(t) + 4000, torch.arange(t) + 131071 - t + 1,
                       torch.tensor([1] * 5 + list(range(70000, 70000 + t - 5)))[torch.randperm(t)]]).to(DEV)
    ck = rnd(g, b, kv, max_len, d, dtype=dtype)                              # sentinel contents
    cv = rnd(g, b, kv, max_len, d, dtype=dtype)
    ck0, cv0, q0, kn0, vn0 = ck.clone(), cv.clone(), q.clone(), kn.clone(), vn.clone()
    ops.rope_kv_append(q, kn, vn, pos, ck, cv, past)
    bits = lambda x: x.view(torch.int16)
    assert torch.equal(bits(kn), bits(kn0)) and torch.equal(bits(vn), bits(vn0)), "k_new / v_new were written"
    outside = torch.ones(max_len, dtype=torch.bool, device=DEV)
    outside[past:past + t] = False
    assert torch.equal(bits(ck[:, :, outside]), bits(ck0[:, :, outside])), "cache_k written outside [past, past + t)"
    assert torch.equal(bits(cv[:, :, outside]), bits(cv0[:, :, outside])), "cache_v written outside [past, past + t)"
    assert torch.equal(bits(cv[:, :, past:past + t]), bits(vn.view(b, t, kv, d).transpose(1, 2))), "v not copied bit for bit"
    for name, x_in, got in (("q", q0.view(b, t, heads, d), q.view(b, t, heads, d)),
                            ("k", kn0.view(b, t, kv, d), ck[:, :, past:past + t].transpose(1, 2))):
        ref, ang = rope_ref(x_in, pos, d)
        tol = rope_tolerance(x_in, ref, ang, d, dtype)
        err = (got.double() - ref).abs()
        bad = err > tol
        assert not bad.any(), (f"{name}: {int(bad.sum())} elements beyond the bound, worst excess "
                               f"{(err - tol).max().item():.3e} at position {pos[bad.nonzero()[0, 0], bad.nonzero()[0, 1]].item()}")


# --------------------------------------------------------------------------------------- module decode with padding
@pytest.mark.parametrize("dtype", DTYPES)
def test_module_decode_honours_key_padding(dtype):
    """A decode step with a [b, 1, 1, kv_len] mask that pads keys matches the module's own reference expressions (on an fp32
    copy of the module) -- the padding must not be dropped on the way to the packed decode kernel."""
    import copy
    b, heads, kv, d, t = 2, 32, 8, 64, 150
    hidden = heads * d
    torch.manual_seed(3)
    att = L.GroupQueryAttention(type("Cfg", (), dict(hidden_size=hidden, n_heads=heads, n_kv_groups=kv, rope_base=500000.0))(),
                                layer_idx=0).to(DEV, dtype).eval()
    att32 = copy.deepcopy(att).float()
    rep = lambda x: x.to(dtype)
    mask2d = torch.ones(b, t + 1, device=DEV)
    mask2d[0, 10:40] = 0
    mask2d[1, :3] = 0
    x = rep(torch.randn(b, t, hidden, device=DEV))
    pos = torch.arange(t, device=DEV)[None].expand(b, -1)
    m4 = O.causal_padding_mask(mask2d[:, :t].cpu(), t).to(DEV)
    cache, cache32 = L.KVCache(), L.KVCache()
    x1 = rep(torch.randn(b, 1, hidden, device=DEV))
    p1 = torch.full((b, 1), t, device=DEV)
    m1 = ((1.0 - mask2d) * torch.finfo(torch.float32).min)[:, None, None, :]        # [b, 1, 1, t + 1]
    with torch.no_grad():
        att(x, attention_mask=m4.to(dtype), position_ids=pos, kv_cache=cache)
        att32._reference_forward(x.float(), m4, pos, cache32)
        y = att(x1, attention_mask=m1.to(dtype), position_ids=p1, kv_cache=cache)
        yr = att32._reference_forward(x1.float(), m1, p1, cache32)
    close(y, yr, FWD, "decode step with padded keys")


# --------------------------------------------------------------------------------------------------- large group
@pytest.mark.parametrize("dtype", DTYPES)
def test_decode_group_larger_than_a_query_tile(dtype):
    """heads 256 over one KV head (a group of 256 rows, two query tiles) at a kv_len that would split: every row computed."""
    batch, heads, kv, d, kv_len = 1, 256, 1, 64, 2048
    q, ck, cv = decode_inputs(batch, heads, kv, kv_len, d, dtype, seed=256, tail=7)
    y, launches = run_decode(q, ck, cv, kv_len)
    close(y, ref_attention(q, ck, cv, kv_len, kv_len - 1, True)[0], FWD, "group 256")
    assert_plan_taken(batch, heads, kv, d, kv_len, launches)
