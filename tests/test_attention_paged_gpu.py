"""The paged KV cache on the GPU: rope_kv_append_paged and gqa_attention_forward_paged (csrc/attention.cu, kPaged instances)
against a float64 restatement over K / V gathered through the block table, bit-identity with the contiguous path, and
PagedKVCache through GroupQueryAttention with continuous batching and one CUDA graph for every decode step.

Block tables are shuffled, non-monotonic and interleave the pages of different sequences, so a wrong page or an off-by-one
row shows; the "needle" cases give one key a dominant score, so the output is exactly that key's value row or visibly not."""
import ctypes

import pytest
import torch

import llama32_b200 as L
from llama32_b200 import ops
from llama32_b200._lib import lib
from oracle import ffn_oracle as O
from test_attention_inference_gpu import DIMS, DTYPES, FWD, HEADS, assert_is_needle, close, gen, num_sms, ref_attention, rnd, split_plan
from test_gpu_parity import _layer

pytestmark = pytest.mark.gpu
DEV = "cuda"
PAGE = 64
LENS = [1, 63, 64, 65, 128, 129, 2048, 8191]


def i32(x):
    return torch.tensor(x, dtype=torch.int32, device=DEV)


def layout(lens, max_pages, extra, seed):
    """Block table [b, max_pages] (int32, device) over a pool of sum(pages) + `extra` pages: a random permutation handed out
    round-robin over the sequences (interleaved, non-monotonic).  Returns (table, num_pages); `extra` pages are in no table."""
    need = [-(-n // PAGE) for n in lens]
    total = sum(need) + extra
    perm = iter(torch.randperm(total, generator=torch.Generator().manual_seed(seed)).tolist())
    table = torch.zeros(len(lens), max_pages, dtype=torch.int32)
    for j in range(max(need)):
        for b, n in enumerate(need):
            if j < n:
                table[b, j] = next(perm)
    return table.to(DEV), total


def gather(pool, table_row, n):
    """[kv, n, d]: the first n rows of a sequence, through its block-table row."""
    pages = table_row[: -(-n // PAGE)].long()
    kv, d = pool.shape[1], pool.shape[3]
    return pool[pages].permute(1, 0, 2, 3).reshape(kv, -1, d)[:, :n]


def ref_paged(q, pk, pv, table, past, new):
    """float64 causal attention of each sequence over its own keys; padded query rows are zeros."""
    b, t, hd = q.shape
    out = torch.zeros(b, t, hd, dtype=torch.float64, device=DEV)
    for i in range(b):
        n = t if new is None else new[i]
        if n == 0:
            continue
        kl = past[i] + n
        k, v = gather(pk, table[i], kl)[None], gather(pv, table[i], kl)[None]
        out[i, :n] = ref_attention(q[i:i + 1, :n], k, v, kl, past[i], True)[0][0]
    return out


def live_rows(table, lens, num_pages):
    """[num_pages, PAGE] bool: the pool rows that hold a key of some sequence."""
    live = torch.zeros(num_pages, PAGE, dtype=torch.bool)
    tab = table.cpu()
    for i, n in enumerate(lens):
        for j0 in range(0, n, PAGE):
            live[tab[i, j0 // PAGE], : min(PAGE, n - j0)] = True
    return live.to(DEV)


def stale(pool, live, value):
    return torch.where(live[:, None, :, None], pool, torch.full_like(pool, value))


def raw_paged(q, pk, pv, table, past, new, max_kv_len, use_ws=True):
    """One l32_gqa_attention_forward_paged call; returns (ctx, kernel launches it took)."""
    b, t = q.shape[0], q.shape[1]
    num_pages, kv, _, d = pk.shape
    heads = q.shape[-1] // d
    need = lib().l32_gqa_attention_workspace_bytes(b, t, heads, kv, d, max_kv_len)
    ws = torch.empty(need, dtype=torch.uint8, device=DEV) if (use_ws and need) else None
    out = torch.empty_like(q)
    n0 = lib().l32_kernel_launch_count()
    ops.check(lib().l32_gqa_attention_forward_paged(q.data_ptr(), pk.data_ptr(), pv.data_ptr(), table.data_ptr(), past.data_ptr(),
                                                    None if new is None else new.data_ptr(), out.data_ptr(),
                                                    None if ws is None else ws.data_ptr(), need if ws is not None else 0, b, t,
                                                    heads, kv, d, num_pages, table.shape[1], max_kv_len, ops._dtype_code(q),
                                                    ops._stream(q)), "l32_gqa_attention_forward_paged")
    return out, lib().l32_kernel_launch_count() - n0


def splits_of(b, heads, kv, max_kv_len, use_ws):
    return split_plan(b, heads, kv, max_kv_len, num_sms())[0] if use_ws else 1


# --------------------------------------------------------------------------------------------- ragged decode batches
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("group", [1, 2, 4, 8])
def test_ragged_decode(group, dtype, d):
    """One decode step over sequences of lengths 1 .. 8191 in one batch: packed and split-KV (the plan from a tight and from a
    far larger max_kv_len, which leaves splits empty), and one pass without a workspace; random queries against float64,
    then needles at the first, a page-edge, the middle and the last key of every sequence."""
    heads, kv = HEADS[group]
    b, max_pages = len(LENS), 4 * 128
    table, num_pages = layout(LENS, max_pages, extra=7, seed=group * 10 + d)
    g = gen(group + d)
    past, new = [n - 1 for n in LENS], [1] * b
    past_d, new_d = i32(past), i32(new)
    pk, pv = rnd(g, num_pages, kv, PAGE, d, dtype=dtype), rnd(g, num_pages, kv, PAGE, d, dtype=dtype)
    q = rnd(g, b, 1, heads * d, dtype=dtype)
    ref = ref_paged(q, pk, pv, table, past, new)
    for max_kv_len in (8192, max_pages * PAGE):
        for use_ws in (True, False):
            y, launches = raw_paged(q, pk, pv, table, past_d, new_d, max_kv_len, use_ws)
            splits = splits_of(b, heads, kv, max_kv_len, use_ws)
            assert launches == (2 if splits > 1 else 1), (launches, splits)
            close(y, ref, FWD, f"group {group} max_kv_len {max_kv_len} ({splits} splits)")
    # needles: keys ~0, one key per sequence with score 4 sqrt(d) against its group's queries (+-1 rows)
    u = (torch.randint(0, 2, (b, kv, 1, d), device=DEV, generator=g) * 2 - 1).float()
    qn = u[:, :, None].expand(b, kv, heads // kv, 1, d).permute(0, 3, 1, 2, 4).reshape(b, 1, heads * d).to(dtype)
    small = (torch.rand(num_pages, kv, PAGE, d, device=DEV, generator=g) * 0.1 - 0.05).to(dtype)
    for where in ("first", "edge", "middle", "last"):
        kn = small.clone()
        want = torch.empty(b, 1, heads * d, device=DEV)
        for i, n in enumerate(LENS):
            pos = {"first": 0, "edge": min(64, n - 1), "middle": n // 2, "last": n - 1}[where]
            page, row = table[i, pos // PAGE].item(), pos % PAGE
            kn[page, :, row] = (u[i, :, 0] * 4).to(dtype)
            want[i, 0] = pv[page, :, row].float()[:, None].expand(kv, heads // kv, d).reshape(-1)
        for max_kv_len in (8192, max_pages * PAGE):
            y = raw_paged(qn, kn, pv, table, past_d, new_d, max_kv_len)[0]
            assert_is_needle(y, want, f"group {group}: needle at the {where} key, max_kv_len {max_kv_len}")


@pytest.mark.parametrize("dtype", DTYPES)
def test_decode_mostly_empty_splits(dtype):
    """b = 1, 512 true keys, a plan for 8192: most splits get no tile, the combine skips their (-inf, 0) partials."""
    heads, kv = HEADS[4]
    d, n, max_kv_len = 128, 512, 8192
    splits = split_plan(1, heads, kv, max_kv_len, num_sms())[0]
    assert splits > 8, splits                                   # more splits than the sequence has tiles
    table, num_pages = layout([n], max_kv_len // PAGE, extra=3, seed=1)
    g = gen(11)
    pk, pv = rnd(g, num_pages, kv, PAGE, d, dtype=dtype), rnd(g, num_pages, kv, PAGE, d, dtype=dtype)
    q = rnd(g, 1, 1, heads * d, dtype=dtype)
    y, launches = raw_paged(q, pk, pv, table, i32([n - 1]), None, max_kv_len)
    assert launches == 2
    close(y, ref_paged(q, pk, pv, table, [n - 1], [1]), FWD, f"512 keys over {splits} splits")


# --------------------------------------------------------------------------------------------- mixed prefill / decode
MIXED = [(200, 150), (1000, 1), (0, 130), (64, 1)]            # (past, new): chunks onto a cache and decode steps, one call


def mixed_inputs(dtype, d, seed, heads=8, kv=2):
    b, t = len(MIXED), max(n for _, n in MIXED)
    past, new = [p for p, _ in MIXED], [n for _, n in MIXED]
    max_pages = 20
    table, num_pages = layout([p + n for p, n in MIXED], max_pages, extra=5, seed=seed)
    g = gen(seed)
    pk, pv = rnd(g, num_pages, kv, PAGE, d, dtype=dtype), rnd(g, num_pages, kv, PAGE, d, dtype=dtype)   # sentinels + cached keys
    q = rnd(g, b, t, heads * d, dtype=dtype)
    kn, vn = rnd(g, b, t, kv * d, dtype=dtype), rnd(g, b, t, kv * d, dtype=dtype)
    pos = torch.stack([torch.arange(p, p + t) for p in past]).to(DEV)
    return table, num_pages, pk, pv, q, kn, vn, pos, past, new


@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("dtype", DTYPES)
def test_mixed_prefill_and_decode_step(dtype, d):
    """Two sequences prefill a chunk onto a non-empty cache (several tiles) while two decode one token, right-padded to a common
    t: the append writes exactly the real tokens (bit-identical to the contiguous append, every other pool row unchanged),
    padded query rows are exact zeros and the rest matches float64."""
    heads, kv = 8, 2
    table, num_pages, pk, pv, q, kn, vn, pos, past, new = mixed_inputs(dtype, d, seed=d + 3)
    b, t = q.shape[0], q.shape[1]
    pk0, pv0, q0 = pk.clone(), pv.clone(), q.clone()
    ops.rope_kv_append_paged(q, kn, vn, pos, pk, pv, table, i32(past), i32(new))
    want_k, want_v = pk0.clone(), pv0.clone()
    for i, (p, n) in enumerate(MIXED):
        qc = q0[i:i + 1, :n].contiguous()
        ck = torch.zeros(1, kv, n, d, dtype=dtype, device=DEV)
        cv = torch.zeros_like(ck)
        ops.rope_kv_append(qc, kn[i:i + 1, :n].contiguous(), vn[i:i + 1, :n].contiguous(), pos[i:i + 1, :n].contiguous(), ck, cv, 0)
        assert torch.equal(q[i, :n].view(torch.int16), qc[0].view(torch.int16)), f"sequence {i}: q rotation differs"
        for j in range(n):
            page, row = table[i, (p + j) // PAGE].item(), (p + j) % PAGE
            want_k[page, :, row] = ck[0, :, j]
            want_v[page, :, row] = cv[0, :, j]
    assert torch.equal(pk.view(torch.int16), want_k.view(torch.int16)), "pool_k: written outside the real tokens, or wrongly"
    assert torch.equal(pv.view(torch.int16), want_v.view(torch.int16)), "pool_v: written outside the real tokens, or wrongly"
    n0 = lib().l32_kernel_launch_count()
    y = ops.gqa_attention_forward_paged(q, pk, pv, table, i32(past), i32(new))
    assert lib().l32_kernel_launch_count() - n0 == 1
    for i, (_, n) in enumerate(MIXED):
        assert (y[i, n:] == 0).all(), f"sequence {i}: padded query rows are not zero"
    close(y, ref_paged(q, pk, pv, table, past, new), FWD, "mixed step")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", ["decode_split", "decode_packed", "decode_group1", "mixed"])
def test_stale_rows_do_not_leak(case, dtype):
    """Every pool row past the sequences' lengths (inside their last pages and in pages no table names) first zero, then
    large finite values: the same bits come out."""
    d = 128
    if case == "mixed":
        heads, kv = 8, 2
        table, num_pages, pk, pv, q, _, _, _, past, new = mixed_inputs(dtype, d, seed=7)
        lens = [p + n for p, n in MIXED]
        use_ws = True
    else:
        heads, kv = HEADS[1 if case == "decode_group1" else 4]
        lens = LENS
        past, new = [n - 1 for n in lens], [1] * len(lens)
        table, num_pages = layout(lens, 128, extra=4, seed=5)
        g = gen(5)
        pk, pv = rnd(g, num_pages, kv, PAGE, d, dtype=dtype), rnd(g, num_pages, kv, PAGE, d, dtype=dtype)
        q = rnd(g, len(lens), 1, heads * d, dtype=dtype)
        use_ws = case == "decode_split"
    live = live_rows(table, lens, num_pages)
    big = torch.finfo(dtype).max / 2
    outs = []
    for val in (0.0, big, -big):
        y, launches = raw_paged(q, stale(pk, live, val), stale(pv, live, val), table, i32(past), i32(new), table.shape[1] * PAGE,
                                use_ws)
        assert torch.isfinite(y).all(), f"{case}: stale {val} reached the output"
        outs.append(y)
    if case == "decode_split":
        assert launches == 2
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2]), f"{case}: stale rows changed the output"


# --------------------------------------------------------------------------------------------- bit-identity with the contiguous path
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape", ["prefill", "packed_decode", "split_decode"])
def test_bit_identical_to_contiguous(shape, dtype, d):
    """Uniform lengths, max_kv_len = kv_len and the same K / V laid out in shuffled pages give the bits of
    l32_gqa_attention_forward (same tile order, same arithmetic), in the same number of launches."""
    if shape == "prefill":
        (heads, kv), b, past, t = (8, 2), 2, 100, 200
    elif shape == "packed_decode":
        (heads, kv), b, past, t = HEADS[4], 64, 2047, 1
    else:
        (heads, kv), b, past, t = HEADS[4], 1, 2046, 1
    kv_len = past + t
    splits = split_plan(b, heads, kv, kv_len, num_sms())[0] if t == 1 else 1
    assert (splits > 1) == (shape == "split_decode")
    g = gen(kv_len + d)
    q = rnd(g, b, t, heads * d, dtype=dtype)
    ck, cv = rnd(g, b, kv, kv_len + 5, d, dtype=dtype), rnd(g, b, kv, kv_len + 5, d, dtype=dtype)
    max_pages = -(-kv_len // PAGE)
    table, num_pages = layout([kv_len] * b, max_pages, extra=3, seed=d)
    pk, pv = rnd(g, num_pages, kv, PAGE, d, dtype=dtype), rnd(g, num_pages, kv, PAGE, d, dtype=dtype)   # finite stale rows
    for i in range(b):
        for j0 in range(0, kv_len, PAGE):
            n = min(PAGE, kv_len - j0)
            page = table[i, j0 // PAGE].item()
            pk[page, :, :n] = ck[i, :, j0:j0 + n]
            pv[page, :, :n] = cv[i, :, j0:j0 + n]
    n0 = lib().l32_kernel_launch_count()
    yc = ops.gqa_attention_forward(q, ck, cv, kv_len, past, causal=True)
    n1 = lib().l32_kernel_launch_count()
    yp = ops.gqa_attention_forward_paged(q, pk, pv, table, i32([past] * b), None, max_kv_len=kv_len)
    n2 = lib().l32_kernel_launch_count()
    assert n1 - n0 == n2 - n1 == (2 if splits > 1 else 1)
    assert torch.equal(yp, yc), f"{shape}: paged differs from contiguous (max |diff| {(yp.float() - yc.float()).abs().max().item():.3e})"


# --------------------------------------------------------------------------------------------- the module: continuous batching
HIDDEN, N_HEADS, N_KV, INTER = 512, 4, 2, 1408
TOL = (1.5e-2, 2.0 ** -5)                                       # a whole layer deep in 16-bit storage (test_gpu_parity)


class Alone:
    """One sequence run by itself through the contiguous KVCache path of the same layer."""

    def __init__(self, blk):
        self.blk, self.cache, self.len = blk, L.KVCache(), 0

    def run(self, x):                                           # x [n, hidden]
        n = x.shape[0]
        pos = torch.arange(self.len, self.len + n, device=DEV)[None]
        mask = (O.causal_padding_mask(torch.ones(1, n), n) if self.len == 0 else torch.zeros(1, 1, 1, 1)).to(DEV, x.dtype)
        if self.len > 0 and n > 1:
            raise AssertionError("chunks onto a cache are not used here")
        with torch.no_grad():
            y = self.blk(x[None], attention_mask=mask, position_ids=pos, kv_cache=self.cache)
        self.len += n
        return y[0]


def paged_step(blk, cache, ids, xs):
    """One step of the paged layer: row r appends xs[r] ([n_r, hidden]) to sequence ids[r]; returns the real output rows."""
    news = [x.shape[0] for x in xs]
    t = max(news)
    x = torch.zeros(len(ids), t, HIDDEN, dtype=xs[0].dtype, device=DEV)
    for r, xr in enumerate(xs):
        x[r, :xr.shape[0]] = xr
    pos = torch.stack([torch.arange(cache.length(s), cache.length(s) + t) for s in ids]).to(DEV)
    cache.set_batch(ids, news)
    with torch.no_grad():
        y = blk(x, position_ids=pos, kv_cache=cache)
    cache.advance()
    return [y[r, :n] for r, n in enumerate(news)]


@pytest.mark.parametrize("dtype", DTYPES)
def test_module_continuous_batching(dtype):
    """norm1 -> attention over a PagedKVCache -> block tail: a ragged prefill of three sequences, decode steps, then one
    sequence finishes and a new one takes its pages (stale finite contents) and prefills in the same step as the others
    decode.  Every sequence's outputs match that sequence run alone through the contiguous KVCache path."""
    blk = _layer(HIDDEN, N_HEADS, N_KV, INTER, dtype)
    cache = L.PagedKVCache(num_pages=12, max_batch=4, max_pages_per_seq=4)
    g = torch.Generator().manual_seed(3)
    tok = lambda n: torch.randn(n, HIDDEN, generator=g).to(DEV, dtype)
    ids = [cache.add_sequence() for _ in range(3)]
    alone = {s: Alone(blk) for s in ids}

    def step(ids, ns, what):
        xs = [tok(n) for n in ns]
        got = paged_step(blk, cache, ids, xs)
        for s, x, y in zip(ids, xs, got):
            close(y, alone[s].run(x), TOL, f"{what}: sequence {s}")

    step(ids, [70, 5, 130], "ragged prefill")
    for i in range(3):
        step(ids, [1, 1, 1], f"decode {i}")
    freed = set(cache.pages(ids[1]))
    cache.free_sequence(ids[1])
    new = cache.add_sequence()
    alone[new] = Alone(blk)
    ids = [ids[0], ids[2], new]
    step(ids, [1, 1, 40], "two decode while one joins")
    assert freed & set(cache.pages(new)), "the new sequence should reuse freed pages"
    for i in range(2):
        step(ids, [1, 1, 1], f"decode after the join {i}")
    assert [cache.length(s) for s in ids] == [76, 136, 42]


@pytest.mark.parametrize("dtype", DTYPES)
def test_one_graph_for_every_decode_step(dtype):
    """One decode step captured ONCE, replayed for 6 steps with set_batch / advance and new inputs between replays (the
    lengths grow, a page boundary is crossed, the split plan is static): every replay gives the bits of the eager step."""
    blk = _layer(HIDDEN, N_HEADS, N_KV, INTER, dtype)
    caches = [L.PagedKVCache(num_pages=16, max_batch=3, max_pages_per_seq=5) for _ in range(2)]   # [graph, eager]
    g = torch.Generator().manual_seed(4)
    lens = [61, 3, 130]
    prefill = [torch.randn(n, HIDDEN, generator=g).to(DEV, dtype) for n in lens]
    ids = None
    for c in caches:
        ids = [c.add_sequence() for _ in lens]
        paged_step(blk, c, ids, prefill)
    b = len(ids)
    x_buf = torch.zeros(b, 1, HIDDEN, dtype=dtype, device=DEV)
    p_buf = torch.zeros(b, 1, dtype=torch.long, device=DEV)
    graph_cache, eager_cache = caches
    gph, y_buf = None, None
    for i in range(6):
        x = torch.randn(b, 1, HIDDEN, generator=g).to(DEV, dtype)
        eager = paged_step(blk, eager_cache, ids, [x[r] for r in range(b)])
        graph_cache.set_batch(ids, [1] * b)
        x_buf.copy_(x)
        p_buf.copy_(torch.tensor([[graph_cache.length(s)] for s in ids], device=DEV))
        if gph is None:
            torch.cuda.synchronize()
            gph = torch.cuda.CUDAGraph()
            with torch.no_grad(), torch.cuda.graph(gph):
                y_buf = blk(x_buf, position_ids=p_buf, kv_cache=graph_cache)
        gph.replay()
        graph_cache.advance()
        torch.cuda.synchronize()
        for r in range(b):
            assert torch.equal(y_buf[r], eager[r]), f"replay {i}: sequence {r} differs from the eager step"
    assert [graph_cache.length(s) for s in ids] == [67, 9, 136]


# --------------------------------------------------------------------------------------------- argument errors
def test_argument_errors_and_out_of_pages():
    """Bad shapes, dtypes and null pointers return L32_ERR_* with real device buffers; running out of pages raises in
    set_batch before anything is launched."""
    d, kv, heads = 128, 2, 8
    table, num_pages = layout([100], 4, extra=0, seed=0)
    pk = torch.zeros(num_pages, kv, PAGE, d, dtype=torch.bfloat16, device=DEV)
    q = torch.zeros(1, 1, heads * d, dtype=torch.bfloat16, device=DEV)
    past = i32([99])
    out = torch.empty_like(q)
    s = ops._stream(q)
    A = lambda *a: lib().l32_gqa_attention_forward_paged(*a)
    ptrs = (q.data_ptr(), pk.data_ptr(), pk.data_ptr(), table.data_ptr(), past.data_ptr(), None, out.data_ptr(), None, 0)
    assert A(*ptrs, 1, 1, heads, kv, 96, num_pages, 4, 256, 0, s) == -2
    assert A(*ptrs, 1, 1, heads, 3, d, num_pages, 4, 256, 0, s) == -2
    assert A(*ptrs, 1, 1, heads, kv, d, num_pages, 4, 257, 0, s) == -2
    assert A(*ptrs, 1, 1, heads, kv, d, num_pages, 4, 256, 4, s) == -1
    assert A(*ptrs[:3], None, *ptrs[4:], 1, 1, heads, kv, d, num_pages, 4, 256, 0, s) == -4
    assert A(*ptrs[:4], None, *ptrs[5:], 1, 1, heads, kv, d, num_pages, 4, 256, 0, s) == -4
    kn = torch.zeros(1, 1, kv * d, dtype=torch.bfloat16, device=DEV)
    pos = torch.zeros(1, 1, dtype=torch.long, device=DEV)
    R = lambda *a: lib().l32_rope_kv_append_paged(*a)
    rp = (q.data_ptr(), kn.data_ptr(), kn.data_ptr(), pos.data_ptr(), pk.data_ptr(), pk.data_ptr(), table.data_ptr(),
          past.data_ptr(), None)
    assert R(*rp, 1, 1, heads, kv, 80, num_pages, 4, ctypes.c_float(500000.0), 0, s) == -2
    assert R(*rp, 1, 1, heads, kv, d, num_pages, 4, ctypes.c_float(500000.0), 2, s) == -1
    assert R(*rp[:4], None, *rp[5:], 1, 1, heads, kv, d, num_pages, 4, ctypes.c_float(500000.0), 0, s) == -4
    with pytest.raises(ops.L32Error):
        ops.gqa_attention_forward_paged(q.float(), pk, pk, table, past)
    with pytest.raises(ops.L32Error):
        ops.gqa_attention_forward_paged(q, pk, pk, table.long(), past)
    cache = L.PagedKVCache(num_pages=3, max_batch=2, max_pages_per_seq=4)
    a, b = cache.add_sequence(), cache.add_sequence()
    cache.set_batch([a], [128])
    cache.advance()
    n0 = lib().l32_kernel_launch_count()
    with pytest.raises(RuntimeError, match="out of pages"):
        cache.set_batch([a, b], [1, 100])
    assert lib().l32_kernel_launch_count() == n0
