"""The cascade decode on the GPU (csrc/attention.cu, kCascade instances + the cascade combine): forked sequences that share
prefix pages, one decode step computed as a prefix pass (each shared prefix read once per query tile of members), an
own-key pass and the combine.  Checked against a float64 restatement over K / V gathered through shuffled, interleaved
block tables, through PagedKVCache.fork and GroupQueryAttention against each sequence run alone, and under a CUDA graph
whose plan changes between replays."""
import pytest
import torch

import llama32_b200 as L
from llama32_b200 import ops
from llama32_b200._lib import lib
from llama32_b200.modules import cascade_items_capacity, cascade_plan
from test_attention_inference_gpu import DIMS, DTYPES, FWD, HEADS, assert_is_needle, close, gen, num_sms, rnd
from test_attention_paged_gpu import HIDDEN, INTER, N_HEADS, N_KV, TOL, Alone, paged_step, ref_paged
from test_gpu_parity import _layer

pytestmark = pytest.mark.gpu
DEV = "cuda"
PAGE = 64
OWN = [1, 63, 64, 65, 700]


def batch_spec(group):
    """(prefix pages, own lengths) per group of members, then unshared rows (prefix None): a group whose members cross a query
    tile's chunk boundary, a 2-member group, a 1-page prefix, and unshared rows."""
    big = {2: 66, 4: 33, 8: 17}[group]
    spec = [(32, [OWN[i % 5] for i in range(big)]), (10, [65, 700]), (1, [1, 64, 63])]
    return spec + [(None, [100]), (None, [1]), (None, [1500])]


def build(spec, seed):
    """Rows' page lists over a shuffled pool (shared prefixes once, every row's own pages interleaved), their lengths (the
    prefix plus own tokens; the decode token is the last) and the table."""
    rng = torch.Generator().manual_seed(seed)
    rows = []                                    # (prefix id, prefix pages, total length)
    for gi, (pp, owns) in enumerate(spec):
        for o in owns:
            rows.append((gi if pp else None, pp or 0, (pp or 0) * PAGE + o))
    own_need = [-(-n // PAGE) - pp for _, pp, n in rows]
    pre_need = [pp for pp, _ in spec if pp]
    total = sum(own_need) + sum(pre_need) + 5
    perm = torch.randperm(total, generator=rng).tolist()
    it = iter(perm)
    prefixes = {gi: [next(it) for _ in range(pp)] for gi, (pp, _) in enumerate(spec) if pp}
    own = [[] for _ in rows]
    for j in range(max(own_need)):               # round-robin: neighbouring pages belong to different rows
        for r, n in enumerate(own_need):
            if j < n:
                own[r].append(next(it))
    tables = [(prefixes[g] if g is not None else []) + own[r] for r, (g, _, _) in enumerate(rows)]
    lens = [n for _, _, n in rows]
    max_pages = max(len(t) for t in tables) + 2
    table = torch.zeros(len(rows), max_pages, dtype=torch.int32)
    for r, t in enumerate(tables):
        table[r, :len(t)] = torch.tensor(t, dtype=torch.int32)
    return tables, lens, table.to(DEV), total


def plan_tensors(plan, b, max_items):
    items, members, seq = plan
    it = torch.zeros(1 + 5 * max_items, dtype=torch.int32)
    it[0] = len(items)
    if items:
        it[1:1 + 5 * len(items)] = torch.tensor(items, dtype=torch.int32).flatten()
    mem = torch.zeros(b, dtype=torch.int32)
    if members:
        mem[:len(members)] = torch.tensor(members, dtype=torch.int32)
    sq = torch.tensor(seq, dtype=torch.int32).reshape(b, 4)
    return it.to(DEV), mem.to(DEV), sq.to(DEV)


def raw_cascade(q, pk, pv, table, past, new, plan, max_items, max_kv_len, fill=None):
    """One l32_gqa_attention_forward_paged_cascade call; `fill` pre-fills the workspace bytes.  Returns (ctx, launches)."""
    b = q.shape[0]
    num_pages, kv, _, d = pk.shape
    heads = q.shape[-1] // d
    need = lib().l32_gqa_attention_cascade_workspace_bytes(b, heads, kv, d, max_kv_len, max_items)
    ws = torch.full((need,), 0 if fill is None else fill, dtype=torch.uint8, device=DEV)
    items, mem, sq = plan
    out = torch.empty_like(q)
    n0 = lib().l32_kernel_launch_count()
    ops.check(lib().l32_gqa_attention_forward_paged_cascade(
        q.data_ptr(), pk.data_ptr(), pv.data_ptr(), table.data_ptr(), past.data_ptr(), None if new is None else new.data_ptr(),
        items.data_ptr(), mem.data_ptr(), sq.data_ptr(), out.data_ptr(), ws.data_ptr(), need, b, heads, kv, d, num_pages,
        table.shape[1], max_kv_len, max_items, ops._dtype_code(q), ops._stream(q)), "l32_gqa_attention_forward_paged_cascade")
    return out, lib().l32_kernel_launch_count() - n0


@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("group", [2, 4, 8])
def test_cascade_against_float64(group, dtype, d):
    """Groups of 66 / 33 / 17 members (over a chunk boundary), of 2 and of 3, unshared rows; prefixes of 32, 10 and 1 pages,
    own lengths 1 .. 700.  Random queries against float64; a NaN-filled workspace gives the same bits; two calls give the
    same bits; then needles at the first and last prefix key and the first and last own key of every row."""
    heads, kv = HEADS[group]
    tables, lens, table, num_pages = build(batch_spec(group), seed=group * 7 + d)
    b = len(lens)
    past = [n - 1 for n in lens]
    max_items = cascade_items_capacity(num_sms(), kv)
    plan = cascade_plan(tables, past, [1] * b, group, max_items, min_shared_pages=1)
    assert plan is not None and len(plan[0]) <= max_items
    shared = [s[0] for s in plan[2]]
    assert sorted(set(shared)) == [0, 1, 10, 32]
    dplan = plan_tensors(plan, b, max_items)
    g = gen(group + d)
    pk, pv = rnd(g, num_pages, kv, PAGE, d, dtype=dtype), rnd(g, num_pages, kv, PAGE, d, dtype=dtype)
    q = rnd(g, b, 1, heads * d, dtype=dtype)
    past_d, new_d = torch.tensor(past, dtype=torch.int32, device=DEV), torch.ones(b, dtype=torch.int32, device=DEV)
    max_kv_len = table.shape[1] * PAGE
    y, launches = raw_cascade(q, pk, pv, table, past_d, new_d, dplan, max_items, max_kv_len)
    assert launches == 2
    close(y, ref_paged(q, pk, pv, table, past, [1] * b), FWD, f"group {group}")
    y_nan = raw_cascade(q, pk, pv, table, past_d, new_d, dplan, max_items, max_kv_len, fill=0xFF)[0]
    y_again = raw_cascade(q, pk, pv, table, past_d, None, dplan, max_items, max_kv_len)[0]
    assert torch.equal(y, y_nan), "a NaN-filled workspace changed the result"
    assert torch.equal(y, y_again), "two calls differ"
    # needles: keys ~0, one key per row with a dominant score against its group's queries
    u = (torch.randint(0, 2, (kv, d), device=DEV, generator=g) * 2 - 1).float()
    qn = u[:, None].expand(kv, heads // kv, d).reshape(1, 1, heads * d).expand(b, 1, heads * d).contiguous().to(dtype)
    small = (torch.rand(num_pages, kv, PAGE, d, device=DEV, generator=g) * 0.1 - 0.05).to(dtype)
    tab = table.cpu()
    for where in ("first prefix", "last prefix", "first own", "last own"):
        kn = small.clone()
        want = torch.empty(b, 1, heads * d, device=DEV)
        for i, n in enumerate(lens):
            p = shared[i] * PAGE
            pos = {"first prefix": 0, "last prefix": max(p - 1, 0), "first own": p, "last own": n - 1}[where]
            page, row = tab[i, pos // PAGE].item(), pos % PAGE
            kn[page, :, row] = (u * 4).to(dtype)
            want[i, 0] = pv[page, :, row].float()[:, None].expand(kv, heads // kv, d).reshape(-1)
        y = raw_cascade(qn, kn, pv, table, past_d, new_d, dplan, max_items, max_kv_len)[0]
        assert_is_needle(y, want, f"group {group}: needle at the {where} key")


@pytest.mark.parametrize("dtype", DTYPES)
def test_cascade_empty_plan_and_padding_rows(dtype):
    """An empty plan is the plain decode over the own-key pass alone; a row with new_len 0 gives zeros."""
    heads, kv = HEADS[4]
    d = 128
    tables, lens, table, num_pages = build([(None, [70, 1, 3000])], seed=5)
    past = [n - 1 for n in lens]
    max_items = cascade_items_capacity(num_sms(), kv)
    empty = plan_tensors(([], [], [(0, 0, 0, 0)] * 3), 3, max_items)
    g = gen(9)
    pk, pv = rnd(g, num_pages, kv, PAGE, d, dtype=dtype), rnd(g, num_pages, kv, PAGE, d, dtype=dtype)
    q = rnd(g, 3, 1, heads * d, dtype=dtype)
    new = [1, 0, 1]
    y = raw_cascade(q, pk, pv, table, torch.tensor(past, dtype=torch.int32, device=DEV),
                    torch.tensor(new, dtype=torch.int32, device=DEV), empty, max_items, table.shape[1] * PAGE, fill=0xFF)[0]
    assert (y[1] == 0).all()
    close(y, ref_paged(q, pk, pv, table, past, new), FWD, "empty plan")


# --------------------------------------------------------------------------------------------- the module
def snapshot(cache, pages):
    return [(k[pages].clone(), v[pages].clone()) for k, v in zip(cache._pool_k, cache._pool_v)]


@pytest.mark.parametrize("dtype", DTYPES)
def test_module_fork_flow(dtype, monkeypatch):
    """A prompt prefilled once and forked; the children prefill their own tokens in a mixed step while the parent decodes;
    cascade decode steps; the parent is freed and a fork of a child joins.  Every sequence's outputs match that sequence run
    alone through the contiguous KVCache; shared pages keep their bits; an unshared batch never takes the cascade."""
    blk = _layer(HIDDEN, N_HEADS, N_KV, INTER, dtype)
    cache = L.PagedKVCache(num_pages=40, max_batch=6, max_pages_per_seq=8)
    g = torch.Generator().manual_seed(5)
    tok = lambda n: torch.randn(n, HIDDEN, generator=g).to(DEV, dtype)
    hist, alone = {}, {}

    def step(ids, ns, what, cascade):
        xs = [tok(n) for n in ns]
        got = paged_step(blk, cache, ids, xs)
        assert cache.cascade == cascade, what
        for s, x, y in zip(ids, xs, got):
            hist[s] = torch.cat([hist[s], x]) if s in hist else x
            if s in alone and (x.shape[0] == 1 or alone[s].len == 0):
                want = alone[s].run(x)
            else:                                 # a fork's first step, or a chunk onto a cache: the whole history at once
                alone[s] = Alone(blk)
                want = alone[s].run(hist[s])[-x.shape[0]:]
            close(y, want, TOL, f"{what}: sequence {s}")

    parent = cache.add_sequence()
    step([parent], [300], "prompt", False)
    kids = [cache.fork(parent) for _ in range(3)]
    for k in kids:
        hist[k] = hist[parent]
    shared = cache.pages(parent)[:300 // PAGE]
    before = snapshot(cache, shared)
    ids = [parent] + kids
    step(ids, [1, 20, 5, 70], "children prefill while the parent decodes", False)
    for i in range(3):
        step(ids, [1, 1, 1, 1], f"cascade decode {i}", True)
    cache.free_sequence(parent)
    new = cache.fork(kids[0])
    hist[new] = hist[kids[0]]
    ids = kids + [new]
    for i in range(3):
        step(ids, [1, 1, 1, 1], f"decode after the parent left and a fork joined {i}", True)
    after = snapshot(cache, shared)
    assert all(torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) for a, b in zip(before, after)), "a shared page changed"
    # unrelated sequences: the plain paged decode, nothing else
    others = [cache.add_sequence() for _ in range(2)]
    step(others, [130, 300], "unrelated prefill", False)

    def refuse(*a, **k):
        raise AssertionError("the cascade ran for an unshared batch")
    monkeypatch.setattr(ops, "gqa_attention_forward_paged_cascade", refuse)
    step(others, [1, 1], "unshared decode", False)


@pytest.mark.parametrize("dtype", DTYPES)
def test_graph_replay_while_groups_change(dtype):
    """A cascade decode captured once and replayed while a member finishes, a fork joins, an unshared sequence joins and
    finally no group is left: every replay equals the eager call with the same plan bit for bit and matches float64."""
    heads, kv = HEADS[4]
    d, b = 128, 6
    cache = L.PagedKVCache(num_pages=200, max_batch=b, max_pages_per_seq=24)
    cache.cascade_geometry = (heads // kv, kv)
    pk, pv = cache.pools(0, kv, d, dtype, DEV)
    g = gen(21)
    pk.copy_(rnd(g, *pk.shape, dtype=dtype))
    pv.copy_(rnd(g, *pv.shape, dtype=dtype))
    root = cache.add_sequence()
    cache.set_batch([root], [600])
    cache.advance()
    ids = [root] + [cache.fork(root) for _ in range(3)]
    solo = cache.add_sequence()
    cache.set_batch([solo], [200])
    cache.advance()
    q_buf = torch.zeros(b, 1, heads * d, dtype=dtype, device=DEV)

    def call():
        return ops.gqa_attention_forward_paged_cascade(q_buf, pk, pv, cache.block_table, cache.past_lens, cache.new_lens,
                                                       cache.plan_items, cache.plan_members, cache.plan_seq,
                                                       cache.cascade_max_items, max_kv_len=cache.max_kv_len)
    events = ["start", "member finishes", "fork joins", "unshared joins", "no group left"]
    gph, y_buf = None, None
    for i, ev in enumerate(events):
        if ev == "member finishes":
            cache.free_sequence(ids.pop(1))
        elif ev == "fork joins":
            ids.append(cache.fork(ids[0]))
        elif ev == "unshared joins":
            ids.append(solo)
        elif ev == "no group left":
            for s in ids[1:-1]:
                cache.free_sequence(s)
            ids = [ids[0], ids[-1]]
        cache.set_batch(ids, [1] * len(ids))
        assert cache.cascade == (ev != "no group left"), ev
        q_buf.copy_(rnd(g, b, 1, heads * d, dtype=dtype))
        if gph is None:
            call()
            torch.cuda.synchronize()
            gph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gph):
                y_buf = call()
        gph.replay()
        eager = call()
        torch.cuda.synchronize()
        assert torch.equal(y_buf, eager), f"{ev}: the replay differs from the eager call"
        n = len(ids)
        tab = cache.block_table[:n]
        close(y_buf[:n], ref_paged(q_buf[:n], pk, pv, tab, [cache.length(s) for s in ids], [1] * n), FWD, ev)
        assert (y_buf[n:] == 0).all()
        cache.advance()
