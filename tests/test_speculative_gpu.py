"""Speculative decoding on the GPU: the verify attention (csrc/attention.cu, kVerify instances) against float64 with K / V
gathered through shuffled, interleaved block tables; the n-gram draft and accept kernels (csrc/speculative.cu) against the
restatement in spec_ref; and SpeculativeDecoder end to end on the paged decoder stack of test_sampling_gpu, whose emitted
streams must equal plain decoding's up to an explained rounding divergence."""
import numpy as np
import pytest
import torch

import llama32_b200 as L
from llama32_b200 import ops
from llama32_b200._lib import lib
from sampling_ref import scores
from spec_ref import accept, ngram_draft
from test_attention_inference_gpu import FWD, close, gen, rnd
from test_attention_paged_gpu import assert_is_needle, layout, live_rows, raw_paged, ref_paged, stale
from test_sampling_gpu import Stack

pytestmark = pytest.mark.gpu
DEV = "cuda"
PAGE = 64
GEOMS = [(8, 2, 64), (32, 8, 128), (64, 8, 128)]          # (heads, kv_heads, head_dim)


def i32(x):
    return torch.tensor(x, dtype=torch.int32, device=DEV)


def raw_verify(q, pk, pv, table, past, new, max_kv_len, use_ws=True, ws_fill=None):
    """One l32_gqa_attention_forward_paged_verify call; returns (ctx, launches)."""
    b, t = q.shape[0], q.shape[1]
    num_pages, kv, _, d = pk.shape
    heads = q.shape[-1] // d
    need = lib().l32_gqa_attention_verify_workspace_bytes(b, t, heads, kv, d, max_kv_len)
    ws = None
    if use_ws and need:
        ws = torch.full((need,), 255 if ws_fill is None else ws_fill, dtype=torch.uint8, device=DEV)   # 0xff..: NaN floats
    out = torch.full_like(q, float("nan"))
    n0 = lib().l32_kernel_launch_count()
    ops.check(lib().l32_gqa_attention_forward_paged_verify(
        q.data_ptr(), pk.data_ptr(), pv.data_ptr(), table.data_ptr(), past.data_ptr(), None if new is None else new.data_ptr(),
        out.data_ptr(), None if ws is None else ws.data_ptr(), need if ws is not None else 0, b, t, heads, kv, d, num_pages,
        table.shape[1], max_kv_len, ops._dtype_code(q), ops._stream(q)), "l32_gqa_attention_forward_paged_verify")
    return out, lib().l32_kernel_launch_count() - n0


def hadamard(n):
    h = torch.ones(1, 1)
    while h.shape[0] < n:
        h = torch.cat([torch.cat([h, h], 1), torch.cat([h, -h], 1)], 0)
    return h


# --------------------------------------------------------------------------------------------- verify attention
def verify_case(heads, kv, d, t, dtype, seed):
    group = heads // kv
    max_pages = 34
    near_max = max_pages * PAGE - t
    past = [0, 1, 63, 64, 65, 2047, near_max, 100]
    new = [t, max(1, t - 1), t, 1, t, t, t, 0]          # ragged, one row out of the step
    lens = [p + n for p, n in zip(past, new)]
    table, num_pages = layout([max(n, 1) for n in lens], max_pages, extra=5, seed=seed)
    g = gen(seed)
    pk, pv = rnd(g, num_pages, kv, PAGE, d, dtype=dtype), rnd(g, num_pages, kv, PAGE, d, dtype=dtype)
    live = live_rows(table, lens, num_pages)
    big = 3.0e4
    pk, pv = stale(pk, live, big), stale(pv, live, -big)  # stale rows: large finite values, never attended
    q = rnd(g, len(past), t, heads * d, dtype=dtype)
    return group, table, past, new, lens, pk, pv, q, max_pages


@pytest.mark.parametrize("geom", GEOMS)
@pytest.mark.parametrize("tsel", ["1", "2", "4", "8", "max"])
def test_verify_attention_vs_fp64(geom, tsel):
    heads, kv, d = geom
    t = 128 // (heads // kv) if tsel == "max" else int(tsel)
    dtype = torch.bfloat16
    group, table, past, new, lens, pk, pv, q, max_pages = verify_case(heads, kv, d, t, dtype, seed=heads + t)
    past_d, new_d = i32(past), i32(new)
    ref = ref_paged(q, pk, pv, table, past, new)
    general = raw_paged(q, pk, pv, table, past_d, new_d, max(lens))[0]
    for max_kv_len in (max(lens), max_pages * PAGE):
        for use_ws in (True, False):
            y, launches = raw_verify(q, pk, pv, table, past_d, new_d, max_kv_len, use_ws)
            what = f"{geom} t {t} max_kv_len {max_kv_len} ws {use_ws}"
            close(y, ref, FWD, what)
            close(y, general, FWD, what + " vs the general paged kernel")
            for i, n in enumerate(new):                  # padded token rows and the row out of the step: exact zeros
                assert (y[i, n:] == 0).all(), (what, i)
            again = raw_verify(q, pk, pv, table, past_d, new_d, max_kv_len, use_ws, ws_fill=0)[0]
            assert torch.equal(y, again), what           # deterministic, whatever the workspace held
            assert launches == (2 if use_ws else 1), what   # 8 sequences: the plan splits at these lengths


@pytest.mark.parametrize("geom", GEOMS)
@pytest.mark.parametrize("t", [2, 4, 8])
def test_verify_causal_mask_by_row(geom, t):
    """Token i's query is the Hadamard row h_i (all its group heads); key past + i holds the needle 4 h_i plus a trap 8 h_(i-1)
    for token i - 1, for which it is the first masked key.  Every live row must be exactly its own needle's value."""
    heads, kv, d = geom
    dtype = torch.bfloat16
    group = heads // kv
    for past in ([0, 1, 63, 64, 65, 127, 2047], [62, 61, 191, 0, 4000, 8, 1000]):
        b = len(past)
        new = [t] * b
        lens = [p + t for p in past]
        max_pages = -(-max(lens) // PAGE)
        table, num_pages = layout(lens, max_pages, extra=3, seed=t + past[1])
        g = gen(t)
        h = hadamard(d)[1:t + 2].to(DEV)                 # orthogonal +-1 rows
        pk = (torch.rand(num_pages, kv, PAGE, d, device=DEV, generator=g) * 0.1 - 0.05).to(dtype)
        pv = rnd(g, num_pages, kv, PAGE, d, dtype=dtype)
        want = torch.zeros(b, t, heads * d, device=DEV)
        tab = table.cpu()
        for s, p0 in enumerate(past):
            for i in range(t):
                pos = p0 + i
                page, row = tab[s, pos // PAGE].item(), pos % PAGE
                key = 4 * h[i] + (8 * h[i - 1] if i > 0 else 0)
                pk[page, :, row] = key.to(dtype)
                want[s, i] = pv[page, :, row].float()[:, None].expand(kv, group, d).reshape(-1)
        q = h[:t][None, :, None, :].expand(b, t, heads, d).reshape(b, t, heads * d).to(dtype).contiguous()
        for max_kv_len in (max(lens), max_pages * PAGE):
            for use_ws in (True, False):
                y = raw_verify(q, pk, pv, table, i32(past), i32(new), max_kv_len, use_ws)[0]
                assert_is_needle(y, want, f"{geom} t {t} past {past} max_kv_len {max_kv_len} ws {use_ws}")


def test_verify_fp16_and_argument_error():
    heads, kv, d, t = 32, 8, 128, 4
    group, table, past, new, lens, pk, pv, q, max_pages = verify_case(heads, kv, d, t, torch.float16, seed=7)
    ref = ref_paged(q, pk, pv, table, past, new)
    y = ops.gqa_attention_forward_paged_verify(q, pk, pv, table, i32(past), i32(new), max_kv_len=max(lens))
    close(y, ref, FWD, "fp16")
    with pytest.raises(ops.L32Error):
        ops.gqa_attention_forward_paged_verify(q[:, :1].expand(-1, 33, -1).contiguous(), pk, pv, table, i32(past), i32(new))


# --------------------------------------------------------------------------------------------- draft kernel
@pytest.mark.parametrize("k", [1, 4, 15])
def test_ngram_draft_matches_restatement(k):
    rng = np.random.default_rng(k)
    lens = [0, 1, 2, 5, 63, 64, 65, 130, 1000, 4095, 8191, 300]
    max_pages = 128
    table, num_pages = layout([max(n, 1) for n in lens], max_pages, extra=4, seed=k)
    tab = table.cpu().clone()
    # forked rows: the last row shares row 7's first page (a shared full page)
    tab[11, 0] = tab[7, 0]
    table = tab.to(DEV)
    pool = torch.full((num_pages, PAGE), -1, dtype=torch.int32)
    hists, pend = [], []
    for r, n in enumerate(lens):
        hst = rng.integers(0, 6 if r % 2 else 40, n).tolist()
        if r == 11:
            hst[:PAGE] = hists[7][:PAGE]
        if n > 200:                                       # a planted repeat of the tail across a page boundary
            hst[124:129] = hst[-5:]
        hists.append(hst)
        pend.append(int(rng.integers(0, 40)))
        for i, tok in enumerate(hst):
            pool[tab[r, i // PAGE], i % PAGE] = tok
    pool = pool.to(DEV)
    for n_min, n_max in ((1, 3), (2, 4), (1, 1), (3, 16)):
        ids = torch.full((len(lens), k + 1), -5, dtype=torch.int64, device=DEV)
        dl = torch.full((len(lens),), -5, dtype=torch.int32, device=DEV)
        ops.ngram_draft(pool, table, i32(lens), torch.tensor(pend, device=DEV), ids, dl, n_min=n_min, n_max=n_max)
        ids, dl = ids.cpu().tolist(), dl.cpu().tolist()
        for r in range(len(lens)):
            want = ngram_draft(hists[r], pend[r], k, n_min, n_max)
            assert (ids[r], dl[r]) == want, (k, n_min, n_max, r, lens[r])


# --------------------------------------------------------------------------------------------- accept kernel
@pytest.mark.parametrize("k", [1, 4, 7])
def test_accept_every_prefix_length(k):
    w = k + 1
    rows = []
    for a in range(k + 1):
        for past in (0, 62, 63, 64 - a, 127):
            rows.append((a, max(0, past)))
    rows.append((0, 10))                                  # a row out of the step
    b = len(rows)
    past = [p for _, p in rows]
    new = [w] * (b - 1) + [0]
    table, num_pages = layout([p + w for p in past], 4, extra=2, seed=k)
    g = torch.Generator().manual_seed(k)
    ids = torch.randint(0, 1000, (b, w), generator=g)
    s = torch.randint(1000, 2000, (b, w), generator=g)   # never equal to a draft ...
    for r, (a, _) in enumerate(rows):
        s[r, :a] = ids[r, 1:a + 1]                        # ... except the planted agreeing prefix
    sentinel = -7
    pool = torch.full((num_pages, PAGE), sentinel, dtype=torch.int32, device=DEV)
    out = torch.full((b, w + 1), -9, dtype=torch.int64, device=DEV)
    ops.speculative_accept(ids.to(DEV), s.to(DEV).reshape(-1), pool, table, i32(past), i32(new), out)
    pool, out, tab = pool.cpu(), out.cpu(), table.cpu()
    expect = torch.full_like(pool, sentinel)
    for r, (a, p0) in enumerate(rows):
        if new[r] == 0:
            assert (out[r] == -9).all()
            continue
        cnt, emitted = accept(ids[r].tolist(), s[r].tolist(), w)
        assert cnt == a + 1
        assert out[r].tolist() == [cnt] + emitted + [-1] * (w - cnt), (k, r)
        for i in range(cnt):
            pos = p0 + i
            expect[tab[r, pos // PAGE], pos % PAGE] = int(ids[r, i])
    assert torch.equal(pool, expect)                      # every other slot keeps its sentinel


# --------------------------------------------------------------------------------------------- end to end
class Hidden(torch.nn.Module):
    """The test Stack without its head: final-normed hidden states [b, t, H] of a paged forward."""

    def __init__(self, stack):
        super().__init__()
        self.stack = stack

    def forward(self, ids, cache):
        b, t = ids.shape
        pos = cache.past_lens[:b].to(torch.int64)[:, None] + torch.arange(t, device=DEV)[None]
        h = self.stack.emb(ids)
        for blk in self.stack.layers:
            h = blk(h, position_ids=pos, kv_cache=cache)
        return self.stack.norm(h)


def plain_decode(stack, prompts, params, steps):
    """Plain decoding: (streams [b][steps + 1], logits [b][steps + 1] float32) where logits[r][p] produced stream token p."""
    cache = L.PagedKVCache(num_pages=64, max_batch=8, max_pages_per_seq=8)
    sampler = L.TokenSampler(8)
    sampler.set_params(**params)
    b = len(prompts)
    ids = [cache.add_sequence() for _ in prompts]
    x = torch.zeros(b, max(len(p) for p in prompts), dtype=torch.int64, device=DEV)
    for r, p in enumerate(prompts):
        x[r, :len(p)] = torch.tensor(p, device=DEV)
    cache.set_batch(ids, [len(p) for p in prompts])
    streams, logits = [[] for _ in prompts], [[] for _ in prompts]
    with torch.no_grad():
        for step in range(steps + 1):
            lg = stack(x, cache)
            tok = sampler(lg, cache.past_lens[:b] + cache.new_lens[:b]).clone()
            cache.advance()
            for r in range(b):
                streams[r].append(int(tok[r]))
                logits[r].append(lg[r].float().cpu())
            x = tok.view(b, 1)
            cache.set_batch(ids, [1] * b)
    return streams, logits


def first_divergence(spec, spec_logits, plain, plain_logits, params, r, pos0):
    """Index of the first differing token of the two streams (len if none).  At a divergence both paths had the same prefix:
    the two logits rows must agree within the stack's tolerance, and the plain path's winning margin there (argmax gap, or
    the Gumbel-key gap of sampling_ref) must be below what the observed logits difference can flip."""
    n = min(len(spec), len(plain))
    for p in range(n):
        if spec[p] == plain[p]:
            continue
        a, b = spec_logits[p], plain_logits[p]
        assert a is not None, f"row {r}: the streams differ at {p} where both paths ran the same prefill"
        diff = (a - b).abs().max().item()
        assert diff <= 2.0 ** -4 * b.abs().max().item() + 0.05, f"row {r} token {p}: logits differ by {diff}"
        t = params["temperature"][r] if isinstance(params["temperature"], list) else params["temperature"]
        if t <= 0:
            top = torch.topk(b, 2).values
            margin, bound = (top[0] - top[1]).item(), 2 * diff
        else:
            sc = scores(b.double().numpy(), t, params["top_k"], params["top_p"], params["seed"][r], pos0 + p)
            top = np.sort(sc[np.isfinite(sc)])[::-1]
            margin, bound = (top[0] - top[1] if top.size > 1 else np.inf), 2 * diff / np.float32(t)
        assert margin <= bound + 1e-6, f"row {r} token {p}: margin {margin} but the logits moved by only {diff}"
        return p
    return n


def spec_run(stack, prompts, params, k, want, drafts_fn=None, graph=False, ngram=(1, 3)):
    """SpeculativeDecoder until every stream holds `want` tokens: (streams, logits per token, accepted counts per step)."""
    b = len(prompts)
    cache = L.PagedKVCache(num_pages=64, max_batch=8, max_pages_per_seq=8)
    dec = L.SpeculativeDecoder(Hidden(stack), stack.head, cache, max_batch=b, k=k, ngram=ngram)
    dec.set_params(**params)
    first = dec.prefill(prompts)
    sids = list(first)
    streams = [list(first[s]) for s in sids]
    logits = [[None] for _ in sids]
    counts = []
    while min(len(s) for s in streams) < want:
        drafts = drafts_fn(streams, len(counts)) if drafts_fn is not None else None
        out = dec.step(sids, drafts=drafts, graph=graph)
        lg = dec.logits.float().cpu()
        counts.append([len(out[s]) for s in sids])
        for r, s in enumerate(sids):
            for i, tok in enumerate(out[s]):
                streams[r].append(tok)
                logits[r].append(lg[r * (k + 1) + i])
    return streams, logits, counts


GREEDY = dict(temperature=0.0, top_k=0, top_p=1.0, seed=[0, 0, 0])
SAMPLED = dict(temperature=1.0, top_k=50, top_p=0.95, seed=[11, 12, 13])


def repetitive_prompts():
    g = torch.Generator().manual_seed(4)
    motif = lambda n: torch.randint(0, 1024, (n,), generator=g).tolist()
    return [motif(9) * 6, motif(5) * 14 + [3], motif(17) * 3]


@pytest.mark.parametrize("params", [GREEDY, SAMPLED], ids=["greedy", "sampled"])
def test_drafts_from_plain_decoding_are_accepted(params):
    stack, k = Stack(1024), 4
    prompts = repetitive_prompts()
    plain, plain_lg = plain_decode(stack, prompts, params, 24)
    corrupt = [None, 0, 2]                                 # second step: row r's draft corrupted at position corrupt[r]

    def drafts(streams, step):
        d = torch.zeros(len(streams), k, dtype=torch.int64)
        for r, s in enumerate(streams):
            d[r] = torch.tensor(plain[r][len(s):len(s) + k])
            if step == 1 and corrupt[r] is not None:
                d[r, corrupt[r]] += 1
        return d.to(DEV)

    spec, spec_lg, counts = spec_run(stack, prompts, params, k, want=2 * (k + 1) + 1, drafts_fn=drafts)
    for r in range(len(prompts)):
        div = first_divergence(spec[r], spec_lg[r], plain[r], plain_lg[r], params, r, len(prompts[r]))
        if div < len(spec[r]):                             # a rounding divergence, explained above: counts say nothing
            continue
        assert counts[0][r] == k + 1, (r, counts)
        want = k + 1 if corrupt[r] is None else corrupt[r] + 1
        assert counts[1][r] == want, (r, counts)


@pytest.mark.parametrize("params", [GREEDY, SAMPLED], ids=["greedy", "sampled"])
@pytest.mark.parametrize("graph", [False, True])
def test_ngram_streams_equal_plain_decoding(params, graph):
    stack, k, n = Stack(1024), 3, 24
    prompts = repetitive_prompts()
    plain, plain_lg = plain_decode(stack, prompts, params, n)
    spec, spec_lg, counts = spec_run(stack, prompts, params, k, want=n + 1, graph=graph)
    for r in range(len(prompts)):                          # equal, or equal up to an explained divergence
        first_divergence(spec[r], spec_lg[r], plain[r], plain_lg[r], params, r, len(prompts[r]))
    assert all(1 <= c <= k + 1 for row in counts for c in row)
    mean = float(np.mean(counts))
    print(f"mean emitted per step ({'graph' if graph else 'eager'}, {'greedy' if params is GREEDY else 'sampled'}): {mean:.2f}")


def test_captured_step_while_the_batch_changes_is_bit_identical_to_eager():
    stack = Stack(1024)
    g = torch.Generator().manual_seed(6)
    pa, pb, pc = (torch.randint(0, 1024, (n,), generator=g).tolist() for n in (20, 35, 9))

    def run(graph):
        cache = L.PagedKVCache(num_pages=64, max_batch=4, max_pages_per_seq=8)
        dec = L.SpeculativeDecoder(Hidden(stack), stack.head, cache, max_batch=3, k=3)
        dec.set_params(1.0, top_k=50, top_p=0.95, seed=[7, 8])
        first = dec.prefill([pa, pb])
        a, b = list(first)
        log = [first[a], first[b]]
        for _ in range(3):
            out = dec.step([a, b], graph=graph)
            log += [out[a], out[b]]
        dec.free_sequence(a)                              # a sequence leaves ...
        dec.set_params(1.0, top_k=50, top_p=0.95, seed=[9])
        (c, fc), = dec.prefill([pc]).items()              # ... and another joins
        log.append(fc)
        dec.set_params(1.0, top_k=50, top_p=0.95, seed=[8, 9])
        for _ in range(3):
            out = dec.step([b, c], graph=graph)
            log += [out[b], out[c]]
        return log

    assert run(False) == run(True)


def test_forked_siblings_speculating():
    stack, k = Stack(1024), 3
    cache = L.PagedKVCache(num_pages=64, max_batch=8, max_pages_per_seq=8)
    dec = L.SpeculativeDecoder(Hidden(stack), stack.head, cache, max_batch=4, k=k)
    prompt = (torch.randint(0, 1024, (14,), generator=torch.Generator().manual_seed(2)).tolist() * 5)[:70]
    dec.set_params(0.0)
    (root, first), = dec.prefill([prompt]).items()
    kids = [dec.fork(root) for _ in range(3)]
    ids = [root] + kids
    shared = cache.pages(root)[:1]
    assert all(cache.pages(s)[:1] == shared for s in kids)
    snap = [p[shared].clone() for p in cache._pool_k + cache._pool_v + [cache.token_pool()]]
    dec.set_params(1.0, top_k=0, top_p=1.0, seed=[5, 5, 6, 5])
    streams = {s: [] for s in ids}
    for _ in range(5):
        out = dec.step(ids, graph=True)
        for s in ids:
            streams[s] += out[s]
    torch.cuda.synchronize()
    now = [p[shared] for p in cache._pool_k + cache._pool_v + [cache.token_pool()]]
    assert all(torch.equal(a, b) for a, b in zip(snap, now))   # shared K / V / token pages bit-unchanged
    n = min(len(v) for v in streams.values())
    assert streams[root][:n] == streams[kids[0]][:n] == streams[kids[2]][:n]
    assert streams[root][:n] != streams[kids[1]][:n]
