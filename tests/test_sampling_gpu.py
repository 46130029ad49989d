"""Next-token sampling on the GPU (csrc/sampling.cu, l32_sample_tokens) against the float64 restatement of its contract
(sampling_ref), and the decode-loop layer around it: last_token_logits, TokenSampler, and a paged decoder stack whose
captured decode graph feeds its sampled tokens back as the next input ids."""
import numpy as np
import pytest
import torch
from scipy.stats import chisquare

import llama32_b200 as L
from llama32_b200 import ops
from sampling_ref import kept_mask, scores, uniforms

pytestmark = pytest.mark.gpu
DEV = "cuda"
DTYPES = [torch.bfloat16, torch.float16]
VOCABS = [8, 1000, 128256, 262144]
BATCHES = [1, 7, 64, 128, 300]


def params(b, temperature, top_k=0, top_p=1.0, seed=0, position=0):
    col = lambda v, dt: torch.tensor(v if isinstance(v, list) else [v] * b, dtype=dt, device=DEV)
    seeds = seed if isinstance(seed, list) else [seed] * b
    seeds = [s - (1 << 64) if s >= 1 << 63 else s for s in seeds]
    return (col(temperature, torch.float32), col(top_k, torch.int32), col(top_p, torch.float32),
            torch.tensor(seeds, dtype=torch.int64, device=DEV), col(position, torch.int64))


def draw(logits, *p):
    tok, kmin = ops.sample_tokens(logits, *p, want_kept_min=True)
    torch.cuda.synchronize()
    return tok.cpu().numpy(), kmin.cpu().numpy()


@pytest.mark.parametrize("vocab", VOCABS)
@pytest.mark.parametrize("dtype", DTYPES)
def test_greedy_is_torch_argmax(dtype, vocab):
    g = torch.Generator(device=DEV).manual_seed(vocab)
    for b in BATCHES:
        x = (torch.randn(b, vocab, generator=g, device=DEV) * 3).to(dtype)
        top = x.float().max() + 1
        x[0, -1] = top                                      # a maximum in the last column
        if b > 1:
            x[1, vocab // 2 - 1] = top                      # the same maximum on both sides of a slice boundary (cluster of 8
            x[1, vocab // 2] = top                          # splits 128256 / 262144 in the middle too)
            x[1, 3 % vocab] = top
        if b > 2:
            x[2] = 0                                        # all ties (-0 and +0 equal)
            x[2, 1::2] = -0.0
        temps = [0.0, -1.0, float("nan")] * b
        tok, kmin = draw(x, *params(b, temps[:b], 5, 0.5, 1, 1))
        ref = torch.argmax(x.float(), dim=1).cpu().numpy()
        assert np.array_equal(tok, ref), (b, np.flatnonzero(tok != ref)[:5])
        assert np.array_equal(kmin, x.float().max(dim=1).values.cpu().numpy())


def check_rows(x64, tok, kmin, rows):
    """Kept set exact (kept_min) and per-draw agreement with the float64 restatement on the same Philox stream."""
    checked = 0
    for r, (t, k, p, seed, pos) in enumerate(rows):
        keep, margin = kept_mask(x64[r], t, k, p, want_margin=True)
        if margin < 1e-5:
            continue                                        # a mass boundary within 1e-5 of top_p: fp32 may go either way
        checked += 1
        assert kmin[r] == x64[r][keep].min(), (r, t, k, p, kmin[r], x64[r][keep].min())
        assert keep[tok[r]], (r, t, k, p, tok[r])
        s = scores(x64[r], t, k, p, seed, pos)
        order = np.argsort(-s, kind="stable")[:2]
        best, second = s[order[0]], s[order[1]] if s.size > 1 else -np.inf
        if best - second > 1e-4 * max(1.0, abs(best)):
            assert tok[r] == order[0], (r, t, k, p, tok[r], order)
        else:
            assert tok[r] in order, (r, t, k, p, tok[r], order)
    return checked


@pytest.mark.parametrize("vocab", [1000, 128256])
@pytest.mark.parametrize("dtype", DTYPES)
def test_kept_set_and_draws_match_restatement(dtype, vocab):
    rows = []
    for t in (1e-3, 0.7, 1.0, 100.0):
        for k in (0, 1, 50, vocab - 1, vocab, vocab + 5):
            for p in (1.0, 0.9, 0.5, 1e-4):
                rows.append((t, k, p, len(rows) * 7919 + 3, len(rows) + 11))
    b = len(rows)
    g = torch.Generator(device=DEV).manual_seed(5)
    x = (torch.randn(b, vocab, generator=g, device=DEV) * 2).to(dtype)
    x[::5, :vocab // 3] = float("-inf")                     # -inf entries are never kept
    tok, kmin = draw(x, *params(b, *[[r[i] for r in rows] for i in range(5)]))
    assert check_rows(x.double().cpu().numpy(), tok, kmin, rows) >= b * 3 // 4


@pytest.mark.parametrize("dtype", DTYPES)
def test_philox_tie_in(dtype):
    vocab, b = 128256, 4
    x = torch.zeros(b, vocab, dtype=dtype, device=DEV)
    seeds, pos = [0, 1, 0xDEADBEEF12345678, (1 << 64) - 1], [0, 5, 1 << 33, 77]
    tok, _ = draw(x, *params(b, 1.0, 0, 1.0, seeds, pos))
    for r in range(b):
        assert tok[r] == int(np.argmax(uniforms(vocab, seeds[r], pos[r]))), r


@pytest.mark.parametrize("tkp", [(0.8, 10, 0.9), (1.3, 0, 1.0)])
def test_distribution_chisquare(tkp):
    t, k, p = tkp
    vocab, b, calls = 1000, 128, 160
    gen = torch.Generator().manual_seed(3)
    row = torch.full((vocab,), -30.0)
    hot = torch.randperm(vocab, generator=gen)[:16]
    row[hot] = torch.randn(16, generator=gen) * 1.2
    x = row.to(torch.bfloat16)
    x64 = x.double().numpy()
    keep, margin = kept_mask(x64, t, k, p, want_margin=True)
    assert margin > 1e-3
    z = np.where(keep, x64 / np.float32(t), -np.inf)
    prob = np.exp(z - z.max())
    prob /= prob.sum()
    logits = x.to(DEV)[None].expand(b, vocab).contiguous()
    counts = np.zeros(vocab)
    for c in range(calls):
        tok, _ = draw(logits, *params(b, t, k, p, [1000 + r for r in range(b)], [c * b + r for r in range(b)]))
        np.add.at(counts, tok, 1)
    assert counts[~keep].sum() == 0
    big = prob * b * calls >= 5
    obs, exp = counts[big], prob[big] * b * calls
    j = int(np.argmin(exp))                                 # the rare tokens join the least likely frequent one
    obs[j] += counts[~big].sum()
    exp[j] += prob[~big].sum() * b * calls
    assert chisquare(obs, exp).pvalue > 1e-3


def test_reproducible_across_rows_batches_calls_and_graphs():
    vocab = 128256
    g = torch.Generator(device=DEV).manual_seed(9)
    base = (torch.randn(8, vocab, generator=g, device=DEV) * 2).to(torch.bfloat16)
    pr = dict(temperature=[0.9, 1.0, 0.7, 1.2, 1.0, 0.0, 1.0, 0.5], top_k=[0, 50, 0, 20, 0, 0, 1000, 0],
              top_p=[1.0, 1.0, 0.9, 0.8, 0.95, 1.0, 0.5, 1.0], seed=[11, 12, 13, 14, 15, 16, 17, 18])
    pos = [100, 101, 102, 103, 104, 105, 106, 107]
    ref, _ = draw(base, *params(8, pr["temperature"], pr["top_k"], pr["top_p"], pr["seed"], pos))
    again, _ = draw(base, *params(8, pr["temperature"], pr["top_k"], pr["top_p"], pr["seed"], pos))
    assert np.array_equal(ref, again)
    perm = [5, 0, 7, 3, 1, 6, 2, 4]                          # other row indices, inside a larger batch of other rows
    big = (torch.randn(40, vocab, generator=g, device=DEV) * 2).to(torch.bfloat16)
    at = [3 + 4 * i for i in range(8)]
    big[at] = base[perm]
    cols = {k: [0.5] * 40 for k in ("temperature",)}
    cols.update(top_k=[0] * 40, top_p=[1.0] * 40, seed=list(range(40)), pos=list(range(40)))
    for i, r in enumerate(perm):
        cols["temperature"][at[i]] = pr["temperature"][r]
        cols["top_k"][at[i]], cols["top_p"][at[i]] = pr["top_k"][r], pr["top_p"][r]
        cols["seed"][at[i]], cols["pos"][at[i]] = pr["seed"][r], pos[r]
    tok, _ = draw(big, *params(40, cols["temperature"], cols["top_k"], cols["top_p"], cols["seed"], cols["pos"]))
    assert np.array_equal(tok[at], ref[perm])

    # a graph replayed while the parameters and positions change between replays, against eager calls
    sampler = L.TokenSampler(16)
    logits = torch.zeros(8, vocab, dtype=torch.bfloat16, device=DEV)
    position = torch.zeros(8, dtype=torch.int64, device=DEV)
    logits.copy_(base)
    sampler.set_params(**pr)
    sampler(logits, position)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = sampler(logits, position)
    for step in range(4):
        seeds = [s + step for s in pr["seed"]]
        sampler.set_params(pr["temperature"], pr["top_k"], pr["top_p"], seeds)
        position.copy_(torch.tensor([p + 3 * step for p in pos], device=DEV))
        graph.replay()
        torch.cuda.synchronize()
        eager, _ = draw(base, *params(8, pr["temperature"], pr["top_k"], pr["top_p"], seeds, [p + 3 * step for p in pos]))
        assert np.array_equal(out.cpu().numpy(), eager), step
    assert out.data_ptr() == sampler.tokens.data_ptr()


@pytest.mark.parametrize("b", [1, 64, 128, 129])
def test_last_token_logits_small_m_and_tiled(b):
    vocab, hidden, t = 128256, 4096, 3
    torch.manual_seed(b)
    head = torch.nn.Linear(hidden, vocab, bias=False).to(DEV, torch.bfloat16)
    hs = torch.randn(b, t, hidden, device=DEV).to(torch.bfloat16)
    with torch.no_grad():
        y = L.last_token_logits(head, hs)
    ref = torch.nn.functional.linear(hs[:, -1].float(), head.weight.float())
    err = (y.float() - ref).norm() / ref.norm()
    assert y.shape == (b, vocab) and y.dtype == torch.bfloat16
    assert err < 1e-2, err.item()
    assert ((y.float() - ref).abs() <= 2.0 ** -5 * ref.abs() + 2e-2 * ref.abs().max()).all()


def test_last_token_logits_paged_mixed_step():
    hidden, vocab = 256, 1024
    cache = L.PagedKVCache(num_pages=8, max_batch=4, max_pages_per_seq=2)
    ids = [cache.add_sequence() for _ in range(3)]
    cache.set_batch(ids, [3, 1, 5])
    head = torch.nn.Linear(hidden, vocab, bias=False).to(DEV, torch.bfloat16)
    hs = torch.randn(3, 5, hidden, device=DEV).to(torch.bfloat16)
    with torch.no_grad():
        y = L.last_token_logits(head, hs, cache.new_lens)
        want = ops.linear_forward(hs[[0, 1, 2], [2, 0, 4]].contiguous(), head.weight)
    assert torch.equal(y, want)


class Stack(torch.nn.Module):
    """Embedding -> decoder layers -> final norm -> head, on a PagedKVCache."""

    def __init__(self, vocab, n_layers=2):
        super().__init__()
        from test_gpu_parity import _layer
        from test_attention_paged_gpu import HIDDEN, INTER, N_HEADS, N_KV
        torch.manual_seed(0)
        self.emb = torch.nn.Embedding(vocab, HIDDEN).to(DEV, torch.bfloat16)
        self.layers = torch.nn.ModuleList([_layer(HIDDEN, N_HEADS, N_KV, INTER, seed=i) for i in range(n_layers)])
        for i, blk in enumerate(self.layers):
            blk.att.layer_idx = i
        self.norm = L.LLAMARMSNorm(HIDDEN, 1e-5).to(DEV, torch.bfloat16)
        self.head = torch.nn.Linear(HIDDEN, vocab, bias=False).to(DEV, torch.bfloat16)
        with torch.no_grad():
            self.head.weight.mul_(8.0)                      # logits of a few units: sampling matters

    def forward(self, ids, cache):
        b, t = ids.shape
        pos = cache.past_lens[:b].to(torch.int64)[:, None] + torch.arange(t, device=DEV)[None]
        h = self.emb(ids)
        for blk in self.layers:
            h = blk(h, position_ids=pos, kv_cache=cache)
        return L.last_token_logits(self.head, self.norm(h), cache.new_lens)


def prefill(model, cache, sampler, prompts):
    ids = [cache.add_sequence() for _ in prompts]
    n = max(len(p) for p in prompts)
    x = torch.zeros(len(prompts), n, dtype=torch.int64, device=DEV)
    for r, p in enumerate(prompts):
        x[r, :len(p)] = torch.tensor(p, device=DEV)
    cache.set_batch(ids, [len(p) for p in prompts])
    with torch.no_grad():
        tok = sampler(model(x, cache), cache.past_lens[:len(ids)] + cache.new_lens[:len(ids)]).clone()
    cache.advance()
    return ids, tok


def decode(model, cache, sampler, ids, first, steps, graph):
    """`steps` decode steps from tokens `first`; each step's sampled tokens are the next step's input ids."""
    b = len(ids)
    buf = first.view(b, 1).clone()
    out = []

    def step():
        logits = model(buf, cache)
        tok = sampler(logits, cache.past_lens[:b] + cache.new_lens[:b])
        buf.copy_(tok.view(b, 1))
        return tok

    g = None
    for _ in range(steps):
        cache.set_batch(ids, [1] * b)
        with torch.no_grad():
            if not graph:
                step()
            else:
                if g is None:
                    keep = buf.clone()
                    step()                                  # warm-up (weight casts, workspaces); it rewrites the same rows
                    buf.copy_(keep)
                    torch.cuda.synchronize()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        step()
                g.replay()
        out.append(buf[:, 0].clone())
        cache.advance()
    torch.cuda.synchronize()
    return torch.stack(out, 1).cpu()


def run_loop(graph, prompts, seeds, temperature=1.0):
    model = Stack(1024)
    cache = L.PagedKVCache(num_pages=64, max_batch=8, max_pages_per_seq=8)
    sampler = L.TokenSampler(8)
    sampler.set_params(temperature, top_k=50, top_p=0.95, seed=seeds)
    ids, first = prefill(model, cache, sampler, prompts)
    return first.cpu(), decode(model, cache, sampler, ids, first, 8, graph)


def test_decode_graph_feeds_tokens_back_bit_identical_to_eager():
    g = torch.Generator().manual_seed(1)
    prompts = [torch.randint(0, 1024, (n,), generator=g).tolist() for n in (5, 70, 13)]
    f_e, toks_e = run_loop(False, prompts, [7, 8, 9])
    f_g, toks_g = run_loop(True, prompts, [7, 8, 9])
    assert torch.equal(f_e, f_g)
    assert torch.equal(toks_e, toks_g)


def test_forked_siblings_diverge_by_seed():
    model = Stack(1024)
    cache = L.PagedKVCache(num_pages=64, max_batch=8, max_pages_per_seq=8)
    sampler = L.TokenSampler(8)
    prompt = torch.randint(0, 1024, (70,), generator=torch.Generator().manual_seed(2)).tolist()
    sampler.set_params(0.0)
    (root,), tok = prefill(model, cache, sampler, [prompt])
    kids = [cache.fork(root) for _ in range(3)]
    ids = [root] + kids
    sampler.set_params(1.0, top_k=0, top_p=1.0, seed=[5, 5, 6, 5])
    first = tok.expand(len(ids)).contiguous()              # every sibling continues from the prompt's greedy token
    toks = decode(model, cache, sampler, ids, first, 8, graph=True)
    assert torch.equal(toks[0], toks[1]) and torch.equal(toks[0], toks[3])
    assert not torch.equal(toks[0], toks[2])
