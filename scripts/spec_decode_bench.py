"""Speculative decoding on the paged KV cache: the verify attention, and a graph-replayed verify step of a decoder stack.

Part 1, attention (one call, CUDA events over replays of a CUDA graph holding `--calls` calls, forms alternated `--rounds`
times, median per call), bf16, head_dim 128, 8 kv heads, geometries 11B (32 query heads) and 90B (64):
  verify   l32_gqa_attention_forward_paged_verify, t new tokens per sequence (the pending token + t - 1 drafts)
  general  l32_gqa_attention_forward_paged on the same step: what the library runs for t > 1 without the verify flag
  decode   l32_gqa_attention_forward_paged with t = 1 (the packed decode): the floor
  b in {1, 8, 32, 64}, past in {512, 2048, 8192}, t in {2, 4, 8}.  `KV` = K + V bytes read once per kv head, `HBM` = those
  bytes over the time as a fraction of 7.7 TB/s (the data-sheet bandwidth; the pools exceed L2 at the larger shapes only).

Part 2, a decoder stack at the 11B geometry (hidden 4096, 32 / 8 heads, intermediate 14336, `--layers` layers, random bf16
weights, V = 128256, every sequence at about 1024 cached tokens):
  plain    one decode step as a CUDA graph (forward, head on b rows, sampler) + set_batch / advance on the host
  verify   SpeculativeDecoder.step(graph=True) at k drafts: the graph (n-gram drafts, forward over b (k + 1) tokens, head on
           b (k + 1) rows, sampler, accept) + one read-back, commit and set_batch on the host
  Reported per step: device time of the graph replay, wall time of the whole step, the host gap (wall - device), and
  tokens/s = b * E[emitted] / wall as a function of the mean emitted count E (1 .. k + 1).  Break-even: the E at which the
  verify step makes as many tokens per second as the plain step.  The weights are random, so the acceptance measured here
  says nothing about real text: it is printed as a statistic only.

Usage: python scripts/spec_decode_bench.py [--calls 10] [--rounds 5] [--layers 4] [--out FILE] [--quick]
"""
from __future__ import annotations

import argparse
import os
import statistics
import subprocess
import sys
import time
from types import SimpleNamespace

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import llama32_b200 as L  # noqa: E402
from llama32_b200 import ops  # noqa: E402

KV, D, PAGE = 8, 128, ops.KV_PAGE
DT = torch.bfloat16
HBM = 7.7e12
GEOMETRIES = {"11B": 32, "90B": 64}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else torch.cuda.get_device_name()


def graphed(fn, calls):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(calls):
            fn()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    return g


def event_us(g, calls, reps=5):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        g.replay()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / (reps * calls)


def paged_step(b, past, t, heads, g):
    """Pools, a table (pages shuffled over the pool), lengths and q for b sequences at `past` cached tokens + t new ones."""
    need = -(-(past + t) // PAGE)
    num = b * need
    perm = torch.randperm(num, generator=g).view(b, need).to(torch.int32)
    table = perm.cuda()
    pk = torch.randn(num, KV, PAGE, D, device="cuda", dtype=DT)
    pv = torch.randn_like(pk)
    past_d = torch.full((b,), past, dtype=torch.int32, device="cuda")
    new_d = torch.full((b,), t, dtype=torch.int32, device="cuda")
    q = torch.randn(b, t, heads * D, device="cuda", dtype=DT)
    return q, pk, pv, table, past_d, new_d, need * PAGE


def bench_attention(args, log):
    log("# part 1: attention of one step; us per call (median of alternated rounds); HBM = K+V once per kv head / time / 7.7 TB/s")
    log(f"{'geom':>5} {'b':>3} {'past':>5} {'t':>2} {'verify':>9} {'general':>9} {'decode':>9} {'ver/dec':>8} {'gen/ver':>8} "
        f"{'KV MB':>8} {'HBM ver':>8}")
    g = torch.Generator().manual_seed(0)
    bs = [1, 64] if args.quick else [1, 8, 32, 64]
    pasts = [2048] if args.quick else [512, 2048, 8192]
    for name, heads in GEOMETRIES.items():
        for b in bs:
            for past in pasts:
                q1, pk, pv, table, past_d, new1, max_kv = paged_step(b, past, 8, heads, g)
                floor = None
                for t in (2, 4, 8):
                    q = torch.randn(b, t, heads * D, device="cuda", dtype=DT)
                    new_d = torch.full((b,), t, dtype=torch.int32, device="cuda")
                    q1 = q[:, :1].contiguous()
                    one = torch.ones(b, dtype=torch.int32, device="cuda")
                    forms = {
                        "verify": lambda: ops.gqa_attention_forward_paged_verify(q, pk, pv, table, past_d, new_d, max_kv_len=max_kv),
                        "general": lambda: ops.gqa_attention_forward_paged(q, pk, pv, table, past_d, new_d, max_kv_len=max_kv),
                        "decode": lambda: ops.gqa_attention_forward_paged(q1, pk, pv, table, past_d, one, max_kv_len=max_kv),
                    }
                    if floor is not None:
                        forms.pop("decode")
                    graphs = {k: graphed(f, args.calls) for k, f in forms.items()}
                    times = {k: [] for k in graphs}
                    for _ in range(args.rounds):
                        for k, gr in graphs.items():
                            times[k].append(event_us(gr, args.calls))
                    us = {k: statistics.median(v) for k, v in times.items()}
                    if floor is None:
                        floor = us["decode"]
                    kv_bytes = b * (past + t) * KV * D * 2 * 2
                    log(f"{name:>5} {b:>3} {past:>5} {t:>2} {us['verify']:>9.2f} {us['general']:>9.2f} {floor:>9.2f} "
                        f"{us['verify'] / floor:>8.2f} {us['general'] / us['verify']:>8.2f} {kv_bytes / 1e6:>8.1f} "
                        f"{kv_bytes / (us['verify'] * 1e-6) / HBM:>8.3f}")
                    del graphs
                del pk, pv
                torch.cuda.empty_cache()


class Block(torch.nn.Module):
    def __init__(self, cfg, i):
        super().__init__()
        self.att = L.GroupQueryAttention(cfg, layer_idx=i)
        self.norm1, self.norm2 = L.LLAMARMSNorm(cfg.hidden_size, 1e-5), L.LLAMARMSNorm(cfg.hidden_size, 1e-5)
        self.ff = L.FusedFeedforward(cfg.hidden_size, cfg.intermediate)

    def forward(self, h, pos, cache):
        a = self.att(self.norm1(h), position_ids=pos, kv_cache=cache)
        return L.block_tail(self.norm2, self.ff, a, h)


class Model(torch.nn.Module):
    """Embedding -> decoder layers -> final norm: hidden states [b, t, H] of a paged forward."""

    def __init__(self, layers, vocab):
        super().__init__()
        cfg = SimpleNamespace(hidden_size=4096, n_heads=32, n_kv_groups=8, intermediate=14336)
        self.emb = torch.nn.Embedding(vocab, cfg.hidden_size)
        self.layers = torch.nn.ModuleList([Block(cfg, i) for i in range(layers)])
        self.norm = L.LLAMARMSNorm(cfg.hidden_size, 1e-5)
        for p in self.parameters():
            torch.nn.init.normal_(p, std=0.02)
        self.norm.weight.data.fill_(1.0)
        for blk in self.layers:
            blk.norm1.weight.data.fill_(1.0)
            blk.norm2.weight.data.fill_(1.0)

    def forward(self, ids, cache):
        b, t = ids.shape
        pos = cache.past_lens[:b].to(torch.int64)[:, None] + torch.arange(t, device=ids.device)[None]
        h = self.emb(ids)
        for blk in self.layers:
            h = blk(h, pos, cache)
        return self.norm(h)


def bench_stack(args, log):
    vocab, ctx = 128256, 1024
    torch.manual_seed(0)
    model = Model(args.layers, vocab).cuda().to(DT).eval()
    head = torch.nn.Linear(4096, vocab, bias=False).cuda().to(DT)
    torch.nn.init.normal_(head.weight, std=0.02)
    log(f"\n# part 2: decoder stack at the 11B geometry, {args.layers} layers, V = {vocab}, ~{ctx} cached tokens per sequence, "
        f"greedy; per step: device (graph replay, CUDA events), wall (whole step incl. host work), host gap = wall - device")
    log(f"{'b':>3} {'form':>9} {'device us':>10} {'wall us':>9} {'host us':>8} {'tok/s @E=1':>11} {'@E=k+1':>10} {'break-even E':>12} "
        f"{'E random':>9}")
    steps = 6 if args.quick else 20
    for b in ([1, 16] if args.quick else [1, 16, 32]):
        g = torch.Generator().manual_seed(b)
        prompts = [torch.randint(0, vocab, (ctx,), generator=g).tolist() for _ in range(b)]
        # plain decode step: graph over forward + head + sampler at b rows
        cache = L.PagedKVCache(num_pages=b * (ctx // PAGE + 8), max_batch=b, max_pages_per_seq=ctx // PAGE + 8)
        dec = L.SpeculativeDecoder(model, head, cache, max_batch=b, k=2)
        dec.set_params(0.0)
        first = dec.prefill(prompts)
        ids = list(first)
        sampler = L.TokenSampler(b)
        sampler.set_params(0.0)
        buf = torch.tensor([first[s][0] for s in ids], device="cuda").view(b, 1)

        def plain():
            h = model(buf, cache)
            tok = sampler(ops.linear_forward(h[:, 0].contiguous(), head.weight), cache.past_lens[:b] + 1)
            buf.copy_(tok.view(b, 1))

        cache.set_batch(ids, [1] * b)
        with torch.no_grad():
            plain()
            torch.cuda.synchronize()
            gp = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gp):
                plain()
        dev, wall = [], []
        for _ in range(steps):
            w0 = time.perf_counter()
            cache.set_batch(ids, [1] * b)
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            gp.replay()
            e.record()
            buf[:, 0].cpu()
            cache.advance()
            wall.append((time.perf_counter() - w0) * 1e6)
            dev.append(a.elapsed_time(e) * 1e3)
        p_dev, p_wall = statistics.median(dev[2:]), statistics.median(wall[2:])
        log(f"{b:>3} {'plain':>9} {p_dev:>10.1f} {p_wall:>9.1f} {p_wall - p_dev:>8.1f} {b / p_wall * 1e6:>11.0f} {'':>10} {'':>12} {'':>9}")
        del gp, dec, cache
        torch.cuda.empty_cache()
        for k in (2, 4, 7):
            cache = L.PagedKVCache(num_pages=b * (ctx // PAGE + 8), max_batch=b, max_pages_per_seq=ctx // PAGE + 8)
            dec = L.SpeculativeDecoder(model, head, cache, max_batch=b, k=k)
            dec.set_params(0.0)
            ids = list(dec.prefill(prompts))
            dec.step(ids, graph=True)                        # capture + warm-up
            dev, wall, emitted = [], [], []
            for _ in range(steps):
                w0 = time.perf_counter()
                out = dec.step(ids, graph=True)
                wall.append((time.perf_counter() - w0) * 1e6)
                emitted += [len(v) for v in out.values()]
            gr = dec._graphs[False]
            for _ in range(5):                               # device time of the captured stages on the current batch
                cache.set_batch(ids, [k + 1] * b, verify=True)
                a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                gr.replay()
                e.record()
                e.synchronize()
                dev.append(a.elapsed_time(e) * 1e3)
                cache.commit([0] * b)
            v_dev, v_wall = statistics.median(dev), statistics.median(wall[2:])
            mean_e = sum(emitted) / len(emitted)
            log(f"{b:>3} {'k=' + str(k):>9} {v_dev:>10.1f} {v_wall:>9.1f} {v_wall - v_dev:>8.1f} {b / v_wall * 1e6:>11.0f} "
                f"{b * (k + 1) / v_wall * 1e6:>10.0f} {v_wall / p_wall:>12.2f} {mean_e:>9.2f}")
            del dec, cache
            torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--layers", type=int, default=4)
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("spec_decode_bench.py measures on a CUDA device; none is available")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"# card, power limit: {card()}")
    log(f"# torch {torch.__version__}")
    bench_attention(args, log)
    bench_stack(args, log)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
