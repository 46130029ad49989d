"""Cascade decode against today's paged decode on batches whose sequences share prefix pages (PagedKVCache.fork).

Each case times one decode-step attention call with CUDA events over replays of a CUDA graph holding `--calls` calls, the
forms alternated `--rounds` times, and prints the median per call with the bytes each form must read (the model below) and
the achieved GB/s, after the card's name and power limit.

  forms      cascade  l32_gqa_attention_forward_paged_cascade with the plan of every group (threshold 1 page, so it is timed
                      below the library's threshold too; `selected` says which form the library takes)
             paged    l32_gqa_attention_forward_paged over the same shared pages: what the library does without the feature
             cascade_unshared  the cascade entry point with an empty plan on the same batch: the cost of the form itself
  geometry   11B (32 / 8 heads) and 90B (64 / 8 heads), head_dim 128, bf16
  workloads  b in {8, 64, 256}, shared prefix in {128, 2048, 8192} tokens, own tokens in {64, 1024}, grouped as one group,
             four groups, or half the batch in one group and half unshared (each with its own copy of the prefix tokens)
  bytes      paged: every sequence's K + V.  cascade: each group's prefix K + V once per query-tile chunk, every sequence's
             own K + V, and the fp32 prefix partials written and read back (members' rows of every item).

Usage: python scripts/cascade_attn_bench.py [--calls 10] [--rounds 5] [--out FILE] [--quick]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from llama32_b200 import ops  # noqa: E402
from llama32_b200.modules import CASCADE_MIN_SHARED_PAGES, cascade_items_capacity, cascade_plan  # noqa: E402

KV, D, PAGE = 8, 128, ops.KV_PAGE
DT = torch.bfloat16
GEOMETRIES = {"11B": 32, "90B": 64}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else torch.cuda.get_device_name()


def timed(fn, calls, rounds_out):
    """Capture `calls` calls of fn in one graph; returns a function that replays it and records us per call."""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(calls):
            fn()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()

    def run():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(5):
            g.replay()
        b.record()
        b.synchronize()
        rounds_out.append(a.elapsed_time(b) * 1e3 / (5 * calls))
    return run


def batch(b, prefix, own, grouping):
    """Page lists and lengths: groups share their prefix pages; unshared rows hold their own prefix copy."""
    n_groups = {"one group": 1, "four groups": 4, "half unshared": 1}[grouping]
    shared_rows = b // 2 if grouping == "half unshared" else b
    pp, total = prefix // PAGE, prefix + own
    nxt = iter(range(1 << 30))
    prefixes = [[next(nxt) for _ in range(pp)] for _ in range(n_groups)]
    tables = []
    for r in range(b):
        head = prefixes[r % n_groups] if r < shared_rows else [next(nxt) for _ in range(pp)]
        tables.append(head + [next(nxt) for _ in range(-(-total // PAGE) - pp)])
    return tables, [total - 1] * b, next(nxt)


def device_plan(plan, b, cap):
    items, members, seq = plan if plan is not None else ([], [], [(0, 0, 0, 0)] * b)
    it = torch.zeros(1 + 5 * cap, dtype=torch.int32)
    it[0] = len(items)
    if items:
        it[1:1 + 5 * len(items)] = torch.tensor(items, dtype=torch.int32).flatten()
    mem = torch.zeros(b, dtype=torch.int32)
    mem[:len(members)] = torch.tensor(members, dtype=torch.int32) if members else mem[:0]
    return it.cuda(), mem.cuda(), torch.tensor(seq, dtype=torch.int32).reshape(b, 4).cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="11B, b = 64 only")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cascade_attn_bench.py measures on the GPU; no CUDA device found")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    head = {"card": card(), "sms": sms, "head_dim": D, "kv_heads": KV, "dtype": "bf16",
            "threshold_pages": CASCADE_MIN_SHARED_PAGES, "timing": f"CUDA events over graph replays of {args.calls} calls"}
    print(json.dumps(head), flush=True)
    rows = [head]
    tok_bytes = KV * D * 2 * 2                                       # K + V of one token, one layer
    for gname, heads in GEOMETRIES.items():
        if args.quick and gname != "11B":
            continue
        group = heads // KV
        cap = cascade_items_capacity(sms, KV)
        for b in ((64,) if args.quick else (8, 64, 256)):
            for prefix in (128, 2048, 8192):
                for own in (64, 1024):
                    for grouping in ("one group", "four groups", "half unshared"):
                        tables, past, num_pages = batch(b, prefix, own, grouping)
                        max_pages = max(len(t) for t in tables)
                        table = torch.zeros(b, max_pages, dtype=torch.int32)
                        for r, t in enumerate(tables):
                            table[r, :len(t)] = torch.tensor(t, dtype=torch.int32)
                        table = table.cuda()
                        pk = torch.randn(num_pages, KV, PAGE, D, device="cuda").to(DT)
                        pv = torch.randn_like(pk)
                        q = torch.randn(b, 1, heads * D, device="cuda").to(DT)
                        past_d, new_d = torch.tensor(past, dtype=torch.int32, device="cuda"), torch.ones(b, dtype=torch.int32, device="cuda")
                        plan = cascade_plan(tables, past, [1] * b, group, cap, min_shared_pages=1)
                        selected = cascade_plan(tables, past, [1] * b, group, cap) is not None
                        dp, de = device_plan(plan, b, cap), device_plan(None, b, cap)
                        mkl = max_pages * PAGE
                        fns = {
                            "cascade": lambda: ops.gqa_attention_forward_paged_cascade(q, pk, pv, table, past_d, new_d, *dp, cap,
                                                                                       max_kv_len=mkl),
                            "paged": lambda: ops.gqa_attention_forward_paged(q, pk, pv, table, past_d, new_d, max_kv_len=mkl),
                            "cascade_unshared": lambda: ops.gqa_attention_forward_paged_cascade(q, pk, pv, table, past_d, new_d,
                                                                                                *de, cap, max_kv_len=mkl),
                        }
                        ref = fns["paged"]()
                        diff = (fns["cascade"]().float() - ref.float()).abs().max().item()
                        times = {k: [] for k in fns}
                        runs = {k: timed(f, args.calls, times[k]) for k, f in fns.items()}
                        for _ in range(args.rounds):
                            for k in fns:
                                runs[k]()
                        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
                        items, _, seq = plan
                        paged_bytes = sum(p + 1 for p in past) * tok_bytes
                        pfx_rows = sum(it[4] * group for it in items) * KV
                        casc_bytes = (sum(it[2] for it in items) * PAGE * tok_bytes
                                      + sum(p + 1 - s[0] * PAGE for p, s in zip(past, seq)) * tok_bytes
                                      + 2 * pfx_rows * (D + 2) * 4)
                        row = {"geometry": gname, "b": b, "prefix": prefix, "own": own, "grouping": grouping,
                               "selected": "cascade" if selected else "paged", "items": len(items),
                               "paged_bytes": paged_bytes, "cascade_bytes": casc_bytes,
                               **{f"{k}_us": round(v, 2) for k, v in med.items()},
                               **{f"{k}_spread_us": [round(min(v), 2), round(max(v), 2)] for k, v in times.items()},
                               "speedup": round(med["paged"] / med["cascade"], 3),
                               "paged_GBps": round(paged_bytes / med["paged"] / 1e3, 1),
                               "cascade_GBps": round(casc_bytes / med["cascade"] / 1e3, 1),
                               "max_abs_diff_vs_paged": diff}
                        print(json.dumps(row), flush=True)
                        rows.append(row)
                        del pk, pv, q, runs
                        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
