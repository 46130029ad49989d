"""Paged against contiguous KV-cache attention at the 11B geometry (32 query / 8 KV heads, head_dim 128, bf16).

Each case times one attention call (l32_gqa_attention_forward / _paged, plus the split-KV combine where planned) with CUDA
events over replays of a CUDA graph holding `--calls` calls, the two layouts alternated `--rounds` times; it prints the
median per call and the K + V bytes the step must read (true keys only), with the card's name and power limit.

  uniform decode   b = 1 x 2048, 8 x 8192, 64 x 2048: same keys, same plan (max_kv_len = kv_len)
  ragged decode    64 sequences, lengths spread over 128 .. 4096: contiguous at the max length with a key_keep mask (the
                   unpacked kernel, today's only option) against paged with the true lengths (packed, split plan for 4096)
  prefill          4 x 2048 causal
  empty splits     b = 1, 512 true keys: paged with max_kv_len 8192 against max_kv_len 512

Usage: python scripts/paged_attn_bench.py [--calls 20] [--rounds 5] [--out FILE]
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

HEADS, KV, D, PAGE = 32, 8, 128, ops.KV_PAGE
DT = torch.bfloat16


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else torch.cuda.get_device_name()


def paged_copy(ck, cv, lens, seed):
    """The same keys in shuffled pages: (pool_k, pool_v, block_table)."""
    b = ck.shape[0]
    need = [-(-n // PAGE) for n in lens]
    perm = torch.randperm(sum(need), generator=torch.Generator().manual_seed(seed)).tolist()
    table = torch.zeros(b, max(need), dtype=torch.int32)
    pk = torch.zeros(sum(need), KV, PAGE, D, dtype=DT, device="cuda")
    pv = torch.zeros_like(pk)
    it = iter(perm)
    for j in range(max(need)):
        for i in range(b):
            if j < need[i]:
                p = next(it)
                table[i, j] = p
                n = min(PAGE, lens[i] - j * PAGE)
                pk[p, :, :n] = ck[i, :, j * PAGE:j * PAGE + n]
                pv[p, :, :n] = cv[i, :, j * PAGE:j * PAGE + n]
    return pk, pv, table.cuda()


def timed(fn, calls, rounds_out):
    """Capture `calls` calls of fn in one graph; returns a function that replays it and returns us per call."""
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


def compare(name, fns, kv_bytes, calls, rounds):
    times = {k: [] for k in fns}
    runs = {k: timed(f, calls, times[k]) for k, f in fns.items()}
    for _ in range(rounds):
        for k in fns:
            runs[k]()
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    row = {"case": name, "kv_bytes_read": kv_bytes, **{f"{k}_us": round(v, 2) for k, v in med.items()},
           **{f"{k}_spread_us": [round(min(v), 2), round(max(v), 2)] for k, v in times.items()}}
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("paged_attn_bench.py measures on the GPU; no CUDA device found")
    torch.manual_seed(0)
    head = {"card": card(), "sms": torch.cuda.get_device_properties(0).multi_processor_count,
            "geometry": f"{HEADS}/{KV} heads x {D}, bf16", "timing": f"CUDA events over graph replays of {args.calls} calls"}
    print(json.dumps(head), flush=True)
    rows = [head]
    kvb = lambda lens: sum(lens) * KV * D * 2 * 2
    i32 = lambda x: torch.tensor(x, dtype=torch.int32, device="cuda")

    for b, n in ((1, 2048), (8, 8192), (64, 2048)):
        ck = torch.randn(b, KV, n, D, device="cuda").to(DT)
        cv = torch.randn_like(ck)
        q = torch.randn(b, 1, HEADS * D, device="cuda").to(DT)
        pk, pv, table = paged_copy(ck, cv, [n] * b, b)
        past = i32([n - 1] * b)
        rows.append(compare(f"uniform decode {b} x {n}", {
            "contiguous": lambda: ops.gqa_attention_forward(q, ck, cv, n, n - 1),
            "paged": lambda: ops.gqa_attention_forward_paged(q, pk, pv, table, past, None, max_kv_len=n),
        }, kvb([n] * b), args.calls, args.rounds))
        del ck, cv, pk, pv

    b, top = 64, 4096
    lens = torch.randint(128, top + 1, (b,), generator=torch.Generator().manual_seed(1)).tolist()
    ck = torch.randn(b, KV, top, D, device="cuda").to(DT)
    cv = torch.randn_like(ck)
    keep = (torch.arange(top, device="cuda")[None] < torch.tensor(lens, device="cuda")[:, None]).to(torch.uint8)
    q = torch.randn(b, 1, HEADS * D, device="cuda").to(DT)
    pk, pv, table = paged_copy(ck, cv, lens, 2)
    past = i32([n - 1 for n in lens])
    rows.append(compare(f"ragged decode 64 x [128, 4096] (sum {sum(lens)})", {
        "contiguous_keep": lambda: ops.gqa_attention_forward(q, ck, cv, top, top - 1, key_keep=keep),
        "paged": lambda: ops.gqa_attention_forward_paged(q, pk, pv, table, past, None, max_kv_len=top),
    }, kvb(lens), args.calls, args.rounds))
    del ck, cv, pk, pv

    b, n = 4, 2048
    ck = torch.randn(b, KV, n, D, device="cuda").to(DT)
    cv = torch.randn_like(ck)
    q = torch.randn(b, n, HEADS * D, device="cuda").to(DT)
    pk, pv, table = paged_copy(ck, cv, [n] * b, 3)
    past = i32([0] * b)
    rows.append(compare(f"causal prefill {b} x {n}", {
        "contiguous": lambda: ops.gqa_attention_forward(q, ck, cv, n, 0),
        "paged": lambda: ops.gqa_attention_forward_paged(q, pk, pv, table, past, None, max_kv_len=n),
    }, kvb([n] * b), args.calls, args.rounds))

    n, cap = 512, 8192
    ck = torch.randn(1, KV, n, D, device="cuda").to(DT)
    cv = torch.randn_like(ck)
    q = torch.randn(1, 1, HEADS * D, device="cuda").to(DT)
    pk, pv, table = paged_copy(ck, cv, [n], 4)
    wide = torch.zeros(1, cap // PAGE, dtype=torch.int32, device="cuda")
    wide[:, :table.shape[1]] = table
    past = i32([n - 1])
    rows.append(compare(f"empty splits: 1 x {n} keys, plan for {cap}", {
        "contiguous": lambda: ops.gqa_attention_forward(q, ck, cv, n, n - 1),
        "paged_tight": lambda: ops.gqa_attention_forward_paged(q, pk, pv, table, past, None, max_kv_len=n),
        "paged_capacity": lambda: ops.gqa_attention_forward_paged(q, pk, pv, wide, past, None, max_kv_len=cap),
    }, kvb([n]), args.calls, args.rounds))
    if args.out:
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
