"""Next-token sampling timings on one GPU (V = 128256, the 11B / 90B vocabulary).

1. l32_sample_tokens against a torch sampler with the same semantics (temperature, top-k, top-p with the kept-ties rule,
   then multinomial): the eager-torch path a decode loop uses today.  b in {1, 16, 64, 128}; modes greedy / T only /
   top-k 50 / top-p 0.9 / k + p.
2. The next-token tail at b = 64, H = 4096: last_token_logits (the head on the last rows only) + the sampler, against
   nn.Linear on every row of a 4-token step + the torch sampler; the head's bytes over HBM bandwidth bound the first.

Each number: CUDA-graph replays of 20 calls, median of 5 rounds, the two sides alternated round by round.  The logits
(33 MB at b = 128) stay in L2 between calls, as they do when the head's epilogue has just written them.
Usage: python scripts/sampling_bench.py [--out profiles/r4_sampling_bench.txt]
"""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import llama32_b200 as L  # noqa: E402

DEV = "cuda"
VOCAB, HIDDEN = 128256, 4096
MODES = {"greedy": (0.0, 0, 1.0), "T only": (0.8, 0, 1.0), "top-k 50": (0.8, 50, 1.0), "top-p 0.9": (0.8, 0, 0.9),
         "k + p": (0.8, 50, 0.9)}
HBM_BPS = 7.7e12


def torch_sample(logits, t, k, p):
    """The same contract in torch ops (ties at the cut-offs kept, like the kernel)."""
    if t <= 0:
        return torch.argmax(logits, dim=-1)
    x = logits.float()
    if 0 < k < x.shape[-1]:
        vk = torch.topk(x, k, dim=-1).values[:, -1:]
        x = x.masked_fill(x < vk, float("-inf"))
    if p < 1:
        sx, _ = torch.sort(x, dim=-1, descending=True)
        prob = torch.softmax(sx / t, dim=-1)
        cum = torch.cumsum(prob, dim=-1)
        cut = (cum < p).sum(dim=-1, keepdim=True).clamp_(max=x.shape[-1] - 1)
        vp = torch.gather(sx, -1, cut)
        x = x.masked_fill(x < vp, float("-inf"))
    return torch.multinomial(torch.softmax(x / t, dim=-1), 1)[:, 0]


def graph_of(fn, calls=20):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(calls):
            fn()
    return g


def time_graph(g, calls=20):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    g.replay()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / calls        # us per call


def compare(fa, fb, rounds=5):
    ga, gb = graph_of(fa), graph_of(fb)
    for _ in range(2):
        time_graph(ga), time_graph(gb)
    ta, tb = [], []
    for _ in range(rounds):
        ta.append(time_graph(ga))
        tb.append(time_graph(gb))
    return statistics.median(ta), statistics.median(tb)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "sampling_bench needs a CUDA device"
    lines = []
    say = lambda s: (print(s, flush=True), lines.append(s))
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    say(f"# card, power limit: {smi.stdout.strip().splitlines()[0] if smi.stdout.strip() else 'unknown'}")
    say(f"# torch {torch.__version__}; V = {VOCAB}; CUDA-graph replays of 20 calls, median of 5 alternated rounds; us per call")
    g = torch.Generator(device=DEV).manual_seed(0)
    say("")
    say(f"{'b':>4} {'mode':>10} {'l32_sample_tokens':>18} {'torch':>10} {'speedup':>8}")
    for b in (1, 16, 64, 128):
        logits = (torch.randn(b, VOCAB, generator=g, device=DEV) * 3).to(torch.bfloat16)
        pos = torch.arange(b, dtype=torch.int64, device=DEV)
        sampler = L.TokenSampler(b)
        for mode, (t, k, p) in MODES.items():
            sampler.set_params(t, top_k=k, top_p=p, seed=list(range(b)))
            ours, ref = compare(lambda: sampler(logits, pos), lambda: torch_sample(logits, t, k, p))
            say(f"{b:>4} {mode:>10} {ours:>18.2f} {ref:>10.2f} {ref / ours:>7.2f}x")

    b, t_step = 64, 4
    say("")
    say(f"next-token tail, b = {b}, H = {HIDDEN}, a {t_step}-token step per sequence, k + p mode")
    head = torch.nn.Linear(HIDDEN, VOCAB, bias=False).to(DEV, torch.bfloat16)
    hs = (torch.randn(b, t_step, HIDDEN, generator=g, device=DEV)).to(torch.bfloat16)
    new_lens = torch.full((b,), t_step, dtype=torch.int32, device=DEV)
    pos = torch.arange(b, dtype=torch.int64, device=DEV)
    sampler = L.TokenSampler(b)
    sampler.set_params(0.8, top_k=50, top_p=0.9, seed=list(range(b)))
    t, k, p = MODES["k + p"]

    def ours():
        return sampler(L.last_token_logits(head, hs, new_lens), pos)

    def ref():
        return torch_sample(head(hs)[:, -1], t, k, p)

    head_only, _ = compare(lambda: L.last_token_logits(head, hs, new_lens), ours)
    a, r = compare(ours, ref)
    bound = VOCAB * HIDDEN * 2 / HBM_BPS * 1e6
    say(f"  last_token_logits + l32_sample_tokens : {a:8.2f} us")
    say(f"  nn.Linear on all rows + torch sampler : {r:8.2f} us  ({r / a:.2f}x)")
    say(f"  last_token_logits alone               : {head_only:8.2f} us; head bytes {VOCAB * HIDDEN * 2 / 1e9:.2f} GB over "
        f"{HBM_BPS / 1e12:.1f} TB/s = {bound:.1f} us -> {bound / head_only:.2f} of HBM bandwidth (data-sheet figure)")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
