"""Restatement of the speculative decoding contract (include/l32_ffn.h: l32_ngram_draft_paged, l32_speculative_accept) in
plain Python.  The tests compare the CUDA kernels with it."""


def ngram_draft(history, pending, k, n_min, n_max):
    """(ids [k + 1], draft_len) for S = history + [pending]: the largest n in [n_min, n_max] whose last-n suffix occurs
    earlier in S (latest occurrence j with j + n < |S|) proposes S[j + n, j + n + k) cut at |S|, padded with its last token
    (pending when there is no proposal)."""
    s = list(history) + [pending]
    prop = []
    for n in range(min(n_max, len(s) - 1), n_min - 1, -1):
        suffix = s[len(s) - n:]
        js = [j for j in range(len(s) - n) if s[j:j + n] == suffix]
        if js:
            j = max(js)
            prop = s[j + n:j + n + k]
            break
    pad = prop[-1] if prop else pending
    return [pending] + prop + [pad] * (k - len(prop)), len(prop)


def accept(ids, sampled, new_len):
    """(kept count a + 1, emitted tokens) of one row: a = leading i < new_len - 1 with ids[i + 1] == sampled[i]."""
    a = 0
    while a < new_len - 1 and ids[a + 1] == sampled[a]:
        a += 1
    return a + 1, list(sampled[:a + 1])
