"""Restatement of the next-token sampling contract (include/l32_ffn.h, l32_sample_tokens) in numpy / float64: the Philox4x32-10
stream, the kept set and the Gumbel-max draw.  The tests compare the CUDA kernel with it."""
import numpy as np

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF


def philox4x32_10(c, k):
    """c: four uint64 arrays (32-bit values), k: two ints -> four uint64 arrays."""
    c = [np.asarray(v, dtype=np.uint64) for v in c]
    k0, k1 = int(k[0]), int(k[1])
    for _ in range(10):
        p0 = c[0] * np.uint64(M0)
        p1 = c[2] * np.uint64(M1)
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & np.uint64(MASK),
             (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1), p0 & np.uint64(MASK)]
        k0, k1 = (k0 + W0) & MASK, (k1 + W1) & MASK
    return c


def uniforms(vocab, seed, position):
    """u_i for i in [0, vocab): ((out[i & 3] >> 8) + 0.5) * 2^-24 of counter (i >> 2, 0, pos_lo, pos_hi), key (seed_lo, seed_hi)."""
    seed, position = int(seed) & ((1 << 64) - 1), int(position) & ((1 << 64) - 1)
    j = np.arange((vocab + 3) // 4, dtype=np.uint64)
    z = np.zeros_like(j)
    out = philox4x32_10([j, z, z + np.uint64(position & MASK), z + np.uint64(position >> 32)], (seed & MASK, seed >> 32))
    r = np.stack(out, axis=1).reshape(-1)[:vocab]
    return ((r >> np.uint64(8)).astype(np.float64) + 0.5) * 2.0 ** -24


def _top_p_cut(x, keep, temperature, top_p):
    """(v_p, margin): the top-p cut-off value over the kept entries of x and the distance of top_p from the nearest mass
    fraction at a value boundary (a kernel in fp32 may only disagree within that distance)."""
    z = x[keep] / np.float64(np.float32(temperature))
    sv = x[keep]
    order = np.argsort(-sv, kind="stable")
    sv, w = sv[order], np.exp(z[order] - z.max())
    frac = np.cumsum(w) / w.sum()
    ends = np.flatnonzero(np.append(sv[1:] != sv[:-1], True))    # last index of each block of equal values
    g = int(np.argmax(frac[ends] >= top_p))
    return sv[ends[g]], float(np.min(np.abs(frac[ends] - top_p)))


def kept_mask(x, temperature, top_k, top_p, want_margin=False):
    """Kept set of a sampled row (temperature > 0): x float64 [V] (the 16-bit logits, -inf allowed)."""
    x = np.asarray(x, dtype=np.float64)
    v = x.size
    keep = x > -np.inf
    margin = np.inf
    if 0 < top_k < v:
        vk = np.sort(x)[::-1][top_k - 1]
        keep &= x >= vk
    if top_p < 1 and keep.any():
        vp, margin = _top_p_cut(x, keep, temperature, top_p)
        keep &= x >= vp
    return (keep, margin) if want_margin else keep


def scores(x, temperature, top_k, top_p, seed, position):
    """Perturbed scores z_i + g_i of the kept tokens (-inf elsewhere), float64."""
    x = np.asarray(x, dtype=np.float64)
    keep = kept_mask(x, temperature, top_k, top_p)
    u = uniforms(x.size, seed, position)
    z = x / np.float64(np.float32(temperature))
    return np.where(keep, z - np.log(-np.log(u)), -np.inf)


def sample(x, temperature, top_k, top_p, seed, position):
    x = np.asarray(x, dtype=np.float64)
    if not temperature > 0:
        return int(np.argmax(x))
    s = scores(x, temperature, top_k, top_p, seed, position)
    return int(np.argmax(s)) if np.isfinite(s).any() else 0
