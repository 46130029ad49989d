"""CPU: the next-token sampling contract restated in float64 (sampling_ref), TokenSampler's host-side validation and staging,
and the l32_sample_tokens argument checks (no compute calls without a GPU)."""
import ctypes
import os

import numpy as np
import pytest

import llama32_b200 as L
from llama32_b200 import _lib
from sampling_ref import kept_mask, philox4x32_10, sample, uniforms

NINF = -np.inf


@pytest.mark.parametrize("ctr, key, want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    got = philox4x32_10([np.array([v], dtype=np.uint64) for v in ctr], key)
    assert tuple(int(g[0]) for g in got) == want


def test_uniforms_strictly_inside_and_keyed():
    u = uniforms(4096, 7, 3)
    assert (u > 0).all() and (u < 1).all()
    assert not np.array_equal(u, uniforms(4096, 8, 3))
    assert not np.array_equal(u, uniforms(4096, 7, 4))
    assert np.array_equal(u[:100], uniforms(100, 7, 3))                  # a draw does not depend on the row's length
    # u_i of counter block i >> 2 only: 4 consecutive tokens share one Philox call
    c = philox4x32_10([np.array([1], np.uint64), np.array([0], np.uint64), np.array([3], np.uint64),
                       np.array([0], np.uint64)], (7, 0))
    assert u[5] == ((int(c[1][0]) >> 8) + 0.5) * 2.0 ** -24


def test_top_k_keeps_ties_whole():
    x = np.array([1, 3, 2, 3, 2, 2, 0, 5], dtype=np.float64)
    assert kept_mask(x, 1.0, 4, 1.0).tolist() == [x_ >= 2 for x_ in x]    # v_4 = 2, and all three 2s survive
    assert kept_mask(x, 1.0, 3, 1.0).tolist() == [x_ >= 3 for x_ in x]
    assert kept_mask(x, 1.0, 1, 1.0).tolist() == [x_ == 5 for x_ in x]
    for k in (0, 8, 9, 100):                                               # off
        assert kept_mask(x, 1.0, k, 1.0).all()


def test_top_p_inside_a_tie_block_and_tiny():
    x = np.log(np.array([4, 2, 2, 1, 1, 0.5, 0.5, 0.5], dtype=np.float64))
    # masses 4, 2, 2, ... of 11.5: 4 / 11.5 < 0.5 <= 8 / 11.5 -> the whole 2-block survives
    assert kept_mask(x, 1.0, 0, 0.5).tolist() == [True, True, True] + [False] * 5
    assert kept_mask(x, 1.0, 0, 1e-4).tolist() == [True] + [False] * 7
    assert kept_mask(x, 1.0, 0, 0.85).tolist() == [True] * 5 + [False] * 3  # 10 / 11.5 = 0.87 >= 0.85
    assert kept_mask(x, 1.0, 0, 0.9).all()                                  # 0.87 < 0.9: the 0.5 block joins
    assert kept_mask(x, 1.0, 3, 0.9).tolist() == [True] * 3 + [False] * 5   # top-k first, then top-p over its survivors


def test_minus_inf_never_kept_and_greedy_is_argmax():
    x = np.array([NINF, 1.0, NINF, 1.0, 0.5, NINF, NINF, NINF])
    assert kept_mask(x, 1.0, 0, 1.0).tolist() == [False, True, False, True, True, False, False, False]
    assert kept_mask(x, 1.0, 5, 1.0).tolist() == [False, True, False, True, True, False, False, False]  # v_5 = -inf
    for t in (0.0, -1.0, float("nan")):
        assert sample(x, t, 0, 1.0, 1, 1) == 1                            # smallest index among the maxima
    for seed in range(20):
        assert sample(x, 1.0, 0, 1.0, seed, 9) in (1, 3, 4)
    assert sample(np.full(8, NINF), 1.0, 0, 1.0, 0, 0) == 0


def test_token_sampler_validates_before_staging():
    s = L.TokenSampler(4)                                                  # host staging only without CUDA
    before = s._host.clone()
    bad = [dict(temperature=-0.1), dict(temperature=float("inf")), dict(temperature=float("nan")),
           dict(temperature=1.0, top_k=-1), dict(temperature=1.0, top_k=2.5), dict(temperature=1.0, top_p=0.0),
           dict(temperature=1.0, top_p=1.5), dict(temperature=1.0, seed=-1), dict(temperature=1.0, seed=1 << 64),
           dict(temperature=[1.0] * 5), dict(temperature=[1.0, 1.0], top_k=[1, 2, 3]), dict(temperature=[])]
    for kw in bad:
        with pytest.raises(ValueError):
            s.set_params(**kw)
        assert s._host.equal(before), kw
    s.set_params(temperature=[0.0, 0.7, 1.3], top_k=[0, 50, 1], top_p=0.9, seed=[1, (1 << 64) - 1, 12345])
    sd, tt, tk, tp = s._views(s._host)
    assert tt.tolist()[:3] == [0.0, np.float32(0.7), np.float32(1.3)] and tt[3] == 0
    assert tk.tolist() == [0, 50, 1, 0]
    assert tp.tolist()[:3] == [np.float32(0.9)] * 3 and tp[3] == 1.0
    assert sd.numpy().view(np.uint64).tolist() == [1, (1 << 64) - 1, 12345, 0]
    s.set_params(0.5)                                                      # scalars: every row
    assert s._views(s._host)[1].tolist() == [0.5] * 4


def test_symbols_in_header_and_signatures():
    assert "l32_sample_tokens" in _lib.header_symbols()
    assert "l32_sample_tokens" in _lib.SIGNATURES
    assert "#define L32_SAMPLE_MAX_VOCAB 262144" in open(_lib.HEADER_PATH).read()


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _lib.lib()


def test_sample_tokens_argument_validation_without_device(lib):
    null = ctypes.c_void_p(0)
    one = ctypes.c_void_p(256)   # never dereferenced: validation fails first
    f = lambda *a: lib.l32_sample_tokens(*a)
    # (logits, temperature, top_k, top_p, seed, position, tokens_out, kept_min, batch, vocab, dtype, stream)
    p8 = [one] * 8
    assert f(*p8, 2, 128256, 2, null) == -1                                 # dtype
    for v in (0, 4, 7, 12, 262152, 1 << 20):                                # V bounds and % 8
        assert f(*p8, 2, v, 0, null) == -2, v
    assert f(*p8, -1, 1000, 0, null) == -2                                  # negative batch
    for i in range(7):                                                      # kept_min (7) may be null
        args = list(p8)
        args[i] = null
        assert f(*args, 2, 1000, 0, null) == -4, i
    assert f(ctypes.c_void_p(8), *p8[1:], 2, 1000, 1, null) == -3           # logits not 16-byte aligned
    assert f(*([null] * 8), 0, 1000, 0, null) == 0                          # empty batch
    assert f(*([null] * 8), 0, 8, 1, null) == 0
