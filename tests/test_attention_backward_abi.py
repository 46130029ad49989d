"""CPU: argument validation of the attention training entry points (l32_gqa_attention_forward_train, _backward and the
backward's workspace size).  Every call here fails validation or is empty, so nothing touches a device."""
import ctypes
import os

import pytest

from llama32_b200 import _lib

BF16, FP16 = 0, 1


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _lib.lib()


def _fwd(lib, q=256, lse=256, batch=2, t=64, heads=8, kv=2, d=128, max_len=64, dtype=BF16):
    p = lambda v: ctypes.c_void_p(v)
    return lib.l32_gqa_attention_forward_train(p(q), p(256), p(256), p(0), p(256), p(lse), batch, t, heads, kv, d, max_len, 1, dtype,
                                               p(0))


def _bwd(lib, dq=256, ws=256, ws_bytes=1 << 20, batch=2, t=64, heads=8, kv=2, d=128, max_len=64, dtype=BF16, base=500000.0):
    p = lambda v: ctypes.c_void_p(v)
    return lib.l32_gqa_attention_backward(p(256), p(256), p(256), p(256), p(256), p(256), p(0), p(256), p(dq), p(256), p(256), p(ws),
                                          ws_bytes, batch, t, heads, kv, d, max_len, 1, base, dtype, p(0))


def test_forward_train_validation(lib):
    assert _fwd(lib, dtype=5) == -1
    assert _fwd(lib, d=96) == -2
    assert _fwd(lib, heads=6, kv=4) == -2
    assert _fwd(lib, max_len=63) == -2              # keys are [0, q_len) of the K / V buffers
    assert _fwd(lib, q=0) == -4
    assert _fwd(lib, lse=0) == -4
    assert _fwd(lib, q=0, lse=0, batch=0) == 0
    assert _fwd(lib, q=0, lse=0, t=0, max_len=1) == 0


def test_backward_validation(lib):
    assert _bwd(lib, dtype=3) == -1
    assert _bwd(lib, d=32) == -2
    assert _bwd(lib, heads=8, kv=3) == -2
    assert _bwd(lib, max_len=10) == -2
    assert _bwd(lib, base=1.0) == -2
    assert _bwd(lib, dq=0) == -4
    assert _bwd(lib, ws=0) == -4
    need = lib.l32_gqa_attention_backward_workspace_bytes(2, 64, 8)
    assert _bwd(lib, ws_bytes=need - 1) == -6
    assert _bwd(lib, dq=0, ws=0, ws_bytes=0, batch=0) == 0
    assert _bwd(lib, dq=0, ws=0, ws_bytes=0, t=0, max_len=1) == 0


def test_backward_workspace_bytes(lib):
    for b, t, h in ((1, 1, 1), (4, 2048, 32), (1, 8192, 32), (3, 300, 8)):
        assert lib.l32_gqa_attention_backward_workspace_bytes(b, t, h) >= 4 * b * h * t
    assert lib.l32_gqa_attention_backward_workspace_bytes(0, 64, 8) == 0
