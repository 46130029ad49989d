"""CPU check of the tiled GEMM's launch plan: the Python restatement in gemm_plan.py, which the GPU tests use to pick a shape
for each tiling regime, must agree with what the library plans (l32_debug_gemm_plan) -- cta_group, tiles, the SwiGLU
act-tile width n_act, the raster group and the persistent grid size."""
import pytest

import gemm_plan as P
from llama32_b200 import _lib

MS = [1, 2, 77, 127, 128, 129, 255, 256, 257, 383, 512, 1000, 2047, 2048, 4096, 6144, 8191, 16384]
NS = [8, 120, 248, 256, 264, 1032, 1792, 4744, 5928, 7112, 8296, 14336, 28672]


@pytest.mark.parametrize("sms", [148, 132, 160])
@pytest.mark.parametrize("epilogue", [P.EPI_STORE, P.EPI_SWIGLU, P.EPI_SWIGLU_BWD, P.EPI_CE])
def test_plan_matches_the_library(sms, epilogue, monkeypatch):
    monkeypatch.delenv("L32_SWIGLU_TILE_N", raising=False)
    monkeypatch.delenv("L32_RASTER_GROUP", raising=False)
    L = _lib.lib()
    for m in MS:
        for n in NS:
            for cta_group in (0, 1, 2):
                for max_ctas in (0, 2, 6, 37, 100, 1000):
                    want = P.plan(epilogue, m, n, sms, cta_group, max_ctas)
                    got = P.library_plan(L, epilogue, m, n, sms, cta_group, max_ctas)
                    assert got == want, (epilogue, m, n, sms, cta_group, max_ctas)


@pytest.mark.parametrize("tile_n,raster", [("16", "1"), ("80", "3"), ("112", None), ("64", "0"), ("136", "1000"), ("24", None)])
def test_plan_follows_the_overrides(tile_n, raster, monkeypatch):
    monkeypatch.setenv("L32_SWIGLU_TILE_N", tile_n)
    if raster is None:
        monkeypatch.delenv("L32_RASTER_GROUP", raising=False)
    else:
        monkeypatch.setenv("L32_RASTER_GROUP", raster)
    L = _lib.lib()
    for epilogue in (P.EPI_STORE, P.EPI_SWIGLU):
        for m in (1, 129, 1000, 8192):
            for n in (8, 1032, 14336):
                want = P.plan(epilogue, m, n, 148, **P.env_knobs())
                assert P.library_plan(L, epilogue, m, n, 148) == want, (epilogue, m, n)


def test_auto_planned_swiglu_widths_on_148_sms():
    """The shapes the GPU tests use to reach each width the wave-cost model can pick (cta_group 2, 148 SMs)."""
    L = _lib.lib()
    for (m, n), n_act in {(256, 4744): 80, (256, 5928): 96, (256, 7112): 112, (256, 8296): 128, (1024, 14336): 112,
                          (512, 14336): 80, (129, 14336): 112, (6144, 14336): 128, (256, 28672): 80, (2048, 28672): 112}.items():
        assert P.library_plan(L, P.EPI_SWIGLU, m, n, 148)["n_act"] == n_act, (m, n)
        assert P.plan(P.EPI_SWIGLU, m, n, 148)["n_act"] == n_act, (m, n)


def test_plan_rejects_bad_arguments():
    L = _lib.lib()
    import ctypes
    out = (ctypes.c_int * 7)()
    assert L.l32_debug_gemm_plan(P.EPI_STORE, 0, 256, 0, 0, 148, out) != 0
    assert L.l32_debug_gemm_plan(P.EPI_STORE, 256, 0, 0, 0, 148, out) != 0
    assert L.l32_debug_gemm_plan(P.EPI_STORE, 256, 256, 3, 0, 148, out) != 0
    assert L.l32_debug_gemm_plan(3, 256, 256, 2, 0, 148, out) != 0      # the tensor-parallel feed-forward is not covered
    assert L.l32_debug_gemm_plan(P.EPI_STORE, 256, 256, 0, 0, 148, None) != 0
