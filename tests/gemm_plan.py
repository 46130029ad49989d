"""Python restatement of the tiled GEMM's launch plan (plan_gemm in csrc/gemm_sm100.cu), shared by the CPU test that
compares it with l32_debug_gemm_plan and the GPU tests that use it to pick a shape for each tiling regime."""
import ctypes
import os

EPI_STORE, EPI_SWIGLU, EPI_SWIGLU_BWD, EPI_CE = 0, 1, 2, 4
BLOCK_M = 128
FIELDS = ("cta_group", "tiles_m", "tiles_n", "n_act", "raster_group", "num_tiles", "ctas")


def cdiv(a, b):
    return -(-a // b)


def plan(epilogue, m, n, sms, cta_group=0, max_ctas=0, tile_n=None, raster=None):
    """dict of FIELDS.  tile_n / raster stand for L32_SWIGLU_TILE_N / L32_RASTER_GROUP (None: unset)."""
    swiglu = epilogue == EPI_SWIGLU
    cg = cta_group or (2 if m > BLOCK_M else 1)
    tiles_m = cdiv(m, BLOCK_M * cg)
    ctas = min(sms, max_ctas) if max_ctas > 0 else sms
    n_act = 128
    if swiglu:
        clusters = max(ctas // cg, 1)
        best = None
        for cand in range(128, 63, -16):      # ties go to the wider tile
            cost = cdiv(tiles_m * cdiv(n, cand), clusters) * (cand + 12)
            if best is None or cost < best:
                best, n_act = cost, cand
        if tile_n is not None and 16 <= tile_n <= 128 and tile_n % 16 == 0:
            n_act = tile_n
    tiles_n = cdiv(n, n_act if swiglu else 256)
    group = (32 if swiglu else 16) // cg
    if raster is not None and raster > 0:
        group = raster
    num_tiles = tiles_m * tiles_n
    clusters = max(min(ctas // cg, num_tiles), 1)
    return dict(cta_group=cg, tiles_m=tiles_m, tiles_n=tiles_n, n_act=n_act, raster_group=group, num_tiles=num_tiles,
                ctas=clusters * cg)


def library_plan(lib, epilogue, m, n, sms, cta_group=0, max_ctas=0):
    """The same plan read from the library (l32_debug_gemm_plan); sms = 0: the current device."""
    out = (ctypes.c_int * 7)()
    rc = lib.l32_debug_gemm_plan(epilogue, m, n, cta_group, max_ctas, sms, out)
    assert rc == 0, f"l32_debug_gemm_plan({epilogue}, {m}, {n}, {cta_group}, {max_ctas}, {sms}) returned {rc}"
    return dict(zip(FIELDS, out))


def env_knobs():
    """The overrides the library reads on every call, as plan() takes them."""
    def num(name):
        v = os.environ.get(name)
        try:
            return int(v) if v else None
        except ValueError:
            return None
    return dict(tile_n=num("L32_SWIGLU_TILE_N"), raster=num("L32_RASTER_GROUP"))
