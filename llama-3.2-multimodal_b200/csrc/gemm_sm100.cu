// K3/K4/K6: persistent warp-specialised tcgen05 GEMM for sm_100a with fused SwiGLU epilogues.
//
//   D[M,N] = sum_p A_p[M,K_p] * B_p[N,K_p]^T        (bf16 / fp16 operands, fp32 accumulation in TMEM)
//
// Replaces the reference's scalar CUDA-core kernels swiglu_forward_kernel / swiglu_down_forward_kernel /
// swiglu_backward_kernel (reference Tools/swiglu/swiglu.cu:58-100, :228-272, :179-223) and the cuBLAS
// F.linear calls of the live PyTorch path (reference Tools/swiglu/FusedSwiglu.py:18-20, Model/model.py:214-217).
//
// Structure (one CTA per SM, 448 threads; optional CTA pair = cta_group::2 with UMMA M = 256):
//   warp 0   : TMA producer  (cp.async.bulk.tensor, 128-byte swizzle, ring of kStages smem slots)
//   warp 1   : MMA issuer    (tcgen05.mma kind::f16, one elected thread of the leader CTA)
//   warp 2   : TMEM allocator
//   warps 4-11: epilogue     (tcgen05.ld -> registers -> fused math -> global stores).  Two groups of four warps
//                            (one warp per TMEM lane quarter each); the SwiGLU epilogues, which read / write several
//                            [M, I] tensors per tile, split the columns of a tile between the groups, EPI_STORE uses one
//   warps 2-3, 12-13: all-gather pullers of the tensor-parallel variant (idle otherwise): NVLink loads from peer memory
// TMEM holds two 256-column fp32 accumulator stages, so the epilogue of tile t overlaps the main loop of
// tile t+1.  Tiles are visited in a grouped raster so concurrently running CTAs share A and B panels in L2.
//
// Epilogues:
//   EPI_STORE      : D tile is 128*cta_group x 256.
//   EPI_SWIGLU     : the 256 accumulator columns are [gate(128) | up(128)] of the same 128 act columns;
//                    act = silu(g) * u is formed in registers, so gate and up never round-trip HBM
//                    (they are written only when the caller asks for the backward caches).
//   EPI_SWIGLU_BWD : D = d_act; reads the gate/up caches, recomputes sigmoid/SiLU in registers and emits
//                    d_gate, d_up (and optionally the recomputed act for the w_down weight gradient).
// Operands may be K-major ([rows][K]) or MN-major ([K][rows]); the latter serves the backward GEMMs
// (dgrad through W^T, wgrad through X^T) without any explicit transpose.
#include "l32_internal.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <type_traits>

namespace l32 {
namespace {

constexpr int kBlockM = 128;   // accumulator rows per CTA (= TMEM lanes)
constexpr int kBlockK = 64;    // one 128-byte swizzle atom of 16-bit elements
constexpr int kUmmaK = 16;
constexpr int kAccCols = 256;  // TMEM columns per accumulator stage (= UMMA N)
constexpr int kThreads = 448;             // warps 0-1 TMA / MMA, 2-3 + 12-13 all-gather pullers (2 allocates TMEM), 4-11 epilogue
constexpr int kPullWarps = 4;
constexpr int kAtomBytes = kBlockK * 128;   // 64 rows x 128 B = 8 KiB: one swizzle-atom column of a tile
constexpr int kEpiRowPitch = 272;           // 256 B of one output row + 16 B so the lanes' st.shared hit distinct banks
constexpr int kEpiStageBytes = 32 * kEpiRowPitch;   // per epilogue warp: one row buffer per lane (EPI_STORE)

template <int kCtaGroup>
struct TileCfg {
    static constexpr int kBRows = kAccCols / kCtaGroup;   // B rows (N) staged by one CTA
    static constexpr int kABytes = kBlockM * kBlockK * 2;
    static constexpr int kBBytes = kBRows * kBlockK * 2;
    static constexpr int kStageBytes = kABytes + kBBytes;
    static constexpr int kStages = (kCtaGroup == 2) ? 6 : 4;
    static constexpr int kNumBarriers = 2 * kStages + 4;
    static constexpr int kSmemBytes = kStages * kStageBytes + 4 * kEpiStageBytes + kNumBarriers * 8 + 16;
};

constexpr int kMaxGroup = 3;
struct GemmKernelParams {
    CUtensorMap map_a[kMaxGroup];   // per accumulation phase -- or, for a grouped launch (nprob > 1), per problem
    CUtensorMap map_b[kMaxGroup];
    int m, n;
    int k[kMaxGroup];
    int num_phases;
    int a_mn_major, b_mn_major;
    int tiles_m, tiles_n, raster_group;
    uint32_t idesc;
    void* d[3];
    const void* e[2];
    const void* bias[2];
    long long ldd;
    int n_act;              // EPI_SWIGLU: act columns per tile (UMMA N = 2 * n_act), multiple of 16, <= 128
    int m_rotate;           // m-tiles are visited starting at this tile index (wrapping around)
    int m_il_world;         // > 0: interleaved visiting order of the fused reduce-scatter -- consecutive m-tiles belong to
    int m_il_tpc;           //      different owner ranks (tiles per owner chunk = m_il_tpc), own rank last in each round
    TpAllGather ag;         // all-gather of A fused into the kernel (world == 0: off)
    TpReduceScatter rs;     // reduce-scatter fused into the EPI_STORE epilogue (world == 0: off)
    // EPI_FFN_TP: the down projection that shares the tile loop (A = act = d[0], K = n, B = w_down shard)
    CUtensorMap map_a_dn, map_b_dn;
    int k_dn, n_dn, tiles_n_dn;
    int ffn_prefix;         // gate/up-only tiles at the head of every mixed round
    uint32_t idesc_dn;
    uint32_t* act_done;
    // Grouped launch (EPI_STORE, one phase): nprob independent problems with the same K and operand majors share ONE
    // persistent tile loop -- e.g. the three weight-gradient GEMMs of a training step: 3 x 896 tiles = 36.3 waves instead of
    // 3 x (12.1 run as 13).  Problem i: D_i = d[i] [gm x gn, pitch gldd], tiles [gstart[i], gstart[i + 1]).
    int nprob;
    int gm[kMaxGroup], gn[kMaxGroup], gtm[kMaxGroup], gtn[kMaxGroup], gstart[kMaxGroup + 1];
    long long gldd[kMaxGroup];
    const long long* ce_labels;   // EPI_CE: target column of every row (int64; anything outside [0, n) never matches)
    float2* ce_partials;          // EPI_CE: [m][tiles_n] (max, sum of exp(v - max)) of the tile's columns of that row
    float* ce_target;             // EPI_CE: [m] logit of the target column (written by the tile that holds it)
    int debug_flags;          // experiments only (L32_BWD_DEBUG): 1 = skip the output stores, 2 = skip the cache loads
    CUtensorMap map_out[3];   // EPI_SWIGLU_BWD: d_gate / d_up / act as [m, n] tensors, box {16 cols, 32 rows}, 32-byte swizzle
    unsigned long long spin_timeout_ns;   // bound of every cross-SM / cross-GPU flag wait
};

// One operand tile of `rows` x 64 (K) elements into shared memory.
//   K-major : a single box {64 (K), rows}; smem = [rows][128 B], swizzled.
//   MN-major: rows/64 boxes {64 (MN), 64 (K)}; smem = rows/64 atoms of [64 (K)][128 B].
template <int kCtaGroup>
L32_DEVICE void load_tile(const CUtensorMap* map, uint8_t* dst, uint64_t* full_bar, int mn_major, int row0, int rows,
                          int k0) {
    if (!mn_major) {
        if constexpr (kCtaGroup == 2) tma_load_2d_pair(dst, map, full_bar, k0, row0, kEvictNormal);
        else tma_load_2d(dst, map, full_bar, k0, row0, kEvictNormal);
    } else {
        for (int i = 0; i < rows / 64; ++i) {
            if constexpr (kCtaGroup == 2) tma_load_2d_pair(dst + i * kAtomBytes, map, full_bar, row0 + i * 64, k0, kEvictNormal);
            else tma_load_2d(dst + i * kAtomBytes, map, full_bar, row0 + i * 64, k0, kEvictNormal);
        }
    }
}

L32_DEVICE void st_global_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// 32-byte streaming read (one full sector per lane in ONE request; read once: first to leave L2).  32-byte aligned address.
L32_DEVICE void ld_global_stream_v8(const void* p, uint4& lo, uint4& hi) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w), "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w) : "l"(p));
}
L32_DEVICE uint4 ld_global_nc_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

L32_DEVICE void st_shared_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(smem_u32(p)), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// Bulk async store of one contiguous row segment (shared -> global), tracked by the issuing thread's bulk group.
L32_DEVICE void bulk_store_row(void* gdst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}
L32_DEVICE void bulk_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
L32_DEVICE void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

struct TileCoord {
    int m_blk, n_blk;
    int prob;   // EPI_FFN_TP: 0 = gate/up tile, 1 = down tile
};
struct TileOrder {
    int tiles_m, tiles_n, group, m_rotate, il_world, il_tpc, il_rank;
};
__host__ L32_DEVICE TileCoord tile_coord(int t, const TileOrder& o) {
    const int per_group = o.group * o.tiles_n;
    const int g = t / per_group;
    const int first_m = g * o.group;
    const int gsize = o.group < o.tiles_m - first_m ? o.group : o.tiles_m - first_m;
    const int r = t - g * per_group;
    TileCoord c;
    const int logical = first_m + r % gsize;
    if (o.il_world > 0) {
        // round-robin over the owner ranks: NVLink stays busy for the whole kernel and every receiver is fed evenly
        const int j = logical / o.il_world, k = logical - j * o.il_world;
        int owner = o.il_rank + 1 + k;
        if (owner >= o.il_world) owner -= o.il_world;
        c.m_blk = owner * o.il_tpc + j;
    } else {
        c.m_blk = logical + o.m_rotate;
        if (c.m_blk >= o.tiles_m) c.m_blk -= o.tiles_m;
    }
    c.n_blk = r / gsize;
    c.prob = 0;
    return c;
}

// EPI_FFN_TP tile sequence.  Rows are processed in groups of `group` m-tiles; round r holds the gate/up tiles of group r
// and the down tiles of group r - 1 (whose act is complete or about to be), interleaved evenly after a gate/up-only
// prefix so that (1) the NVLink pushes of the down epilogues are spread over the whole kernel instead of only its last
// third and (2) nobody waits long for the act of the previous group.  Every tile depends only on tiles with a smaller
// index, and every cluster walks its tiles in increasing order, so the waits cannot deadlock.
struct FfnOrder {
    int tiles_m, n_gu, n_dn, group, m_rotate, prefix;
};
__host__ L32_DEVICE TileCoord ffn_tile_coord(int t, const FfnOrder& o) {
    const int A = o.group * o.n_gu, B = o.group * o.n_dn;
    const int rounds = o.tiles_m / o.group;
    int r, idx, prob;
    if (t < A) {
        r = 0; idx = t; prob = 0;
    } else {
        const int tt = t - A;
        r = 1 + tt / (A + B);
        const int i = tt - (r - 1) * (A + B);
        if (r == rounds) {
            idx = i; prob = 1;
        } else if (i < o.prefix) {
            idx = i; prob = 0;
        } else {
            const int i2 = i - o.prefix, A2 = A - o.prefix, T2 = A2 + B;
            const int c0 = static_cast<int>(static_cast<long long>(i2) * A2 / T2);
            const int c1 = static_cast<int>(static_cast<long long>(i2 + 1) * A2 / T2);
            if (c1 > c0) { idx = o.prefix + c0; prob = 0; }
            else { idx = i2 - c0; prob = 1; }
        }
    }
    // within a group the tiles are m-major (all n-tiles of one row block, then the next row block): a row block's act is
    // complete long before its down tiles come up (>= 1.5 waves of distance, also in the down-only last round)
    const int g = prob ? r - 1 : r;
    const int nt = prob ? o.n_dn : o.n_gu;
    TileCoord c;
    c.prob = prob;
    c.m_blk = g * o.group + idx / nt + o.m_rotate;
    if (c.m_blk >= o.tiles_m) c.m_blk -= o.tiles_m;
    c.n_blk = idx % nt;
    return c;
}

// All-gather fused into the kernel: this warp's share of pulling chunk after chunk of A rows out of peer memory
// (NVLink loads that bypass the non-coherent L1) into the local A buffer, in the order the tiles consume them.
L32_DEVICE void ag_pull(const TpAllGather& ag, int m, size_t row_bytes, int puller, int num_pullers, uint32_t lane,
                        uint64_t timeout_ns) {
    constexpr int kUnroll = 8;   // measured (scripts/nvlink_probe.py): 4 warps/SM x 8 loads in flight saturate NVLink pulls; 16 is slower
    // copy_own: the A buffer is NOT the buffer the peers pull from, so the own rows are copied too (a local copy, first)
    for (int j = ag.copy_own ? 0 : 1; j < ag.world; ++j) {
        const int s = (ag.rank + j) % ag.world;
        const long long r0 = static_cast<long long>(s) * ag.rows_per_rank;
        long long rows = static_cast<long long>(m) - r0;
        if (rows > ag.rows_per_rank) rows = ag.rows_per_rank;
        if (rows > 0) {
            if (lane == 0 && j != 0) wait_flag_ge<true>(&ag.ready[s], ag.epoch, timeout_ns);   // rank s has written its own rows
            __syncwarp();
            const long long nvec = rows * static_cast<long long>(row_bytes / 16);
            const long long v0 = nvec * puller / num_pullers, v1 = nvec * (puller + 1) / num_pullers;
            const uint8_t* src = static_cast<const uint8_t*>(ag.peer_src[s]) + static_cast<size_t>(r0) * row_bytes;
            uint8_t* dst = static_cast<uint8_t*>(ag.local_dst) + static_cast<size_t>(r0) * row_bytes;
            for (long long v = v0 + lane; v < v1; v += 32 * kUnroll) {
                uint4 buf[kUnroll];
#pragma unroll
                for (int u = 0; u < kUnroll; ++u)
                    if (v + u * 32 < v1) buf[u] = ld_relaxed_sys_v4(src + static_cast<size_t>(v + u * 32) * 16);
#pragma unroll
                for (int u = 0; u < kUnroll; ++u)
                    if (v + u * 32 < v1)
                        st_global_v4(dst + static_cast<size_t>(v + u * 32) * 16, buf[u].x, buf[u].y, buf[u].z, buf[u].w);
            }
            __threadfence();
        }
        __syncwarp();
        if (lane == 0) red_release_gpu_add_u32(&ag.done[s], 1u);
    }
}


// Store 32 consecutive columns of one row (16 packed registers), 8 columns per 16-byte store.
L32_DEVICE void store_row32(void* base, const uint32_t (&v)[16], int n_valid) {
    uint8_t* p = static_cast<uint8_t*>(base);
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (j * 8 < n_valid) st_global_v4(p + j * 16, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}
L32_DEVICE void load_row32(const void* base, uint32_t (&v)[16], int n_valid) {
    const uint8_t* p = static_cast<const uint8_t*>(base);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint4 t = make_uint4(0, 0, 0, 0);
        if (j * 8 < n_valid) t = ld_global_nc_v4(p + j * 16);
        v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
    }
}

template <int kCtaGroup, int kEpi, typename T>
__global__ void __launch_bounds__(kThreads, 1) gemm_kernel(const __grid_constant__ GemmKernelParams p) {
    using Cfg = TileCfg<kCtaGroup>;
    constexpr int kStages = Cfg::kStages;
    constexpr bool kTp = (kEpi == EPI_FFN_TP);
    const int kTileNOut = (kEpi == EPI_SWIGLU || kTp) ? p.n_act : 256;   // output columns per (gate/up) tile
    constexpr int kEpiWarps = (kEpi == EPI_STORE || kEpi == EPI_CE) ? 4 : 8;        // epilogue warps per CTA that take part
    // bytes the pair's TMA loads deliver per ring stage (EPI_SWIGLU stages n_act gate + n_act up weight rows)
    const uint32_t stage_tx_full = static_cast<uint32_t>(Cfg::kStageBytes * kCtaGroup);
    const uint32_t stage_tx = (kEpi == EPI_SWIGLU || kTp) ? static_cast<uint32_t>(kCtaGroup * Cfg::kABytes + 2 * p.n_act * 128)
                                                          : stage_tx_full;

    // 128-byte-swizzled tiles need 1024-byte alignment; the kernel has no static shared memory, so the dynamic window
    // starts aligned (checked: a misaligned base traps instead of corrupting tiles).
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    if ((smem_u32(smem_raw) & 1023u) != 0) __trap();
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + kStages * Cfg::kABytes;
    uint8_t* epi_stage = smem + kStages * Cfg::kStageBytes;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(epi_stage + 4 * kEpiStageBytes);
    uint64_t* empty_bar = full_bar + kStages;
    uint64_t* tfull_bar = empty_bar + kStages;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const uint32_t warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const uint32_t lane = lane_id();
    const uint32_t rank = (kCtaGroup == 2) ? cluster_ctarank() : 0u;
    const int cluster_id = blockIdx.x / kCtaGroup;
    const int num_clusters = gridDim.x / kCtaGroup;
    const bool grouped = (kEpi == EPI_STORE) && p.nprob > 1;
    const int num_tiles = grouped ? p.gstart[p.nprob] : p.tiles_m * (p.tiles_n + (kTp ? p.tiles_n_dn : 0));
    const TileOrder order = {p.tiles_m, p.tiles_n, p.raster_group, p.m_rotate, p.m_il_world, p.m_il_tpc, p.rs.rank};
    const FfnOrder forder = {p.tiles_m, p.tiles_n, p.tiles_n_dn, p.raster_group, p.m_rotate, p.ffn_prefix};
    auto get_tile = [&](int t) -> TileCoord {
        if constexpr (kTp) {
            return ffn_tile_coord(t, forder);
        } else {
            if (grouped) {
                int pr = 0;
                while (pr + 1 < p.nprob && t >= p.gstart[pr + 1]) ++pr;
                // m_rotate is nonzero only with the all-gather, where every problem has the same rows
                const TileOrder go = {p.gtm[pr], p.gtn[pr], p.raster_group, p.m_rotate, 0, 0, 0};
                TileCoord c = tile_coord(t - p.gstart[pr], go);
                c.prob = pr;                                   // here: index of the problem of the group
                return c;
            }
            return tile_coord(t, order);
        }
    };

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.map_a[0]);
        tma_prefetch_desc(&p.map_b[0]);
        if (p.num_phases > 1 || p.nprob > 1) tma_prefetch_desc(&p.map_a[1]);
        if (p.nprob > 2 || p.num_phases > 2) {
            tma_prefetch_desc(&p.map_a[2]);
            tma_prefetch_desc(&p.map_b[2]);
        }
        if (p.num_phases > 1 || p.nprob > 1 || kEpi == EPI_SWIGLU || kTp) tma_prefetch_desc(&p.map_b[1]);
        if constexpr (kEpi == EPI_SWIGLU_BWD) {
            tma_prefetch_desc(&p.map_out[0]);
            tma_prefetch_desc(&p.map_out[1]);
            if (p.d[2] != nullptr) tma_prefetch_desc(&p.map_out[2]);
        }
        if constexpr (kTp) {
            tma_prefetch_desc(&p.map_a_dn);
            tma_prefetch_desc(&p.map_b_dn);
        }
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < kStages; ++i) {
            mbar_init(&full_bar[i], kCtaGroup);    // one producer arrival per CTA of the pair (+ tx bytes)
            mbar_init(&empty_bar[i], 1);           // one tcgen05.commit
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull_bar[i], 1);               // one tcgen05.commit
            mbar_init(&tempty_bar[i], kEpiWarps * kCtaGroup);  // one arrival per (active) epilogue warp of every CTA
        }
        fence_mbar_init();
    }
    if constexpr (kCtaGroup == 2) cluster_sync_all();   // both CTAs resident before the paired TMEM allocation
    if (warp == 2) {
        tmem_alloc<kCtaGroup>(tmem_slot, 512);
        tmem_relinquish<kCtaGroup>();
    }
    tc_fence_before();
    if constexpr (kCtaGroup == 2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
    // Programmatic dependent launch: everything above (barriers, TMEM, descriptor prefetch) overlapped the tail of the
    // previous kernel of the stream; from here on its results are needed.  The next kernel may be scheduled as soon as
    // SM resources free up (it orders itself behind this grid with griddepcontrol.wait).
    pdl_launch_dependents();
    pdl_wait_prior_grid();

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        // (elect.sync, not lane == 0: ptxas then knows the branch is single-lane and emits the TMA / tcgen05 instructions
        //  back to back; behind a lane test it wraps each of them in an ELECT ... BRA.U.ANY loop, ~100 clocks apiece)
        if (elect_one()) {
            uint32_t stage = 0, phase = 0;
            for (int t = cluster_id; t < num_tiles; t += num_clusters) {
                const TileCoord tc = get_tile(t);
                const bool dn = kTp && tc.prob == 1;                       // down tile of the fused feed-forward
                const bool swiglu_tile = (kEpi == EPI_SWIGLU) || (kTp && !dn);
                const int m0 = tc.m_blk * (kBlockM * kCtaGroup) + static_cast<int>(rank) * kBlockM;
                const int n0 = tc.n_blk * (dn ? kAccCols : kTileNOut);
                if (dn) {
                    // its A operand is the act of this m-tile: every epilogue warp of every gate/up tile of the row
                    // block must have stored (generic proxy, other SMs) before the TMA (async proxy) may read it
                    wait_flag_ge<false>(&p.act_done[tc.m_blk], static_cast<uint32_t>(p.tiles_n * kEpiWarps * kCtaGroup), p.spin_timeout_ns);
                    fence_proxy_async_all();
                }
                if (!dn && p.ag.world > 1 && m0 < p.m) {
                    // the A rows of this tile may belong to other ranks: wait until every puller warp has landed them
                    const int c_lo = m0 / p.ag.rows_per_rank;
                    const int c_hi = (min(m0 + kBlockM, p.m) - 1) / p.ag.rows_per_rank;
                    bool waited = false;
                    for (int c = c_lo; c <= c_hi; ++c) {
                        if (c == p.ag.rank && !p.ag.copy_own) continue;
                        wait_flag_ge<false>(&p.ag.done[c], p.ag.done_base + gridDim.x * static_cast<uint32_t>(kPullWarps), p.spin_timeout_ns);
                        waited = true;
                    }
                    if (waited) fence_proxy_async_all();   // generic-proxy stores of other SMs -> TMA (async proxy) loads
                }
                for (int ph = 0; ph < p.num_phases; ++ph) {
                    const int num_kb = ((dn ? p.k_dn : p.k[ph]) + kBlockK - 1) / kBlockK;
                    const CUtensorMap* map_a = dn ? &p.map_a_dn : &p.map_a[grouped ? tc.prob : ph];
                    const CUtensorMap* map_b = dn ? &p.map_b_dn : &p.map_b[grouped ? tc.prob : ph];
                    for (int kb = 0; kb < num_kb; ++kb) {
                        mbar_wait(&empty_bar[stage], phase ^ 1u);
                        uint8_t* sa = smem_a + stage * Cfg::kABytes;
                        uint8_t* sb = smem_b + stage * Cfg::kBBytes;
                        if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], swiglu_tile ? stage_tx : stage_tx_full);
                        load_tile<kCtaGroup>(map_a, sa, &full_bar[stage], p.a_mn_major, m0, kBlockM, kb * kBlockK);
                        if (swiglu_tile) {
                            if constexpr (kCtaGroup == 2) {
                                // leader stages the gate rows, its peer the up rows of the same 128 act columns
                                load_tile<2>(&p.map_b[rank], sb, &full_bar[stage], 0, n0, 128, kb * kBlockK);
                            } else {
                                load_tile<1>(&p.map_b[0], sb, &full_bar[stage], 0, n0, 128, kb * kBlockK);
                                load_tile<1>(&p.map_b[1], sb + p.n_act * 128, &full_bar[stage], 0, n0, 128, kb * kBlockK);
                            }
                        } else {
                            load_tile<kCtaGroup>(map_b, sb, &full_bar[stage], p.b_mn_major,
                                                 n0 + static_cast<int>(rank) * Cfg::kBRows, Cfg::kBRows, kb * kBlockK);
                        }
                        if (rank != 0) mbar_arrive_remote(&full_bar[stage], 0);
                        if (++stage == kStages) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (leader CTA only)
        if (rank == 0 && elect_one()) {
            const uint32_t a_kstep = p.a_mn_major ? (kUmmaK * 128) : (kUmmaK * 2);   // bytes per UMMA K step
            const uint32_t b_kstep = p.b_mn_major ? (kUmmaK * 128) : (kUmmaK * 2);
            const uint32_t a_lbo = p.a_mn_major ? kAtomBytes : 0;
            const uint32_t b_lbo = p.b_mn_major ? kAtomBytes : 0;
            uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
            for (int t = cluster_id; t < num_tiles; t += num_clusters) {
                bool dn = false;
                if constexpr (kTp) dn = get_tile(t).prob == 1;
                const uint32_t idesc = dn ? p.idesc_dn : p.idesc;
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * kAccCols;
                uint32_t accumulate = 0;
                for (int ph = 0; ph < p.num_phases; ++ph) {
                    const int num_kb = ((dn ? p.k_dn : p.k[ph]) + kBlockK - 1) / kBlockK;
                    for (int kb = 0; kb < num_kb; ++kb) {
                        mbar_wait(&full_bar[stage], phase);
                        tc_fence_after();
                        const uint32_t a_addr = smem_u32(smem_a + stage * Cfg::kABytes);
                        const uint32_t b_addr = smem_u32(smem_b + stage * Cfg::kBBytes);
#pragma unroll
                        for (int k = 0; k < kBlockK / kUmmaK; ++k) {
                            const uint64_t adesc = make_smem_desc_sw128(a_addr + k * a_kstep, a_lbo, 1024);
                            const uint64_t bdesc = make_smem_desc_sw128(b_addr + k * b_kstep, b_lbo, 1024);
                            umma_f16<kCtaGroup>(d_tmem, adesc, bdesc, idesc, accumulate);
                            accumulate = 1;
                        }
                        umma_commit<kCtaGroup>(&empty_bar[stage]);   // smem slot reusable once these MMAs retire
                        if (++stage == kStages) { stage = 0; phase ^= 1u; }
                    }
                }
                umma_commit<kCtaGroup>(&tfull_bar[acc]);             // accumulator complete -> epilogue
                acc ^= 1u;
                if (acc == 0) acc_phase ^= 1u;
            }
        }
    } else if (warp == 2 || warp == 3 || warp >= 12) {
        // ------------------------------------------------------------------ all-gather pullers (tensor-parallel only)
        if (p.ag.world > 1) {
            const int idx = static_cast<int>(warp >= 12 ? warp - 10 : warp - 2);   // 0..3
            ag_pull(p.ag, p.m, static_cast<size_t>(p.k[0]) * sizeof(T), static_cast<int>(blockIdx.x) * kPullWarps + idx,
                    static_cast<int>(gridDim.x) * kPullWarps, lane, p.spin_timeout_ns);
        }
    } else if (warp >= 4 && warp < 4 + kEpiWarps) {
        // ------------------------------------------------------------------ epilogue
        const uint32_t q = (warp - 4) & 3u;                // TMEM lane quarter owned by this warp (warp id % 4)
        const uint32_t eg = (warp - 4) >> 2;               // epilogue group: which share of the tile's columns
        uint32_t acc = 0, acc_phase = 0;
        const size_t esz = sizeof(T);
        for (int t = cluster_id; t < num_tiles; t += num_clusters) {
            const TileCoord tc = get_tile(t);
            const bool dn = kTp && tc.prob == 1;
            const bool store_tile = (kEpi == EPI_STORE) || (kEpi == EPI_CE) || dn;
            const bool swiglu_tile = (kEpi == EPI_SWIGLU) || (kTp && !dn);
            const int tile_n = dn ? p.n_dn : (grouped ? p.gn[tc.prob] : p.n);   // valid output columns of this problem
            const size_t tile_ldd = static_cast<size_t>(dn ? p.n_dn : (grouped ? p.gldd[tc.prob] : p.ldd));  // and its row pitch
            const int row = tc.m_blk * (kBlockM * kCtaGroup) + static_cast<int>(rank) * kBlockM + q * 32 + lane;
            const int n0 = tc.n_blk * (dn ? kAccCols : kTileNOut);
            const bool row_ok = row < (grouped ? p.gm[tc.prob] : p.m);
            const size_t row_off = static_cast<size_t>(row_ok ? row : 0) * tile_ldd;
            // EPI_SWIGLU_BWD: the gate / up cache rows of step c + 2 (this warp's next step) are requested before step c is
            // computed, the first ones before the accumulator is even complete (they do not depend on it)
            // 32-byte loads need 32-byte aligned rows: row pitch a multiple of 16 elements and 32-byte aligned bases
            const bool wide_ok = (kEpi == EPI_SWIGLU_BWD) && (p.ldd % 16) == 0 &&
                                 ((reinterpret_cast<uintptr_t>(p.e[0]) | reinterpret_cast<uintptr_t>(p.e[1])) & 31u) == 0;
            auto load_gu = [&](int c, uint4 (&gq)[2], uint4 (&uq)[2]) {
                const int col = n0 + c * 16;
                const int nv = (row_ok && c < kAccCols / 16 && !(p.debug_flags & 2)) ? (p.n - col) : 0;
                const uint8_t* gsrc = static_cast<const uint8_t*>(p.e[0]) + (row_off + col) * esz;
                const uint8_t* usrc = static_cast<const uint8_t*>(p.e[1]) + (row_off + col) * esz;
                if (nv >= 16 && wide_ok && !(p.debug_flags & 8)) {
                    ld_global_stream_v8(gsrc, gq[0], gq[1]);
                    ld_global_stream_v8(usrc, uq[0], uq[1]);
                    return;
                }
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    gq[j] = make_uint4(0, 0, 0, 0);
                    uq[j] = make_uint4(0, 0, 0, 0);
                    if (j * 8 < nv) {
                        gq[j] = ld_global_nc_v4(gsrc + j * 16);
                        uq[j] = ld_global_nc_v4(usrc + j * 16);
                    }
                }
            };
            uint4 gq[2], uq[2], gn[2], un[2];
            if constexpr (kEpi == EPI_SWIGLU_BWD) load_gu(static_cast<int>(eg), gq, uq);
            mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((q * 32u) << 16) + acc * kAccCols;

            if (store_tile) {
              if (eg == 0) {   // EPI_STORE runs on one group of four epilogue warps
                // Every lane parks 128 columns (256 B) of its own row in shared memory and ships them with ONE bulk
                // async store (cp.async.bulk shared -> global): whole 256-byte row segments on the wire, which is what
                // NVLink needs when the reduce-scatter is fused in (the row then goes straight to the rank that owns
                // it -- a peer store), no second pass through the LSU, and the TMEM stage is released without waiting
                // for the stores.  Row pitch 272 B keeps the 16-byte st.shared of the 32 lanes conflict-free.
                uint8_t* my_row = epi_stage + q * kEpiStageBytes + lane * kEpiRowPitch;
                const T* bias = kTp ? nullptr : static_cast<const T*>(p.bias[0]);
                uint8_t* d_row = nullptr;
                if (row_ok) {
                    if (p.rs.world > 0) {
                        int owner = row / p.rs.rows_per_rank;
                        if (owner >= p.rs.world) owner = p.rs.world - 1;
                        d_row = static_cast<uint8_t*>(p.rs.peer_dst[owner]) +
                                static_cast<size_t>(row - owner * p.rs.rows_per_rank) * tile_ldd * esz;
                    } else {
                        d_row = static_cast<uint8_t*>(p.d[grouped ? tc.prob : 0]) + row_off * esz;
                    }
                }
                const uint8_t* add_row = (!kTp && p.e[0] != nullptr) ? static_cast<const uint8_t*>(p.e[0]) + row_off * esz : nullptr;
                // EPI_CE (lm_head + cross entropy): besides storing the logits, every row keeps a running (max, sum of exp) over
                // the tile's columns -- of the values ROUNDED to the storage type, so that the softmax the backward forms from
                // the stored logits sums to one -- and the tile that holds the row's target column records that logit.
                float ce_m = -INFINITY, ce_s = 0.f, ce_t = 0.f;
                bool ce_hit = false;
                long long ce_lab = -1;
                if constexpr (kEpi == EPI_CE) {
                    if (row_ok) ce_lab = p.ce_labels[row];
                }
#pragma unroll 1
                for (int c = 0; c < kAccCols / 128; ++c) {
                    const int col = n0 + c * 128;
                    if (col >= tile_n) break;
                    bulk_store_wait_read();   // the previous store of this lane has finished reading its row buffer
#pragma unroll
                    for (int part = 0; part < 4; ++part) {
                        const int pcol = col + part * 32;
                        if (pcol >= tile_n) break;
                        uint32_t v[32];
                        tmem_ld_32x32b_x32(taddr + c * 128 + part * 32, v);
                        tmem_ld_wait();
                        uint32_t o[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            float lo = __uint_as_float(v[2 * j]), hi = __uint_as_float(v[2 * j + 1]);
                            if (bias != nullptr) {
                                if (pcol + 2 * j < tile_n) lo += static_cast<float>(bias[pcol + 2 * j]);
                                if (pcol + 2 * j + 1 < tile_n) hi += static_cast<float>(bias[pcol + 2 * j + 1]);
                            }
                            o[j] = Pack2<T>::pack(lo, hi);
                        }
                        if constexpr (kEpi == EPI_CE) {
                            float r[32];
#pragma unroll
                            for (int j = 0; j < 16; ++j) {
                                const float2 f = Pack2<T>::unpack(o[j]);
                                r[2 * j] = f.x; r[2 * j + 1] = f.y;
                            }
                            float cm = -INFINITY;
#pragma unroll
                            for (int j = 0; j < 32; ++j) if (pcol + j < tile_n) cm = fmaxf(cm, r[j]);
                            const float nm = fmaxf(ce_m, cm);
                            float acc = 0.f;
#pragma unroll
                            for (int j = 0; j < 32; ++j) if (pcol + j < tile_n) acc += __expf(r[j] - nm);
                            ce_s = ce_s * __expf(ce_m - nm) + acc;   // first chunk: ce_s = 0, exp(-inf) = 0
                            ce_m = nm;
                            const long long d = ce_lab - pcol;
                            if (d >= 0 && d < 32 && ce_lab < tile_n) {
                                ce_hit = true;
#pragma unroll
                                for (int j = 0; j < 32; ++j) if (j == static_cast<int>(d)) ce_t = r[j];
                            }
                        }
                        if (add_row != nullptr && row_ok) {   // fused "+ addend" (block tail: attn_out + ff_out, model.py:273)
                            uint32_t ad[16];
                            load_row32(add_row + static_cast<size_t>(pcol) * esz, ad, tile_n - pcol);
#pragma unroll
                            for (int j = 0; j < 16; ++j) {
                                const float2 a = Pack2<T>::unpack(o[j]), b = Pack2<T>::unpack(ad[j]);
                                o[j] = Pack2<T>::pack(a.x + b.x, a.y + b.y);
                            }
                        }
#pragma unroll
                        for (int j4 = 0; j4 < 4; ++j4)
                            st_shared_v4(my_row + part * 64 + j4 * 16, o[4 * j4], o[4 * j4 + 1], o[4 * j4 + 2], o[4 * j4 + 3]);
                    }
                    fence_proxy_async_smem();   // generic-proxy st.shared -> async-proxy bulk store
                    if (row_ok) {
                        const int ncols = min(tile_n - col, 128);
                        bulk_store_row(d_row + static_cast<size_t>(col) * esz, my_row, static_cast<uint32_t>(ncols) * static_cast<uint32_t>(esz));
                    }
                    bulk_store_commit();
                }
                if constexpr (kEpi == EPI_CE) {
                    if (row_ok) {
                        p.ce_partials[static_cast<size_t>(row) * p.tiles_n + tc.n_blk] = make_float2(ce_m, ce_s);
                        if (ce_hit) p.ce_target[row] = ce_t;
                    }
                }
              }
            } else if (swiglu_tile) {
                // accumulator columns [0, n_act) = gate, [n_act, 2 n_act) = up of the same act columns
                const T* bg = static_cast<const T*>(p.bias[0]);
                const T* bu = static_cast<const T*>(p.bias[1]);
                auto finish = [&](auto& g, auto& u, int col, auto ncols_tag) {
                    constexpr int kCols = decltype(ncols_tag)::value;
                    if (bg != nullptr || bu != nullptr) {
#pragma unroll
                        for (int j = 0; j < kCols; ++j) {
                            if (col + j < p.n) {
                                if (bg != nullptr) g[j] = __float_as_uint(__uint_as_float(g[j]) + static_cast<float>(bg[col + j]));
                                if (bu != nullptr) u[j] = __float_as_uint(__uint_as_float(u[j]) + static_cast<float>(bu[col + j]));
                            }
                        }
                    }
                    uint32_t o[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) o[j] = 0;
#pragma unroll
                    for (int j = 0; j < kCols / 2; ++j) {
                        const float g0 = __uint_as_float(g[2 * j]), g1 = __uint_as_float(g[2 * j + 1]);
                        const float u0 = __uint_as_float(u[2 * j]), u1 = __uint_as_float(u[2 * j + 1]);
                        o[j] = Pack2<T>::pack(silu_f32(g0) * u0, silu_f32(g1) * u1);
                    }
                    const int n_valid = min(p.n - col, kCols);
                    if (row_ok) store_row32(static_cast<uint8_t*>(p.d[0]) + (row_off + col) * esz, o, n_valid);
                    if (p.d[1] != nullptr) {   // backward caches
#pragma unroll
                        for (int j = 0; j < kCols / 2; ++j) o[j] = Pack2<T>::pack(__uint_as_float(g[2 * j]), __uint_as_float(g[2 * j + 1]));
                        if (row_ok) store_row32(static_cast<uint8_t*>(p.d[1]) + (row_off + col) * esz, o, n_valid);
#pragma unroll
                        for (int j = 0; j < kCols / 2; ++j) o[j] = Pack2<T>::pack(__uint_as_float(u[2 * j]), __uint_as_float(u[2 * j + 1]));
                        if (row_ok) store_row32(static_cast<uint8_t*>(p.d[2]) + (row_off + col) * esz, o, n_valid);
                    }
                };
                int c0 = 0;
#pragma unroll 1
                for (; c0 + 32 <= p.n_act; c0 += 32) {
                    const int col = n0 + c0;
                    if (col >= p.n) break;
                    if (((c0 >> 5) & 1) != static_cast<int>(eg)) continue;   // the other warp group's chunk
                    uint32_t g[32], u[32];
                    tmem_ld_32x32b_x32(taddr + c0, g);
                    tmem_ld_32x32b_x32(taddr + p.n_act + c0, u);
                    tmem_ld_wait();
                    finish(g, u, col, std::integral_constant<int, 32>{});
                }
                if (c0 < p.n_act && n0 + c0 < p.n && ((c0 >> 5) & 1) == static_cast<int>(eg)) {   // n_act = 32 k + 16: 16-column tail
                    uint32_t g[16], u[16];
                    tmem_ld_32x32b_x16(taddr + c0, g);
                    tmem_ld_32x32b_x16(taddr + p.n_act + c0, u);
                    tmem_ld_wait();
                    finish(g, u, n0 + c0, std::integral_constant<int, 16>{});
                }
            } else if constexpr (kEpi == EPI_SWIGLU_BWD) {
                // Five [M, I] tensors pass through this epilogue.  The three outputs leave through shared memory and TMA
                // tensor stores (one 32-row x 16-column box per tensor per step: full 32-byte sectors, three requests
                // instead of 96 per-lane 16-byte stores to 32 different rows); TMA clips the ragged edges.  The staging
                // rows use the 32-byte swizzle of the tensor map (16-byte chunk index ^= bit 2 of the row), which also
                // makes the lanes' st.shared conflict-free.
                uint8_t* stg = epi_stage + (warp - 4) * (3 * 1024);
                const int row0 = tc.m_blk * (kBlockM * kCtaGroup) + static_cast<int>(rank) * kBlockM + q * 32;
                const uint32_t sw = (lane >> 2) & 1u;
                uint8_t* my = stg + lane * 32;
#pragma unroll 1
                for (int c = static_cast<int>(eg); c < kAccCols / 16; c += 2) {
                    const int col = n0 + c * 16;
                    if (col >= p.n) break;
                    uint32_t v[16];
                    tmem_ld_32x32b_x16(taddr + c * 16, v);
                    load_gu(c + 2, gn, un);
                    tmem_ld_wait();
                    const uint32_t gp[8] = {gq[0].x, gq[0].y, gq[0].z, gq[0].w, gq[1].x, gq[1].y, gq[1].z, gq[1].w};
                    const uint32_t up[8] = {uq[0].x, uq[0].y, uq[0].z, uq[0].w, uq[1].x, uq[1].y, uq[1].z, uq[1].w};
                    uint32_t odg[8], odu[8], oact[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float2 g = Pack2<T>::unpack(gp[j]);
                        const float2 u = Pack2<T>::unpack(up[j]);
                        const float da0 = __uint_as_float(v[2 * j]), da1 = __uint_as_float(v[2 * j + 1]);
                        const float s0 = sigmoid_f32(g.x), s1 = sigmoid_f32(g.y);
                        const float silu0 = g.x * s0, silu1 = g.y * s1;
                        // d silu(g)/dg = s * (1 + g * (1 - s))
                        odg[j] = Pack2<T>::pack(da0 * u.x * (s0 * (1.0f + g.x * (1.0f - s0))),
                                                da1 * u.y * (s1 * (1.0f + g.y * (1.0f - s1))));
                        odu[j] = Pack2<T>::pack(da0 * silu0, da1 * silu1);
                        oact[j] = Pack2<T>::pack(silu0 * u.x, silu1 * u.y);
                    }
                    if (lane == 0) bulk_store_wait_read();   // the previous step's tensor stores have read the staging rows
                    __syncwarp();
                    st_shared_v4(my + ((0u ^ sw) << 4), odg[0], odg[1], odg[2], odg[3]);
                    st_shared_v4(my + ((1u ^ sw) << 4), odg[4], odg[5], odg[6], odg[7]);
                    st_shared_v4(my + 1024 + ((0u ^ sw) << 4), odu[0], odu[1], odu[2], odu[3]);
                    st_shared_v4(my + 1024 + ((1u ^ sw) << 4), odu[4], odu[5], odu[6], odu[7]);
                    if (p.d[2] != nullptr) {
                        st_shared_v4(my + 2048 + ((0u ^ sw) << 4), oact[0], oact[1], oact[2], oact[3]);
                        st_shared_v4(my + 2048 + ((1u ^ sw) << 4), oact[4], oact[5], oact[6], oact[7]);
                    }
                    fence_proxy_async_smem();   // generic-proxy st.shared -> async-proxy tensor store
                    __syncwarp();
                    if (lane == 0 && row0 < p.m && !(p.debug_flags & 1)) {
                        const uint64_t hint = (p.debug_flags & 4) ? kEvictNormal : kEvictFirst;
                        tma_store_2d_hint(&p.map_out[0], stg, col, row0, hint);
                        tma_store_2d_hint(&p.map_out[1], stg + 1024, col, row0, hint);
                        if (p.d[2] != nullptr) tma_store_2d_hint(&p.map_out[2], stg + 2048, col, row0, hint);
                        tma_store_commit();
                    }
#pragma unroll
                    for (int j = 0; j < 2; ++j) { gq[j] = gn[j]; uq[j] = un[j]; }
                }
            }
            // accumulator stage drained: hand it back to the MMA issuer of the leader CTA
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (rank == 0) mbar_arrive(&tempty_bar[acc]);
                else mbar_arrive_remote(&tempty_bar[acc], 0);
            }
            if constexpr (kTp) {
                // This warp's share of the act tile is stored: publish it to the producers of the down tiles.  Done AFTER
                // the TMEM stage went back to the MMA issuer -- the fence waits for the stores to be acknowledged, which
                // takes microseconds under load and must not sit between a short down tile and the next main loop.
                if (swiglu_tile) {
                    __threadfence();
                    __syncwarp();
                    if (lane == 0) red_release_gpu_add_u32(&p.act_done[tc.m_blk], 1u);
                }
            }
            acc ^= 1u;
            if (acc == 0) acc_phase ^= 1u;
        }
        if (kEpi == EPI_STORE || kEpi == EPI_CE || kEpi == EPI_SWIGLU_BWD || kTp) bulk_store_wait_read();   // shared memory must outlive the last bulk stores
    }

    __syncwarp();
    tc_fence_before();
    if constexpr (kCtaGroup == 2) cluster_sync_all(); else __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc<kCtaGroup>(tmem_base, 512);
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    });
    return fn;
}

// ctas: grid size from plan_ctas (a multiple of kCtaGroup)
template <int kCtaGroup, int kEpi, typename T>
int launch(const GemmKernelParams& kp, int ctas, cudaStream_t s) {
    using Cfg = TileCfg<kCtaGroup>;
    auto* kernel = gemm_kernel<kCtaGroup, kEpi, T>;
    static bool configured_dev[kMaxDevices] = {};   // per instantiation and device
    bool& configured = configured_dev[current_device_slot()];
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
        if (e != cudaSuccess) return static_cast<int>(e);
        configured = true;
    }
    int clusters = ctas / kCtaGroup;

    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(clusters * kCtaGroup));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = kCtaGroup;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
    if (kp.ag.world > 1 || kEpi == EPI_FFN_TP) {
        // These variants spin on counters that only fill when EVERY CTA of the persistent grid is running (all-gather
        // arrival counts, act_done): the whole grid must be co-resident.  Ask the driver how many clusters fit on the SMs
        // this context may use (MPS limits, green contexts) and shrink the grid to that; no room at all is an error.
        static int max_clusters_dev[kMaxDevices] = {};
        int& max_clusters = max_clusters_dev[current_device_slot()];
        if (max_clusters == 0) {
            int n = 0;
            cudaError_t q = cudaOccupancyMaxActiveClusters(&n, kernel, &cfg);
            if (q != cudaSuccess) return static_cast<int>(q);
            max_clusters = n > 0 ? n : -1;
        }
        if (max_clusters < 0) return L32_ERR_NOT_RESIDENT;
        if (clusters > max_clusters) {
            clusters = max_clusters;
            cfg.gridDim = dim3(static_cast<unsigned>(clusters * kCtaGroup));
        }
    }
    cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, kp);
    if (e == cudaSuccess) count_launch();
    return static_cast<int>(e);
}

template <int kCtaGroup, typename T>
int launch_epi(const GemmKernelParams& kp, int epi, int ctas, cudaStream_t s) {
    switch (epi) {
        case EPI_STORE: return launch<kCtaGroup, EPI_STORE, T>(kp, ctas, s);
        case EPI_CE: return launch<kCtaGroup, EPI_CE, T>(kp, ctas, s);
        case EPI_SWIGLU: return launch<kCtaGroup, EPI_SWIGLU, T>(kp, ctas, s);
        case EPI_SWIGLU_BWD: return launch<kCtaGroup, EPI_SWIGLU_BWD, T>(kp, ctas, s);
        case EPI_FFN_TP:
            if constexpr (kCtaGroup == 2) return launch<2, EPI_FFN_TP, T>(kp, ctas, s);
            else return L32_ERR_BAD_SHAPE;
        default: return L32_ERR_BAD_SHAPE;
    }
}

// CTAs of the persistent grid: one cluster of cta_group CTAs per SM pair (or SM), never more clusters than tiles.
int plan_ctas(int num_tiles, int cta_group, int max_ctas, int sms) {
    int ctas = sms;
    if (max_ctas > 0 && max_ctas < ctas) ctas = max_ctas;
    int clusters = ctas / cta_group;
    if (clusters > num_tiles) clusters = num_tiles;
    if (clusters < 1) clusters = 1;
    return clusters * cta_group;
}

// The host decisions of one (not grouped) launch of gemm_sm100.  EPI_FFN_TP adds its down tiles, and a grouped launch its
// problems' tiles, to num_tiles afterwards (and re-plans ctas).
struct GemmPlan {
    int cta_group, tiles_m, tiles_n, n_act, raster_group, num_tiles, ctas;
};

int plan_gemm(int epilogue, int m, int n, int cta_group_req, int raster_group_req, int max_ctas, int sms, GemmPlan& pl) {
    const bool swiglu_like = epilogue == EPI_SWIGLU || epilogue == EPI_FFN_TP;
    int cta_group = cta_group_req;
    if (cta_group == 0) cta_group = (m > kBlockM) ? 2 : 1;
    if (cta_group != 1 && cta_group != 2) return L32_ERR_BAD_SHAPE;
    pl.cta_group = cta_group;
    const int tile_m = kBlockM * cta_group;
    pl.tiles_m = (m + tile_m - 1) / tile_m;
    // EPI_SWIGLU: pick the act-column tile width (multiple of 16) that minimises waves x tile cost -- e.g. a
    // tensor-parallel shard of 1792 act columns is 7 waves of 112 columns instead of 7 waves of 128 (the last one
    // nearly empty).  Ties go to the wider tile.
    int n_act = 128;
    if (swiglu_like) {
        int ctas = sms;
        if (max_ctas > 0 && max_ctas < ctas) ctas = max_ctas;
        const long long clusters = ctas / cta_group > 0 ? ctas / cta_group : 1;
        long long best = -1;
        for (int cand = 128; cand >= 64; cand -= 16) {
            const long long tiles = static_cast<long long>(pl.tiles_m) * ((n + cand - 1) / cand);
            const long long cost = ((tiles + clusters - 1) / clusters) * (cand + 12);   // + fixed per-tile overhead
            if (best < 0 || cost < best) { best = cost; n_act = cand; }
        }
        if (const char* env = getenv("L32_SWIGLU_TILE_N")) {   // tuning knob for experiments only
            const int v = atoi(env);
            if (v >= 16 && v <= 128 && (v % 16) == 0) n_act = v;
        }
    }
    pl.n_act = n_act;
    const int tile_n_out = swiglu_like ? n_act : 256;
    pl.tiles_n = (n + tile_n_out - 1) / tile_n_out;
    // m-tiles per raster group: 2048 rows for the plain / backward epilogues, 4096 rows for the fused gate/up GEMM (its B
    // operand -- two weight matrices -- is the big one: larger groups re-read it from HBM half as often; measured
    // +1.8 % at the 11B shape, scripts/raster_ab.py)
    pl.raster_group = raster_group_req > 0 ? raster_group_req : (swiglu_like ? 32 : 16) / cta_group;
    if (const char* env = getenv("L32_RASTER_GROUP")) {   // tuning knob for experiments only
        const int v = atoi(env);
        if (v > 0) pl.raster_group = v;
    }
    pl.num_tiles = pl.tiles_m * pl.tiles_n;
    pl.ctas = plan_ctas(pl.num_tiles, cta_group, max_ctas, sms);
    return L32_OK;
}

}  // namespace

int num_sms() {
    static int cached[kMaxDevices] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    int& n = cached[(dev >= 0 && dev < kMaxDevices) ? dev : 0];
    if (n == 0) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) return 148;
        n = v;
    }
    return n;
}

int make_tensor_map_2d(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                       uint32_t box_rows, uint32_t box_cols, int dtype) {
    return make_tensor_map_2d_sw(map, ptr, rows, cols, ld_elems, box_rows, box_cols, dtype, 128);
}

// swizzle_bytes: 128 (box_cols = 64), 64 (box_cols = 32) or 32 (box_cols = 16) -- the box row is exactly one swizzle span
int make_tensor_map_2d_sw(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                          uint32_t box_rows, uint32_t box_cols, int dtype, int swizzle_bytes) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (fn == nullptr) return L32_ERR_DRIVER;
    if (!is_aligned16(ptr) || (ld_elems % 8) != 0) return L32_ERR_BAD_ALIGN;
    if (box_rows == 0 || box_rows > 256 || static_cast<int>(box_cols) * 2 != swizzle_bytes) return L32_ERR_BAD_SHAPE;
    const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                  : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                  : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
    if (sw == CU_TENSOR_MAP_SWIZZLE_NONE) return L32_ERR_BAD_SHAPE;
    const cuuint64_t gdim[2] = {cols, rows};
    const cuuint64_t gstride[1] = {ld_elems * 2};
    const cuuint32_t box[2] = {box_cols, box_rows};
    const cuuint32_t estride[2] = {1, 1};
    const CUtensorMapDataType dt = (dtype == L32_BF16) ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    CUresult r = fn(map, dt, 2, const_cast<void*>(ptr), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r == CUDA_ERROR_INVALID_CONTEXT || r == CUDA_ERROR_NOT_INITIALIZED) {
        // A thread that has not touched the runtime yet (e.g. autograd's backward thread calling this library first) has no
        // current driver context although the process has a primary one: bind it through the runtime and retry once.
        if (cudaFree(nullptr) == cudaSuccess)
            r = fn(map, dt, 2, const_cast<void*>(ptr), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    if (r != CUDA_SUCCESS && getenv("L32_DEBUG") != nullptr)
        fprintf(stderr, "[l32] cuTensorMapEncodeTiled failed (%d): ptr %p rows %llu cols %llu ld %llu box %u x %u swizzle %d\n",
                static_cast<int>(r), ptr, static_cast<unsigned long long>(rows), static_cast<unsigned long long>(cols),
                static_cast<unsigned long long>(ld_elems), box_rows, box_cols, swizzle_bytes);
    return r == CUDA_SUCCESS ? L32_OK : L32_ERR_DRIVER;
}

int make_tensor_map_3d(CUtensorMap* map, const void* ptr, uint64_t planes, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                       uint64_t plane_elems, uint32_t box_rows, int dtype) {
    return make_tensor_map_3d_box(map, ptr, planes, rows, cols, ld_elems, plane_elems, box_rows, 1, dtype);
}

int make_tensor_map_3d_box(CUtensorMap* map, const void* ptr, uint64_t planes, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                           uint64_t plane_elems, uint32_t box_rows, uint32_t box_planes, int dtype) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (fn == nullptr) return L32_ERR_DRIVER;
    if (!is_aligned16(ptr) || (ld_elems % 8) != 0 || (plane_elems % 8) != 0) return L32_ERR_BAD_ALIGN;
    if (box_rows == 0 || box_rows > 256 || box_planes == 0 || box_planes > 256 || planes == 0 || rows == 0) return L32_ERR_BAD_SHAPE;
    const cuuint64_t gdim[3] = {cols, rows, planes};
    const cuuint64_t gstride[2] = {ld_elems * 2, plane_elems * 2};
    const cuuint32_t box[3] = {64, box_rows, box_planes};
    const cuuint32_t estride[3] = {1, 1, 1};
    const CUtensorMapDataType dt = (dtype == L32_BF16) ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    auto encode = [&] {
        return fn(map, dt, 3, const_cast<void*>(ptr), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    };
    CUresult r = encode();
    if ((r == CUDA_ERROR_INVALID_CONTEXT || r == CUDA_ERROR_NOT_INITIALIZED) && cudaFree(nullptr) == cudaSuccess)
        r = encode();   // no current driver context on this thread yet: see make_tensor_map_2d_sw
    if (r != CUDA_SUCCESS && getenv("L32_DEBUG") != nullptr)
        fprintf(stderr, "[l32] cuTensorMapEncodeTiled (3-D) failed (%d): ptr %p planes %llu rows %llu cols %llu\n", static_cast<int>(r),
                ptr, static_cast<unsigned long long>(planes), static_cast<unsigned long long>(rows),
                static_cast<unsigned long long>(cols));
    return r == CUDA_SUCCESS ? L32_OK : L32_ERR_DRIVER;
}

// Host-side view of the persistent kernels' tile sequences (tests/test_tile_order.py checks on the CPU that every tile is
// visited exactly once and that every down tile of EPI_FFN_TP comes well after the act tiles it consumes).
void debug_tile_order(int t, int tiles_m, int tiles_n, int group, int m_rotate, int il_world, int il_tpc, int il_rank, int* out3) {
    const TileOrder o = {tiles_m, tiles_n, group, m_rotate, il_world, il_tpc, il_rank};
    const TileCoord c = tile_coord(t, o);
    out3[0] = c.prob; out3[1] = c.m_blk; out3[2] = c.n_blk;
}
void debug_ffn_tile_order(int t, int tiles_m, int n_gu, int n_dn, int group, int m_rotate, int prefix, int* out3) {
    const FfnOrder o = {tiles_m, n_gu, n_dn, group, m_rotate, prefix};
    const TileCoord c = ffn_tile_coord(t, o);
    out3[0] = c.prob; out3[1] = c.m_blk; out3[2] = c.n_blk;
}
// The launch plan gemm_sm100 would use (tests/test_gemm_plan.py restates it; the GPU tests pick their shapes with it).
int debug_gemm_plan(int epilogue, int m, int n, int cta_group, int max_ctas, int sms, int* out7) {
    if (m <= 0 || n <= 0 || sms < 0) return L32_ERR_BAD_SHAPE;
    GemmPlan pl;
    const int rc = plan_gemm(epilogue, m, n, cta_group, 0, max_ctas, sms > 0 ? sms : num_sms(), pl);
    if (rc != L32_OK) return rc;
    const int v[7] = {pl.cta_group, pl.tiles_m, pl.tiles_n, pl.n_act, pl.raster_group, pl.num_tiles, pl.ctas};
    for (int i = 0; i < 7; ++i) out7[i] = v[i];
    return L32_OK;
}

int gemm_sm100(const GemmProblem& g, cudaStream_t s) {
    const bool ffn_tp = g.epilogue == EPI_FFN_TP;
    const bool swiglu_like = g.epilogue == EPI_SWIGLU || ffn_tp;
    if (g.dtype != L32_BF16 && g.dtype != L32_FP16) return L32_ERR_BAD_DTYPE;
    if (g.m < 0 || g.n <= 0 || g.num_phases < 1 || g.num_phases > kMaxGroup) return L32_ERR_BAD_SHAPE;
    if (g.m == 0) return L32_OK;
    if ((g.n % 8) != 0 || (g.ldd % 8) != 0) return L32_ERR_BAD_ALIGN;
    if (swiglu_like && (g.num_phases != 1 || g.b[0].mn_major || g.b[1].mn_major)) return L32_ERR_BAD_SHAPE;
    for (int i = 0; i < 3; ++i)
        if (g.d[i] != nullptr && !is_aligned16(g.d[i])) return L32_ERR_BAD_ALIGN;
    if (g.d[0] == nullptr && g.rs.world == 0) return L32_ERR_NULL;
    if (g.epilogue == EPI_SWIGLU && (g.d[1] == nullptr) != (g.d[2] == nullptr)) return L32_ERR_NULL;
    if (g.epilogue == EPI_SWIGLU_BWD) {
        if (g.d[1] == nullptr || g.e[0] == nullptr || g.e[1] == nullptr) return L32_ERR_NULL;
        if (!is_aligned16(g.e[0]) || !is_aligned16(g.e[1])) return L32_ERR_BAD_ALIGN;
    }

    const int sms = num_sms();
    GemmPlan plan;
    if (const int rc = plan_gemm(g.epilogue, g.m, g.n, g.cta_group, g.raster_group, g.max_ctas, sms, plan); rc != L32_OK) return rc;
    const int cta_group = plan.cta_group;
    if (ffn_tp) {
        if (cta_group != 2 || g.dn.w == nullptr || g.dn.n <= 0 || (g.dn.n % 8) != 0 || g.dn.act_done == nullptr ||
            g.rs.world < 1 || g.d[0] == nullptr || g.d[1] != nullptr || g.a[0].mn_major || g.bias[0] != nullptr ||
            g.bias[1] != nullptr)
            return L32_ERR_BAD_SHAPE;
    }

    GemmKernelParams kp;
    memset(&kp, 0, sizeof(kp));
    kp.m = g.m;
    kp.n = g.n;
    kp.num_phases = g.num_phases;
    kp.a_mn_major = g.a[0].mn_major;
    kp.b_mn_major = g.b[0].mn_major;
    const int tile_m = kBlockM * cta_group;
    kp.tiles_m = plan.tiles_m;
    const int n_act = plan.n_act;
    kp.n_act = n_act;
    kp.tiles_n = plan.tiles_n;
    kp.raster_group = plan.raster_group;
    kp.idesc = make_idesc_f16(g.dtype == L32_BF16, static_cast<uint32_t>(tile_m),
                              swiglu_like ? static_cast<uint32_t>(2 * n_act) : static_cast<uint32_t>(kAccCols),
                              g.a[0].mn_major != 0, g.b[0].mn_major != 0);
    for (int i = 0; i < 3; ++i) kp.d[i] = g.d[i];
    kp.e[0] = g.e[0]; kp.e[1] = g.e[1];
    kp.bias[0] = g.bias[0]; kp.bias[1] = g.bias[1];
    kp.ldd = g.ldd;
    kp.m_rotate = (g.m_rotate_rows > 0) ? (g.m_rotate_rows / tile_m) % kp.tiles_m : 0;
    if (g.rs.world > 1 && g.rs.rows_per_rank > 0 && (g.rs.rows_per_rank % tile_m) == 0 &&
        kp.tiles_m == g.rs.world * (g.rs.rows_per_rank / tile_m)) {
        kp.m_il_world = g.rs.world;
        kp.m_il_tpc = g.rs.rows_per_rank / tile_m;
        if (const char* env = getenv("L32_RS_INTERLEAVE")) {   // tuning knob for experiments only
            if (atoi(env) == 0) kp.m_il_world = 0;
        }
    }
    kp.ag = g.ag;
    kp.spin_timeout_ns = spin_timeout_ns();
    if (const char* env = getenv("L32_BWD_DEBUG")) kp.debug_flags = atoi(env);
    kp.rs = g.rs;
    if (g.ag.world > kMaxTpWorld || g.rs.world > kMaxTpWorld) return L32_ERR_BAD_SHAPE;
    if (g.ag.world > 1) {
        // the pulled chunk is treated as a flat byte range: A must be K-major with a dense row pitch
        if (g.a[0].mn_major || g.num_phases != 1 || g.a[0].ld != g.k[0] || g.ag.rows_per_rank <= 0 ||
            g.ag.local_dst != g.a[0].ptr || g.ag.ready == nullptr || g.ag.done == nullptr)
            return L32_ERR_BAD_SHAPE;
    }
    if (g.rs.world > 0 && ((g.epilogue != EPI_STORE && !ffn_tp) || g.rs.rows_per_rank <= 0 || g.e[0] != nullptr)) return L32_ERR_BAD_SHAPE;
    if (g.epilogue == EPI_STORE && g.e[0] != nullptr && !is_aligned16(g.e[0])) return L32_ERR_BAD_ALIGN;

    const int b_box_rows = swiglu_like ? 128 : kAccCols / cta_group;
    for (int ph = 0; ph < g.num_phases; ++ph) {
        if (g.k[ph] <= 0) return L32_ERR_BAD_SHAPE;   // any K: TMA zero-fills the ragged last k-block
        if (g.a[ph].mn_major != g.a[0].mn_major || g.b[ph].mn_major != g.b[0].mn_major) return L32_ERR_BAD_SHAPE;
        kp.k[ph] = g.k[ph];
        int rc;
        if (!g.a[ph].mn_major) rc = make_tensor_map_2d(&kp.map_a[ph], g.a[ph].ptr, g.m, g.k[ph], g.a[ph].ld, kBlockM, kBlockK, g.dtype);
        else rc = make_tensor_map_2d(&kp.map_a[ph], g.a[ph].ptr, g.k[ph], g.m, g.a[ph].ld, kBlockK, 64, g.dtype);
        if (rc != L32_OK) return rc;
        if (!swiglu_like) {
            if (!g.b[ph].mn_major) rc = make_tensor_map_2d(&kp.map_b[ph], g.b[ph].ptr, g.n, g.k[ph], g.b[ph].ld, b_box_rows, kBlockK, g.dtype);
            else rc = make_tensor_map_2d(&kp.map_b[ph], g.b[ph].ptr, g.k[ph], g.n, g.b[ph].ld, kBlockK, 64, g.dtype);
            if (rc != L32_OK) return rc;
        }
    }
    if (swiglu_like) {
        for (int i = 0; i < 2; ++i) {
            int rc = make_tensor_map_2d(&kp.map_b[i], g.b[i].ptr, g.n, g.k[0], g.b[i].ld, n_act, kBlockK, g.dtype);
            if (rc != L32_OK) return rc;
        }
    }
    if (g.group_count > 1) {
        // a grouped launch: every problem shares K, the operand majors and the dtype; no bias / addend / reduce-scatter.
        // The all-gather is allowed when every problem reads the same gathered A (e.g. the q / k / v projections of one
        // tensor-parallel attention shard): the pullers fetch it once and every tile waits for the chunk it reads.
        if (g.group_count > kMaxGroup || g.epilogue != EPI_STORE || g.num_phases != 1 || g.e[0] != nullptr || g.bias[0] != nullptr ||
            g.rs.world > 0 || cta_group != 2 || g.k[0] <= 0)
            return L32_ERR_BAD_SHAPE;
        if (g.ag.world > 1) {
            for (int i = 0; i < g.group_count; ++i)
                if (g.group[i].a != g.a[0].ptr || g.group[i].lda != g.k[0] || g.group[i].m != g.m) return L32_ERR_BAD_SHAPE;
        }
        kp.nprob = g.group_count;
        int start = 0;
        for (int i = 0; i < g.group_count; ++i) {
            const GroupMember& q = g.group[i];
            if (q.m <= 0 || q.n <= 0 || (q.n % 8) != 0 || (q.ldd % 8) != 0 || q.d == nullptr || !is_aligned16(q.d)) return L32_ERR_BAD_SHAPE;
            kp.gm[i] = q.m; kp.gn[i] = q.n; kp.gldd[i] = q.ldd;
            kp.gtm[i] = (q.m + tile_m - 1) / tile_m;
            kp.gtn[i] = (q.n + kAccCols - 1) / kAccCols;
            kp.gstart[i] = start;
            start += kp.gtm[i] * kp.gtn[i];
            kp.d[i] = q.d;
            int rc;
            if (!g.a[0].mn_major) rc = make_tensor_map_2d(&kp.map_a[i], q.a, q.m, g.k[0], q.lda, kBlockM, kBlockK, g.dtype);
            else rc = make_tensor_map_2d(&kp.map_a[i], q.a, g.k[0], q.m, q.lda, kBlockK, 64, g.dtype);
            if (rc != L32_OK) return rc;
            if (!g.b[0].mn_major) rc = make_tensor_map_2d(&kp.map_b[i], q.b, q.n, g.k[0], q.ldb, kAccCols / cta_group, kBlockK, g.dtype);
            else rc = make_tensor_map_2d(&kp.map_b[i], q.b, g.k[0], q.n, q.ldb, kBlockK, 64, g.dtype);
            if (rc != L32_OK) return rc;
        }
        kp.gstart[g.group_count] = start;
        kp.k[0] = g.k[0];
        kp.m_il_world = 0;
        if (g.ag.world <= 1) kp.m_rotate = 0;   // all-gather: own rows first (setup_allgather's rotation), in every problem
        const int ctas = plan_ctas(start, 2, g.max_ctas, sms);
        if (g.dtype == L32_BF16) return launch_epi<2, __nv_bfloat16>(kp, EPI_STORE, ctas, s);
        return launch_epi<2, __half>(kp, EPI_STORE, ctas, s);
    }
    if (g.epilogue == EPI_CE) {
        if (g.ce.labels == nullptr || g.ce.partials == nullptr || g.ce.target == nullptr) return L32_ERR_NULL;
        if (g.e[0] != nullptr || g.bias[0] != nullptr || g.rs.world > 0 || g.ag.world > 0) return L32_ERR_BAD_SHAPE;
        kp.ce_labels = g.ce.labels;
        kp.ce_partials = static_cast<float2*>(g.ce.partials);
        kp.ce_target = g.ce.target;
    }
    if (g.epilogue == EPI_SWIGLU_BWD) {
        for (int i = 0; i < 3; ++i) {
            if (g.d[i] == nullptr) continue;
            int rc = make_tensor_map_2d_sw(&kp.map_out[i], g.d[i], g.m, g.n, g.ldd, 32, 16, g.dtype, 32);
            if (rc != L32_OK) return rc;
        }
    }
    if (ffn_tp) {
        // second problem: y_partial = act (= d[0], [m, n] with pitch ldd) * w_down_shard^T, 256-column tiles, RS epilogue
        kp.k_dn = g.n;
        kp.n_dn = g.dn.n;
        kp.tiles_n_dn = (g.dn.n + kAccCols - 1) / kAccCols;
        kp.idesc_dn = make_idesc_f16(g.dtype == L32_BF16, static_cast<uint32_t>(tile_m), kAccCols, false, false);
        kp.act_done = g.dn.act_done;
        int rc = make_tensor_map_2d(&kp.map_a_dn, g.d[0], g.m, g.n, g.ldd, kBlockM, kBlockK, g.dtype);
        if (rc != L32_OK) return rc;
        rc = make_tensor_map_2d(&kp.map_b_dn, g.dn.w, g.dn.n, g.n, g.dn.ld, kAccCols / cta_group, kBlockK, g.dtype);
        if (rc != L32_OK) return rc;
        // the tile sequence works on whole groups of m-tiles: largest group size <= the requested one that divides tiles_m
        int grp = kp.raster_group < 1 ? 1 : kp.raster_group;
        if (grp > kp.tiles_m) grp = kp.tiles_m;
        while (kp.tiles_m % grp != 0) --grp;
        kp.raster_group = grp;
        int ctas = sms;
        if (g.max_ctas > 0 && g.max_ctas < ctas) ctas = g.max_ctas;
        const int a_tiles = grp * kp.tiles_n;
        kp.ffn_prefix = a_tiles < ctas / 2 ? a_tiles : ctas / 2;   // one wave of gate/up-only tiles at the head of a round
        if (const char* env = getenv("L32_FFN_PREFIX")) {   // tuning knob for experiments only
            const int v = atoi(env);
            if (v >= 0 && v <= a_tiles) kp.ffn_prefix = v;
        }
        kp.m_il_world = 0;
        plan.num_tiles = kp.tiles_m * (kp.tiles_n + kp.tiles_n_dn);
        plan.ctas = plan_ctas(plan.num_tiles, cta_group, g.max_ctas, sms);
    }

    if (g.dtype == L32_BF16) {
        if (cta_group == 2) return launch_epi<2, __nv_bfloat16>(kp, g.epilogue, plan.ctas, s);
        return launch_epi<1, __nv_bfloat16>(kp, g.epilogue, plan.ctas, s);
    }
    if (cta_group == 2) return launch_epi<2, __half>(kp, g.epilogue, plan.ctas, s);
    return launch_epi<1, __half>(kp, g.epilogue, plan.ctas, s);
}

}  // namespace l32
