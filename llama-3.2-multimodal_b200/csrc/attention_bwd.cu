// K10: grouped-query attention backward for training calls on tcgen05 (no KV cache, past_len = 0, keys = queries).
//
// Replaces the autograd backward of GroupQueryAttention.forward's attention core (reference Model/model.py:238-253 under
// autograd): the saved [B, heads, S, S] softmax, repeat_kv's expanded K / V and the backward of the rotary embedding
// (:195-198).  Three kernels, chained with programmatic dependent launch, deterministic (no floating-point atomics):
//
//   attention_bwd_delta_kernel   delta[b, head, i] = sum_d dO . O  (fp32, from the 16-bit ctx and d_ctx)
//   attention_bwd_kernel<dKdV>   key-tile-stationary: one CTA per (batch, KV head, 128 keys).  Keys are the TMEM lanes:
//                                S^T = K Q^T and dP^T = V dO^T into TMEM, P^T = exp2(S^T c - lse), dS^T = P^T (dP^T - delta)
//                                back into TMEM as 16-bit A operands, dV += P^T dO and dK += dS^T Q (Q / dO MN-major).  The
//                                walk covers every query head of the KV group, so dK / dV sum the group in TMEM: this is the
//                                GQA reduction, with no atomics and no repeat_kv.
//   attention_bwd_kernel<dQ>     query-tile-stationary (the forward's structure): S = Q K^T, dP = dO V^T, dS = P (dP - delta)
//                                into TMEM, dQ += dS K (K MN-major).  P is exact from the saved lse: no online maximum.
//
// Both epilogues own one TMEM lane = one whole row of head_dim columns, which holds both halves of every rotation pair: dq and
// dk are rotated back (the transpose of RoPE) in registers with the angles of rope_kv_append_kernel (rope_cos_sin) and scaled
// by 1 / sqrt(head_dim), then stored once in 16 bit as the gradients of the projection outputs: dq [b, t, heads * d],
// dk / dv [b, t, kv_heads * d].
//
// Mask semantics are the forward's: causal (key <= query), key_keep, keys [0, q_len).  A query row that sees no key has
// lse = +inf: its probabilities are exactly 0, so it gets dq = 0 and contributes nothing; a padded key gets dk = dv = 0.
#include "l32_internal.cuh"

#include <cstring>

namespace l32 {
namespace {

constexpr int kBwdThreads = 160;   // warps 0-3: one TMEM lane (row) per thread; warp 4: TMA producer + MMA issuer
constexpr int kRows = 128;         // rows of the stationary tile (TMEM lanes): keys (dK/dV) or queries (dQ)
constexpr int kCols = 64;          // rows of each streamed tile = columns of S / dP: queries (dK/dV) or keys (dQ)
constexpr int kStages = 3;         // streamed tile ring
constexpr int kUmmaK = 16;

struct AttnBwdParams {
    CUtensorMap map_q, map_do;   // [batch * q_len, heads * head_dim], box {64, 64}
    CUtensorMap map_k, map_v;    // [batch * kv_heads * max_len, head_dim], box {64, 64}
    const float* lse;            // [batch, heads, q_len] log2 domain, +inf = row without keys
    const float* delta;          // [batch, heads, q_len]
    const uint8_t* keep;         // optional [batch, q_len]: 0 = padded key
    const long long* pos;        // [batch, q_len]
    void* dq;                    // [batch * q_len, heads * head_dim]
    void* dk;                    // [batch * q_len, kv_heads * head_dim]
    void* dv;
    int batch, q_len, heads, kv_heads, max_len, causal;
    float scale_log2;            // log2(e) / sqrt(head_dim)
    float scale;                 // 1 / sqrt(head_dim)
    float log2_base;             // log2(rope_base)
    uint32_t idesc_s, idesc_o;
};

L32_DEVICE float exp2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// One 16-bit row segment of 32 columns -> global (4 x 16-byte stores).
template <typename T>
L32_DEVICE void store_row32(T* dst, const float (&v)[32]) {
#pragma unroll
    for (int j4 = 0; j4 < 4; ++j4) {
        uint4 w;
        w.x = Pack2<T>::pack(v[8 * j4], v[8 * j4 + 1]);
        w.y = Pack2<T>::pack(v[8 * j4 + 2], v[8 * j4 + 3]);
        w.z = Pack2<T>::pack(v[8 * j4 + 4], v[8 * j4 + 5]);
        w.w = Pack2<T>::pack(v[8 * j4 + 6], v[8 * j4 + 7]);
        *reinterpret_cast<uint4*>(dst + 8 * j4) = w;
    }
}

// Epilogue of one row held in TMEM at `acc` (kD fp32 columns of this thread's lane): dst[i] = scale * acc[i], rotated back by
// the RoPE angle of `pos` when `rope` (dx[i] = dy[i] cos + dy[i + d/2] sin, dx[i + d/2] = dy[i + d/2] cos - dy[i] sin).
// `zero`: store zeros (dead row / padded key).  The TMEM loads are warp-collective: every lane executes them.
template <int kD, typename T>
L32_DEVICE void store_grad_row(uint32_t acc, T* dst, bool store, bool zero, bool rope, float pos, float scale, float log2_base) {
    constexpr int kHalf = kD / 2;
#pragma unroll 1
    for (int c = 0; c < kHalf / 32; ++c) {
        uint32_t lo[32], hi[32];
        tmem_ld_32x32b_x32(acc + c * 32, lo);
        tmem_ld_32x32b_x32(acc + kHalf + c * 32, hi);
        tmem_ld_wait();
        float a[32], bb[32];
#pragma unroll
        for (int e = 0; e < 32; ++e) {
            float y0 = zero ? 0.f : __uint_as_float(lo[e]) * scale;
            float y1 = zero ? 0.f : __uint_as_float(hi[e]) * scale;
            if (rope) {
                float cs, sn;
                rope_cos_sin(pos, c * 32 + e, kD, log2_base, cs, sn);
                a[e] = y0 * cs + y1 * sn;
                bb[e] = y1 * cs - y0 * sn;
            } else {
                a[e] = y0;
                bb[e] = y1;
            }
        }
        if (store) {
            store_row32<T>(dst + c * 32, a);
            store_row32<T>(dst + kHalf + c * 32, bb);
        }
    }
}

// kKV = true: dK / dV kernel (stationary = K, V of 128 keys; streamed = Q, dO tiles of 64 queries of every head of the group).
// kKV = false: dQ kernel (stationary = Q, dO of 128 queries; streamed = K, V tiles of 64 keys).
// TMEM (512 columns): buffer s in {0, 1}: X = S or S^T at [128 s, 128 s + 64), Y = dP or dP^T at [128 s + 64, 128 s + 128);
// accumulators from column 256: dQ, or dV then dK.
template <bool kKV, int kD, typename T>
__global__ void __launch_bounds__(kBwdThreads, 1) attention_bwd_kernel(const __grid_constant__ AttnBwdParams p) {
    constexpr int kDAtoms = kD / 64;
    constexpr int kABytes = kRows * kD * 2;     // one stationary operand
    constexpr int kBBytes = kCols * kD * 2;     // one streamed operand
    extern __shared__ __align__(1024) uint8_t bwd_smem[];
    if ((smem_u32(bwd_smem) & 1023u) != 0) __trap();
    uint8_t* sa0 = bwd_smem;                    // Q (dQ) or K (dK/dV)
    uint8_t* sa1 = sa0 + kABytes;               // dO (dQ) or V (dK/dV)
    uint8_t* sb = sa1 + kABytes;                // [stage][2][kBBytes]: (K, V) (dQ) or (Q, dO) (dK/dV)
    float* col_stats = reinterpret_cast<float*>(sb + kStages * 2 * kBBytes);   // dK/dV: [2][lse 64 | delta 64]
    uint64_t* bar_a = reinterpret_cast<uint64_t*>(col_stats + 2 * 2 * kCols);
    uint64_t* bar_b = bar_a + 1;                // [kStages] streamed tiles landed
    uint64_t* bar_s = bar_b + kStages;          // [2] X and Y of a tile complete
    uint64_t* bar_p = bar_s + 2;                // [2] 16-bit operands of a tile are in TMEM (128 arrivals)
    uint64_t* bar_o = bar_p + 2;                // accumulating MMAs of a tile complete (stage and TMEM buffer free)
    uint64_t* bar_done = bar_o + 1;             // every MMA complete
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_done + 1);

    const int tid = threadIdx.x;
    const uint32_t warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int group = p.heads / p.kv_heads;
    const int nq = (p.q_len + kCols - 1) / kCols;          // dK/dV: query tiles per head
    int b, head, kvh, r0, ntiles, qt0 = 0;
    if constexpr (kKV) {
        // grid (kv_heads, batch, key tiles), key tile 0 first: under a causal mask it sees the most queries
        kvh = blockIdx.x;
        b = blockIdx.y;
        r0 = blockIdx.z * kRows;
        head = kvh * group;
        qt0 = p.causal ? r0 / kCols : 0;                   // first query tile that sees any of keys [r0, r0 + 128)
        ntiles = group * (nq - qt0);
    } else {
        // grid (heads, batch, query tiles), the last query tile first (the forward's order)
        head = blockIdx.x;
        b = blockIdx.y;
        r0 = static_cast<int>(gridDim.z - 1 - blockIdx.z) * kRows;
        kvh = head / group;
        const int q_last = min(r0 + kRows, p.q_len) - 1;
        const int hi = p.causal ? q_last + 1 : p.q_len;
        ntiles = (hi + kCols - 1) / kCols;
    }
    const int kv_row0 = (b * p.kv_heads + kvh) * p.max_len;

    if (tid == 0) {
        tma_prefetch_desc(&p.map_q);
        tma_prefetch_desc(&p.map_do);
        tma_prefetch_desc(&p.map_k);
        tma_prefetch_desc(&p.map_v);
        mbar_init(bar_a, 1);
        for (int i = 0; i < kStages; ++i) mbar_init(&bar_b[i], 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bar_s[i], 1);
            mbar_init(&bar_p[i], kRows);
        }
        mbar_init(bar_o, 1);
        mbar_init(bar_done, 1);
        fence_mbar_init();
    }
    constexpr uint32_t kTmemCols = 512u;
    if (warp == 4) {
        tmem_alloc<1>(tmem_slot, kTmemCols);
        tmem_relinquish<1>();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
    const uint32_t tmem_acc = tmem_base + 256;
    pdl_launch_dependents();
    pdl_wait_prior_grid();

    // streamed tile t: dK/dV -> (query head, first query row); dQ -> first key row
    auto tile_head = [&](int t) { return kKV ? head + t / (nq - qt0) : head; };
    auto tile_col0 = [&](int t) { return kKV ? (qt0 + t % (nq - qt0)) * kCols : t * kCols; };

    if (warp == 4) {
        // ------------------------------------------------------------------ TMA producer + MMA issuer (one elected thread)
        if (ntiles > 0 && elect_one()) {
            auto load_b = [&](int t) {
                const int st = t % kStages;
                uint8_t* dst = sb + st * 2 * kBBytes;
                mbar_arrive_expect_tx(&bar_b[st], 2 * kBBytes);
#pragma unroll
                for (int a = 0; a < kDAtoms; ++a) {
                    if constexpr (kKV) {
                        const int col = tile_head(t) * kD + a * 64, row = b * p.q_len + tile_col0(t);
                        tma_load_2d(dst + a * (kCols * 128), &p.map_q, &bar_b[st], col, row, kEvictNormal);
                        tma_load_2d(dst + kBBytes + a * (kCols * 128), &p.map_do, &bar_b[st], col, row, kEvictNormal);
                    } else {
                        const int row = kv_row0 + tile_col0(t);
                        tma_load_2d(dst + a * (kCols * 128), &p.map_k, &bar_b[st], a * 64, row, kEvictNormal);
                        tma_load_2d(dst + kBBytes + a * (kCols * 128), &p.map_v, &bar_b[st], a * 64, row, kEvictNormal);
                    }
                }
            };
            mbar_arrive_expect_tx(bar_a, 2 * kABytes);
#pragma unroll
            for (int a = 0; a < kDAtoms; ++a) {
#pragma unroll
                for (int h = 0; h < kRows / 64; ++h) {      // 128 rows as two 64-row boxes (same swizzled layout)
                    uint8_t* d0 = sa0 + a * (kRows * 128) + h * (64 * 128);
                    uint8_t* d1 = sa1 + a * (kRows * 128) + h * (64 * 128);
                    if constexpr (kKV) {
                        tma_load_2d(d0, &p.map_k, bar_a, a * 64, kv_row0 + r0 + h * 64, kEvictNormal);
                        tma_load_2d(d1, &p.map_v, bar_a, a * 64, kv_row0 + r0 + h * 64, kEvictNormal);
                    } else {
                        const int col = head * kD + a * 64, row = b * p.q_len + r0 + h * 64;
                        tma_load_2d(d0, &p.map_q, bar_a, col, row, kEvictNormal);
                        tma_load_2d(d1, &p.map_do, bar_a, col, row, kEvictNormal);
                    }
                }
            }
            for (int t = 0; t < kStages && t < ntiles; ++t) load_b(t);
            const uint32_t a0_addr = smem_u32(sa0), a1_addr = smem_u32(sa1);
            // X = A0 B0^T and Y = A1 B1^T of tile t into TMEM buffer t & 1
            auto issue_xy = [&](int t) {
                const int st = t % kStages;
                mbar_wait(&bar_b[st], (t / kStages) & 1u);
                tc_fence_after();
                const uint32_t b0 = smem_u32(sb + st * 2 * kBBytes), b1 = b0 + kBBytes;
                const uint32_t x = tmem_base + (t & 1) * 128, y = x + 64;
#pragma unroll
                for (int kk = 0; kk < kD / kUmmaK; ++kk) {
                    const uint32_t aoff = (kk / 4) * (kRows * 128) + (kk % 4) * 32;
                    const uint32_t boff = (kk / 4) * (kCols * 128) + (kk % 4) * 32;
                    umma_f16<1>(x, make_smem_desc_sw128(a0_addr + aoff, 0, 1024), make_smem_desc_sw128(b0 + boff, 0, 1024), p.idesc_s,
                                kk > 0 ? 1u : 0u);
                    umma_f16<1>(y, make_smem_desc_sw128(a1_addr + aoff, 0, 1024), make_smem_desc_sw128(b1 + boff, 0, 1024), p.idesc_s,
                                kk > 0 ? 1u : 0u);
                }
                umma_commit<1>(&bar_s[t & 1]);
            };
            mbar_wait(bar_a, 0);
            issue_xy(0);
            if (ntiles > 1) issue_xy(1);
            for (int t = 0; t < ntiles; ++t) {
                const int s = t & 1, st = t % kStages;
                mbar_wait(&bar_p[s], (t >> 1) & 1u);
                tc_fence_after();
                const uint32_t b0 = smem_u32(sb + st * 2 * kBBytes), b1 = b0 + kBBytes;
                const uint32_t x = tmem_base + s * 128, y = x + 64;
                // accumulate over the 64 columns of the tile (the K of these MMAs); streamed operands consumed MN-major
#pragma unroll
                for (int kk = 0; kk < kCols / kUmmaK; ++kk) {
                    const uint32_t acc = (t > 0 || kk > 0) ? 1u : 0u;
                    const uint32_t boff = kk * (kUmmaK * 128);
                    if constexpr (kKV) {
                        umma_f16_ts(tmem_acc, x + kk * (kUmmaK / 2), make_smem_desc_sw128(b1 + boff, kCols * 128, 1024), p.idesc_o,
                                    acc);                                               // dV += P^T dO
                        umma_f16_ts(tmem_acc + kD, y + kk * (kUmmaK / 2), make_smem_desc_sw128(b0 + boff, kCols * 128, 1024),
                                    p.idesc_o, acc);                                    // dK += dS^T Q
                    } else {
                        umma_f16_ts(tmem_acc, x + kk * (kUmmaK / 2), make_smem_desc_sw128(b0 + boff, kCols * 128, 1024), p.idesc_o,
                                    acc);                                               // dQ += dS K
                    }
                }
                umma_commit<1>(bar_o);
                // the tensor pipe runs in issue order: X / Y of tile t + 2 overwrite buffer s only after the MMAs above read it
                if (t + 2 < ntiles) issue_xy(t + 2);
                if (t + kStages < ntiles) {                  // stage st is free once the MMAs of tile t are complete
                    mbar_wait(bar_o, t & 1u);
                    load_b(t + kStages);
                }
            }
            umma_commit<1>(bar_done);
        }
    } else {
        // ------------------------------------------------------------------ one row (TMEM lane) per thread
        const uint32_t lane_off = (warp * 32u) << 16;
        const int row = r0 + tid;                          // key (dK/dV) or query (dQ) index
        const bool row_ok = row < p.q_len;
        float row_lse = INFINITY, row_delta = 0.f;         // dQ: this query row's statistics
        bool key_ok = row_ok;                              // dK/dV: this key is visible at all
        if constexpr (kKV) {
            if (row_ok && p.keep != nullptr) key_ok = p.keep[static_cast<size_t>(b) * p.q_len + row] != 0;
        } else {
            if (row_ok) {
                const size_t i = (static_cast<size_t>(b) * p.heads + head) * p.q_len + row;
                row_lse = p.lse[i];
                row_delta = p.delta[i];
            }
        }
        const uint8_t* keep_row = p.keep != nullptr ? p.keep + static_cast<size_t>(b) * p.q_len : nullptr;
        for (int t = 0; t < ntiles; ++t) {
            const int s = t & 1;
            const int c0 = tile_col0(t);
            float* stats = col_stats + s * 2 * kCols;
            uint32_t vis_lo = 0xffffffffu, vis_hi = 0xffffffffu;   // columns of the tile that pass the mask tests
            if constexpr (kKV) {
                // per-column lse / delta of the tile's 64 queries, staged through shared memory (buffer s: the write of
                // tile t + 2 follows the barrier of tile t + 1, which every reader of tile t has passed)
                const int h = tile_head(t);
                const int q = c0 + (tid & (kCols - 1));
                const size_t i = (static_cast<size_t>(b) * p.heads + h) * p.q_len + q;
                if (tid < kCols) stats[tid] = q < p.q_len ? p.lse[i] : INFINITY;
                else stats[tid] = q < p.q_len ? p.delta[i] : 0.f;
                named_bar_sync(1, kRows);
                if (!key_ok) {
                    vis_lo = vis_hi = 0u;
                } else if (p.causal) {                     // query c0 + j sees this key iff c0 + j >= row
                    const int lim = row - c0;              // columns j < lim are masked
                    vis_lo = lim <= 0 ? 0xffffffffu : (lim >= 32 ? 0u : ~((1u << lim) - 1u));
                    vis_hi = lim <= 32 ? 0xffffffffu : (lim >= 64 ? 0u : ~((1u << (lim - 32)) - 1u));
                }
            } else {
                // keys of the tile: length / causal limit, then the key-padding bytes as two ballot words per warp
                uint32_t keep_lo = 0xffffffffu, keep_hi = 0xffffffffu;
                if (keep_row != nullptr) {
                    const int ka = c0 + static_cast<int>(lane_id()), kb = ka + 32;
                    keep_lo = __ballot_sync(0xffffffffu, ka < p.q_len && keep_row[ka] != 0);
                    keep_hi = __ballot_sync(0xffffffffu, kb < p.q_len && keep_row[kb] != 0);
                }
                const int lim = min(p.q_len, p.causal ? row + 1 : p.q_len) - c0;   // keys [0, lim) of the tile
                vis_lo = (lim >= 32 ? 0xffffffffu : (lim > 0 ? (1u << lim) - 1u : 0u)) & keep_lo;
                vis_hi = (lim >= 64 ? 0xffffffffu : (lim > 32 ? (1u << (lim - 32)) - 1u : 0u)) & keep_hi;
            }
            mbar_wait(&bar_s[s], (t >> 1) & 1u);
            tc_fence_after();
            const uint32_t x = tmem_base + s * 128 + lane_off, y = x + 64;
            uint32_t sx[64], sy[64];
            {
                uint32_t (&x0)[32] = *reinterpret_cast<uint32_t (*)[32]>(&sx[0]);
                uint32_t (&x1)[32] = *reinterpret_cast<uint32_t (*)[32]>(&sx[32]);
                uint32_t (&y0)[32] = *reinterpret_cast<uint32_t (*)[32]>(&sy[0]);
                uint32_t (&y1)[32] = *reinterpret_cast<uint32_t (*)[32]>(&sy[32]);
                tmem_ld_32x32b_x32(x, x0);
                tmem_ld_32x32b_x32(x + 32, x1);
                tmem_ld_32x32b_x32(y, y0);
                tmem_ld_32x32b_x32(y + 32, y1);
                tmem_ld_wait();
            }
            uint32_t pk[32], dk[32];
#pragma unroll
            for (int j2 = 0; j2 < 32; ++j2) {
                float pv[2], dv[2];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int j = 2 * j2 + u;
                    const float lse = kKV ? stats[j] : row_lse;
                    const float dl = kKV ? stats[kCols + j] : row_delta;
                    const bool vis = (j < 32 ? (vis_lo >> j) : (vis_hi >> (j - 32))) & 1u;
                    const float pr = vis ? exp2_approx(fmaf(__uint_as_float(sx[j]), p.scale_log2, -lse)) : 0.f;
                    pv[u] = pr;
                    dv[u] = vis ? pr * (__uint_as_float(sy[j]) - dl) : 0.f;
                }
                pk[j2] = Pack2<T>::pack(pv[0], pv[1]);
                dk[j2] = Pack2<T>::pack(dv[0], dv[1]);
            }
            // dQ: dS over the first 32 columns of X.  dK/dV: P^T over X, dS^T over Y.
            {
                uint32_t (&d0)[16] = *reinterpret_cast<uint32_t (*)[16]>(&dk[0]);
                uint32_t (&d1)[16] = *reinterpret_cast<uint32_t (*)[16]>(&dk[16]);
                if constexpr (kKV) {
                    uint32_t (&p0)[16] = *reinterpret_cast<uint32_t (*)[16]>(&pk[0]);
                    uint32_t (&p1)[16] = *reinterpret_cast<uint32_t (*)[16]>(&pk[16]);
                    tmem_st_32x32b_x16(x, p0);
                    tmem_st_32x32b_x16(x + 16, p1);
                    tmem_st_32x32b_x16(y, d0);
                    tmem_st_32x32b_x16(y + 16, d1);
                } else {
                    tmem_st_32x32b_x16(x, d0);
                    tmem_st_32x32b_x16(x + 16, d1);
                }
            }
            tmem_st_wait();
            tc_fence_before();
            mbar_arrive(&bar_p[s]);
        }
        if (ntiles > 0) {
            mbar_wait(bar_done, 0);
            tc_fence_after();
        }
        const float pos = row_ok ? static_cast<float>(p.pos[static_cast<size_t>(b) * p.q_len + row]) : 0.f;
        const size_t tok = static_cast<size_t>(b) * p.q_len + (row_ok ? row : 0);
        if constexpr (kKV) {
            T* dv_row = static_cast<T*>(p.dv) + tok * (static_cast<size_t>(p.kv_heads) * kD) + kvh * kD;
            T* dk_row = static_cast<T*>(p.dk) + tok * (static_cast<size_t>(p.kv_heads) * kD) + kvh * kD;
            store_grad_row<kD, T>(tmem_acc + lane_off, dv_row, row_ok, !key_ok || ntiles == 0, false, pos, 1.f, p.log2_base);
            store_grad_row<kD, T>(tmem_acc + kD + lane_off, dk_row, row_ok, !key_ok || ntiles == 0, true, pos, p.scale, p.log2_base);
        } else {
            T* dq_row = static_cast<T*>(p.dq) + tok * (static_cast<size_t>(p.heads) * kD) + head * kD;
            store_grad_row<kD, T>(tmem_acc + lane_off, dq_row, row_ok, ntiles == 0, true, pos, p.scale, p.log2_base);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        tmem_dealloc<1>(tmem_base, kTmemCols);
    }
}

// delta[b, head, i] = sum_d dO[b, i, head, d] * O[b, i, head, d] in fp32.  One warp per (token, head) row.
template <typename T>
__global__ void __launch_bounds__(256) attention_bwd_delta_kernel(const T* __restrict__ d_ctx, const T* __restrict__ ctx,
                                                                   float* __restrict__ delta, int batch, int q_len, int heads, int d) {
    pdl_launch_dependents();
    pdl_wait_prior_grid();
    const long long w = blockIdx.x * 8ll + (threadIdx.x >> 5);     // row = (b * q_len + i) * heads + head
    const int lane = threadIdx.x & 31;
    if (w >= static_cast<long long>(batch) * q_len * heads) return;
    const T* go = d_ctx + w * d;
    const T* o = ctx + w * d;
    float acc = 0.f;
    for (int c = 2 * lane; c < d; c += 64) {
        const float2 a = Pack2<T>::unpack(*reinterpret_cast<const uint32_t*>(go + c));
        const float2 bb = Pack2<T>::unpack(*reinterpret_cast<const uint32_t*>(o + c));
        acc = fmaf(a.x, bb.x, fmaf(a.y, bb.y, acc));
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) {
        const int head = static_cast<int>(w % heads);
        const long long tok = w / heads;
        const int i = static_cast<int>(tok % q_len), b = static_cast<int>(tok / q_len);
        delta[(static_cast<size_t>(b) * heads + head) * q_len + i] = acc;
    }
}

template <bool kKV, int kD, typename T>
int launch_bwd(const AttnBwdParams& p, cudaStream_t s) {
    auto* kernel = attention_bwd_kernel<kKV, kD, T>;
    // the 512-column TMEM allocation needs the SM to itself: at least 116 KB of shared memory keeps a second CTA away
    size_t smem = 2 * kRows * kD * 2 + kStages * 2 * kCols * kD * 2 + 2 * 2 * kCols * 4 + 128;
    if (smem < 116 * 1024) smem = 116 * 1024;
    static bool configured_dev[kMaxDevices] = {};
    bool& configured = configured_dev[current_device_slot()];
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) return static_cast<int>(e);
        configured = true;
    }
    cudaLaunchConfig_t cfg = {};
    if (kKV)
        cfg.gridDim = dim3(static_cast<unsigned>(p.kv_heads), static_cast<unsigned>(p.batch),
                           static_cast<unsigned>((p.q_len + kRows - 1) / kRows));
    else
        cfg.gridDim = dim3(static_cast<unsigned>(p.heads), static_cast<unsigned>(p.batch),
                           static_cast<unsigned>((p.q_len + kRows - 1) / kRows));
    cfg.blockDim = dim3(kBwdThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, p);
    if (e == cudaSuccess) count_launch();
    return static_cast<int>(e);
}

template <int kD, typename T>
int launch_bwd_pair(const AttnBwdParams& p, cudaStream_t s) {
    int rc = launch_bwd<true, kD, T>(p, s);
    if (rc != L32_OK) return rc;
    return launch_bwd<false, kD, T>(p, s);
}

}  // namespace

size_t gqa_attention_backward_workspace_bytes(int batch, int q_len, int heads) {
    if (batch <= 0 || q_len <= 0 || heads <= 0) return 0;
    return static_cast<size_t>(batch) * heads * q_len * sizeof(float);
}

int gqa_attention_backward(const void* d_ctx, const void* q, const void* cache_k, const void* cache_v, const void* ctx, const float* lse,
                           const uint8_t* keep, const long long* position_ids, void* dq, void* dk, void* dv, void* workspace, int batch,
                           int q_len, int heads, int kv_heads, int head_dim, int max_len, int causal, float rope_base, int dtype,
                           cudaStream_t s) {
    if (head_dim != 64 && head_dim != 128) return L32_ERR_BAD_SHAPE;
    if (batch <= 0 || q_len <= 0) return L32_OK;
    float* delta = static_cast<float*>(workspace);
    {
        const long long rows = static_cast<long long>(batch) * q_len * heads;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(static_cast<unsigned>((rows + 7) / 8));
        cfg.blockDim = dim3(256);
        cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        cudaError_t e;
        if (dtype == L32_BF16)
            e = cudaLaunchKernelEx(&cfg, attention_bwd_delta_kernel<__nv_bfloat16>, static_cast<const __nv_bfloat16*>(d_ctx),
                                   static_cast<const __nv_bfloat16*>(ctx), delta, batch, q_len, heads, head_dim);
        else
            e = cudaLaunchKernelEx(&cfg, attention_bwd_delta_kernel<__half>, static_cast<const __half*>(d_ctx),
                                   static_cast<const __half*>(ctx), delta, batch, q_len, heads, head_dim);
        if (e != cudaSuccess) return static_cast<int>(e);
        count_launch();
    }
    AttnBwdParams p;
    memset(&p, 0, sizeof(p));
    p.lse = lse;
    p.delta = delta;
    p.keep = keep;
    p.pos = position_ids;
    p.dq = dq; p.dk = dk; p.dv = dv;
    p.batch = batch; p.q_len = q_len; p.heads = heads; p.kv_heads = kv_heads; p.max_len = max_len; p.causal = causal;
    p.scale = 1.0f / sqrtf(static_cast<float>(head_dim));
    p.scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(head_dim));
    p.log2_base = log2f(rope_base);
    p.idesc_s = make_idesc_f16(dtype == L32_BF16, kRows, kCols, false, false);
    p.idesc_o = make_idesc_f16(dtype == L32_BF16, kRows, static_cast<uint32_t>(head_dim), false, true);
    const uint64_t tok = static_cast<uint64_t>(batch) * q_len;
    int rc = make_tensor_map_2d(&p.map_q, q, tok, static_cast<uint64_t>(heads) * head_dim, static_cast<uint64_t>(heads) * head_dim, kCols,
                                64, dtype);
    if (rc != L32_OK) return rc;
    rc = make_tensor_map_2d(&p.map_do, d_ctx, tok, static_cast<uint64_t>(heads) * head_dim, static_cast<uint64_t>(heads) * head_dim, kCols,
                            64, dtype);
    if (rc != L32_OK) return rc;
    const uint64_t kv_rows = static_cast<uint64_t>(batch) * kv_heads * max_len;
    rc = make_tensor_map_2d(&p.map_k, cache_k, kv_rows, head_dim, head_dim, kCols, 64, dtype);
    if (rc != L32_OK) return rc;
    rc = make_tensor_map_2d(&p.map_v, cache_v, kv_rows, head_dim, head_dim, kCols, 64, dtype);
    if (rc != L32_OK) return rc;
    if (dtype == L32_BF16)
        return head_dim == 128 ? launch_bwd_pair<128, __nv_bfloat16>(p, s) : launch_bwd_pair<64, __nv_bfloat16>(p, s);
    return head_dim == 128 ? launch_bwd_pair<128, __half>(p, s) : launch_bwd_pair<64, __half>(p, s);
}

}  // namespace l32
