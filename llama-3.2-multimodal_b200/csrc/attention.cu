// K7/K8: grouped-query attention with a preallocated KV cache for sm_100a (SURVEY.md 8f rank 3).
//
// Replaces GroupQueryAttention.forward between the projections (reference Model/model.py:238-253): RoPE on q / k
// (apply_rotary_pos_emb, :195-198; cos / sin from position_ids, LLAMARotaryEmbedding :176-186), the KV cache update
// (KVCache.update, :21-29 -- a torch.cat per layer per step), repeat_kv copies (:124-132), the materialised
// [B, heads, S, S] score tensor, the dense additive mask and the softmax / PV products (:246-252).
//
//   rope_kv_append_kernel   RoPE on q in place and on k while it is written into the cache; v copied next to it.  The cache
//                           is preallocated [batch, kv_heads, max_len, head_dim]: appending is a store at `past_len`, not a
//                           reallocation.  Angles are computed in fp32 from position_ids (explicit positions also fix the
//                           reference's decode bug, SURVEY.md 0.9: `_prepare_position_ids` restarts at 0 for every step).
//   gqa_attention_kernel    flash-style forward: one CTA = one (batch, query head, 128-query tile); the key / value tiles of the
//                           head's KV group stream through shared memory (TMA, double-buffered), S = Q K^T and P V run on
//                           tcgen05 with the accumulators in TMEM, the online softmax runs in registers (one query row per
//                           thread = one TMEM lane), scores never leave the SM.  Causal tiles beyond the diagonal are never
//                           visited.  head_dim 64 or 128.
// Masking = the reference's additive mask restated as predicates: causal (key position <= query position; the reference's
// triu(-inf, 1), model.py:314-317), key padding (model.py:318, as a per-key keep byte) and the cache length.
#include "l32_internal.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace l32 {
namespace {

constexpr int kQTile = 128;      // query rows per CTA = TMEM lanes = softmax threads
constexpr int kKvTile = 64;      // keys per iteration (one 128-byte swizzle atom of P)
constexpr int kAttThreads = 160;   // warps 0-3: softmax (one query row per thread); warp 4: TMA producer + MMA issuer
constexpr int kUmmaKAtt = 16;

struct AttnParams {
    CUtensorMap map_q;   // [batch * q_len, heads * head_dim], box {64, 128}
    CUtensorMap map_k;   // [batch * kv_heads][kv_len][head_dim] with planes max_len * head_dim apart, box {64, 64, 1}: the
                         // rows [kv_len, tile end) of the last tile arrive as zeros, whatever the cache holds there
    CUtensorMap map_v;   // same tensor shape as K, box {64, 64, 1}
    void* out;           // [batch * q_len, heads * head_dim]
    const uint8_t* keep; // optional [batch, kv_len]: 0 = padded key (never attended)
    int batch, q_len, heads, kv_heads, max_len, kv_len, past_len, causal;
    float scale_log2;    // log2(e) / sqrt(head_dim)
    uint32_t idesc_s, idesc_o;
    // split-KV (decode): gridDim.x = splits CTAs per (batch, head), each over `tiles_per_split` key tiles; unnormalised partial
    // outputs and (reference, sum) pairs go to the workspace, attention_combine_kernel merges them.  splits == 1: off.
    int splits, tiles_per_split;
    float* part_o;       // [batch][heads][splits][q_len][head_dim] fp32
    float2* part_ml;     // [batch][heads][splits][q_len] (m_ref in the log2 domain, l)
    float* lse;          // optional [batch, heads, q_len] (training): m_ref + log2(l) in the log2 domain, +inf for a row that
                         // sees no key (the backward then forms exact zero probabilities for it).  Never with split-KV.
    // Paged cache (kPaged instances only).  map_k / map_v are then {d, kKvTile, num_pages * page_kv_heads}: key tile t of a
    // sequence is page block_table[seq][t], plane page * page_kv_heads + kv head.  kv_len / past_len / tiles_per_split above
    // are unused: each CTA reads its sequence's lengths from device memory and divides its own tiles over the splits.
    const int* block_table;   // [sequences, pages_per_seq]
    const int* past_lens;     // [sequences]
    const int* new_lens;      // [sequences], or null: every sequence has q_len new tokens (the packed decode: one)
    int pages_per_seq, page_kv_heads;
    int packed;               // packed decode: CTA batch index = sequence * page_kv_heads + kv head, its q_len rows are the
                              // query heads of ONE query
};
static_assert(L32_KV_PAGE == kKvTile, "a KV-cache page is one key tile");

// L32_ATT_NOEXP / L32_ATT_NOPV / L32_ATT_NOLD: experiment builds only (wrong results) -- what the kernel costs without the
// exponentials, without the P V MMAs, without the S reads from TMEM.
L32_DEVICE float fast_exp2(float x) {
#ifdef L32_ATT_NOEXP
    return x * 0.001f;
#else
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));   // not volatile: a pure function the scheduler may interleave freely
    return y;
#endif
}

// Packed fp32 pairs (Blackwell FFMA2 / FADD2): half the FMA-pipe instructions of the exponent arguments and the row sums.
L32_DEVICE uint64_t pack_f32x2(uint32_t lo, uint32_t hi) {
    uint64_t d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
    return d;
}
L32_DEVICE void unpack_f32x2(uint64_t v, float& lo, float& hi) {
    uint32_t a, b;
    asm("mov.b64 {%0, %1}, %2;" : "=r"(a), "=r"(b) : "l"(v));
    lo = __uint_as_float(a);
    hi = __uint_as_float(b);
}
L32_DEVICE uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
L32_DEVICE uint64_t add_f32x2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// kLse: training forward, also stores the per-row log-sum-exp (a separate instantiation: the inference kernel is unchanged)
// kPaged: K / V from a paged cache, lengths per sequence from device memory (AttnParams, "paged cache")
template <int kD, typename T, bool kLse, bool kPaged>
__global__ void __maxnreg__(160) gqa_attention_kernel(const __grid_constant__ AttnParams p) {
    constexpr int kDAtoms = kD / 64;                       // 64-element (128-byte) column blocks of a head
    constexpr int kQBytes = kQTile * kD * 2;
    constexpr int kKBytes = kKvTile * kD * 2;              // also the V tile
    // 128-byte-swizzled tiles need 1024-byte alignment; the kernel has no static shared memory, so the dynamic window
    // starts aligned (checked: a misaligned base traps instead of corrupting tiles)
    extern __shared__ __align__(1024) uint8_t att_smem[];
    if ((smem_u32(att_smem) & 1023u) != 0) __trap();
    uint8_t* sq = att_smem;
    uint8_t* sk = sq + kQBytes;                            // 2 stages
    uint8_t* sv = sk + 2 * kKBytes;                        // 2 stages
    uint64_t* bar_q = reinterpret_cast<uint64_t*>(sv + 2 * kKBytes);
    uint64_t* bar_k = bar_q + 1;                           // [2] K tile landed
    uint64_t* bar_v = bar_k + 2;                           // [2] V tile landed
    uint64_t* bar_s = bar_v + 2;                           // [2] S = Q K^T complete (two accumulators: S of tile t + 1 runs
                                                           //     on the tensor cores while the softmax of tile t is computed)
    uint64_t* bar_o = bar_s + 2;                           // P V complete (P and the V stage may be reused)
    uint64_t* bar_p = bar_o + 1;                           // [2] P of the tile is in tensor memory (128 arrivals).  Two, used
                                                           //     alternately: a warp whose rows are all masked can finish tile
                                                           //     t + 1 before a slow warp has handed over tile t (nothing makes
                                                           //     it wait for the previous P V any more), and must not arrive
                                                           //     on the phase of tile t a second time
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_p + 2);

    const int tid = threadIdx.x;
    const uint32_t warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    // grid: split-KV (decode) = (splits, heads, batch); otherwise (heads, batch, query tiles) with the LAST query tile first:
    // under a causal mask the late tiles see the most keys, so the long CTAs start first and the short ones fill the tail,
    // and the CTAs running at the same time are the query heads of the same KV groups (their K / V tiles meet in L2)
    const int split = p.splits > 1 ? static_cast<int>(blockIdx.x) : 0;
    const int q0 = p.splits > 1 ? 0 : static_cast<int>(gridDim.z - 1 - blockIdx.z) * kQTile;
    const int head = p.splits > 1 ? blockIdx.y : blockIdx.x;
    const int b = p.splits > 1 ? blockIdx.z : blockIdx.y;
    const int kvh = head / (p.heads / p.kv_heads);

    if (tid == 0) {
        tma_prefetch_desc(&p.map_q);
        tma_prefetch_desc(&p.map_k);
        tma_prefetch_desc(&p.map_v);
        mbar_init(bar_q, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bar_k[i], 1);
            mbar_init(&bar_v[i], 1);
            mbar_init(&bar_s[i], 1);
        }
        mbar_init(bar_o, 1);
        mbar_init(&bar_p[0], kQTile);
        mbar_init(&bar_p[1], kQTile);
        fence_mbar_init();
    }
    constexpr uint32_t kTmemCols = 256u;                   // S[2] (2 x 64 columns) + P V (kD columns)
    if (warp == 4) {
        tmem_alloc<1>(tmem_slot, kTmemCols);
        tmem_relinquish<1>();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
    const uint32_t tmem_o = tmem_base + 2 * kKvTile;   // S of even / odd tiles: columns [0, 64) / [64, 128); P V: [128, 128 + kD)
    pdl_launch_dependents();
    pdl_wait_prior_grid();

    // paged: the CTA's sequence, its kv head in the pool and its lengths (written by earlier work of the stream).  Query rows
    // [q_rows, q_len) are right padding of a ragged call: they see no key and store zeros.
    int kv_len = p.kv_len, past_len = p.past_len, q_rows = p.q_len, tiles_per_split = p.tiles_per_split;
    int seq = b, kvh_pool = kvh;
    if constexpr (kPaged) {
        if (p.packed) {
            seq = b / p.page_kv_heads;
            kvh_pool = b % p.page_kv_heads;
        }
        past_len = p.past_lens[seq];
        const int n_new = p.new_lens != nullptr ? p.new_lens[seq] : (p.packed ? 1 : p.q_len);
        kv_len = past_len + n_new;
        q_rows = p.packed ? (n_new > 0 ? p.q_len : 0) : min(n_new, p.q_len);
    }
    // keys this query tile can see: [0, hi)
    const int q_last = min(q0 + kQTile, q_rows) - 1;
    int hi = kv_len;
    if (p.causal) hi = min(hi, past_len + q_last + 1);
    if constexpr (kPaged) {
        if (q_last < q0) hi = 0;                                          // the whole query tile is padding
    }
    const int total_tiles = (hi + kKvTile - 1) / kKvTile;
    if constexpr (kPaged) tiles_per_split = (total_tiles + p.splits - 1) / p.splits;   // the host plan, per sequence
    const int tile0 = split * tiles_per_split;                            // first key tile of this CTA (0 without split-KV)
    const int ntiles = p.splits > 1 ? max(0, min(tiles_per_split, total_tiles - tile0)) : total_tiles;
    const int kv_plane = b * p.kv_heads + kvh;
    const int key0 = tile0 * kKvTile;

    if (warp == 4) {
        // ------------------------------------------------------------------ TMA producer + MMA issuer (one thread)
        // The softmax warps never issue anything: the serial descriptor / tcgen05.mma stream of this thread is off their
        // critical path (measured: with the issuer inside softmax warp 0 the other warps spent a third of the kernel at the
        // CTA barrier waiting for it).
        if (ntiles > 0 && elect_one()) {   // elect.sync: ptxas knows the branch is single-lane (a lane == 0 test makes it wrap every
                                              // tcgen05.mma / TMA instruction in an ELECT ... BRA.U.ANY loop: ~140 clocks per MMA)
            // K tile, K-major: [64 keys][64 dims] per column block;  V tile: the same boxes, consumed as an MN-major B operand.
            // pg: paged, the pool page of tile t
            auto load_k = [&](int t, int pg) {
                const int s = t & 1;
                mbar_arrive_expect_tx(&bar_k[s], kKBytes);
#pragma unroll
                for (int a = 0; a < kDAtoms; ++a) {
                    if constexpr (kPaged)
                        tma_load_3d(sk + s * kKBytes + a * (kKvTile * 128), &p.map_k, &bar_k[s], a * 64, 0,
                                    pg * p.page_kv_heads + kvh_pool, kEvictNormal);
                    else
                        tma_load_3d(sk + s * kKBytes + a * (kKvTile * 128), &p.map_k, &bar_k[s], a * 64, key0 + t * kKvTile, kv_plane,
                                    kEvictNormal);
                }
            };
            auto load_v = [&](int t, int pg) {
                const int s = t & 1;
                mbar_arrive_expect_tx(&bar_v[s], kKBytes);
#pragma unroll
                for (int a = 0; a < kDAtoms; ++a) {
                    if constexpr (kPaged)
                        tma_load_3d(sv + s * kKBytes + a * (kKvTile * 128), &p.map_v, &bar_v[s], a * 64, 0,
                                    pg * p.page_kv_heads + kvh_pool, kEvictNormal);
                    else
                        tma_load_3d(sv + s * kKBytes + a * (kKvTile * 128), &p.map_v, &bar_v[s], a * 64, key0 + t * kKvTile, kv_plane,
                                    kEvictNormal);
                }
            };
            // Paged: the block-table entries are read a tile before the load that needs them (pg2 / pg3 = pages of tiles
            // t + 2 / t + 3 at step t), so no global-load latency sits in the TMA issue chain.
            const int* pages = nullptr;
            int pg0 = 0, pg1 = 0, pg2 = 0, pg3 = 0;
            auto page = [&](int t) { return t < ntiles ? __ldg(pages + t) : 0; };
            if constexpr (kPaged) {
                pages = p.block_table + static_cast<size_t>(seq) * p.pages_per_seq + tile0;
                pg0 = page(0); pg1 = page(1); pg2 = page(2); pg3 = page(3);
            }
            // S[128, 64] = Q[128, kD] K[64, kD]^T of tile t into accumulator t & 1
            const uint32_t q_addr = smem_u32(sq);
            auto issue_s = [&](int t) {
                const int s = t & 1;
                mbar_wait(&bar_k[s], (t >> 1) & 1u);
                tc_fence_after();
                const uint32_t k_addr = smem_u32(sk + s * kKBytes);
#pragma unroll
                for (int kk = 0; kk < kD / kUmmaKAtt; ++kk) {
                    const uint32_t qoff = (kk / 4) * (kQTile * 128) + (kk % 4) * 32;      // column block, then 32 B per K step
                    const uint32_t koff = (kk / 4) * (kKvTile * 128) + (kk % 4) * 32;
                    umma_f16<1>(tmem_base + s * kKvTile, make_smem_desc_sw128(q_addr + qoff, 0, 1024),
                                make_smem_desc_sw128(k_addr + koff, 0, 1024), p.idesc_s, kk > 0 ? 1u : 0u);
                }
                umma_commit<1>(&bar_s[s]);
            };
            mbar_arrive_expect_tx(bar_q, kQBytes);
#pragma unroll
            for (int a = 0; a < kDAtoms; ++a)
                tma_load_2d(sq + a * (kQTile * 128), &p.map_q, bar_q, head * kD + a * 64, b * p.q_len + q0, kEvictNormal);
            load_k(0, pg0);
            if (ntiles > 1) load_k(1, pg1);
            load_v(0, pg0);
            if (ntiles > 1) load_v(1, pg1);
            // P (16-bit) is written by the softmax warps over the first 32 columns of the S accumulator it was computed from,
            // and P V takes it from there (A operand in tensor memory): no shared-memory P tile, no generic -> async proxy
            // fence.  The tensor pipe executes in issue order, so S of tile t + 2 -- issued right behind P V of tile t --
            // overwrites that accumulator only after P V has read P from it.
            mbar_wait(bar_q, 0);
            issue_s(0);
            if (ntiles > 1) issue_s(1);
            if (ntiles > 2) {                             // K stage 0 is free once S of tile 0 is complete
                mbar_wait(&bar_s[0], 0);
                load_k(2, pg2);
            }
            for (int t = 0; t < ntiles; ++t) {
                const int s = t & 1;
                int pg_next = 0;
                if constexpr (kPaged) pg_next = page(t + 4);   // used at step t + 1: its latency hides behind this step's waits
                // O[128, kD] (+)= P[128, 64] V[64, kD]   (V consumed MN-major: [64 keys][kD]); tile 0 overwrites
                mbar_wait(&bar_p[s], (t >> 1) & 1u);
                mbar_wait(&bar_v[s], (t >> 1) & 1u);
                tc_fence_after();
                const uint32_t v_addr = smem_u32(sv + s * kKBytes);
                const uint32_t p_tmem = tmem_base + s * kKvTile;
#ifndef L32_ATT_NOPV
#pragma unroll
                for (int kk = 0; kk < kKvTile / kUmmaKAtt; ++kk)
                    umma_f16_ts(tmem_o, p_tmem + kk * (kUmmaKAtt / 2),
                                make_smem_desc_sw128(v_addr + kk * (kUmmaKAtt * 128), kKvTile * 128, 1024), p.idesc_o,
                                (t > 0 || kk > 0) ? 1u : 0u);
#endif
                umma_commit<1>(bar_o);
                if (t + 2 < ntiles) issue_s(t + 2);       // (K of tile t + 2 was requested a tile ago)
                if (t + 3 < ntiles) {                     // K stage (t + 1) & 1 is free once S of tile t + 1 is complete
                    mbar_wait(&bar_s[s ^ 1], ((t + 1) >> 1) & 1u);
                    load_k(t + 3, pg3);
                }
                if (t + 2 < ntiles) {                     // V stage t & 1 is free once P V of tile t is complete
                    mbar_wait(bar_o, t & 1u);
                    load_v(t + 2, pg2);
                }
                pg2 = pg3;
                pg3 = pg_next;
            }
        }
    } else {
        // ------------------------------------------------------------------ softmax warps: one query row per thread = one TMEM lane
        const int qi = q0 + tid;                       // query index inside the sequence
        const int qpos = past_len + qi;                // its absolute position
        const bool row_ok = qi < p.q_len;
        // Online softmax with a LAZY reference: the output accumulator stays in TMEM across the key tiles (P V accumulates
        // there) and is rescaled -- a TMEM read-modify-write of this thread's row -- only when the row maximum outgrows the
        // reference by more than 2^kLazyLog2 (probabilities then stay <= 2^kLazyLog2: exact in fp32, harmless in the 16-bit
        // P).  TMEM reads are the scarce resource here (64 B / clock / SM): S is read once per tile, O once at the end.
        constexpr float kLazyLog2 = 8.0f;
        float m_ref = -INFINITY, l = 0.f;
        const uint32_t lane_off = (warp * 32u) << 16;
        const uint8_t* keep_row = p.keep != nullptr ? p.keep + static_cast<size_t>(b) * p.kv_len : nullptr;

        // One tile: `cur` holds the raw scores of tile t (read from TMEM during the previous tile); the scores of tile t + 1
        // are requested into `nxt` before the exponentials of tile t are computed, so the TMEM read (64 B / clock / SM) and
        // the wait for S hide behind the MUFU work.  The exponentials go to registers first: the previous tile's P V only has
        // to be complete when P is stored and when the accumulator is rescaled.
        auto process = [&](int t, uint32_t (&cur)[kKvTile], uint32_t (&nxt)[kKvTile]) {
            const int j0 = (tile0 + t) * kKvTile;
            // key padding: the tile's 64 keep bytes become two ballot words per warp (lane = key; every lane of the warp takes
            // part: keep_row is CTA-uniform) -- two byte loads per thread and tile instead of a loop over the keys
            uint32_t keep_lo = 0xffffffffu, keep_hi = 0xffffffffu;
            if (keep_row != nullptr) {
                const int ka = j0 + static_cast<int>(lane_id()), kb = ka + 32;
                keep_lo = __ballot_sync(0xffffffffu, ka < p.kv_len && keep_row[ka] != 0);
                keep_hi = __ballot_sync(0xffffffffu, kb < p.kv_len && keep_row[kb] != 0);
            }
            // A tile every key of which is visible needs no per-element predicates (all but the diagonal / last / padded tiles).
            int kvl = p.kv_len;
            if constexpr (kPaged) kvl = kv_len;
            const bool full = (j0 + kKvTile <= kvl) && (!p.causal || j0 + kKvTile - 1 <= qpos) && (keep_lo & keep_hi) == 0xffffffffu;
            if (!full) {
                // keys [0, lim) of the tile pass the length / causal tests
                const int lim = min(kvl, p.causal ? qpos + 1 : kvl) - j0;
                const uint32_t vis_lo = (lim >= 32 ? 0xffffffffu : (lim > 0 ? (1u << lim) - 1u : 0u)) & keep_lo;
                const uint32_t vis_hi = (lim >= 64 ? 0xffffffffu : (lim > 32 ? (1u << (lim - 32)) - 1u : 0u)) & keep_hi;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    if (!(vis_lo & (1u << j))) cur[j] = 0xff800000u;      // -inf
                    if (!(vis_hi & (1u << j))) cur[32 + j] = 0xff800000u;
                }
            }
            float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
            for (int j = 0; j < kKvTile; j += 4) {
#pragma unroll
                for (int q4 = 0; q4 < 4; ++q4) mx[q4] = fmaxf(mx[q4], __uint_as_float(cur[j + q4]));
            }
            const float tmax = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])) * p.scale_log2;   // scale > 0: max commutes with it
            // tcgen05.ld / .st are warp-collective: the rescale is taken by the whole warp as soon as one of its rows needs a
            // new reference; the other rows rescale by exactly 1
            const bool want = tmax > m_ref + kLazyLog2;                   // also true for the first visible key (m_ref = -inf)
            const bool any = __any_sync(0xffffffffu, want);
            float alpha = 1.f;
            if (any) {
                alpha = want ? fast_exp2(m_ref - tmax) : 1.f;             // m_ref = -inf: 0
                l *= alpha;
                if (want) m_ref = tmax;
            }
            // ---- probabilities (registers): ALL the MUFU work of the tile comes before anything that depends on the previous
            // tile's P V.  A masked score is -inf: 2^(-inf * scale - m) = 0 as long as m is finite.  A row that has not seen a
            // visible key yet has m_ref = -inf (and only -inf scores): its exponent reference is taken as 0 so that no nan
            // appears.
            const float neg_m = (m_ref == -INFINITY) ? 0.f : -m_ref;
            const uint64_t scale2 = pack_f32x2(__float_as_uint(p.scale_log2), __float_as_uint(p.scale_log2));
            const uint64_t neg_m2 = pack_f32x2(__float_as_uint(neg_m), __float_as_uint(neg_m));
            uint64_t ps2[2] = {0ull, 0ull};         // four independent row-sum chains, two per packed accumulator
            uint32_t pk[kKvTile / 2];
#pragma unroll
            for (int j = 0; j < kKvTile / 2; ++j) {
                float x0, x1;
                unpack_f32x2(fma_f32x2(pack_f32x2(cur[2 * j], cur[2 * j + 1]), scale2, neg_m2), x0, x1);
                const float p0 = fast_exp2(x0), p1 = fast_exp2(x1);
                pk[j] = Pack2<T>::pack(p0, p1);
                ps2[j & 1] = add_f32x2(ps2[j & 1], pack_f32x2(__float_as_uint(p0), __float_as_uint(p1)));
            }
            {
                float s0, s1, s2, s3;
                unpack_f32x2(ps2[0], s0, s1);
                unpack_f32x2(ps2[1], s2, s3);
                l += (s0 + s1) + (s2 + s3);
            }
            // ---- next tile's scores: S of tile t + 1 was issued behind P V of tile t - 1 and has had the whole exponential
            // phase to complete; the read is awaited after P is handed over
            if (t + 1 < ntiles) {
                mbar_wait(&bar_s[(t + 1) & 1], ((t + 1) >> 1) & 1u);
                tc_fence_after();
                const uint32_t tmem_s_next = tmem_base + ((t + 1) & 1) * kKvTile + lane_off;
                uint32_t (&lo)[32] = *reinterpret_cast<uint32_t (*)[32]>(&nxt[0]);
                uint32_t (&hi32)[32] = *reinterpret_cast<uint32_t (*)[32]>(&nxt[32]);
                tmem_ld_32x32b_x32(tmem_s_next, lo);
                tmem_ld_32x32b_x32(tmem_s_next + 32, hi32);
            } else {                                  // (defined on every path: the old contents are dead for the compiler too)
#pragma unroll
                for (int j = 0; j < kKvTile; ++j) nxt[j] = 0u;
            }
            // ---- the accumulator is touched only when a row of this warp needs a new reference (rare after the first
            // tiles): only then does the previous tile's P V have to be complete here
            if (t > 0 && any) {
                mbar_wait(bar_o, (t - 1) & 1u);
                tc_fence_after();
#pragma unroll
                for (int c = 0; c < kD / 8; ++c) {                    // small chunks keep the register need of the rare path low
                    uint32_t v[8];
                    tmem_ld_32x32b_x8(tmem_o + lane_off + c * 8, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) * alpha);
                    tmem_st_32x32b_x8(tmem_o + lane_off + c * 8, v);
                }
            }
            // ---- P -> tensor memory, over the first 32 columns of the accumulator S of this tile came from (this thread's
            // lane; it read those columns into registers a tile ago): the A operand of P V
            {
                const uint32_t tmem_p = tmem_base + (t & 1) * kKvTile + lane_off;
                uint32_t (&p_lo)[16] = *reinterpret_cast<uint32_t (*)[16]>(&pk[0]);
                uint32_t (&p_hi)[16] = *reinterpret_cast<uint32_t (*)[16]>(&pk[16]);
                tmem_st_32x32b_x16(tmem_p, p_lo);
                tmem_st_32x32b_x16(tmem_p + 16, p_hi);
            }
            tmem_st_wait();
            // Every thread watches EVERY phase of bar_o (a parity wait can only tell the current phase from the previous one:
            // a thread that skipped a phase would take "tile t - 2 complete" for "tile t complete", or hang on a parity that
            // has come round again).  Here P V of tile t - 1 has had the whole tile to finish, and P V of tile t cannot have
            // been issued yet (this thread has not arrived), so the wait is free and unambiguous.
            if (t > 0 && !any) mbar_wait(bar_o, (t - 1) & 1u);
            tc_fence_before();             // this thread's tcgen05.ld / .st are ordered before the issuer's next tcgen05.mma
            mbar_arrive(&bar_p[t & 1]);
            if (t + 1 < ntiles) tmem_ld_wait();    // the next tile's scores are in registers
        };
        uint32_t sc_a[kKvTile], sc_b[kKvTile];
        if (ntiles > 0) {
            mbar_wait(&bar_s[0], 0);
            tc_fence_after();
            uint32_t (&lo)[32] = *reinterpret_cast<uint32_t (*)[32]>(&sc_a[0]);
            uint32_t (&hi32)[32] = *reinterpret_cast<uint32_t (*)[32]>(&sc_a[32]);
            tmem_ld_32x32b_x32(tmem_base + lane_off, lo);
            tmem_ld_32x32b_x32(tmem_base + lane_off + 32, hi32);
            tmem_ld_wait();
        }
        for (int t = 0; t < ntiles; t += 2) {
            process(t, sc_a, sc_b);
            if (t + 1 < ntiles) {
                process(t + 1, sc_b, sc_a);
            } else {                                  // (dead values: tells the compiler sc_a is not live across tile t)
#pragma unroll
                for (int j = 0; j < kKvTile; ++j) sc_a[j] = 0u;
            }
        }
        if (ntiles > 0) {
            mbar_wait(bar_o, (ntiles - 1) & 1u);
            tc_fence_after();
        }
        if (p.splits > 1) {
            // split-KV: the unnormalised accumulator row and its (reference, sum) leave for the combine kernel
            const size_t slot = ((static_cast<size_t>(b) * p.heads + head) * p.splits + split) * p.q_len + (row_ok ? qi : 0);
            if (row_ok) p.part_ml[slot] = make_float2(ntiles > 0 ? m_ref : -INFINITY, ntiles > 0 ? l : 0.f);
            float* dstf = p.part_o + slot * kD;
#pragma unroll
            for (int c = 0; c < kD / 32; ++c) {
                uint32_t v[32];
                if (ntiles > 0) {
                    tmem_ld_32x32b_x32(tmem_o + lane_off + c * 32, v);
                    tmem_ld_wait();
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = 0u;
                }
                if (row_ok) {
#pragma unroll
                    for (int j4 = 0; j4 < 8; ++j4)
                        *reinterpret_cast<uint4*>(dstf + c * 32 + 4 * j4) = make_uint4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
                }
            }
        } else {
        const float inv = (ntiles > 0 && l > 0.f) ? 1.f / l : 0.f;     // a row without any visible key gives zeros
        if (kLse && row_ok)
            p.lse[(static_cast<size_t>(b) * p.heads + head) * p.q_len + qi] = inv > 0.f ? m_ref + log2f(l) : INFINITY;
        T* dst = static_cast<T*>(p.out) + (static_cast<size_t>(b) * p.q_len + (row_ok ? qi : 0)) * (static_cast<size_t>(p.heads) * kD) +
                 head * kD;
#pragma unroll
        for (int c = 0; c < kD / 32; ++c) {
            uint32_t v[32];
            if (ntiles > 0) {                          // CTA-uniform; the loads are warp-collective (every lane takes part)
                tmem_ld_32x32b_x32(tmem_o + lane_off + c * 32, v);
                tmem_ld_wait();
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = 0u;
            }
            if constexpr (kPaged) {
                if (qi >= q_rows) {                    // right padding: exact zeros
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = 0u;
                }
            }
            if (row_ok) {
#pragma unroll
                for (int j4 = 0; j4 < 4; ++j4) {
                    uint4 w;
                    w.x = Pack2<T>::pack(__uint_as_float(v[8 * j4]) * inv, __uint_as_float(v[8 * j4 + 1]) * inv);
                    w.y = Pack2<T>::pack(__uint_as_float(v[8 * j4 + 2]) * inv, __uint_as_float(v[8 * j4 + 3]) * inv);
                    w.z = Pack2<T>::pack(__uint_as_float(v[8 * j4 + 4]) * inv, __uint_as_float(v[8 * j4 + 5]) * inv);
                    w.w = Pack2<T>::pack(__uint_as_float(v[8 * j4 + 6]) * inv, __uint_as_float(v[8 * j4 + 7]) * inv);
                    *reinterpret_cast<uint4*>(dst + c * 32 + 8 * j4) = w;
                }
            }
        }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        tmem_dealloc<1>(tmem_base, kTmemCols);
    }
}

// Split-KV combine: out[row] = sum_s O_s 2^(m_s - M) / sum_s l_s 2^(m_s - M), M = max_s m_s.  One warp per (batch, head, row).
template <typename T>
__global__ void __launch_bounds__(128) attention_combine_kernel(const float* __restrict__ part_o, const float2* __restrict__ part_ml,
                                                               T* __restrict__ out, int batch, int heads, int q_len, int splits,
                                                               int d) {
    pdl_wait_prior_grid();
    const long long w = blockIdx.x * 4ll + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    const long long total = static_cast<long long>(batch) * heads * q_len;
    if (w >= total) return;
    const int qi = static_cast<int>(w % q_len);
    const long long bh = w / q_len;                       // b * heads + head
    float mx = -INFINITY;
    for (int s = 0; s < splits; ++s) mx = fmaxf(mx, part_ml[(bh * splits + s) * q_len + qi].x);
    float lsum = 0.f;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};                  // d <= 128: 4 columns per lane
    for (int s = 0; s < splits; ++s) {
        const size_t slot = (bh * splits + s) * q_len + qi;
        const float2 ml = part_ml[slot];
        if (ml.x == -INFINITY) continue;
        const float sc = exp2f(ml.x - mx);
        lsum += ml.y * sc;
        for (int c = 0; c < 4; ++c) {
            const int col = lane + 32 * c;
            if (col < d) acc[c] = fmaf(part_o[slot * d + col], sc, acc[c]);
        }
    }
    const float inv = lsum > 0.f ? 1.f / lsum : 0.f;
    const int b = static_cast<int>(bh / heads), head = static_cast<int>(bh % heads);
    T* dst = out + (static_cast<size_t>(b) * q_len + qi) * (static_cast<size_t>(heads) * d) + static_cast<size_t>(head) * d;
    for (int c = 0; c < 4; ++c) {
        const int col = lane + 32 * c;
        if (col < d) dst[col] = static_cast<T>(acc[c] * inv);
    }
}

// RoPE + cache append, the rotate_half form
//   out[i] = x[i] cos - x[i + d/2] sin,  out[i + d/2] = x[i + d/2] cos + x[i] sin,  angle = position * base^(-2 i / d)
// (reference Model/model.py:188-198; cos / sin in fp32 instead of the reference's storage-dtype cos / sin).
// One CTA per token.  The d / 2 angles of the token are computed ONCE (the first d / 2 threads, fp32 sincosf) and shared by
// its heads + 2 kv_heads head rows through shared memory; every thread then moves 16-byte vectors: thread (slot, j) takes
// elements [8 j, 8 j + 8) of both halves of the head rows slot, slot + 16, ... (q heads rotated in place, k heads rotated
// into the cache, v heads copied into the cache).
// kPaged: the cache is a page pool [num_pages, kv_heads, kKvTile, d]; token t of sequence b goes to position pos = past_lens[b]
// + t, i.e. row pos % kKvTile of page block_table[b][pos / kKvTile].  A token t >= new_lens[b] (right padding) writes no
// cache row (its q is still rotated).
template <typename T, bool kPaged>
__global__ void __launch_bounds__(128) rope_kv_append_kernel(T* q, const T* __restrict__ k_new, const T* __restrict__ v_new,
                                                            const long long* __restrict__ position_ids, T* cache_k, T* cache_v,
                                                            int q_len, int heads, int kv_heads, int d, int max_len,
                                                            int past_len, float log2_base, const int* __restrict__ block_table,
                                                            const int* __restrict__ past_lens, const int* __restrict__ new_lens,
                                                            int pages_per_seq) {
    __shared__ float cs_sh[64], sn_sh[64];             // d / 2 <= 64
    pdl_wait_prior_grid();
    const int half = d >> 1;
    const long long tok = blockIdx.x;                    // b * q_len + t
    const int t = static_cast<int>(tok % q_len);
    const int b = static_cast<int>(tok / q_len);
    if (static_cast<int>(threadIdx.x) < half) {
        const int i = threadIdx.x;
        rope_cos_sin(static_cast<float>(position_ids[tok]), i, d, log2_base, cs_sh[i], sn_sh[i]);
    }
    __syncthreads();
    const int vph = d >> 4;                              // 16-byte vectors per half row
    const int j = threadIdx.x % vph;
    const int slot = threadIdx.x / vph;                  // 0 .. 15
    float cs[8], sn[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        cs[e] = cs_sh[8 * j + e];
        sn[e] = sn_sh[8 * j + e];
    }
    int units = heads + 2 * kv_heads;
    long long page = 0;
    int row = 0;
    if constexpr (kPaged) {
        const int pos = past_lens[b] + t;
        if (new_lens != nullptr && t >= new_lens[b])
            units = heads;
        else
            page = block_table[static_cast<long long>(b) * pages_per_seq + pos / kKvTile];
        row = pos % kKvTile;
    }
    for (int u = slot; u < units; u += 16) {
        const T* src;
        T* dst;
        bool rotate = true;
        if (u < heads) {
            T* x = q + (tok * heads + u) * d;
            src = x;
            dst = x;
        } else if (u < heads + kv_heads) {
            const int h = u - heads;
            src = k_new + (tok * kv_heads + h) * d;
            if constexpr (kPaged)
                dst = cache_k + ((page * kv_heads + h) * kKvTile + row) * d;
            else
                dst = cache_k + ((static_cast<long long>(b) * kv_heads + h) * max_len + past_len + t) * d;
        } else {
            const int h = u - heads - kv_heads;
            src = v_new + (tok * kv_heads + h) * d;
            if constexpr (kPaged)
                dst = cache_v + ((page * kv_heads + h) * kKvTile + row) * d;
            else
                dst = cache_v + ((static_cast<long long>(b) * kv_heads + h) * max_len + past_len + t) * d;
            rotate = false;
        }
        const uint4 lo = *reinterpret_cast<const uint4*>(src + 8 * j);
        const uint4 hi = *reinterpret_cast<const uint4*>(src + half + 8 * j);
        if (!rotate) {
            *reinterpret_cast<uint4*>(dst + 8 * j) = lo;
            *reinterpret_cast<uint4*>(dst + half + 8 * j) = hi;
            continue;
        }
        const T* a = reinterpret_cast<const T*>(&lo);
        const T* c = reinterpret_cast<const T*>(&hi);
        uint4 olo, ohi;
        T* oa = reinterpret_cast<T*>(&olo);
        T* oc = reinterpret_cast<T*>(&ohi);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const float av = static_cast<float>(a[e]), cv = static_cast<float>(c[e]);
            oa[e] = static_cast<T>(av * cs[e] - cv * sn[e]);
            oc[e] = static_cast<T>(cv * cs[e] + av * sn[e]);
        }
        *reinterpret_cast<uint4*>(dst + 8 * j) = olo;
        *reinterpret_cast<uint4*>(dst + half + 8 * j) = ohi;
    }
}

template <int kD, typename T, bool kLse, bool kPaged>
int launch_attention(const AttnParams& p, cudaStream_t s) {
    auto* kernel = gqa_attention_kernel<kD, T, kLse, kPaged>;
    size_t smem = kQTile * kD * 2 + 4 * kKvTile * kD * 2 + 128;   // tiles + barriers
    if (const char* v = getenv("L32_ATT_ONE_CTA_PER_SM")) {   // experiments only: pad so that only one CTA fits per SM
        if (*v == '1') smem = 160 * 1024;
    }
    static bool configured_dev[kMaxDevices] = {};
    bool& configured = configured_dev[current_device_slot()];
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return static_cast<int>(e);
        configured = true;
        if (getenv("L32_ATT_DEBUG") != nullptr) {
            int nb = 0;
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, kAttThreads, smem);
            cudaFuncAttributes fa;
            cudaFuncGetAttributes(&fa, kernel);
            fprintf(stderr, "[l32] gqa_attention_kernel<%d>: %d CTAs / SM, %d registers, %zu B local, %zu B dynamic smem\n", kD, nb,
                    fa.numRegs, fa.localSizeBytes, smem);
        }
    }
    cudaLaunchConfig_t cfg = {};
    if (p.splits > 1)
        cfg.gridDim = dim3(static_cast<unsigned>(p.splits), static_cast<unsigned>(p.heads), static_cast<unsigned>(p.batch));
    else
        cfg.gridDim = dim3(static_cast<unsigned>(p.heads), static_cast<unsigned>(p.batch),
                           static_cast<unsigned>((p.q_len + kQTile - 1) / kQTile));
    cfg.blockDim = dim3(kAttThreads);
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

// Fields every attention launch shares: shapes, scale, instruction descriptors and the Q map.
int attention_setup(AttnParams& p, const void* q, void* out, int batch, int q_len, int heads, int kv_heads, int head_dim,
                    int causal, int dtype) {
    memset(&p, 0, sizeof(p));
    p.out = out;
    p.batch = batch; p.q_len = q_len; p.heads = heads; p.kv_heads = kv_heads; p.causal = causal;
    p.scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(head_dim));
    p.idesc_s = make_idesc_f16(dtype == L32_BF16, kQTile, kKvTile, false, false);
    p.idesc_o = make_idesc_f16(dtype == L32_BF16, kQTile, static_cast<uint32_t>(head_dim), false, true);
    return make_tensor_map_2d(&p.map_q, q, static_cast<uint64_t>(batch) * q_len, static_cast<uint64_t>(heads) * head_dim,
                              static_cast<uint64_t>(heads) * head_dim, kQTile, 64, dtype);
}

// Split-KV: `splits` CTAs per (batch, head) over the key tiles of kv_len keys; the partials go to the workspace.
void attention_split(AttnParams& p, int splits, int kv_len, int head_dim, void* workspace) {
    p.splits = splits > 1 ? splits : 1;
    if (p.splits > 1) {
        const int tiles = (kv_len + kKvTile - 1) / kKvTile;
        p.tiles_per_split = (tiles + p.splits - 1) / p.splits;
        const size_t rows = static_cast<size_t>(p.batch) * p.heads * p.splits * p.q_len;
        p.part_o = static_cast<float*>(workspace);
        p.part_ml = reinterpret_cast<float2*>(static_cast<uint8_t*>(workspace) + ((rows * head_dim * sizeof(float) + 255) & ~static_cast<size_t>(255)));
    }
}

// The inference kernel, then (split-KV) the merge of its partials.
template <bool kPaged>
int attention_run(const AttnParams& p, int head_dim, int dtype, cudaStream_t s) {
    int rc;
    if (dtype == L32_BF16) {
        rc = head_dim == 128 ? launch_attention<128, __nv_bfloat16, false, kPaged>(p, s) : launch_attention<64, __nv_bfloat16, false, kPaged>(p, s);
    } else {
        rc = head_dim == 128 ? launch_attention<128, __half, false, kPaged>(p, s) : launch_attention<64, __half, false, kPaged>(p, s);
    }
    if (rc != L32_OK || p.splits == 1) return rc;
    // merge the split-KV partials
    const long long rows = static_cast<long long>(p.batch) * p.heads * p.q_len;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>((rows + 3) / 4));
    cfg.blockDim = dim3(128);
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const float* po = p.part_o;
    const float2* pml = p.part_ml;
    cudaError_t e;
    if (dtype == L32_BF16)
        e = cudaLaunchKernelEx(&cfg, attention_combine_kernel<__nv_bfloat16>, po, pml, static_cast<__nv_bfloat16*>(p.out), p.batch,
                               p.heads, p.q_len, p.splits, head_dim);
    else
        e = cudaLaunchKernelEx(&cfg, attention_combine_kernel<__half>, po, pml, static_cast<__half*>(p.out), p.batch, p.heads, p.q_len,
                               p.splits, head_dim);
    if (e == cudaSuccess) count_launch();
    return static_cast<int>(e);
}

// Paged-cache arguments of rope_kv_append_kernel (null: the contiguous cache).
struct RopePages {
    const int* block_table;
    const int* past_lens;
    const int* new_lens;
    int pages_per_seq;
};

template <typename T, bool kPaged>
cudaError_t launch_rope(const cudaLaunchConfig_t& cfg, void* q, const void* k_new, const void* v_new, const long long* position_ids,
                        void* cache_k, void* cache_v, int q_len, int heads, int kv_heads, int head_dim, int max_len, int past_len,
                        float log2_base, const RopePages& pg) {
    return cudaLaunchKernelEx(&cfg, rope_kv_append_kernel<T, kPaged>, static_cast<T*>(q), static_cast<const T*>(k_new),
                              static_cast<const T*>(v_new), position_ids, static_cast<T*>(cache_k), static_cast<T*>(cache_v), q_len,
                              heads, kv_heads, head_dim, max_len, past_len, log2_base, pg.block_table, pg.past_lens, pg.new_lens,
                              pg.pages_per_seq);
}

int rope_append(void* q, const void* k_new, const void* v_new, const long long* position_ids, void* cache_k, void* cache_v,
                int batch, int q_len, int heads, int kv_heads, int head_dim, int max_len, int past_len, float rope_base, int dtype,
                cudaStream_t s, const RopePages* pages) {
    const long long tokens = static_cast<long long>(batch) * q_len;
    if (tokens == 0) return L32_OK;
    if (head_dim != 64 && head_dim != 128) return L32_ERR_BAD_SHAPE;
    if (tokens > 0x7fffffffll) return L32_ERR_BAD_SHAPE;
    if (!is_aligned16(q) || !is_aligned16(k_new) || !is_aligned16(v_new) || !is_aligned16(cache_k) || !is_aligned16(cache_v))
        return L32_ERR_BAD_ALIGN;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(tokens));
    cfg.blockDim = dim3(static_cast<unsigned>((head_dim / 16) * 16));
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const float log2_base = log2f(rope_base);
    const RopePages none = {nullptr, nullptr, nullptr, 0};
    const RopePages& pg = pages != nullptr ? *pages : none;
    cudaError_t e;
    if (dtype == L32_BF16)
        e = pages != nullptr ? launch_rope<__nv_bfloat16, true>(cfg, q, k_new, v_new, position_ids, cache_k, cache_v, q_len, heads,
                                                                kv_heads, head_dim, max_len, past_len, log2_base, pg)
                             : launch_rope<__nv_bfloat16, false>(cfg, q, k_new, v_new, position_ids, cache_k, cache_v, q_len, heads,
                                                                 kv_heads, head_dim, max_len, past_len, log2_base, pg);
    else
        e = pages != nullptr ? launch_rope<__half, true>(cfg, q, k_new, v_new, position_ids, cache_k, cache_v, q_len, heads, kv_heads,
                                                         head_dim, max_len, past_len, log2_base, pg)
                             : launch_rope<__half, false>(cfg, q, k_new, v_new, position_ids, cache_k, cache_v, q_len, heads, kv_heads,
                                                          head_dim, max_len, past_len, log2_base, pg);
    if (e == cudaSuccess) count_launch();
    return static_cast<int>(e);
}

}  // namespace

int gqa_attention_packed(const void* q, const void* cache_k, const void* cache_v, void* out, int batch2, int group, int head_dim,
                         int max_len, int kv_len, int splits, void* workspace, int dtype, cudaStream_t s);
int gqa_attention_launch(const void* q, const void* cache_k, const void* cache_v, const uint8_t* keep, void* out, int batch, int q_len,
                         int heads, int kv_heads, int head_dim, int max_len, int kv_len, int past_len, int causal, int splits,
                         void* workspace, int dtype, cudaStream_t s, float* lse = nullptr);

int rope_kv_append(void* q, const void* k_new, const void* v_new, const long long* position_ids, void* cache_k, void* cache_v,
                   int batch, int q_len, int heads, int kv_heads, int head_dim, int max_len, int past_len, float rope_base,
                   int dtype, cudaStream_t s) {
    return rope_append(q, k_new, v_new, position_ids, cache_k, cache_v, batch, q_len, heads, kv_heads, head_dim, max_len, past_len,
                       rope_base, dtype, s, nullptr);
}

int rope_kv_append_paged(void* q, const void* k_new, const void* v_new, const long long* position_ids, void* pool_k, void* pool_v,
                         const int* block_table, const int* past_lens, const int* new_lens, int batch, int q_len, int heads,
                         int kv_heads, int head_dim, int max_pages_per_seq, float rope_base, int dtype, cudaStream_t s) {
    const RopePages pages = {block_table, past_lens, new_lens, max_pages_per_seq};
    return rope_append(q, k_new, v_new, position_ids, pool_k, pool_v, batch, q_len, heads, kv_heads, head_dim, kKvTile, 0, rope_base,
                       dtype, s, &pages);
}

// Split-KV plan of a decode call without key padding: the number of key splits (1 = none).  Only the packed decode path
// splits: one query per sequence, the `group` query heads of a KV group as the rows of ONE query tile (a split CTA covers
// rows [0, kQTile) only, so a larger group is not split).
static int decode_splits(int batch, int q_len, int heads, int kv_heads, int kv_len) {
    const int group = heads / kv_heads;
    if (q_len != 1 || batch <= 0 || group < 2 || group > kQTile) return 1;
    const int tiles = (kv_len + kKvTile - 1) / kKvTile;
    const int ctas = batch * kv_heads;                    // decode packs the heads of a KV group into one CTA
    int splits = (2 * num_sms() + ctas - 1) / ctas;       // aim at two CTAs per SM
    if (splits > tiles / 2) splits = tiles / 2;           // at least two key tiles (128 keys) per split
    return splits < 2 ? 1 : splits;
}

size_t gqa_attention_workspace_bytes(int batch, int q_len, int heads, int kv_heads, int head_dim, int kv_len) {
    const int splits = decode_splits(batch, q_len, heads, kv_heads, kv_len);
    if (splits < 2) return 0;
    return static_cast<size_t>(batch) * heads * splits * (static_cast<size_t>(head_dim) + 2) * sizeof(float) + 256;
}

int gqa_attention(const void* q, const void* cache_k, const void* cache_v, const uint8_t* keep, void* out, int batch, int q_len,
                  int heads, int kv_heads, int head_dim, int max_len, int kv_len, int past_len, int causal, void* workspace,
                  size_t workspace_bytes, int dtype, cudaStream_t s) {
    if (head_dim != 64 && head_dim != 128) return L32_ERR_BAD_SHAPE;
    if (batch <= 0 || q_len <= 0) return L32_OK;
    if (q_len == 1 && heads > kv_heads && keep == nullptr) {
        // Decode: the query heads of one KV group become the ROWS of one tile (q is [batch, kv_heads, group, head_dim] in
        // memory), so every K / V tile is read once per group instead of once per query head.  One query per sequence sees
        // the whole cache: no causal predicate needed.
        const int group = heads / kv_heads;
        const size_t need = gqa_attention_workspace_bytes(batch, 1, heads, kv_heads, head_dim, kv_len);
        const int splits = (need > 0 && workspace != nullptr && workspace_bytes >= need) ? decode_splits(batch, 1, heads, kv_heads, kv_len)
                                                                                         : 1;   // too short: one pass
        return gqa_attention_packed(q, cache_k, cache_v, out, batch * kv_heads, group, head_dim, max_len, kv_len, splits, workspace,
                                    dtype, s);
    }
    return gqa_attention_launch(q, cache_k, cache_v, keep, out, batch, q_len, heads, kv_heads, head_dim, max_len, kv_len, past_len,
                                causal, 1, nullptr, dtype, s);
}

// Paged cache: the same three launch shapes (packed decode, its split-KV form, the general causal kernel) with K / V tiles
// read through the block table and each sequence's lengths read from device memory.  The split plan is the contiguous
// path's for kv_len = max_kv_len (a host bound on every sequence's length); each sequence then divides its own key tiles over
// those splits.
int gqa_attention_paged(const void* q, const void* pool_k, const void* pool_v, const int* block_table, const int* past_lens,
                        const int* new_lens, void* out, void* workspace, size_t workspace_bytes, int batch, int q_len, int heads,
                        int kv_heads, int head_dim, int num_pages, int max_pages_per_seq, int max_kv_len, int dtype, cudaStream_t s) {
    if (head_dim != 64 && head_dim != 128) return L32_ERR_BAD_SHAPE;
    if (batch <= 0 || q_len <= 0) return L32_OK;
    const bool packed = q_len == 1 && heads > kv_heads;
    AttnParams p;
    int rc = packed ? attention_setup(p, q, out, batch * kv_heads, heads / kv_heads, 1, 1, head_dim, 0, dtype)
                    : attention_setup(p, q, out, batch, q_len, heads, kv_heads, head_dim, 1, dtype);
    if (rc != L32_OK) return rc;
    p.block_table = block_table;
    p.past_lens = past_lens;
    p.new_lens = new_lens;
    p.pages_per_seq = max_pages_per_seq;
    p.page_kv_heads = kv_heads;
    p.packed = packed ? 1 : 0;
    // K / V: one plane per (page, kv head) of kKvTile rows.  Rows of a page past its sequence's length are read as they are
    // and get P = 0: the pool's contract keeps them finite (include/l32_ffn.h).
    const uint64_t planes = static_cast<uint64_t>(num_pages) * kv_heads, plane_elems = static_cast<uint64_t>(kKvTile) * head_dim;
    rc = make_tensor_map_3d(&p.map_k, pool_k, planes, kKvTile, head_dim, head_dim, plane_elems, kKvTile, dtype);
    if (rc != L32_OK) return rc;
    rc = make_tensor_map_3d(&p.map_v, pool_v, planes, kKvTile, head_dim, head_dim, plane_elems, kKvTile, dtype);
    if (rc != L32_OK) return rc;
    int splits = 1;
    if (packed) {
        const size_t need = gqa_attention_workspace_bytes(batch, 1, heads, kv_heads, head_dim, max_kv_len);
        if (need > 0 && workspace != nullptr && workspace_bytes >= need) splits = decode_splits(batch, 1, heads, kv_heads, max_kv_len);
    }
    attention_split(p, splits, max_kv_len, head_dim, workspace);
    return attention_run<true>(p, head_dim, dtype, s);
}

// Training forward: keys [0, q_len) of the K / V buffers, no past, no split-KV; also writes the per-row log-sum-exp.
int gqa_attention_train(const void* q, const void* cache_k, const void* cache_v, const uint8_t* keep, void* out, float* lse, int batch,
                        int q_len, int heads, int kv_heads, int head_dim, int max_len, int causal, int dtype, cudaStream_t s) {
    if (head_dim != 64 && head_dim != 128) return L32_ERR_BAD_SHAPE;
    if (batch <= 0 || q_len <= 0) return L32_OK;
    return gqa_attention_launch(q, cache_k, cache_v, keep, out, batch, q_len, heads, kv_heads, head_dim, max_len, q_len, 0, causal, 1,
                                nullptr, dtype, s, lse);
}

// Decode layout: batch' = batch * kv_heads sequences of `group` query rows, one head.
int gqa_attention_packed(const void* q, const void* cache_k, const void* cache_v, void* out, int batch2, int group, int head_dim,
                         int max_len, int kv_len, int splits, void* workspace, int dtype, cudaStream_t s) {
    return gqa_attention_launch(q, cache_k, cache_v, nullptr, out, batch2, group, 1, 1, head_dim, max_len, kv_len, 0, 0, splits,
                                workspace, dtype, s);
}

int gqa_attention_launch(const void* q, const void* cache_k, const void* cache_v, const uint8_t* keep, void* out, int batch, int q_len,
                         int heads, int kv_heads, int head_dim, int max_len, int kv_len, int past_len, int causal, int splits,
                         void* workspace, int dtype, cudaStream_t s, float* lse) {
    AttnParams p;
    int rc = attention_setup(p, q, out, batch, q_len, heads, kv_heads, head_dim, causal, dtype);
    if (rc != L32_OK) return rc;
    p.lse = lse;
    p.keep = keep;
    p.max_len = max_len; p.kv_len = kv_len; p.past_len = past_len;
    // K / V: one plane per (batch, kv head), cut at kv_len.  Masked keys get P = 0, but 0 * NaN and 0 * Inf are NaN in the
    // P V product: the rows of the last tile beyond kv_len (stale cache capacity, or the next head's keys) must not reach
    // shared memory with whatever they hold, so TMA fills them with zeros.
    const uint64_t planes = static_cast<uint64_t>(batch) * kv_heads, plane_elems = static_cast<uint64_t>(max_len) * head_dim;
    const uint64_t kv_rows = static_cast<uint64_t>(kv_len > 0 ? kv_len : 1);   // kv_len 0: no tile is loaded
    rc = make_tensor_map_3d(&p.map_k, cache_k, planes, kv_rows, head_dim, head_dim, plane_elems, kKvTile, dtype);
    if (rc != L32_OK) return rc;
    rc = make_tensor_map_3d(&p.map_v, cache_v, planes, kv_rows, head_dim, head_dim, plane_elems, kKvTile, dtype);
    if (rc != L32_OK) return rc;
    attention_split(p, splits, kv_len, head_dim, workspace);
    if (lse != nullptr) {
        if (dtype == L32_BF16)
            return head_dim == 128 ? launch_attention<128, __nv_bfloat16, true, false>(p, s) : launch_attention<64, __nv_bfloat16, true, false>(p, s);
        return head_dim == 128 ? launch_attention<128, __half, true, false>(p, s) : launch_attention<64, __half, true, false>(p, s);
    }
    return attention_run<false>(p, head_dim, dtype, s);
}

}  // namespace l32
