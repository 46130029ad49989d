// Next-token sampling (K11): greedy / temperature / top-k / top-p over 16-bit logits, drawn by Gumbel-max with a Philox
// stream keyed by the request's seed and counted by the token position (contract: include/l32_ffn.h, l32_sample_tokens).
//
// One thread-block cluster per row; CTA r of the cluster owns the contiguous slice [r * S, r * S + n_r) of the row and
// keeps it in shared memory for every pass (one bulk copy).  A 16-bit logit maps to a 16-bit key whose unsigned order is
// the order of the values (-0 folded onto +0), so both cut-offs are exact two-round radix selects over 256-bin histograms:
//   max pass      : (key, smallest index) of the row maximum         -- greedy, and the softmax shift of top-p
//   top-k rounds  : count histograms of the high byte, then of the low byte inside the chosen bucket, giving v_k
//   top-p rounds  : the same over the survivors' softmax mass exp(z - z_max), in 2^-40 fixed point, giving v_p
//   Gumbel pass   : argmax over kept i of z_i - log(-log u_i), Philox noise drawn only for groups holding a survivor
// Histograms are integers (counts, fixed-point mass), so their sums do not depend on the order of the atomics; the CTAs
// merge them and their per-slice candidates through DSMEM in rank order, so every result is deterministic.
#include "l32_internal.cuh"

#include <type_traits>

namespace l32 {
namespace {

constexpr int kThreads = 512;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxCluster = 8;
constexpr int kSliceTarget = 16384;        // tokens per CTA before the cluster grows (V = 128256: 8 slices of 16032)
constexpr float kMassScale = 1099511627776.0f;   // 2^40: the mass of the row maximum; sums stay below 2^58

struct SampleParams {
    const void* logits;
    const float* temperature;
    const int* top_k;
    const float* top_p;
    const unsigned long long* seed;
    const long long* position;
    long long* tokens;
    float* kept_min;
    int vocab;
    int slice;                              // S: tokens per CTA, a multiple of 8
};

// Shared memory: the slice first (16-byte aligned for the bulk copy), then this block.
struct SampleSmem {
    unsigned long long hist[2][256];        // double-buffered: a round clears the buffer its peers read two rounds ago
    unsigned long long red[kWarps];
    unsigned long long cl_max;              // this CTA's (key, ~index) of the max pass, read by the peers
    unsigned long long cl_cand;             // this CTA's Gumbel candidate
    unsigned int cl_min;                    // this CTA's smallest kept key
    unsigned long long wt[8];               // suffix-scan warp totals
    unsigned long long sel_above;           // mass / count strictly above the selected bin
    int sel_bin;
    unsigned int red32[kWarps];
    uint64_t bar;
};

L32_DEVICE uint32_t key16(uint32_t b) {
    b &= 0xffffu;
    if (b == 0x8000u) b = 0;                // -0 == +0
    return (b & 0x8000u) ? (~b & 0xffffu) : (b | 0x8000u);
}
template <typename T>
L32_DEVICE float key_value(uint32_t key) {
    const uint32_t b = (key & 0x8000u) ? (key & 0x7fffu) : (~key & 0xffffu);
    if constexpr (std::is_same<T, __nv_bfloat16>::value) return __uint_as_float(b << 16);
    else return __half2float(__ushort_as_half(static_cast<unsigned short>(b)));
}
template <typename T>
constexpr uint32_t ninf_key() {
    return std::is_same<T, __nv_bfloat16>::value ? 0x007fu : 0x03ffu;   // key16(0xff80) / key16(0xfc00)
}

L32_DEVICE uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
        const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}

// -log(u) of u = (m + 0.5) 2^-24, m < 2^24.  m + 0.5 has 25 significant bits for u >= 0.5, where fp32 would round the largest
// u to 1 and the noise to +inf; 1 - u = (2^24 - 1 - m + 0.5) 2^-24 is exact there, so log1p takes it.
L32_DEVICE float neg_log_u(uint32_t m) {
    if (m < (1u << 23)) return -logf((static_cast<float>(m) + 0.5f) * 5.9604644775390625e-8f);
    return -log1pf(-(static_cast<float>((1u << 24) - 1u - m) + 0.5f) * 5.9604644775390625e-8f);
}

L32_DEVICE uint32_t float_order(float f) {
    const uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

L32_DEVICE unsigned long long ld_dsmem_u64(const void* local, uint32_t rank) {
    unsigned long long v;
    asm volatile(
        "{\n\t"
        ".reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %1, %2;\n\t"
        "ld.shared::cluster.u64 %0, [ra];\n\t"
        "}\n"
        : "=l"(v)
        : "r"(smem_u32(local)), "r"(rank)
        : "memory");
    return v;
}
L32_DEVICE uint32_t ld_dsmem_u32(const void* local, uint32_t rank) {
    uint32_t v;
    asm volatile(
        "{\n\t"
        ".reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %1, %2;\n\t"
        "ld.shared::cluster.u32 %0, [ra];\n\t"
        "}\n"
        : "=r"(v)
        : "r"(smem_u32(local)), "r"(rank)
        : "memory");
    return v;
}
L32_DEVICE void bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// Block-wide max of a u64 (every thread gets it).
L32_DEVICE unsigned long long block_max_u64(unsigned long long v, SampleSmem& s) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
        v = w > v ? w : v;
    }
    const int warp = threadIdx.x / 32;
    __syncthreads();                        // red[] of a previous reduction has been read
    if (lane_id() == 0) s.red[warp] = v;
    __syncthreads();
    v = s.red[0];
    for (int w = 1; w < kWarps; ++w) v = s.red[w] > v ? s.red[w] : v;
    return v;
}
L32_DEVICE uint32_t block_min_u32(uint32_t v, SampleSmem& s) {
    v = __reduce_min_sync(0xffffffffu, v);
    const int warp = threadIdx.x / 32;
    __syncthreads();
    if (lane_id() == 0) s.red32[warp] = v;
    __syncthreads();
    v = s.red32[0];
    for (int w = 1; w < kWarps; ++w) v = s.red32[w] < v ? s.red32[w] : v;
    return v;
}

// One radix round: histogram of the survivors (key >= lo) whose high byte is `prefix` (round 2; round 1: any), binned by
// the high byte (round 1) or the low byte (round 2), weighted by 1 (counts) or by the fixed-point softmax mass.  Then the
// cluster's histograms are summed and the largest non-empty bin b whose mass at or above it reaches `target` is selected:
// s.sel_bin = b (-1 if none), s.sel_above = the mass strictly above b.  Returns the row total.
template <typename T, bool kMass>
L32_DEVICE double radix_round(const uint16_t* sl, int n, int buf, bool round2, uint32_t prefix, uint32_t lo, float temp,
                              float zmax, double target_frac_or_abs, bool target_is_frac, int csize, SampleSmem& s) {
    unsigned long long* h = s.hist[buf];
    for (int i = threadIdx.x; i < 256; i += kThreads) h[i] = 0;
    __syncthreads();
    const uint32_t lane = lane_id();
    for (int base = 0; base < n; base += kThreads * 8) {
        const int li = base + static_cast<int>(threadIdx.x) * 8;
        const bool valid = li < n;
        uint4 raw = valid ? *reinterpret_cast<const uint4*>(sl + li) : make_uint4(0, 0, 0, 0);
        const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t bits = (w[j >> 1] >> ((j & 1) * 16)) & 0xffffu;
            const uint32_t key = key16(bits);
            const bool in = valid && key >= lo && (!round2 || (key >> 8) == prefix);
            const uint32_t bin = in ? (round2 ? (key & 0xffu) : (key >> 8)) : 0x100u;
            const uint32_t grp = __match_any_sync(0xffffffffu, bin);
            const bool leader = lane == static_cast<uint32_t>(__ffs(grp) - 1);
            if constexpr (kMass) {
                const unsigned long long v =
                    in ? __float2ull_rn(expf(__fdiv_rn(key_value<T>(key), temp) - zmax) * kMassScale) : 0ull;
                const uint32_t hi = __reduce_add_sync(grp, static_cast<uint32_t>(v >> 20));
                const uint32_t lw = __reduce_add_sync(grp, static_cast<uint32_t>(v & 0xfffffu));
                if (leader && bin < 256u) atomicAdd(&h[bin], (static_cast<unsigned long long>(hi) << 20) + lw);
            } else {
                if (leader && bin < 256u) atomicAdd(&h[bin], static_cast<unsigned long long>(__popc(grp)));
            }
        }
    }
    cluster_sync_all();                     // every CTA's histogram complete and visible cluster-wide
    const int t = threadIdx.x;
    unsigned long long mine = 0;
    if (t < 256) {
        for (int c = 0; c < csize; ++c) mine += ld_dsmem_u64(&h[t], static_cast<uint32_t>(c));
    }
    // suffix sums over the 256 bins (threads 0..255 = warps 0..7)
    unsigned long long suf = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long v = __shfl_down_sync(0xffffffffu, suf, o);
        if (static_cast<int>(lane) + o < 32) suf += v;
    }
    if (t < 256 && lane == 0) s.wt[t / 32] = suf;
    if (t == 0) s.sel_bin = -1;
    __syncthreads();
    unsigned long long total = 0;
    for (int w = 0; w < 8; ++w) total += s.wt[w];
    if (t < 256) {
        for (int w = t / 32 + 1; w < 8; ++w) suf += s.wt[w];
        const double target = target_is_frac ? target_frac_or_abs * static_cast<double>(total) : target_frac_or_abs;
        if (mine > 0 && static_cast<double>(suf) >= target) atomicMax(&s.sel_bin, t);
    }
    __syncthreads();
    if (t < 256 && t == s.sel_bin) s.sel_above = suf - mine;
    __syncthreads();
    return static_cast<double>(total);
}

template <typename T>
__global__ void __launch_bounds__(kThreads, 1) sample_tokens_kernel(const __grid_constant__ SampleParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint32_t cs;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(cs));
    const int nclu = static_cast<int>(cs);
    const uint32_t rank = cluster_ctarank();
    const int row = static_cast<int>(blockIdx.x) / nclu;
    const int slice0 = static_cast<int>(rank) * p.slice;
    int n = p.vocab - slice0;
    if (n > p.slice) n = p.slice;
    if (n < 0) n = 0;
    uint16_t* sl = reinterpret_cast<uint16_t*>(smem);
    SampleSmem& s = *reinterpret_cast<SampleSmem*>(smem + static_cast<size_t>(p.slice) * 2);
    const int t = threadIdx.x;

    if (t == 0) {
        mbar_init(&s.bar, 1);
        fence_mbar_init();
    }
    __syncthreads();
    pdl_wait_prior_grid();                  // logits and parameters come from the preceding kernels
    if (t == 0) {
        const uint32_t bytes = static_cast<uint32_t>(n) * 2u;
        mbar_arrive_expect_tx(&s.bar, bytes);
        if (bytes) bulk_load(sl, static_cast<const uint16_t*>(p.logits) + static_cast<size_t>(row) * p.vocab + slice0, bytes, &s.bar);
    }
    const float temp = p.temperature[row];
    const int top_k = p.top_k[row];
    const float top_p = p.top_p[row];
    const unsigned long long seed = p.seed[row];
    const unsigned long long pos = static_cast<unsigned long long>(p.position[row]);
    mbar_wait(&s.bar, 0);
    pdl_launch_dependents();

    const bool greedy = !(temp > 0.0f);
    const bool topk_on = top_k > 0 && top_k < p.vocab;
    const bool topp_on = top_p < 1.0f;
    const uint32_t ninf = ninf_key<T>();

    // ---- max pass (greedy; the shift of the top-p softmax)
    unsigned long long gmax = 0;
    if (greedy || topp_on) {
        unsigned long long best = 0;
        for (int li = t * 8; li < n; li += kThreads * 8) {
            const uint4 raw = *reinterpret_cast<const uint4*>(sl + li);
            const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const uint32_t key = key16((w[j >> 1] >> ((j & 1) * 16)) & 0xffffu);
                const unsigned long long v = (static_cast<unsigned long long>(key) << 32) |
                                             (0xffffffffu - static_cast<uint32_t>(slice0 + li + j));
                best = v > best ? v : best;
            }
        }
        best = block_max_u64(best, s);
        if (t == 0) s.cl_max = best;
        cluster_sync_all();
        for (int c = 0; c < nclu; ++c) {
            const unsigned long long v = ld_dsmem_u64(&s.cl_max, static_cast<uint32_t>(c));
            gmax = v > gmax ? v : gmax;
        }
    }
    if (greedy) {
        if (rank == 0 && t == 0) {
            p.tokens[row] = static_cast<long long>(0xffffffffu - static_cast<uint32_t>(gmax));
            if (p.kept_min != nullptr) p.kept_min[row] = key_value<T>(static_cast<uint32_t>(gmax >> 32));
        }
        cluster_sync_all();                 // no CTA leaves while a peer may still read its cl_max
        return;
    }

    // ---- top-k: v_k = the k-th largest key counted with multiplicity (-inf never counted)
    uint32_t lo = ninf + 1;
    int buf = 0;
    if (topk_on) {
        radix_round<T, false>(sl, n, buf, false, 0, lo, temp, 0.f, static_cast<double>(top_k), false, nclu, s);
        const int b1 = s.sel_bin;
        const double above = static_cast<double>(s.sel_above);
        buf ^= 1;
        if (b1 >= 0) {
            radix_round<T, false>(sl, n, buf, true, static_cast<uint32_t>(b1), lo, temp, 0.f,
                                  static_cast<double>(top_k) - above, false, nclu, s);
            buf ^= 1;
            const uint32_t thr = (static_cast<uint32_t>(b1) << 8) | static_cast<uint32_t>(s.sel_bin);
            lo = thr > lo ? thr : lo;
        }
    }
    // ---- top-p: v_p = the largest survivor value whose survivors at or above it carry >= top_p of their mass
    if (topp_on) {
        const float zmax = __fdiv_rn(key_value<T>(static_cast<uint32_t>(gmax >> 32)), temp);
        const double frac = top_p > 0.0f ? static_cast<double>(top_p) : 0.0;
        const double total = radix_round<T, true>(sl, n, buf, false, 0, lo, temp, zmax, frac, true, nclu, s);
        const int b1 = s.sel_bin;
        const double above = static_cast<double>(s.sel_above);
        buf ^= 1;
        if (b1 >= 0) {
            radix_round<T, true>(sl, n, buf, true, static_cast<uint32_t>(b1), lo, temp, zmax, frac * total - above, false,
                                 nclu, s);
            buf ^= 1;
            const uint32_t thr = (static_cast<uint32_t>(b1) << 8) | static_cast<uint32_t>(s.sel_bin);
            lo = thr > lo ? thr : lo;
        }
    }

    // ---- Gumbel-max over the kept tokens
    const uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
    const uint32_t c2 = static_cast<uint32_t>(pos), c3 = static_cast<uint32_t>(pos >> 32);
    const bool want_min = p.kept_min != nullptr;
    unsigned long long best = 0;
    uint32_t kmin = 0x10000u;
    for (int li = t * 8; li < n; li += kThreads * 8) {
        const uint4 raw = *reinterpret_cast<const uint4*>(sl + li);
        const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int g = 0; g < 2; ++g) {
            uint32_t keys[4];
            bool any = false;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int e = g * 4 + j;
                keys[j] = key16((w[e >> 1] >> ((e & 1) * 16)) & 0xffffu);
                any |= keys[j] >= lo;
            }
            if (!any) continue;
            const uint32_t gi = static_cast<uint32_t>(slice0 + li + g * 4);
            const uint4 r = philox4x32_10(make_uint4(gi >> 2, 0u, c2, c3), k0, k1);
            const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (keys[j] < lo) continue;
                const float score = __fdiv_rn(key_value<T>(keys[j]), temp) - logf(neg_log_u(rr[j] >> 8));
                const unsigned long long v = (static_cast<unsigned long long>(float_order(score)) << 32) | (0xffffffffu - (gi + j));
                best = v > best ? v : best;
                if (want_min) kmin = keys[j] < kmin ? keys[j] : kmin;
            }
        }
    }
    best = block_max_u64(best, s);
    if (want_min) kmin = block_min_u32(kmin, s);
    if (t == 0) {
        s.cl_cand = best;
        s.cl_min = kmin;
    }
    cluster_sync_all();
    if (rank == 0 && t == 0) {
        unsigned long long win = 0;
        uint32_t m = 0x10000u;
        for (int c = 0; c < nclu; ++c) {
            const unsigned long long v = ld_dsmem_u64(&s.cl_cand, static_cast<uint32_t>(c));
            win = v > win ? v : win;
            if (want_min) {
                const uint32_t mc = ld_dsmem_u32(&s.cl_min, static_cast<uint32_t>(c));
                m = mc < m ? mc : m;
            }
        }
        // nothing kept <=> no finite logit: every entry is a maximum, the smallest index is 0
        p.tokens[row] = win == 0 ? 0ll : static_cast<long long>(0xffffffffu - static_cast<uint32_t>(win));
        if (want_min) p.kept_min[row] = m > 0xffffu ? -INFINITY : key_value<T>(m);
    }
    cluster_sync_all();                     // no CTA leaves while rank 0 may still read its candidate
}

template <typename T>
int launch_sample(const SampleParams& p, int batch, int csize, cudaStream_t s) {
    auto* kernel = sample_tokens_kernel<T>;
    const size_t smem = static_cast<size_t>(p.slice) * 2 + sizeof(SampleSmem);
    static size_t configured_dev[kMaxDevices] = {};
    size_t& configured = configured_dev[current_device_slot()];
    if (smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) return static_cast<int>(e);
        configured = smem;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(batch * csize));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = static_cast<unsigned>(csize);
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, p);
    if (e == cudaSuccess) count_launch();
    return static_cast<int>(e);
}

}  // namespace

int sample_tokens(const void* logits, const float* temperature, const int* top_k, const float* top_p,
                  const unsigned long long* seed, const long long* position, long long* tokens_out, float* kept_min_logit,
                  int batch, int vocab, int dtype, cudaStream_t s) {
    int csize = (vocab + kSliceTarget - 1) / kSliceTarget;
    if (csize > kMaxCluster) csize = kMaxCluster;
    int slice = (vocab + csize - 1) / csize;
    slice = (slice + 7) & ~7;
    SampleParams p;
    p.logits = logits;
    p.temperature = temperature;
    p.top_k = top_k;
    p.top_p = top_p;
    p.seed = seed;
    p.position = position;
    p.tokens = tokens_out;
    p.kept_min = kept_min_logit;
    p.vocab = vocab;
    p.slice = slice;
    if (dtype == L32_BF16) return launch_sample<__nv_bfloat16>(p, batch, csize, s);
    return launch_sample<__half>(p, batch, csize, s);
}

}  // namespace l32
