// K1/K2: fused residual Add-RMSNorm forward and RMSNorm backward for sm_100a.
//
// Replaces the reference kernels rmsnorm_kernel_fused / rmsnorm_backward_kernel
// (reference Tools/rmsnorm/rmsnorm.cuh:13-108 and :110-154) behind the host entry points
// rmsnorm_forward / rmsnorm_backward (reference Tools/rmsnorm/rmsnorm.cu:7-61).
//
// Design (HBM-bound; algorithmic traffic 3*C*2 B per row fwd with residual, 3*C*2 B per row bwd):
//  * forward : one CTA per row, the whole row lives in registers (single read of x and residual),
//              128-bit coalesced loads/stores, fp32 add + sum of squares, warp-shuffle reduction plus
//              one shared-memory hop, rsqrtf; optional h = x + residual output (training) and
//              optional in-place residual update (raw reference ABI).
//  * backward: 512-thread CTAs, each row handled by a group of threads, grid-stride over rows,
//              d_weight accumulated in registers per thread and written once per CTA as an fp32
//              partial row; a second tiny kernel column-reduces the partials (no per-element atomics,
//              deterministic).
#include "l32_internal.cuh"

#include <cstdlib>

namespace l32 {

template <typename T>
L32_DEVICE void unpack8(const uint4& v, float (&f)[8]) {
    float2 a = Pack2<T>::unpack(v.x), b = Pack2<T>::unpack(v.y), c = Pack2<T>::unpack(v.z), d = Pack2<T>::unpack(v.w);
    f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
template <typename T>
L32_DEVICE uint4 pack8(const float (&f)[8]) {
    uint4 v;
    v.x = Pack2<T>::pack(f[0], f[1]); v.y = Pack2<T>::pack(f[2], f[3]);
    v.z = Pack2<T>::pack(f[4], f[5]); v.w = Pack2<T>::pack(f[6], f[7]);
    return v;
}
L32_DEVICE uint4 ld_stream_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
L32_DEVICE uint4 ld_v4(const void* p) {   // plain (coherent) load: used when the buffer is also written
    uint4 r;
    asm volatile("ld.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
L32_DEVICE void st_v4(void* p, const uint4& v) {
    asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
L32_DEVICE float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sum over a group of RT consecutive threads (RT multiple of 32). `slot` = per-group smem scratch
// of RT/32 floats. All threads of the group get the result.
template <int RT>
L32_DEVICE float group_sum(float v, float* slot, int tid_in_group, int bar_id) {
    v = warp_sum(v);
    if constexpr (RT == 32) {
        return v;
    } else {
        constexpr int NW = RT / 32;
        if ((tid_in_group & 31) == 0) slot[tid_in_group >> 5] = v;
        if constexpr (RT == 512) __syncthreads(); else named_bar_sync(bar_id, RT);
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < NW; ++i) s += slot[i];
        return s;
    }
}

// ------------------------------------------------------------------------------------------------
// Forward, fast path: C % 8 == 0, C <= RT * VPT * 8. One CTA (RT threads) per row.
// ------------------------------------------------------------------------------------------------
template <typename T, int RT, int VPT, bool kHasResidual, bool kWriteH>
__global__ void __launch_bounds__(RT) add_rmsnorm_fwd_kernel(
    const T* __restrict__ x, const T* residual, const T* __restrict__ weight, T* __restrict__ y,
    T* h_out, float* __restrict__ rms_out, int64_t rows, int C, float eps) {
    __shared__ float red[16];
    const int tid = threadIdx.x;
    const int nvec = C >> 3;
    const int64_t row = blockIdx.x;
    const size_t base = static_cast<size_t>(row) * C;

    uint4 xv[VPT], rv[VPT], wv[VPT];
    // Programmatic dependent launch: the next kernel of the stream may be scheduled now (it orders itself with
    // griddepcontrol.wait); the weight does not depend on the previous kernel, x / residual do.
    pdl_launch_dependents();
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
        const int v = tid + i * RT;
        if (v < nvec) wv[i] = __ldg(reinterpret_cast<const uint4*>(weight) + v);
    }
    pdl_wait_prior_grid();
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
        const int v = tid + i * RT;
        if (v < nvec) xv[i] = ld_stream_v4(x + base + (size_t)v * 8);
    }
    if constexpr (kHasResidual) {
#pragma unroll
        for (int i = 0; i < VPT; ++i) {
            const int v = tid + i * RT;
            // h_out may alias residual (raw reference ABI updates residual in place): coherent load.
            if (v < nvec) rv[i] = ld_v4(residual + base + (size_t)v * 8);
        }
    }

    float h[VPT][8];
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
        const int v = tid + i * RT;
        if (v < nvec) {
            unpack8<T>(xv[i], h[i]);
            if constexpr (kHasResidual) {
                float r[8];
                unpack8<T>(rv[i], r);
#pragma unroll
                for (int j = 0; j < 8; ++j) h[i][j] += r[j];
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) ss = fmaf(h[i][j], h[i][j], ss);
        }
    }
    if constexpr (kWriteH) {
#pragma unroll
        for (int i = 0; i < VPT; ++i) {
            const int v = tid + i * RT;
            if (v < nvec) st_v4(h_out + base + (size_t)v * 8, pack8<T>(h[i]));
        }
    }
    ss = group_sum<RT>(ss, red, tid, 1);
    const float var = ss / static_cast<float>(C) + eps;
    const float inv = rsqrtf(var);
    if (rms_out != nullptr && tid == 0) rms_out[row] = sqrtf(var);

#pragma unroll
    for (int i = 0; i < VPT; ++i) {
        const int v = tid + i * RT;
        if (v < nvec) {
            float w[8], o[8];
            unpack8<T>(wv[i], w);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = h[i][j] * inv * w[j];
            st_v4(y + base + (size_t)v * 8, pack8<T>(o));
        }
    }
}

// Forward, generic path: any C, scalar accesses, two passes (second pass re-reads, L2-resident).
template <typename T>
__global__ void __launch_bounds__(256) add_rmsnorm_fwd_generic_kernel(
    const T* x, const T* residual, const T* weight, T* y, T* h_out, float* rms_out, int64_t rows, int C, float eps) {
    __shared__ float red[8];
    const int64_t row = blockIdx.x;
    const size_t base = static_cast<size_t>(row) * C;
    float ss = 0.f;
    for (int i = threadIdx.x; i < C; i += 256) {
        float h = static_cast<float>(x[base + i]);
        if (residual != nullptr) h += static_cast<float>(residual[base + i]);
        ss = fmaf(h, h, ss);
    }
    ss = group_sum<256>(ss, red, threadIdx.x, 1);
    const float var = ss / static_cast<float>(C) + eps;
    const float inv = rsqrtf(var);
    if (rms_out != nullptr && threadIdx.x == 0) rms_out[row] = sqrtf(var);
    for (int i = threadIdx.x; i < C; i += 256) {
        float h = static_cast<float>(x[base + i]);
        if (residual != nullptr) h += static_cast<float>(residual[base + i]);
        if (h_out != nullptr) h_out[base + i] = static_cast<T>(h);   // each element touched by one thread only
        y[base + i] = static_cast<T>(h * inv * static_cast<float>(weight[i]));
    }
}

// ------------------------------------------------------------------------------------------------
// Backward, fast path: C % 8 == 0, C <= RT * VPT * 8.  Persistent, one CTA per SM.
//   rstd = 1/rms; xhat = h*rstd; wdy = dy*w; c1 = mean(xhat*wdy)
//   dx = (wdy - xhat*c1) * rstd;   dw[c] = sum_rows dy*xhat
// (same algebra as reference rmsnorm.cuh:124-152 with inp := h, minus its extra 1e-6 and atomics)
//
// HBM-bound (3*C*2 B per row).  A producer warp streams whole rows of dy and h into a shared-memory ring with
// 1-D bulk copies (cp.async.bulk, mbarrier completion), so up to ~190 KB of loads per SM are in flight
// independently of the register file.  512 consumer threads form G = 512/RT row groups that work on alternate
// ring stages; the row reduction is one shuffle tree + one named barrier per row.  d_weight is accumulated in
// registers over all rows of the CTA and leaves as ONE fp32 partial row per CTA (deterministic, no atomics).
// ------------------------------------------------------------------------------------------------
constexpr int kBwdConsumersMax = 512;
constexpr int kBwdStagesWanted = 12;   // ring depth, rounded up to a multiple of the row groups (see launch_bwd_fast)
constexpr int kBwdMaxStages = 16;
constexpr int kBwdBarrierBytes = 2 * kBwdMaxStages * 8;
constexpr int kBwdRedBytes = 2 * 16 * 16 * 4 * 2;   // [parity][group][row of the iteration (<= 2)][warp of the group]

L32_DEVICE void bulk_load_row(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(smem_dst)),
        "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "l"(kEvictFirst)
        : "memory");
}
L32_DEVICE uint4 lds_v4(const void* p) {
    uint4 r;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(smem_u32(p)));
    return r;
}

template <typename T, int RT, int VPT, bool kAddend, int kBwdConsumers, int RPI>
__global__ void __launch_bounds__(kBwdConsumers + 32, 1) rmsnorm_bwd_kernel(
    const T* __restrict__ dy, const T* __restrict__ h, const T* __restrict__ weight, const float* __restrict__ rms,
    const T* __restrict__ addend, T* __restrict__ dx, T* __restrict__ dx_plain, float* __restrict__ dw_partial,
    int64_t rows, int C, int stages) {
    constexpr int G = kBwdConsumers / RT;
    constexpr int kBwdThreads = kBwdConsumers + 32;
    static_assert(kBwdConsumers % RT == 0 && G >= 1 && G <= 14, "row groups");
    extern __shared__ __align__(128) uint8_t bwd_smem[];
    const uint32_t row_bytes = static_cast<uint32_t>(C) * sizeof(T);
    const uint32_t stage_bytes = 2 * row_bytes;
    uint8_t* ring = bwd_smem;
    uint8_t* w_sm = ring + static_cast<size_t>(stages) * stage_bytes;          // gamma, raw T (row_bytes)
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(w_sm + row_bytes);
    uint64_t* empty_bar = full_bar + kBwdMaxStages;
    float* red = reinterpret_cast<float*>(empty_bar + kBwdMaxStages);

    const int tid = threadIdx.x;
    const int nvec = C >> 3;
    const int64_t n_local = rows > blockIdx.x ? (rows - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (tid == 0) {
        for (int i = 0; i < stages; ++i) {
            mbar_init(&full_bar[i], 1);          // the producer's arrive.expect_tx
            mbar_init(&empty_bar[i], RT / 32);   // one arrival per consumer warp of the owning row group
        }
        fence_mbar_init();
    }
    // gamma lives in shared memory (raw 16-bit): the registers it would take (VPT * 8 fp32) are what allows four vectors
    // per thread, i.e. half as many threads per row and twice as many rows in flight per SM
    for (int v = tid; v < nvec; v += kBwdThreads)
        *reinterpret_cast<uint4*>(w_sm + static_cast<size_t>(v) * 16) = __ldg(reinterpret_cast<const uint4*>(weight) + v);
    __syncthreads();
    pdl_launch_dependents();   // the d_weight column reduce may be scheduled; it waits for this grid to finish
    pdl_wait_prior_grid();     // dy / h / rms come from earlier kernels of the stream; dx may still be read by them

    if (tid >= kBwdConsumers) {
        // ------------------------------------------------------------------ producer warp
        if (tid == kBwdConsumers) {
            for (int64_t i = 0; i < n_local; ++i) {
                const int s = static_cast<int>(i % stages);
                const uint32_t use = static_cast<uint32_t>(i / stages);
                if (use > 0) mbar_wait(&empty_bar[s], (use & 1u) ^ 1u);
                const size_t base = static_cast<size_t>(i * gridDim.x + blockIdx.x) * C;
                uint8_t* dst = ring + static_cast<size_t>(s) * stage_bytes;
                mbar_arrive_expect_tx(&full_bar[s], stage_bytes);
                bulk_load_row(dst, dy + base, row_bytes, &full_bar[s]);
                bulk_load_row(dst + row_bytes, h + base, row_bytes, &full_bar[s]);
            }
        }
        return;
    }

    // ---------------------------------------------------------------------- consumers
    // Per element (p = dy*h):  dot' += p*w;  dw += p*rstd;  dx = (dy*w)*rstd - h*c2,  c2 = rstd^3 * dot' / C
    // -- algebraically the formulas above with rstd factored out of the row sums, 6 fp32 ops per element.
    // The row is latency-bound (wait -> reduce -> barrier -> store), so what counts is how many rows an SM has in flight:
    // dy / h stay PACKED in registers between the two passes (unpacking is a shift), which leaves room for VPT = 4.
    const int g = tid / RT;
    const int t = tid % RT;
    constexpr bool kWRegs = (VPT <= 2);   // two vectors per thread: gamma fits into registers next to everything else
    float dwacc[VPT][8], wreg[kWRegs ? VPT : 1][8];
#pragma unroll
    for (int i = 0; i < VPT; ++i) {
#pragma unroll
        for (int j = 0; j < 8; ++j) dwacc[i][j] = 0.f;
        if constexpr (kWRegs) {
            const int v = t + i * RT;
            unpack8<T>(v < nvec ? lds_v4(w_sm + static_cast<size_t>(v) * 16) : make_uint4(0, 0, 0, 0), wreg[i]);
        }
    }
    const float invC = 1.0f / static_cast<float>(C);

    // One iteration of a row group handles RPI rows (i, i + G, ...): their wait -> reduce -> barrier -> store chains are
    // independent, so the warp interleaves them (twice the rows in flight for VPT * 8 more registers per extra row).
    float rms_next[RPI];
#pragma unroll
    for (int r = 0; r < RPI; ++r) {
        const int64_t i = g + static_cast<int64_t>(r) * G;
        rms_next[r] = (i < n_local) ? rms[i * gridDim.x + blockIdx.x] : 1.f;
    }
    for (int64_t i0 = g; i0 < n_local; i0 += static_cast<int64_t>(G) * RPI) {
        uint4 graw[RPI][VPT], hraw[RPI][VPT];
        float rstd[RPI], dot[RPI];
        size_t base[RPI];
        bool live[RPI];
#pragma unroll
        for (int r = 0; r < RPI; ++r) {
            const int64_t i = i0 + static_cast<int64_t>(r) * G;
            live[r] = i < n_local;
            const int64_t row = (live[r] ? i : i0) * gridDim.x + blockIdx.x;
            base[r] = static_cast<size_t>(row) * C;
            rstd[r] = __frcp_rn(rms_next[r]);
            const int64_t inext = i + static_cast<int64_t>(G) * RPI;   // prefetch for the next turn (a global load per row
            if (inext < n_local) rms_next[r] = rms[inext * gridDim.x + blockIdx.x];   // must not sit in the row's chain)
        }
        uint4 av[kAddend ? RPI : 1][kAddend ? VPT : 1];
        if constexpr (kAddend) {
#pragma unroll
            for (int r = 0; r < RPI; ++r)
#pragma unroll
                for (int k = 0; k < VPT; ++k) {
                    const int v = t + k * RT;
                    av[r][k] = make_uint4(0, 0, 0, 0);
                    if (v < nvec && live[r]) av[r][k] = ld_stream_v4(addend + base[r] + (size_t)v * 8);
                }
        }
#pragma unroll
        for (int r = 0; r < RPI; ++r) {
            const int64_t i = i0 + static_cast<int64_t>(r) * G;
#pragma unroll
            for (int k = 0; k < VPT; ++k) {
                graw[r][k] = make_uint4(0, 0, 0, 0);
                hraw[r][k] = make_uint4(0, 0, 0, 0);
            }
            if (live[r]) {
                const int s = static_cast<int>(i % stages);
                const uint32_t use = static_cast<uint32_t>(i / stages);
                mbar_wait(&full_bar[s], use & 1u);
                const uint8_t* src = ring + static_cast<size_t>(s) * stage_bytes;
#pragma unroll
                for (int k = 0; k < VPT; ++k) {
                    const int v = t + k * RT;
                    if (v < nvec) {
                        graw[r][k] = lds_v4(src + static_cast<size_t>(v) * 16);
                        hraw[r][k] = lds_v4(src + row_bytes + static_cast<size_t>(v) * 16);
                    }
                }
                // The refill is a bulk copy (async proxy). Without this fence the arrive does not wait for the loads
                // above, and a late ld.shared could read part of the next row of the stage.
                fence_proxy_async_smem();
                __syncwarp();
                if ((t & 31) == 0) mbar_arrive(&empty_bar[s]);   // stage may be refilled
            }
            dot[r] = 0.f;
        }
#pragma unroll
        for (int k = 0; k < VPT; ++k) {
            const int v = t + k * RT;
            float w[8];
            if constexpr (kWRegs) {
#pragma unroll
                for (int j = 0; j < 8; ++j) w[j] = wreg[k][j];
            } else {
                unpack8<T>(v < nvec ? lds_v4(w_sm + static_cast<size_t>(v) * 16) : make_uint4(0, 0, 0, 0), w);
            }
#pragma unroll
            for (int r = 0; r < RPI; ++r) {
                float gg[8], hh[8];
                unpack8<T>(graw[r][k], gg);
                unpack8<T>(hraw[r][k], hh);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float pr = gg[j] * hh[j];
                    dot[r] = fmaf(pr, w[j], dot[r]);
                    dwacc[k][j] = fmaf(pr, rstd[r], dwacc[k][j]);   // a dead row contributes zeros (graw = hraw = 0)
                }
            }
        }
#pragma unroll
        for (int r = 0; r < RPI; ++r) dot[r] = warp_sum(dot[r]);
        if constexpr (RT > 32) {
            // double-buffered: one barrier per iteration
            float* slot = red + ((static_cast<int>(i0 / (G * RPI)) & 1) * 16 + g) * (16 * RPI);
            if ((t & 31) == 0) {
#pragma unroll
                for (int r = 0; r < RPI; ++r) slot[r * 16 + (t >> 5)] = dot[r];
            }
            named_bar_sync(1 + g, RT);
#pragma unroll
            for (int r = 0; r < RPI; ++r) {
                dot[r] = 0.f;
#pragma unroll
                for (int k = 0; k < RT / 32; ++k) dot[r] += slot[r * 16 + k];
            }
        }
#pragma unroll
        for (int r = 0; r < RPI; ++r) {
            if (!live[r]) continue;
            const float c2 = dot[r] * invC * rstd[r] * rstd[r] * rstd[r];
#pragma unroll
            for (int k = 0; k < VPT; ++k) {
                const int v = t + k * RT;
                if (v < nvec) {
                    float gg[8], hh[8], w[8], o[8];
                    unpack8<T>(graw[r][k], gg);
                    unpack8<T>(hraw[r][k], hh);
                    if constexpr (kWRegs) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) w[j] = wreg[k][j];
                    } else {
                        unpack8<T>(lds_v4(w_sm + static_cast<size_t>(v) * 16), w);
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) o[j] = fmaf(-hh[j], c2, gg[j] * w[j] * rstd[r]);
                    if constexpr (kAddend) {   // dx += addend (a gradient that bypasses the norm, e.g. the block tail's "+ attn_out")
                        if (dx_plain != nullptr) st_v4(dx_plain + base[r] + (size_t)v * 8, pack8<T>(o));   // and the plain one
                        float ad[8];
                        unpack8<T>(av[r][k], ad);
#pragma unroll
                        for (int j = 0; j < 8; ++j) o[j] += ad[j];
                    }
                    st_v4(dx + base[r] + (size_t)v * 8, pack8<T>(o));
                }
            }
        }
    }

    // Fold the G row groups of this CTA through the (now idle) ring, then one fp32 partial row per CTA.
    float* fold = reinterpret_cast<float*>(ring);
    if constexpr (G > 1) {
        named_bar_sync(15, kBwdConsumers);   // every consumer is done reading the ring
        if (g > 0) {
#pragma unroll
            for (int k = 0; k < VPT; ++k) {
                const int v = t + k * RT;
                if (v < nvec) {
                    float4* dst = reinterpret_cast<float4*>(fold + (size_t)(g - 1) * C + (size_t)v * 8);
                    dst[0] = make_float4(dwacc[k][0], dwacc[k][1], dwacc[k][2], dwacc[k][3]);
                    dst[1] = make_float4(dwacc[k][4], dwacc[k][5], dwacc[k][6], dwacc[k][7]);
                }
            }
        }
        named_bar_sync(15, kBwdConsumers);
    }
    if (g == 0) {
#pragma unroll
        for (int k = 0; k < VPT; ++k) {
            const int v = t + k * RT;
            if (v < nvec) {
                float sacc[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) sacc[j] = dwacc[k][j];
                if constexpr (G > 1) {
                    for (int gg = 1; gg < G; ++gg) {
                        const float4* src = reinterpret_cast<const float4*>(fold + (size_t)(gg - 1) * C + (size_t)v * 8);
                        const float4 a = src[0], b = src[1];
                        sacc[0] += a.x; sacc[1] += a.y; sacc[2] += a.z; sacc[3] += a.w;
                        sacc[4] += b.x; sacc[5] += b.y; sacc[6] += b.z; sacc[7] += b.w;
                    }
                }
                float4* dst = reinterpret_cast<float4*>(dw_partial + (size_t)blockIdx.x * C + (size_t)v * 8);
                dst[0] = make_float4(sacc[0], sacc[1], sacc[2], sacc[3]);
                dst[1] = make_float4(sacc[4], sacc[5], sacc[6], sacc[7]);
            }
        }
    }
}

// Backward, generic path: one CTA (256 threads) per grid-stride row, scalar accesses,
// dw partial per CTA accumulated in global memory owned by that CTA (no atomics).
template <typename T>
__global__ void __launch_bounds__(256) rmsnorm_bwd_generic_kernel(
    const T* dy, const T* h, const T* weight, const float* rms, const T* addend, T* dx, T* dx_plain, float* dw_partial,
    int64_t rows, int C) {
    __shared__ float red[8];
    float* my_dw = dw_partial + (size_t)blockIdx.x * C;
    for (int i = threadIdx.x; i < C; i += 256) my_dw[i] = 0.f;
    const float invC = 1.0f / static_cast<float>(C);
    for (int64_t row = blockIdx.x; row < rows; row += gridDim.x) {
        const size_t base = static_cast<size_t>(row) * C;
        const float rstd = 1.0f / rms[row];
        float dot = 0.f;
        for (int i = threadIdx.x; i < C; i += 256) {
            const float gg = static_cast<float>(dy[base + i]);
            const float xh = static_cast<float>(h[base + i]) * rstd;
            dot = fmaf(xh, gg * static_cast<float>(weight[i]), dot);
            my_dw[i] += gg * xh;   // index i is owned by exactly one thread of this CTA
        }
        dot = group_sum<256>(dot, red, threadIdx.x, 1);
        const float c1 = dot * invC;
        for (int i = threadIdx.x; i < C; i += 256) {
            const float gg = static_cast<float>(dy[base + i]);
            const float xh = static_cast<float>(h[base + i]) * rstd;
            float o = (gg * static_cast<float>(weight[i]) - xh * c1) * rstd;
            if (addend != nullptr) {
                if (dx_plain != nullptr) dx_plain[base + i] = static_cast<T>(o);
                o += static_cast<float>(addend[base + i]);
            }
            dx[base + i] = static_cast<T>(o);
        }
        __syncthreads();
    }
}

// dw[c] = sum_p partial[p][c], cast to T.  Latency-bound (the partials are L2-resident), so it is laid out for one
// round of independent loads: CTA = 32 columns x 32 partial groups (1024 threads); a warp reads 32 consecutive
// columns of one partial row (coalesced 128 B) and every thread issues its <= 8 loads back to back.  Fixed
// summation order (deterministic).
constexpr int kDwGroups = 32;
constexpr int kDwMaxPerThread = 8;   // covers up to 256 partial rows (<= 2 x SM count)
template <typename T>
__global__ void __launch_bounds__(32 * kDwGroups) rmsnorm_dw_reduce_kernel(const float* __restrict__ partial,
                                                                           T* __restrict__ dw, int nparts, int C) {
    __shared__ float sm[kDwGroups][33];
    const int cl = threadIdx.x & 31, pg = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + cl;
    pdl_launch_dependents();
    pdl_wait_prior_grid();   // partial rows come from the backward kernel launched just before
    float v[kDwMaxPerThread];
#pragma unroll
    for (int k = 0; k < kDwMaxPerThread; ++k) {
        const int p = pg + k * kDwGroups;
        v[k] = (c < C && p < nparts) ? partial[(size_t)p * C + c] : 0.f;
    }
    float s = ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
    for (int p = pg + kDwMaxPerThread * kDwGroups; p < nparts; p += kDwGroups)   // only for > 256 partial rows
        if (c < C) s += partial[(size_t)p * C + c];
    sm[pg][cl] = s;
    __syncthreads();
    if (pg == 0 && c < C) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < kDwGroups; ++k) t += sm[k][cl];
        dw[c] = static_cast<T>(t);
    }
}

// ------------------------------------------------------------------------------------------------
// Host launchers
// ------------------------------------------------------------------------------------------------
template <typename T, int RT, int VPT>
static cudaError_t launch_fwd_fast(const T* x, const T* residual, const T* weight, T* y, T* h_out, float* rms,
                                   int64_t rows, int C, float eps, cudaStream_t s) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(rows));
    cfg.blockDim = dim3(RT);
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const T* rc = residual;
    cudaError_t e;
    if (residual != nullptr) {
        if (h_out != nullptr) e = cudaLaunchKernelEx(&cfg, add_rmsnorm_fwd_kernel<T, RT, VPT, true, true>, x, rc, weight, y, h_out, rms, rows, C, eps);
        else e = cudaLaunchKernelEx(&cfg, add_rmsnorm_fwd_kernel<T, RT, VPT, true, false>, x, rc, weight, y, h_out, rms, rows, C, eps);
    } else {
        if (h_out != nullptr) e = cudaLaunchKernelEx(&cfg, add_rmsnorm_fwd_kernel<T, RT, VPT, false, true>, x, rc, weight, y, h_out, rms, rows, C, eps);
        else e = cudaLaunchKernelEx(&cfg, add_rmsnorm_fwd_kernel<T, RT, VPT, false, false>, x, rc, weight, y, h_out, rms, rows, C, eps);
    }
    if (e == cudaSuccess) count_launch();
    return e;
}

template <typename T>
static cudaError_t add_rmsnorm_fwd_t(const T* x, const T* residual, const T* weight, T* y, T* h_out, float* rms,
                                     int64_t rows, int C, float eps, cudaStream_t s) {
    if (rows == 0) return cudaSuccess;
    const bool aligned = (C % 8 == 0) && is_aligned16(x) && is_aligned16(residual) && is_aligned16(weight) &&
                         is_aligned16(y) && is_aligned16(h_out);
    if (aligned && C <= 16384) {
        if (C <= 32 * 4 * 8) return launch_fwd_fast<T, 32, 4>(x, residual, weight, y, h_out, rms, rows, C, eps, s);
        if (C <= 64 * 4 * 8) return launch_fwd_fast<T, 64, 4>(x, residual, weight, y, h_out, rms, rows, C, eps, s);
        if (C <= 128 * 4 * 8) return launch_fwd_fast<T, 128, 4>(x, residual, weight, y, h_out, rms, rows, C, eps, s);
        if (C <= 256 * 4 * 8) return launch_fwd_fast<T, 256, 4>(x, residual, weight, y, h_out, rms, rows, C, eps, s);
        return launch_fwd_fast<T, 512, 4>(x, residual, weight, y, h_out, rms, rows, C, eps, s);
    }
    add_rmsnorm_fwd_generic_kernel<T><<<static_cast<unsigned>(rows), 256, 0, s>>>(x, residual, weight, y, h_out, rms, rows, C, eps);
    count_launch();
    return cudaGetLastError();
}

static int bwd_grid(int64_t rows) {
    const int64_t cap = num_sms();
    return static_cast<int>(rows < cap ? (rows < 1 ? 1 : rows) : cap);
}

template <typename T, int RT, int VPT, bool kAddend, int kBwdConsumers, int RPI>
static cudaError_t launch_bwd_fast(const T* dy, const T* h, const T* weight, const float* rms, const T* addend, T* dx,
                                   T* dx_plain, float* partial, int64_t rows, int C, int grid, cudaStream_t s) {
    constexpr int G = kBwdConsumers / RT;
    const size_t row_bytes = static_cast<size_t>(C) * sizeof(T);
    const size_t stage_bytes = 2 * row_bytes;
    int stages = static_cast<int>((200 * 1024 - row_bytes) / stage_bytes);
    // Row i goes to stage i % stages and to row group i % G. With stages a multiple of G every stage has one consumer
    // group, which waits for its uses in order, so the parity wait on full_bar[s] cannot pass on use u - 2's phase while
    // use u - 1 (a bulk copy of another group's row, which need not complete in issue order) is still in flight.
    constexpr int kStagesCap = (kBwdStagesWanted + G - 1) / G * G;   // at least kBwdStagesWanted where the ring fits them
    static_assert(kStagesCap <= kBwdMaxStages, "barrier slots");
    if (stages > kStagesCap) stages = kStagesCap;
    stages -= stages % G;
    // the d_weight fold reuses the ring: (G - 1) fp32 rows must fit into it
    if (stages < 2 || static_cast<size_t>(stages) * stage_bytes < static_cast<size_t>(G - 1) * C * sizeof(float))
        return cudaErrorInvalidConfiguration;
    const size_t smem = stages * stage_bytes + row_bytes + kBwdBarrierBytes + kBwdRedBytes;
    static_assert(RPI >= 1 && RPI <= 2, "rows per iteration");
    auto* k = rmsnorm_bwd_kernel<T, RT, VPT, kAddend, kBwdConsumers, RPI>;
    static bool configured_dev[kMaxDevices] = {};   // per instantiation and device
    bool& configured = configured_dev[current_device_slot()];
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(kBwdConsumers + 32);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, k, dy, h, weight, rms, addend, dx, dx_plain, partial, rows, C, stages);
    if (e == cudaSuccess) count_launch();
    return e;
}

// workspace layout: [grid][C] fp32, grid <= 2 * num_sms
size_t rmsnorm_bwd_workspace_bytes(int64_t rows, int C) {
    (void)rows;
    return static_cast<size_t>(num_sms()) * 2 * static_cast<size_t>(C) * sizeof(float);
}

template <typename T, int RT, int VPT, int NC = kBwdConsumersMax, int RPI = 1>
static cudaError_t launch_bwd_sel(const T* dy, const T* h, const T* weight, const float* rms, const T* addend, T* dx,
                                  T* dx_plain, float* partial, int64_t rows, int C, int grid, cudaStream_t s) {
    if (addend != nullptr) return launch_bwd_fast<T, RT, VPT, true, NC, RPI>(dy, h, weight, rms, addend, dx, dx_plain, partial, rows, C, grid, s);
    return launch_bwd_fast<T, RT, VPT, false, NC, RPI>(dy, h, weight, rms, addend, dx, dx_plain, partial, rows, C, grid, s);
}

template <typename T>
static cudaError_t rmsnorm_bwd_t(const T* dy, const T* h, const T* weight, const float* rms, const T* addend, T* dx,
                                 T* dx_plain, T* dw,
                                 float* workspace, int64_t rows, int C, cudaStream_t s) {
    if (rows == 0) {
        if (dw != nullptr) return cudaMemsetAsync(dw, 0, sizeof(T) * C, s);
        return cudaSuccess;
    }
    const bool aligned = (C % 8 == 0) && is_aligned16(dy) && is_aligned16(h) && is_aligned16(weight) && is_aligned16(dx) &&
                         is_aligned16(addend) && is_aligned16(dx_plain);
    int grid;
    cudaError_t e;
    if (aligned && C <= 16384) {
        grid = bwd_grid(rows);
        // threads per row (RT) x 16-byte vectors per thread (VPT): as few threads per row as the registers allow, so that
        // 512 / RT rows are in flight per SM (the per-row wait -> reduce -> barrier -> store chain is latency-bound)
        static const int variant = [] { const char* v = getenv("L32_RMSBWD_VARIANT"); return v ? atoi(v) : 0; }();   // tuning knob
        if (C <= 64 * 2 * 8) e = launch_bwd_sel<T, 64, 2>(dy, h, weight, rms, addend, dx, dx_plain, workspace, rows, C, grid, s);
        else if (C <= 128 * 2 * 8) e = launch_bwd_sel<T, 128, 2>(dy, h, weight, rms, addend, dx, dx_plain, workspace, rows, C, grid, s);
        else if (C <= 128 * 4 * 8) {
            if (variant == 1) e = launch_bwd_sel<T, 128, 4, 256, 2>(dy, h, weight, rms, addend, dx, dx_plain, workspace, rows, C, grid, s);
            else if (variant == 2) e = launch_bwd_sel<T, 256, 2, 512, 2>(dy, h, weight, rms, addend, dx, dx_plain, workspace, rows, C, grid, s);
            else e = launch_bwd_sel<T, 128, 4, 384, 1>(dy, h, weight, rms, addend, dx, dx_plain, workspace, rows, C, grid, s);
        } else if (C <= 256 * 4 * 8) {
            if (variant == 1) e = launch_bwd_sel<T, 256, 4, 256, 1>(dy, h, weight, rms, addend, dx, dx_plain, workspace, rows, C, grid, s);
            else if (variant == 2) e = launch_bwd_sel<T, 384, 3, 384, 1>(dy, h, weight, rms, addend, dx, dx_plain, workspace, rows, C, grid, s);
            else e = launch_bwd_sel<T, 512, 2, 512, 1>(dy, h, weight, rms, addend, dx, dx_plain, workspace, rows, C, grid, s);
        } else e = launch_bwd_sel<T, 512, 4, 512, 1>(dy, h, weight, rms, addend, dx, dx_plain, workspace, rows, C, grid, s);
    } else {
        grid = 2 * bwd_grid(rows);
        rmsnorm_bwd_generic_kernel<T><<<grid, 256, 0, s>>>(dy, h, weight, rms, addend, dx, dx_plain, workspace, rows, C);
        count_launch();
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return e;
    if (dw != nullptr) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(static_cast<unsigned>((C + 31) / 32));
        cfg.blockDim = dim3(32 * kDwGroups);
        cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        const float* part = workspace;
        e = cudaLaunchKernelEx(&cfg, rmsnorm_dw_reduce_kernel<T>, part, dw, grid, C);
        if (e == cudaSuccess) count_launch();
    }
    return e;
}

cudaError_t add_rmsnorm_fwd(const void* x, const void* residual, const void* weight, void* y, void* h_out, float* rms,
                            int64_t rows, int C, float eps, int dtype, cudaStream_t s) {
    if (dtype == L32_BF16)
        return add_rmsnorm_fwd_t<__nv_bfloat16>((const __nv_bfloat16*)x, (const __nv_bfloat16*)residual, (const __nv_bfloat16*)weight,
                                                (__nv_bfloat16*)y, (__nv_bfloat16*)h_out, rms, rows, C, eps, s);
    return add_rmsnorm_fwd_t<__half>((const __half*)x, (const __half*)residual, (const __half*)weight, (__half*)y,
                                     (__half*)h_out, rms, rows, C, eps, s);
}

cudaError_t rmsnorm_bwd(const void* dy, const void* h, const void* weight, const float* rms, const void* addend, void* dx,
                        void* dx_plain, void* dw, float* workspace, int64_t rows, int C, int dtype, cudaStream_t s) {
    if (addend == nullptr) dx_plain = nullptr;
    if (dtype == L32_BF16)
        return rmsnorm_bwd_t<__nv_bfloat16>((const __nv_bfloat16*)dy, (const __nv_bfloat16*)h, (const __nv_bfloat16*)weight, rms,
                                            (const __nv_bfloat16*)addend, (__nv_bfloat16*)dx, (__nv_bfloat16*)dx_plain,
                                            (__nv_bfloat16*)dw, workspace, rows, C, s);
    return rmsnorm_bwd_t<__half>((const __half*)dy, (const __half*)h, (const __half*)weight, rms, (const __half*)addend,
                                 (__half*)dx, (__half*)dx_plain, (__half*)dw, workspace, rows, C, s);
}

}  // namespace l32
