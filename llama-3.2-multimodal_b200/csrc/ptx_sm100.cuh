// Hand-written sm_100a PTX wrappers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM),
// cluster helpers.  No CUTLASS/CuTe dependency.  Compile with
//   -gencode arch=compute_100a,code=sm_100a
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace l32 {

#define L32_DEVICE __device__ __forceinline__

// ------------------------------------------------------------------------------------------------
// misc
// ------------------------------------------------------------------------------------------------
L32_DEVICE uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
L32_DEVICE uint32_t lane_id() {
    uint32_t l;
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
    return l;
}
L32_DEVICE uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
L32_DEVICE uint64_t globaltimer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
L32_DEVICE bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
L32_DEVICE void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
L32_DEVICE void named_bar_sync(uint32_t id, uint32_t nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// Programmatic dependent launch (no-ops when the launch did not opt in).
L32_DEVICE void pdl_wait_prior_grid() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
L32_DEVICE void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------
// cross-SM / cross-GPU flags and peer-memory access (tensor-parallel kernels)
// ------------------------------------------------------------------------------------------------
L32_DEVICE uint32_t ld_acquire_sys_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
L32_DEVICE uint32_t ld_acquire_gpu_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
L32_DEVICE void st_release_sys_u32(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
L32_DEVICE void red_release_gpu_add_u32(uint32_t* p, uint32_t v) {
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// 16-byte load that never hits a (non-coherent) L1 line: peer memory rewritten every step by another GPU.
L32_DEVICE uint4 ld_relaxed_sys_v4(const void* p) {
    uint4 r;
    asm volatile("ld.relaxed.sys.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
    return r;
}
L32_DEVICE void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
// Bounded spin on a flag another SM / GPU will raise: a protocol bug traps after `timeout_ns` instead of hanging the GPU
// for ever.  The bound comes from the host (l32::spin_timeout_ns(): 120 s unless L32_TP_TIMEOUT_S says otherwise) -- long
// enough that a peer rank stalled by lazy initialisation, checkpointing or a data hiccup does not cost the context.
template <bool kSys>
L32_DEVICE void wait_flag_ge(const uint32_t* flag, uint32_t target, uint64_t timeout_ns) {
    uint64_t t0 = 0;
    uint32_t spins = 0;
    while (true) {
        const uint32_t v = kSys ? ld_acquire_sys_u32(flag) : ld_acquire_gpu_u32(flag);
        if (static_cast<int32_t>(v - target) >= 0) return;
        if ((++spins & 0xffu) == 0) {
            const uint64_t now = globaltimer_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > timeout_ns) __trap();
            __nanosleep(64);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------------
L32_DEVICE void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
L32_DEVICE void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
L32_DEVICE void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

L32_DEVICE void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
L32_DEVICE void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
// Arrive on the barrier that lives at the same smem offset in CTA `cta_rank` of this cluster.
// Deliberately the default (.release.cta) form, like CUTLASS' ClusterBarrier::arrive(cta_id): a
// `.release.cluster` arrive compiles to MEMBAR.ALL + ERRBAR, which also waits for this thread's
// outstanding TMA loads and serialised the peer CTA's producer (one k-block per TMA latency, measured).
L32_DEVICE void mbar_arrive_remote(uint64_t* bar, uint32_t cta_rank) {
    asm volatile(
        "{\n\t"
        ".reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(cta_rank)
        : "memory");
}
L32_DEVICE bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps after ~4 s instead of hanging the GPU.
L32_DEVICE void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    uint64_t t0 = 0;
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++spins & 0x3ffu) == 0) {
            uint64_t now = globaltimer_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ull) __trap();
        }
    }
}

// ------------------------------------------------------------------------------------------------
// TMA
// ------------------------------------------------------------------------------------------------
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;

L32_DEVICE void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
// 2-D tile load, completion on this CTA's mbarrier.
L32_DEVICE void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1,
                            uint64_t hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(hint)
        : "memory");
}
// 3-D tile load, completion on this CTA's mbarrier (elements outside the map's extent arrive as zeros).
L32_DEVICE void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1, int32_t c2,
                            uint64_t hint) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "l"(hint)
        : "memory");
}
// 2-D tile load issued by either CTA of a cta_group::2 pair; the transaction bytes are
// credited to the LEADER (even) CTA's mbarrier at the same smem offset.
L32_DEVICE void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1,
                                 uint64_t hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "l"(hint)
        : "memory");
}
// 2-D tile load multicast to every CTA in `mask` (same smem offset, each CTA's own mbarrier).
L32_DEVICE void tma_load_2d_mcast(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1,
                                  uint16_t mask, uint64_t hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster.L2::cache_hint"
        " [%0], [%1, {%4, %5}], [%2], %3, %6;" ::"r"(smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(bar)), "h"(mask), "r"(c0), "r"(c1), "l"(hint)
        : "memory");
}
L32_DEVICE void tma_store_2d(const CUtensorMap* map, const void* smem_src, int32_t c0, int32_t c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}
// The same with an L2 eviction-priority hint (kEvictFirst for streaming outputs that nobody re-reads soon).
L32_DEVICE void tma_store_2d_hint(const CUtensorMap* map, const void* smem_src, int32_t c0, int32_t c1, uint64_t hint) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;" ::"l"(map),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "l"(hint)
                 : "memory");
}
L32_DEVICE void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
L32_DEVICE void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
L32_DEVICE void tma_store_wait_all() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation, MMA, commit, TMEM loads
// ------------------------------------------------------------------------------------------------
template <int kCtaGroup>
L32_DEVICE void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
    if constexpr (kCtaGroup == 1)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
                     "r"(ncols)
                     : "memory");
    else
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
                     "r"(ncols)
                     : "memory");
}
template <int kCtaGroup>
L32_DEVICE void tmem_relinquish() {
    if constexpr (kCtaGroup == 1)
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    else
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCtaGroup>
L32_DEVICE void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    if constexpr (kCtaGroup == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
    else
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
L32_DEVICE void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
L32_DEVICE void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::f16 covers bf16 and fp16 inputs, fp32 accumulate.
template <int kCtaGroup>
L32_DEVICE void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    if constexpr (kCtaGroup == 1)
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
            "}\n" ::"r"(tmem_d),
            "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
            : "memory");
    else
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
            "}\n" ::"r"(tmem_d),
            "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
            : "memory");
}
// Same with the A operand in TENSOR MEMORY (lane = row of D, 16-bit elements packed two per 32-bit column, K-major):
// D[tmem] (+)= A[tmem] * B[smem desc].
L32_DEVICE void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Make an mbarrier track completion of all prior tcgen05.mma of this thread.
// cta_group::2 : arrives on the barrier at this smem offset in BOTH CTAs of the pair.
template <int kCtaGroup>
L32_DEVICE void umma_commit(uint64_t* bar) {
    if constexpr (kCtaGroup == 1) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                         smem_u32(bar))
                     : "memory");
    } else {
        const uint16_t mask = 0b11;
        asm volatile(
            "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                smem_u32(bar)),
            "h"(mask)
            : "memory");
    }
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (one row per thread).
L32_DEVICE void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
L32_DEVICE void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
L32_DEVICE void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
        : "r"(taddr)
        : "memory");
}
L32_DEVICE void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
L32_DEVICE void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
                 "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
L32_DEVICE void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
        "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
// registers -> TMEM: this warp's 32 lanes x 32 consecutive fp32 columns (one row per thread)
L32_DEVICE void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
        "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
        "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]),
        "r"(r[31])
        : "memory");
}
L32_DEVICE void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------
// UMMA descriptors (bit layouts per the PTX ISA "tcgen05 matrix/instruction descriptor" tables)
// ------------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, 128-byte swizzle:
//   [0,14)  start address >> 4        [16,30) leading-dim byte offset >> 4
//   [32,46) stride-dim byte offset >> 4     [46,48) version = 1 (sm_100)
//   [49,52) base offset = 0           [61,64) layout: 2 = SWIZZLE_128B
L32_DEVICE uint64_t make_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFFu);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}
// Instruction descriptor for kind::f16, fp32 accumulate:
//   [4,6) D format (1 = f32)   [7,10) A format (0 = f16, 1 = bf16)   [10,13) B format
//   [15] A major (0 = K, 1 = MN)   [16] B major   [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_f16(bool is_bf16, uint32_t m, uint32_t n, bool a_mn_major,
                                                      bool b_mn_major) {
    return (1u << 4) | ((is_bf16 ? 1u : 0u) << 7) | ((is_bf16 ? 1u : 0u) << 10) |
           ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

// ------------------------------------------------------------------------------------------------
// numeric helpers
// ------------------------------------------------------------------------------------------------
template <typename T>
struct Pack2;
template <>
struct Pack2<__nv_bfloat16> {
    static L32_DEVICE uint32_t pack(float lo, float hi) {
        __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
        return *reinterpret_cast<uint32_t*>(&v);
    }
    static L32_DEVICE float2 unpack(uint32_t u) {
        return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u));
    }
};
template <>
struct Pack2<__half> {
    static L32_DEVICE uint32_t pack(float lo, float hi) {
        __half2 v = __floats2half2_rn(lo, hi);
        return *reinterpret_cast<uint32_t*>(&v);
    }
    static L32_DEVICE float2 unpack(uint32_t u) { return __half22float2(*reinterpret_cast<__half2*>(&u)); }
};

// silu(g) = g * sigmoid(g); fp32, fast exp + fast reciprocal (rel. error ~1e-6, far below bf16 ulp).
L32_DEVICE float sigmoid_f32(float g) { return __frcp_rn(1.0f + __expf(-g)); }
L32_DEVICE float silu_f32(float g) { return g * sigmoid_f32(g); }

}  // namespace l32
