// Inline-PTX wrappers shared by the sm_100a kernels: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (alloc / mma / commit / ld), cluster helpers, and the deadlock-guarded barrier wait.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace triad {
namespace ptx {

constexpr unsigned long long kWatchdogNs = 4000000000ull;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank)); return r;
}
__device__ __forceinline__ unsigned long long globaltimer() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_local(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Arrive on a (possibly remote) CTA's barrier.  Default semantics (.release at CTA scope), as CUTLASS's
// ClusterBarrier::arrive: what crosses this barrier is TENSOR memory, ordered by tcgen05.wait::ld +
// tcgen05.fence::before_thread_sync, not global/shared data — the explicit .release.cluster form makes
// ptxas emit MEMBAR.ALL.GPU + ERRBAR per arrive (once per tile and epilogue warp), which stalls the hand-back
// of the accumulator until the warp's outstanding global stores have drained.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// Wait with a deadlock guard: if the barrier does not flip within kWatchdogNs the kernel raises the
// global abort flag and every role drains out, so a pipeline bug costs an error code, not a hung GPU.
static __device__ __noinline__ bool mbar_wait_slow(uint32_t bar, uint32_t parity, int* abort_flag, int code) {
    const unsigned long long t0 = globaltimer();
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++spins & 63u) == 0u) {
            if (*(volatile int*)abort_flag != 0) return false;
            if (globaltimer() - t0 > kWatchdogNs) { atomicCAS(abort_flag, 0, code); return false; }
        }
    }
    return true;
}
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity, int* abort_flag, int code) {
    if (mbar_try_wait(bar, parity)) return true;
    return mbar_wait_slow(bar, parity, abort_flag, code);
}

__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire;" ::: "memory"); }

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int kCtaGroup>
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
    if constexpr (kCtaGroup == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
}
template <int kCtaGroup>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    if constexpr (kCtaGroup == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
    else
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> fp32
template <int kCtaGroup>
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    if constexpr (kCtaGroup == 1) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    }
}
// D[tmem] (+)= A[smem] * B[smem]^T, e4m3 x e4m3 -> fp32 (K = 32 per instruction: the same 32 bytes of a 128-byte
// swizzle row as one bf16 K = 16 step, so the descriptors and their per-step advance are those of umma_bf16)
template <int kCtaGroup>
__device__ __forceinline__ void umma_e4m3(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    if constexpr (kCtaGroup == 1) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    }
}
// One lane of a fully active warp (the lowest): lets a WHOLE warp run a role's loop with warp-uniform control
// flow — descriptors and barrier addresses then live in uniform registers — while only this lane issues the
// single-thread instructions (tcgen05.mma / tcgen05.commit / TMA).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

// arrive on `bar` (same offset in every CTA of the pair) once all previously issued MMAs completed
template <int kCtaGroup>
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    if constexpr (kCtaGroup == 1) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
    } else {
        const uint16_t mask = 3;
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                     ::"r"(bar), "h"(mask) : "memory");
    }
}

template <int kCtaGroup>
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    if constexpr (kCtaGroup == 1) {
        asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                     ::"r"(dst), "l"((uint64_t)map), "r"(bar), "r"(c0), "r"(c1) : "memory");
    } else {
        asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                     ::"r"(dst), "l"((uint64_t)map), "r"(bar), "r"(c0), "r"(c1) : "memory");
    }
}
template <int kCtaGroup>
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
    if constexpr (kCtaGroup == 1) {
        asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                     ::"r"(dst), "l"((uint64_t)map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
    } else {
        asm volatile("cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                     ::"r"(dst), "l"((uint64_t)map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
    }
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// 32 consecutive fp32 columns of this thread's TMEM lane, as raw bits.  The load is ASYNCHRONOUS: the
// registers are defined only after tmem_wait_ld(); callers must not touch `r` (not even to bit-cast it)
// before that and must keep the issue unconditional (a conditional load makes the compiler merge old and
// new values with moves that read the registers too early).  The address is warp-uniform (tcgen05.ld is
// a warp-collective instruction): per-thread column offsets are NOT possible.
__device__ __forceinline__ void tmem_ld32_raw(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 "version 1"): rows are 128 bytes,
// 8-row core groups 1024 bytes apart (SBO); LBO is unused for swizzled K-major layouts.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);          // start address  [0,14)
    d |= (uint64_t)1 << 16;                                // LBO (ignored)  [16,30)
    d |= (uint64_t)(1024 >> 4) << 32;                      // SBO            [32,46)
    d |= (uint64_t)1 << 46;                                // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                                // SWIZZLE_128B
    return d;
}
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, M x N
__device__ __forceinline__ uint32_t make_idesc(int M, int N) {
    uint32_t d = 0;
    d |= 1u << 4;                  // c_format = F32
    d |= 1u << 7;                  // a_format = BF16
    d |= 1u << 10;                 // b_format = BF16
    d |= (uint32_t)(N >> 3) << 17;
    d |= (uint32_t)(M >> 4) << 24;
    return d;
}
// kind::f8f6f4 instruction descriptor: D=f32, A=B=e4m3 (format code 0), both K-major, M x N
__device__ __forceinline__ uint32_t make_idesc_e4m3(int M, int N) {
    uint32_t d = 0;
    d |= 1u << 4;                  // c_format = F32; a_format = b_format = E4M3 (0)
    d |= (uint32_t)(N >> 3) << 17;
    d |= (uint32_t)(M >> 4) << 24;
    return d;
}


}  // namespace ptx
}  // namespace triad
