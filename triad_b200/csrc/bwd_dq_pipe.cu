// dQ of the max-mean backward, bf16, Nv <= 256 — the software-pipelined shared-memory gather
// (SURVEY.md §8 a5; autograd backward of src/model.py:387-391):
//
//   dq[r, :] = T * row_scale[r] * sum_j g[i(r), j] * v[j, idx[j][r], :]
//
// A CTA owns 512 token rows x one 64-element slice of D, keeps the 512 x 64 fp32 accumulators in
// registers for the whole sweep over the images, and gathers from a TMA ring of V slices (Nv x 128 B
// per image) in shared memory.  Staging each image's winners and weights through shared memory (the
// round-1 kernel, DESIGN.md K3a) left every warp waiting on a dependent chain per image (barrier wait
// -> staged offsets -> gathered rows -> FMAs) with nothing saturated, and there are no registers for
// more warps.  This kernel removes the chain instead:
//
//   * ROWS ARE ADDRESSED IN THE PADDED INDEX SPACE of the argmax buffer (x = i*nq_pad + a, nq_pad a
//     multiple of 16), so the 8 rows of an 8-lane group always belong to ONE query: their weight
//     g[i, j] is one register per image, and their 8 winners are 8 consecutive bytes of idx[j] — one
//     8-byte load per image, prefetched two images ahead straight into registers.  No shared-memory
//     staging, no staging registers, no __syncthreads.
//   * the byte -> shared-memory address conversion is one IDP.4A per row (dot product of the packed
//     winners with a one-hot 0x80 selector, added to the lane's base): no unpacking, no table.
//   * the gather is SOFTWARE PIPELINED by a quarter image: rows 2k..2k+1 of image j are accumulated
//     while rows 2k+2..2k+3 are in flight, and the first pair of image j+1 (whose barrier is tested in
//     between) is requested before the last pair of image j is consumed — a warp never waits for its
//     own loads.
//   * a dedicated producer warpgroup refills the 7-deep ring (setmaxnreg: 24 registers for it, 112 for
//     the consumers), so no consumer warp blocks on the slowest warp's release of a slot and the warps
//     drift freely.
//   * the pipeline watchdog does not vote: a timed-out wait marks the launch (abort flag) and the
//     kernel finishes with NaNs in dq, so a pipeline bug is LOUD downstream instead of silent.
//
// Masked text queries: the launcher passes a list of the 8-row groups that hold at least one
// kept token (pack.cu); rows with weight 0 inside such a group are swept and scaled by 0.
#include "common.cuh"
#include "ptx.cuh"

namespace triad {
namespace dq4 {
using namespace ptx;

constexpr int kGroupsPerTile = 64;                  // 8-row groups per CTA = 512 padded rows
constexpr int kConsumerWarps = 16;
constexpr int kThreads = (kConsumerWarps + 4) * 32;     // + the producer warpgroup (one lane of it works)
constexpr int kSlice = 64;                          // bf16 elements of D per CTA (one 128-byte line)
constexpr int kMaxNv = 256;
constexpr uint32_t kStageBytes = kMaxNv * kSlice * 2;   // 32 KB per image slice
constexpr int kVS = 7;                              // ring depth (images)
constexpr uint32_t kSmemBytes = kVS * kStageBytes + 16 * kVS + 128;

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 u;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(addr));
    return u;
}
__device__ __forceinline__ uint2 ldg64(const uint8_t* p) {
    uint2 u;
    asm volatile("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(u.x), "=r"(u.y) : "l"(p));
    return u;
}
__device__ __forceinline__ float ldg32f(const float* p) {
    float f;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(f) : "l"(p));
    return f;
}
// acc (lo,hi) += w * (bf16 pair of one 32-bit word): FFMA2, two fp32 FMAs per issue slot
__device__ __forceinline__ void ffma2(float2& acc, float w, uint32_t pair) {
    float2 wv = make_float2(w, w);
    float2 vv = make_float2(__uint_as_float(pair << 16), __uint_as_float(pair & 0xffff0000u));
    unsigned long long a = *reinterpret_cast<unsigned long long*>(&acc);
    const unsigned long long b = *reinterpret_cast<unsigned long long*>(&wv);
    const unsigned long long c = *reinterpret_cast<unsigned long long*>(&vv);
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a) : "l"(b), "l"(c));
    acc = *reinterpret_cast<float2*>(&a);
}
__device__ __forceinline__ void fma_row(float2 (&a)[4], float w, const uint4& u) {
    ffma2(a[0], w, u.x); ffma2(a[1], w, u.y); ffma2(a[2], w, u.z); ffma2(a[3], w, u.w);
}
// shared-memory address of winner byte k (0..3) of `packed`: base + 128 * byte_k
__device__ __forceinline__ uint32_t row_addr(uint32_t packed, int k, uint32_t base) {
    return __dp4a(packed, 0x80u << (8 * k), base);
}

// The guarded wait of ptx.cuh with its slow path INLINED: ptxas cannot allocate registers per role
// (setmaxnreg) in a kernel that contains a function call.
__device__ __forceinline__ bool wait_guarded(uint32_t bar, uint32_t parity, int* abort_flag, int code) {
    if (mbar_try_wait(bar, parity)) return true;
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

struct Params {
    const uint8_t* idx;        // [Bv][Bq][nq_pad]
    const float* g;            // [Bq][Bv]
    const float* row_scale;    // [Bq*Nq]
    const float* T;
    const int* glist;          // padded row index of each active 8-row group, or null (all groups)
    const int* n_groups;       // device count of glist entries (null with glist == null)
    __nv_bfloat16* dq;
    int* abort_flag;
    int Bq, Bv, Nq, Nv, D, nq_pad, gq;     // gq = ceil(Nq / 8) groups per query
};

// 640 threads: 16 consumer warps and the producer warpgroup.  setmaxnreg gives the consumers 112 registers —
// 512*112 + 128*24 is exactly the 640*96 the CTA is launched with.
__global__ void __launch_bounds__(kThreads, 1)
dq_pipe_kernel(const __grid_constant__ CUtensorMap tmap_v, const Params p) {
    const int n_groups = p.glist ? *p.n_groups : p.Bq * p.gq;
    if ((int)blockIdx.y * kGroupsPerTile >= n_groups) return;

    extern __shared__ unsigned char dq4_smem[];
    const uint32_t s0 = smem_u32(dq4_smem);
    uint32_t sbase = (s0 + 127u) & ~127u;
    asm volatile("mov.u32 %0, %0;" : "+r"(sbase));   // opaque: ptxas otherwise re-derives the shared-window base inside the loop
    const uint32_t bar_full = sbase + kVS * kStageBytes;
    const uint32_t bar_empty = bar_full + 8 * kVS;

    uint32_t tid = threadIdx.x;
    asm volatile("mov.u32 %0, %0;" : "+r"(tid));
    const int warp = tid >> 5, lane = tid & 31;
    const int slice = blockIdx.x;
    const int Bv = p.Bv;

    if (tid == 0) {
        prefetch_tmap(&tmap_v);
        for (int s = 0; s < kVS; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, kConsumerWarps); }
        fence_barrier_init();
    }
    __syncthreads();                                   // the only CTA-wide barrier

    const uint32_t stage_tx = (uint32_t)p.Nv * (kSlice * 2);
    if (warp >= kConsumerWarps) {
        // ---- producer warpgroup: hands its registers to the consumers; one lane streams the V slices ----
        asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
        if (warp == kConsumerWarps && lane == 0) {
            int s = 0;
            uint32_t par = 1;                          // parity of the consumers' PREVIOUS release of slot s
            for (int j = 0; j < Bv; ++j) {
                if (j >= kVS && !wait_guarded(bar_empty + 8 * s, par, p.abort_flag, 12)) break;
                mbar_expect_tx(bar_full + 8 * s, stage_tx);
                tma_load_3d<1>(sbase + s * kStageBytes, &tmap_v, bar_full + 8 * s, slice * kSlice, 0, j);
                if (++s == kVS) { s = 0; par ^= 1; }
            }
        }
        return;
    }
    asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");

    // ---- consumer: 8-lane group gi owns 8 consecutive padded rows of one query; lane c owns 8 elements ----
    const int gi = warp * 4 + (lane >> 3), c = lane & 7;
    const int k = blockIdx.y * kGroupsPerTile + gi;
    const bool gvalid = k < n_groups;
    int qi = 0, a0 = 0;
    if (gvalid) {
        if (p.glist) { const int x0 = p.glist[k]; qi = x0 / p.nq_pad; a0 = x0 - qi * p.nq_pad; }
        else { qi = k / p.gq; a0 = (k - qi * p.gq) * 8; }
    }
    const size_t pitch = (size_t)p.Bq * p.nq_pad;
    const uint32_t lane_base = sbase + (uint32_t)c * 16u;
    const bool lane0 = lane == 0;

    float2 acc[8][4];
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[r][e] = make_float2(0.f, 0.f);

    // Winners / weight of images j and j+1 live in two register sets that alternate with the parity of j; the
    // request for image j+2 goes into the set image j has just finished with (winners: right after the last
    // addresses of image j are formed; weight: after the last FMA), so there is no third set and no register moves.
    // Addresses are a uniform 64-bit base (advanced by one image per image) plus a 32-bit per-lane offset.
    const int last = Bv - 1;
    const uint32_t x0 = (uint32_t)(qi * p.nq_pad + a0);    // < 2^31 (checked by the launcher)
    const uint8_t* ibase = p.idx;                          // uniform: winners of image j+2 start at ibase + x0
    const float* gbase = p.g;                              // uniform: weight of image j+2 is gbase[goff]
    const uint32_t goff = (uint32_t)qi * (uint32_t)Bv;
    uint2 W0 = ldg64(ibase + x0), W1 = ldg64(ibase + (size_t)(last < 1 ? last : 1) * pitch + x0);
    float w0 = ldg32f(gbase + goff), w1 = ldg32f(gbase + goff + (last < 1 ? last : 1));
    ibase += 2 * pitch;
    gbase += 2;

    wait_guarded(bar_full, 0, p.abort_flag, 11);
    uint32_t cur = lane_base;                              // this lane's base inside the slot of image j
    uint32_t fbar = bar_full;                              // full barrier of image j's slot (empty = +8*kVS)
    uint32_t par = 0;                                      // parity of image j's slot
    int slot = 0;
    auto advance = [&]() {
        cur += kStageBytes; fbar += 8;
        if (++slot == kVS) { slot = 0; cur = lane_base; fbar = bar_full; par ^= 1u; }
    };

    // Quarter-image pipelining: two 2-row buffers (16 registers; half-image buffers spill at 112 registers).
    uint4 dX[2], dY[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) dX[r] = lds128(row_addr(W0.x, r, lane_base));
// One image.  HAS_NEXT: image j+1 exists (its first pair is requested before the last pair of j is consumed);
// PREFETCH: image j+2 exists.
#define TRIAD_DQ_IMAGE(Wc, wc, Wn, HAS_NEXT, PREFETCH)                                                   \
    {                                                                                                    \
        _Pragma("unroll") for (int r = 0; r < 2; ++r) dY[r] = lds128(row_addr(Wc.x, 2 + r, cur));        \
        _Pragma("unroll") for (int r = 0; r < 2; ++r) fma_row(acc[r], wc, dX[r]);                        \
        _Pragma("unroll") for (int r = 0; r < 2; ++r) dX[r] = lds128(row_addr(Wc.y, r, cur));            \
        _Pragma("unroll") for (int r = 0; r < 2; ++r) fma_row(acc[2 + r], wc, dY[r]);                    \
        _Pragma("unroll") for (int r = 0; r < 2; ++r) dY[r] = lds128(row_addr(Wc.y, 2 + r, cur));        \
        if (PREFETCH) { Wc = ldg64(ibase + x0); ibase += pitch; }                                        \
        _Pragma("unroll") for (int r = 0; r < 2; ++r) fma_row(acc[4 + r], wc, dX[r]);                    \
        const uint32_t ebar = fbar + 8 * kVS;                                                            \
        if (HAS_NEXT) {                                                                                  \
            advance();                                                                                   \
            wait_guarded(fbar, par, p.abort_flag, 11);                                                   \
            _Pragma("unroll") for (int r = 0; r < 2; ++r) dX[r] = lds128(row_addr(Wn.x, r, cur));        \
        }                                                                                                \
        _Pragma("unroll") for (int r = 0; r < 2; ++r) fma_row(acc[6 + r], wc, dY[r]);                    \
        __syncwarp();                                                                                    \
        if (lane0) mbar_arrive_local(ebar);                                                              \
        if (PREFETCH) { wc = ldg32f(gbase + goff); ++gbase; }                                            \
    }
    int j = 0;
    for (; j + 3 <= last; j += 2) {                        // both images of the pair have a successor two ahead
        TRIAD_DQ_IMAGE(W0, w0, W1, true, true)
        TRIAD_DQ_IMAGE(W1, w1, W0, true, true)
    }
    for (; j <= last; ++j) {                               // the last two or three images
        if (j & 1) TRIAD_DQ_IMAGE(W1, w1, W0, j < last, j + 2 <= last)
        else TRIAD_DQ_IMAGE(W0, w0, W1, j < last, j + 2 <= last)
    }
#undef TRIAD_DQ_IMAGE

    // ---- epilogue: scale, round to bf16, one 16-byte store per row and lane (128 B per row and group) ----
    const bool poisoned = *(volatile int*)p.abort_flag != 0;   // a timed-out wait anywhere in the grid: make it loud
    if (gvalid) {
        const float Tval = *p.T;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int a = a0 + r;
            if (a < p.Nq) {
                const size_t row = (size_t)qi * p.Nq + a;
                float sc = Tval * p.row_scale[row];
                if (poisoned) sc = __int_as_float(0x7fc00000);
                uint4 o;
                uint32_t* w32 = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float2 f = acc[r][e];
                    __nv_bfloat162 h = __floats2bfloat162_rn(f.x * sc, f.y * sc);
                    w32[e] = *reinterpret_cast<uint32_t*>(&h);
                }
                *reinterpret_cast<uint4*>(p.dq + row * p.D + slice * kSlice + c * 8) = o;
            }
        }
    }
}

}  // namespace dq4

bool dq_pipe_supported(int Nv, int D, int dtype) {
    return dtype == TRIAD_DTYPE_BF16 && D % dq4::kSlice == 0 && Nv <= dq4::kMaxNv;
}

// glist / n_groups_dev: active 8-row groups (device), or null for "all rows of all queries".
int launch_dq_pipe(const void* v, const void* idx, const float* g, const float* row_scale, const float* Tp,
                   int Bq, int Bv, int Nq, int Nv, int D, void* dq, int* abort_flag,
                   const int* glist, const int* n_groups_dev, cudaStream_t st) {
    using namespace dq4;
    CUtensorMap mv;
    cuuint64_t dims[3] = {(cuuint64_t)D, (cuuint64_t)Nv, (cuuint64_t)Bv};
    cuuint64_t strides[2] = {(cuuint64_t)D * 2, (cuuint64_t)Nv * D * 2};
    cuuint32_t box[3] = {(cuuint32_t)kSlice, (cuuint32_t)Nv, 1};
    int rc = encode_tmap(&mv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, v, 3, dims, strides, box, Swizzle::kNone);
    if (rc) return rc;
    Params p;
    p.idx = (const uint8_t*)idx; p.g = g; p.row_scale = row_scale; p.T = Tp;
    p.glist = glist; p.n_groups = n_groups_dev; p.dq = (__nv_bfloat16*)dq; p.abort_flag = abort_flag;
    p.Bq = Bq; p.Bv = Bv; p.Nq = Nq; p.Nv = Nv; p.D = D; p.nq_pad = nq_padded(Nq); p.gq = ceil_div(Nq, 8);
    const int max_groups = Bq * p.gq;
    if (glist) TRIAD_CUDA_CHECK(cudaMemsetAsync(dq, 0, (size_t)Bq * Nq * D * 2, st));   // rows of inactive groups: zero gradient
    if ((long long)Bq * p.nq_pad > 0x7fffffffLL || (long long)Bq * Bv > 0x7fffffffLL)
        return fail_msg(TRIAD_ERR_BAD_SHAPE, "dq_pipe: Bq*nq_pad and Bq*Bv must fit in 31 bits");
    TRIAD_SET_MAX_SMEM(dq_pipe_kernel, kSmemBytes);
    const dim3 grid((unsigned)(D / kSlice), (unsigned)ceil_div(max_groups, kGroupsPerTile));
    dq_pipe_kernel<<<grid, kThreads, kSmemBytes, st>>>(mv, p);
    TRIAD_LAUNCH_CHECK("dq_pipe_kernel");
    return TRIAD_OK;
}

}  // namespace triad
