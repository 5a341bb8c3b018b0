// dQ of the max-mean backward, bf16, Nv > 256 (uint16 winners), tiled for on-chip reuse (SURVEY.md §8 a5;
// Nv <= 256 is served by the shared-memory pipeline of bwd_dq_pipe.cu):
//
//   dq[r, :] = T * row_scale[r] * sum_j g[i(r), j] * v[j, idx[j][r], :]
//
// The arithmetic is 2*D MACs per (row, image) pair — 2/Nv of the forward — but every MAC
// needs one bf16 of a GATHERED patch row: M*Bv rows of D*2 bytes (16.8 GB at B=256, 250x256,
// D=512).  Served from L2 that is the whole cost (the generic kernel in maxmean_bwd.cu runs
// at the L2 limit).  This kernel makes the gather an ON-CHIP one:
//
//   * a CTA owns R = 512 consecutive token rows and ONE 64-element (128-byte = one cache line)
//     slice of D, and keeps the 512 x 64 fp32 accumulators in registers (128 KB = half the
//     register file of the SM) for the whole sweep over the images;
//   * for one image the 512 rows pick their winners among only Nv (256) patches, so the CTA
//     touches at most Nv distinct 128-byte lines per image — a 32 KB working set that lives in
//     L1: every line is fetched from L2 once and then re-read by the other rows that chose the
//     same patch (Nv*(1-exp(-R/Nv)) = 221 of 512 reads miss for uniformly random winners, far
//     fewer when the winners concentrate, as they do for trained embeddings);
//   * all CTAs walk the images in the same order, so the lines they miss on are hot in L2.
//
// Thread mapping: warp w owns tile rows [32w, 32w+32); its four 8-lane groups own 8 rows each;
// lane c of a group owns elements [8c, 8c+8) of the slice, so one LDG.128 per lane fetches a
// whole line per group (4 rows per warp instruction, no bank or sector waste).  The winners and
// weights g[i(r), j] of 8 images at a time are staged through shared memory (thread t stages
// tile row t), double buffered, one __syncthreads per 8 images.
#include "common.cuh"

namespace triad {
namespace dq2 {

constexpr int kRows = 512;
constexpr int kThreads = 512;
constexpr int kSlice = 64;      // bf16 elements per CTA slice (128 bytes)
constexpr int kJG = 8;          // images per staging group

__device__ __forceinline__ uint4 ldg_line(const char* p) {
    uint4 u;
    asm("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "l"(p));
    return u;
}

__device__ __forceinline__ void prefetch_l1(const char* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

__device__ __forceinline__ void fma8(float (&a)[8], float w, const uint4& u) {
    a[0] = fmaf(w, __uint_as_float(u.x << 16), a[0]);
    a[1] = fmaf(w, __uint_as_float(u.x & 0xffff0000u), a[1]);
    a[2] = fmaf(w, __uint_as_float(u.y << 16), a[2]);
    a[3] = fmaf(w, __uint_as_float(u.y & 0xffff0000u), a[3]);
    a[4] = fmaf(w, __uint_as_float(u.z << 16), a[4]);
    a[5] = fmaf(w, __uint_as_float(u.z & 0xffff0000u), a[5]);
    a[6] = fmaf(w, __uint_as_float(u.w << 16), a[6]);
    a[7] = fmaf(w, __uint_as_float(u.w & 0xffff0000u), a[7]);
}

constexpr int kStages = 3;      // staging ring: group G computes, G+1 is the prefetch target, G+2 is being loaded

using IdxT = uint16_t;           // winners: this kernel serves Nv > 256
constexpr size_t kSmemBytes = (size_t)kStages * kJG * kRows * (sizeof(IdxT) + sizeof(float));

// kPF = prefetch distance in images: before the rows of image j are gathered, every lane asks for
// the line ONE of its group's rows will need at image j+kPF (prefetch.global.L1), so that by the
// time the LDG.128s are issued they hit L1 instead of waiting ~700 cycles on L2.
constexpr int kPF = 2;

__global__ void __launch_bounds__(kThreads, 1)
dq_tile_kernel(const __nv_bfloat16* __restrict__ v, const IdxT* __restrict__ idx, const float* __restrict__ g,
               const float* __restrict__ row_scale, const float* __restrict__ Tptr,
               int M, int Bv, int Nq, int Nv, int D, int nq_pad, int g_vec, __nv_bfloat16* __restrict__ dq) {
    extern __shared__ __align__(16) unsigned char dq_smem[];
    float (*w_s)[kJG][kRows] = reinterpret_cast<float (*)[kJG][kRows]>(dq_smem);
    IdxT (*idx_s)[kJG][kRows] = reinterpret_cast<IdxT (*)[kJG][kRows]>(dq_smem + (size_t)kStages * kJG * kRows * sizeof(float));

    const int t = threadIdx.x;
    const int slice = blockIdx.x;
    const int row0 = blockIdx.y * kRows;

    // ---- staging role: thread t = tile row t -------------------------------------------------
    const int rs = row0 + t;
    const bool rs_valid = rs < M;
    const int qi = rs_valid ? rs / Nq : 0;
    const size_t pitch = (size_t)(M / Nq) * nq_pad;
    const IdxT* idx_row = idx + (size_t)qi * nq_pad + (rs_valid ? rs - qi * Nq : 0);
    const float* g_row = g + (size_t)qi * Bv;

    // ---- compute role -------------------------------------------------------------------------
    const int warp = t >> 5, lane = t & 31, grp = lane >> 3, c = lane & 7;
    const int rb = warp * 32 + grp * 8;                      // first tile row of this 8-lane group
    const char* vslice = reinterpret_cast<const char*>(v) + (size_t)slice * (kSlice * 2);
    const char* vbase = vslice + c * 16;
    const size_t img_bytes = (size_t)Nv * D * 2;
    const uint32_t row_bytes = (uint32_t)D * 2u;

    float acc[8][8];
#pragma unroll
    for (int k = 0; k < 8; ++k)
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[k][e] = 0.f;

    auto stage = [&](int j0, int st) {
        IdxT pi[kJG];
        float pw[kJG];
        if (rs_valid && g_vec && j0 + kJG <= Bv) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(g_row + j0));
            const float4 b = __ldg(reinterpret_cast<const float4*>(g_row + j0 + 4));
            pw[0] = a.x; pw[1] = a.y; pw[2] = a.z; pw[3] = a.w; pw[4] = b.x; pw[5] = b.y; pw[6] = b.z; pw[7] = b.w;
#pragma unroll
            for (int jj = 0; jj < kJG; ++jj) pi[jj] = __ldcs(idx_row + (size_t)(j0 + jj) * pitch);
        } else {
#pragma unroll
            for (int jj = 0; jj < kJG; ++jj) {
                const int j = j0 + jj;
                const bool ok = rs_valid && j < Bv;
                pi[jj] = ok ? __ldcs(idx_row + (size_t)j * pitch) : (IdxT)0;
                pw[jj] = ok ? __ldg(g_row + j) : 0.f;
            }
        }
#pragma unroll
        for (int jj = 0; jj < kJG; ++jj) { idx_s[st][jj][t] = pi[jj]; w_s[st][jj][t] = pw[jj]; }
    };

    stage(0, 0);
    if (kJG < Bv) stage(kJG, 1);
    __syncthreads();
#pragma unroll
    for (int jp = 0; jp < kPF; ++jp)                          // warm-up: the first kPF images
        if (jp < Bv) prefetch_l1(vslice + (size_t)jp * img_bytes + (uint32_t)idx_s[0][jp][rb + c] * row_bytes);
    int st = 0;
    for (int j0 = 0; j0 < Bv; j0 += kJG) {
        const int jn = min(kJG, Bv - j0);
        const int st1 = (st + 1 == kStages) ? 0 : st + 1;
        const int st2 = (st1 + 1 == kStages) ? 0 : st1 + 1;
#pragma unroll
        for (int jj = 0; jj < kJG; ++jj) {
            if (jj < jn) {
                const int jp = jj + kPF;                                   // compile-time after unrolling
                if (j0 + jp < Bv) {
                    const uint32_t pp = (jp < kJG) ? idx_s[st][jp % kJG][rb + c] : idx_s[st1][jp % kJG][rb + c];
                    prefetch_l1(vslice + (size_t)(j0 + jp) * img_bytes + pp * row_bytes);
                }
                const char* vj = vbase + (size_t)(j0 + jj) * img_bytes;
                const uint4 pk = *reinterpret_cast<const uint4*>(&idx_s[st][jj][rb]);
                const uint32_t p[8] = {pk.x & 0xffffu, pk.x >> 16, pk.y & 0xffffu, pk.y >> 16,
                                       pk.z & 0xffffu, pk.z >> 16, pk.w & 0xffffu, pk.w >> 16};
                const float4 wa = *reinterpret_cast<const float4*>(&w_s[st][jj][rb]);
                const float4 wb = *reinterpret_cast<const float4*>(&w_s[st][jj][rb + 4]);
                const float w[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
                uint4 d[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) d[k] = ldg_line(vj + p[k] * row_bytes);
#pragma unroll
                for (int k = 0; k < 8; ++k) fma8(acc[k], w[k], d[k]);
            }
        }
        if (j0 + 2 * kJG < Bv) stage(j0 + 2 * kJG, st2);
        __syncthreads();
        st = st1;
    }

    const float Tval = *Tptr;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int r = row0 + rb + k;
        if (r < M) {
            const float s = Tval * row_scale[r];
            uint4 o;
            uint32_t* w32 = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                __nv_bfloat162 h = __floats2bfloat162_rn(acc[k][2 * e] * s, acc[k][2 * e + 1] * s);
                w32[e] = *reinterpret_cast<uint32_t*>(&h);
            }
            *reinterpret_cast<uint4*>(dq + (size_t)r * D + slice * kSlice + c * 8) = o;
        }
    }
}

}  // namespace dq2

bool dq_tile_supported(int D, int dtype) { return dtype == TRIAD_DTYPE_BF16 && D % dq2::kSlice == 0; }

int launch_dq_tile(const void* v, const void* idx, const float* g, const float* row_scale, const float* Tp,
                   int M, int Bv, int Nq, int Nv, int D, void* dq, cudaStream_t st) {
    using namespace dq2;
    TRIAD_SET_MAX_SMEM(dq_tile_kernel, kSmemBytes);
    const dim3 grid((unsigned)(D / kSlice), (unsigned)ceil_div(M, kRows));
    const int g_vec = (Bv % 4 == 0) && (((uintptr_t)g & 15) == 0);
    dq_tile_kernel<<<grid, kThreads, kSmemBytes, st>>>((const __nv_bfloat16*)v, (const uint16_t*)idx, g, row_scale, Tp,
                                                      M, Bv, Nq, Nv, D, nq_padded(Nq), g_vec, (__nv_bfloat16*)dq);
    TRIAD_LAUNCH_CHECK("dq_tile_kernel");
    return TRIAD_OK;
}

}  // namespace triad
