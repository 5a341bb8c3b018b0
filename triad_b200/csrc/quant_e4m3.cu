// Per-row e4m3 quantizer of the fp8 retrieval gallery (and of the query that is scored against it).
//
// For a row x[0..D) (fp32, or bf16 widened exactly):
//   amax = max_k |x_k|,  s = fp32(amax / 448)  (IEEE division, round to nearest),
//   c_k  = e4m3_rn_satfinite(fp32(x_k / s))  if s > 0,   c_k = 0  if s == 0 (an all-zero row, or amax so small that
//   s underflows).
// A row holding an inf or a NaN gets s = NaN (and codes 0), so every score that reads the row is NaN, never finite.
// This is torch.clamp(x / s, -448, 448).to(torch.float8_e4m3fn) on the CPU for every finite row.  The library is
// built without --use_fast_math, so the divisions are IEEE and subnormals are kept.
//
// One warp per row, lane l owns elements [16 l, 16 l + 16): D <= 512, codes leave in one 16-byte store per lane.  The
// kernel is an HBM stream (read 2 or 4 bytes, write 1 byte per element).
#include "common.cuh"

#include <float.h>

namespace triad {

namespace {

__device__ __forceinline__ float fmax_nan_q(float a, float b) {
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}

// two fp32 -> two e4m3 bytes, `lo` in the low byte (the element at the lower address)
__device__ __forceinline__ uint32_t cvt_e4m3x2(float lo, float hi) {
    uint16_t h;
    asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(h) : "f"(hi), "f"(lo));
    return (uint32_t)h;
}

__device__ __forceinline__ void load16(const float* p, float (&v)[16]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(p) + i);
        v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
    }
}
__device__ __forceinline__ void load16(const __nv_bfloat16* p, float (&v)[16]) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const uint4 t = __ldg(reinterpret_cast<const uint4*>(p) + i);
        const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            v[8 * i + 2 * k] = __uint_as_float(w[k] << 16);
            v[8 * i + 2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u);
        }
    }
}

// kGather: output row r quantizes source row rowmap[r], or a zero row (scale 0, codes 0) where rowmap[r] is negative or
// not below src_rows (the ragged gallery's pack: a slot's rows after its last caption)
template <typename T, bool kGather>
__global__ void __launch_bounds__(256)
quantize_e4m3_kernel(const T* __restrict__ x, long long rows, int D, uint8_t* __restrict__ codes, float* __restrict__ scales,
                     const int* __restrict__ rowmap, long long src_rows) {
    const int lane = threadIdx.x & 31;
    const bool act = lane < D / 16;
    const long long step = (long long)gridDim.x * 8;
    for (long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += step) {
        float v[16];
        bool ld = act;
        long long src = r;
        if constexpr (kGather) {
            const int m = __ldg(rowmap + r);
            ld = act && m >= 0 && m < src_rows;
            src = m;
        }
        if (ld) load16(x + src * D + lane * 16, v);
        else {
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = 0.f;
        }
        float am = 0.f;
#pragma unroll
        for (int e = 0; e < 16; ++e) am = fmax_nan_q(am, fabsf(v[e]));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) am = fmax_nan_q(am, __shfl_xor_sync(0xffffffffu, am, o));
        float s = am / 448.0f;
        if (!(am <= FLT_MAX)) s = __int_as_float(0x7fc00000);          // inf or NaN in the row
        if (act) {
            uint32_t w[4] = {0u, 0u, 0u, 0u};
            if (s > 0.f) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    w[k] = cvt_e4m3x2(v[4 * k] / s, v[4 * k + 1] / s) | (cvt_e4m3x2(v[4 * k + 2] / s, v[4 * k + 3] / s) << 16);
            }
            *reinterpret_cast<uint4*>(codes + r * D + lane * 16) = make_uint4(w[0], w[1], w[2], w[3]);
        }
        if (lane == 0) scales[r] = s;
    }
}

}  // namespace

int launch_quantize_e4m3(const void* x, int dtype, long long rows, int D, void* codes, float* scales, cudaStream_t st,
                         const int* rowmap, long long src_rows) {
    long long blocks = (rows + 7) / 8;
    if (blocks > (1ll << 20)) blocks = 1ll << 20;                  // grid-stride beyond 8 M rows
    const unsigned g = (unsigned)blocks;
    uint8_t* c = (uint8_t*)codes;
    if (dtype == TRIAD_DTYPE_BF16) {
        const __nv_bfloat16* xb = (const __nv_bfloat16*)x;
        if (rowmap) quantize_e4m3_kernel<__nv_bfloat16, true><<<g, 256, 0, st>>>(xb, rows, D, c, scales, rowmap, src_rows);
        else quantize_e4m3_kernel<__nv_bfloat16, false><<<g, 256, 0, st>>>(xb, rows, D, c, scales, nullptr, 0);
    } else {
        const float* xf = (const float*)x;
        if (rowmap) quantize_e4m3_kernel<float, true><<<g, 256, 0, st>>>(xf, rows, D, c, scales, rowmap, src_rows);
        else quantize_e4m3_kernel<float, false><<<g, 256, 0, st>>>(xf, rows, D, c, scales, nullptr, 0);
    }
    TRIAD_LAUNCH_CHECK("quantize_e4m3_kernel");
    return TRIAD_OK;
}

}  // namespace triad

using namespace triad;

extern "C" int triad_quantize_e4m3(const void* x, int dtype, long long rows, int D, void* codes, float* scales, void* stream) {
    if (!x || !codes || !scales) return fail_msg(TRIAD_ERR_BAD_ARG, "quantize_e4m3: null pointer");
    if (dtype != TRIAD_DTYPE_F32 && dtype != TRIAD_DTYPE_BF16) return fail_msg(TRIAD_ERR_BAD_ARG, "quantize_e4m3: dtype");
    if (rows <= 0 || D <= 0 || D % 16 != 0 || D > 512) return fail_msg(TRIAD_ERR_BAD_SHAPE, "quantize_e4m3: need rows >= 1, D % 16 == 0, D <= 512");
    if ((((uintptr_t)x | (uintptr_t)codes) & 15) || ((uintptr_t)scales & 3))
        return fail_msg(TRIAD_ERR_ALIGNMENT, "quantize_e4m3: x and codes 16-byte aligned, scales 4-byte aligned");
    return launch_quantize_e4m3(x, dtype, rows, D, codes, scales, (cudaStream_t)stream);
}
