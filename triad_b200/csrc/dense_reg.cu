// Dense "non-negative pressure" regulariser of the reference's loss (SURVEY.md §8 f1):
//
//   l_nonneg = mean over ALL (query token, patch) pairs of clamp(S, lo, 0)^2,   S = T * <q, v>
//   (src/model.py:411-412 with lo = -60 for audio-visual, :525-526 with lo = -20 for text-visual;
//    padded text tokens and zero-padded patches take part, exactly as in the reference.)
//
// Unlike the max-mean path its gradient dL/dS = 2/numel * clamp(S,lo,0) * [lo <= S <= 0] is DENSE
// (about half of all pairs), so the backward is two real GEMMs.  With D = 512 a fused
// flash-attention-style kernel needs the 128 x 512 fp32 dQ (or dV) accumulator = all 512 TMEM
// columns, leaving none for the recomputed S tile; splitting D doubles the S recompute (6 GEMM
// units).  Going through HBM with a bf16 S chunk costs 4 bytes per 1024 flops, so the path is:
// library GEMM (S chunk) -> THIS kernel (in place: S -> dL/d<q,v>, plus the two reductions)
// -> two library GEMMs (dQ += N V, dV = N^T Q), 3 GEMM units in total.  See DESIGN.md §4 K5.
//
// The kernel is a pure HBM stream: one 16-byte load and one 16-byte store per 8 (bf16) or 4
// (fp32) pairs, fp64 block partials reduced in a fixed order by a second launch (deterministic).
#include "common.cuh"

namespace triad {
namespace dense {

constexpr int kThreads = 256;
constexpr int kMaxBlocks = 148 * 8;

template <typename T> struct Pack;
template <> struct Pack<__nv_bfloat16> {
    static constexpr int kElems = 8;
    __device__ static __forceinline__ void load(const void* p, float (&f)[8]) {
        const uint4 u = *reinterpret_cast<const uint4*>(p);
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            f[2 * k] = __uint_as_float(w[k] << 16);
            f[2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u);
        }
    }
    __device__ static __forceinline__ void store(void* p, const float (&f)[8]) {
        uint4 u;
        uint32_t* w = reinterpret_cast<uint32_t*>(&u);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * k], f[2 * k + 1]);
            w[k] = *reinterpret_cast<uint32_t*>(&h);
        }
        *reinterpret_cast<uint4*>(p) = u;
    }
    // the reference's token_sims element: bf16(bf16 GEMM output * fp32 T)  (model.py:387 under autocast)
    __device__ static __forceinline__ float scaled(float raw, float Tv) { return __bfloat162float(__float2bfloat16_rn(raw * Tv)); }
    __device__ static __forceinline__ float scalar(const void* p) { return __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(p)); }
    __device__ static __forceinline__ void put(void* p, float x) { *reinterpret_cast<__nv_bfloat16*>(p) = __float2bfloat16_rn(x); }
};
template <> struct Pack<float> {
    static constexpr int kElems = 4;
    __device__ static __forceinline__ void load(const void* p, float (&f)[4]) {
        const float4 u = *reinterpret_cast<const float4*>(p);
        f[0] = u.x; f[1] = u.y; f[2] = u.z; f[3] = u.w;
    }
    __device__ static __forceinline__ void store(void* p, const float (&f)[4]) {
        *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
    }
    __device__ static __forceinline__ float scaled(float raw, float Tv) { return raw * Tv; }
    __device__ static __forceinline__ float scalar(const void* p) { return *reinterpret_cast<const float*>(p); }
    __device__ static __forceinline__ void put(void* p, float x) { *reinterpret_cast<float*>(p) = x; }
};

// one element: accumulates clamp^2 and dS*raw, returns dL/d(raw) = coef * clamp(S,lo,0) * [S >= lo] * T
// (s2, sT are fp32 sums over ONE 16-byte vector; the caller adds them to its fp64 accumulators once per vector —
//  an fp64 add per element would cost as much as the HBM stream itself)
__device__ __forceinline__ float one(float raw, float Tv, float lo, float coefT, float& s2, float& sT,
                                     float s /* = scaled(raw) */) {
    const float n = fminf(fmaxf(s, lo), 0.f);
    s2 = fmaf(n, n, s2);
    const float pass = (s >= lo) ? n : 0.f;          // clamp's gradient is 1 on [lo, 0] (n == 0 beyond 0 anyway)
    sT = fmaf(pass, raw, sT);                        // dS/dT = <q,v> = raw; the constant coef is applied once per block
    return coefT * pass;
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
nonneg_kernel(void* __restrict__ S, size_t n, const float* __restrict__ Tptr, float lo, float coef, int write_grad,
              double* __restrict__ partials) {
    constexpr int E = Pack<T>::kElems;
    const float Tv = *Tptr;
    const float coefT = coef * Tv;
    double s2 = 0.0, sT = 0.0;
    char* base = reinterpret_cast<char*>(S);
    const size_t nvec = n / E;
    // kUnroll independent 16-byte loads in flight per thread (a pure HBM stream: bytes in flight are the throughput)
    constexpr int kUnroll = 4;
    const size_t stride = (size_t)gridDim.x * kThreads;
    size_t k = (size_t)blockIdx.x * kThreads + threadIdx.x;
    for (; k + (kUnroll - 1) * stride < nvec; k += kUnroll * stride) {
        float f[kUnroll][E];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) Pack<T>::load(base + (k + u * stride) * E * sizeof(T), f[u]);
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            float o[E], a2 = 0.f, aT = 0.f;
#pragma unroll
            for (int c = 0; c < E; ++c) o[c] = one(f[u][c], Tv, lo, coefT, a2, aT, Pack<T>::scaled(f[u][c], Tv));
            s2 += (double)a2; sT += (double)aT;
            if (write_grad) Pack<T>::store(base + (k + u * stride) * E * sizeof(T), o);
        }
    }
    for (; k < nvec; k += stride) {
        float f[E], o[E], a2 = 0.f, aT = 0.f;
        Pack<T>::load(base + k * E * sizeof(T), f);
#pragma unroll
        for (int c = 0; c < E; ++c) o[c] = one(f[c], Tv, lo, coefT, a2, aT, Pack<T>::scaled(f[c], Tv));
        s2 += (double)a2; sT += (double)aT;
        if (write_grad) Pack<T>::store(base + k * E * sizeof(T), o);
    }
    // tail (n % E elements), handled by block 0
    if (blockIdx.x == 0) {
        for (size_t k = nvec * E + threadIdx.x; k < n; k += kThreads) {
            const float raw = Pack<T>::scalar(base + k * sizeof(T));
            float a2 = 0.f, aT = 0.f;
            const float o = one(raw, Tv, lo, coefT, a2, aT, Pack<T>::scaled(raw, Tv));
            s2 += (double)a2; sT += (double)aT;
            if (write_grad) Pack<T>::put(base + k * sizeof(T), o);
        }
    }
    __shared__ double r2[kThreads / 32], rT[kThreads / 32];
    s2 = warp_sum_d(s2);
    sT = warp_sum_d(sT);
    if ((threadIdx.x & 31) == 0) { r2[threadIdx.x >> 5] = s2; rT[threadIdx.x >> 5] = sT; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int w = 0; w < kThreads / 32; ++w) { a += r2[w]; b += rT[w]; }
        partials[2 * blockIdx.x] = a;
        partials[2 * blockIdx.x + 1] = b * (double)coef;
    }
}

// sums[0] += sum clamp^2 ; sums[1] += sum dS * <q,v>   (fixed order over the block partials)
__global__ void nonneg_finish_kernel(const double* __restrict__ partials, int nblocks, double* __restrict__ sums) {
    double a = 0.0, b = 0.0;
    for (int k = threadIdx.x; k < nblocks; k += 32) { a += partials[2 * k]; b += partials[2 * k + 1]; }
    a = warp_sum_d(a);
    b = warp_sum_d(b);
    if (threadIdx.x == 0) { sums[0] += a; sums[1] += b; }
}

}  // namespace dense

int launch_nonneg_finish(const double* partials, int n, double* sums, cudaStream_t st) {
    dense::nonneg_finish_kernel<<<1, 32, 0, st>>>(partials, n, sums);
    TRIAD_LAUNCH_CHECK("nonneg_finish_kernel");
    return TRIAD_OK;
}
}  // namespace triad

using namespace triad;

extern "C" size_t triad_nonneg_workspace_bytes(void) { return (size_t)dense::kMaxBlocks * 2 * sizeof(double); }

extern "C" int triad_nonneg_chunk(void* S, size_t n, int dtype, const float* temperature, float lo, float coef,
                                  int write_grad, double* sums, void* ws, size_t ws_bytes, void* stream) {
    if (!S || !temperature || !sums || !ws) return fail_msg(TRIAD_ERR_BAD_ARG, "nonneg_chunk: null pointer");
    if (dtype != TRIAD_DTYPE_F32 && dtype != TRIAD_DTYPE_BF16) return fail_msg(TRIAD_ERR_BAD_ARG, "nonneg_chunk: dtype");
    if (n == 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "nonneg_chunk: empty chunk");
    if (!(lo < 0.f)) return fail_msg(TRIAD_ERR_BAD_ARG, "nonneg_chunk: lo must be negative");
    if ((uintptr_t)S & 15) return fail_msg(TRIAD_ERR_ALIGNMENT, "nonneg_chunk: S must be 16-byte aligned");
    if (ws_bytes < triad_nonneg_workspace_bytes()) return fail_msg(TRIAD_ERR_WORKSPACE, "nonneg_chunk: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const int E = dtype == TRIAD_DTYPE_BF16 ? 8 : 4;
    size_t want = (n / E + dense::kThreads - 1) / dense::kThreads;
    int blocks = (int)(want < 1 ? 1 : (want > (size_t)dense::kMaxBlocks ? (size_t)dense::kMaxBlocks : want));
    double* partials = (double*)ws;
    if (dtype == TRIAD_DTYPE_BF16)
        dense::nonneg_kernel<__nv_bfloat16><<<blocks, dense::kThreads, 0, st>>>(S, n, temperature, lo, coef, write_grad, partials);
    else
        dense::nonneg_kernel<float><<<blocks, dense::kThreads, 0, st>>>(S, n, temperature, lo, coef, write_grad, partials);
    TRIAD_LAUNCH_CHECK("nonneg_kernel");
    dense::nonneg_finish_kernel<<<1, 32, 0, st>>>(partials, blocks, sums);
    TRIAD_LAUNCH_CHECK("nonneg_finish_kernel");
    return TRIAD_OK;
}

// ---------------------------------------------------------------------------------------------
// Fused variant for bf16 (D % 64 == 0, D <= 512, Nv <= 256, Nv % 8 == 0): the tcgen05 forward kernel itself
// produces N = dL/d<q,v> (maxmean_tc.cu, kEmitN) — no materialised S chunk, no separate elementwise pass.
// ---------------------------------------------------------------------------------------------
extern "C" size_t triad_nonneg_fused_workspace_bytes(void) { return kCtrlBlockBytes + (size_t)kNonnegFusedPartials * 2 * sizeof(double); }

extern "C" int triad_nonneg_fused_chunk(const void* q, const void* v, const float* temperature,
                                        int Bq, int Bv, int Nq, int Nv, int D, float lo, float coef,
                                        void* n_out, long long ldn, int write_grad, double* sums,
                                        void* ws, size_t ws_bytes, void* stream) {
    if (!q || !v || !temperature || !sums || !ws || (write_grad && !n_out)) return fail_msg(TRIAD_ERR_BAD_ARG, "nonneg_fused: null pointer");
    if (Bq <= 0 || Bv <= 0 || Nq <= 0 || Nv <= 0 || D <= 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "nonneg_fused: bad shape");
    if (!(lo < 0.f)) return fail_msg(TRIAD_ERR_BAD_ARG, "nonneg_fused: lo must be negative");
    if ((long long)Bq * Nq > 0x7fffffffLL) return fail_msg(TRIAD_ERR_BAD_SHAPE, "nonneg_fused: Bq*Nq overflows int32");
    if (!tc_emit_supported(Nv, D)) return fail_msg(TRIAD_ERR_UNSUPPORTED, "nonneg_fused: needs D % 64 == 0, D <= 512, Nv <= 256, Nv % 8 == 0");
    if (write_grad && (ldn < (long long)Bv * Nv || ldn % 8 != 0)) return fail_msg(TRIAD_ERR_BAD_SHAPE, "nonneg_fused: ldn");
    if (write_grad && (long long)ldn * 2 >= (1ll << 40)) return fail_msg(TRIAD_ERR_BAD_SHAPE, "nonneg_fused: row pitch beyond the tensor map's 2^40 bytes");
    if (((uintptr_t)q | (uintptr_t)v | (uintptr_t)n_out | (uintptr_t)ws) & 15) return fail_msg(TRIAD_ERR_ALIGNMENT, "nonneg_fused: 16-byte alignment");
    if (ws_bytes < triad_nonneg_fused_workspace_bytes()) return fail_msg(TRIAD_ERR_WORKSPACE, "nonneg_fused: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    TRIAD_CUDA_CHECK(cudaMemsetAsync(ws, 0, kCtrlBlockBytes, st));
    EmitNArgs e{n_out, ldn, lo, coef, write_grad ? 1 : 0, (double*)((char*)ws + kCtrlBlockBytes), sums, 0};
    return launch_maxmean_tc(q, v, nullptr, temperature, 0, Bq * Nq, Bv, Nq, Nv, D, nullptr, nullptr, (int*)ws, 2, 0,
                             nullptr, &e, nullptr, st);
}
