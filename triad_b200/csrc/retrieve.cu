// Retrieval helpers: top-k of a score vector, rank of the diagonal (recall@k), and the
// per-pair normalised similarity matrix used by the visualisers.
// Replaces src/retrieval.py:117-144 (numpy argsort per row) and src/model.py:355-368.
#include "common.cuh"

namespace triad {

// order-preserving key: larger score -> larger key; among equal scores the LOWER id is larger,
// i.e. a descending sort of keys is a stable descending argsort of the scores.  -0.0 and +0.0 are
// equal scores, so both get the key of +0.0 (f32_key alone would rank every +0.0 above every -0.0).
__device__ __forceinline__ unsigned long long make_key(float s, uint32_t id) {
    const uint32_t k = s == 0.f ? f32_key(0.f) : f32_key(s);
    return ((unsigned long long)k << 32) | (unsigned long long)(0xffffffffu - id);
}

constexpr int kTopkChunk = 4096;

__global__ void topk_keys_kernel(const float* __restrict__ scores, int n, unsigned long long* __restrict__ keys) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = make_key(scores[i], (uint32_t)i);
}

// each CTA sorts one chunk of kTopkChunk keys (descending, bitonic in shared memory) and keeps
// the first `keep`
__global__ void __launch_bounds__(1024)
topk_chunk_kernel(const unsigned long long* __restrict__ in, int n, int keep, unsigned long long* __restrict__ out) {
    __shared__ unsigned long long s[kTopkChunk];
    const int base = blockIdx.x * kTopkChunk;
    for (int t = threadIdx.x; t < kTopkChunk; t += 1024) s[t] = (base + t < n) ? in[base + t] : 0ull;
    __syncthreads();
    for (int k = 2; k <= kTopkChunk; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = threadIdx.x; t < kTopkChunk; t += 1024) {
                const int ixj = t ^ j;
                if (ixj > t) {
                    const bool desc = ((t & k) == 0);
                    const unsigned long long a = s[t], b = s[ixj];
                    if ((a < b) == desc) { s[t] = b; s[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
    for (int t = threadIdx.x; t < keep; t += 1024) out[(size_t)blockIdx.x * keep + t] = s[t];
}

// the score is read back from the input rather than decoded from the key: a -0.0 keeps its sign bit
__global__ void topk_emit_kernel(const unsigned long long* __restrict__ keys, const float* __restrict__ scores, int k,
                                 float* __restrict__ out_scores, int32_t* __restrict__ out_ids) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k) return;
    const uint32_t id = 0xffffffffu - (uint32_t)(keys[i] & 0xffffffffull);
    out_scores[i] = scores[id];
    out_ids[i] = (int32_t)id;
}

// ranks[i] = #{j: sim[i,j] > sim[i,i]} + #{j < i: sim[i,j] == sim[i,i]}  (position of i in a
// stable descending argsort of row i, retrieval.py:129-131).  NaN sorts last there, so a NaN
// diagonal ranks after every non-NaN entry and after the NaNs to its left: a forward whose
// watchdog fired (NaN scores) must not count as a hit.
__global__ void diag_ranks_kernel(const float* __restrict__ sim, int N, int32_t* __restrict__ ranks) {
    const int i = blockIdx.x;
    const float d = sim[(size_t)i * N + i];
    const bool d_nan = d != d;
    int cnt = 0;
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        const float x = sim[(size_t)i * N + j];
        cnt += d_nan ? (x == x || j < i) : (x > d || (x == d && j < i));
    }
    __shared__ int red[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int a = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) a += red[w];
        ranks[i] = a;
    }
}

// out[b,n1,n2] = T * <f1[b,n1], f2[b,n2]> / (max(|f1|,eps) * max(|f2|,eps))   (F.normalize eps = 1e-12)
__global__ void __launch_bounds__(256)
simmat_kernel(const float* __restrict__ f1, const float* __restrict__ f2, const float* __restrict__ Tptr,
              int N1, int N2, int D, float* __restrict__ out) {
    const int b = blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n1 = blockIdx.x * 8 + warp;
    if (n1 >= N1) return;
    const float* a = f1 + ((size_t)b * N1 + n1) * D;
    float na = 0.f;
    for (int d = lane; d < D; d += 32) na += a[d] * a[d];
    na = fmaxf(sqrtf(warp_sum(na)), 1e-12f);
    const float Tval = *Tptr;
    for (int n2 = blockIdx.y; n2 < N2; n2 += gridDim.y) {
        const float* c = f2 + ((size_t)b * N2 + n2) * D;
        float nb = 0.f, dot = 0.f;
        for (int d = lane; d < D; d += 32) { const float x = c[d]; nb += x * x; dot += (a[d] / na) * x; }
        nb = fmaxf(sqrtf(warp_sum(nb)), 1e-12f);
        dot = warp_sum(dot);
        if (lane == 0) out[((size_t)b * N1 + n1) * N2 + n2] = (dot / nb) * Tval;
    }
}

}  // namespace triad

using namespace triad;

extern "C" size_t triad_topk_workspace_bytes(int n, int k) {
    if (n <= 0 || k <= 0) return 0;
    // two ping-pong key buffers, each large enough for the first level
    const size_t nchunk = ceil_div(n, kTopkChunk);
    const size_t lvl = (size_t)n > nchunk * kTopkChunk ? (size_t)n : nchunk * kTopkChunk;
    return 2 * align_up(lvl * 8, 256);
}

extern "C" int triad_topk(const float* scores, int n, int k, float* out_scores, int32_t* out_ids,
                          void* ws, size_t ws_bytes, void* stream) {
    if (!scores || !out_scores || !out_ids || !ws) return fail_msg(TRIAD_ERR_BAD_ARG, "topk: null pointer");
    if (n <= 0 || k <= 0 || k > n || k > kTopkChunk / 2) return fail_msg(TRIAD_ERR_BAD_SHAPE, "topk: need 1 <= k <= min(n, 2048)");
    if (ws_bytes < triad_topk_workspace_bytes(n, k)) return fail_msg(TRIAD_ERR_WORKSPACE, "topk: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t half = triad_topk_workspace_bytes(n, k) / 2;
    unsigned long long* a = (unsigned long long*)ws;
    unsigned long long* b = (unsigned long long*)((char*)ws + half);
    topk_keys_kernel<<<ceil_div(n, 256), 256, 0, st>>>(scores, n, a);
    TRIAD_LAUNCH_CHECK("topk_keys_kernel");
    int cur = n;
    for (;;) {
        const int nchunk = ceil_div(cur, kTopkChunk);
        const int keep = nchunk == 1 ? (cur < kTopkChunk ? (cur < k ? cur : k) : k) : k;
        topk_chunk_kernel<<<nchunk, 1024, 0, st>>>(a, cur, keep, b);
        TRIAD_LAUNCH_CHECK("topk_chunk_kernel");
        unsigned long long* t = a; a = b; b = t;
        cur = nchunk * keep;
        if (nchunk == 1) break;
    }
    topk_emit_kernel<<<ceil_div(k, 256), 256, 0, st>>>(a, scores, k, out_scores, out_ids);
    TRIAD_LAUNCH_CHECK("topk_emit_kernel");
    return TRIAD_OK;
}

extern "C" int triad_diag_ranks(const float* sim, int N, int32_t* ranks, void* stream) {
    if (!sim || !ranks) return fail_msg(TRIAD_ERR_BAD_ARG, "diag_ranks: null pointer");
    if (N <= 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "diag_ranks: N");
    diag_ranks_kernel<<<N, 256, 0, (cudaStream_t)stream>>>(sim, N, ranks);
    TRIAD_LAUNCH_CHECK("diag_ranks_kernel");
    return TRIAD_OK;
}

extern "C" int triad_similarity_matrix(const float* f1, const float* f2, const float* temperature,
                                       int B, int N1, int N2, int D, float* out, void* stream) {
    if (!f1 || !f2 || !temperature || !out) return fail_msg(TRIAD_ERR_BAD_ARG, "similarity_matrix: null pointer");
    if (B <= 0 || N1 <= 0 || N2 <= 0 || D <= 0 || B > 65535) return fail_msg(TRIAD_ERR_BAD_SHAPE, "similarity_matrix: bad shape");
    dim3 grid(ceil_div(N1, 8), N2 < 64 ? N2 : 64, B);
    simmat_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(f1, f2, temperature, N1, N2, D, out);
    TRIAD_LAUNCH_CHECK("simmat_kernel");
    return TRIAD_OK;
}
