// Symmetric InfoNCE on a row block of the B x B clip matrix: row / column log-sum-exp via
// warp-shuffle reductions, closed-form gradient, and the reference's similarity statistics.
// Replaces src/model.py:435-459 (AV) and :553-578 (TV).  Row-sharding aware: a rank owns rows
// [row0,row0+rows) and exchanges only 2*B floats of column partials.
//
// Everything is deterministic: per-block partials are combined in a fixed order (no float
// atomics).
#include "common.cuh"

namespace triad {

constexpr int kNceRowsPerBlock = 32;    // rows handled by one CTA of the partial / finish kernels
constexpr int kNceThreads = 256;

struct NceWs {
    float* chunk_part;   // [nblk][2][B]
    float* col_lse;      // [B]
    double* blk_sums;    // [nblk][8]
};

static inline int nce_blocks(int rows) { return ceil_div(rows, kNceRowsPerBlock); }

static inline size_t nce_ws_bytes(int rows, int B) {
    const size_t nblk = nce_blocks(rows);
    return align_up(nblk * 2 * (size_t)B * 4, 256) + align_up((size_t)B * 4, 256) + align_up(nblk * 8 * 8, 256);
}
static inline NceWs nce_ws_carve(void* ws, int rows, int B) {
    const size_t nblk = nce_blocks(rows);
    char* p = (char*)ws;
    NceWs w;
    w.chunk_part = (float*)p; p += align_up(nblk * 2 * (size_t)B * 4, 256);
    w.col_lse = (float*)p;    p += align_up((size_t)B * 4, 256);
    w.blk_sums = (double*)p;
    return w;
}

// The hardest negative (the max of the off-diagonal entries) propagates NaN like the reference's torch max: fmaxf /
// fmax return the other operand, which would report a finite hardest negative next to a NaN loss.
__device__ __forceinline__ float nan_max(float a, float b) { return (a != a || b != b) ? a + b : fmaxf(a, b); }
__device__ __forceinline__ double nan_max(double a, double b) { return (a != a || b != b) ? a + b : fmax(a, b); }
__device__ __forceinline__ float warp_nan_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = nan_max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- step 1a: one CTA = 32 rows; warps reduce rows, then threads own columns ---------------
__global__ void __launch_bounds__(kNceThreads)
nce_partial_kernel(const float* __restrict__ clip, int rows, int B, int rpb,
                   float* __restrict__ row_lse, float* __restrict__ chunk_part, unsigned int* __restrict__ ticket) {
    if (ticket && blockIdx.x == 0 && threadIdx.x == 0) *ticket = 0u;     // the fused head's "last block" ticket
    const int blk = blockIdx.x;
    const int r0 = blk * rpb;
    const int nr = min(rpb, rows - r0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // row log-sum-exp: 8 warps x 4 rows each, two shuffle reductions per row
    for (int rr = warp; rr < nr; rr += kNceThreads / 32) {
        const float* x = clip + (size_t)(r0 + rr) * B;
        float m = -INFINITY;
        for (int c = lane; c < B; c += 32) m = fmaxf(m, x[c]);
        m = warp_max(m);
        float s = 0.f;
        for (int c = lane; c < B; c += 32) s += expf(x[c] - m);
        s = warp_sum(s);
        if (lane == 0) row_lse[r0 + rr] = m + logf(s);
    }
    // per-column (max, sum exp) over this block's rows; consecutive threads read consecutive columns
    for (int c = threadIdx.x; c < B; c += kNceThreads) {
        float m = -INFINITY;
        for (int rr = 0; rr < nr; ++rr) m = fmaxf(m, clip[(size_t)(r0 + rr) * B + c]);
        float s = 0.f;
        for (int rr = 0; rr < nr; ++rr) s += expf(clip[(size_t)(r0 + rr) * B + c] - m);
        chunk_part[((size_t)blk * 2 + 0) * B + c] = m;
        chunk_part[((size_t)blk * 2 + 1) * B + c] = s;
    }
}

// ---- combine [n][2][B] (max, sumexp) partials over n in fixed order ---------------------
// out_mode 0: write (max,sum) as [2][B];  out_mode 1: write lse = max + log(sum) as [B]
__global__ void nce_combine_kernel(const float* __restrict__ parts, int n, int B, int out_mode,
                                   float* __restrict__ out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= B) return;
    float m = -INFINITY;
    for (int k = 0; k < n; ++k) m = fmaxf(m, parts[((size_t)k * 2 + 0) * B + c]);
    float s = 0.f;
    for (int k = 0; k < n; ++k)
        s += parts[((size_t)k * 2 + 1) * B + c] * expf(parts[((size_t)k * 2 + 0) * B + c] - m);
    if (out_mode == 0) { out[c] = m; out[(size_t)B + c] = s; }
    else out[c] = m + logf(s);
}

// ---- step 2: gradient + loss terms + statistics -------------------------------------------
__global__ void __launch_bounds__(kNceThreads)
nce_finish_kernel(const float* __restrict__ clip, int rows, int B, int row0,
                  const float* __restrict__ row_lse, const float* __restrict__ col_lse,
                  float grad_scale, float* __restrict__ g, double* __restrict__ blk_sums) {
    const int blk = blockIdx.x;
    const int r0 = blk * kNceRowsPerBlock;
    const int nr = min(kNceRowsPerBlock, rows - r0);
    const float inv2B = 0.5f / (float)B;

    double loss = 0.0, sd = 0.0, sd2 = 0.0, so = 0.0, so2 = 0.0, gc = 0.0;
    float mo = -INFINITY;
    for (int rr = 0; rr < nr; ++rr) {
        const int i = r0 + rr;
        const int diag = row0 + i;
        const float rl = row_lse[i];
        const float* x = clip + (size_t)i * B;
        float* gi = g + (size_t)i * B;
        for (int c = threadIdx.x; c < B; c += kNceThreads) {
            const float xc = x[c];
            const float cl = col_lse[c];
            float gv = expf(xc - rl) + expf(xc - cl);
            if (c == diag) {
                gv -= 2.f;
                loss += (double)(rl - xc) + (double)(cl - xc);
                sd += xc; sd2 += (double)xc * xc;
            } else {
                so += xc; so2 += (double)xc * xc; mo = nan_max(mo, xc);
            }
            gv *= inv2B;
            gc += (double)gv * xc;
            gi[c] = gv * grad_scale;
        }
    }
    __shared__ double red[kNceThreads / 32][7];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    loss = warp_sum_d(loss); sd = warp_sum_d(sd); sd2 = warp_sum_d(sd2);
    so = warp_sum_d(so); so2 = warp_sum_d(so2); gc = warp_sum_d(gc); mo = warp_nan_max(mo);
    if (lane == 0) {
        red[warp][0] = loss; red[warp][1] = sd; red[warp][2] = sd2; red[warp][3] = so;
        red[warp][4] = so2; red[warp][5] = (double)mo; red[warp][6] = gc;
    }
    __syncthreads();
    if (threadIdx.x < 7) {
        const int k = threadIdx.x;
        double a = red[0][k];
        for (int w = 1; w < kNceThreads / 32; ++w) a = (k == 5) ? nan_max(a, red[w][k]) : a + red[w][k];
        blk_sums[(size_t)blk * 8 + k] = a;
    }
}

__global__ void nce_final_reduce_kernel(const double* __restrict__ blk_sums, int nblk,
                                        double* __restrict__ sums) {
    const int k = threadIdx.x;
    if (k >= 8) return;
    if (k == 7) { sums[7] = 0.0; return; }
    double a = blk_sums[k];
    for (int b = 1; b < nblk; ++b) a = (k == 5) ? nan_max(a, blk_sums[(size_t)b * 8 + k]) : a + blk_sums[(size_t)b * 8 + k];
    sums[k] = a;
}


// ---------------------------------------------------------------------------------------------
// Fused single-device head (the whole B x B matrix on this GPU): two launches instead of five
// kernels plus the torch glue around them (loss division, temperature calibration, casts).
//   launch 1: nce_partial_kernel (row LSE + per-block column partials); block 0 also zeroes the ticket.
//   launch 2: nce_head_kernel — every CTA combines the column partials of ALL blocks itself (nblk <= 64:
//             nblk*B floats out of L2), then gradient + statistics for its 32 rows; the last CTA to take a
//             ticket reduces the per-block sums in block order (deterministic) and writes the scalars:
//               out[0] = contrastive loss = sums[0] / (2B)                      (model.py:453-459)
//               out[1] = 20 * relu(-log T)^2        (the l_cal term, model.py:420-427; 0 without T)
//               out[2] = out[0] + out[1]
//               out[3] = d out[1] / dT
// ---------------------------------------------------------------------------------------------
constexpr int kHeadMaxBlocks = 64;

__global__ void __launch_bounds__(kNceThreads)
nce_head_kernel(const float* __restrict__ clip, int B, int rpb, const float* __restrict__ row_lse,
                const float* __restrict__ chunk_part, int nblk, const float* __restrict__ Tptr,
                float* __restrict__ g, double* __restrict__ blk_sums, unsigned int* __restrict__ ticket,
                double* __restrict__ sums, float* __restrict__ out) {
    extern __shared__ float col_lse_s[];                 // [B]
    for (int c = threadIdx.x; c < B; c += kNceThreads) {
        float m = -INFINITY;
        for (int k = 0; k < nblk; ++k) m = fmaxf(m, chunk_part[((size_t)k * 2 + 0) * B + c]);
        float s = 0.f;
        for (int k = 0; k < nblk; ++k)
            s += chunk_part[((size_t)k * 2 + 1) * B + c] * expf(chunk_part[((size_t)k * 2 + 0) * B + c] - m);
        col_lse_s[c] = m + logf(s);
    }
    __syncthreads();

    const int blk = blockIdx.x;
    const int r0 = blk * rpb;
    const int nr = min(rpb, B - r0);
    const float inv2B = 0.5f / (float)B;
    double loss = 0.0, sd = 0.0, sd2 = 0.0, so = 0.0, so2 = 0.0, gc = 0.0;
    float mo = -INFINITY;
    for (int rr = 0; rr < nr; ++rr) {
        const int i = r0 + rr;
        const float rl = row_lse[i];
        const float* x = clip + (size_t)i * B;
        float* gi = g + (size_t)i * B;
        for (int c = threadIdx.x; c < B; c += kNceThreads) {
            const float xc = x[c];
            const float cl = col_lse_s[c];
            float gv = expf(xc - rl) + expf(xc - cl);
            if (c == i) {
                gv -= 2.f;
                loss += (double)(rl - xc) + (double)(cl - xc);
                sd += xc; sd2 += (double)xc * xc;
            } else {
                so += xc; so2 += (double)xc * xc; mo = nan_max(mo, xc);
            }
            gv *= inv2B;
            gc += (double)gv * xc;
            gi[c] = gv;
        }
    }
    __shared__ double red[kNceThreads / 32][7];
    __shared__ bool is_last;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    loss = warp_sum_d(loss); sd = warp_sum_d(sd); sd2 = warp_sum_d(sd2);
    so = warp_sum_d(so); so2 = warp_sum_d(so2); gc = warp_sum_d(gc); mo = warp_nan_max(mo);
    if (lane == 0) {
        red[warp][0] = loss; red[warp][1] = sd; red[warp][2] = sd2; red[warp][3] = so;
        red[warp][4] = so2; red[warp][5] = (double)mo; red[warp][6] = gc;
    }
    __syncthreads();
    if (threadIdx.x < 7) {
        const int k = threadIdx.x;
        double a = red[0][k];
        for (int w = 1; w < kNceThreads / 32; ++w) a = (k == 5) ? nan_max(a, red[w][k]) : a + red[w][k];
        blk_sums[(size_t)blk * 8 + k] = a;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();                                  // this block's sums are visible before its ticket
        is_last = atomicAdd(ticket, 1u) == (unsigned)gridDim.x - 1u;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    if (threadIdx.x < 8) {
        const int k = threadIdx.x;
        double a = 0.0;
        if (k < 7) {
            a = ((volatile double*)blk_sums)[k];
            for (int b = 1; b < (int)gridDim.x; ++b) {
                const double t = ((volatile double*)blk_sums)[(size_t)b * 8 + k];
                a = (k == 5) ? nan_max(a, t) : a + t;
            }
        }
        sums[k] = a;
        if (k == 0) {
            const float con = (float)(a / (2.0 * (double)B));
            float cal = 0.f, dcal = 0.f;
            if (Tptr) {
                const float T = *Tptr;
                const float nl = -logf(T);
                if (nl > 0.f) { cal = 20.f * nl * nl; dcal = -40.f * nl / T; }
            }
            out[0] = con; out[1] = cal; out[2] = con + cal; out[3] = dcal;
        }
    }
}

}  // namespace triad

using namespace triad;

extern "C" size_t triad_infonce_workspace_bytes(int rows, int B) {
    if (rows <= 0 || B <= 0) return 0;
    return nce_ws_bytes(rows, B);
}

extern "C" int triad_infonce_partial(const float* clip_rows, int rows, int B, int row0,
                                     float* row_lse, float* col_part,
                                     void* ws, size_t ws_bytes, void* stream) {
    if (!clip_rows || !row_lse || !col_part || !ws) return fail_msg(TRIAD_ERR_BAD_ARG, "infonce_partial: null pointer");
    if (rows <= 0 || B <= 0 || row0 < 0 || row0 + rows > B) return fail_msg(TRIAD_ERR_BAD_SHAPE, "infonce_partial: bad rows/B/row0");
    if (ws_bytes < nce_ws_bytes(rows, B)) return fail_msg(TRIAD_ERR_WORKSPACE, "infonce_partial: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    NceWs w = nce_ws_carve(ws, rows, B);
    const int nblk = nce_blocks(rows);
    nce_partial_kernel<<<nblk, kNceThreads, 0, st>>>(clip_rows, rows, B, kNceRowsPerBlock, row_lse, w.chunk_part, nullptr);
    TRIAD_LAUNCH_CHECK("nce_partial_kernel");
    nce_combine_kernel<<<ceil_div(B, 256), 256, 0, st>>>(w.chunk_part, nblk, B, 0, col_part);
    TRIAD_LAUNCH_CHECK("nce_combine_kernel");
    return TRIAD_OK;
}

extern "C" int triad_infonce_finish(const float* clip_rows, int rows, int B, int row0,
                                    const float* row_lse, const float* col_parts, int nparts,
                                    float grad_scale, float* g, double* sums,
                                    void* ws, size_t ws_bytes, void* stream) {
    if (!clip_rows || !row_lse || !col_parts || !g || !sums || !ws) return fail_msg(TRIAD_ERR_BAD_ARG, "infonce_finish: null pointer");
    if (rows <= 0 || B <= 0 || row0 < 0 || row0 + rows > B || nparts <= 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "infonce_finish: bad rows/B/row0/nparts");
    if (ws_bytes < nce_ws_bytes(rows, B)) return fail_msg(TRIAD_ERR_WORKSPACE, "infonce_finish: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    NceWs w = nce_ws_carve(ws, rows, B);
    const int nblk = nce_blocks(rows);
    nce_combine_kernel<<<ceil_div(B, 256), 256, 0, st>>>(col_parts, nparts, B, 1, w.col_lse);
    TRIAD_LAUNCH_CHECK("nce_combine_kernel(lse)");
    nce_finish_kernel<<<nblk, kNceThreads, 0, st>>>(clip_rows, rows, B, row0, row_lse, w.col_lse,
                                                     grad_scale, g, w.blk_sums);
    TRIAD_LAUNCH_CHECK("nce_finish_kernel");
    nce_final_reduce_kernel<<<1, 32, 0, st>>>(w.blk_sums, nblk, sums);
    TRIAD_LAUNCH_CHECK("nce_final_reduce_kernel");
    return TRIAD_OK;
}

// Fused head: rows per CTA.  Every CTA combines the column partials of ALL row blocks itself (2*nblk dependent-latency
// loads per thread), so few blocks are better than many: about 16 (B = 256: 16 CTAs of 16 rows — measured 19 us with
// 64 blocks of 4 rows, 28 us with the sharded path's 8 blocks of 32), never more than kHeadMaxBlocks.
static inline int head_rows_per_block(int B) {
    int rpb = 4;
    while (ceil_div(B, rpb) > 16) rpb *= 2;
    while (rpb > 32 && ceil_div(B, rpb / 2) <= kHeadMaxBlocks) rpb /= 2;     // large B: keep blocks <= 32 rows if the partials allow
    return rpb;
}
struct HeadWs { float* chunk_part; float* row_lse; double* blk_sums; unsigned int* ticket; size_t total; };
static inline HeadWs head_ws_carve(void* ws, int B) {
    const size_t nblk = ceil_div(B, head_rows_per_block(B));
    char* p = (char*)ws;
    HeadWs w;
    w.chunk_part = (float*)p; p += align_up(nblk * 2 * (size_t)B * 4, 256);
    w.row_lse = (float*)p;    p += align_up((size_t)B * 4, 256);
    w.blk_sums = (double*)p;  p += align_up(nblk * 8 * 8, 256);
    w.ticket = (unsigned int*)p; p += 256;
    w.total = (size_t)(p - (char*)ws);
    return w;
}

extern "C" size_t triad_contrastive_head_workspace_bytes(int B) {
    if (B <= 0) return 0;
    return head_ws_carve(nullptr, B).total;
}

extern "C" int triad_contrastive_head(const float* clip, int B, const float* temperature,
                                      float* g, double* sums, float* out4,
                                      void* ws, size_t ws_bytes, void* stream) {
    if (!clip || !g || !sums || !out4 || !ws) return fail_msg(TRIAD_ERR_BAD_ARG, "contrastive_head: null pointer");
    if (B <= 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "contrastive_head: bad B");
    if (B > kHeadMaxBlocks * 32 || (size_t)B * 4 > 96 * 1024)
        return fail_msg(TRIAD_ERR_UNSUPPORTED, "contrastive_head: B too large for the fused head (use infonce_partial/finish)");
    if (ws_bytes < triad_contrastive_head_workspace_bytes(B)) return fail_msg(TRIAD_ERR_WORKSPACE, "contrastive_head: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const HeadWs w = head_ws_carve(ws, B);
    const int rpb = head_rows_per_block(B);
    const int nblk = ceil_div(B, rpb);
    nce_partial_kernel<<<nblk, kNceThreads, 0, st>>>(clip, B, B, rpb, w.row_lse, w.chunk_part, w.ticket);
    TRIAD_LAUNCH_CHECK("nce_partial_kernel");
    nce_head_kernel<<<nblk, kNceThreads, (size_t)B * 4, st>>>(clip, B, rpb, w.row_lse, w.chunk_part, nblk, temperature, g,
                                                              w.blk_sums, w.ticket, sums, out4);
    TRIAD_LAUNCH_CHECK("nce_head_kernel");
    return TRIAD_OK;
}
