// Shared declarations for the triad_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/triad_b200.h"
#include "triad_round.h"

namespace triad {

int cuda_fail(cudaError_t e, const char* where);   // records triad_last_error(), returns TRIAD_ERR_CUDA
int fail_msg(int status, const char* msg);

#define TRIAD_CUDA_CHECK(expr)                                              \
    do {                                                                    \
        cudaError_t e__ = (expr);                                           \
        if (e__ != cudaSuccess) return ::triad::cuda_fail(e__, #expr);      \
    } while (0)

// Opt a kernel in to > 48 KB of dynamic shared memory.  The attribute is PER DEVICE, so the "already done" state is a
// bit per device ordinal (one process may drive several GPUs, and autograd runs backward on its own threads).
#define TRIAD_SET_MAX_SMEM(kern, bytes)                                                                       \
    do {                                                                                                      \
        static std::atomic<unsigned long long> done__{0ull};                                                  \
        int dev__ = 0;                                                                                        \
        TRIAD_CUDA_CHECK(cudaGetDevice(&dev__));                                                              \
        const unsigned long long bit__ = 1ull << (dev__ & 63);                                                \
        if (!(done__.load(std::memory_order_acquire) & bit__)) {                                              \
            TRIAD_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))); \
            done__.fetch_or(bit__, std::memory_order_release);                                                \
        }                                                                                                     \
    } while (0)

void count_launch();                                // triad_launch_count(): kernels launched by this library

#define TRIAD_LAUNCH_CHECK(what)                                            \
    do {                                                                    \
        cudaError_t e__ = cudaGetLastError();                               \
        if (e__ != cudaSuccess) return ::triad::cuda_fail(e__, what);       \
        ::triad::count_launch();                                            \
    } while (0)

// Launches kKernel as clusters of cta_group CTAs with smem bytes of dynamic shared memory, and counts the launch.
template <auto kKernel, typename... Args>
int launch_clusters(int cta_group, int n_clusters, int threads, uint32_t smem, cudaStream_t st, const Args&... args) {
    TRIAD_SET_MAX_SMEM(kKernel, smem);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(n_clusters * cta_group));
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cta_group;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    TRIAD_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kKernel, args...));
    count_launch();
    return TRIAD_OK;
}

// Multiprocessor count of the current device.  On a CUDA error it returns TRIAD_ERR_CUDA and leaves *sms = 148 (a
// B200): the workspace-size functions, which cannot report an error, size for that.
int device_sms(int* sms);

// Tiled tensor map over bf16, fp32 or uint8 elements (rank 2 or 3, element strides 1, 256-byte L2 promotion, zero fill).
enum class Swizzle { kNone, k128B };
int encode_tmap(CUtensorMap* map, CUtensorMapDataType type, const void* base, int rank, const cuuint64_t* dims,
                const cuuint64_t* strides, const cuuint32_t* box, Swizzle swizzle);

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// The control block at the start of a workspace, cleared before each call: the kernels' watchdog abort flag at [0]
// (and the backward's dT ticket at [16]).
constexpr size_t kCtrlBlockBytes = 256;

// ---- forward partial-sum layout ---------------------------------------------------------
// The forward kernels reduce row maxima per 32-row GROUP (one warp of the epilogue) and per
// query inside the group, deterministically (shuffle tree), into
//     part[j][g][s]   j < Bv, g < G = ceil(M/32), s < S = 31/Nq + 2
// where slot s of group g belongs to query (32*g)/Nq + s.  finalize_clip() then sums, for
// every (i,j), the groups that hold rows of query i in ascending g — a fixed order, so clip
// is bit-reproducible run to run (no float atomics anywhere on the forward path).
struct PartLayout {
    int G;   // 32-row groups
    int S;   // query slots per group
};
static inline PartLayout part_layout(int M, int Nq) {
    PartLayout p; p.G = ceil_div(M, 32); p.S = 31 / Nq + 2; return p;
}

// ---- division by a runtime constant (n < 2^31, 1 <= d < 2^31): one multiply-high and a shift -----------
struct FastDiv {
    uint32_t d, mul, shift;      // n / d == umulhi(n, mul) >> shift   (round-up method, exact for n < 2^31)
};
static inline FastDiv make_fastdiv(uint32_t d) {
    FastDiv f; f.d = d;
    if (d <= 1) { f.mul = 0; f.shift = 0; return f; }            // handled separately (n / 1)
    uint32_t l = 0;
    while ((1ull << l) < d) ++l;                                   // l = ceil(log2 d)
    f.shift = l - 1;                                               // n < 2^31: a 32-bit multiplier with shift l-1 is exact
    f.mul = (uint32_t)((((1ull << (31 + l)) + d - 1) / d) & 0xffffffffull);
    return f;
}

// ---- argmax index layout ------------------------------------------------------------------
// idx[j][i][a], a < nq_pad = Nq rounded up to 16: every query's run of winners starts 16-byte
// aligned, so the backward can fetch 8 or 16 consecutive rows' winners with one vector load.
static inline int nq_padded(int Nq) { return (Nq + 15) / 16 * 16; }

// launchers implemented in the .cu files -------------------------------------------------
int launch_row_scale(const int64_t* mask, int Bq, int Nq, float* row_scale, cudaStream_t st);
int launch_maxmean_simt(const void* q, const void* v, const float* row_scale, const float* T,
                        int inv_T, int M, int Bv, int Nq, int Nv, int D, int dtype,
                        float* part, void* idx, cudaStream_t st);   // idx: [Bv][M/Nq][nq_padded(Nq)]
// dense-regulariser modes of the tcgen05 forward (maxmean_tc.cu, kMode): the epilogue writes N = dL/d<q,v> of the
// non-negative-pressure term — instead of reducing each tile (with_maxmean = 0) or next to the max-mean reduction
// (with_maxmean = 1: clip partials, idx and N from ONE pass over the similarities).  Every epilogue warp of every CTA
// owns one slot of [SMs * kEmitEpiWarps][2] double partials; the launch clears them and adds them to sums[0..1].
struct EmitNArgs { void* n_out; long long ldn; float lo, coef; int write_n; double* partials; double* sums; int with_maxmean; };
constexpr int kEmitEpiWarps = 8;                                      // epilogue warps 4-11 of the emitting kernel
constexpr int kNonnegFusedPartials = 512 * kEmitEpiWarps;             // partial slots: devices of up to 512 SMs
bool tc_emit_supported(int Nv, int D);
// e4m3 retrieval operands (kFp8): q and v hold e4m3 codes, scaled per token (q_scale [M]) and per patch
// (g_scale [Bv][Nv]); divides by T, no idx, D in {128, 256, 384, 512}
struct E4m3Args { const float* q_scale; const float* g_scale; };
bool tc_e4m3_supported(int Nv, int D);
// ragged caption gallery (ragged.cu): captions packed whole into kSlotRows-row slots, zero rows at a slot's end.
// slot_meta [slots][kSlotMetaInts] int32: first caption id, caption count, used rows, 0, the caption-start mask (bit
// r of word r/32 = a caption starts at row r), the caption-end mask (its last row); cap_info [captions][2] int32:
// first row (slot * kSlotRows + offset), length (1..kSlotRows)
constexpr int kSlotRows = 256;
constexpr int kSlotMetaCap0 = 0, kSlotMetaCount = 1, kSlotMetaUsed = 2, kSlotMetaStarts = 4, kSlotMetaEnds = 12;
constexpr int kSlotMetaInts = 20;
// direction 0: q = the query's tokens, v = the slots (Bv = slots, Nv = kSlotRows), partials part[caption][group];
// direction 1: q = the slot rows (M = slots * kSlotRows), v = the query (Bv = 1), one weighted row max per slot row
struct RaggedArgs { const int* slot_meta; const int* cap_info; int direction; };
int launch_maxmean_tc(const void* q, const void* v, const float* row_scale, const float* T,
                      int inv_T, int M, int Bv, int Nq, int Nv, int D,
                      float* part, void* idx, int* abort_flag, int cta_group, int flags, const int* pack_maps,
                      const EmitNArgs* emit, const E4m3Args* e4m3, cudaStream_t st, const RaggedArgs* ragged = nullptr);
// cta_group of the unpacked tcgen05 forwards (capi.cu)
int fwd_cta_group(int M, int flags);
// sums[0..1] += the per-warp partials of a dense-regulariser forward, in slot order (dense_reg.cu)
int launch_nonneg_finish(const double* partials, int n, double* sums, cudaStream_t st);
int launch_finalize_clip(const float* part, int Bq, int Bv, int Nq, float* clip, const int* abort_flag, cudaStream_t st);
// packed rows (pack.cu): maps = off[Bq+1] | rowmap[Bq*Nq] | scratch
size_t pack_map_bytes(int Bq, int Nq);
int launch_pack_map(const float* row_scale, int Bq, int Nq, void* maps, cudaStream_t st);
int launch_pack_groups(const float* row_scale, int Bq, int Nq, void* maps, cudaStream_t st);   // goff[Bq+1] | glist | cnt
int launch_pack_copy(const void* q, const void* maps, int Bq, int Nq, int D, int elt_bytes, void* qp, cudaStream_t st);
int launch_finalize_clip_packed(const float* part, const int* pack_off, int Bq, int Bv, int Nq, float* clip,
                                const int* abort_flag, cudaStream_t st);
// partial sums of the packed forward: part[(j*Bq + i)*pieces + piece], piece = (32-row group of the packed row)
// - (group of the query's first packed row); a query of <= Nq kept rows spans at most (Nq+30)/32 + 1 groups
static inline int packed_pieces(int Nq) { return (Nq + 30) / 32 + 1; }
bool tc_supported(int Nv, int D);
// rows x D (fp32 or bf16) -> e4m3 codes [rows][D] + one fp32 scale per row (quant_e4m3.cu); D % 16 == 0, D <= 512.
// With a rowmap, output row r is source row rowmap[r] of the src_rows rows of x, or a zero row where it is negative
// or not below src_rows.
int launch_quantize_e4m3(const void* x, int dtype, long long rows, int D, void* codes, float* scales, cudaStream_t st,
                         const int* rowmap = nullptr, long long src_rows = 0);
// tiled dQ of the backward, bf16 only.  Nv <= 256 (uint8 winners): the software-pipelined shared-memory gather
// (bwd_dq_pipe.cu); Nv > 256 (uint16 winners): the L1-resident gather (bwd_dq_tile.cu)
bool dq_pipe_supported(int Nv, int D, int dtype);
int launch_dq_pipe(const void* v, const void* idx, const float* g, const float* row_scale, const float* Tp,
                   int Bq, int Bv, int Nq, int Nv, int D, void* dq, int* abort_flag,
                   const int* glist, const int* n_groups_dev, cudaStream_t st);
// the projection head backward's products on the dense-gradient GEMM (dense_gemm.cu): mode 0 out[M][D] = N . x,
// mode 1 out[Kc][D] = N^T . x, any D % 64 == 0 (512-column output slices), fp32 (out_f32) or bf16 out
size_t head_gemm_workspace_bytes(int M, int Kc, int D, int mode);
int launch_head_gemm(const void* n_mat, long long ldn, int M, int Kc, const void* x, int D, int mode, void* out,
                     int out_f32, void* ws, size_t ws_bytes, cudaStream_t st);
bool dq_tile_supported(int D, int dtype);
int launch_dq_tile(const void* v, const void* idx, const float* g, const float* row_scale, const float* Tp,
                   int M, int Bv, int Nq, int Nv, int D, void* dq, cudaStream_t st);

// ---- device helpers -----------------------------------------------------------------------
#if defined(__CUDACC__)

__device__ __forceinline__ uint32_t fast_div(uint32_t n, const FastDiv& f) {
    return f.d <= 1 ? n : (__umulhi(n, f.mul) >> f.shift);
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One warp holds 32 consecutive token rows (row = row0 + lane) of image j: `val` is the row's
// weighted maximum (0 for rows >= M).  Segmented shuffle reduction keyed by the query id
// (rows of one query are contiguous, so segments are contiguous lane ranges); the first lane
// of each segment stores part[j][g][qid - qfirst].
__device__ __forceinline__ void store_group_partials(float* __restrict__ part, int j, int g,
                                                     int G, int S, int row0, int M, int Nq,
                                                     float val, int lane) {
    const int r = row0 + lane;
    const int qid = (r < M) ? r / Nq : 0x7fffffff;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        float t = __shfl_down_sync(0xffffffffu, val, o);
        int tq = __shfl_down_sync(0xffffffffu, qid, o);
        if (lane + o < 32 && tq == qid) val += t;
    }
    const int prev = __shfl_up_sync(0xffffffffu, qid, 1);
    const bool head = (lane == 0) || (prev != qid);
    if (head && r < M) {
        const int qfirst = (g * 32) / Nq;
        part[((size_t)j * G + g) * S + (qid - qfirst)] = val;
    }
}

// Packed rows: the same segmented reduction; the head lane of each query segment stores the segment's sum in
// the query's slot for this 32-row group.
__device__ __forceinline__ void store_group_partials_packed(float* __restrict__ part, int j, int Bq, int pieces,
                                                            int qid, int piece, float val, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        float t = __shfl_down_sync(0xffffffffu, val, o);
        int tq = __shfl_down_sync(0xffffffffu, qid, o);
        if (lane + o < 32 && tq == qid) val += t;
    }
    const int prev = __shfl_up_sync(0xffffffffu, qid, 1);
    const bool head = (lane == 0) || (prev != qid);
    if (head && qid != 0x7fffffff) part[((size_t)j * Bq + qid) * pieces + piece] = val;
}

#endif  // __CUDACC__
}  // namespace triad
