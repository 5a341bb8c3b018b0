// Projection head of the three embedders (SURVEY.md §8 f3): the producer of the hot path's inputs.
//
//   feats = projection2( layer_norm( projection1(x) ) )            src/model.py:32-34,68 (audio),
//                                                                  :81-83,116 (text), :253-255,326 (visual)
//   (+ F.normalize(feats, dim=-1) for audio-visual retrieval:      src/retrieval.py:93-94)
//
// The reference runs three library kernels per embedder (Linear, LayerNorm, Linear) with the 512-wide hidden
// activations going through HBM twice.  Here one CTA owns 128 token rows end to end and the hidden row never leaves
// the chip:
//
//   GEMM 1   h[128 x 512] = x[128 x Din] . W1^T            tcgen05.mma, fp32 accumulators = all 512 TMEM columns
//   epilogue LayerNorm over the 512 columns of each row (one thread = one TMEM lane = one token): + bias, rounded
//            to bf16 (the Linear's output dtype under autocast), fp32 mean / variance / affine (autocast keeps
//            layer_norm in fp32), rounded to bf16 and written into shared memory in the SWIZZLE_128B K-major
//            layout, i.e. directly as the A operand of
//   GEMM 2   out[128 x Dout] = ln[128 x 512] . W2^T          (same TMEM columns, overwritten)
//   epilogue + bias, bf16, optional L2 normalisation of the row, one contiguous 2*Dout-byte store per token: the
//            [B, N, D] K-major layout the similarity kernel's TMA maps read.
//
// Weights stream through a TMA ring (nn.Linear's [out, in] layout IS the K-major B operand: no transposes).
// Warp roles: warp 0 TMA producer, warp 1 TMEM allocator + MMA issuer, warps 2-5 epilogue.  The kernel is a few
// per cent of a training step (84 GFLOP at the B=256 audio shape); it is built for fusion, not tuned to the last
// cycle: one tile per CTA, no overlap between a tile's phases.
#include "common.cuh"
#include "ptx.cuh"

namespace triad {
namespace proj {
using namespace ptx;

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;
constexpr int kUmmaK = 16;
constexpr int kHidden = 512;
constexpr int kHalfN = 256;
constexpr int kThreads = 192;
constexpr uint32_t kAkb = kBlockM * kBlockK * 2;        // 16 KB: one k-block of a 128-row A tile
constexpr uint32_t kBst = kHalfN * kBlockK * 2;         // 32 KB: one k-block of 256 weight rows
constexpr int kStages1 = 4;
constexpr uint32_t kStage1 = kAkb + kBst;               // 48 KB
constexpr uint32_t kA2 = (kHidden / kBlockK) * kAkb;    // 128 KB: the LayerNorm output as GEMM 2's A operand
constexpr int kStages2 = 3;
constexpr uint32_t kRing = kA2 + kStages2 * kBst;       // 224 KB >= kStages1 * kStage1 (192 KB)
constexpr uint32_t kSmemBytes = kRing + 1024 + 1024;    // + barriers + alignment slack

struct Params {
    const float* b1; const float* ln_g; const float* ln_b; const float* b2;
    __nv_bfloat16* out;
    int* abort_flag;
    int M, Din, Dout, normalize;
    float eps;
};

__device__ __forceinline__ float bf16r(float x) { return __bfloat162float(__float2bfloat16(x)); }

__global__ void __launch_bounds__(kThreads, 1)
proj_head_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w1,
                 const __grid_constant__ CUtensorMap tmap_w2, const Params p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar = base + kRing;
    const uint32_t full1 = bar, empty1 = bar + 8 * kStages1;
    const uint32_t full2 = empty1 + 8 * kStages1, empty2 = full2 + 8 * kStages2;
    const uint32_t t_full1 = empty2 + 8 * kStages2, a2_ready = t_full1 + 8, t_full2 = a2_ready + 8;
    const uint32_t tmem_slot = t_full2 + 8;
    uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(gen + (tmem_slot - base));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * kBlockM;
    const int nkb1 = p.Din / kBlockK;
    const int n_halves = p.Dout > kHalfN ? 2 : 1;

    if (warp == 0 && lane == 0) { prefetch_tmap(&tmap_x); prefetch_tmap(&tmap_w1); prefetch_tmap(&tmap_w2); }
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < kStages1; ++s) { mbar_init(full1 + 8 * s, 1); mbar_init(empty1 + 8 * s, 1); }
            for (int s = 0; s < kStages2; ++s) { mbar_init(full2 + 8 * s, 1); mbar_init(empty2 + 8 * s, 1); }
            mbar_init(t_full1, 1); mbar_init(a2_ready, 4 * 32); mbar_init(t_full2, 1);
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc<1>(tmem_slot, 512);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem0 = *tmem_slot_gen;

    if (warp == 0) {
        // =============================== TMA producer ===================================
        if (lane == 0) {
            int s = 0; uint32_t ph = 0; bool ok = true;
            for (int half = 0; half < 2 && ok; ++half)
                for (int kb = 0; kb < nkb1; ++kb) {
                    ok = mbar_wait(empty1 + 8 * s, ph ^ 1, p.abort_flag, 21);
                    if (!ok) break;
                    mbar_expect_tx(full1 + 8 * s, kStage1);
                    tma_load_2d<1>(base + s * kStage1, &tmap_x, full1 + 8 * s, kb * kBlockK, m0);
                    tma_load_2d<1>(base + s * kStage1 + kAkb, &tmap_w1, full1 + 8 * s, kb * kBlockK, half * kHalfN);
                    if (++s == kStages1) { s = 0; ph ^= 1; }
                }
            // the second ring lives behind the LayerNorm tile, inside what the first ring used: wait until every
            // MMA of GEMM 1 has read its operands
            ok = ok && mbar_wait(t_full1, 0, p.abort_flag, 22);
            s = 0; ph = 0;
            for (int half = 0; half < n_halves && ok; ++half)
                for (int kb = 0; kb < kHidden / kBlockK; ++kb) {
                    ok = mbar_wait(empty2 + 8 * s, ph ^ 1, p.abort_flag, 23);
                    if (!ok) break;
                    mbar_expect_tx(full2 + 8 * s, kBst);
                    tma_load_2d<1>(base + kA2 + s * kBst, &tmap_w2, full2 + 8 * s, kb * kBlockK, half * kHalfN);
                    if (++s == kStages2) { s = 0; ph ^= 1; }
                }
        }
    } else if (warp == 1) {
        // =============================== MMA issuer =====================================
        if (lane == 0) {
            int s = 0; uint32_t ph = 0; bool ok = true;
            const uint32_t idesc1 = make_idesc(kBlockM, kHalfN);
            for (int half = 0; half < 2 && ok; ++half)
                for (int kb = 0; kb < nkb1; ++kb) {
                    ok = mbar_wait(full1 + 8 * s, ph, p.abort_flag, 24);
                    if (!ok) break;
                    tc_fence_after();
                    const uint64_t a_desc = make_smem_desc(base + s * kStage1);
                    const uint64_t b_desc = make_smem_desc(base + s * kStage1 + kAkb);
#pragma unroll
                    for (int k = 0; k < kBlockK / kUmmaK; ++k)
                        umma_bf16<1>(tmem0 + half * kHalfN, a_desc + 2u * k, b_desc + 2u * k, idesc1, (uint32_t)((kb | k) != 0));
                    umma_commit<1>(empty1 + 8 * s);
                    if (++s == kStages1) { s = 0; ph ^= 1; }
                }
            if (ok) umma_commit<1>(t_full1);                       // h complete (and the first ring's memory free)
            // GEMM 2 overwrites the same TMEM columns and reads the LayerNorm tile: both are handed over by a2_ready
            ok = ok && mbar_wait(a2_ready, 0, p.abort_flag, 25);
            tc_fence_after();
            s = 0; ph = 0;
            for (int half = 0; half < n_halves && ok; ++half) {
                const int n = min(kHalfN, p.Dout - half * kHalfN);
                const uint32_t idesc2 = make_idesc(kBlockM, (n + 15) / 16 * 16);
                for (int kb = 0; kb < kHidden / kBlockK; ++kb) {
                    ok = mbar_wait(full2 + 8 * s, ph, p.abort_flag, 26);
                    if (!ok) break;
                    tc_fence_after();
                    const uint64_t a_desc = make_smem_desc(base + kb * kAkb);
                    const uint64_t b_desc = make_smem_desc(base + kA2 + s * kBst);
#pragma unroll
                    for (int k = 0; k < kBlockK / kUmmaK; ++k)
                        umma_bf16<1>(tmem0 + half * kHalfN, a_desc + 2u * k, b_desc + 2u * k, idesc2, (uint32_t)((kb | k) != 0));
                    umma_commit<1>(empty2 + 8 * s);
                    if (++s == kStages2) { s = 0; ph ^= 1; }
                }
            }
            if (ok) umma_commit<1>(t_full2);
        }
    } else {
        // =============================== epilogue: one thread = one token row ============
        const int quarter = warp & 3;                              // TMEM lanes this warp may touch: 32*(warp % 4)
        const int r = quarter * 32 + lane;                         // row inside the tile
        const int row = m0 + r;
        const uint32_t taddr = tmem0 + ((uint32_t)(quarter * 32) << 16);
        bool ok = mbar_wait(t_full1, 0, p.abort_flag, 27);
        tc_fence_after();
        uint32_t buf[32];
        // ---- LayerNorm: mean, variance (two passes over the accumulator), then normalise + affine ----
        float sum = 0.f;
        for (int c = 0; c < kHidden / 32; ++c) {
            tmem_ld32_raw(taddr + c * 32, buf);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 32; ++e) sum += bf16r(__uint_as_float(buf[e]) + bf16r(__ldg(p.b1 + c * 32 + e)));
        }
        const float mean = sum * (1.f / kHidden);
        float sq = 0.f;
        for (int c = 0; c < kHidden / 32; ++c) {
            tmem_ld32_raw(taddr + c * 32, buf);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                const float d = bf16r(__uint_as_float(buf[e]) + bf16r(__ldg(p.b1 + c * 32 + e))) - mean;
                sq = fmaf(d, d, sq);
            }
        }
        const float rstd = rsqrtf(sq * (1.f / kHidden) + p.eps);
        for (int c = 0; c < kHidden / 32; ++c) {
            tmem_ld32_raw(taddr + c * 32, buf);
            tmem_wait_ld();
            const int kb = c >> 1;                                 // 64 columns per k-block
            const uint32_t rowaddr = base + kb * kAkb + (uint32_t)r * 128u;
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {                       // four 16-byte chunks (8 columns each)
                uint32_t w[4];
#pragma unroll
                for (int e2 = 0; e2 < 4; ++e2) {
                    const int col = c * 32 + ch * 8 + e2 * 2;
                    const float h0 = bf16r(__uint_as_float(buf[ch * 8 + e2 * 2]) + bf16r(__ldg(p.b1 + col)));
                    const float h1 = bf16r(__uint_as_float(buf[ch * 8 + e2 * 2 + 1]) + bf16r(__ldg(p.b1 + col + 1)));
                    const float y0 = (h0 - mean) * rstd * __ldg(p.ln_g + col) + __ldg(p.ln_b + col);
                    const float y1 = (h1 - mean) * rstd * __ldg(p.ln_g + col + 1) + __ldg(p.ln_b + col + 1);
                    __nv_bfloat162 pk = __floats2bfloat162_rn(y0, y1);
                    w[e2] = *reinterpret_cast<uint32_t*>(&pk);
                }
                const uint32_t chunk = (uint32_t)((c & 1) * 4 + ch);                   // 16-byte chunk inside the 128-byte row
                const uint32_t addr = rowaddr + ((chunk ^ ((uint32_t)r & 7u)) << 4);   // SWIZZLE_128B
                asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]) : "memory");
            }
        }
        tc_fence_before();                 // our tcgen05.ld of h are done (waited) before GEMM 2 may overwrite it
        fence_proxy_async();               // the st.shared above become visible to the tensor core's (async-proxy) reads
        mbar_arrive_local(a2_ready);

        // ---- output: + bias, bf16, optional L2 normalisation, one contiguous row store ----
        ok = ok && mbar_wait(t_full2, 0, p.abort_flag, 28);
        tc_fence_after();
        const int nch = (p.Dout + 31) / 32;
        float inv = 1.f;
        if (p.normalize) {
            float ss = 0.f;
            for (int c = 0; c < nch; ++c) {
                tmem_ld32_raw(taddr + c * 32, buf);
                tmem_wait_ld();
#pragma unroll
                for (int e = 0; e < 32; ++e) {
                    const int col = c * 32 + e;
                    if (col < p.Dout) { const float o = bf16r(__uint_as_float(buf[e]) + bf16r(__ldg(p.b2 + col))); ss = fmaf(o, o, ss); }
                }
            }
            inv = 1.f / fmaxf(sqrtf(ss), 1e-12f);                  // F.normalize: x / max(||x||, eps)
        }
        const bool poisoned = !ok || *(volatile int*)p.abort_flag != 0;
        for (int c = 0; c < nch; ++c) {
            tmem_ld32_raw(taddr + c * 32, buf);
            tmem_wait_ld();
            if (row < p.M) {
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) {
                    const int col0 = c * 32 + ch * 8;
                    if (col0 < p.Dout) {                           // Dout % 8 == 0
                        uint32_t w[4];
#pragma unroll
                        for (int e2 = 0; e2 < 4; ++e2) {
                            const int col = col0 + e2 * 2;
                            float o0 = bf16r(__uint_as_float(buf[ch * 8 + e2 * 2]) + bf16r(__ldg(p.b2 + col))) * inv;
                            float o1 = bf16r(__uint_as_float(buf[ch * 8 + e2 * 2 + 1]) + bf16r(__ldg(p.b2 + col + 1))) * inv;
                            if (poisoned) o0 = o1 = __int_as_float(0x7fc00000);
                            __nv_bfloat162 pk = __floats2bfloat162_rn(o0, o1);
                            w[e2] = *reinterpret_cast<uint32_t*>(&pk);
                        }
                        *reinterpret_cast<uint4*>(p.out + (size_t)row * p.Dout + col0) = make_uint4(w[0], w[1], w[2], w[3]);
                    }
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem_dealloc<1>(tmem0, 512); }
}

// ================================ backward: the row pass ===========================================================
// With gy = dL/dout (bf16 [M, Dout], the layout triad_maxmean_bwd writes dq / dv in), one CTA per 128-token tile:
//
//   GEMM 1   h = x . W1^T recomputed into all 512 TMEM columns, exactly as the forward; the epilogue rounds
//            h = bf16(acc + bf16(b1)) into shared memory (the forward's LayerNorm tile layout) and takes the row mean
//            and rstd with the forward's arithmetic, so xh is bit for bit what the forward normalised
//   GEMM 2'  gln = gy . W2 (K = Dout, N = 512) into the same TMEM columns; W2 [Dout, 512] is read as an MN-major B
//            operand as stored (64 x 64 SWIZZLE_128B boxes, the dense-gradient GEMMs' layout): no transposed copy
//   epilogue one thread per row: gxh = gln * gamma, gh = rstd * (gxh - mean(gxh) - xh * mean(gxh * xh)) -> bf16 gh,
//            ln = bf16(xh * gamma + beta) -> bf16 ln (projection2's weight gradient reads it), and per-tile fp32
//            column sums of gln * xh (d gamma), gln (d beta), gh (d b1, before rounding) and gy (d b2): each warp adds
//            its 32 rows by a fixed shuffle tree, the four warps are added in warp order, one partial row per tile;
//            proj_bwd_finish_kernel adds the tiles in tile order (deterministic, no float atomics).
//
// Shared memory: GEMM 1 uses the forward's 4-stage ring; the h tile (128 KB) then takes the ring's first 128 KB and
// GEMM 2' streams through a 2-stage ring behind it (gy k-block 16 KB + one 256-column half of a W2 k-block 32 KB).
constexpr int kStagesB = 2;
constexpr uint32_t kW2Box = 64 * 128;                   // 64 n x 64 k bf16
constexpr uint32_t kStageB = kAkb + 4 * kW2Box;         // 48 KB
static_assert(kA2 + kStagesB * kStageB <= kRing, "GEMM 2' ring");
constexpr int kPartRows = 4;                            // d gamma, d beta, d b1, d b2

struct BwdParams {
    const float* b1; const float* ln_g; const float* ln_b;
    const __nv_bfloat16* gy;
    __nv_bfloat16* gh; __nv_bfloat16* ln;
    float* part;                                        // [tiles][kPartRows][512]
    int* abort_flag;
    int M, Din, Dout;
    float eps;
};

// v[i] of lane l = this lane's value of column i (32 columns); returns, in lane l, the sum of column l over the 32 lanes.
// Fixed butterfly order: the result does not depend on timing.
__device__ __forceinline__ float column_sums32(float (&v)[32], int lane) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const bool upper = (lane & s) != 0;
#pragma unroll
        for (int i = 0; i < s; ++i) {
            const float send = upper ? v[i] : v[i + s];
            const float keep = upper ? v[i + s] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
        }
    }
    return v[0];
}

// 32 consecutive h columns (chunk c) of row r from the swizzled bf16 tile
__device__ __forceinline__ void load_h32(uint32_t base, int r, int c, float (&h)[32]) {
    const uint32_t rowaddr = base + (uint32_t)(c >> 1) * kAkb + (uint32_t)r * 128u;
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
        const uint32_t chunk = (uint32_t)((c & 1) * 4 + ch);
        uint32_t w[4];
        asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3])
                     : "r"(rowaddr + ((chunk ^ ((uint32_t)r & 7u)) << 4)) : "memory");
#pragma unroll
        for (int e2 = 0; e2 < 4; ++e2) {
            const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[e2]));
            h[ch * 8 + e2 * 2] = f.x; h[ch * 8 + e2 * 2 + 1] = f.y;
        }
    }
}

__device__ __forceinline__ void store_row32(__nv_bfloat16* dst, const float (&v)[32], bool poisoned) {
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
        uint32_t w[4];
#pragma unroll
        for (int e2 = 0; e2 < 4; ++e2) {
            float a = v[ch * 8 + e2 * 2], b = v[ch * 8 + e2 * 2 + 1];
            if (poisoned) a = b = __int_as_float(0x7fc00000);
            __nv_bfloat162 pk = __floats2bfloat162_rn(a, b);
            w[e2] = *reinterpret_cast<uint32_t*>(&pk);
        }
        reinterpret_cast<uint4*>(dst)[ch] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

__global__ void __launch_bounds__(kThreads, 1)
proj_head_bwd_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w1,
                     const __grid_constant__ CUtensorMap tmap_gy, const __grid_constant__ CUtensorMap tmap_w2,
                     const BwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar = base + kRing;
    const uint32_t full1 = bar, empty1 = bar + 8 * kStages1;
    const uint32_t full2 = empty1 + 8 * kStages1, empty2 = full2 + 8 * kStagesB;
    const uint32_t t_full1 = empty2 + 8 * kStagesB, t_free = t_full1 + 8, t_full2 = t_free + 8;
    const uint32_t tmem_slot = t_full2 + 8;
    uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(gen + (tmem_slot - base));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * kBlockM;
    const int nkb1 = p.Din / kBlockK;
    const int nkb2 = (p.Dout + kBlockK - 1) / kBlockK;

    if (warp == 0 && lane == 0) { prefetch_tmap(&tmap_x); prefetch_tmap(&tmap_w1); prefetch_tmap(&tmap_gy); prefetch_tmap(&tmap_w2); }
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < kStages1; ++s) { mbar_init(full1 + 8 * s, 1); mbar_init(empty1 + 8 * s, 1); }
            for (int s = 0; s < kStagesB; ++s) { mbar_init(full2 + 8 * s, 1); mbar_init(empty2 + 8 * s, 1); }
            mbar_init(t_full1, 1); mbar_init(t_free, 4 * 32); mbar_init(t_full2, 1);
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc<1>(tmem_slot, 512);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem0 = *tmem_slot_gen;

    if (warp == 0) {
        // =============================== TMA producer ===================================
        if (lane == 0) {
            int s = 0; uint32_t ph = 0; bool ok = true;
            for (int half = 0; half < 2 && ok; ++half)
                for (int kb = 0; kb < nkb1; ++kb) {
                    ok = mbar_wait(empty1 + 8 * s, ph ^ 1, p.abort_flag, 41);
                    if (!ok) break;
                    mbar_expect_tx(full1 + 8 * s, kStage1);
                    tma_load_2d<1>(base + s * kStage1, &tmap_x, full1 + 8 * s, kb * kBlockK, m0);
                    tma_load_2d<1>(base + s * kStage1 + kAkb, &tmap_w1, full1 + 8 * s, kb * kBlockK, half * kHalfN);
                    if (++s == kStages1) { s = 0; ph ^= 1; }
                }
            // the second ring lies inside what the first one used: wait until every MMA of GEMM 1 has read its operands
            ok = ok && mbar_wait(t_full1, 0, p.abort_flag, 42);
            s = 0; ph = 0;
            for (int half = 0; half < 2 && ok; ++half)
                for (int kb = 0; kb < nkb2; ++kb) {
                    ok = mbar_wait(empty2 + 8 * s, ph ^ 1, p.abort_flag, 43);
                    if (!ok) break;
                    const uint32_t st = base + kA2 + s * kStageB;
                    mbar_expect_tx(full2 + 8 * s, kStageB);
                    tma_load_2d<1>(st, &tmap_gy, full2 + 8 * s, kb * kBlockK, m0);                       // {64 k, 128 rows}
#pragma unroll
                    for (int j = 0; j < 4; ++j)                                                            // {64 n, 64 k}
                        tma_load_2d<1>(st + kAkb + j * kW2Box, &tmap_w2, full2 + 8 * s, half * kHalfN + j * 64, kb * kBlockK);
                    if (++s == kStagesB) { s = 0; ph ^= 1; }
                }
        }
    } else if (warp == 1) {
        // =============================== MMA issuer =====================================
        if (lane == 0) {
            int s = 0; uint32_t ph = 0; bool ok = true;
            const uint32_t idesc1 = make_idesc(kBlockM, kHalfN);
            for (int half = 0; half < 2 && ok; ++half)
                for (int kb = 0; kb < nkb1; ++kb) {
                    ok = mbar_wait(full1 + 8 * s, ph, p.abort_flag, 44);
                    if (!ok) break;
                    tc_fence_after();
                    const uint64_t a_desc = make_smem_desc(base + s * kStage1);
                    const uint64_t b_desc = make_smem_desc(base + s * kStage1 + kAkb);
#pragma unroll
                    for (int k = 0; k < kBlockK / kUmmaK; ++k)
                        umma_bf16<1>(tmem0 + half * kHalfN, a_desc + 2u * k, b_desc + 2u * k, idesc1, (uint32_t)((kb | k) != 0));
                    umma_commit<1>(empty1 + 8 * s);
                    if (++s == kStages1) { s = 0; ph ^= 1; }
                }
            if (ok) umma_commit<1>(t_full1);
            // GEMM 2' overwrites the accumulator: the epilogue hands it back once h is in shared memory
            ok = ok && mbar_wait(t_free, 0, p.abort_flag, 45);
            tc_fence_after();
            const uint32_t idesc2 = make_idesc(kBlockM, kHalfN) | (1u << 16);                 // B MN-major
            s = 0; ph = 0;
            for (int half = 0; half < 2 && ok; ++half)
                for (int kb = 0; kb < nkb2; ++kb) {
                    ok = mbar_wait(full2 + 8 * s, ph, p.abort_flag, 46);
                    if (!ok) break;
                    tc_fence_after();
                    const uint32_t st = base + kA2 + s * kStageB;
                    const uint64_t a_desc = make_smem_desc(st);
                    const uint64_t b_desc = make_smem_desc(st + kAkb);
                    // MN-major B: 64-element n groups kW2Box apart (LBO), 8-row k groups 1 KB apart (SBO)
                    const uint64_t b_mn = (b_desc & ~(0x3FFFull << 16)) | ((uint64_t)(kW2Box >> 4) << 16);
#pragma unroll
                    for (int k = 0; k < kBlockK / kUmmaK; ++k)                                         // K = 16: 32 B of A, 2 KB of B
                        umma_bf16<1>(tmem0 + half * kHalfN, a_desc + 2u * k, b_mn + 128u * k, idesc2, (uint32_t)((kb | k) != 0));
                    umma_commit<1>(empty2 + 8 * s);
                    if (++s == kStagesB) { s = 0; ph ^= 1; }
                }
            if (ok) umma_commit<1>(t_full2);
        }
    } else {
        // =============================== epilogue: one thread = one token row ============
        const int quarter = warp & 3;
        const int r = quarter * 32 + lane;
        const int row = m0 + r;
        const bool valid = row < p.M;
        const uint32_t taddr = tmem0 + ((uint32_t)(quarter * 32) << 16);
        bool ok = mbar_wait(t_full1, 0, p.abort_flag, 47);
        tc_fence_after();
        uint32_t buf[32];
        // ---- h = bf16(acc + bf16(b1)) into shared memory, row sum (the forward's order) ----
        float sum = 0.f;
        for (int c = 0; c < kHidden / 32; ++c) {
            tmem_ld32_raw(taddr + c * 32, buf);
            tmem_wait_ld();
            const uint32_t rowaddr = base + (uint32_t)(c >> 1) * kAkb + (uint32_t)r * 128u;
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {
                uint32_t w[4];
#pragma unroll
                for (int e2 = 0; e2 < 4; ++e2) {
                    const int e = ch * 8 + e2 * 2;
                    const float h0 = bf16r(__uint_as_float(buf[e]) + bf16r(__ldg(p.b1 + c * 32 + e)));
                    const float h1 = bf16r(__uint_as_float(buf[e + 1]) + bf16r(__ldg(p.b1 + c * 32 + e + 1)));
                    sum += h0; sum += h1;
                    __nv_bfloat162 pk = __floats2bfloat162_rn(h0, h1);
                    w[e2] = *reinterpret_cast<uint32_t*>(&pk);
                }
                const uint32_t chunk = (uint32_t)((c & 1) * 4 + ch);
                asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(rowaddr + ((chunk ^ ((uint32_t)r & 7u)) << 4)),
                             "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]) : "memory");
            }
        }
        tc_fence_before();                 // the accumulator has been read: GEMM 2' may overwrite it
        mbar_arrive_local(t_free);
        const float mean = sum * (1.f / kHidden);
        float sq = 0.f;
        float h[32];
        for (int c = 0; c < kHidden / 32; ++c) {
            load_h32(base, r, c, h);
#pragma unroll
            for (int e = 0; e < 32; ++e) { const float d = h[e] - mean; sq = fmaf(d, d, sq); }
        }
        const float rstd = rsqrtf(sq * (1.f / kHidden) + p.eps);

        ok = mbar_wait(t_full2, 0, p.abort_flag, 48) && ok;
        tc_fence_after();
        const bool poisoned = !ok || *(volatile int*)p.abort_flag != 0;
        // GEMM 2' has completed, so its ring is free: it holds the per-warp column sums [kPartRows][4 warps][512]
        float* colsum = reinterpret_cast<float*>(gen + kA2);
        auto stash = [&](int q, int c, float (&v)[32]) {
            const float t = column_sums32(v, lane);
            colsum[(q * 4 + quarter) * kHidden + c * 32 + lane] = t;
        };
        // ---- pass A: the two row means of gxh; column sums of gln * xh and gln ----
        float s1 = 0.f, s2 = 0.f;
        for (int c = 0; c < kHidden / 32; ++c) {
            tmem_ld32_raw(taddr + c * 32, buf);
            tmem_wait_ld();
            load_h32(base, r, c, h);
            float a[32], b[32];
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                const float gln = valid ? __uint_as_float(buf[e]) : 0.f;
                const float xh = (h[e] - mean) * rstd;
                const float gxh = gln * __ldg(p.ln_g + c * 32 + e);
                s1 += gxh; s2 = fmaf(gxh, xh, s2);
                a[e] = gln * xh; b[e] = gln;
            }
            stash(0, c, a);
            stash(1, c, b);
        }
        const float m1 = s1 * (1.f / kHidden), m2 = s2 * (1.f / kHidden);
        // ---- pass B: gh and ln rows out; column sums of gh ----
        __nv_bfloat16* gh_row = p.gh + (size_t)row * kHidden;
        __nv_bfloat16* ln_row = p.ln + (size_t)row * kHidden;
        for (int c = 0; c < kHidden / 32; ++c) {
            tmem_ld32_raw(taddr + c * 32, buf);
            tmem_wait_ld();
            load_h32(base, r, c, h);
            float gh[32], ln[32];
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                const int col = c * 32 + e;
                const float gln = valid ? __uint_as_float(buf[e]) : 0.f;
                const float xh = (h[e] - mean) * rstd;
                const float gxh = gln * __ldg(p.ln_g + col);
                gh[e] = rstd * (gxh - m1 - xh * m2);
                ln[e] = (h[e] - mean) * rstd * __ldg(p.ln_g + col) + __ldg(p.ln_b + col);     // the forward's expression
            }
            if (valid) { store_row32(gh_row + c * 32, gh, poisoned); store_row32(ln_row + c * 32, ln, poisoned); }
            stash(2, c, gh);
        }
        // ---- column sums of gy (d b2) ----
        for (int c = 0; c * 32 < p.Dout; ++c) {
            float g[32];
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {
                const int col0 = c * 32 + ch * 8;
                uint4 u = make_uint4(0u, 0u, 0u, 0u);
                if (valid && col0 < p.Dout) u = __ldg(reinterpret_cast<const uint4*>(p.gy + (size_t)row * p.Dout + col0));   // Dout % 16 == 0
                const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
                for (int e2 = 0; e2 < 4; ++e2) {
                    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[e2]));
                    g[ch * 8 + e2 * 2] = f.x; g[ch * 8 + e2 * 2 + 1] = f.y;
                }
            }
            stash(3, c, g);
        }
        tc_fence_before();
        // ---- the four warps' sums, in warp order: one partial row per tile ----
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const int t = threadIdx.x - 64;
        float* part = p.part + (size_t)blockIdx.x * kPartRows * kHidden;
        for (int k = t; k < kPartRows * kHidden; k += 128) {
            const int q = k / kHidden, col = k - q * kHidden;
            float v = colsum[(q * 4 + 0) * kHidden + col];
            v += colsum[(q * 4 + 1) * kHidden + col];
            v += colsum[(q * 4 + 2) * kHidden + col];
            v += colsum[(q * 4 + 3) * kHidden + col];
            part[k] = poisoned ? __int_as_float(0x7fc00000) : v;
        }
    }
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem_dealloc<1>(tmem0, 512); }
}

// d gamma, d beta, d b1 [512] and d b2 [Dout] (fp32): the tiles' partial rows added in tile order; NaN if the row
// pass's watchdog fired.  A NULL output is skipped.
__global__ void __launch_bounds__(256)
proj_bwd_finish_kernel(const float* __restrict__ part, int n_tiles, int Dout, float* dg, float* db, float* db1,
                       float* db2, const int* __restrict__ abort_flag) {
    const int k = blockIdx.x * 256 + threadIdx.x;
    if (k >= kPartRows * kHidden) return;
    const int q = k / kHidden, col = k - q * kHidden;
    float* out = q == 0 ? dg : q == 1 ? db : q == 2 ? db1 : db2;
    if (out == nullptr || (q == 3 && col >= Dout)) return;
    float v = 0.f;
#pragma unroll 8
    for (int t = 0; t < n_tiles; ++t) v += part[(size_t)t * kPartRows * kHidden + k];
    out[col] = *abort_flag != 0 ? __int_as_float(0x7fc00000) : v;
}

// ---- patch dropout compaction (src/model.py:268-308): kept patches to the front of each image, zero rows behind ----
// pos_s[n] = slot of patch n of image b among the image's kept patches (ballot prefix in patch order), or -1; returns
// the image's kept count.  Every thread of the 256-thread block calls it.
__device__ __forceinline__ int patch_slots(const uint8_t* __restrict__ keep, int b, int N, int* pos_s, int* warp_tot, int* carry_s) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) *carry_s = 0;
    __syncthreads();
    for (int n0 = 0; n0 < N; n0 += 256) {
        const int n = n0 + tid;
        const bool k = n < N && keep[(size_t)b * N + n] != 0;
        const unsigned m = __ballot_sync(0xffffffffu, k);
        if (lane == 0) warp_tot[warp] = __popc(m);
        __syncthreads();
        int off = *carry_s;
        for (int w = 0; w < warp; ++w) off += warp_tot[w];
        if (n < N) pos_s[n] = k ? off + __popc(m & ((1u << lane) - 1u)) : -1;
        __syncthreads();
        if (tid == 0) { int t = 0; for (int w = 0; w < 8; ++w) t += warp_tot[w]; *carry_s += t; }
        __syncthreads();
    }
    return *carry_s;
}

// one CTA per image; keep[b][n] != 0 marks a kept patch; out is [B][max_len][D]; rows are copied in 16-byte chunks
__global__ void __launch_bounds__(256)
patch_compact_kernel(const uint4* __restrict__ x, const uint8_t* __restrict__ keep, int N, int chunks, int max_len,
                     uint4* __restrict__ out) {
    extern __shared__ int pos_s[];                 // slot of patch n, or -1
    __shared__ int warp_tot[8];
    __shared__ int carry_s;
    const int b = blockIdx.x, tid = threadIdx.x;
    const int kept = patch_slots(keep, b, N, pos_s, warp_tot, &carry_s);
    const uint4* xb = x + (size_t)b * N * chunks;
    uint4* ob = out + (size_t)b * max_len * chunks;
    for (long long t = tid; t < (long long)N * chunks; t += 256) {
        const int n = (int)(t / chunks), c = (int)(t - (long long)n * chunks);
        const int ps = pos_s[n];
        if (ps >= 0) ob[(size_t)ps * chunks + c] = __ldg(xb + (size_t)n * chunks + c);
    }
    for (long long t = (long long)kept * chunks + tid; t < (long long)max_len * chunks; t += 256) ob[t] = make_uint4(0u, 0u, 0u, 0u);
}

// its backward: gx[b][n] = keep[b][n] ? gy[b][slot(n)] : 0, gy [B][max_len][D], gx [B][N][D]; a slot at or beyond max_len
// (a max_len smaller than the kept count, which the forward never produces) reads as zero
__global__ void __launch_bounds__(256)
patch_expand_kernel(const uint4* __restrict__ gy, const uint8_t* __restrict__ keep, int N, int chunks, int max_len,
                    uint4* __restrict__ gx) {
    extern __shared__ int pos_s[];
    __shared__ int warp_tot[8];
    __shared__ int carry_s;
    const int b = blockIdx.x, tid = threadIdx.x;
    patch_slots(keep, b, N, pos_s, warp_tot, &carry_s);
    const uint4* gb = gy + (size_t)b * max_len * chunks;
    uint4* xb = gx + (size_t)b * N * chunks;
    for (long long t = tid; t < (long long)N * chunks; t += 256) {
        const int n = (int)(t / chunks), c = (int)(t - (long long)n * chunks);
        const int ps = pos_s[n];
        xb[t] = (ps >= 0 && ps < max_len) ? __ldg(gb + (size_t)ps * chunks + c) : make_uint4(0u, 0u, 0u, 0u);
    }
}

}  // namespace proj
}  // namespace triad

using namespace triad;

extern "C" size_t triad_project_workspace_bytes(void) { return kCtrlBlockBytes; }

extern "C" int triad_project_tokens(const void* x, const void* w1, const float* b1, const float* ln_g, const float* ln_b,
                                    float ln_eps, const void* w2, const float* b2, int M, int Din, int Dout, int l2_normalize,
                                    void* out, void* ws, size_t ws_bytes, void* stream) {
    using namespace proj;
    if (!x || !w1 || !b1 || !ln_g || !ln_b || !w2 || !b2 || !out || !ws) return fail_msg(TRIAD_ERR_BAD_ARG, "project_tokens: null pointer");
    if (M <= 0 || Din <= 0 || Dout <= 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "project_tokens: bad shape");
    if (Din % kBlockK != 0 || Dout % 16 != 0 || Dout > kHidden)
        return fail_msg(TRIAD_ERR_UNSUPPORTED, "project_tokens: needs Din % 64 == 0, Dout % 16 == 0, Dout <= 512 (hidden width is 512)");
    if (((uintptr_t)x | (uintptr_t)w1 | (uintptr_t)w2 | (uintptr_t)out | (uintptr_t)ws) & 15) return fail_msg(TRIAD_ERR_ALIGNMENT, "project_tokens: 16-byte alignment");
    if (ws_bytes < kCtrlBlockBytes) return fail_msg(TRIAD_ERR_WORKSPACE, "project_tokens: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    TRIAD_CUDA_CHECK(cudaMemsetAsync(ws, 0, kCtrlBlockBytes, st));
    CUtensorMap mx, mw1, mw2;
    {
        cuuint64_t dims[2] = {(cuuint64_t)Din, (cuuint64_t)M};
        cuuint64_t strides[1] = {(cuuint64_t)Din * 2};
        cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)kBlockM};
        int rc = encode_tmap(&mx, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, x, 2, dims, strides, box, Swizzle::k128B);
        if (rc) return rc;
    }
    {
        cuuint64_t dims[2] = {(cuuint64_t)Din, (cuuint64_t)kHidden};
        cuuint64_t strides[1] = {(cuuint64_t)Din * 2};
        cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)kHalfN};
        int rc = encode_tmap(&mw1, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, w1, 2, dims, strides, box, Swizzle::k128B);
        if (rc) return rc;
    }
    {
        cuuint64_t dims[2] = {(cuuint64_t)kHidden, (cuuint64_t)Dout};
        cuuint64_t strides[1] = {(cuuint64_t)kHidden * 2};
        cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)kHalfN};
        int rc = encode_tmap(&mw2, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, w2, 2, dims, strides, box, Swizzle::k128B);
        if (rc) return rc;
    }
    Params p;
    p.b1 = b1; p.ln_g = ln_g; p.ln_b = ln_b; p.b2 = b2; p.out = (__nv_bfloat16*)out; p.abort_flag = (int*)ws;
    p.M = M; p.Din = Din; p.Dout = Dout; p.normalize = l2_normalize ? 1 : 0; p.eps = ln_eps;
    TRIAD_SET_MAX_SMEM(proj_head_kernel, kSmemBytes);
    proj_head_kernel<<<ceil_div(M, kBlockM), kThreads, kSmemBytes, st>>>(mx, mw1, mw2, p);
    TRIAD_LAUNCH_CHECK("proj_head_kernel");
    return TRIAD_OK;
}

// workspace of triad_project_tokens_bwd: [abort flag | gh bf16 [M][512] | ln bf16 [M][512] | partial rows | GEMM scratch]
struct BwdWs { size_t gh, ln, part, gemm, total; };
static BwdWs bwd_ws_layout(int M, int Din, int Dout) {
    using namespace proj;
    BwdWs w;
    w.gh = kCtrlBlockBytes;
    w.ln = w.gh + align_up((size_t)M * kHidden * 2, 256);
    w.part = w.ln + align_up((size_t)M * kHidden * 2, 256);
    w.gemm = w.part + align_up((size_t)ceil_div(M, kBlockM) * kPartRows * kHidden * 4, 256);
    size_t g = head_gemm_workspace_bytes(M, Dout, kHidden, 1);                 // dW2 = gy^T . ln
    const size_t g1 = head_gemm_workspace_bytes(M, kHidden, Din, 1);         // dW1 = gh^T . x
    const size_t g0 = head_gemm_workspace_bytes(M, kHidden, Din, 0);         // dx  = gh . W1
    if (g1 > g) g = g1;
    if (g0 > g) g = g0;
    w.total = w.gemm + g;
    return w;
}

extern "C" size_t triad_project_tokens_bwd_workspace_bytes(int M, int Din, int Dout) {
    if (M <= 0 || Din <= 0 || Dout <= 0) return 0;
    return bwd_ws_layout(M, Din, Dout).total;
}

extern "C" int triad_project_tokens_bwd(const void* x, const void* w1, const float* b1, const float* ln_g, const float* ln_b,
                                        float ln_eps, const void* w2, const void* gy, int M, int Din, int Dout,
                                        void* dx, float* dw1, float* db1, float* dln_g, float* dln_b, float* dw2, float* db2,
                                        void* ws, size_t ws_bytes, void* stream) {
    using namespace proj;
    if (!x || !w1 || !b1 || !ln_g || !ln_b || !w2 || !gy || !ws) return fail_msg(TRIAD_ERR_BAD_ARG, "project_tokens_bwd: null pointer");
    if (M <= 0 || Din <= 0 || Dout <= 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "project_tokens_bwd: bad shape");
    if (Din % kBlockK != 0 || Dout % 16 != 0 || Dout > kHidden)
        return fail_msg(TRIAD_ERR_UNSUPPORTED, "project_tokens_bwd: needs Din % 64 == 0, Dout % 16 == 0, Dout <= 512 (hidden width is 512)");
    if (((uintptr_t)x | (uintptr_t)w1 | (uintptr_t)w2 | (uintptr_t)gy | (uintptr_t)dx | (uintptr_t)dw1 | (uintptr_t)dw2 | (uintptr_t)ws) & 15)
        return fail_msg(TRIAD_ERR_ALIGNMENT, "project_tokens_bwd: 16-byte alignment");
    if (((uintptr_t)b1 | (uintptr_t)ln_g | (uintptr_t)ln_b | (uintptr_t)db1 | (uintptr_t)dln_g | (uintptr_t)dln_b | (uintptr_t)db2) & 3)
        return fail_msg(TRIAD_ERR_ALIGNMENT, "project_tokens_bwd: 4-byte alignment of the fp32 vectors");
    const BwdWs L = bwd_ws_layout(M, Din, Dout);
    if (ws_bytes < L.total) return fail_msg(TRIAD_ERR_WORKSPACE, "project_tokens_bwd: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    char* wsb = (char*)ws;
    __nv_bfloat16* gh = (__nv_bfloat16*)(wsb + L.gh);
    __nv_bfloat16* ln = (__nv_bfloat16*)(wsb + L.ln);
    float* part = (float*)(wsb + L.part);
    TRIAD_CUDA_CHECK(cudaMemsetAsync(ws, 0, kCtrlBlockBytes, st));
    CUtensorMap mx, mw1, mgy, mw2;
    int rc;
    {
        cuuint64_t dims[2] = {(cuuint64_t)Din, (cuuint64_t)M};
        cuuint64_t strides[1] = {(cuuint64_t)Din * 2};
        cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)kBlockM};
        if ((rc = encode_tmap(&mx, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, x, 2, dims, strides, box, Swizzle::k128B))) return rc;
    }
    {
        cuuint64_t dims[2] = {(cuuint64_t)Din, (cuuint64_t)kHidden};
        cuuint64_t strides[1] = {(cuuint64_t)Din * 2};
        cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)kHalfN};
        if ((rc = encode_tmap(&mw1, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, w1, 2, dims, strides, box, Swizzle::k128B))) return rc;
    }
    {                      // gy as GEMM 2's K-major A operand: {64 k, 128 rows}
        cuuint64_t dims[2] = {(cuuint64_t)Dout, (cuuint64_t)M};
        cuuint64_t strides[1] = {(cuuint64_t)Dout * 2};
        cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)kBlockM};
        if ((rc = encode_tmap(&mgy, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, gy, 2, dims, strides, box, Swizzle::k128B))) return rc;
    }
    {                      // W2 [Dout][512] as the MN-major B operand: {64 n, 64 k}
        cuuint64_t dims[2] = {(cuuint64_t)kHidden, (cuuint64_t)Dout};
        cuuint64_t strides[1] = {(cuuint64_t)kHidden * 2};
        cuuint32_t box[2] = {64, 64};
        if ((rc = encode_tmap(&mw2, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, w2, 2, dims, strides, box, Swizzle::k128B))) return rc;
    }
    BwdParams p;
    p.b1 = b1; p.ln_g = ln_g; p.ln_b = ln_b; p.gy = (const __nv_bfloat16*)gy;
    p.gh = gh; p.ln = ln; p.part = part; p.abort_flag = (int*)ws;
    p.M = M; p.Din = Din; p.Dout = Dout; p.eps = ln_eps;
    const int n_tiles = ceil_div(M, kBlockM);
    TRIAD_SET_MAX_SMEM(proj_head_bwd_kernel, kSmemBytes);
    proj_head_bwd_kernel<<<n_tiles, kThreads, kSmemBytes, st>>>(mx, mw1, mgy, mw2, p);
    TRIAD_LAUNCH_CHECK("proj_head_bwd_kernel");
    if (dln_g || dln_b || db1 || db2) {
        proj_bwd_finish_kernel<<<kPartRows * kHidden / 256, 256, 0, st>>>(part, n_tiles, Dout, dln_g, dln_b, db1, db2, (const int*)ws);
        TRIAD_LAUNCH_CHECK("proj_bwd_finish_kernel");
    }
    void* gws = wsb + L.gemm;
    const size_t gws_bytes = ws_bytes - L.gemm;
    if (dw2 && (rc = launch_head_gemm(gy, Dout, M, Dout, ln, kHidden, 1, dw2, 1, gws, gws_bytes, st))) return rc;
    if (dw1 && (rc = launch_head_gemm(gh, kHidden, M, kHidden, x, Din, 1, dw1, 1, gws, gws_bytes, st))) return rc;
    if (dx && (rc = launch_head_gemm(gh, kHidden, M, kHidden, w1, Din, 0, dx, 0, gws, gws_bytes, st))) return rc;
    return TRIAD_OK;
}

extern "C" int triad_patch_compact(const void* x, const uint8_t* keep, int B, int N, int D, int elt_bytes, int max_len,
                                   void* out, void* stream) {
    if (!x || !keep || !out) return fail_msg(TRIAD_ERR_BAD_ARG, "patch_compact: null pointer");
    if (B <= 0 || N <= 0 || D <= 0 || max_len < 0 || (D * elt_bytes) % 16 != 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "patch_compact: bad shape (row bytes % 16)");
    if (((uintptr_t)x | (uintptr_t)out) & 15) return fail_msg(TRIAD_ERR_ALIGNMENT, "patch_compact: 16-byte alignment");
    if (max_len == 0) return TRIAD_OK;
    if ((size_t)N * 4 > 200 * 1024) return fail_msg(TRIAD_ERR_UNSUPPORTED, "patch_compact: too many patches per image");
    auto kern = proj::patch_compact_kernel;
    if ((size_t)N * 4 > 48 * 1024) TRIAD_SET_MAX_SMEM(kern, N * 4);
    kern<<<B, 256, (size_t)N * 4, (cudaStream_t)stream>>>((const uint4*)x, keep, N, D * elt_bytes / 16, max_len, (uint4*)out);
    TRIAD_LAUNCH_CHECK("patch_compact_kernel");
    return TRIAD_OK;
}

extern "C" int triad_patch_expand(const void* gy, const uint8_t* keep, int B, int N, int D, int elt_bytes, int max_len,
                                  void* gx, void* stream) {
    if (!gy || !keep || !gx) return fail_msg(TRIAD_ERR_BAD_ARG, "patch_expand: null pointer");
    if (B <= 0 || N <= 0 || D <= 0 || max_len < 0 || (D * elt_bytes) % 16 != 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "patch_expand: bad shape (row bytes % 16)");
    if (((uintptr_t)gy | (uintptr_t)gx) & 15) return fail_msg(TRIAD_ERR_ALIGNMENT, "patch_expand: 16-byte alignment");
    if ((size_t)N * 4 > 200 * 1024) return fail_msg(TRIAD_ERR_UNSUPPORTED, "patch_expand: too many patches per image");
    auto kern = proj::patch_expand_kernel;
    if ((size_t)N * 4 > 48 * 1024) TRIAD_SET_MAX_SMEM(kern, N * 4);
    kern<<<B, 256, (size_t)N * 4, (cudaStream_t)stream>>>((const uint4*)gy, keep, N, D * elt_bytes / 16, max_len, (uint4*)gx);
    TRIAD_LAUNCH_CHECK("patch_expand_kernel");
    return TRIAD_OK;
}
