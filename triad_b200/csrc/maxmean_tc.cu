// tcgen05 / TMEM / TMA forward of the max-mean similarity for bf16 inputs (sm_100a).
//
// Replaces src/model.py:384-391 (AV) and :502-512 (TV): the reference clones both operands B
// times, runs a batched GEMM with batch B^2 and sweeps the resulting Bq x Bv x Nq x Nv tensor
// four more times (*T, max, mean).  Here that tensor only ever exists as 128 x Nv fp32
// accumulator tiles in tensor memory:
//
//   * rows   = query tokens, flattened over the batch (M = Bq*Nq), 128 per CTA = the 128 TMEM lanes;
//   * cols   = the Nv patches of ONE image (UMMA N = Nv rounded up to 16, <= 256); images with more
//              patches (high-resolution DINOv2: 1024) are walked as consecutive 256-patch SUB-TILES and
//              the epilogue keeps a running (rounded max, first argmax) per row across them;
//   * K      = D (<= 512) in 64-element (128-byte, SWIZZLE_128B) k-blocks.
//
// Work decomposition (persistent, one CTA or CTA pair per SM / SM pair):
//   the (m-tile, image) space is linearised image-chunk-major, m-tile, image-in-chunk and cut
//   into equal contiguous ranges, so a CTA keeps its 128 x D QUERY tile stationary in shared
//   memory (128 KB) while it streams images, and all CTAs walk the same chunk of images at the
//   same time (L2 reuse of V when V does not fit in L2).  Only V k-blocks go through the
//   multi-stage TMA ring.  With cta_group::2 the pair shares each V tile (each CTA loads half
//   of the patches), halving L2->SMEM traffic per SM.
//
// Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane), warp 2 = TMEM
// allocator, warps 4-7 = epilogue (TMEM lane quarter = warp & 3).  Accumulators are double
// buffered in TMEM (2 x 256 columns) so the epilogue of tile t overlaps the MMAs of tile t+1.
//
// Epilogue (per thread = one token row): pass 1 fmax over the Nv raw accumulators; the exact
// first-argmax threshold of triad_round.h; pass 2 finds the first column >= threshold (this
// reproduces torch.max's first-index tie-break on the double-rounded bf16 values bit-exactly);
// then a deterministic segmented shuffle reduction over the 32 rows of the warp into
// per-(image, 32-row group, query) partial sums (common.cuh).
#include "common.cuh"
#include "ptx.cuh"

#include <cuda.h>
#include <string.h>

namespace triad {
namespace tc {

using namespace ptx;

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;            // bf16 per 128-byte swizzle row
constexpr int kUmmaK = 16;
constexpr int kMaxKB = 8;              // D <= 512
constexpr int kMaxN = 256;
constexpr int kThreads = 256;
constexpr int kEpiWarp0 = 4;
constexpr int kTmemCols = 512;
constexpr uint32_t kQkbBytes = kBlockM * kBlockK * 2;        // 16 KB
constexpr uint32_t kQBytes = kMaxKB * kQkbBytes;             // 128 KB
constexpr uint32_t kVRingBytes = 96 * 1024;
constexpr uint32_t kBarBytes = 1024;          // mbarriers, the TMEM base, and the 512-byte argmax exchange of the epilogue pairs
constexpr uint32_t kSmemBytes = kQBytes + kVRingBytes + kBarBytes + 1024;   // + alignment slack

struct Params {
    int M, Bv, Nq, Nv;
    int n_umma;        // UMMA N (Nv rounded up to 16; 256 when the image is split into sub-tiles)
    int n_sub;         // 256-patch sub-tiles per image (1 when Nv <= 256)
    int idx16;         // idx elements are uint16 (Nv > 256)
    int num_kb;        // D / 64
    int n_m;           // number of (128*cta_group)-row tiles
    int C;             // images per chunk
    int sync;          // TileIter mode: all clusters walk the same image chunk at the same time
    int G, S;          // partial layout
    int nq_pad;        // idx row pitch per query
    int inv_T;
    const float* row_scale;
    const float* T;
    float* part;
    uint8_t* idx;
    int* abort_flag;
    // packed rows (pack.cu): the GEMM rows are the kept rows only; maps = off[Bq+1] | rowmap[M], M' = off[Bq]
    const int* pack_off;     // NULL = rows are the original rows
    const int* rowmap;
    int Bq;
    int pieces;              // packed partial layout: part[(j*Bq + i)*pieces + (group - first group of query i)]
    // kEmitN (dense regulariser, dense_reg.cu): the epilogue writes N = dL/d<q,v> of the non-negative pressure
    // term for every (row, patch) instead of reducing the tile
    __nv_bfloat16* n_out;    // [M][ldn] bf16; image j of this call occupies columns [j*Nv, (j+1)*Nv)
    long long ldn;
    float lo, coef;          // clamp floor (< 0), 2*weight/numel
    int write_n;             // 0: value only
    double* n_partials;      // [gridDim.x*8][2]: sum clamp^2, sum dS*<q,v>; slot blockIdx.x*8 + (warp - 4), written by the
                             // emission warps 8-11 (slots of the other epilogue warps stay as cleared)
    // kFp8 (e4m3 retrieval): per-patch scales [Bv][Nv] of the gallery codes, per-token scales [M] of the query codes
    const float* col_scale;
    const float* q_scale;
    // kMode 3 / 4 (ragged caption gallery, ragged.cu): per-slot metadata [slots][kSlotMetaInts] and per-caption
    // {first slot row, length} [captions]
    const int* slot_meta;
    const int* cap_info;
};

__device__ __forceinline__ float fmax3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }

// maximum of one 32-column chunk of a row; columns >= Nv (TMA zero fill / stale TMEM) do not take part
__device__ __forceinline__ float chunk_max32(const uint32_t (&r)[32], int col0, int Nv) {
    float v[32];
#pragma unroll
    for (int e = 0; e < 32; ++e) v[e] = __uint_as_float(r[e]);
    if (col0 + 32 > Nv) {
#pragma unroll
        for (int e = 0; e < 32; ++e) if (col0 + e >= Nv) v[e] = -INFINITY;
    }
    float m[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {                       // four independent chains of 8
        m[k] = fmax3(v[8 * k], v[8 * k + 1], v[8 * k + 2]);
        m[k] = fmax3(m[k], v[8 * k + 3], v[8 * k + 4]);
        m[k] = fmax3(m[k], v[8 * k + 5], v[8 * k + 6]);
        m[k] = fmaxf(m[k], v[8 * k + 7]);
    }
    return fmaxf(fmax3(m[0], m[1], m[2]), m[3]);
}

// maximum that returns NaN when either operand is NaN (fmaxf drops it): a NaN patch scale must reach the score
__device__ __forceinline__ float fmax_nan(float a, float b) {
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
// e4m3 epilogue: maximum over one 32-column chunk of sg[c] * acc[c], the patch scales sg of the chunk's columns read
// from shared memory (the same address in every lane: a broadcast); columns >= Nv do not take part, a NaN product does.
// Scaled and reduced four columns at a time, so the products never occupy a second 32-register buffer.
__device__ __forceinline__ float chunk_max32_scaled(const uint32_t (&r)[32], const float4* sg, int col0, int Nv) {
    const bool part = col0 + 32 > Nv;
    float m[4];
#pragma unroll
    for (int g = 0; g < 8; ++g) {
        const float4 s = sg[g];
        float v0 = __uint_as_float(r[4 * g]) * s.x, v1 = __uint_as_float(r[4 * g + 1]) * s.y;
        float v2 = __uint_as_float(r[4 * g + 2]) * s.z, v3 = __uint_as_float(r[4 * g + 3]) * s.w;
        if (part) {
            if (col0 + 4 * g >= Nv) v0 = -INFINITY;
            if (col0 + 4 * g + 1 >= Nv) v1 = -INFINITY;
            if (col0 + 4 * g + 2 >= Nv) v2 = -INFINITY;
            if (col0 + 4 * g + 3 >= Nv) v3 = -INFINITY;
        }
        const float a = fmax_nan(fmax_nan(v0, v1), fmax_nan(v2, v3));
        m[g & 3] = g < 4 ? a : fmax_nan(m[g & 3], a);                // four independent chains
    }
    return fmax_nan(fmax_nan(m[0], m[1]), fmax_nan(m[2], m[3]));
}

// best = lowest column of this chunk with value >= theta, if any (columns >= Nv never qualify)
__device__ __forceinline__ void first_ge32(const uint32_t (&r)[32], int col0, int Nv, float theta, int& best) {
    const int lim = Nv - col0;                          // >= 32 for every chunk but the last partial one
    int b[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {                       // four independent chains of 8 (descending: lowest sticks)
        b[k] = 64;
#pragma unroll
        for (int e = 7; e >= 0; --e) if (__uint_as_float(r[8 * k + e]) >= theta) b[k] = 8 * k + e;
    }
    const int lo = min(min(b[0], b[1]), min(b[2], b[3]));
    if (lo < min(lim, 32)) best = col0 + lo;            // 64 = "none"; columns >= lim are padding
}

// ---- ragged caption gallery, direction 0 (kMode 3): segmented row maximum over one 256-row slot -------------------
// r[b] of a 32-column chunk, b warp-uniform but not a compile-time constant: a five-level select tree keeps r in
// registers (an indexed access would put it in local memory)
__device__ __forceinline__ float pick32(const uint32_t (&r)[32], int b) {
    uint32_t a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = (b & 1) ? r[2 * i + 1] : r[2 * i];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = (b & 2) ? a[2 * i + 1] : a[2 * i];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = (b & 4) ? a[2 * i + 1] : a[2 * i];
#pragma unroll
    for (int i = 0; i < 2; ++i) a[i] = (b & 8) ? a[2 * i + 1] : a[2 * i];
    return __uint_as_float((b & 16) ? a[1] : a[0]);
}
// One 32-column chunk of the slot: `starts` / `ends` are the chunk's words of the slot's caption-start and
// caption-end masks (warp-uniform).  A running maximum restarts at every caption start; r[i] becomes the maximum of
// the open caption up to column i, so at every end column it is that caption's row maximum.  Each caption that ends
// in the chunk is weighted (val = round_sim(max) * row weight, as the dense epilogue) and reduced over the warp's 32
// query rows into its partial part[caption][32-row group] (store_group_partials with one slot per group), captions
// numbered from `cap` in slot order.
__device__ __forceinline__ void ragged_chunk(uint32_t (&r)[32], uint32_t starts, uint32_t ends, float& run, int& cap,
                                             bool valid, float Tval, float rs, const Params& p, int row0, int lane) {
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        const float x = __uint_as_float(r[i]);
        run = ((starts >> i) & 1u) ? x : fmaxf(run, x);
        r[i] = __float_as_uint(run);
    }
    while (ends != 0u) {                                    // warp-uniform: one iteration per caption ending here
        const int b = __ffs(ends) - 1;
        ends &= ends - 1u;
        const float val = valid ? round_sim<true>(pick32(r, b), Tval) * rs : 0.f;
        store_group_partials(p.part, cap, row0 >> 5, p.G, 1, row0, p.M, p.Nq, val, lane);
        ++cap;
    }
}
// e4m3 variant (kFp8): every column is first multiplied by its slot-row scale sg[c] (broadcast from shared memory, as
// chunk_max32_scaled), the running maximum propagates NaN, and a caption's maximum is weighted by the row factor
// rs = t_a with no bf16 rounding.  A caption row with a NaN scale makes that caption's maximum NaN and no other's,
// since the running maximum restarts at every caption start.
__device__ __forceinline__ void ragged_chunk_scaled(uint32_t (&r)[32], const float4* sg, uint32_t starts, uint32_t ends,
                                                    float& run, int& cap, bool valid, float rs, const Params& p, int row0,
                                                    int lane) {
#pragma unroll
    for (int g = 0; g < 8; ++g) {
        const float4 s = sg[g];
        const float sc[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int i = 4 * g + e;
            const float x = __uint_as_float(r[i]) * sc[e];
            run = ((starts >> i) & 1u) ? x : fmax_nan(run, x);
            r[i] = __float_as_uint(run);
        }
    }
    while (ends != 0u) {
        const int b = __ffs(ends) - 1;
        ends &= ends - 1u;
        const float val = valid ? pick32(r, b) * rs : 0.f;
        store_group_partials(p.part, cap, row0 >> 5, p.G, 1, row0, p.M, p.Nq, val, lane);
        ++cap;
    }
}

// ---- dense-regulariser epilogue (kMode 1: instead of the max-mean reduction; kMode 2: next to it) -----------------
// N = coef*T*min(T*acc, 0) = (coef*T^2) * min(acc, 0) for T > 0, written as bf16.  A thread owns a ROW of the
// accumulator, so storing straight from registers would hit 32 different rows per store instruction.  Each emission
// warp instead stages a 32-row x 64-column box (4 KB, the SWIZZLE_128B layout of a TMA box: 16-byte piece c of row
// r sits at piece c ^ (r & 7), so the 32 lanes' st.shared.v4 are conflict-free) and ONE lane hands it to the TMA
// unit (cp.async.bulk.tensor store): no per-lane global stores, no address arithmetic, and rows >= M / columns >= Nv
// are clipped by the tensor map {Nv, images, M}.  Round 1's version (per-lane 16-byte stores out of a transposing
// staging buffer) spent 4 dependent STS -> LDS -> STG round trips per chunk: 3.8 ms per pass against 2.45 ms for
// the plain forward.
constexpr int kEmitThreads = (kEpiWarp0 + kEmitEpiWarps) * 32;      // 384
constexpr uint32_t kStgBytesPerWarp = 32 * 128;                     // one 32 x 64 bf16 box
constexpr uint32_t kStgBytes = 4 * 2 * kStgBytesPerWarp;            // four emission warps x two boxes: 32 KB, carved
                                                                    // from the end of the V ring
constexpr uint16_t kNoCol = 0xffffu;                                // "no column of my half reaches the threshold"

__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ float fmin3(float a, float b, float c) { return fminf(fminf(a, b), c); }
// compensated (Kahan) fp32 accumulation: s + c-correction carries ~fp64 accuracy over a few thousand terms
__device__ __forceinline__ void kahan_add(float& s, float& c, float x) {
    const float y = x - c;
    const float t = s + y;
    c = (t - s) - y;
    s = t;
}
__device__ __forceinline__ void ffma2(float2& acc, float2 a, float2 b) {
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(reinterpret_cast<unsigned long long&>(acc))
        : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    float2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<unsigned long long&>(r))
        : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
    return r;
}

// One 32-column chunk of the warp's 32 rows, fast path: n = min(acc, 0); a2 += n^2 (two packed chains; the tile's sum
// is scaled by T^2 afterwards); mn = row minimum (to detect the clamp floor); bf16(n * cT2) into the staging box
// (`sub` = which 64-byte half of the 128-byte staged row).  Columns >= Nv (stale TMEM beyond n_umma) are zeroed in
// the last, partial chunk only (kFull = false).
template <bool kFull>
__device__ __forceinline__ void emit_chunk_t(const uint32_t (&r)[32], int col0, int Nv, float2 cT2, float2 (&a2)[2],
                                             float (&mn)[2], uint32_t (&w)[16]) {
#pragma unroll
    for (int e = 0; e < 32; e += 2) {
        float x0 = __uint_as_float(r[e]), x1 = __uint_as_float(r[e + 1]);
        if constexpr (!kFull) { if (col0 + e >= Nv) x0 = 0.f; if (col0 + e + 1 >= Nv) x1 = 0.f; }
        const float2 n = make_float2(fminf(x0, 0.f), fminf(x1, 0.f));
        ffma2(a2[(e >> 1) & 1], n, n);
        mn[(e >> 1) & 1] = fmin3(mn[(e >> 1) & 1], n.x, n.y);
        const float2 o = fmul2(n, cT2);
        __nv_bfloat162 hh = __floats2bfloat162_rn(o.x, o.y);
        w[e >> 1] = *reinterpret_cast<uint32_t*>(&hh);
    }
}
__device__ __forceinline__ void emit_chunk(const uint32_t (&r)[32], int col0, int Nv, float2 cT2, float2 (&a2)[2],
                                           float (&mn)[2], uint32_t (&w)[16]) {
    if (col0 >= Nv) return;                                         // warp-uniform; the staged half is clipped by TMA
    if (col0 + 32 <= Nv) emit_chunk_t<true>(r, col0, Nv, cT2, a2, mn, w);
    else emit_chunk_t<false>(r, col0, Nv, cT2, a2, mn, w);
}
// the chunk's 32 bf16 (64 bytes) of this lane's row into the staging box; `sub` = which half of the 128-byte row
__device__ __forceinline__ void stage_chunk(const uint32_t (&w)[16], uint32_t stg_row, int lane, int sub) {
#pragma unroll
    for (int g = 0; g < 4; ++g)
        sts128(stg_row + ((uint32_t)((sub * 4 + g) ^ (lane & 7)) << 4), w[4 * g], w[4 * g + 1], w[4 * g + 2], w[4 * g + 3]);
}
// Exact variant of one chunk (some similarity of the warp's rows is at the clamp floor `lo`): near the floor the
// reference's own rounding decides the gradient gate — token_sims is bf16(bf16(<q,v>) * T) under autocast
// (model.py:387), clamp and its gradient act on that.  e2 += clamp(S,lo,0)^2, eT += dS * <q,v> (both unscaled by coef).
__device__ __forceinline__ void emit_chunk_exact(const uint32_t (&r)[32], int col0, int Nv, float Tval, float coefT, float lo,
                                                 float& e2, float& eT, uint32_t (&w)[16]) {
    if (col0 >= Nv) return;
#pragma unroll
    for (int e = 0; e < 32; e += 2) {
        float o[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const float raw = __bfloat162float(__float2bfloat16_rn(__uint_as_float(r[e + h])));
            const float sv = (col0 + e + h < Nv) ? __bfloat162float(__float2bfloat16_rn(raw * Tval)) : 0.f;
            const float n = fminf(sv, 0.f);
            const float nc = fmaxf(n, lo);
            e2 = fmaf(nc, nc, e2);
            const float pass = (sv >= lo) ? n : 0.f;
            eT = fmaf(pass, raw, eT);
            o[h] = pass * coefT;
        }
        __nv_bfloat162 hh = __floats2bfloat162_rn(o[0], o[1]);
        w[e >> 1] = *reinterpret_cast<uint32_t*>(&hh);
    }
}
// the staged box -> N[row0 .. row0+32)[image j][col0 .. col0+64): the writes of all 32 lanes are made visible to the
// async proxy, then one lane issues the bulk tensor store and commits it as a bulk group
__device__ __forceinline__ void emit_box_store(const CUtensorMap* tmap_n, uint32_t stg, int col0, int j, int row0, int lane) {
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
        asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                     ::"l"(reinterpret_cast<uint64_t>(tmap_n)), "r"(stg), "r"(col0), "r"(j), "r"(row0) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
}
// before the staging box is written again: the TMA unit must have READ the previous one
__device__ __forceinline__ void emit_box_reusable(int lane) {
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
}
// all of this warp's bulk stores have been performed (before generic stores to the same addresses / kernel exit)
__device__ __forceinline__ void emit_box_drain(int lane) {
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    __syncwarp();
}

struct Tile { int m, j; };
__device__ __forceinline__ Tile decode_tile(uint32_t L, int n_m, int Bv, int C) {
    const uint32_t per_chunk = (uint32_t)n_m * (uint32_t)C;
    const uint32_t full = (uint32_t)Bv / (uint32_t)C;
    uint32_t jc = L / per_chunk;
    Tile t;
    if (jc < full) {
        const uint32_t rem = L - jc * per_chunk;
        t.m = (int)(rem / (uint32_t)C);
        t.j = (int)(jc * C + rem % (uint32_t)C);
    } else {
        const uint32_t rem = L - full * per_chunk;
        const uint32_t cl = (uint32_t)Bv - full * (uint32_t)C;
        t.m = (int)(rem / cl);
        t.j = (int)(full * C + rem % cl);
    }
    return t;
}

// The sequence of (m-tile, image) work items of one cluster; the three warp roles walk it in lockstep.
//   sync == 0: one contiguous range of the chunk-major linearisation (chunks of C images; C = 1..64 for a huge
//              gallery with few query tiles, C = Bv when V is small) — a cluster keeps to its own images and
//              changes its query tile as rarely as the chunking allows;
//   sync == 1: every image chunk is cut into one range per cluster, so ALL clusters stream the SAME chunk of
//              C images at the same time — V is then read from HBM once per pass over the chunk, whatever
//              its total size (B = 8192: 2.1 GB), at the price of re-loading the (small) query tiles per chunk.
// launch_maxmean_tc() picks the mode from the size of V and the number of query tiles.
struct TileIter {
    uint32_t n_m, Bv, C, cid, ncl, sync;
    uint32_t L, Lend, j0, cl;
    __device__ __forceinline__ void range(uint32_t per) {
        L = (uint32_t)(((unsigned long long)per * cid) / ncl);
        Lend = (uint32_t)(((unsigned long long)per * (cid + 1)) / ncl);
    }
    __device__ __forceinline__ void init(int n_m_, int Bv_, int C_, int sync_, uint32_t cid_, uint32_t ncl_) {
        n_m = (uint32_t)n_m_; Bv = (uint32_t)Bv_; C = (uint32_t)C_; sync = (uint32_t)sync_; cid = cid_; ncl = ncl_;
        j0 = 0; cl = min(C, Bv);
        range(sync ? n_m * cl : n_m * Bv);
    }
    __device__ __forceinline__ bool next(Tile& t) {
        if (!sync) {
            if (L >= Lend) return false;
            t = decode_tile(L++, (int)n_m, (int)Bv, (int)C);
            return true;
        }
        while (L >= Lend) {
            j0 += C;
            if (j0 >= Bv) return false;
            cl = min(C, Bv - j0);
            range(n_m * cl);
        }
        t.m = (int)(L / cl);
        t.j = (int)(j0 + L % cl);
        ++L;
        return true;
    }
};

// ---------------------------------------------------------------------------------------------
// kernel
// ---------------------------------------------------------------------------------------------
// kSub = false: one accumulator tile per image (Nv <= 256), the training shapes' hot path;
// kSub = true : n_sub 256-patch sub-tiles per image.
// kMode 0: max-mean reduction (the contrastive forward / retrieval); 2: BOTH the max-mean reduction (warps 4-7) and
// the dense regulariser (emission warps 8-11 write N = dL/d<q,v> of the non-negative pressure term) in one pass over
// the similarities — the training step with the reference's full loss needs both of the very same tiles; 1: kMode 2
// without the max-mean warps (the regulariser-only pass).
// kFp8: e4m3 operands (kMode 0, 3 or 4, no idx: the retrieval forward on a quantized gallery).  A 128-byte swizzle row then
// holds 128 elements, so a k-block is 128 wide (num_kb = D/128 <= 4) and one kind::f8f6f4 MMA step covers K = 32;
// the ring, the descriptors and the issue loops are those of bf16.  The epilogue multiplies every column by its
// patch scale before the max and the row by t_a = fp32(fp32(q_scale * row_scale) * (1/T)) after it.  The scales of
// the current 256-patch sub-tile are staged per epilogue warp in the upper half of the query region (num_kb <= 4
// leaves it unused).
// kMode 3 / 4: a ragged caption gallery (ragged.cu), stored as 256-row slots that each hold whole captions.
//   kMode 3 (direction 0: mean over the query's tokens of the max over each caption's tokens): rows = the query's
//   tokens, "images" = the slots (Nv = 256).  The epilogue walks each row's 256 columns with a running maximum that
//   restarts at every caption start (ragged_chunk) and reduces each caption's row maxima over the warp's 32 rows into
//   part[caption][group]; no idx.
//   kMode 4 (direction 1: mean over each caption's tokens of the max over the query's tokens): rows = the slot rows,
//   the one "image" = the query (sub-tiles when it has more than 256 tokens).  The row's caption and its weight
//   1/length come from the slot metadata in place (the gallery is not copied); each slot row's weighted maximum is
//   stored as it is, part[row] (the zero rows at a slot's end store nothing), and the finalize sums each caption's
//   rows in token order.  A warp reduction would add a caption's rows in an order set by its offset within a 32-row
//   group, so the same caption packed after another prefix could score differently in the last bit; this order
//   depends on the caption alone.  cta_group::2 only (the rows are whole 256-row slots).
//   With kFp8 the column scales are the slot-row scales in kMode 3 (ragged_chunk_scaled) and the query's token scales
//   in kMode 4, where the row weight becomes w_t = fp32(fp32(s_t * (1/length)) * (1/T)) with s_t the slot row's scale.
constexpr int kModeRaggedMax = 3, kModeRaggedMean = 4;
template <int kCtaGroup, bool kSub, int kMode = 0, bool kFp8 = false>
__global__ void __launch_bounds__(kEmitThreads, 1)
maxmean_tc_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_v,
                  const __grid_constant__ CUtensorMap tmap_n, const Params p) {
    static_assert(!kFp8 || kMode == 0 || kMode == kModeRaggedMax || kMode == kModeRaggedMean,
                  "the e4m3 forward is the max-mean reduction, dense or ragged, only");
    static_assert(kMode != kModeRaggedMax || !kSub, "ragged direction 0: one 256-row slot per tile");
    constexpr bool kEmitN = kMode == 1 || kMode == 2;
    constexpr bool kRagged = kMode == kModeRaggedMax || kMode == kModeRaggedMean;
    constexpr int kKbElems = kFp8 ? 128 : kBlockK;                          // elements per 128-byte k-block row
    constexpr int kVStageBytes = (kMaxN / kCtaGroup) * kBlockK * 2;       // 32 KB / 16 KB
    // the dense-regulariser modes give the last 32 KB of the ring to the epilogue's store staging: four emission warps x
    // two 4 KB boxes (32 rows x 64 columns).  (Two 2 KB boxes of 32 columns per emission warp, i.e. 5 ring stages
    // instead of 4, were measured: no faster, twice the bulk stores.)
    constexpr uint32_t kStgTotal = kEmitN ? kStgBytes : 0u;
    constexpr int kStages = (kVRingBytes - kStgTotal) / kVStageBytes;                  // 3 / 6  (2 / 4)
    constexpr int kTileRows = kBlockM * kCtaGroup;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t q_smem = smem_base;
    const uint32_t v_smem = smem_base + kQBytes;
    const uint32_t bar_base = v_smem + kVRingBytes;
    // barrier map (8 bytes each)
    const uint32_t bar_q_full = bar_base;                       // [kMaxKB]
    const uint32_t bar_q_empty = bar_q_full + 8 * kMaxKB;       // [1]
    const uint32_t bar_v_full = bar_q_empty + 8;                // [kStages]
    const uint32_t bar_v_empty = bar_v_full + 8 * kStages;      // [kStages]
    const uint32_t bar_t_full = bar_v_empty + 8 * kStages;      // [2]
    const uint32_t bar_t_empty = bar_t_full + 16;               // [2]
    const uint32_t tmem_ptr_smem = bar_t_empty + 16;            // u32
    const uint32_t xch_smem = bar_base + 512;                   // u16 [2 parities][128 rows]: epilogue pair exchange
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_ptr_smem - smem_base));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t cta_rank = (kCtaGroup == 2) ? cluster_ctarank() : 0u;
    const bool is_leader = (cta_rank == 0);
    const uint32_t cluster_id = blockIdx.x / kCtaGroup;
    const uint32_t n_clusters = gridDim.x / kCtaGroup;

    // work items are (m-tile, image) pairs; each is n_sub consecutive accumulator tiles
    // packed rows: the number of kept rows is only known on the device (no host synchronisation)
    const int M_eff = p.pack_off ? p.pack_off[p.Bq] : p.M;
    const int n_m_eff = p.pack_off ? (M_eff + kBlockM * kCtaGroup - 1) / (kBlockM * kCtaGroup) : p.n_m;
    TileIter it;
    it.init(n_m_eff, p.Bv, p.C, p.sync, cluster_id, n_clusters);
    const int n_sub = kSub ? p.n_sub : 1;

    const int n_half = p.n_umma / kCtaGroup;                    // patch rows this CTA loads per image
    const uint32_t v_tx_bytes = (uint32_t)n_half * kBlockK * 2u;

    // ---- one-time setup -------------------------------------------------------------------
    if (warp == 0 && lane == 0) { prefetch_tmap(&tmap_q); prefetch_tmap(&tmap_v); }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < kMaxKB; ++i) mbar_init(bar_q_full + 8 * i, 1);
        mbar_init(bar_q_empty, 1);
        for (int i = 0; i < kStages; ++i) { mbar_init(bar_v_full + 8 * i, 1); mbar_init(bar_v_empty + 8 * i, 1); }
        // arrivals that free an accumulator: kMode 2 its four max-mean and four emission warps, kMode 1 the four
        // emission warps, kMode 0 the eight max-mean warps (four when no idx is wanted: the upper halves sit out)
        const int t_empty_warps = kMode == 2 ? 8 : kMode == 1 ? 4 : (p.idx != nullptr ? 8 : 4);
        for (int i = 0; i < 2; ++i) { mbar_init(bar_t_full + 8 * i, 1); mbar_init(bar_t_empty + 8 * i, t_empty_warps * kCtaGroup); }
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc<kCtaGroup>(tmem_ptr_smem, kTmemCols);
    tc_fence_before();
    if constexpr (kCtaGroup == 2) { cluster_arrive(); cluster_wait(); } else { __syncthreads(); }
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_gen;

    if (warp == 0) {
        // =============================== TMA producer ===================================
        // (whole warp in the loop, one elected lane issues — see the MMA role)
        {
            const bool issuer = elect_one();
            // in a pair, every load signals the LEADER's barrier (the only MMA issuer waits there)
            const uint32_t q_full_sig = (kCtaGroup == 2) ? mapa(bar_q_full, 0) : bar_q_full;
            const uint32_t v_full_sig = (kCtaGroup == 2) ? mapa(bar_v_full, 0) : bar_v_full;
            int stage = 0; uint32_t phase = 0, qe_phase = 0; int prev_m = -1;
            bool ok = true;
            Tile t;
            while (ok && it.next(t)) {
                const bool new_m = (t.m != prev_m);
                if (new_m && prev_m >= 0) {
                    ok = mbar_wait(bar_q_empty, qe_phase, p.abort_flag, 1);
                    qe_phase ^= 1;
                    if (!ok) break;
                }
                for (int sb = 0; sb < n_sub && ok; ++sb) {
                    for (int kb = 0; kb < p.num_kb; ++kb) {
                        if (new_m && sb == 0 && issuer) {
                            if (is_leader) mbar_expect_tx(bar_q_full + 8 * kb, kQkbBytes * kCtaGroup);
                            tma_load_2d<kCtaGroup>(q_smem + kb * kQkbBytes, &tmap_q, q_full_sig + 8 * kb,
                                                   kb * kKbElems, t.m * kTileRows + (int)cta_rank * kBlockM);
                        }
                        ok = mbar_wait(bar_v_empty + 8 * stage, phase ^ 1, p.abort_flag, 2);
                        if (!ok) break;
                        if (issuer) {
                            if (is_leader) mbar_expect_tx(bar_v_full + 8 * stage, v_tx_bytes * kCtaGroup);
                            // patches beyond Nv (last sub-tile) are zero-filled by TMA and masked in the epilogue
                            tma_load_3d<kCtaGroup>(v_smem + stage * kVStageBytes, &tmap_v, v_full_sig + 8 * stage,
                                                   kb * kKbElems, sb * kMaxN + (int)cta_rank * n_half, t.j);
                        }
                        __syncwarp();
                        if (++stage == kStages) { stage = 0; phase ^= 1; }
                    }
                }
                prev_m = t.m;
            }
        }
    } else if (warp == 1) {
        // =============================== MMA issuer =====================================
        // The whole warp walks the loop (warp-uniform control flow, so tile decoding, stage bookkeeping and the
        // shared-memory descriptors stay in uniform registers); one elected lane issues the tcgen05 instructions.
        // (With the loop under `if (lane == 0)` every MMA cost an ELECT + five R2UR.BROADCAST + a lane loop and
        // the issuing thread, not the tensor pipe, set the pace: ncu showed it busy 85 % of the time.)
        if (is_leader) {
            const bool issuer = elect_one();
            const uint32_t idesc = kFp8 ? make_idesc_e4m3(kTileRows, p.n_umma) : make_idesc(kTileRows, p.n_umma);
            const uint32_t tmem0 = __shfl_sync(0xffffffffu, tmem_base, 0);
            const uint64_t a_desc0 = make_smem_desc(q_smem);
            const uint64_t b_desc0 = make_smem_desc(v_smem);
            int stage = 0; uint32_t phase = 0, qf_phase = 0; int prev_m = -1; uint32_t t_cnt = 0;
            bool ok = true;
            Tile t;
            while (ok && it.next(t)) {
                const bool new_m = (t.m != prev_m);
              for (int sb = 0; sb < n_sub && ok; ++sb, ++t_cnt) {
                const uint32_t acc = t_cnt & 1u, acc_phase = (t_cnt >> 1) & 1u;
                ok = mbar_wait(bar_t_empty + 8 * acc, acc_phase ^ 1, p.abort_flag, 3);
                if (!ok) break;
                tc_fence_after();
                const uint32_t d_tmem = tmem0 + acc * kMaxN;
                for (int kb = 0; kb < p.num_kb; ++kb) {
                    if (new_m && sb == 0) { ok = mbar_wait(bar_q_full + 8 * kb, qf_phase, p.abort_flag, 4); if (!ok) break; }
                    ok = mbar_wait(bar_v_full + 8 * stage, phase, p.abort_flag, 5);
                    if (!ok) break;
                    tc_fence_after();
                    // start-address field is (addr >> 4): whole k-blocks / stages are added to the base descriptors
                    const uint64_t a_desc = a_desc0 + (uint64_t)((uint32_t)kb * (kQkbBytes >> 4));
                    const uint64_t b_desc = b_desc0 + (uint64_t)((uint32_t)stage * (uint32_t)(kVStageBytes >> 4));
                    if (issuer) {
#pragma unroll
                        for (int k = 0; k < kBlockK / kUmmaK; ++k) {
                            // +32 bytes per K=16 (bf16) / K=32 (e4m3) step inside the 128-byte swizzle row (address
                            // field is >>4)
                            if constexpr (kFp8)
                                umma_e4m3<kCtaGroup>(d_tmem, a_desc + 2u * k, b_desc + 2u * k, idesc, (uint32_t)((kb | k) != 0));
                            else
                                umma_bf16<kCtaGroup>(d_tmem, a_desc + 2u * k, b_desc + 2u * k, idesc, (uint32_t)((kb | k) != 0));
                        }
                        umma_commit<kCtaGroup>(bar_v_empty + 8 * stage);      // frees the V stage in both CTAs
                    }
                    __syncwarp();
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
                if (!ok) break;
                if (issuer) umma_commit<kCtaGroup>(bar_t_full + 8 * acc);            // accumulator ready (both CTAs)
                __syncwarp();
              }
                if (!ok) break;
                TileIter peek = it;
                Tile tn;
                const bool next_new_m = !peek.next(tn) || tn.m != t.m;
                if (next_new_m && issuer) umma_commit<kCtaGroup>(bar_q_empty);     // query tile may be overwritten
                __syncwarp();
                if (new_m) qf_phase ^= 1;
                prev_m = t.m;
            }
        }
    } else if (kEmitN && warp >= kEpiWarp0 + 4) {
        // ============ emission warps: N = coef*T*min(S,0) for every pair (one warp per TMEM lane quarter) =============
        // One pass over the accumulator: n = min(acc, 0); the tile's sum of n^2 (times T^2) feeds the value and,
        // because n*s == n^2, also dL/dT (sum dS*<q,v> = sum n^2 / T).  The clamp floor `lo` (-60 / -20) is far
        // outside the data range; a tile that does come near it (row minimum within two bf16 ulps of lo) is redone
        // with the reference's bf16 rounding of S, clamp and gradient gate before its accumulator is released.
        // Padded text tokens take part, as in the reference (model.py:525).
        // In kMode 2 the max-mean epilogue runs beside these warps in warps 4-7 (one warp per quarter, the round-1
        // arrangement): two independent ~1 000-instruction chains per scheduler instead of two ~1 500-instruction ones
        // doing both jobs; in kMode 1 warps 4-7 have no work.  The 8 KB of staging per warp are two 32 x 64 boxes: a
        // box leaves through the TMA unit while the next one is filled (cp.async.bulk.wait_group.read 1).
        const int quarter = warp & 3;
        const uint32_t t_empty_sig = (kCtaGroup == 2) ? mapa(bar_t_empty, 0) : bar_t_empty;
        const float Tval = *p.T;
        const float coefT = p.coef * Tval;
        const float2 cT2 = make_float2(coefT * Tval, coefT * Tval);
        const float T2f = Tval * Tval;
        const uint32_t stg0 = v_smem + (uint32_t)kStages * (uint32_t)kVStageBytes + (uint32_t)(warp - kEpiWarp0 - 4) * 2u * kStgBytesPerWarp;
        const bool wn = p.write_n != 0;
        // per-tile sums are added with a compensated fp32 sum (an fp64 add per tile and lane is 1/64-rate on this chip)
        float s2 = 0.f, s2c = 0.f, sT = 0.f, sTc = 0.f;
        uint32_t t_cnt = 0, nbox = 0;                               // nbox: bulk groups committed so far (staging box = nbox & 1)
        bool alive = true;
        Tile t;
        while (alive && it.next(t)) {
            const int wrow0 = t.m * kTileRows + (int)cta_rank * kBlockM + quarter * 32;      // the warp's first row
            const bool vrow = wrow0 + lane < p.M;
            const uint32_t acc = t_cnt & 1u, acc_phase = (t_cnt >> 1) & 1u;
            ++t_cnt;
            bool ok = mbar_wait(bar_t_full + 8 * acc, acc_phase, p.abort_flag, 6);
            ok = __all_sync(0xffffffffu, ok);
            if (!ok) { alive = false; break; }
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * kMaxN;
            float2 a2[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
            float mn[2] = {0.f, 0.f};
            {
                uint32_t bufA[32], bufB[32], w[16];
                tmem_ld32_raw(taddr, bufA);
                tmem_wait_ld();
#pragma unroll 1
                for (int b = 0; b < 4; ++b) {                                             // (rolled: I-cache)
                    const int c = 2 * b;
                    const uint32_t stg = stg0 + (nbox & 1u) * kStgBytesPerWarp;
                    const uint32_t stg_row = stg + (uint32_t)lane * 128u;
                    tmem_ld32_raw(taddr + (c + 1) * 32, bufB);
                    emit_chunk(bufA, c * 32, p.Nv, cT2, a2, mn, w);
                    if (wn) {
                        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // the box before last has been read
                        __syncwarp();
                        stage_chunk(w, stg_row, lane, 0);
                    }
                    tmem_wait_ld();
                    tmem_ld32_raw(taddr + ((c + 2) & 7) * 32, bufA);                     // (b == 3: a harmless re-load of chunk 0)
                    emit_chunk(bufB, (c + 1) * 32, p.Nv, cT2, a2, mn, w);
                    if (wn) { stage_chunk(w, stg_row, lane, 1); if (c * 32 < p.Nv) { emit_box_store(&tmap_n, stg, c * 32, t.j, wrow0, lane); ++nbox; } }
                    tmem_wait_ld();
                }
            }
            const float a2s = (a2[0].x + a2[0].y) + (a2[1].x + a2[1].y);
            const float mns = fminf(mn[0], mn[1]) * Tval;
            // (margin of two bf16 ulps: the reference clamps the bf16-ROUNDED similarity, so a value a hair above
            //  the floor in fp32 can sit on it after rounding)
            if (!__any_sync(0xffffffffu, vrow && mns < p.lo * (1.0f - 1.0f / 64.0f))) {
                if (vrow) { kahan_add(s2, s2c, a2s * T2f); kahan_add(sT, sTc, a2s * Tval); }
            } else {
                // exact pass (some similarity of this warp's rows is below the clamp floor): redo the tile with the
                // clamp and its gradient gate applied, overwriting what the fast pass stored
                float e2 = 0.f, eT = 0.f;
                if (wn) emit_box_drain(lane);
                for (int b = 0; b < 4; ++b) {
                    const int c = 2 * b;
                    if (c * 32 >= p.Nv) break;                                           // warp-uniform
                    const uint32_t stg = stg0 + (nbox & 1u) * kStgBytesPerWarp;
                    const uint32_t stg_row = stg + (uint32_t)lane * 128u;
                    uint32_t buf[32], w[16];
                    tmem_ld32_raw(taddr + c * 32, buf);
                    tmem_wait_ld();
                    emit_chunk_exact(buf, c * 32, p.Nv, Tval, coefT, p.lo, e2, eT, w);
                    if (wn) { emit_box_reusable(lane); stage_chunk(w, stg_row, lane, 0); }
                    tmem_ld32_raw(taddr + (c + 1) * 32, buf);
                    tmem_wait_ld();
                    emit_chunk_exact(buf, (c + 1) * 32, p.Nv, Tval, coefT, p.lo, e2, eT, w);
                    if (wn) { stage_chunk(w, stg_row, lane, 1); emit_box_store(&tmap_n, stg, c * 32, t.j, wrow0, lane); ++nbox; }
                }
                if (vrow) { kahan_add(s2, s2c, e2); kahan_add(sT, sTc, eT); }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (kCtaGroup == 2) mbar_arrive_cluster(t_empty_sig + 8 * acc);
                else mbar_arrive_local(bar_t_empty + 8 * acc);
            }
        }
        emit_box_reusable(lane);                                    // the staging boxes must outlive the last bulk reads
        const double s2d = warp_sum_d((double)s2 - (double)s2c);
        const double sTd = warp_sum_d((double)sT - (double)sTc);
        if (lane == 0) {
            p.n_partials[(size_t)(blockIdx.x * kEmitEpiWarps + (warp - kEpiWarp0)) * 2] = s2d;
            p.n_partials[(size_t)(blockIdx.x * kEmitEpiWarps + (warp - kEpiWarp0)) * 2 + 1] = sTd * (double)p.coef;
        }
    } else if (kMode != 1 && warp >= kEpiWarp0 && (p.idx != nullptr || warp < kEpiWarp0 + 4)) {
        // =============================== epilogue =======================================
        // Two warps per TMEM lane quarter (one per scheduler pair): both take the row maximum over all columns
        // (cheap: FMNMX3), then each searches ITS half of the columns for the first one that reaches the
        // threshold (the expensive pass); the upper half hands its result to the lower-half warp through 2 bytes
        // of shared memory and a 64-thread named barrier, and the lower-half warp alone writes idx / partial sums.
        // (One warp per scheduler has to issue ~1 600 dependent instructions per tile within the tile's MMA time.)
        // Forward-only calls (no idx) have no second pass: the upper-half warps sit out.
        // kMode 2: ONE warp per lane quarter does the whole max-mean epilogue (all columns in both passes, no exchange);
        // the other four epilogue warps are the emission warps above.
        constexpr bool kSolo = kMode == 2;
        const int quarter = warp & 3;
        const int half = (warp - kEpiWarp0) >> 2;
        const uint32_t t_empty_sig = (kCtaGroup == 2) ? mapa(bar_t_empty, 0) : bar_t_empty;
        float Tval = *p.T;
        if (p.inv_T) Tval = 1.0f / Tval;
        int prev_m = -1; float rs = 0.f; uint32_t t_cnt = 0;
        size_t idx_off = 0;                       // (i*nq_pad + a) of this thread's row
        int r_orig = -1, qi = 0, piece = 0;       // original row (-1: no such row), its query, packed partial slot
        const size_t idx_pitch = (size_t)(p.M / p.Nq) * p.nq_pad;
        float R_run = 0.f; int best_run = 0;      // running (rounded max, first argmax) across the sub-tiles of an image
        bool alive = true;
        Tile t;
        while (alive && it.next(t)) {
            const int row0 = t.m * kTileRows + (int)cta_rank * kBlockM + quarter * 32;
            const int r = row0 + lane;                   // GEMM row (packed row number when rows are packed)
            if constexpr (kMode == kModeRaggedMean) {
                // the warp's 32 rows are word w of their slot's caption-start mask: the row's caption is the number
                // of starts up to it, counted from the slot's first caption
                if (t.m != prev_m) {
                    const int* meta = p.slot_meta + (size_t)(row0 >> 8) * kSlotMetaInts;
                    const int w = (row0 >> 5) & 7;
                    int before = 0;
                    for (int i = 0; i < w; ++i) before += __popc((uint32_t)__ldg(meta + kSlotMetaStarts + i));
                    const uint32_t sw = (uint32_t)__ldg(meta + kSlotMetaStarts + w);
                    const bool valid = (row0 & (kSlotRows - 1)) + lane < __ldg(meta + kSlotMetaUsed);
                    const int cap = __ldg(meta + kSlotMetaCap0) + before + __popc(sw & (0xffffffffu >> (31 - lane))) - 1;
                    r_orig = valid ? r : -1;
                    rs = valid ? 1.0f / (float)__ldg(p.cap_info + 2 * (size_t)cap + 1) : 0.f;
                    if constexpr (kFp8) { if (valid) rs = (__ldg(p.q_scale + r) * rs) * Tval; }     // w_t
                    prev_m = t.m;
                }
            } else if (t.m != prev_m) {
                r_orig = (r < M_eff) ? (p.pack_off ? p.rowmap[r] : r) : -1;
                rs = (r_orig >= 0) ? p.row_scale[r_orig] : 0.f;
                if constexpr (kFp8) { if (r_orig >= 0) rs = (p.q_scale[r_orig] * rs) * Tval; }     // t_a
                qi = (r_orig >= 0) ? r_orig / p.Nq : 0x7fffffff;
                idx_off = (r_orig >= 0) ? (size_t)qi * p.nq_pad + (r_orig - qi * p.Nq) : 0;
                if (p.pack_off && r_orig >= 0) piece = (row0 >> 5) - (p.pack_off[qi] >> 5);
                prev_m = t.m;
            }
          for (int sb = 0; sb < n_sub; ++sb, ++t_cnt) {
            const uint32_t acc = t_cnt & 1u, acc_phase = (t_cnt >> 1) & 1u;
            // e4m3: this sub-tile's 256 patch scales into the warp's slot (lane l: columns 8l .. 8l+7), loaded
            // while the MMAs run; 0 beyond the last patch (those columns are masked anyway)
            const uint32_t sg_smem = q_smem + 4u * kQkbBytes + (uint32_t)quarter * 1024u;
            const float4* sg_gen = reinterpret_cast<const float4*>(smem_gen + (sg_smem - smem_base));
            if constexpr (kFp8) {
                const int c0 = sb * kMaxN + 8 * lane;
                const float* src = p.col_scale + (size_t)t.j * p.Nv;
                uint32_t s[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) s[e] = __float_as_uint(c0 + e < p.Nv ? __ldg(src + c0 + e) : 0.f);
                __syncwarp();                                 // every lane is done with the previous sub-tile's scales
                sts128(sg_smem + (uint32_t)lane * 32u, s[0], s[1], s[2], s[3]);
                sts128(sg_smem + (uint32_t)lane * 32u + 16u, s[4], s[5], s[6], s[7]);
                __syncwarp();
            }
            bool ok = mbar_wait(bar_t_full + 8 * acc, acc_phase, p.abort_flag, 6);
            ok = __all_sync(0xffffffffu, ok);
            if (!ok) { alive = false; break; }
            tc_fence_after();
            const int Nv = p.Nv - sb * kMaxN;                // patches of this sub-tile that exist (may exceed 256)
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * kMaxN;

            if constexpr (kMode == kModeRaggedMax) {
                // ---- segmented walk of the slot's used columns, two 32-column chunks per step; the mask words
                //      are read with the same address in every lane (one broadcast load each) ----
                const int* meta = p.slot_meta + (size_t)t.j * kSlotMetaInts;
                const int used = __ldg(meta + kSlotMetaUsed);
                int cap = __ldg(meta + kSlotMetaCap0);
                float run = -INFINITY;
#pragma unroll 1
                for (int c = 0; c < kMaxN / 32 && c * 32 < used; c += 2) {
                    uint32_t bufA[32], bufB[32];
                    tmem_ld32_raw(taddr + c * 32, bufA);
                    tmem_ld32_raw(taddr + (c + 1) * 32, bufB);
                    const int2 sw = __ldg(reinterpret_cast<const int2*>(meta + kSlotMetaStarts + c));
                    const int2 ew = __ldg(reinterpret_cast<const int2*>(meta + kSlotMetaEnds + c));
                    tmem_wait_ld();
                    if constexpr (kFp8) {
                        ragged_chunk_scaled(bufA, sg_gen + 8 * c, (uint32_t)sw.x, (uint32_t)ew.x, run, cap, r_orig >= 0,
                                            rs, p, row0, lane);
                        ragged_chunk_scaled(bufB, sg_gen + 8 * (c + 1), (uint32_t)sw.y, (uint32_t)ew.y, run, cap,
                                            r_orig >= 0, rs, p, row0, lane);
                    } else {
                        ragged_chunk(bufA, (uint32_t)sw.x, (uint32_t)ew.x, run, cap, r_orig >= 0, Tval, rs, p, row0, lane);
                        ragged_chunk(bufB, (uint32_t)sw.y, (uint32_t)ew.y, run, cap, r_orig >= 0, Tval, rs, p, row0, lane);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if constexpr (kCtaGroup == 2) mbar_arrive_cluster(t_empty_sig + 8 * acc);
                    else mbar_arrive_local(bar_t_empty + 8 * acc);
                }
                continue;
            }

            // ---- pass 1: row maximum over the raw accumulators.  32-column loads, software pipelined
            //      (chunk c+1 in flight while chunk c is reduced), four independent FMNMX3 chains per chunk.
            //      All kMaxN/32 chunks are always loaded — columns >= n_umma hold stale but allocated TMEM and
            //      are masked by Nv — which keeps every load unconditional (see tmem_ld32_raw). ----
            constexpr int kCh = kMaxN / 32;
            float mx = -INFINITY;
            if constexpr (kFp8) {
                // the same loads; every column scaled by its patch scale before the (NaN-propagating) max
                uint32_t bufA[32], bufB[32];
                tmem_ld32_raw(taddr, bufA);
                tmem_wait_ld();
#pragma unroll
                for (int c = 0; c < kCh; c += 2) {
                    tmem_ld32_raw(taddr + (c + 1) * 32, bufB);
                    mx = fmax_nan(mx, chunk_max32_scaled(bufA, sg_gen + 8 * c, c * 32, Nv));
                    tmem_wait_ld();
                    if (c + 2 < kCh) tmem_ld32_raw(taddr + (c + 2) * 32, bufA);          // compile-time condition
                    mx = fmax_nan(mx, chunk_max32_scaled(bufB, sg_gen + 8 * (c + 1), (c + 1) * 32, Nv));
                    tmem_wait_ld();
                }
            } else {
                uint32_t bufA[32], bufB[32];
                tmem_ld32_raw(taddr, bufA);
                tmem_wait_ld();
#pragma unroll
                for (int c = 0; c < kCh; c += 2) {
                    tmem_ld32_raw(taddr + (c + 1) * 32, bufB);
                    mx = fmaxf(mx, chunk_max32(bufA, c * 32, Nv));
                    tmem_wait_ld();
                    if (c + 2 < kCh) tmem_ld32_raw(taddr + (c + 2) * 32, bufA);          // compile-time condition
                    mx = fmaxf(mx, chunk_max32(bufB, (c + 1) * 32, Nv));
                    tmem_wait_ld();
                }
            }
            float R;
            float theta = 0.f;
            if constexpr (kFp8) R = mx;
            else if constexpr (kRagged) R = round_sim<true>(mx, Tval);       // no idx: no threshold
            else theta = argmax_threshold<true>(mx, Tval, &R);

            // ---- pass 2: first column whose accumulator reaches the threshold (the reference's first-index
            //      argmax).  Same pipelined loads, walking the chunks from the last to the first so the lowest
            //      qualifying column is the one that sticks; inside a chunk four independent 8-column
            //      compare/select chains instead of one 256-long dependent chain. ----
            int best = (int)kNoCol;
            if (!kFp8 && !kRagged && p.idx != nullptr) {
                constexpr int kHalfCh = kSolo ? kCh : kCh / 2;
                const int cb = kSolo ? 0 : half * kHalfCh;       // this warp's chunks: [cb, cb + kHalfCh)
                uint32_t bufA[32], bufB[32];
                tmem_ld32_raw(taddr + (cb + kHalfCh - 1) * 32, bufA);
                tmem_wait_ld();
#pragma unroll
                for (int cc = kHalfCh - 1; cc >= 0; cc -= 2) {
                    const int c = cb + cc;
                    tmem_ld32_raw(taddr + (c - 1) * 32, bufB);
                    first_ge32(bufA, c * 32, Nv, theta, best);
                    tmem_wait_ld();
                    if (cc - 2 >= 0) tmem_ld32_raw(taddr + (c - 2) * 32, bufA);          // compile-time condition
                    first_ge32(bufB, (c - 1) * 32, Nv, theta, best);
                    tmem_wait_ld();
                }
            }
            // TMEM stage drained: hand it back to the MMA issuer before touching global memory
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (kCtaGroup == 2) mbar_arrive_cluster(t_empty_sig + 8 * acc);
                else mbar_arrive_local(bar_t_empty + 8 * acc);
            }
            if (p.idx != nullptr && !kSolo && !kRagged) {
                // pair exchange (double buffered by tile parity: the upper-half warp may already be one tile ahead)
                const uint32_t slot = xch_smem + ((t_cnt & 1u) * 128u + (uint32_t)(quarter * 32 + lane)) * 2u;
                if (half == 1) asm volatile("st.shared.u16 [%0], %1;" ::"r"(slot), "h"((uint16_t)best) : "memory");
                asm volatile("bar.sync %0, 64;" ::"r"(1 + quarter) : "memory");
                if (half == 0) {
                    uint16_t other;
                    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(other) : "r"(slot) : "memory");
                    if (best == (int)kNoCol) best = (other == kNoCol) ? 0 : (int)other;
                }
            }
            if (kSolo && best == (int)kNoCol) best = 0;
            if (half == 1) continue;                             // the lower-half warp owns the outputs
            // Equal rounded maxima in two sub-tiles: the earlier one holds the first index (torch.max), and
            // inside a sub-tile `best` already is the first column of that rounded value.
            if constexpr (kFp8) R_run = sb == 0 ? R : fmax_nan(R_run, R);
            else if (sb == 0 || R > R_run) { R_run = R; best_run = best + sb * kMaxN; }
          }
            if (!alive) break;
            if (half == 1 || kMode == kModeRaggedMax) continue;     // kMode 3 stored its partials during the walk
            if (!kRagged && p.idx != nullptr && r_orig >= 0) {
                if (p.idx16) reinterpret_cast<uint16_t*>(p.idx)[(size_t)t.j * idx_pitch + idx_off] = (uint16_t)best_run;
                else p.idx[(size_t)t.j * idx_pitch + idx_off] = (uint8_t)best_run;
            }
            const float val = (r_orig >= 0) ? R_run * rs : 0.f;
            if constexpr (kMode == kModeRaggedMean) {
                if (r_orig >= 0) p.part[r] = val;                  // one weighted row maximum per slot row
            } else if (p.pack_off == nullptr) store_group_partials(p.part, t.j, row0 >> 5, p.G, p.S, row0, p.M, p.Nq, val, lane);
            else store_group_partials_packed(p.part, t.j, p.Bq, p.pieces, qi, piece, val, lane);
        }
    }

    // ---- teardown ---------------------------------------------------------------------------
    __syncwarp();
    tc_fence_before();
    if constexpr (kCtaGroup == 2) { cluster_arrive(); cluster_wait(); } else { __syncthreads(); }
    if (warp == 2) tmem_dealloc<kCtaGroup>(tmem_base, kTmemCols);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// Tile order (TileIter).  V up to ~48 MB: any order, V stays in L2.  Larger: if there are enough query tiles to
// give every cluster a few items per ~16 MB image chunk, ALL clusters walk the same chunk at the same time —
// V is read from HBM once per pass whatever its size (cfg 4: 2.1 GB), and even at cfg 2 (67 MB, nominally
// L2-sized) the hot set shrinks from V + Q to one chunk + the query tiles (measured 3.34 -> 3.17 ms).
// Otherwise (retrieval: one or a few query tiles against a huge gallery) each cluster keeps to its own images
// and runs all query tiles against a handful of them back to back, so the re-reads hit L2.
// img_bytes = Nv * D * element size.
static void pick_tile_order(Params& p, size_t img_bytes, int Bv, int n_m, int n_clusters) {
    const size_t v_bytes = (size_t)Bv * img_bytes;
    p.C = Bv;
    p.sync = 0;
    if (v_bytes > (size_t)48 << 20) {
        size_t c16 = ((size_t)16 << 20) / img_bytes;
        if (c16 < 1) c16 = 1;
        if ((size_t)n_m * c16 >= (size_t)4 * n_clusters) {
            p.C = (int)(c16 > (size_t)Bv ? (size_t)Bv : c16);
            p.sync = 1;
        } else {
            size_t c = ((size_t)48 << 20) / ((size_t)n_clusters * img_bytes);
            p.C = (int)(c < 1 ? 1 : (c > 64 ? 64 : c));
            if (p.C > Bv) p.C = Bv;
        }
    }
}

template <int kCtaGroup, bool kSub, int kMode = 0, bool kFp8 = false>
static int launch_t(const CUtensorMap& mq, const CUtensorMap& mv, const CUtensorMap& mn, const Params& p, int n_clusters,
                    cudaStream_t st) {
    return launch_clusters<maxmean_tc_kernel<kCtaGroup, kSub, kMode, kFp8>>(kCtaGroup, n_clusters, kEmitThreads, kSmemBytes,
                                                                            st, mq, mv, mn, p);
}

}  // namespace tc

bool tc_supported(int Nv, int D) { return Nv >= 1 && Nv <= 65535 && D % tc::kBlockK == 0 && D >= tc::kBlockK && D <= tc::kMaxKB * tc::kBlockK; }
bool tc_emit_supported(int Nv, int D) { return tc_supported(Nv, D) && Nv <= tc::kMaxN && Nv % 8 == 0; }
bool tc_e4m3_supported(int Nv, int D) { return Nv >= 1 && Nv <= 65535 && D % 128 == 0 && D >= 128 && D <= 512; }

int launch_maxmean_tc(const void* q, const void* v, const float* row_scale, const float* T,
                      int inv_T, int M, int Bv, int Nq, int Nv, int D,
                      float* part, void* idx, int* abort_flag, int cta_group, int flags, const int* pack_maps,
                      const EmitNArgs* emit, const E4m3Args* e4m3, cudaStream_t st, const RaggedArgs* ragged) {
    using namespace tc;
    if (e4m3 ? !tc_e4m3_supported(Nv, D) : !tc_supported(Nv, D))
        return fail_msg(TRIAD_ERR_UNSUPPORTED, e4m3 ? "tcgen05 e4m3 forward: needs D in {128, 256, 384, 512}"
                                                    : "tcgen05 forward: needs D in {64,...,512} (multiple of 64)");
    const int tile_rows = kBlockM * cta_group;
    const int n_m = ceil_div(M, tile_rows);
    const int n_sub = ceil_div(Nv, kMaxN);
    if ((long long)n_m * Bv * n_sub >= 0x7fffffffLL) return fail_msg(TRIAD_ERR_UNSUPPORTED, "tcgen05 forward: too many tiles");

    int sms = 0;
    int rc = device_sms(&sms);
    if (rc) return rc;

    // one 128-byte swizzle row of a k-block holds 64 bf16 or 128 e4m3 elements
    const int elt = e4m3 ? 1 : 2, kb_elems = 128 / elt;
    const CUtensorMapDataType ttype = e4m3 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    Params p;
    memset(&p, 0, sizeof p);
    p.M = M; p.Bv = Bv; p.Nq = Nq; p.Nv = Nv;
    p.n_umma = n_sub > 1 ? kMaxN : (Nv + 15) / 16 * 16;
    p.n_sub = n_sub;
    p.idx16 = !e4m3 && Nv > 256;
    p.num_kb = D / kb_elems;
    p.n_m = n_m;
    int n_clusters = sms / cta_group;
    pick_tile_order(p, (size_t)Nv * D * elt, Bv, n_m, n_clusters);
    if (flags & TRIAD_FWD_SYNC_CHUNKS) { p.C = Bv < 3 ? Bv : 3; p.sync = 1; }     // tests: tiny chunks on small shapes
    PartLayout pl = part_layout(M, Nq);
    p.G = pl.G; p.S = pl.S;
    p.nq_pad = nq_padded(Nq);
    p.inv_T = inv_T;
    p.row_scale = row_scale; p.T = T; p.part = part; p.idx = (uint8_t*)idx; p.abort_flag = abort_flag;
    p.Bq = M / Nq;
    p.pack_off = pack_maps;                                   // q then points at the PACKED rows
    p.rowmap = pack_maps ? pack_maps + p.Bq + 1 : nullptr;
    p.pieces = packed_pieces(Nq);
    if (emit) {
        if (!tc_emit_supported(Nv, D) || pack_maps) return fail_msg(TRIAD_ERR_UNSUPPORTED, "dense-regulariser forward: needs Nv <= 256, Nv % 8 == 0");
        if (emit->with_maxmean && (!idx || !part || inv_T)) return fail_msg(TRIAD_ERR_BAD_ARG, "dense-regulariser + max-mean forward: needs idx and the partial buffer");
        if (sms * kEmitEpiWarps > kNonnegFusedPartials) return fail_msg(TRIAD_ERR_UNSUPPORTED, "dense-regulariser forward: too many SMs for the partial buffer");
        p.n_out = (__nv_bfloat16*)emit->n_out; p.ldn = emit->ldn; p.lo = emit->lo; p.coef = emit->coef;
        p.write_n = emit->write_n; p.n_partials = emit->partials;
    }
    if (e4m3) { p.col_scale = e4m3->g_scale; p.q_scale = e4m3->q_scale; }

    CUtensorMap mq, mv;
    {
        cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)M};
        cuuint64_t strides[1] = {(cuuint64_t)D * elt};
        cuuint32_t box[2] = {(cuuint32_t)kb_elems, (cuuint32_t)kBlockM};
        if ((rc = encode_tmap(&mq, ttype, q, 2, dims, strides, box, Swizzle::k128B))) return rc;
    }
    {
        cuuint64_t dims[3] = {(cuuint64_t)D, (cuuint64_t)Nv, (cuuint64_t)Bv};
        cuuint64_t strides[2] = {(cuuint64_t)D * elt, (cuuint64_t)Nv * D * elt};
        cuuint32_t box[3] = {(cuuint32_t)kb_elems, (cuuint32_t)(p.n_umma / cta_group), 1};
        if ((rc = encode_tmap(&mv, ttype, v, 3, dims, strides, box, Swizzle::k128B))) return rc;
    }
    // N[row][image][patch] as a rank-3 tensor {Nv, images, M} (row pitch ldn): the epilogue's 32-row x 64-column store
    // boxes are clipped at the image's last patch and at the last row by the TMA unit itself
    CUtensorMap mn = mq;
    if (emit && emit->write_n) {
        cuuint64_t dims[3] = {(cuuint64_t)Nv, (cuuint64_t)Bv, (cuuint64_t)M};
        cuuint64_t strides[2] = {(cuuint64_t)Nv * 2, (cuuint64_t)emit->ldn * 2};
        cuuint32_t box[3] = {64, 1, 32};
        if ((rc = encode_tmap(&mn, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, emit->n_out, 3, dims, strides, box, Swizzle::k128B))) return rc;
    }
    const long long total = (long long)n_m * Bv;
    if ((long long)n_clusters > total) n_clusters = (int)total;
    if (n_clusters < 1) n_clusters = 1;
    if (ragged) {
        p.slot_meta = ragged->slot_meta;
        p.cap_info = ragged->cap_info;
        if (ragged->direction == 0) {
            p.S = 1;                                          // part[caption][group]
            if (e4m3)
                return cta_group == 2 ? launch_t<2, false, kModeRaggedMax, true>(mq, mv, mn, p, n_clusters, st)
                                      : launch_t<1, false, kModeRaggedMax, true>(mq, mv, mn, p, n_clusters, st);
            return cta_group == 2 ? launch_t<2, false, kModeRaggedMax>(mq, mv, mn, p, n_clusters, st)
                                  : launch_t<1, false, kModeRaggedMax>(mq, mv, mn, p, n_clusters, st);
        }
        if (cta_group != 2) return fail_msg(TRIAD_ERR_UNSUPPORTED, "ragged direction 1: cta_group::2 only");
        if (e4m3)
            return n_sub > 1 ? launch_t<2, true, kModeRaggedMean, true>(mq, mv, mn, p, n_clusters, st)
                             : launch_t<2, false, kModeRaggedMean, true>(mq, mv, mn, p, n_clusters, st);
        return n_sub > 1 ? launch_t<2, true, kModeRaggedMean>(mq, mv, mn, p, n_clusters, st)
                         : launch_t<2, false, kModeRaggedMean>(mq, mv, mn, p, n_clusters, st);
    }
    if (emit) {
        // one slot per epilogue warp of every CTA, written only by the emission warps of CTAs that get work: clear all
        TRIAD_CUDA_CHECK(cudaMemsetAsync(emit->partials, 0, (size_t)sms * kEmitEpiWarps * 2 * sizeof(double), st));
        if (emit->with_maxmean)
            rc = cta_group == 2 ? launch_t<2, false, 2>(mq, mv, mn, p, n_clusters, st) : launch_t<1, false, 2>(mq, mv, mn, p, n_clusters, st);
        else
            rc = cta_group == 2 ? launch_t<2, false, 1>(mq, mv, mn, p, n_clusters, st) : launch_t<1, false, 1>(mq, mv, mn, p, n_clusters, st);
        return rc ? rc : launch_nonneg_finish(emit->partials, sms * kEmitEpiWarps, emit->sums, st);
    }
    if (!e4m3) {
        if (n_sub > 1) return cta_group == 2 ? launch_t<2, true>(mq, mv, mn, p, n_clusters, st) : launch_t<1, true>(mq, mv, mn, p, n_clusters, st);
        return cta_group == 2 ? launch_t<2, false>(mq, mv, mn, p, n_clusters, st) : launch_t<1, false>(mq, mv, mn, p, n_clusters, st);
    }
    if (n_sub > 1) return cta_group == 2 ? launch_t<2, true, 0, true>(mq, mv, mn, p, n_clusters, st) : launch_t<1, true, 0, true>(mq, mv, mn, p, n_clusters, st);
    return cta_group == 2 ? launch_t<2, false, 0, true>(mq, mv, mn, p, n_clusters, st) : launch_t<1, false, 0, true>(mq, mv, mn, p, n_clusters, st);
}

}  // namespace triad
