// Backward of the max-mean similarity through the saved argmax indices (SURVEY.md §8 a5;
// replaces autograd's backward of src/model.py:387-391, which materialises a zero dS of the
// full Bq x Bv x Nq x Nv size, scatters into it and runs two dense bmm backward GEMMs).
//
//   dq[r,:]   = T*row_scale[r] * sum_j g[i(r),j] * v[j, idx[j][r], :]        (gather)
//   dv[j,p,:] = sum_{r: idx[j][r]==p} T*row_scale[r]*g[i(r),j] * q[r,:]      (scatter)
//   dT        = sum_ij g[i,j]*clip[i,j] / T
//
// Both passes are L2- and issue-bound CUDA-core work (2*D MACs per (row,image) pair, i.e. 2/Nv
// of the forward's flops); they are deliberately NOT reshaped into one-hot GEMMs (that would
// cost a full forward each).  The scatter is turned into a gather: a stable per-image counting
// sort of the rows by winning patch (one byte keys) gives every (image, patch) its list of
// (row, weight) pairs, and a warp then accumulates that list in registers — no atomics, fixed
// summation order, bit-reproducible.
//
// dv code paths, for Nv <= kDvMaxNv (all produce the same lists in the same order, hence bit-identical results; the
// tests compare them):
//   bf16, Nv <= kGroupMaxNv (the training shapes): dv_group_sort_kernel (shared-memory sort per image x 8192-row group)
//                                            -> dv_gather_grouped_kernel (packed rows, FFMA2, 64 registers);
//   bf16, Nv  > kGroupMaxNv:                 dv_count / dv_offsets / dv_scatter_sort (global sort)
//                                            -> dv_gather_grouped_kernel over the image's one list;
//   fp32 inputs or TRIAD_BWD_GENERIC_DV:     the global sort -> dv_gather_kernel (generic, the cross-check).
// dq code paths:
//   bf16, Nv <= 256, D % 64 == 0:            dq_pipe_kernel (bwd_dq_pipe.cu, shared-memory gather);
//   bf16, Nv  > 256, D % 64 == 0:            dq_tile_kernel (bwd_dq_tile.cu, L1-resident gather);
//   otherwise or TRIAD_BWD_GENERIC_DQ:       dq_gather_kernel here (generic, the cross-check: same summation order).
#include "common.cuh"

#include <type_traits>

namespace triad {

template <typename T> struct Vec16;            // one 16-byte chunk of a row
template <> struct Vec16<__nv_bfloat16> {
    static constexpr int kElems = 8;
    __device__ static __forceinline__ void load(const __nv_bfloat16* p, float (&f)[8]) {
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            f[2 * k] = __uint_as_float(w[k] << 16);
            f[2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u);
        }
    }
    __device__ static __forceinline__ void store(__nv_bfloat16* p, const float (&f)[8]) {
        uint4 u;
        uint32_t* w = reinterpret_cast<uint32_t*>(&u);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * k], f[2 * k + 1]);
            w[k] = *reinterpret_cast<uint32_t*>(&h);
        }
        *reinterpret_cast<uint4*>(p) = u;
    }
};
template <> struct Vec16<float> {
    static constexpr int kElems = 4;
    __device__ static __forceinline__ void load(const float* p, float (&f)[4]) {
        const float4 u = __ldg(reinterpret_cast<const float4*>(p));
        f[0] = u.x; f[1] = u.y; f[2] = u.z; f[3] = u.w;
    }
    __device__ static __forceinline__ void store(float* p, const float (&f)[4]) {
        *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
    }
};

// store E fp32 values as OutT (float or the input type)
template <typename OutT, int E> struct StoreAs;
template <int E> struct StoreAs<float, E> {
    __device__ static __forceinline__ void put(float* p, const float (&f)[E]) {
#pragma unroll
        for (int c = 0; c < E; c += 4) *reinterpret_cast<float4*>(p + c) = make_float4(f[c], f[c + 1], f[c + 2], f[c + 3]);
    }
};
template <> struct StoreAs<__nv_bfloat16, 8> {
    __device__ static __forceinline__ void put(__nv_bfloat16* p, const float (&f)[8]) { Vec16<__nv_bfloat16>::store(p, f); }
};

template <typename OutT, int E> struct LoadAs;
template <int E> struct LoadAs<float, E> {
    __device__ static __forceinline__ void get(const float* p, float (&f)[E]) {
#pragma unroll
        for (int c = 0; c < E; c += 4) {
            const float4 u = *reinterpret_cast<const float4*>(p + c);
            f[c] = u.x; f[c + 1] = u.y; f[c + 2] = u.z; f[c + 3] = u.w;
        }
    }
};
template <> struct LoadAs<__nv_bfloat16, 8> {
    __device__ static __forceinline__ void get(const __nv_bfloat16* p, float (&f)[8]) { Vec16<__nv_bfloat16>::load(p, f); }
};

// fp32 scratch -> output dtype (used when dv is accumulated over several query blocks)
template <typename OutT>
__global__ void __launch_bounds__(256)
dv_convert_kernel(const float* __restrict__ src, size_t n, OutT* __restrict__ dst) {
    for (size_t k = (size_t)blockIdx.x * 256 + threadIdx.x; k < n; k += (size_t)gridDim.x * 256) dst[k] = (OutT)src[k];
}

// ---------------------------------------------------------------------------------------
// dq (generic gather): one CTA = 32 consecutive token rows; 8 warps x 4 rows; lanes own
// 16-byte chunks of D; winners and weights of 32 images at a time are staged in shared memory.
// ---------------------------------------------------------------------------------------
constexpr int kDqRows = 32;
constexpr int kDqJ = 32;          // images staged per step

template <typename T, typename IdxT, int KCH>
__global__ void __launch_bounds__(256)
dq_gather_kernel(const T* __restrict__ v, const IdxT* __restrict__ idx, const float* __restrict__ g,
                 const float* __restrict__ row_scale, const float* __restrict__ Tptr,
                 int M, int Bv, int Nq, int Nv, int D, int nq_pad, T* __restrict__ dq) {
    constexpr int E = Vec16<T>::kElems;
    __shared__ IdxT idx_s[kDqJ][kDqRows];
    __shared__ float w_s[kDqRows][kDqJ + 1];
    __shared__ int ioff_s[kDqRows];      // (i*nq_pad + a) of each row
    __shared__ int iq_s[kDqRows];        // query index of each row

    const int row0 = blockIdx.x * kDqRows;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nchunk = D / E;
    const size_t pitch = (size_t)(M / Nq) * nq_pad;
    if (threadIdx.x < kDqRows) {
        const int r = row0 + threadIdx.x;
        const int qi = (r < M) ? r / Nq : 0;
        iq_s[threadIdx.x] = qi;
        ioff_s[threadIdx.x] = (r < M) ? qi * nq_pad + (r - qi * Nq) : -1;
    }

    float acc[4][KCH][E];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < KCH; ++b)
#pragma unroll
            for (int c = 0; c < E; ++c) acc[a][b][c] = 0.f;

    for (int j0 = 0; j0 < Bv; j0 += kDqJ) {
        __syncthreads();
        for (int t = threadIdx.x; t < kDqJ * kDqRows; t += 256) {
            const int jj = t / kDqRows, rr = t % kDqRows;
            const int j = j0 + jj;
            const int off = ioff_s[rr];
            IdxT p = 0; float w = 0.f;
            if (j < Bv && off >= 0) {
                p = idx[(size_t)j * pitch + off];
                w = g[(size_t)iq_s[rr] * Bv + j];
            }
            idx_s[jj][rr] = p;
            w_s[rr][jj] = w;
        }
        __syncthreads();
        const int jn = min(kDqJ, Bv - j0);
        for (int jj = 0; jj < jn; ++jj) {
            const T* vj = v + (size_t)(j0 + jj) * Nv * D;
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const int rr = warp * 4 + a;
                const float w = w_s[rr][jj];
                const T* src = vj + (size_t)idx_s[jj][rr] * D;
#pragma unroll
                for (int b = 0; b < KCH; ++b) {
                    const int ch = lane + 32 * b;
                    if (ch < nchunk) {
                        float f[E];
                        Vec16<T>::load(src + ch * E, f);
#pragma unroll
                        for (int c = 0; c < E; ++c) acc[a][b][c] = fmaf(w, f[c], acc[a][b][c]);
                    }
                }
            }
        }
    }
    const float Tval = *Tptr;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int r = row0 + warp * 4 + a;
        if (r >= M) continue;
        const float s = Tval * row_scale[r];
#pragma unroll
        for (int b = 0; b < KCH; ++b) {
            const int ch = lane + 32 * b;
            if (ch < nchunk) {
                float f[E];
#pragma unroll
                for (int c = 0; c < E; ++c) f[c] = acc[a][b][c] * s;
                Vec16<T>::store(dq + (size_t)r * D + ch * E, f);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// dv step 1: stable counting sort of one image's rows by winning patch.
//   The Bq queries are cut into kSortGroups groups; warp (j,c) owns group c of image j.
//   count  : per-(j,c) histogram of the winners            -> cnt[j][c][p]
//   offsets: exclusive scan over (p major, c minor)        -> start[j][c][p], seg[j][p]
//   scatter: rows in order, rank inside a 32-row chunk via __match_any_sync => stable
//   entry = { row index into q, weight = row_scale[r] * g[i][j] }
// ---------------------------------------------------------------------------------------
constexpr int kSortGroups = 8;
constexpr int kSortWarps = 4;
// The largest patch count the dv pass handles: the global sort keeps kSortWarps counters of Nv words in (at most the
// default 48 KB of) dynamic shared memory.
constexpr int kDvMaxNv = 3072;
static_assert((size_t)kSortWarps * kDvMaxNv * 4 <= 48 * 1024, "dv global sort: per-warp counters exceed 48 KB");

struct __align__(8) DvEntry { uint32_t row; float w; };

template <typename IdxT>
__global__ void __launch_bounds__(kSortWarps * 32)
dv_count_kernel(const IdxT* __restrict__ idx, const float* __restrict__ row_scale, size_t img_pitch,
                int j0, int nj, int Bq, int Nq, int Nv, int nq_pad, uint32_t* __restrict__ cnt) {
    extern __shared__ uint32_t sm_cnt[];                       // [kSortWarps][Nv]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int item = blockIdx.x * kSortWarps + warp;           // (jl, c)
    uint32_t* my = sm_cnt + warp * Nv;
    for (int p = lane; p < Nv; p += 32) my[p] = 0;
    __syncwarp();
    if (item < nj * kSortGroups) {
        const int jl = item / kSortGroups, c = item % kSortGroups;
        const int qper = (Bq + kSortGroups - 1) / kSortGroups;
        const int i0 = c * qper, i1 = min(Bq, i0 + qper);
        const IdxT* base = idx + (size_t)(j0 + jl) * img_pitch;
        for (int i = i0; i < i1; ++i)
            for (int a = lane; a < Nq; a += 32)
                if (row_scale[i * Nq + a] != 0.f) atomicAdd(&my[(int)base[(size_t)i * nq_pad + a]], 1u);
        __syncwarp();
        uint32_t* out = cnt + ((size_t)jl * kSortGroups + c) * Nv;
        for (int p = lane; p < Nv; p += 32) out[p] = my[p];
    }
}

// one thread per (jl, p): running offsets over the groups; then an in-block scan over p
__global__ void __launch_bounds__(1024)
dv_offsets_kernel(const uint32_t* __restrict__ cnt, int nj, int Nv, uint32_t* __restrict__ start,
                  uint32_t* __restrict__ seg) {
    // one block per image, Nv <= 65535 handled with a strided serial scan over 1024-wide tiles
    __shared__ uint32_t tile[1024];
    __shared__ uint32_t carry;
    const int jl = blockIdx.x;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int p0 = 0; p0 < Nv; p0 += 1024) {
        const int p = p0 + threadIdx.x;
        uint32_t tot = 0;
        if (p < Nv)
            for (int c = 0; c < kSortGroups; ++c) tot += cnt[((size_t)jl * kSortGroups + c) * Nv + p];
        tile[threadIdx.x] = tot;
        __syncthreads();
        // Hillis-Steele inclusive scan
        for (int o = 1; o < 1024; o <<= 1) {
            uint32_t x = (threadIdx.x >= (unsigned)o) ? tile[threadIdx.x - o] : 0u;
            __syncthreads();
            tile[threadIdx.x] += x;
            __syncthreads();
        }
        const uint32_t excl = carry + tile[threadIdx.x] - tot;
        if (p < Nv) {
            seg[(size_t)jl * (Nv + 1) + p] = excl;
            uint32_t run = excl;
            for (int c = 0; c < kSortGroups; ++c) {
                start[((size_t)jl * kSortGroups + c) * Nv + p] = run;
                run += cnt[((size_t)jl * kSortGroups + c) * Nv + p];
            }
        }
        __syncthreads();
        if (threadIdx.x == 1023) carry += tile[1023];
        __syncthreads();
    }
    if (threadIdx.x == 0) seg[(size_t)jl * (Nv + 1) + Nv] = carry;
}

template <typename IdxT>
__global__ void __launch_bounds__(kSortWarps * 32)
dv_scatter_sort_kernel(const IdxT* __restrict__ idx, const float* __restrict__ g,
                       const float* __restrict__ row_scale, const uint32_t* __restrict__ start, size_t img_pitch,
                       int j0, int nj, int Bq, int Bv, int Nq, int Nv, int nq_pad, size_t Mrows,
                       DvEntry* __restrict__ entries) {
    extern __shared__ uint32_t sm_cur[];                       // [kSortWarps][Nv]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int item = blockIdx.x * kSortWarps + warp;
    if (item >= nj * kSortGroups) return;
    const int jl = item / kSortGroups, c = item % kSortGroups;
    uint32_t* cur = sm_cur + warp * Nv;
    const uint32_t* st = start + ((size_t)jl * kSortGroups + c) * Nv;
    for (int p = lane; p < Nv; p += 32) cur[p] = st[p];
    __syncwarp();
    const int j = j0 + jl;
    const int qper = (Bq + kSortGroups - 1) / kSortGroups;
    const int i0 = c * qper, i1 = min(Bq, i0 + qper);
    const IdxT* base = idx + (size_t)j * img_pitch;
    DvEntry* out = entries + (size_t)jl * Mrows;
    const uint32_t lt = (1u << lane) - 1u;
    for (int i = i0; i < i1; ++i) {
        const float gij = g[(size_t)i * Bv + j];
        for (int a0 = 0; a0 < Nq; a0 += 32) {
            const int a = a0 + lane;
            // rows with zero weight (padded text tokens, model.py:510) contribute nothing: not listed
            const float rs = (a < Nq) ? row_scale[i * Nq + a] : 0.f;
            const bool valid = rs != 0.f;
            const int p = valid ? (int)base[(size_t)i * nq_pad + a] : -1 - lane;   // distinct dummies
            const uint32_t peers = __match_any_sync(0xffffffffu, p);
            uint32_t pos = 0;
            if (valid) pos = cur[p] + __popc(peers & lt);
            __syncwarp();
            if (valid && (peers & lt) == 0u) cur[p] += __popc(peers);            // group leader advances the cursor
            __syncwarp();
            if (valid) {
                const int r = i * Nq + a;
                DvEntry e; e.row = (uint32_t)r; e.w = rs * gij;
                out[pos] = e;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// dv step 1, grouped variant (bf16 path, Nv <= kGroupMaxNv): NO global count / offset pass.
//   ncu on the three kernels above at cfg 2: count 120 us + offsets 9 us + scatter 320 us, the scatter
//   writing 315 MB to DRAM for a 131 MB list (16.4 M lone 8-byte stores, each dirtying its own sector).
//   Here the rows of a query block are cut into GROUPS of kGroupRows consecutive rows; one CTA sorts one
//   (image, group) by winning patch entirely in shared memory — every lane loads its 32 winners up front
//   (independent loads), per-warp histograms, one scan, a stable placement of 16-bit local row numbers —
//   and writes the group's list as ONE contiguous, fully coalesced run into the group's own region of the
//   entry buffer.  The per-(image, group) segment table replaces the global offsets; the gather walks a
//   patch's list group by group.  Order inside a patch is still "rows ascending", so dv is bit-identical to
//   the global sort's.
// ---------------------------------------------------------------------------------------
constexpr int kGroupRows = 8192;
constexpr int kGroupWarps = 8;
constexpr int kGroupPerLane = kGroupRows / (kGroupWarps * 32);      // 32 rows per lane
constexpr int kGroupMaxQueries = kGroupRows / 16 + 2;               // queries one group touches (nq_pad >= 16)
// Above kGroupMaxNv patches bf16 takes the global sort: the dv pass measured slower with the grouped sort at Nv = 2048
// and 3072, where its tables leave room for one CTA per SM (DESIGN.md, K3b).
constexpr int kGroupMaxNv = 1024;

static constexpr size_t group_sort_smem(int Nv) { return (size_t)kGroupRows * 2 + (size_t)(kGroupWarps + 2) * Nv * 4 + 16; }
static_assert(group_sort_smem(kGroupMaxNv) + kGroupMaxQueries * sizeof(float) <= 227 * 1024,
              "dv grouped sort: shared memory exceeds 227 KB per block");

// Rows are walked in the PADDED index space of the argmax buffer (x = i*nq_pad + a): one image's winners are then
// one contiguous byte string, fetched 16 bytes (16 rows) per lane and load instead of a byte at a time, and the
// (i, a) of a vector comes from one division.  Pad entries (a >= Nq) and zero-weight rows are simply not listed.
// ncu on the byte-at-a-time version: 139 us at cfg 2 with the L1/LSU pipe at 74 % — 64 scalar loads per lane.
template <typename IdxT>
__global__ void __launch_bounds__(kGroupWarps * 32, 3)
dv_group_sort_kernel(const IdxT* __restrict__ idx, const float* __restrict__ g, const float* __restrict__ row_scale,
                     const int masked, size_t img_pitch, int j0, int n_groups, int Mpad, int Bv, int Nq, int Nv, int nq_pad,
                     const FastDiv div_pad, uint32_t* __restrict__ segc, DvEntry* __restrict__ entries) {
    extern __shared__ __align__(16) unsigned char gs_smem[];
    uint16_t* sorted = reinterpret_cast<uint16_t*>(gs_smem);                              // [kGroupRows] local padded row numbers
    uint32_t* hist = reinterpret_cast<uint32_t*>(gs_smem + (size_t)kGroupRows * 2);       // [warps][Nv]
    uint32_t* lbase = hist + kGroupWarps * Nv;                                            // [Nv]
    uint32_t* tot = lbase + Nv;                                                           // [Nv]
    uint32_t* total_s = tot + Nv;

    // 4 rows per load and lane: a warp instruction covers 128 consecutive rows.  (16 rows per lane — one 16-byte load —
    // was tried: fewer loads, but rows then reach the placement step far from row order — the order inside a
    // 512-row window becomes (element, lane) — and the insertion sort of step 3b, which assumes almost sorted runs,
    // grew to 45 % of the kernel: 164 us instead of 139.)
    constexpr int kVec = 4;                                       // rows per load
    constexpr int kLoads = kGroupPerLane / kVec;                  // loads per lane (32 rows per lane)
    using LoadT = typename std::conditional<sizeof(IdxT) == 1, uint32_t, uint2>::type;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int jl = blockIdx.x / n_groups, c = blockIdx.x - jl * n_groups;
    const int j = j0 + jl;
    const int x_group = c * kGroupRows;
    const IdxT* base = idx + (size_t)j * img_pitch;

    for (int k = tid; k < kGroupWarps * Nv; k += blockDim.x) hist[k] = 0;
    // g[i][j] of the queries this group touches (<= kGroupMaxQueries of them): step 4 looks its weights up here
    // instead of issuing one scattered global load per entry (32 sectors per warp instruction)
    __shared__ float gq_s[kGroupMaxQueries];
    const uint32_t i_first = fast_div((uint32_t)x_group, div_pad);
    {
        const int x_last = min(x_group + kGroupRows, Mpad) - 1;
        const int nq_here = (int)fast_div((uint32_t)x_last, div_pad) - (int)i_first + 1;
        for (int t = tid; t < nq_here; t += blockDim.x) gq_s[t] = g[(size_t)(i_first + t) * Bv + j];
    }
    __syncthreads();

    // ---- 1. every lane fetches its 32 winners (kLoads independent vector loads), then the per-warp histogram.
    //         Winners are kept packed two per register (0xffff = pad entry, row beyond the block, or zero weight).
    //         Lane's local row of (load v, element e): warp*1024 + v*32*kVec + lane*kVec + e. ----
    uint32_t pv[kGroupPerLane / 2];
    uint32_t* myh = hist + warp * Nv;
    {
        LoadT raw[kLoads];
#pragma unroll
        for (int v = 0; v < kLoads; ++v) {
            const int x = x_group + warp * (kGroupPerLane * 32) + v * 32 * kVec + lane * kVec;
            raw[v] = LoadT();
            if (x < Mpad) raw[v] = __ldg(reinterpret_cast<const LoadT*>(base + x));        // nq_pad % 16 == 0: never straddles
        }
#pragma unroll
        for (int v = 0; v < kLoads; ++v) {
            const int x = x_group + warp * (kGroupPerLane * 32) + v * 32 * kVec + lane * kVec;
            const uint32_t qi = fast_div((uint32_t)x, div_pad);
            const int a0 = x - (int)qi * nq_pad;
            uint32_t w32[2];
            if constexpr (sizeof(IdxT) == 1) { w32[0] = raw[v]; w32[1] = 0u; } else { w32[0] = raw[v].x; w32[1] = raw[v].y; }
#pragma unroll
            for (int e = 0; e < kVec; ++e) {
                uint32_t p = sizeof(IdxT) == 1 ? (w32[0] >> (8 * e)) & 0xffu : (w32[e >> 1] >> (16 * (e & 1))) & 0xffffu;
                bool ok = x < Mpad && a0 + e < Nq;
                if (masked && ok) ok = row_scale[(size_t)qi * Nq + a0 + e] != 0.f;
                if (!ok) p = 0xffffu;
                const int k = v * kVec + e;
                if (k & 1) pv[k >> 1] |= p << 16; else pv[k >> 1] = p;
            }
        }
#pragma unroll
        for (int k = 0; k < kGroupPerLane; ++k) {
            const uint32_t p = (pv[k >> 1] >> ((k & 1) * 16)) & 0xffffu;
            if (p != 0xffffu) atomicAdd(&myh[p], 1u);
        }
    }
    __syncthreads();
    // ---- 2. per patch: exclusive prefix over the warps, then an exclusive scan over the patches ----
    for (int p = tid; p < Nv; p += blockDim.x) {
        uint32_t run = 0;
        for (int w = 0; w < kGroupWarps; ++w) { const uint32_t t = hist[w * Nv + p]; hist[w * Nv + p] = run; run += t; }
        tot[p] = run;
    }
    __syncthreads();
    uint32_t* seg_out = segc + (size_t)blockIdx.x * (Nv + 1);
    if (warp == 0) {
        uint32_t carry = 0;
        for (int p0 = 0; p0 < Nv; p0 += 32) {
            const int p = p0 + lane;
            const uint32_t v = (p < Nv) ? tot[p] : 0u;
            uint32_t incl = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
            if (p < Nv) { lbase[p] = carry + incl - v; seg_out[p] = carry + incl - v; }
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) { *total_s = carry; seg_out[Nv] = carry; }
    }
    __syncthreads();
    // ---- 3. placement.  Slot = run start + this warp's prefix + a shared-memory atomic counter; step 3b sorts every
    //         patch's run by row (insertion sort over an almost sorted run of ~Rows/Nv 16-bit values, one thread per
    //         patch), which makes the order "rows ascending" whatever order the atomics resolved in. ----
#pragma unroll
    for (int k = 0; k < kGroupPerLane; ++k) {
        const uint32_t pk = (pv[k >> 1] >> ((k & 1) * 16)) & 0xffffu;
        if (pk != 0xffffu) {
            const uint32_t slot = lbase[pk] + atomicAdd(&myh[pk], 1u);
            const int v = k / kVec, e = k - v * kVec;
            sorted[slot] = (uint16_t)(warp * (kGroupPerLane * 32) + v * 32 * kVec + lane * kVec + e);
        }
    }
    __syncthreads();
    for (int p = tid; p < Nv; p += blockDim.x) {
        const uint32_t b0 = lbase[p], cnt = tot[p];
        for (uint32_t u = 1; u < cnt; ++u) {
            const uint16_t key = sorted[b0 + u];
            uint32_t v = u;
            while (v > 0 && sorted[b0 + v - 1] > key) { sorted[b0 + v] = sorted[b0 + v - 1]; --v; }
            sorted[b0 + v] = key;
        }
    }
    __syncthreads();
    // ---- 4. the group's list leaves as one contiguous run; the (unpadded) row number and the weight are attached here ----
    const uint32_t n = *total_s;
    DvEntry* out = entries + (size_t)blockIdx.x * kGroupRows;
    const float rs_uniform = masked ? 0.f : row_scale[0];                      // no mask: every row weighs 1/Nq
#pragma unroll 8
    for (uint32_t t = tid; t < n; t += kGroupWarps * 32) {
        const uint32_t x = (uint32_t)x_group + (uint32_t)sorted[t];
        const uint32_t i = fast_div(x, div_pad);
        const uint32_t r = x - i * (uint32_t)(nq_pad - Nq);                    // i*Nq + a
        DvEntry d; d.row = r; d.w = (masked ? row_scale[r] : rs_uniform) * gq_s[i - i_first];
        out[t] = d;
    }
}

// ---------------------------------------------------------------------------------------
// dv step 2: one warp per (image, patch) segment and 32-chunk column block of D (a 512-byte
// bf16 column block per warp: D = 512 -> 2 warps per segment); lanes own 16-byte chunks; the
// (row, weight) list is read 32 entries at a time (the next 32 prefetched) and broadcast with
// shuffles; kU rows in flight per warp.  The pass is L2-latency bound, so it is shaped for
// bytes in flight: few registers per thread (many resident warps) x kU independent loads each.
// ---------------------------------------------------------------------------------------
constexpr int kDvU = 8;

template <typename T, typename OutT>
__global__ void __launch_bounds__(256)
dv_gather_kernel(const T* __restrict__ q, const DvEntry* __restrict__ entries, const uint32_t* __restrict__ seg,
                 const float* __restrict__ Tptr, int j0, int nj, int Nv, int D, int wps, size_t Mrows,
                 int accumulate, OutT* __restrict__ dv) {
    constexpr int E = Vec16<T>::kElems;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long wid = (long long)blockIdx.x * 8 + warp;
    const long long sid = wid / wps;
    const int ch = (int)(wid - sid * wps) * 32 + lane;          // this lane's 16-byte chunk of the row
    if (sid >= (long long)nj * Nv) return;
    const bool act = ch * E < D;
    const int jl = (int)(sid / Nv), p = (int)(sid % Nv);
    const uint32_t e0 = seg[(size_t)jl * (Nv + 1) + p], e1 = seg[(size_t)jl * (Nv + 1) + p + 1];
    const DvEntry* list = entries + (size_t)jl * Mrows;
    const T* qc = q + (act ? ch * E : 0);

    float acc[E];
#pragma unroll
    for (int c = 0; c < E; ++c) acc[c] = 0.f;

    DvEntry next; next.row = 0; next.w = 0.f;
    if (e0 + lane < e1) next = list[e0 + lane];
    for (uint32_t base = e0; base < e1; base += 32) {
        const DvEntry mine = next;
        next.row = 0; next.w = 0.f;
        if (base + 32 + lane < e1) next = list[base + 32 + lane];
        const int n = min(32u, e1 - base);
        for (int l = 0; l < n; l += kDvU) {
            float f[kDvU][E];
            float w[kDvU];
#pragma unroll
            for (int u = 0; u < kDvU; ++u) {
                // slots past n re-read the segment's last entry with weight 0: no branch in the batch
                const int src = min(l + u, n - 1);
                const uint32_t r = __shfl_sync(0xffffffffu, mine.row, src);
                const float ww = __shfl_sync(0xffffffffu, mine.w, src);
                w[u] = (l + u < n) ? ww : 0.f;
                Vec16<T>::load(qc + (size_t)r * D, f[u]);
            }
#pragma unroll
            for (int u = 0; u < kDvU; ++u)
#pragma unroll
                for (int c = 0; c < E; ++c) acc[c] = fmaf(w[u], f[u][c], acc[c]);
        }
    }
    if (act) {
        const float Tval = *Tptr;
        float o[E];
#pragma unroll
        for (int c = 0; c < E; ++c) o[c] = acc[c] * Tval;
        OutT* dst = dv + ((size_t)(j0 + jl) * Nv + p) * D + ch * E;
        if (accumulate) {                       // later query blocks add to the fp32 partial of the earlier ones
            float prev[E];
            LoadAs<OutT, E>::get(dst, prev);
#pragma unroll
            for (int c = 0; c < E; ++c) o[c] = __fmaf_rn(acc[c], Tval, prev[c]);    // explicit: both gather kernels round alike
        }
        StoreAs<OutT, E>::put(dst, o);
    }
}

// dv step 2, bf16: the gather above over the GROUPED lists of dv_group_sort_kernel, shaped for the two things ncu
// shows the generic kernel short of — bytes in flight (its 102 registers allow 16 warps/SM; L2 throughput sits at
// 44 %) and issue slots (54 % busy, mostly bf16 unpacking and scalar FMAs):
//   * rows stay PACKED (one uint4 per lane and row) until they are consumed, so kU rows in flight cost
//     4*kU registers instead of 8*kU and kMinBlocks CTAs fit per SM;
//   * FFMA2 (two fp32 FMAs per issue slot) on the (lo,hi) halves of every 32-bit word;
//   * the byte offset of the row is computed once per entry, before the broadcast.
// Same summation order as the generic kernel (entries in list order, fp32), so the results are
// bit-identical to it.
__device__ __forceinline__ void ffma2_pair(float2& acc, float w, uint32_t pair) {
    float2 wv = make_float2(w, w);
    float2 vv = make_float2(__uint_as_float(pair << 16), __uint_as_float(pair & 0xffff0000u));
    unsigned long long a = *reinterpret_cast<unsigned long long*>(&acc);
    const unsigned long long b = *reinterpret_cast<unsigned long long*>(&wv);
    const unsigned long long c = *reinterpret_cast<unsigned long long*>(&vv);
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a) : "l"(b), "l"(c));
    acc = *reinterpret_cast<float2*>(&a);
}

// The (row, weight) list of (image, patch) is the concatenation, over the groups c, of
// entries[jl][c][segc[jl][c][p] .. segc[jl][c][p+1]), with Mrows entry slots per image: n_groups * kGroupRows for
// the lists of dv_group_sort_kernel; the global sort's list is one group of the block's rows.  The first batch of
// the next group is requested before the current group's rows are consumed.
// kW = 16-byte chunks per lane and row: kW = 1 -> a warp covers 512 bytes of the row (D = 512: two warps per
// segment, each walking the entry list); kW = 2 -> one warp covers 1 KB with two loads per row, halving the
// list/shuffle overhead per byte.
template <typename OutT, int kU, int kW, int kMinBlocks>
__global__ void __launch_bounds__(256, kMinBlocks)
dv_gather_grouped_kernel(const __nv_bfloat16* __restrict__ q, const DvEntry* __restrict__ entries,
                         const uint32_t* __restrict__ segc, const float* __restrict__ Tptr, int j0, int nj, int n_groups,
                         size_t Mrows, int Nv, int D, int wps, int accumulate, OutT* __restrict__ dv) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long wid = (long long)blockIdx.x * 8 + warp;
    const long long sid = wid / wps;
    const int ch0 = (int)(wid - sid * wps) * 32 * kW + lane;
    if (sid >= (long long)nj * Nv) return;
    const int jl = (int)(sid / Nv), p = (int)(sid % Nv);
    // 32-bit byte offsets from the (uniform) block base: a query block is <= 64 MB (dv_plan), so the
    // address is one register per row in flight instead of two
    const char* qbase = reinterpret_cast<const char*>(q);
    const uint32_t row_bytes = (uint32_t)D * 2u;
    bool act[kW];
    uint32_t lane_off[kW];
#pragma unroll
    for (int k = 0; k < kW; ++k) { act[k] = (ch0 + 32 * k) * 8 < D; lane_off[k] = act[k] ? (uint32_t)(ch0 + 32 * k) * 16u : 0u; }

    float2 acc[kW][4];
#pragma unroll
    for (int k = 0; k < kW; ++k)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[k][c] = make_float2(0.f, 0.f);

    const uint32_t* sg = segc + (size_t)jl * n_groups * (Nv + 1) + p;
    const DvEntry* lists = entries + (size_t)jl * Mrows;
    // segment bounds of 32 groups at a time live in lane registers (lane c <-> group c0 + c): no dependent
    // table load per group
    uint32_t myE0 = 0, myE1 = 0;
    if (lane < n_groups) { myE0 = sg[(size_t)lane * (Nv + 1)]; myE1 = sg[(size_t)lane * (Nv + 1) + 1]; }
    uint32_t e0 = __shfl_sync(0xffffffffu, myE0, 0), e1 = __shfl_sync(0xffffffffu, myE1, 0);
    DvEntry next; next.row = 0; next.w = 0.f;
    if (e0 + lane < e1) next = lists[e0 + lane];
    for (int c = 0; c < n_groups; ++c) {
        const DvEntry* list = lists + (size_t)c * kGroupRows;
        uint32_t f0 = 0, f1 = 0;                                   // the next group's segment
        if (c + 1 < n_groups) {
            if (((c + 1) & 31) == 0) {                             // refill the lane registers
                myE0 = myE1 = 0;
                if (c + 1 + lane < n_groups) { myE0 = sg[(size_t)(c + 1 + lane) * (Nv + 1)]; myE1 = sg[(size_t)(c + 1 + lane) * (Nv + 1) + 1]; }
            }
            f0 = __shfl_sync(0xffffffffu, myE0, (c + 1) & 31);
            f1 = __shfl_sync(0xffffffffu, myE1, (c + 1) & 31);
        }
        const DvEntry* nlist = list + kGroupRows;
        if (e0 >= e1) {                                            // empty here: `next` must become the next group's first batch
            next.row = 0; next.w = 0.f;
            if (f0 + lane < f1) next = nlist[f0 + lane];
        }
        for (uint32_t base = e0; base < e1; base += 32) {
            const uint32_t my_row = next.row;
            const float my_w = next.w;
            next.row = 0; next.w = 0.f;
            if (base + 32 < e1) { if (base + 32 + lane < e1) next = list[base + 32 + lane]; }
            else if (f0 + lane < f1) next = nlist[f0 + lane];
            const int n = min(32u, e1 - base);
            for (int l = 0; l < n; l += kU) {
                uint4 d[kU][kW];
                float w[kU];
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    const int src = min(l + u, n - 1);
                    const uint32_t row = __shfl_sync(0xffffffffu, my_row, src);
                    const float ww = __shfl_sync(0xffffffffu, my_w, src);
                    w[u] = (l + u < n) ? ww : 0.f;
#pragma unroll
                    for (int k = 0; k < kW; ++k)
                        d[u][k] = __ldg(reinterpret_cast<const uint4*>(qbase + (row * row_bytes + lane_off[k])));
                }
#pragma unroll
                for (int u = 0; u < kU; ++u)
#pragma unroll
                    for (int k = 0; k < kW; ++k) {
                        ffma2_pair(acc[k][0], w[u], d[u][k].x); ffma2_pair(acc[k][1], w[u], d[u][k].y);
                        ffma2_pair(acc[k][2], w[u], d[u][k].z); ffma2_pair(acc[k][3], w[u], d[u][k].w);
                    }
            }
        }
        e0 = f0; e1 = f1;
    }
    const float Tval = *Tptr;
#pragma unroll
    for (int k = 0; k < kW; ++k) {
        if (!act[k]) continue;
        float o[8];
#pragma unroll
        for (int c = 0; c < 4; ++c) { o[2 * c] = acc[k][c].x * Tval; o[2 * c + 1] = acc[k][c].y * Tval; }
        OutT* dst = dv + ((size_t)(j0 + jl) * Nv + p) * D + (ch0 + 32 * k) * 8;
        if (accumulate) {
            float prev[8];
            LoadAs<OutT, 8>::get(dst, prev);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                o[2 * c] = __fmaf_rn(acc[k][c].x, Tval, prev[2 * c]);
                o[2 * c + 1] = __fmaf_rn(acc[k][c].y, Tval, prev[2 * c + 1]);
            }
        }
        StoreAs<OutT, 8>::put(dst, o);
    }
}

// ---------------------------------------------------------------------------------------
// dT = sum g*clip / T.  Up to kDtMaxBlocks CTAs sum contiguous chunks (fp64, fixed order inside a
// CTA); the last CTA to take a ticket adds the per-CTA partials in CTA order — deterministic, and
// a B = 8192 rank block (8 M elements) is no longer read by a single SM.
// ---------------------------------------------------------------------------------------
constexpr int kDtMaxBlocks = 128;
constexpr size_t kCtrlBytes = 4096;        // workspace control block: [0] abort flag, [16] dT ticket, [64..] dT partials

__global__ void __launch_bounds__(1024)
dT_kernel(const float* __restrict__ g, const float* __restrict__ clip, size_t n, size_t per_block,
          const float* __restrict__ Tptr, float* __restrict__ dT, double* __restrict__ partials,
          unsigned int* __restrict__ ticket) {
    __shared__ double red[32];
    __shared__ bool is_last;
    const size_t k0 = (size_t)blockIdx.x * per_block;
    const size_t k1 = k0 + per_block < n ? k0 + per_block : n;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;      // four independent chains: the loads of one thread overlap
    size_t k = k0 + threadIdx.x;
    for (; k + 3 * 1024 < k1; k += 4 * 1024) {
        const float g0 = g[k], g1 = g[k + 1024], g2 = g[k + 2048], g3 = g[k + 3072];
        const float c0 = clip[k], c1 = clip[k + 1024], c2 = clip[k + 2048], c3 = clip[k + 3072];
        a0 += (double)g0 * (double)c0; a1 += (double)g1 * (double)c1;
        a2 += (double)g2 * (double)c2; a3 += (double)g3 * (double)c3;
    }
    for (; k < k1; k += 1024) a0 += (double)g[k] * (double)clip[k];
    double a = (a0 + a1) + (a2 + a3);
    a = warp_sum_d(a);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x < 32) {
        double b = red[threadIdx.x];
        b = warp_sum_d(b);
        if (threadIdx.x == 0) {
            partials[blockIdx.x] = b;
            __threadfence();
            is_last = atomicAdd(ticket, 1u) == gridDim.x - 1u;
        }
    }
    __syncthreads();
    if (is_last && threadIdx.x == 0) {
        __threadfence();
        double t = 0.0;
        for (unsigned b = 0; b < gridDim.x; ++b) t += ((volatile double*)partials)[b];
        *dT = (float)(t / (double)*Tptr);
        *ticket = 0u;
    }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
// The dv pass is tiled twice so that its working sets stay on chip whatever the batch size:
//   * over QUERY BLOCKS of <= kDvBlockBytes of q rows (64 MB: the block a warp gathers from stays
//     L2-resident; at B=256 the whole q is one block) — later blocks accumulate into the output;
//   * over IMAGE BATCHES that bound the sorted entry list to ~1 GiB.
constexpr size_t kDvBlockBytes = (size_t)64 << 20;
struct DvPlan {
    int jb;                 // images per batch
    int qb;                 // queries per block
    int nblk;               // number of query blocks
    bool scratch;           // fp32 scratch needed (several blocks and a non-fp32 output)
    size_t off_cnt, off_start, off_seg, off_segc, off_entries, off_scratch, total;
};
static DvPlan dv_plan(int Bq, int Bv, int Nq, int Nv, int D, int elt_bytes, bool out_f32, size_t block_bytes = kDvBlockBytes) {
    DvPlan pl;
    size_t qb = block_bytes / ((size_t)Nq * D * elt_bytes);
    if (qb < 1) qb = 1;
    if (qb > (size_t)Bq) qb = Bq;
    pl.qb = (int)qb;
    pl.nblk = (int)(((size_t)Bq + qb - 1) / qb);
    pl.scratch = pl.nblk > 1 && !out_f32;
    const size_t Mb = qb * Nq;                                       // rows per block
    const size_t Mp = qb * (size_t)nq_padded(Nq);                    // ... in the padded index space the grouped sort walks
    const size_t ng = (Mp + kGroupRows - 1) / kGroupRows;            // sort groups per block (grouped path)
    const size_t Me = ng * kGroupRows > Mb ? ng * kGroupRows : Mb;   // entry slots per image (both sort paths fit)
    size_t jb = ((size_t)1 << 30) / (Me * sizeof(DvEntry));
    if (pl.scratch) {                                                // keep the fp32 scratch <= 256 MB
        const size_t js = ((size_t)256 << 20) / ((size_t)Nv * D * 4);
        if (jb > js) jb = js;
    }
    if (jb < 1) jb = 1;
    if (jb > (size_t)Bv) jb = Bv;
    pl.jb = (int)jb;
    size_t o = kCtrlBytes;                                // control block (watchdog flag, dT ticket and partials)
    pl.off_cnt = o;     o += align_up(jb * kSortGroups * (size_t)Nv * 4, 256);
    pl.off_start = o;   o += align_up(jb * kSortGroups * (size_t)Nv * 4, 256);
    pl.off_seg = o;     o += align_up(jb * ((size_t)Nv + 1) * 4, 256);
    pl.off_segc = o;    o += align_up(jb * ng * ((size_t)Nv + 1) * 4, 256);
    pl.off_entries = o; o += align_up(jb * Me * sizeof(DvEntry), 256);
    pl.off_scratch = o; o += pl.scratch ? align_up(jb * (size_t)Nv * D * 4, 256) : 0;
    pl.total = o;
    return pl;
}

template <typename T, typename IdxT>
static int bwd_typed(const void* q, const void* v, const void* idx, const float* g,
                     const float* clip, const float* row_scale, const float* Tp,
                     int Bq, int Bv, int Nq, int Nv, int D,
                     void* dq, void* dv, int dv_f32, float* dT, void* ws, size_t pack_maps_offset, int bwd_flags, cudaStream_t st) {
    const int M = Bq * Nq;
    const int nq_pad = nq_padded(Nq);
    constexpr int E = Vec16<T>::kElems;
    const int kch = ceil_div(D / E, 32);
    if (dq && (kch < 1 || kch > 4)) return fail_msg(TRIAD_ERR_UNSUPPORTED, "maxmean_bwd: D too large (max 1024 bf16 / 512 fp32)");
    if (dq && sizeof(T) == 2 && !(bwd_flags & TRIAD_BWD_GENERIC_DQ) &&
        (sizeof(IdxT) == 1 ? dq_pipe_supported(Nv, D, TRIAD_DTYPE_BF16) : dq_tile_supported(D, TRIAD_DTYPE_BF16))) {
        if constexpr (sizeof(IdxT) == 1) {
            // the software-pipelined shared-memory gather (bwd_dq_pipe.cu); TRIAD_BWD_PACK_ROWS (masked text queries):
            // only the 8-row groups that hold a row with a non-zero weight are swept
            const int* glist = nullptr;
            const int* n_groups = nullptr;
            if (bwd_flags & TRIAD_BWD_PACK_ROWS) {
                void* maps = (char*)ws + pack_maps_offset;
                const int rcm = launch_pack_groups(row_scale, Bq, Nq, maps, st);
                if (rcm) return rcm;
                n_groups = (const int*)maps + Bq;
                glist = (const int*)maps + Bq + 1;
            }
            const int rc = launch_dq_pipe(v, idx, g, row_scale, Tp, Bq, Bv, Nq, Nv, D, dq, (int*)ws, glist, n_groups, st);
            if (rc) return rc;
        } else {
            // the L1-resident gather (bwd_dq_tile.cu) sweeps every row, TRIAD_BWD_PACK_ROWS or not
            const int rc = launch_dq_tile(v, idx, g, row_scale, Tp, M, Bv, Nq, Nv, D, dq, st);
            if (rc) return rc;
        }
    } else if (dq) {
        const int grid = ceil_div(M, kDqRows);
#define TRIAD_DQ(K) dq_gather_kernel<T, IdxT, K><<<grid, 256, 0, st>>>( \
        (const T*)v, (const IdxT*)idx, g, row_scale, Tp, M, Bv, Nq, Nv, D, nq_pad, (T*)dq)
        switch (kch) {
            case 1: TRIAD_DQ(1); break;
            case 2: TRIAD_DQ(2); break;
            case 3: TRIAD_DQ(3); break;
            default: TRIAD_DQ(4); break;
        }
#undef TRIAD_DQ
        TRIAD_LAUNCH_CHECK("dq_gather_kernel");
    }
    if (dv) {
        const bool out_f32 = dv_f32 || sizeof(T) == 4;
        // TRIAD_BWD_SMALL_BLOCKS (tests): 64 KB query blocks, so small shapes exercise the multi-block path
        const DvPlan pl = dv_plan(Bq, Bv, Nq, Nv, D, (int)sizeof(T), out_f32,
                                  (bwd_flags & TRIAD_BWD_SMALL_BLOCKS) ? ((size_t)64 << 10) : kDvBlockBytes);
        uint32_t* cnt = (uint32_t*)((char*)ws + pl.off_cnt);
        uint32_t* start = (uint32_t*)((char*)ws + pl.off_start);
        uint32_t* seg = (uint32_t*)((char*)ws + pl.off_seg);
        uint32_t* segc = (uint32_t*)((char*)ws + pl.off_segc);
        DvEntry* entries = (DvEntry*)((char*)ws + pl.off_entries);
        float* scratch = (float*)((char*)ws + pl.off_scratch);
        const size_t smem = (size_t)kSortWarps * Nv * 4;                          // <= 48 KB: Nv <= kDvMaxNv
        // bf16: the packed FFMA2 gather, over the grouped sort's lists up to kGroupMaxNv patches and over the global
        // sort's list beyond; fp32 and TRIAD_BWD_GENERIC_DV: the global sort and the generic gather
        const bool packed = sizeof(T) == 2 && !(bwd_flags & TRIAD_BWD_GENERIC_DV);
        const bool grouped = packed && Nv <= kGroupMaxNv;
        const size_t img_pitch = (size_t)Bq * nq_pad;
        const int wps = ceil_div(D / E, 32);                                       // warps per segment
        const bool add_first = (bwd_flags & TRIAD_BWD_ACCUMULATE_DV) != 0;        // fp32 out (checked): no scratch
        for (int j0 = 0; j0 < Bv; j0 += pl.jb) {
            const int nj = (Bv - j0 < pl.jb) ? (Bv - j0) : pl.jb;
            const int sort_grid = ceil_div(nj * kSortGroups, kSortWarps);
            const long long nwarps = (long long)nj * Nv * wps;
            const unsigned ggrid = (unsigned)((nwarps + 7) / 8);
            for (int b = 0; b < pl.nblk; ++b) {
                const int q0 = b * pl.qb;
                const int nq = (Bq - q0 < pl.qb) ? (Bq - q0) : pl.qb;
                const size_t Mb = (size_t)nq * Nq;
                const IdxT* idx_b = (const IdxT*)idx + (size_t)q0 * nq_pad;
                const float* rs_b = row_scale + (size_t)q0 * Nq;
                const float* g_b = g + (size_t)q0 * Bv;
                const T* q_b = (const T*)q + (size_t)q0 * Nq * D;
                // the sort leaves n_groups lists per image (Mrows entry slots per image) and their segment table in segs
                const uint32_t* segs = seg;
                int n_groups = 1;
                size_t Mrows = Mb;
                if (grouped) {                                     // shared-memory sort per (image, row group)
                    const int Mpad = nq * nq_pad;
                    n_groups = ceil_div(Mpad, kGroupRows);
                    Mrows = (size_t)n_groups * kGroupRows;
                    segs = segc;
                    auto skern = dv_group_sort_kernel<IdxT>;
                    TRIAD_SET_MAX_SMEM(skern, group_sort_smem(kGroupMaxNv));
                    skern<<<nj * n_groups, kGroupWarps * 32, group_sort_smem(Nv), st>>>(
                        idx_b, g_b, rs_b, (bwd_flags & TRIAD_BWD_UNIFORM_SCALE) ? 0 : 1, img_pitch, j0, n_groups, Mpad, Bv, Nq, Nv,
                        nq_pad, make_fastdiv((uint32_t)nq_pad), segc, entries);
                    TRIAD_LAUNCH_CHECK("dv_group_sort_kernel");
                } else {                                           // global sort: one list per image
                    dv_count_kernel<IdxT><<<sort_grid, kSortWarps * 32, smem, st>>>(idx_b, rs_b, img_pitch, j0, nj, nq, Nq, Nv, nq_pad, cnt);
                    TRIAD_LAUNCH_CHECK("dv_count_kernel");
                    dv_offsets_kernel<<<nj, 1024, 0, st>>>(cnt, nj, Nv, start, seg);
                    TRIAD_LAUNCH_CHECK("dv_offsets_kernel");
                    dv_scatter_sort_kernel<IdxT><<<sort_grid, kSortWarps * 32, smem, st>>>(
                        idx_b, g_b, rs_b, start, img_pitch, j0, nj, nq, Bv, Nq, Nv, nq_pad, Mb, entries);
                    TRIAD_LAUNCH_CHECK("dv_scatter_sort_kernel");
                }
                // the gather
                if (packed) {
                    const __nv_bfloat16* qb16 = (const __nv_bfloat16*)q_b;
                    // rows of more than 512 bytes: one warp per segment, two 16-byte loads per lane and row
                    // (measured at cfg 2: 1.46 -> 1.36 ms for the whole dv pass); otherwise one load per lane
                    const bool wide_rows = D > 256;
#define TRIAD_DVG_K(OUT, DST, J0, U, W, MB) do { \
                        const int wps_ = ceil_div(D / 8, 32 * W); \
                        const unsigned grid_ = (unsigned)(((long long)nj * Nv * wps_ + 7) / 8); \
                        dv_gather_grouped_kernel<OUT, U, W, MB><<<grid_, 256, 0, st>>>(qb16, entries, segs, Tp, J0, nj, n_groups, Mrows, Nv, D, wps_, b > 0 || add_first, DST); \
                    } while (0)
#define TRIAD_DVG(OUT, DST, J0) \
                    if (wide_rows) TRIAD_DVG_K(OUT, DST, J0, 4, 2, 4); else TRIAD_DVG_K(OUT, DST, J0, 8, 1, 3);
                    if (pl.scratch) { TRIAD_DVG(float, scratch, 0) }
                    else if (out_f32) { TRIAD_DVG(float, (float*)dv, j0) }
                    else { TRIAD_DVG(__nv_bfloat16, (__nv_bfloat16*)dv, j0) }
#undef TRIAD_DVG
#undef TRIAD_DVG_K
                    TRIAD_LAUNCH_CHECK("dv_gather_grouped_kernel");
                } else {
                    if (pl.scratch)      // accumulate this image batch in fp32 scratch (local image index), convert at the end
                        dv_gather_kernel<T, float><<<ggrid, 256, 0, st>>>(q_b, entries, seg, Tp, 0, nj, Nv, D, wps, Mb, b > 0, scratch);
                    else if (out_f32)
                        dv_gather_kernel<T, float><<<ggrid, 256, 0, st>>>(q_b, entries, seg, Tp, j0, nj, Nv, D, wps, Mb, b > 0 || add_first, (float*)dv);
                    else
                        dv_gather_kernel<T, T><<<ggrid, 256, 0, st>>>(q_b, entries, seg, Tp, j0, nj, Nv, D, wps, Mb, b > 0, (T*)dv);
                    TRIAD_LAUNCH_CHECK("dv_gather_kernel");
                }
            }
            if (pl.scratch) {
                const size_t n = (size_t)nj * Nv * D;
                dv_convert_kernel<T><<<(unsigned)((n + 2047) / 2048 > 4096 ? 4096 : (n + 2047) / 2048), 256, 0, st>>>(
                    scratch, n, (T*)dv + (size_t)j0 * Nv * D);
                TRIAD_LAUNCH_CHECK("dv_convert_kernel");
            }
        }
    }
    if (dT) {
        const size_t n = (size_t)Bq * Bv;
        int nb = (int)((n + 16383) / 16384);
        if (nb > kDtMaxBlocks) nb = kDtMaxBlocks;
        const size_t per_block = (n + nb - 1) / nb;
        dT_kernel<<<nb, 1024, 0, st>>>(g, clip, n, per_block, Tp, dT, (double*)((char*)ws + 64), (unsigned int*)((char*)ws + 16));
        TRIAD_LAUNCH_CHECK("dT_kernel");
    }
    return TRIAD_OK;
}

}  // namespace triad

using namespace triad;

// every TRIAD_BWD_* bit; any other bit is an error rather than silently ignored
static constexpr int kBwdFlags = TRIAD_BWD_GENERIC_DQ | TRIAD_BWD_GENERIC_DV | TRIAD_BWD_SMALL_BLOCKS | TRIAD_BWD_PACK_ROWS |
                                 TRIAD_BWD_UNIFORM_SCALE | TRIAD_BWD_TEST_TRIP_WATCHDOG | TRIAD_BWD_ACCUMULATE_DV;

extern "C" size_t triad_maxmean_bwd_workspace_bytes(int Bq, int Bv, int Nq, int Nv, int D, int dtype) {
    if (Bq <= 0 || Bv <= 0 || Nq <= 0 || Nv <= 0 || D <= 0) return 0;
    // the caller may ask for dv in `dtype` (fp32 scratch when several query blocks) or as an fp32 partial
    const int eb = dtype == TRIAD_DTYPE_BF16 ? 2 : 4;
    size_t best = 0;
    for (int f32 = 0; f32 < 2; ++f32)
        for (int small = 0; small < 2; ++small) {
            const size_t t = dv_plan(Bq, Bv, Nq, Nv, D, eb, f32 != 0, small ? ((size_t)64 << 10) : kDvBlockBytes).total;
            if (t > best) best = t;
        }
    return best + pack_map_bytes(Bq, Nq);                 // the packing maps of TRIAD_BWD_PACK_ROWS live at the end
}

extern "C" int triad_maxmean_bwd(const void* q, const void* v, const void* idx, const float* g,
                                 const float* clip, const float* row_scale, const float* temperature,
                                 int Bq, int Bv, int Nq, int Nv, int D, int dtype,
                                 void* dq, void* dv, int dv_f32, float* dT,
                                 void* ws, size_t ws_bytes, int flags, void* stream) {
    if (!q || !v || !idx || !g || !row_scale || !temperature) return fail_msg(TRIAD_ERR_BAD_ARG, "maxmean_bwd: null pointer");
    if (dT && !clip) return fail_msg(TRIAD_ERR_BAD_ARG, "maxmean_bwd: dT needs clip");
    if (Bq <= 0 || Bv <= 0 || Nq <= 0 || Nv <= 0 || D <= 0 || D % 8 != 0 || Nv > 65535)
        return fail_msg(TRIAD_ERR_BAD_SHAPE, "maxmean_bwd: bad shape");
    if (dtype != TRIAD_DTYPE_F32 && dtype != TRIAD_DTYPE_BF16) return fail_msg(TRIAD_ERR_BAD_ARG, "maxmean_bwd: dtype");
    if (flags & ~kBwdFlags) return fail_msg(TRIAD_ERR_BAD_ARG, "maxmean_bwd: unknown flag bit");
    if ((flags & TRIAD_BWD_ACCUMULATE_DV) && !dv_f32 && dtype != TRIAD_DTYPE_F32)
        return fail_msg(TRIAD_ERR_BAD_ARG, "maxmean_bwd: TRIAD_BWD_ACCUMULATE_DV needs an fp32 dv");
    if (dv && Nv > kDvMaxNv) return fail_msg(TRIAD_ERR_UNSUPPORTED, "maxmean_bwd: dv needs Nv <= 3072");
    if (((uintptr_t)q | (uintptr_t)v | (uintptr_t)dq | (uintptr_t)dv | (uintptr_t)ws) & 15) return fail_msg(TRIAD_ERR_ALIGNMENT, "maxmean_bwd: 16-byte alignment");
    if (!ws || ws_bytes < ((dv || (flags & TRIAD_BWD_PACK_ROWS)) ? triad_maxmean_bwd_workspace_bytes(Bq, Bv, Nq, Nv, D, dtype) : kCtrlBytes))
        return fail_msg(TRIAD_ERR_WORKSPACE, "maxmean_bwd: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    TRIAD_CUDA_CHECK(cudaMemsetAsync(ws, 0, kCtrlBlockBytes, st));      // abort flag + dT ticket
    if (flags & TRIAD_BWD_TEST_TRIP_WATCHDOG) TRIAD_CUDA_CHECK(cudaMemsetAsync(ws, 1, 4, st));
    const bool wide = Nv > 256;
    const size_t pmo = triad_maxmean_bwd_workspace_bytes(Bq, Bv, Nq, Nv, D, dtype) - pack_map_bytes(Bq, Nq);
    if (dtype == TRIAD_DTYPE_BF16) {
        return wide ? bwd_typed<__nv_bfloat16, uint16_t>(q, v, idx, g, clip, row_scale, temperature, Bq, Bv, Nq, Nv, D, dq, dv, dv_f32, dT, ws, pmo, flags, st)
                    : bwd_typed<__nv_bfloat16, uint8_t>(q, v, idx, g, clip, row_scale, temperature, Bq, Bv, Nq, Nv, D, dq, dv, dv_f32, dT, ws, pmo, flags, st);
    }
    return wide ? bwd_typed<float, uint16_t>(q, v, idx, g, clip, row_scale, temperature, Bq, Bv, Nq, Nv, D, dq, dv, dv_f32, dT, ws, pmo, flags, st)
                : bwd_typed<float, uint8_t>(q, v, idx, g, clip, row_scale, temperature, Bq, Bv, Nq, Nv, D, dq, dv, dv_f32, dT, ws, pmo, flags, st);
}
