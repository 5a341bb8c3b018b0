// The two backward GEMMs of the dense "non-negative pressure" regulariser (SURVEY.md §8 f1), hand-written for
// sm_100a: with N = dL/d<q,v> ([M = Bq*Nq rows][Kc = Bv*Nv columns], bf16, row-major — what the tcgen05 forward's
// epilogue emits, maxmean_tc.cu kMode 1 / 2),
//
//     mode 0   dQ[M , D] = N   . V2        V2 = the patches, [Kc][D]      (autograd of src/model.py:384-387 w.r.t. the
//     mode 1   dV[Kc, D] = N^T . Q2        Q2 = the tokens,  [M ][D]       query / patch embeddings, dense dS)
//
// Neither needs a transposed copy of anything: tcgen05.mma reads MN-major operands (instruction-descriptor bits 15 /
// 16), so B = V2 / Q2 is taken as stored (D contiguous), A = N as stored for mode 0 (K-major) and, for mode 1, the
// SAME row-major N read as an MN-major operand (its columns are the M dimension of that product).
//
// One CTA pair (cta_group::2) owns a 256-row x D output tile: fp32 accumulators = 128 lanes x 512 TMEM columns per
// CTA, two N = 256 halves per K step.  Operands stream through a 4-stage TMA ring (48 KB per stage and CTA: A 16 KB,
// B 2 x 16 KB; the pair shares every B tile, each CTA loads half of its rows).  MN-major tiles are loaded as
// 64-element x 64-row SWIZZLE_128B boxes (k = the box row): exactly the canonical MN-major layout
// ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units, LBO = 8 KB between 64-element groups, SBO = 1 KB between 8-row
// k groups; a K = 16 step advances the start address by 2 KB.
//
// Work = (row tile, K split); the K range is split so that the number of items is close to a multiple of the cluster
// count (cfg 2: 250 row tiles x 2 = 500 items on 74 pairs).  Every item writes an fp32 partial tile (TMA bulk-tensor
// stores of swizzled 32 x 32 boxes, as the forward's N emission); a second launch adds the splits in order and rounds
// to bf16 once — deterministic, no atomics.  Out-of-range rows / columns / K are zero-filled by the loads and clipped
// by the stores (the tensor maps carry the true extents).  triad_dense_grad_gemm_f32 differs in that second launch
// only: it writes the fp32 sum, or adds it to the caller's fp32 output (an accumulator carried across image chunks, or
// one chunk's rows of a per-rank dV partial).
//
// The projection head's backward (proj_head.cu) runs its three products on the same kernel through
// launch_head_gemm: outputs wider than 512 columns are cut into 512-column slices (work item = row tile x slice x
// K split), and the K splits are planned for few output tiles over a long K (the weight gradients: 1-4 tiles, K = the
// token count).  A call with D <= 512 is one slice, so the public entry points run exactly as before.
#include "common.cuh"
#include "ptx.cuh"

#include <cuda.h>

namespace triad {
namespace dgemm {
using namespace ptx;

constexpr int kBlockK = 64;
constexpr int kUmmaK = 16;
constexpr int kTileM = 256;                 // per pair
constexpr int kCtaM = 128;
constexpr int kHalfN = 256;
constexpr int kThreads = 256;
constexpr int kStages = 4;
constexpr uint32_t kBoxBytes = 64 * 128;                        // one 64 x 64 bf16 box
constexpr uint32_t kABytes = 2 * kBoxBytes;                     // 16 KB: 128 rows x 64 k (either major)
constexpr uint32_t kBHalfBytes = 2 * kBoxBytes;                 // 16 KB: this CTA's 128 of a half's 256 columns x 64 k
constexpr uint32_t kStageBytes = kABytes + 2 * kBHalfBytes;     // 48 KB
constexpr uint32_t kStgPerWarp = 32 * 128;                      // 32 rows x 32 fp32
constexpr uint32_t kSmemBytes = kStages * kStageBytes + 4 * 2 * kStgPerWarp + 1024 + 1024;   // 226 KB

struct Params {
    int n_tiles;          // 256-row tiles of the output
    int splits;           // K splits
    int kb_per_split;     // k-blocks per split (the last one may be shorter)
    int nkb;              // k-blocks in all
    int n_halves;         // 1 when D <= 256
    int D;                // output columns in all
    int n_slices;         // 512-column output slices (1 when D <= 512)
    int* abort_flag;
};

// MN-major, SWIZZLE_128B: 64-element groups LBO apart, 8-row k groups SBO apart
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(kBoxBytes >> 4) << 16;                 // LBO
    d |= (uint64_t)(1024 >> 4) << 32;                      // SBO
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

template <bool kAMN, int kHalves>
__global__ void __launch_bounds__(kThreads, 1)
dgemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
             const __grid_constant__ CUtensorMap tmap_c, const Params p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t stg0 = base + kStages * kStageBytes;
    const uint32_t bar = stg0 + 4 * 2 * kStgPerWarp;
    const uint32_t bar_full = bar, bar_empty = bar + 8 * kStages;
    const uint32_t bar_t_full = bar_empty + 8 * kStages, bar_t_empty = bar_t_full + 8;
    const uint32_t tmem_slot = bar_t_empty + 8;
    uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(gen + (tmem_slot - base));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t cta_rank = cluster_ctarank();
    const bool is_leader = cta_rank == 0;
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    const int n_items = p.n_tiles * p.n_slices * p.splits;
    constexpr uint32_t b_bytes = (uint32_t)kHalves * kBHalfBytes;

    if (warp == 0 && lane == 0) { prefetch_tmap(&tmap_a); prefetch_tmap(&tmap_b); prefetch_tmap(&tmap_c); }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        mbar_init(bar_t_full, 1);
        mbar_init(bar_t_empty, 4 * 2);
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc<2>(tmem_slot, 512);
    tc_fence_before();
    cluster_arrive(); cluster_wait();
    tc_fence_after();
    const uint32_t tmem0 = *tmem_slot_gen;

    if (warp == 0) {
        // =============================== TMA producer (both CTAs) =========================
        const bool issuer = elect_one();
        const uint32_t full_sig = mapa(bar_full, 0);                  // every load signals the LEADER's barrier
        int s = 0; uint32_t ph = 0; bool ok = true;
        for (int it = cluster_id; it < n_items && ok; it += n_clusters) {
            const int unit = it / p.splits, sp = it - unit * p.splits;
            const int tile = unit / p.n_slices, col0 = (unit - tile * p.n_slices) * (2 * kHalfN);
            const int kb0 = sp * p.kb_per_split, kb1 = min(p.nkb, kb0 + p.kb_per_split);
            const int m0 = tile * kTileM + (int)cta_rank * kCtaM;
            for (int kb = kb0; kb < kb1; ++kb) {
                ok = mbar_wait(bar_empty + 8 * s, ph ^ 1, p.abort_flag, 31);
                if (!ok) break;
                if (issuer) {
                    const uint32_t st = base + s * kStageBytes;
                    if (is_leader) mbar_expect_tx(bar_full + 8 * s, 2u * (kABytes + b_bytes));
                    if constexpr (!kAMN) {
                        tma_load_2d<2>(st, &tmap_a, full_sig + 8 * s, kb * kBlockK, m0);                     // box {64 k, 128 rows}
                    } else {
                        tma_load_2d<2>(st, &tmap_a, full_sig + 8 * s, m0, kb * kBlockK);                     // boxes {64 m, 64 k}
                        tma_load_2d<2>(st + kBoxBytes, &tmap_a, full_sig + 8 * s, m0 + 64, kb * kBlockK);
                    }
#pragma unroll
                    for (int h = 0; h < kHalves; ++h) {
                        const int n0 = col0 + h * kHalfN + (int)cta_rank * (kHalfN / 2);
                        const uint32_t bs = st + kABytes + h * kBHalfBytes;
                        tma_load_2d<2>(bs, &tmap_b, full_sig + 8 * s, n0, kb * kBlockK);
                        tma_load_2d<2>(bs + kBoxBytes, &tmap_b, full_sig + 8 * s, n0 + 64, kb * kBlockK);
                    }
                }
                __syncwarp();
                if (++s == kStages) { s = 0; ph ^= 1; }
            }
        }
    } else if (warp == 1) {
        // =============================== MMA issuer (leader CTA) ==========================
        if (is_leader) {
            const bool issuer = elect_one();
            const uint32_t idesc = make_idesc(kTileM, kHalfN) | (kAMN ? (1u << 15) : 0u) | (1u << 16);
            const uint32_t tm = __shfl_sync(0xffffffffu, tmem0, 0);
            // descriptors of stage 0; a stage / a K = 16 step / an N half are added to the start-address field (>> 4), so
            // everything stays in uniform registers and the eight MMAs of a k-block issue back to back
            const uint64_t a_desc0 = kAMN ? make_desc_mn(base) : make_smem_desc(base);
            const uint64_t b_desc0 = make_desc_mn(base + kABytes);
            int s = 0; uint32_t ph = 0, tph = 0; bool ok = true;
            for (int it = cluster_id; it < n_items && ok; it += n_clusters) {
                const int tile = it / p.splits, sp = it - tile * p.splits;
                const int kb0 = sp * p.kb_per_split, kb1 = min(p.nkb, kb0 + p.kb_per_split);
                ok = mbar_wait(bar_t_empty, tph ^ 1, p.abort_flag, 32);         // the epilogue has drained the accumulators
                if (!ok) break;
                tc_fence_after();
                for (int kb = kb0; kb < kb1; ++kb) {
                    ok = mbar_wait(bar_full + 8 * s, ph, p.abort_flag, 33);
                    if (!ok) break;
                    tc_fence_after();
                    const uint64_t a_desc = a_desc0 + (uint64_t)((uint32_t)s * (kStageBytes >> 4));
                    const uint64_t b_desc = b_desc0 + (uint64_t)((uint32_t)s * (kStageBytes >> 4));
                    if (issuer) {
#pragma unroll
                        for (int k = 0; k < kBlockK / kUmmaK; ++k) {
#pragma unroll
                            for (int h = 0; h < kHalves; ++h)
                                umma_bf16<2>(tm + h * kHalfN, a_desc + (uint64_t)(kAMN ? 128u * k : 2u * k),       // 2 KB / 32 B per K = 16 step
                                             b_desc + (uint64_t)(h * (kBHalfBytes >> 4) + 128u * k), idesc, (uint32_t)((kb != kb0) | (k != 0)));
                        }
                        umma_commit<2>(bar_empty + 8 * s);
                    }
                    __syncwarp();
                    if (++s == kStages) { s = 0; ph ^= 1; }
                }
                if (!ok) break;
                if (issuer) umma_commit<2>(bar_t_full);
                __syncwarp();
                tph ^= 1;
            }
        }
    } else if (warp >= 4) {
        // =============================== epilogue (both CTAs): fp32 partial tile out ======
        const int quarter = warp & 3;
        const uint32_t t_empty_sig = mapa(bar_t_empty, 0);
        const uint32_t stg_w = stg0 + (uint32_t)quarter * 2u * kStgPerWarp;      // two boxes: one leaves while the other fills
        const uint32_t taddr = tmem0 + ((uint32_t)(quarter * 32) << 16);
        uint32_t tph = 0, nbox = 0; bool ok = true;
        for (int it = cluster_id; it < n_items && ok; it += n_clusters) {
            const int unit = it / p.splits, sp = it - unit * p.splits;
            const int tile = unit / p.n_slices, col0 = (unit - tile * p.n_slices) * (2 * kHalfN);
            const int width = min(2 * kHalfN, p.D - col0);
            const int row0 = tile * kTileM + (int)cta_rank * kCtaM + quarter * 32;
            ok = mbar_wait(bar_t_full, tph, p.abort_flag, 34);
            ok = __all_sync(0xffffffffu, ok);
            if (!ok) break;
            tc_fence_after();
            for (int c = 0; c * 32 < width; ++c, ++nbox) {
                const uint32_t stg = stg_w + (nbox & 1u) * kStgPerWarp;
                const uint32_t stg_row = stg + (uint32_t)lane * 128u;
                uint32_t buf[32];
                tmem_ld32_raw(taddr + c * 32, buf);
                tmem_wait_ld();
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");     // the box before last has been read
                __syncwarp();
#pragma unroll
                for (int g = 0; g < 8; ++g)
                    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(stg_row + ((uint32_t)(g ^ (lane & 7)) << 4)),
                                 "r"(buf[4 * g]), "r"(buf[4 * g + 1]), "r"(buf[4 * g + 2]), "r"(buf[4 * g + 3]) : "memory");
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                                 ::"l"(reinterpret_cast<uint64_t>(&tmap_c)), "r"(stg), "r"(col0 + c * 32), "r"(row0), "r"(sp) : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(t_empty_sig);
            tph ^= 1;
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncwarp();
    }
    __syncwarp();
    tc_fence_before();
    cluster_arrive(); cluster_wait();
    if (warp == 2) tmem_dealloc<2>(tmem0, 512);
}

// What the split reduction writes: bf16(sum), the fp32 sum, or out + sum in fp32 (the splits are added in order
// first, then to out once, so accumulating onto zeros gives the bits of kOutF32)
enum { kOutBf16 = 0, kOutF32 = 1, kOutF32Add = 2 };

// out[r][d] = sum over splits, in order, of part[s][r][d]; NaN everywhere if the GEMM's watchdog fired
template <int kOut>
__global__ void __launch_bounds__(256)
reduce_kernel(const float4* __restrict__ part, size_t n4, int splits, void* __restrict__ out, const int* __restrict__ abort_flag) {
    const bool poisoned = *abort_flag != 0;
    for (size_t k = (size_t)blockIdx.x * 256 + threadIdx.x; k < n4; k += (size_t)gridDim.x * 256) {
        float4 a = part[k];
        for (int s = 1; s < splits; ++s) {
            const float4 b = part[(size_t)s * n4 + k];
            a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
        }
        if constexpr (kOut == kOutF32Add) {
            const float4 o = reinterpret_cast<const float4*>(out)[k];
            a.x = o.x + a.x; a.y = o.y + a.y; a.z = o.z + a.z; a.w = o.w + a.w;
        }
        if (poisoned) a.x = a.y = a.z = a.w = __int_as_float(0x7fc00000);
        if constexpr (kOut == kOutBf16) {
            __nv_bfloat162 lo = __floats2bfloat162_rn(a.x, a.y), hi = __floats2bfloat162_rn(a.z, a.w);
            reinterpret_cast<uint2*>(out)[k] = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
        } else {
            reinterpret_cast<float4*>(out)[k] = a;
        }
    }
}

static int pick_splits(int n_tiles, int nkb, int n_clusters) {
    int best = 1; double best_eff = 0.0;
    const int cand[] = {1, 2, 3, 4, 6, 8, 12, 16};
    for (int s : cand) {
        if (s > nkb) break;
        const long long items = (long long)n_tiles * s;
        const long long rounds = (items + n_clusters - 1) / n_clusters;
        // every extra split costs one more fp32 pass over the output in the reduction
        const double eff = (double)items / (double)(rounds * n_clusters) - 0.01 * (s - 1);
        if (eff > best_eff + 1e-9) { best_eff = eff; best = s; }
    }
    return best;
}

}  // namespace dgemm
}  // namespace triad

using namespace triad;

// CTA pairs the split plans are made for (the workspace sizes depend on the plan, so a failed query plans for a B200)
static int plan_clusters() {
    int sms;
    device_sms(&sms);
    return max(1, sms / 2);
}

static int plan_splits(int M, int Kc, int mode, int* n_tiles, int* nkb, int* kb_per_split) {
    const int rows_out = mode == 0 ? M : Kc, K = mode == 0 ? Kc : M;
    *n_tiles = ceil_div(rows_out, dgemm::kTileM);
    *nkb = ceil_div(K, dgemm::kBlockK);
    int splits = dgemm::pick_splits(*n_tiles, *nkb, plan_clusters());
    *kb_per_split = ceil_div(*nkb, splits);
    return ceil_div(*nkb, *kb_per_split);             // no empty split
}

// The head backward's plan: with fewer (row tile, column slice) units than CTA pairs (the weight gradients: K = the
// token count, 1-4 units) the K range is cut so that every pair gets one item; otherwise the shared heuristic.
static int plan_head_splits(int M, int Kc, int D, int mode, int* n_tiles, int* n_slices, int* nkb, int* kb_per_split) {
    const int clusters = plan_clusters();
    const int rows_out = mode == 0 ? M : Kc, K = mode == 0 ? Kc : M;
    *n_tiles = ceil_div(rows_out, dgemm::kTileM);
    *n_slices = ceil_div(D, 2 * dgemm::kHalfN);
    *nkb = ceil_div(K, dgemm::kBlockK);
    const int units = *n_tiles * *n_slices;
    int splits = units >= clusters ? dgemm::pick_splits(units, *nkb, clusters) : clusters / units;
    splits = max(1, min(splits, *nkb));
    *kb_per_split = ceil_div(*nkb, splits);
    return ceil_div(*nkb, *kb_per_split);
}

extern "C" size_t triad_dense_grad_gemm_workspace_bytes(int M, int Kc, int D, int mode) {
    if (M <= 0 || Kc <= 0 || D <= 0) return 0;
    int n_tiles, nkb, kbs;
    const int splits = plan_splits(M, Kc, mode, &n_tiles, &nkb, &kbs);
    return kCtrlBlockBytes + (size_t)splits * (size_t)(mode == 0 ? M : Kc) * (size_t)D * sizeof(float);
}

namespace triad {
size_t head_gemm_workspace_bytes(int M, int Kc, int D, int mode) {
    int n_tiles, n_slices, nkb, kbs;
    const int splits = plan_head_splits(M, Kc, D, mode, &n_tiles, &n_slices, &nkb, &kbs);
    return kCtrlBlockBytes + (size_t)splits * (size_t)(mode == 0 ? M : Kc) * (size_t)D * sizeof(float);
}
}  // namespace triad

// Launches the GEMM and the split reduction for a validated call and a plan in p (n_tiles, n_slices, splits,
// kb_per_split, nkb).
static int dgemm_launch(dgemm::Params p, const void* n_mat, long long ldn, int M, int Kc, const void* x, int D, int mode,
                        void* out, int out_kind, void* ws, size_t ws_bytes, cudaStream_t st) {
    using namespace dgemm;
    int sms = 0;
    int rc = device_sms(&sms);
    if (rc) return rc;
    const int rows_out = mode == 0 ? M : Kc;          // rows of the product
    const int K = mode == 0 ? Kc : M;                 // contraction length
    int n_clusters = sms / 2;
    p.n_halves = D > kHalfN ? 2 : 1;
    p.D = D;
    p.abort_flag = (int*)ws;
    const size_t part_bytes = (size_t)p.splits * rows_out * D * sizeof(float);
    if (ws_bytes < kCtrlBlockBytes + part_bytes) return fail_msg(TRIAD_ERR_WORKSPACE, "dense_grad_gemm: workspace too small");
    float* part = (float*)((char*)ws + kCtrlBlockBytes);
    TRIAD_CUDA_CHECK(cudaMemsetAsync(ws, 0, kCtrlBlockBytes, st));

    CUtensorMap ma, mb, mc;
    if (mode == 0) {       // A = N, K-major: dims {Kc, M}, box {64 k, 128 rows}
        cuuint64_t dims[2] = {(cuuint64_t)Kc, (cuuint64_t)M};
        cuuint64_t strides[1] = {(cuuint64_t)ldn * 2};
        cuuint32_t box[2] = {64, 128};
        rc = encode_tmap(&ma, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, n_mat, 2, dims, strides, box, Swizzle::k128B);
    } else {               // A = N^T read MN-major from the same rows: dims {Kc (the product's rows), M (k)}, box {64, 64}
        cuuint64_t dims[2] = {(cuuint64_t)Kc, (cuuint64_t)M};
        cuuint64_t strides[1] = {(cuuint64_t)ldn * 2};
        cuuint32_t box[2] = {64, 64};
        rc = encode_tmap(&ma, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, n_mat, 2, dims, strides, box, Swizzle::k128B);
    }
    if (rc) return rc;
    {                      // B = V2 / Q2, [K][D], MN-major: dims {D, K}, box {64 n, 64 k}
        cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)K};
        cuuint64_t strides[1] = {(cuuint64_t)D * 2};
        cuuint32_t box[2] = {64, 64};
        rc = encode_tmap(&mb, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, x, 2, dims, strides, box, Swizzle::k128B);
        if (rc) return rc;
    }
    {                      // fp32 partials [splits][rows_out][D]: box {32 cols, 32 rows, 1}
        cuuint64_t dims[3] = {(cuuint64_t)D, (cuuint64_t)rows_out, (cuuint64_t)p.splits};
        cuuint64_t strides[2] = {(cuuint64_t)D * 4, (cuuint64_t)rows_out * D * 4};
        cuuint32_t box[3] = {32, 32, 1};
        rc = encode_tmap(&mc, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, part, 3, dims, strides, box, Swizzle::k128B);
        if (rc) return rc;
    }
    const int n_items = p.n_tiles * p.n_slices * p.splits;
    if (n_clusters > n_items) n_clusters = n_items;
    if (mode == 0) rc = p.n_halves == 2 ? launch_clusters<dgemm_kernel<false, 2>>(2, n_clusters, kThreads, kSmemBytes, st, ma, mb, mc, p)
                                        : launch_clusters<dgemm_kernel<false, 1>>(2, n_clusters, kThreads, kSmemBytes, st, ma, mb, mc, p);
    else           rc = p.n_halves == 2 ? launch_clusters<dgemm_kernel<true, 2>>(2, n_clusters, kThreads, kSmemBytes, st, ma, mb, mc, p)
                                        : launch_clusters<dgemm_kernel<true, 1>>(2, n_clusters, kThreads, kSmemBytes, st, ma, mb, mc, p);
    if (rc) return rc;
    const size_t n4 = (size_t)rows_out * D / 4;
    size_t want = (n4 + 255) / 256;
    const int blocks = (int)(want > (size_t)(148 * 16) ? (size_t)(148 * 16) : (want < 1 ? 1 : want));
    if (out_kind == kOutBf16)     reduce_kernel<kOutBf16><<<blocks, 256, 0, st>>>((const float4*)part, n4, p.splits, out, (const int*)ws);
    else if (out_kind == kOutF32) reduce_kernel<kOutF32><<<blocks, 256, 0, st>>>((const float4*)part, n4, p.splits, out, (const int*)ws);
    else                          reduce_kernel<kOutF32Add><<<blocks, 256, 0, st>>>((const float4*)part, n4, p.splits, out, (const int*)ws);
    TRIAD_LAUNCH_CHECK("dense_grad_gemm reduce_kernel");
    return TRIAD_OK;
}

static int dense_grad_gemm_run(const void* n_mat, long long ldn, int M, int Kc, const void* x, int D, int mode,
                               void* out, int out_kind, void* ws, size_t ws_bytes, void* stream) {
    using namespace dgemm;
    if (!n_mat || !x || !out || !ws) return fail_msg(TRIAD_ERR_BAD_ARG, "dense_grad_gemm: null pointer");
    if (mode != 0 && mode != 1) return fail_msg(TRIAD_ERR_BAD_ARG, "dense_grad_gemm: mode");
    if (M <= 0 || Kc <= 0 || D <= 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "dense_grad_gemm: bad shape");
    if (D % 8 != 0 || D > 512 || ldn % 8 != 0 || ldn < Kc || (long long)ldn * 2 >= (1ll << 40))
        return fail_msg(TRIAD_ERR_UNSUPPORTED, "dense_grad_gemm: needs D % 8 == 0, D <= 512, ldn % 8 == 0");
    if (((uintptr_t)n_mat | (uintptr_t)x | (uintptr_t)out | (uintptr_t)ws) & 15) return fail_msg(TRIAD_ERR_ALIGNMENT, "dense_grad_gemm: 16-byte alignment");
    Params p;
    p.splits = plan_splits(M, Kc, mode, &p.n_tiles, &p.nkb, &p.kb_per_split);
    p.n_slices = 1;
    return dgemm_launch(p, n_mat, ldn, M, Kc, x, D, mode, out, out_kind, ws, ws_bytes, (cudaStream_t)stream);
}

namespace triad {
// The projection head's products (arguments validated by triad_project_tokens_bwd): D % 64 == 0, any width
int launch_head_gemm(const void* n_mat, long long ldn, int M, int Kc, const void* x, int D, int mode, void* out,
                     int out_f32, void* ws, size_t ws_bytes, cudaStream_t st) {
    dgemm::Params p;
    p.splits = plan_head_splits(M, Kc, D, mode, &p.n_tiles, &p.n_slices, &p.nkb, &p.kb_per_split);
    return dgemm_launch(p, n_mat, ldn, M, Kc, x, D, mode, out, out_f32 ? dgemm::kOutF32 : dgemm::kOutBf16, ws, ws_bytes, st);
}
}  // namespace triad

extern "C" int triad_dense_grad_gemm(const void* n_mat, long long ldn, int M, int Kc, const void* x, int D, int mode,
                                     void* out, void* ws, size_t ws_bytes, void* stream) {
    return dense_grad_gemm_run(n_mat, ldn, M, Kc, x, D, mode, out, dgemm::kOutBf16, ws, ws_bytes, stream);
}

extern "C" int triad_dense_grad_gemm_f32(const void* n_mat, long long ldn, int M, int Kc, const void* x, int D, int mode,
                                         float* out, int accumulate, void* ws, size_t ws_bytes, void* stream) {
    if (accumulate != 0 && accumulate != 1) return fail_msg(TRIAD_ERR_BAD_ARG, "dense_grad_gemm_f32: accumulate must be 0 or 1");
    return dense_grad_gemm_run(n_mat, ldn, M, Kc, x, D, mode, out, accumulate ? dgemm::kOutF32Add : dgemm::kOutF32,
                               ws, ws_bytes, stream);
}
