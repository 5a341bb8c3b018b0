// Ragged caption gallery: captions of different lengths stored whole in 256-row slots, and the retrieval scores of
// one query against it in both aggregation directions (the tcgen05 forward's kMode 3 / 4, maxmean_tc.cu).
//
// Layout (planned on the host from the lengths, triad_ragged_plan): captions are placed greedily in order; a caption
// that does not fit in the rest of the current slot starts a new one, so no caption straddles a slot, and a slot's
// rows after its last caption are zero.  The zero-padded alternative [n, 77, D] reads 77 rows per caption and
// scores the padding; at cfg 3's lengths (U[8, 77]) about 90 % of the slot rows are caption rows.
//
// The slots are bf16 (triad_ragged_pack) or e4m3 codes with one fp32 scale per slot row (triad_ragged_pack_e4m3, the
// per-row quantizer of quant_e4m3.cu gathering through the same row map); both storages share the plan, the workspace
// and the finalize.
#include "common.cuh"

#include <string.h>

namespace triad {

// dst[r] = bf16(src[rowmap[r]]), or a zero row where rowmap[r] is negative or not below src_rows; 8 elements per
// thread and step
__global__ void __launch_bounds__(256)
ragged_pack_kernel(const void* __restrict__ src, int dtype, long long src_rows, int D, const int* __restrict__ rowmap,
                   long long dst_rows, __nv_bfloat16* __restrict__ dst) {
    const int per_row = D / 8;
    const long long total = dst_rows * per_row;
    for (long long t = (long long)blockIdx.x * 256 + threadIdx.x; t < total; t += (long long)gridDim.x * 256) {
        const long long r = t / per_row;
        const int c = (int)(t - r * per_row);
        const int s = rowmap[r];
        uint4 out = make_uint4(0u, 0u, 0u, 0u);
        if (s >= 0 && s < src_rows) {
            if (dtype == TRIAD_DTYPE_BF16) {
                out = __ldg(reinterpret_cast<const uint4*>(src) + (size_t)s * per_row + c);
            } else {
                const float4* f = reinterpret_cast<const float4*>(src) + ((size_t)s * per_row + c) * 2;
                const float4 a = __ldg(f), b = __ldg(f + 1);
                __nv_bfloat162 h[4] = {__floats2bfloat162_rn(a.x, a.y), __floats2bfloat162_rn(a.z, a.w),
                                       __floats2bfloat162_rn(b.x, b.y), __floats2bfloat162_rn(b.z, b.w)};
                memcpy(&out, h, sizeof out);
            }
        }
        reinterpret_cast<uint4*>(dst)[(size_t)r * per_row + c] = out;
    }
}

// scores[c] = the caption's partials summed in ascending order: direction 0 its G query-row-group partials
// part[c][g] (cap_info == NULL), direction 1 its rows' weighted maxima part[first row + t], t < length.  Neither order
// depends on where the caption sits in the gallery.  A tripped watchdog turns every score into NaN, as the dense
// finalize does.
__global__ void __launch_bounds__(256)
ragged_finalize_kernel(const float* __restrict__ part, int n_cap, int G, const int2* __restrict__ cap_info,
                       float* __restrict__ scores, const int* __restrict__ abort_flag) {
    const int c = blockIdx.x * 256 + threadIdx.x;
    if (c >= n_cap) return;
    float acc = 0.f;
    if (cap_info == nullptr) {
        for (int g = 0; g < G; ++g) acc += part[(size_t)c * G + g];
    } else {
        const int2 ci = cap_info[c];
        for (int t = 0; t < ci.y; ++t) acc += part[(size_t)ci.x + t];
    }
    if (*abort_flag != 0) acc = __int_as_float(0x7fc00000);
    scores[c] = acc;
}

// workspace: row weights [Nq] (direction 0) | control block | partials: direction 0 [n_cap][ceil(Nq/32)],
// direction 1 [n_slots * 256]
static size_t ragged_part_bytes(int Nq, int n_slots, int n_cap, int direction) {
    const size_t n = direction == 0 ? (size_t)n_cap * ceil_div(Nq, 32) : (size_t)n_slots * kSlotRows;
    return align_up(n * sizeof(float), 256);
}

}  // namespace triad

using namespace triad;

extern "C" int triad_ragged_plan(const int32_t* lengths, int n_cap, int32_t* slot_meta, int32_t* cap_info, int* n_slots) {
    if (!lengths || !slot_meta || !cap_info || !n_slots) return fail_msg(TRIAD_ERR_BAD_ARG, "ragged_plan: null pointer");
    if (n_cap <= 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "ragged_plan: need at least one caption");
    for (int c = 0; c < n_cap; ++c)
        if (lengths[c] < 1 || lengths[c] > kSlotRows) return fail_msg(TRIAD_ERR_BAD_SHAPE, "ragged_plan: caption lengths must be 1..256");
    int slot = -1, used = kSlotRows;
    for (int c = 0; c < n_cap; ++c) {
        const int len = lengths[c];
        if (used + len > kSlotRows) {                        // does not fit: a new slot
            ++slot;
            used = 0;
            int32_t* m = slot_meta + (size_t)slot * kSlotMetaInts;
            memset(m, 0, kSlotMetaInts * sizeof(int32_t));
            m[kSlotMetaCap0] = c;
        }
        int32_t* m = slot_meta + (size_t)slot * kSlotMetaInts;
        const int last = used + len - 1;
        m[kSlotMetaCount] += 1;
        m[kSlotMetaStarts + (used >> 5)] |= (int32_t)(1u << (used & 31));
        m[kSlotMetaEnds + (last >> 5)] |= (int32_t)(1u << (last & 31));
        cap_info[2 * (size_t)c] = slot * kSlotRows + used;
        cap_info[2 * (size_t)c + 1] = len;
        used += len;
        m[kSlotMetaUsed] = used;
        if ((long long)(slot + 1) * kSlotRows > 0x7fffffffLL) return fail_msg(TRIAD_ERR_BAD_SHAPE, "ragged_plan: too many slots");
    }
    *n_slots = slot + 1;
    return TRIAD_OK;
}

extern "C" int triad_ragged_pack(const void* src, int dtype, long long src_rows, int D, const int32_t* rowmap,
                                 long long dst_rows, void* dst, void* stream) {
    if (!src || !rowmap || !dst) return fail_msg(TRIAD_ERR_BAD_ARG, "ragged_pack: null pointer");
    if (dtype != TRIAD_DTYPE_F32 && dtype != TRIAD_DTYPE_BF16) return fail_msg(TRIAD_ERR_BAD_ARG, "ragged_pack: dtype");
    if (src_rows <= 0 || dst_rows <= 0 || dst_rows % kSlotRows != 0 || D <= 0 || D % 8 != 0)
        return fail_msg(TRIAD_ERR_BAD_SHAPE, "ragged_pack: bad shape (need D % 8 == 0, dst_rows a multiple of 256)");
    if (src_rows > 0x7fffffffLL || dst_rows > 0x7fffffffLL) return fail_msg(TRIAD_ERR_BAD_SHAPE, "ragged_pack: more than 2^31 rows");
    if (((uintptr_t)src | (uintptr_t)dst) & 15) return fail_msg(TRIAD_ERR_ALIGNMENT, "ragged_pack: src and dst 16-byte aligned");
    if ((uintptr_t)rowmap & 3) return fail_msg(TRIAD_ERR_ALIGNMENT, "ragged_pack: rowmap 4-byte aligned");
    const long long chunks = dst_rows * (D / 8);
    const long long blocks = (chunks + 255) / 256;
    ragged_pack_kernel<<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, (cudaStream_t)stream>>>(
        src, dtype, src_rows, D, rowmap, dst_rows, (__nv_bfloat16*)dst);
    TRIAD_LAUNCH_CHECK("ragged_pack_kernel");
    return TRIAD_OK;
}

extern "C" int triad_ragged_pack_e4m3(const void* src, int dtype, long long src_rows, int D, const int32_t* rowmap,
                                      long long dst_rows, void* codes, float* scales, void* stream) {
    if (!src || !rowmap || !codes || !scales) return fail_msg(TRIAD_ERR_BAD_ARG, "ragged_pack_e4m3: null pointer");
    if (dtype != TRIAD_DTYPE_F32 && dtype != TRIAD_DTYPE_BF16) return fail_msg(TRIAD_ERR_BAD_ARG, "ragged_pack_e4m3: dtype");
    if (src_rows <= 0 || dst_rows <= 0 || dst_rows % kSlotRows != 0)
        return fail_msg(TRIAD_ERR_BAD_SHAPE, "ragged_pack_e4m3: bad shape (need dst_rows a multiple of 256)");
    if (src_rows > 0x7fffffffLL || dst_rows > 0x7fffffffLL) return fail_msg(TRIAD_ERR_BAD_SHAPE, "ragged_pack_e4m3: more than 2^31 rows");
    if (!tc_e4m3_supported(kSlotRows, D)) return fail_msg(TRIAD_ERR_UNSUPPORTED, "ragged_pack_e4m3: needs D in {128, 256, 384, 512}");
    if (((uintptr_t)src | (uintptr_t)codes) & 15) return fail_msg(TRIAD_ERR_ALIGNMENT, "ragged_pack_e4m3: src and codes 16-byte aligned");
    if (((uintptr_t)rowmap | (uintptr_t)scales) & 3) return fail_msg(TRIAD_ERR_ALIGNMENT, "ragged_pack_e4m3: rowmap and scales 4-byte aligned");
    return launch_quantize_e4m3(src, dtype, dst_rows, D, codes, scales, (cudaStream_t)stream, rowmap, src_rows);
}

extern "C" size_t triad_retrieve_ragged_workspace_bytes(int Nq, int n_slots, int n_cap, int direction) {
    if (Nq <= 0 || n_slots <= 0 || n_cap <= 0 || (direction != 0 && direction != 1)) return 0;
    return align_up((size_t)Nq * 4, 256) + kCtrlBlockBytes + ragged_part_bytes(Nq, n_slots, n_cap, direction);
}

// the scores of the ragged forward (both storages): the workspace split, the kernel and the finalize; the arguments
// have been checked.  q_scales == NULL: q and slots are bf16; otherwise both hold e4m3 codes, scaled per row by
// q_scales and slot_scales.
static int retrieve_ragged(const void* q, const float* q_scales, int Nq, const void* slots, const float* slot_scales,
                           const int32_t* slot_meta, const int32_t* cap_info, int n_slots, int n_cap, int D,
                           const float* temperature, int direction, float* scores, void* ws, cudaStream_t st) {
    float* rs = (float*)ws;
    char* fws = (char*)ws + align_up((size_t)Nq * 4, 256);
    int* abort_flag = (int*)fws;
    float* part = (float*)(fws + kCtrlBlockBytes);
    TRIAD_CUDA_CHECK(cudaMemsetAsync(abort_flag, 0, kCtrlBlockBytes, st));
    const RaggedArgs ragged{slot_meta, cap_info, direction};
    int rc;
    if (direction == 0) {
        // rows = the query's tokens (weight 1/Nq), images = the slots
        const E4m3Args e4m3{q_scales, slot_scales};
        rc = launch_row_scale(nullptr, 1, Nq, rs, st);
        if (rc) return rc;
        rc = launch_maxmean_tc(q, slots, rs, temperature, 1, Nq, n_slots, Nq, kSlotRows, D, part, nullptr, abort_flag,
                               fwd_cta_group(Nq, 0), 0, nullptr, nullptr, q_scales ? &e4m3 : nullptr, st, &ragged);
    } else {
        // rows = the slot rows (weight 1/length of their caption), the one image = the query
        const E4m3Args e4m3{slot_scales, q_scales};
        rc = launch_maxmean_tc(slots, q, nullptr, temperature, 1, n_slots * kSlotRows, 1, kSlotRows, Nq, D, part, nullptr,
                               abort_flag, 2, 0, nullptr, nullptr, q_scales ? &e4m3 : nullptr, st, &ragged);
    }
    if (rc) return rc;
    ragged_finalize_kernel<<<ceil_div(n_cap, 256), 256, 0, st>>>(part, n_cap, ceil_div(Nq, 32),
                                                                 direction == 0 ? nullptr : (const int2*)cap_info, scores,
                                                                 abort_flag);
    TRIAD_LAUNCH_CHECK("ragged_finalize_kernel");
    return TRIAD_OK;
}

static bool ragged_shape_ok(int Nq, int n_slots, int n_cap, int D) {
    return !(Nq <= 0 || Nq > 65535 || n_slots <= 0 || n_cap < n_slots || (long long)n_cap > (long long)n_slots * kSlotRows ||
             (long long)n_slots * kSlotRows > 0x7fffffffLL || D <= 0);
}

extern "C" int triad_retrieve_scores_ragged(const void* q, int Nq, const void* slots, const int32_t* slot_meta,
                                            const int32_t* cap_info, int n_slots, int n_cap, int D,
                                            const float* temperature, int direction, float* scores,
                                            void* ws, size_t ws_bytes, void* stream) {
    if (!q || !slots || !slot_meta || !cap_info || !temperature || !scores || !ws)
        return fail_msg(TRIAD_ERR_BAD_ARG, "retrieve_scores_ragged: null pointer");
    if (direction != 0 && direction != 1) return fail_msg(TRIAD_ERR_BAD_ARG, "retrieve_scores_ragged: direction must be 0 or 1");
    if (!ragged_shape_ok(Nq, n_slots, n_cap, D))
        return fail_msg(TRIAD_ERR_BAD_SHAPE, "retrieve_scores_ragged: bad shape (need 1 <= Nq <= 65535, n_slots <= n_cap <= 256 n_slots)");
    if (!tc_supported(kSlotRows, D)) return fail_msg(TRIAD_ERR_UNSUPPORTED, "retrieve_scores_ragged: needs D in {64,...,512} (multiple of 64)");
    if ((((uintptr_t)q | (uintptr_t)slots | (uintptr_t)ws) & 15) || (((uintptr_t)slot_meta | (uintptr_t)cap_info) & 7) ||
        ((uintptr_t)scores & 3))
        return fail_msg(TRIAD_ERR_ALIGNMENT, "retrieve_scores_ragged: q, slots and ws 16-byte, metadata 8-byte, scores 4-byte aligned");
    if (ws_bytes < triad_retrieve_ragged_workspace_bytes(Nq, n_slots, n_cap, direction))
        return fail_msg(TRIAD_ERR_WORKSPACE, "retrieve_scores_ragged: workspace too small");
    return retrieve_ragged(q, nullptr, Nq, slots, nullptr, slot_meta, cap_info, n_slots, n_cap, D, temperature, direction,
                           scores, ws, (cudaStream_t)stream);
}

extern "C" int triad_retrieve_scores_ragged_e4m3(const void* q_codes, const float* q_scales, int Nq, const void* codes,
                                                 const float* scales, const int32_t* slot_meta, const int32_t* cap_info,
                                                 int n_slots, int n_cap, int D, const float* temperature, int direction,
                                                 float* scores, void* ws, size_t ws_bytes, void* stream) {
    if (!q_codes || !q_scales || !codes || !scales || !slot_meta || !cap_info || !temperature || !scores || !ws)
        return fail_msg(TRIAD_ERR_BAD_ARG, "retrieve_scores_ragged_e4m3: null pointer");
    if (direction != 0 && direction != 1)
        return fail_msg(TRIAD_ERR_BAD_ARG, "retrieve_scores_ragged_e4m3: direction must be 0 or 1");
    if (!ragged_shape_ok(Nq, n_slots, n_cap, D))
        return fail_msg(TRIAD_ERR_BAD_SHAPE, "retrieve_scores_ragged_e4m3: bad shape (need 1 <= Nq <= 65535, n_slots <= n_cap <= 256 n_slots)");
    if (!tc_e4m3_supported(kSlotRows, D))
        return fail_msg(TRIAD_ERR_UNSUPPORTED, "retrieve_scores_ragged_e4m3: needs D in {128, 256, 384, 512}");
    if ((((uintptr_t)q_codes | (uintptr_t)codes | (uintptr_t)ws) & 15) || (((uintptr_t)slot_meta | (uintptr_t)cap_info) & 7) ||
        (((uintptr_t)q_scales | (uintptr_t)scales | (uintptr_t)scores) & 3))
        return fail_msg(TRIAD_ERR_ALIGNMENT, "retrieve_scores_ragged_e4m3: codes and ws 16-byte, metadata 8-byte, scales and "
                                             "scores 4-byte aligned");
    if (ws_bytes < triad_retrieve_ragged_workspace_bytes(Nq, n_slots, n_cap, direction))
        return fail_msg(TRIAD_ERR_WORKSPACE, "retrieve_scores_ragged_e4m3: workspace too small");
    return retrieve_ragged(q_codes, q_scales, Nq, codes, scales, slot_meta, cap_info, n_slots, n_cap, D, temperature,
                           direction, scores, ws, (cudaStream_t)stream);
}
