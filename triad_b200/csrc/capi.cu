// extern "C" entry points of libtriad_b200.so (see include/triad_b200.h).
#include "common.cuh"

#include <string.h>

#include <atomic>

namespace triad {

static thread_local char g_last_error[256] = "";

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int cuda_fail(cudaError_t e, const char* where) {
    snprintf(g_last_error, sizeof g_last_error, "%s: %s", where, cudaGetErrorString(e));
    return TRIAD_ERR_CUDA;
}
int fail_msg(int status, const char* msg) {
    snprintf(g_last_error, sizeof g_last_error, "%s", msg);
    return status;
}

int device_sms(int* sms) {
    int dev = 0;
    *sms = 148;
    TRIAD_CUDA_CHECK(cudaGetDevice(&dev));
    TRIAD_CUDA_CHECK(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
    return TRIAD_OK;
}

// forward workspace: control block (kCtrlBlockBytes), then the partial sums
static size_t fwd_part_bytes(int M, int Bv, int Nq) {
    PartLayout pl = part_layout(M, Nq);
    return align_up((size_t)Bv * pl.G * pl.S * sizeof(float), 256);
}

}  // namespace triad

using namespace triad;

extern "C" int triad_abi_version(void) { return 1; }

extern "C" const char* triad_status_string(int s) {
    switch (s) {
        case TRIAD_OK: return "ok";
        case TRIAD_ERR_BAD_ARG: return "bad argument";
        case TRIAD_ERR_BAD_SHAPE: return "bad shape";
        case TRIAD_ERR_ALIGNMENT: return "pointer not 16-byte aligned";
        case TRIAD_ERR_WORKSPACE: return "workspace too small";
        case TRIAD_ERR_CUDA: return "CUDA error";
        case TRIAD_ERR_ARCH: return "device is not sm_100";
        case TRIAD_ERR_UNSUPPORTED: return "unsupported shape";
        case TRIAD_ERR_TIMEOUT: return "kernel watchdog timeout";
        default: return "unknown status";
    }
}

extern "C" const char* triad_last_error(void) { return g_last_error; }

extern "C" long long triad_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

extern "C" int triad_device_check(int device) {
    int major = 0;
    TRIAD_CUDA_CHECK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) return fail_msg(TRIAD_ERR_ARCH, "triad_b200 kernels are built for sm_100a only");
    return TRIAD_OK;
}

extern "C" int triad_row_scale(const int64_t* mask, int Bq, int Nq, float* row_scale, void* stream) {
    if (!row_scale) return fail_msg(TRIAD_ERR_BAD_ARG, "row_scale: null output");
    if (Bq <= 0 || Nq <= 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "row_scale: bad shape");
    return launch_row_scale(mask, Bq, Nq, row_scale, (cudaStream_t)stream);
}

// packed forward (TRIAD_FWD_PACK_ROWS): control block | partial sums (packed layout) | packing maps | packed q
static size_t fwd_part_bytes_packed(int Bq, int Bv, int Nq) {
    return align_up((size_t)Bv * Bq * packed_pieces(Nq) * sizeof(float), 256);
}

extern "C" size_t triad_maxmean_fwd_workspace_bytes_ex(int Bq, int Bv, int Nq, int Nv, int D, int dtype, int flags) {
    (void)Nv;
    if (Bq <= 0 || Bv <= 0 || Nq <= 0) return 0;
    size_t n = kCtrlBlockBytes + fwd_part_bytes(Bq * Nq, Bv, Nq);
    if ((flags & TRIAD_FWD_PACK_ROWS) && dtype == TRIAD_DTYPE_BF16 && D > 0) {
        const size_t packed = kCtrlBlockBytes + fwd_part_bytes_packed(Bq, Bv, Nq) + pack_map_bytes(Bq, Nq) +
                              align_up((size_t)Bq * Nq * D * 2, 256);
        if (packed > n) n = packed;
    }
    return n;
}

extern "C" size_t triad_maxmean_fwd_workspace_bytes(int Bq, int Bv, int Nq, int Nv, int D, int dtype) {
    return triad_maxmean_fwd_workspace_bytes_ex(Bq, Bv, Nq, Nv, D, dtype, 0);
}

// cta_group of the unpacked tcgen05 forwards.  A single row tile of <= 128 tokens (one text query against a gallery):
// cta_group::1 — a pair would spend a 256-row MMA on <= 128 rows, and at one tile per image that MMA time equals the
// HBM time of the image, leaving no slack to overlap; alone, each SM streams its own images at twice that rate.
int triad::fwd_cta_group(int M, int flags) { return ((flags & TRIAD_FWD_FORCE_1CTA) || M <= 128) ? 1 : 2; }

static int fwd_impl(const void* q, const void* v, const float* row_scale, const float* temperature, int inv_T,
                    int Bq, int Bv, int Nq, int Nv, int D, int dtype, float* clip, void* idx,
                    void* ws, size_t ws_bytes, int flags, cudaStream_t st) {
    if (!q || !v || !row_scale || !temperature || !clip || !ws) return fail_msg(TRIAD_ERR_BAD_ARG, "maxmean_fwd: null pointer");
    if (dtype != TRIAD_DTYPE_F32 && dtype != TRIAD_DTYPE_BF16) return fail_msg(TRIAD_ERR_BAD_ARG, "maxmean_fwd: dtype");
    if (Bq <= 0 || Bv <= 0 || Nq <= 0 || Nv <= 0 || D <= 0 || D % 8 != 0 || Nv > 65535)
        return fail_msg(TRIAD_ERR_BAD_SHAPE, "maxmean_fwd: bad shape (need D % 8 == 0, Nv <= 65535)");
    if ((long long)Bq * Nq > 0x7fffffffLL) return fail_msg(TRIAD_ERR_BAD_SHAPE, "maxmean_fwd: Bq*Nq overflows int32");
    if (((uintptr_t)q | (uintptr_t)v | (uintptr_t)ws) & 15) return fail_msg(TRIAD_ERR_ALIGNMENT, "maxmean_fwd: q, v and ws must be 16-byte aligned");
    if (ws_bytes < triad_maxmean_fwd_workspace_bytes_ex(Bq, Bv, Nq, Nv, D, dtype, flags)) return fail_msg(TRIAD_ERR_WORKSPACE, "maxmean_fwd: workspace too small");

    const int M = Bq * Nq;
    int* abort_flag = (int*)ws;
    float* part = (float*)((char*)ws + kCtrlBlockBytes);
    TRIAD_CUDA_CHECK(cudaMemsetAsync(abort_flag, 0, kCtrlBlockBytes, st));

    const bool use_tc = dtype == TRIAD_DTYPE_BF16 && !(flags & TRIAD_FWD_FORCE_SIMT) && tc_supported(Nv, D);
    int rc;
    if (use_tc && (flags & TRIAD_FWD_PACK_ROWS)) {
        // masked text queries: drop the zero-weight rows before the tensor cores (pack.cu)
        char* maps = (char*)ws + kCtrlBlockBytes + fwd_part_bytes_packed(Bq, Bv, Nq);
        void* qp = maps + pack_map_bytes(Bq, Nq);
        rc = launch_pack_map(row_scale, Bq, Nq, maps, st);
        if (rc) return rc;
        rc = launch_pack_copy(q, maps, Bq, Nq, D, 2, qp, st);
        if (rc) return rc;
        if (idx) TRIAD_CUDA_CHECK(cudaMemsetAsync(idx, 0, (size_t)Bv * Bq * nq_padded(Nq) * (Nv > 256 ? 2 : 1), st));
        const int cta_group = (flags & TRIAD_FWD_FORCE_1CTA) ? 1 : 2;
        rc = launch_maxmean_tc(qp, v, row_scale, temperature, inv_T, M, Bv, Nq, Nv, D, part, idx, abort_flag, cta_group, flags,
                               (const int*)maps, nullptr, nullptr, st);
        if (rc) return rc;
        if (flags & TRIAD_FWD_TEST_TRIP_WATCHDOG) TRIAD_CUDA_CHECK(cudaMemsetAsync(abort_flag, 1, 4, st));
        return launch_finalize_clip_packed(part, (const int*)maps, Bq, Bv, Nq, clip, abort_flag, st);
    }
    if (use_tc) {
        rc = launch_maxmean_tc(q, v, row_scale, temperature, inv_T, M, Bv, Nq, Nv, D, part, idx, abort_flag,
                               fwd_cta_group(M, flags), flags, nullptr, nullptr, nullptr, st);
    } else {
        rc = launch_maxmean_simt(q, v, row_scale, temperature, inv_T, M, Bv, Nq, Nv, D, dtype, part, idx, st);
    }
    if (rc) return rc;
    if (flags & TRIAD_FWD_TEST_TRIP_WATCHDOG) TRIAD_CUDA_CHECK(cudaMemsetAsync(abort_flag, 1, 4, st));
    return launch_finalize_clip(part, Bq, Bv, Nq, clip, abort_flag, st);
}

extern "C" int triad_maxmean_fwd(const void* q, const void* v, const float* row_scale, const float* temperature,
                                 int Bq, int Bv, int Nq, int Nv, int D, int dtype,
                                 float* clip, void* idx, void* ws, size_t ws_bytes, int flags, void* stream) {
    return fwd_impl(q, v, row_scale, temperature, (flags & TRIAD_FWD_DIVIDE_BY_T) ? 1 : 0, Bq, Bv, Nq, Nv, D, dtype, clip, idx,
                    ws, ws_bytes, flags, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// max-mean forward + dense non-negative-pressure regulariser from ONE pass over the similarities (bf16, tcgen05)
// workspace: control block | max-mean partial sums | regulariser partials
// ---------------------------------------------------------------------------------------------
extern "C" size_t triad_maxmean_fwd_nonneg_workspace_bytes(int Bq, int Bv, int Nq, int Nv, int D) {
    (void)Nv; (void)D;
    if (Bq <= 0 || Bv <= 0 || Nq <= 0) return 0;
    return kCtrlBlockBytes + fwd_part_bytes(Bq * Nq, Bv, Nq) + (size_t)kNonnegFusedPartials * 2 * sizeof(double);
}

extern "C" int triad_maxmean_fwd_nonneg(const void* q, const void* v, const float* row_scale, const float* temperature,
                                        int Bq, int Bv, int Nq, int Nv, int D, float* clip, void* idx,
                                        float lo, float coef, void* n_out, long long ldn, double* sums,
                                        void* ws, size_t ws_bytes, int flags, void* stream) {
    if (!q || !v || !row_scale || !temperature || !clip || !idx || !n_out || !sums || !ws)
        return fail_msg(TRIAD_ERR_BAD_ARG, "maxmean_fwd_nonneg: null pointer");
    if (Bq <= 0 || Bv <= 0 || Nq <= 0 || Nv <= 0 || D <= 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "maxmean_fwd_nonneg: bad shape");
    if ((long long)Bq * Nq > 0x7fffffffLL) return fail_msg(TRIAD_ERR_BAD_SHAPE, "maxmean_fwd_nonneg: Bq*Nq overflows int32");
    if (!tc_emit_supported(Nv, D))
        return fail_msg(TRIAD_ERR_UNSUPPORTED, "maxmean_fwd_nonneg: needs D % 64 == 0, D <= 512, Nv <= 256, Nv % 8 == 0");
    if (!(lo < 0.f)) return fail_msg(TRIAD_ERR_BAD_ARG, "maxmean_fwd_nonneg: lo must be negative");
    if (ldn < (long long)Bv * Nv || ldn % 8 != 0 || (long long)ldn * 2 >= (1ll << 40)) return fail_msg(TRIAD_ERR_BAD_SHAPE, "maxmean_fwd_nonneg: ldn");
    if (((uintptr_t)q | (uintptr_t)v | (uintptr_t)n_out | (uintptr_t)ws) & 15) return fail_msg(TRIAD_ERR_ALIGNMENT, "maxmean_fwd_nonneg: 16-byte alignment");
    if (ws_bytes < triad_maxmean_fwd_nonneg_workspace_bytes(Bq, Bv, Nq, Nv, D)) return fail_msg(TRIAD_ERR_WORKSPACE, "maxmean_fwd_nonneg: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const int M = Bq * Nq;
    int* abort_flag = (int*)ws;
    float* part = (float*)((char*)ws + kCtrlBlockBytes);
    double* npart = (double*)((char*)ws + kCtrlBlockBytes + fwd_part_bytes(M, Bv, Nq));
    TRIAD_CUDA_CHECK(cudaMemsetAsync(abort_flag, 0, kCtrlBlockBytes, st));
    EmitNArgs e{n_out, ldn, lo, coef, 1, npart, sums, 1};
    const int cta_group = (flags & TRIAD_FWD_FORCE_1CTA) ? 1 : 2;
    const int rc = launch_maxmean_tc(q, v, row_scale, temperature, 0, M, Bv, Nq, Nv, D, part, idx, abort_flag, cta_group,
                                     flags, nullptr, &e, nullptr, st);
    if (rc) return rc;
    if (flags & TRIAD_FWD_TEST_TRIP_WATCHDOG) TRIAD_CUDA_CHECK(cudaMemsetAsync(abort_flag, 1, 4, st));
    return launch_finalize_clip(part, Bq, Bv, Nq, clip, abort_flag, st);
}

// Synchronises `stream` and reports whether the forward kernel that last used `ws` hit its
// deadlock watchdog (debug / test aid; the hot path never calls it).
extern "C" int triad_maxmean_fwd_status(const void* ws, void* stream) {
    if (!ws) return fail_msg(TRIAD_ERR_BAD_ARG, "fwd_status: null workspace");
    int flag = 0;
    TRIAD_CUDA_CHECK(cudaMemcpyAsync(&flag, ws, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    TRIAD_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    if (flag != 0) {
        char buf[96];
        snprintf(buf, sizeof buf, "forward kernel watchdog fired at wait site %d", flag);
        return fail_msg(TRIAD_ERR_TIMEOUT, buf);
    }
    return TRIAD_OK;
}

// ---------------------------------------------------------------------------------------------
// retrieval scores: one query against a gallery (both directions are the same max-mean kernel;
// direction 1 swaps the operands: rows = gallery patches, "image" = the query's tokens)
// ---------------------------------------------------------------------------------------------
extern "C" size_t triad_retrieve_workspace_bytes(int Nq, int n_img, int Nv, int D, int dtype) {
    if (Nq <= 0 || n_img <= 0 || Nv <= 0) return 0;
    const size_t scale_rows = (size_t)(Nq > (long long)n_img * Nv ? Nq : (size_t)n_img * Nv);
    const size_t a = triad_maxmean_fwd_workspace_bytes(1, n_img, Nq, Nv, D, dtype);
    const size_t b = triad_maxmean_fwd_workspace_bytes(n_img, 1, Nv, Nq, D, dtype);
    return align_up(scale_rows * 4, 256) + (a > b ? a : b);
}

extern "C" int triad_retrieve_scores(const void* q, int Nq, const void* gallery, int n_img, int Nv, int D,
                                     int dtype, const float* temperature, int divide_by_T, int direction,
                                     float* scores, void* ws, size_t ws_bytes, void* stream) {
    if (!q || !gallery || !temperature || !scores || !ws) return fail_msg(TRIAD_ERR_BAD_ARG, "retrieve_scores: null pointer");
    if (Nq <= 0 || n_img <= 0 || Nv <= 0 || D <= 0) return fail_msg(TRIAD_ERR_BAD_SHAPE, "retrieve_scores: bad shape");
    if (direction != 0 && direction != 1) return fail_msg(TRIAD_ERR_BAD_ARG, "retrieve_scores: direction");
    if (ws_bytes < triad_retrieve_workspace_bytes(Nq, n_img, Nv, D, dtype)) return fail_msg(TRIAD_ERR_WORKSPACE, "retrieve_scores: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t scale_rows = (size_t)(Nq > (long long)n_img * Nv ? Nq : (size_t)n_img * Nv);
    float* rs = (float*)ws;
    void* fws = (char*)ws + align_up(scale_rows * 4, 256);
    const size_t fws_bytes = ws_bytes - align_up(scale_rows * 4, 256);
    if (direction == 0) {
        int rc = launch_row_scale(nullptr, 1, Nq, rs, st);
        if (rc) return rc;
        return fwd_impl(q, gallery, rs, temperature, divide_by_T, 1, n_img, Nq, Nv, D, dtype, scores, nullptr, fws, fws_bytes, 0, st);
    }
    int rc = launch_row_scale(nullptr, n_img, Nv, rs, st);
    if (rc) return rc;
    return fwd_impl(gallery, q, rs, temperature, divide_by_T, n_img, 1, Nv, Nq, D, dtype, scores, nullptr, fws, fws_bytes, 0, st);
}

// ---------------------------------------------------------------------------------------------
// retrieval scores on an e4m3 gallery (direction 0, divides by T)
// workspace: row weights [Nq] | control block | partial sums
// ---------------------------------------------------------------------------------------------
extern "C" size_t triad_retrieve_e4m3_workspace_bytes(int Nq, int n_img, int Nv, int D) {
    (void)Nv; (void)D;
    if (Nq <= 0 || n_img <= 0) return 0;
    return align_up((size_t)Nq * 4, 256) + kCtrlBlockBytes + fwd_part_bytes(Nq, n_img, Nq);
}

extern "C" int triad_retrieve_scores_e4m3(const void* q_codes, const float* q_scales, int Nq, const void* g_codes,
                                          const float* g_scales, int n_img, int Nv, int D, const float* temperature,
                                          float* scores, void* ws, size_t ws_bytes, void* stream) {
    if (!q_codes || !q_scales || !g_codes || !g_scales || !temperature || !scores || !ws)
        return fail_msg(TRIAD_ERR_BAD_ARG, "retrieve_scores_e4m3: null pointer");
    if (Nq <= 0 || n_img <= 0 || Nv <= 0 || D <= 0 || Nv > 65535)
        return fail_msg(TRIAD_ERR_BAD_SHAPE, "retrieve_scores_e4m3: bad shape (need Nq, n_img >= 1, 1 <= Nv <= 65535)");
    if (!tc_e4m3_supported(Nv, D)) return fail_msg(TRIAD_ERR_UNSUPPORTED, "retrieve_scores_e4m3: needs D % 128 == 0, D <= 512");
    if ((((uintptr_t)q_codes | (uintptr_t)g_codes | (uintptr_t)ws) & 15) ||
        (((uintptr_t)q_scales | (uintptr_t)g_scales | (uintptr_t)scores) & 3))
        return fail_msg(TRIAD_ERR_ALIGNMENT, "retrieve_scores_e4m3: codes and ws 16-byte aligned, scales and scores 4-byte aligned");
    if (ws_bytes < triad_retrieve_e4m3_workspace_bytes(Nq, n_img, Nv, D))
        return fail_msg(TRIAD_ERR_WORKSPACE, "retrieve_scores_e4m3: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    float* rs = (float*)ws;
    char* fws = (char*)ws + align_up((size_t)Nq * 4, 256);
    int* abort_flag = (int*)fws;
    float* part = (float*)(fws + kCtrlBlockBytes);
    TRIAD_CUDA_CHECK(cudaMemsetAsync(abort_flag, 0, kCtrlBlockBytes, st));
    int rc = launch_row_scale(nullptr, 1, Nq, rs, st);
    if (rc) return rc;
    const E4m3Args e4m3{q_scales, g_scales};
    rc = launch_maxmean_tc(q_codes, g_codes, rs, temperature, 1, Nq, n_img, Nq, Nv, D, part, nullptr, abort_flag,
                           fwd_cta_group(Nq, 0), 0, nullptr, nullptr, &e4m3, st);
    if (rc) return rc;
    return launch_finalize_clip(part, 1, n_img, Nq, scores, abort_flag, st);
}
