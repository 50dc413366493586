// api_align.cu -- extern "C" entry points for the photometric alignment stages (marshalling only).
#include <algorithm>

#include <cstring>

#include "common.cuh"

using namespace ygzb;

namespace {

template <typename T>
int h2d(ygzb_ctx* ctx, T* dst, const T* src, size_t count) {
    if (!count) return YGZB_OK;
    return check_cuda(ctx, cudaMemcpyAsync(dst, src, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream), "H2D");
}
template <typename T>
int d2h(ygzb_ctx* ctx, T* dst, const T* src, size_t count) {
    if (!count) return YGZB_OK;
    return check_cuda(ctx, cudaMemcpyAsync(dst, src, count * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream), "D2H");
}
#define TRY(x)                       \
    do {                             \
        int _rc = (x);               \
        if (_rc != YGZB_OK) return _rc; \
    } while (0)

int check_slots(ygzb_frames* f, const int32_t* s, int n, const char* what) {
    for (int i = 0; i < n; ++i)
        if (s[i] < 0 || s[i] >= f->capacity) return set_error(f->ctx, YGZB_ERR_INVALID, "%s[%d] = %d out of range", what, i, s[i]);
    return YGZB_OK;
}

}  // namespace

extern "C" {

int ygzb_align2d(ygzb_frames* f, int n, const int32_t* slot, const uint8_t* level, const uint8_t* ref_border, const uint8_t* ref,
                 int n_iter, double* uv, uint8_t* ok) {
    if (!f || n < 0 || (n && (!slot || !level || !ref_border || !uv || !ok))) return YGZB_ERR_INVALID;
    if (n == 0) return YGZB_OK;
    ygzb_ctx* ctx = f->ctx;
    cudaSetDevice(ctx->device);
    TRY(check_slots(f, slot, n, "slot"));
    for (int i = 0; i < n; ++i)
        if (level[i] >= ctx->geo.n_levels) return set_error(ctx, YGZB_ERR_INVALID, "level[%d] out of range", i);
    const size_t N = (size_t)n;
    Carver sz(nullptr);
    sz.take<int32_t>(N); sz.take<uint8_t>(N); sz.take<uint8_t>(N * 100); sz.take<uint8_t>(N * 64); sz.take<double>(2 * N); sz.take<uint8_t>(N);
    void* buf = dev_scratch(ctx, 6, sz.bytes());
    if (!buf) return YGZB_ERR_CUDA;
    Carver c(buf);
    int32_t* d_slot = c.take<int32_t>(N);
    uint8_t* d_level = c.take<uint8_t>(N);
    uint8_t* d_rb = c.take<uint8_t>(N * 100);
    uint8_t* d_ref = c.take<uint8_t>(N * 64);
    double* d_uv = c.take<double>(2 * N);
    uint8_t* d_ok = c.take<uint8_t>(N);
    TRY(h2d(ctx, d_slot, slot, N));
    TRY(h2d(ctx, d_level, level, N));
    TRY(h2d(ctx, d_rb, ref_border, N * 100));
    if (ref) TRY(h2d(ctx, d_ref, ref, N * 64));
    TRY(h2d(ctx, d_uv, uv, 2 * N));
    TRY(launch_align2d(f, n, d_slot, d_level, d_rb, ref ? d_ref : nullptr, n_iter, d_uv, d_ok));
    TRY(d2h(ctx, uv, d_uv, 2 * N));
    TRY(d2h(ctx, ok, d_ok, N));
    YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return YGZB_OK;
}

int ygzb_align1d(ygzb_frames* f, int n, const int32_t* slot, const uint8_t* level, const float* dir, const uint8_t* ref_border,
                 const uint8_t* ref, int n_iter, double* uv, uint8_t* ok, double* h_inv) {
    if (!f || n < 0 || (n && (!slot || !level || !dir || !ref_border || !uv || !ok || !h_inv))) return YGZB_ERR_INVALID;
    if (n == 0) return YGZB_OK;
    ygzb_ctx* ctx = f->ctx;
    cudaSetDevice(ctx->device);
    TRY(check_slots(f, slot, n, "slot"));
    for (int i = 0; i < n; ++i)
        if (level[i] >= ctx->geo.n_levels) return set_error(ctx, YGZB_ERR_INVALID, "level[%d] out of range", i);
    const size_t N = (size_t)n;
    Carver sz(nullptr);
    sz.take<int32_t>(N); sz.take<uint8_t>(N); sz.take<float>(2 * N); sz.take<uint8_t>(N * 100); sz.take<uint8_t>(N * 64); sz.take<double>(2 * N);
    sz.take<uint8_t>(N); sz.take<double>(N);
    void* buf = dev_scratch(ctx, 6, sz.bytes());
    if (!buf) return YGZB_ERR_CUDA;
    Carver c(buf);
    int32_t* d_slot = c.take<int32_t>(N);
    uint8_t* d_level = c.take<uint8_t>(N);
    float* d_dir = c.take<float>(2 * N);
    uint8_t* d_rb = c.take<uint8_t>(N * 100);
    uint8_t* d_ref = c.take<uint8_t>(N * 64);
    double* d_uv = c.take<double>(2 * N);
    uint8_t* d_ok = c.take<uint8_t>(N);
    double* d_h = c.take<double>(N);
    TRY(h2d(ctx, d_slot, slot, N));
    TRY(h2d(ctx, d_level, level, N));
    TRY(h2d(ctx, d_dir, dir, 2 * N));
    TRY(h2d(ctx, d_rb, ref_border, N * 100));
    if (ref) TRY(h2d(ctx, d_ref, ref, N * 64));
    TRY(h2d(ctx, d_uv, uv, 2 * N));
    TRY(launch_align1d(f, n, d_slot, d_level, d_dir, d_rb, ref ? d_ref : nullptr, n_iter, d_uv, d_ok, d_h));
    TRY(d2h(ctx, uv, d_uv, 2 * N));
    TRY(d2h(ctx, ok, d_ok, N));
    TRY(d2h(ctx, h_inv, d_h, N));
    YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return YGZB_OK;
}

int ygzb_project_align(ygzb_frames* f, int n, const int32_t* ref_slot, const int32_t* cur_slot, int n_poses, const double* poses,
                       const int32_t* ref_pose, const int32_t* cur_pose, const double* ref_px, const double* ref_depth,
                       const uint8_t* ref_level, double* cur_px, uint8_t* search_level, uint8_t* ok) {
    if (!f || n < 0 || n_poses < 1 || !poses) return YGZB_ERR_INVALID;
    if (n == 0) return YGZB_OK;
    if (!ref_slot || !cur_slot || !ref_pose || !cur_pose || !ref_px || !ref_depth || !ref_level || !cur_px || !search_level || !ok)
        return YGZB_ERR_INVALID;
    ygzb_ctx* ctx = f->ctx;
    cudaSetDevice(ctx->device);
    TRY(check_slots(f, ref_slot, n, "ref_slot"));
    TRY(check_slots(f, cur_slot, n, "cur_slot"));
    for (int i = 0; i < n; ++i) {
        if (ref_pose[i] < 0 || ref_pose[i] >= n_poses || cur_pose[i] < 0 || cur_pose[i] >= n_poses)
            return set_error(ctx, YGZB_ERR_INVALID, "candidate %d: pose index out of range", i);
        if (ref_level[i] >= ctx->geo.n_levels) return set_error(ctx, YGZB_ERR_INVALID, "ref_level[%d] out of range", i);
    }
    const size_t N = (size_t)n, P = (size_t)n_poses;
    Carver sz(nullptr);
    sz.take<int32_t>(4 * N); sz.take<double>(12 * P); sz.take<double>(2 * N); sz.take<double>(N); sz.take<double>(2 * N);
    sz.take<uint8_t>(N); sz.take<uint8_t>(N); sz.take<uint8_t>(N);
    void* buf = dev_scratch(ctx, 6, sz.bytes());
    if (!buf) return YGZB_ERR_CUDA;
    Carver c(buf);
    int32_t* d_idx = c.take<int32_t>(4 * N);
    double* d_poses = c.take<double>(12 * P);
    double* d_rpx = c.take<double>(2 * N);
    double* d_depth = c.take<double>(N);
    double* d_cpx = c.take<double>(2 * N);
    uint8_t* d_rlevel = c.take<uint8_t>(N);
    uint8_t* d_slevel = c.take<uint8_t>(N);
    uint8_t* d_ok = c.take<uint8_t>(N);
    // the inputs are the first six sub-buffers, contiguous on the device: assemble them in pinned memory with the same
    // layout and move them with ONE copy (nine pageable copies cost more than the kernel itself)
    const size_t in_bytes = (size_t)((uint8_t*)(d_rlevel + N) - (uint8_t*)buf);
    uint8_t* stage = (uint8_t*)host_scratch(ctx, 1, in_bytes);
    if (!stage) return YGZB_ERR_CUDA;
    YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    auto put = [&](const void* dev_ptr, const void* src, size_t bytes) { memcpy(stage + ((const uint8_t*)dev_ptr - (uint8_t*)buf), src, bytes); };
    put(d_idx, ref_slot, N * 4);
    put(d_idx + N, cur_slot, N * 4);
    put(d_idx + 2 * N, ref_pose, N * 4);
    put(d_idx + 3 * N, cur_pose, N * 4);
    put(d_poses, poses, 12 * P * 8);
    put(d_rpx, ref_px, 2 * N * 8);
    put(d_depth, ref_depth, N * 8);
    put(d_cpx, cur_px, 2 * N * 8);
    put(d_rlevel, ref_level, N);
    YGZB_CUDA(ctx, cudaMemcpyAsync(buf, stage, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    TRY(launch_project_align(f, n, d_idx, d_idx + N, d_poses, d_idx + 2 * N, d_idx + 3 * N, d_rpx, d_depth, d_rlevel, d_cpx, d_slevel,
                             d_ok));
    TRY(d2h(ctx, cur_px, d_cpx, 2 * N));
    TRY(d2h(ctx, search_level, d_slevel, N));
    TRY(d2h(ctx, ok, d_ok, N));
    YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return YGZB_OK;
}

int ygzb_sparse_align(ygzb_frames* f, int n_problems, const int32_t* ref_slot, const int32_t* cur_slot, const int32_t* offsets,
                      const double* px, const double* depth, const uint8_t* has_mappoint, const double* T_cw_ref, double* T_cw_cur,
                      int max_level, int min_level, int n_iter, double eps, int32_t* n_meas, int32_t* iters_per_level) {
    if (!f || n_problems < 1 || !ref_slot || !cur_slot || !offsets || !T_cw_ref || !T_cw_cur || !n_meas) return YGZB_ERR_INVALID;
    ygzb_ctx* ctx = f->ctx;
    cudaSetDevice(ctx->device);
    TRY(check_slots(f, ref_slot, n_problems, "ref_slot"));
    TRY(check_slots(f, cur_slot, n_problems, "cur_slot"));
    if (max_level >= ctx->geo.n_levels || min_level < 0 || min_level > max_level)
        return set_error(ctx, YGZB_ERR_INVALID, "levels [%d, %d] outside the %d-level pyramid", min_level, max_level, ctx->geo.n_levels);
    TRY(check_offsets(ctx, offsets, n_problems, "offsets"));
    const size_t P = (size_t)n_problems, T = (size_t)offsets[n_problems];
    if (T && (!px || !depth || !has_mappoint)) return YGZB_ERR_INVALID;
    int max_feat = 0;
    for (int p = 0; p < n_problems; ++p) max_feat = std::max(max_feat, offsets[p + 1] - offsets[p]);
    Carver sz(nullptr);
    sz.take<int32_t>(2 * P); sz.take<int32_t>(P + 1); sz.take<double>(2 * T); sz.take<double>(T); sz.take<uint8_t>(T);
    sz.take<double>(12 * P); sz.take<double>(12 * P); sz.take<int32_t>(P); sz.take<int32_t>(P * kMaxLevels);
    sz.take<uint8_t>(sparse_align_scratch_bytes(T));
    void* buf = dev_scratch(ctx, 6, sz.bytes());
    if (!buf) return YGZB_ERR_CUDA;
    Carver c(buf);
    int32_t* d_slots = c.take<int32_t>(2 * P);
    int32_t* d_off = c.take<int32_t>(P + 1);
    double* d_px = c.take<double>(2 * T);
    double* d_depth = c.take<double>(T);
    uint8_t* d_mp = c.take<uint8_t>(T);
    double* d_Tref = c.take<double>(12 * P);
    double* d_Tcur = c.take<double>(12 * P);
    int32_t* d_nmeas = c.take<int32_t>(P);
    int32_t* d_iters = c.take<int32_t>(P * kMaxLevels);
    void* d_feat = c.take<uint8_t>(sparse_align_scratch_bytes(T));
    {   // the inputs are the first seven sub-buffers of `buf`: one pinned staging copy instead of eight pageable ones
        const size_t in_bytes = (size_t)((uint8_t*)(d_Tcur + 12 * P) - (uint8_t*)buf);
        uint8_t* stage = (uint8_t*)host_scratch(ctx, 1, in_bytes);
        if (!stage) return YGZB_ERR_CUDA;
        YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        auto put = [&](const void* dev_ptr, const void* src, size_t bytes) {
            if (bytes) memcpy(stage + ((const uint8_t*)dev_ptr - (uint8_t*)buf), src, bytes);
        };
        put(d_slots, ref_slot, P * 4);
        put(d_slots + P, cur_slot, P * 4);
        put(d_off, offsets, (P + 1) * 4);
        put(d_px, px, 2 * T * 8);
        put(d_depth, depth, T * 8);
        put(d_mp, has_mappoint, T);
        put(d_Tref, T_cw_ref, 12 * P * 8);
        put(d_Tcur, T_cw_cur, 12 * P * 8);
        YGZB_CUDA(ctx, cudaMemcpyAsync(buf, stage, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    YGZB_CUDA(ctx, cudaMemsetAsync(d_iters, 0, P * kMaxLevels * sizeof(int32_t), ctx->stream));
    TRY(launch_sparse_align(f, n_problems, d_slots, d_slots + P, d_off, max_feat, d_px, d_depth, d_mp, d_Tref, d_Tcur, max_level,
                            min_level, n_iter, eps, d_nmeas, d_iters, d_feat));
    TRY(d2h(ctx, T_cw_cur, d_Tcur, 12 * P));
    TRY(d2h(ctx, n_meas, d_nmeas, P));
    if (iters_per_level) TRY(d2h(ctx, iters_per_level, d_iters, P * kMaxLevels));
    YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return YGZB_OK;
}

}  // extern "C"
