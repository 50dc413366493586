// common.cuh -- shared declarations of libygz_b200.so (context, slot storage, launch helpers).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "../../include/ygz_b200.h"

namespace ygzb {

constexpr int kMaxLevels = YGZB_MAX_LEVELS;

// FAST / cell-selection tile (level pixels).  80 x 40 is a whole number of 10-px grid cells on the
// three levels that can yield features (8x4, 16x8, 32x16 cells).
constexpr int kTileW = 80;
constexpr int kTileH = 40;

struct LevelGeom {
    int w, h, pitch;   // pitch in bytes, multiple of 16
    unsigned off;      // byte offset of the level inside a slot
};

struct Geometry {
    LevelGeom lv[kMaxLevels];
    int n_levels;
    int n_sel_levels;  // levels [0, n_sel_levels) can pass Frame::InFrame(px, 20, L); the others never yield features
    int W, H;          // full resolution (image.width / image.height)
    int cell_size, grid_cols, grid_rows, n_cells;
    int threshold;
    int tile_begin[kMaxLevels + 1];  // prefix sums of tiles per level
    int tiles_x[kMaxLevels];
    // exact division by small runtime constants without the ~20-instruction integer divide: n / d == (n * magic) >> 24
    // with magic = ceil(2^24 / d), valid while n * d < 2^24 (checked by build_geometry)
    unsigned tiles_x_magic[kMaxLevels];
    unsigned cell_magic;
    int cpt_x[kMaxLevels], cpt_y[kMaxLevels];  // grid cells per FAST tile row / column on the selectable levels
};

__host__ __device__ __forceinline__ unsigned div_magic(unsigned n, unsigned magic) {
    return (unsigned)(((unsigned long long)n * magic) >> 24);
}

}  // namespace ygzb

struct ygzb_ctx {
    int device;
    cudaStream_t stream;
    ygzb_params prm;
    ygzb::Geometry geo;
    size_t slot_stride;  // bytes per frame slot (pyramid), multiple of 256
    int sm_count;
    long long launches;
    char err[512];
    // growable device / pinned scratch owned by the context
    void* d_scratch[8];
    size_t d_scratch_bytes[8];
    void* h_scratch[4];
    size_t h_scratch_bytes[4];
    // optional per-stage CUDA-event timing (ygzb_profile_*): events bracket each kernel on ctx->stream
    int prof_on;
    void* prof;  // std::vector<ygzb::ProfRec>*
    cudaEvent_t timer[2];   // ygzb_timer_start / ygzb_timer_stop
    cudaEvent_t block_ev;   // ygzb_synchronize_blocking (created on first use)
};

struct ygzb_frames {
    ygzb_ctx* ctx;
    int capacity;
    uint8_t* d_pyr;       // capacity * slot_stride
    // device feature store, per slot, capacity n_cells features each (cell-index order)
    int32_t* d_count;     // [capacity]
    int16_t* d_fx;        // level coordinates
    int16_t* d_fy;
    uint8_t* d_flevel;
    float* d_fscore;
    float* d_fangle;
    int32_t* d_fcell;
    uint8_t* d_fdesc;     // [capacity][n_cells][32]
    // detect scratch (sized for `capacity` items)
    unsigned long long* d_best_key;   // [capacity][n_sel][n_cells]
    unsigned long long* d_first_key;  // [capacity][n_sel][n_cells]
    int32_t* d_stats;                 // [capacity][n_levels][2]
    int32_t* d_slots;                 // [capacity] slot list of the current call
    uint8_t* d_occupied;              // [capacity][n_cells]
    // TMA descriptors (CUtensorMap, 128 B each) of the first pyramid levels: 3-D tensors (x, y, slot) of u8 with a
    // 112 x 50 x 1 box = one FAST tile + halo; tma_levels == 0 disables the TMA path
    alignas(64) unsigned char tile_maps[3][128];
    void* d_tile_maps;                // device copy of tile_maps
    int tma_levels;
    int32_t* d_offsets;               // [capacity+1]
    int last_n;
};

namespace ygzb {

int set_error(ygzb_ctx* ctx, int code, const char* fmt, ...);
int check_cuda(ygzb_ctx* ctx, cudaError_t e, const char* what);
// offsets arrays of the batched entry points: off[0] == 0, non-decreasing, int-range total (returns YGZB_ERR_INVALID before
// anything is allocated or indexed)
inline int check_offsets(ygzb_ctx* ctx, const int32_t* off, int n, const char* what) {
    if (!off || n < 0) return set_error(ctx, YGZB_ERR_INVALID, "%s: null offsets", what);
    if (off[0] != 0) return set_error(ctx, YGZB_ERR_INVALID, "%s[0] must be 0", what);
    for (int i = 0; i < n; ++i)
        if (off[i + 1] < off[i]) return set_error(ctx, YGZB_ERR_INVALID, "%s must be non-decreasing (entry %d)", what, i + 1);
    return YGZB_OK;
}
// grow-only scratch buffers
void* dev_scratch(ygzb_ctx* ctx, int which, size_t bytes);
void* host_scratch(ygzb_ctx* ctx, int which, size_t bytes);

#define YGZB_CUDA(ctx, call)                                               \
    do {                                                                   \
        int _rc = ygzb::check_cuda((ctx), (call), #call);                  \
        if (_rc != YGZB_OK) return _rc;                                    \
    } while (0)

#define YGZB_LAUNCHED(ctx)                                                 \
    do {                                                                   \
        (ctx)->launches++;                                                 \
        int _rc = ygzb::check_cuda((ctx), cudaGetLastError(), "kernel launch"); \
        if (_rc != YGZB_OK) return _rc;                                    \
    } while (0)

// ---- per-stage device timing -------------------------------------------------------------------
enum Stage {
    kStageBgr2Gray = 0, kStagePyrDown, kStageFastCells, kStageMergeCells, kStageDescribe, kStageMatch,
    kStageMatchFinalize, kStagePack, kStageOther, kStageAlign2D, kStageProjectAlign, kStageSparseAlign, kStagePoseOnly,
    kStageLocalBA, kStageKLT, kNumStages
};
struct ProfRec {
    cudaEvent_t a, b;
    int stage;
};
void prof_begin(ygzb_ctx* ctx, int stage);
void prof_end(ygzb_ctx* ctx);
struct ProfScope {
    ygzb_ctx* c;
    ProfScope(ygzb_ctx* ctx, int stage) : c(ctx) { if (c->prof_on) prof_begin(c, stage); }
    ~ProfScope() { if (c->prof_on) prof_end(c); }
};

// ---- stage launchers (one .cu each) -----------------------------------------------------------
int launch_pyramid(ygzb_frames* f, int first, int count, const uint8_t* d_bgr /* or null */);
int launch_pyrdown_ptrs(ygzb_ctx* ctx, const uint8_t* const* d_src_ptr, uint8_t* const* d_dst_ptr, int sw, int sh, int spitch,
                        int dw, int dh, int dpitch, int count);
int launch_detect(ygzb_frames* f, int n, bool have_occupied);
int build_tile_maps(ygzb_frames* f);
int launch_describe_store(ygzb_frames* f, int n);
int launch_describe_list(ygzb_frames* f, int n, const int32_t* d_slot_of, int total, const double* d_x, const double* d_y,
                         const uint8_t* d_level, float* d_angle, uint8_t* d_desc);
int launch_fast_debug(ygzb_frames* f, int slot, int level, uint8_t* d_score_map, uint8_t* d_nonmax_map);
int launch_offsets(ygzb_ctx* ctx, const int32_t* d_counts, const int32_t* d_sets, int n, int32_t* d_offsets);
int launch_match(ygzb_ctx* ctx, const uint8_t* d_base, size_t set_stride, const int32_t* d_counts, const int32_t* d_a_sets,
                 const int32_t* d_b_sets, int n_pairs, int cap, int cross_check, unsigned* d_fwd_key, unsigned* d_col_key,
                 const int32_t* d_q_offsets, int32_t* d_train_idx, int32_t* d_dist);
int launch_hamming_pairs(ygzb_ctx* ctx, const uint8_t* d_A, const uint8_t* d_B, const int32_t* d_ia, const int32_t* d_ib,
                         int n, int32_t* d_dist);
int launch_align2d(ygzb_frames* f, int n, const int32_t* d_slot, const uint8_t* d_level, const uint8_t* d_ref_border,
                   const uint8_t* d_ref, int n_iter, double* d_uv, uint8_t* d_ok);
int launch_align1d(ygzb_frames* f, int n, const int32_t* d_slot, const uint8_t* d_level, const float* d_dir, const uint8_t* d_ref_border,
                   const uint8_t* d_ref, int n_iter, double* d_uv, uint8_t* d_ok, double* d_hinv);
int launch_project_align(ygzb_frames* f, int n, const int32_t* d_ref_slot, const int32_t* d_cur_slot, const double* d_poses,
                         const int32_t* d_ref_pose, const int32_t* d_cur_pose, const double* d_ref_px, const double* d_ref_depth,
                         const uint8_t* d_ref_level, double* d_cur_px, uint8_t* d_search_level, uint8_t* d_ok);
// max_feat: the largest feature count of a problem; d_feat_scratch: sparse_align_scratch_bytes(d_offsets[n_problems])
int launch_sparse_align(ygzb_frames* f, int n_problems, const int32_t* d_ref_slot, const int32_t* d_cur_slot,
                        const int32_t* d_offsets, int max_feat, const double* d_px, const double* d_depth, const uint8_t* d_has_mp,
                        const double* d_T_ref, double* d_T_cur, int max_level, int min_level, int n_iter, double eps,
                        int32_t* d_n_meas, int32_t* d_iters, void* d_feat_scratch);
size_t sparse_align_scratch_bytes(size_t n_features);

// bump allocator over one scratch buffer (all sub-buffers 256-byte aligned)
struct Carver {
    uint8_t* base;
    size_t off = 0;
    explicit Carver(void* p) : base(static_cast<uint8_t*>(p)) {}
    template <typename T>
    T* take(size_t count) {
        off = (off + 255) & ~(size_t)255;
        T* r = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off += count * sizeof(T);
        return r;
    }
    size_t bytes() const { return off + 256; }
};

// device helpers shared by kernels ---------------------------------------------------------------
__device__ __forceinline__ unsigned float_orderable(float f) {
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float orderable_float(unsigned o) {
    unsigned u = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
    return __uint_as_float(u);
}

}  // namespace ygzb
