// track.cuh -- device-resident local map (key-frame ring per stream) and the per-batch work arrays of the fused
// tracking chain; shared by align.cu (sparse alignment / direct projection kernels), ba.cu (pose-only) and track.cu
// (the ygzb_tracker_* entry points, key-frame insertion, local-BA problem assembly).
#pragma once

#include <stdint.h>

#include "../../include/ygz_b200.h"

struct ygzb_frames;

namespace ygzb {

constexpr int kTrackMaxLocal = 4;   // ring entries per stream = local key-frames + 1 (a new key-frame is written before the oldest leaves)

struct TrackStore {
    int S, R, cells, W, H;
    double fx, fy, cx, cy;      // caller-side intrinsics in double (config/default.yaml camera.*): candidate projection, map points
    // ring entry e = stream * R + entry
    double* kf_T;               // [S*R][12]   T_cw
    int32_t* kf_n;              // [S*R]       features = map points created by the key-frame
    int32_t* kf_slot;           // [S*R]       frame slot that keeps its pyramid
    long long* kf_mp0;          // [S*R]       ids of its map points are [mp0, mp0 + n)
    double* kf_px;              // [S*R][cells][2]  full-resolution pixel (Feature::_pixel)
    uint8_t* kf_level;          // [S*R][cells]
    double* kf_depth;           // [S*R][cells]
    double* kf_pw;              // [S*R][cells][3]  MapPoint::_pos_world
    int32_t* kf_nobs;           // [S*R]       older map points tracked into the key-frame ...
    long long* kf_obs_id;       // [S*R][kTrackMaxLocal*cells]
    double* kf_obs_px;          // [S*R][kTrackMaxLocal*cells][2]
    const double* depth_map;    // [S][W*H]    depth image of the frame that becomes a key-frame (stand-in for the TUM depth)
};

struct TrackBatch {
    int J;                      // jobs of the batch
    int cap;                    // candidate capacity per job = kTrackMaxLocal * cells
    const ygzb_track_job* jobs; // device copy
    // sparse alignment (SparseImgAlign::run): problem j owns scratch features [offsets[j], offsets[j] + n_feat[j])
    int32_t *ref_slot, *cur_slot, *offsets, *in_off, *n_feat, *n_meas;
    double *T_ref, *T_cur;      // [J][12]; T_cur: reference pose in, aligned pose, then pose-only result
    void* feat_scratch;         // [J * cells] features: global fall-back of the kernel's per-feature staging
    // Matcher::SparseImageAlignment's motion check, poses relative to the local key-frames
    int32_t* aligned;           // [J]
    double* rel;                // [J][kTrackMaxLocal][12]
    // FindCandidates + FindDirectProjection, dense over (local key-frame, feature)
    uint8_t* cand_ok;           // [J][cap]
    double* cand_px;            // [J][cap][2]
    int32_t* n_cand;            // [J]
    // successfully projected points, compacted in candidate order
    int32_t *c_cnt, *c_off;     // [J], [J+1]
    int32_t* c_src;             // [J][cap]  dense candidate index (local key-frame * cells + feature)
    double *c_pw, *c_px, *c_depth;
    uint8_t *inlier, *enable;
    int32_t* n_inl;
    double* pose_ws;
    ygzb_track_result* results; // [J]
};

// align.cu
int launch_track_chain_front(ygzb_frames* f, const TrackStore& st, const TrackBatch& b, int sparse_cluster);
int launch_track_chain_mid(ygzb_frames* f, const TrackStore& st, const TrackBatch& b);
// ba.cu
int launch_pose_only_dev(ygzb_ctx* ctx, int n_problems, const int32_t* d_offsets, const int32_t* d_counts, const double* d_pw,
                         const double* d_px, double* d_T_cw, uint8_t* d_inlier, double* d_depth, int32_t* d_n_inlier, uint8_t* d_enable,
                         double* d_ws, int cluster, int max_points);
size_t pose_only_ws_doubles(int n_problems);

}  // namespace ygzb
