// track.cu -- device-resident local map and the fused tracking entry points (ygzb_tracker_*).
//
// Replaces the CALLER-SIDE data flow of the reference's per-frame path, so that nothing but one small record per frame
// crosses PCIe:
//   VisualOdometry::TrackRefFrame / LocalMapping::TrackLocalMap     src/Module/VisualOdometry.cpp:281-302,
//                                                                   src/Module/LocalMapping.cpp:24-140
//   VisualOdometry::SetKeyframe (Detect, map points, LocalBA)       src/Module/VisualOdometry.cpp:182-218,
//                                                                   src/Module/LocalMapping.cpp:149-172
// The numeric stages are the kernels of align.cu (sparse alignment, direct projection), ba.cu (pose-only), fast.cu /
// describe.cu (Detect) and ba2.cu (LocalBAG2O); this file owns the key-frame ring, the key-frame insertion kernel, the
// assembly of the local-BA problems (landmark-major, straight from the ring) and the write-back of the BA result.
// Compiled with -fmad=false: the map-point creation and candidate bookkeeping follow the host loops
// (host/vo_driver.cpp, ygz_slam_b200/vo.py) operation by operation.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <new>

#include "ba2.cuh"
#include "common.cuh"
#include "se3.cuh"
#include "track.cuh"

using namespace ygzb;

struct ygzb_tracker {
    ygzb_frames* f;
    ygzb_ctx* ctx;
    TrackStore st;
    TrackBatch b;          // arrays sized for max_jobs
    int max_jobs;
    void* d_store;         // one allocation behind st.*
    void* d_batch;         // one allocation behind b.*
    double* d_depth;       // [S][W*H]
    // staging (page-locked) + device copies of the job arrays
    ygzb_track_job* h_jobs;
    ygzb_keyframe_job* h_kfjobs;
    ygzb_keyframe_job* d_kfjobs;
    ygzb_keyframe_result* d_kfres;
    cudaEvent_t staged;    // the last H2D copy out of the staging buffers
    int last_J;
    // local BA problems of a key-frame batch (device-built, capacity based)
    void* d_ba;            // problem arrays + scratch of ba2
    size_t ba_bytes;
    int pcap, ocap;        // points / observations capacity per problem
    cudaStream_t front;    // second stream: uploads + pyramid + sparse alignment of the next batch run here, concurrently with a
                           // local BA on the context's stream (they need the new key-frame's features, not its refined pose)
    cudaEvent_t e_fill;    // recorded on the main stream after the key-frame insertion kernel (features + ring entry written)
    cudaEvent_t e_front;   // recorded on the front stream after the sparse alignment
    cudaEvent_t e_up;      // recorded on the front stream after every upload: a key-frame insertion (Detect) waits for it
    cudaEvent_t e_main;    // recorded on the main stream after a tracking chain: the front stream must not overwrite its arrays earlier
    int cluster;           // CTAs per tracking problem (sparse alignment, pose-only): fixed, so that a frame's result does not
                           // depend on how many other frames share its batch (the summation order follows the cluster size)
};

namespace {

template <typename T>
int dalloc(ygzb_ctx* ctx, T** p, size_t count) {
    return check_cuda(ctx, cudaMalloc((void**)p, std::max(count, (size_t)1) * sizeof(T)), "cudaMalloc");
}

__device__ __forceinline__ void mat34_inv(const double* A, double* C) {
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) C[4 * r + c] = A[4 * c + r];
        C[4 * r + 3] = -(A[r] * A[3] + A[4 + r] * A[7] + A[8 + r] * A[11]);
    }
}

__global__ void track_finish_kernel(TrackBatch b) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= b.J) return;
    ygzb_track_result r;
    for (int c = 0; c < 12; ++c) r.T_cw[c] = b.T_cur[12 * (size_t)j + c];
    r.n_meas = b.n_meas[j];
    r.aligned = b.aligned[j];
    r.n_candidates = b.n_cand[j];
    r.n_projected = b.c_cnt[j];
    r.n_inliers = b.aligned[j] ? b.n_inl[j] : 0;
    r.pad[0] = r.pad[1] = r.pad[2] = 0;
    b.results[j] = r;
}

// inclusive scan of one int per thread over a 1024-thread CTA: shuffles inside the warps, the 32 warp totals scanned by warp 0
// (two barriers instead of the twenty of a shared-memory Hillis-Steele scan); s_w = 33 ints; returns the CTA total in *total
__device__ __forceinline__ int block_scan_1024(int v, int* s_w, int* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xFFFFFFFFu, v, o);
        if (lane >= o) v += u;
    }
    if (lane == 31) s_w[warp] = v;
    __syncthreads();
    if (warp == 0) {
        int w = s_w[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xFFFFFFFFu, w, o);
            if (lane >= o) w += u;
        }
        s_w[lane] = w;
        if (lane == 31) s_w[32] = w;
    }
    __syncthreads();
    const int out = v + (warp ? s_w[warp - 1] : 0);
    *total = s_w[32];
    __syncthreads();   // s_w may be rewritten by the next call
    return out;
}

// SetKeyframe for job blockIdx.x: the features Detect left in the frame slot's store become the key-frame's features and
// map points (depth image -> camera point -> world, VisualOdometry.cpp:182-218 with the depth initialisation of
// test/test_feature_alignment.cpp:72-85), the inlier observations of its tracking job become its observations of older points
__global__ void __launch_bounds__(1024) kf_fill_kernel(TrackStore st, TrackBatch b, const ygzb_keyframe_job* __restrict__ jobs,
                                                      const int32_t* __restrict__ f_count, const int16_t* __restrict__ f_x,
                                                      const int16_t* __restrict__ f_y, const uint8_t* __restrict__ f_level, int n_cells,
                                                      ygzb_keyframe_result* __restrict__ res) {
    __shared__ int s_scan[1024];
    __shared__ int s_carry;
    __shared__ double s_T[12], s_Tin[12];
    const ygzb_keyframe_job kj = jobs[blockIdx.x];
    const int tid = threadIdx.x, e = kj.stream * st.R + kj.entry;
    const int n = min(f_count[kj.frame_slot], st.cells);
    if (tid < 12) s_T[tid] = kj.track_job >= 0 ? b.T_cur[12 * (size_t)kj.track_job + tid] : ((tid == 0 || tid == 5 || tid == 10) ? 1.0 : 0.0);
    if (tid == 0) s_carry = 0;
    __syncthreads();
    if (tid == 0) mat34_inv(s_T, s_Tin);
    __syncthreads();
    if (tid < 12) st.kf_T[12 * (size_t)e + tid] = s_T[tid];
    if (tid == 0) {
        st.kf_n[e] = n;
        st.kf_slot[e] = kj.kf_slot;
        st.kf_mp0[e] = kj.mp0;
        res[blockIdx.x].n_features = n;
    }
    const double* depth = st.depth_map + (size_t)kj.stream * st.W * st.H;
    for (int g = tid; g < n; g += 1024) {
        const size_t s = (size_t)kj.frame_slot * n_cells + g, fe = (size_t)e * st.cells + g;
        const int L = f_level[s];
        const double x = (double)((int)f_x[s] << L), y = (double)((int)f_y[s] << L);   // Feature::_pixel = level coordinate * 2^level
        const double d = depth[(size_t)(int)y * st.W + (int)x];
        st.kf_px[2 * fe] = x;
        st.kf_px[2 * fe + 1] = y;
        st.kf_level[fe] = (uint8_t)L;
        st.kf_depth[fe] = d;
        const double pc0 = (x - st.cx) * d / st.fx, pc1 = (y - st.cy) * d / st.fy, pc2 = d;
        for (int r = 0; r < 3; ++r)
            st.kf_pw[3 * fe + r] = s_Tin[4 * r] * pc0 + s_Tin[4 * r + 1] * pc1 + s_Tin[4 * r + 2] * pc2 + s_Tin[4 * r + 3];
    }
    // observations of older map points: the inliers of the tracking job, in candidate order
    int total = 0;
    if (kj.track_job >= 0) {
        const int tj = kj.track_job;
        const ygzb_track_job job = b.jobs[tj];
        const int cnt = b.aligned[tj] ? b.c_cnt[tj] : 0;
        for (int base = 0; base < cnt; base += 1024) {
            const int q = base + tid;
            const size_t at = (size_t)tj * b.cap + q;
            const int flag = (q < cnt && b.inlier[at]) ? 1 : 0;
            int chunk_total;
            const int incl = block_scan_1024(flag, s_scan, &chunk_total);
            if (flag) {
                const size_t dst = (size_t)e * b.cap + s_carry + incl - 1;
                const int c = b.c_src[at], k = c / st.cells, f = c - k * st.cells;
                st.kf_obs_id[dst] = st.kf_mp0[job.stream * st.R + job.entry[k]] + f;
                st.kf_obs_px[2 * dst] = b.c_px[2 * at];
                st.kf_obs_px[2 * dst + 1] = b.c_px[2 * at + 1];
            }
            __syncthreads();
            if (tid == 0) s_carry += chunk_total;
            __syncthreads();
        }
        total = s_carry;
    }
    if (tid == 0) st.kf_nobs[e] = total;
}

struct BABuild {   // device arrays of the batch of local-BA problems (capacity based: problem p owns fixed ranges)
    int32_t *kf_off, *pt_off, *obs_off;   // [P + 1]
    int32_t *n_kf, *n_pt;                 // [P]
    double* poses;                        // [P][kTrackMaxLocal][6]
    uint8_t* fixed;                       // [P][kTrackMaxLocal]
    double* pts;                          // [P][pcap][3]
    int32_t* lm_start;                    // [P][pcap]
    int32_t* so_kf;                       // [P][ocap]
    double* so_uv;                        // [P][ocap][2]
    int32_t* owner;                       // [P][pcap]  dense index (local key-frame * cells + feature) of every BA point
    int32_t* tab;                         // [P][kTrackMaxLocal][kTrackMaxLocal * cells]  observation of point i in key-frame k' (+1)
    int32_t* prob_of;                     // [n key-frame jobs] -> problem or -1
    int pcap, ocap;
};

// LocalMapping::LocalBA problem of key-frame job kf_job[blockIdx.x] (if it runs a BA): the local key-frames and the points
// at least two of them observe (a key-frame observes its own points and the older points tracked into it), landmark-major
__global__ void __launch_bounds__(1024) ba_build_kernel(TrackStore st, const ygzb_keyframe_job* __restrict__ jobs, BABuild B, int cap_obs) {
    __shared__ int s_scan[1024];
    __shared__ int s_cpt, s_cobs;
    const int p = B.prob_of[blockIdx.x];
    if (p < 0) return;
    const ygzb_keyframe_job kj = jobs[blockIdx.x];
    const int tid = threadIdx.x, nk = kj.n_local, dense = nk * st.cells;
    int e[kTrackMaxLocal], nf[kTrackMaxLocal];
    long long m0[kTrackMaxLocal];
    for (int k = 0; k < kTrackMaxLocal; ++k) {
        e[k] = kj.stream * st.R + kj.local_entry[k < nk ? k : 0];
        nf[k] = k < nk ? st.kf_n[e[k]] : 0;
        m0[k] = st.kf_mp0[e[k]];
    }
    int32_t* tab = B.tab + (size_t)p * kTrackMaxLocal * kTrackMaxLocal * st.cells;
    for (int i = tid; i < nk * dense; i += 1024) tab[(size_t)(i / dense) * kTrackMaxLocal * st.cells + (i % dense)] = 0;
    if (tid == 0) s_cpt = s_cobs = 0;
    __syncthreads();
    for (int k2 = 0; k2 < nk; ++k2) {
        const int nobs = st.kf_nobs[e[k2]];
        for (int q = tid; q < nobs; q += 1024) {
            const long long id = st.kf_obs_id[(size_t)e[k2] * cap_obs + q];
            for (int k = 0; k < nk; ++k)
                if (id >= m0[k] && id < m0[k] + nf[k]) {
                    tab[(size_t)k2 * kTrackMaxLocal * st.cells + k * st.cells + (int)(id - m0[k])] = q + 1;
                    break;
                }
        }
    }
    __syncthreads();
    const int p0 = p * B.pcap, o0 = p * B.ocap;
    // every thread takes `per` CONSECUTIVE dense indices (so the output order is the dense order), finds their degrees with all
    // the table loads in flight at once, and ONE block scan of the per-thread (points, observations) totals places them
    constexpr int kMaxPer = (kTrackMaxLocal * 4096 + 1023) / 1024;   // cells <= 4096
    const int per = (dense + 1023) / 1024;
    int degs[kMaxPer];
    int my_pts = 0, my_obs = 0;
#pragma unroll
    for (int r = 0; r < kMaxPer; ++r) {
        degs[r] = 0;
        const int i = tid * per + r;
        if (r < per && i < dense) {
            const int k = i / st.cells, g = i - k * st.cells;
            if (g < nf[k]) {
                int deg = 1;
                for (int k2 = 0; k2 < nk; ++k2) deg += tab[(size_t)k2 * kTrackMaxLocal * st.cells + i] != 0;
                if (deg >= 2) {
                    degs[r] = deg;
                    my_pts += 1;
                    my_obs += deg;
                }
            }
        }
    }
    int total_packed;
    const int incl = block_scan_1024(my_pts | (my_obs << 15), s_scan, &total_packed);   // 15 bits of points, 17 of observations
    int pt = (incl & 0x7FFF) - my_pts, ob = (int)((unsigned)incl >> 15) - my_obs;   // exclusive prefix of this thread
#pragma unroll
    for (int r = 0; r < kMaxPer; ++r) {
        const int deg = degs[r];
        if (!deg) continue;
        const int i = tid * per + r, k = i / st.cells, g = i - k * st.cells;
        const size_t P = (size_t)p0 + pt, fe = (size_t)e[k] * st.cells + g;
        B.pts[3 * P] = st.kf_pw[3 * fe];
        B.pts[3 * P + 1] = st.kf_pw[3 * fe + 1];
        B.pts[3 * P + 2] = st.kf_pw[3 * fe + 2];
        B.lm_start[P] = o0 + ob;
        B.owner[P] = i;
        size_t o = (size_t)o0 + ob;
        B.so_kf[o] = k;
        B.so_uv[2 * o] = st.kf_px[2 * fe];
        B.so_uv[2 * o + 1] = st.kf_px[2 * fe + 1];
        ++o;
        for (int k2 = 0; k2 < nk; ++k2) {
            const int q = tab[(size_t)k2 * kTrackMaxLocal * st.cells + i];
            if (!q) continue;
            B.so_kf[o] = k2;
            B.so_uv[2 * o] = st.kf_obs_px[2 * ((size_t)e[k2] * cap_obs + q - 1)];
            B.so_uv[2 * o + 1] = st.kf_obs_px[2 * ((size_t)e[k2] * cap_obs + q - 1) + 1];
            ++o;
        }
        pt += 1;
        ob += deg;
    }
    if (tid == 0) {
        s_cpt = total_packed & 0x7FFF;
        s_cobs = (int)((unsigned)total_packed >> 15);
    }
    __syncthreads();
    if (tid == 0) {
        B.lm_start[(size_t)p0 + s_cpt] = o0 + s_cobs;
        B.n_kf[p] = nk;
        B.n_pt[p] = s_cpt;
        B.kf_off[p] = p * kTrackMaxLocal;
        B.pt_off[p] = p0;
        B.obs_off[p] = o0;
    }
    if (tid < nk) {
        double lg[6];
        se3_log(se3_from_mat(st.kf_T + 12 * (size_t)e[tid]), lg);
        double* g2o = B.poses + 6 * ((size_t)p * kTrackMaxLocal + tid);
        g2o[0] = lg[3]; g2o[1] = lg[4]; g2o[2] = lg[5]; g2o[3] = lg[0]; g2o[4] = lg[1]; g2o[5] = lg[2];   // VertexSE3Sophus: [omega; upsilon]
        B.fixed[p * kTrackMaxLocal + tid] = tid == 0 ? 1 : 0;   // the oldest local key-frame fixes the gauge (key-frame 0 in the reference)
    }
}

// BA result back into the ring (poses of every local key-frame, refined map points) and into the result records
__global__ void __launch_bounds__(256) ba_writeback_kernel(TrackStore st, const ygzb_keyframe_job* __restrict__ jobs, BABuild B,
                                                           const double* __restrict__ ba_stats, ygzb_keyframe_result* __restrict__ res) {
    const ygzb_keyframe_job kj = jobs[blockIdx.x];
    const int p = B.prob_of[blockIdx.x], tid = threadIdx.x, nk = kj.n_local;
    ygzb_keyframe_result* r = res + blockIdx.x;
    if (p >= 0) {
        if (tid < nk) {
            const double* g = B.poses + 6 * ((size_t)p * kTrackMaxLocal + tid);
            const double v[6] = {g[3], g[4], g[5], g[0], g[1], g[2]};
            se3_to_mat(se3_exp(v), st.kf_T + 12 * (size_t)(kj.stream * st.R + kj.local_entry[tid]));
        }
        const int npt = B.n_pt[p];
        for (int q = tid; q < npt; q += 256) {
            const int i = B.owner[(size_t)p * B.pcap + q], k = i / st.cells, g = i - k * st.cells;
            const size_t fe = (size_t)(kj.stream * st.R + kj.local_entry[k]) * st.cells + g;
            for (int c = 0; c < 3; ++c) st.kf_pw[3 * fe + c] = B.pts[3 * ((size_t)p * B.pcap + q) + c];
        }
        if (tid == 0) {
            const double* s = ba_stats + 8 * (size_t)p;
            r->ba_points = npt;
            r->ba_observations = B.lm_start[(size_t)p * B.pcap + npt] - p * B.ocap;
            r->ba_iters = (int)s[0];
            r->ba_trials = (int)s[1];
            r->chi2_initial = s[2];
            r->chi2_final = s[3];
            r->pad = 0;
        }
    } else if (tid == 0) {
        r->ba_points = r->ba_observations = r->ba_iters = r->ba_trials = r->pad = 0;
        r->chi2_initial = r->chi2_final = 0;
    }
    __syncthreads();
    if (tid < 12 * nk) r->T_cw[tid / 12][tid % 12] = st.kf_T[12 * (size_t)(kj.stream * st.R + kj.local_entry[tid / 12]) + tid % 12];
}

size_t babuild_carve(Carver& c, BABuild& B, size_t P, int cells, int n_jobs) {
    B.kf_off = c.take<int32_t>(P + 1); B.pt_off = c.take<int32_t>(P + 1); B.obs_off = c.take<int32_t>(P + 1);
    B.n_kf = c.take<int32_t>(P); B.n_pt = c.take<int32_t>(P);
    B.poses = c.take<double>(P * kTrackMaxLocal * 6);
    B.fixed = c.take<uint8_t>(P * kTrackMaxLocal);
    B.pts = c.take<double>(P * B.pcap * 3);
    B.lm_start = c.take<int32_t>(P * B.pcap);
    B.so_kf = c.take<int32_t>(P * B.ocap);
    B.so_uv = c.take<double>(P * B.ocap * 2);
    B.owner = c.take<int32_t>(P * B.pcap);
    B.tab = c.take<int32_t>(P * kTrackMaxLocal * kTrackMaxLocal * cells);
    B.prob_of = c.take<int32_t>((size_t)n_jobs);
    return c.bytes();
}

}  // namespace

extern "C" {

int ygzb_tracker_create(ygzb_frames* f, int n_streams, int max_jobs, const double K[4], ygzb_tracker** out) {
    if (!f || !out || n_streams < 1 || max_jobs < 1 || !K) return YGZB_ERR_INVALID;
    *out = nullptr;
    ygzb_ctx* ctx = f->ctx;
    cudaSetDevice(ctx->device);
    if (ctx->geo.n_cells > 4096) return set_error(ctx, YGZB_ERR_CAPACITY, "tracker: %d grid cells (the BA assembly handles up to 4096)", ctx->geo.n_cells);
    ygzb_tracker* t = new (std::nothrow) ygzb_tracker();
    if (!t) return YGZB_ERR_INVALID;
    memset(t, 0, sizeof(*t));
    t->f = f;
    t->ctx = ctx;
    t->max_jobs = max_jobs;
    t->cluster = 4;
    if (const char* e = getenv("YGZB_TRACK_CLUSTER")) {   // tuning knob: 1, 2, 4 or 8
        const int v = atoi(e);
        if (v == 1 || v == 2 || v == 4 || v == 8) t->cluster = v;
    }
    const Geometry& g = ctx->geo;
    const size_t S = (size_t)n_streams, R = YGZB_TRACK_RING, cells = (size_t)g.n_cells, E = S * R, cap = kTrackMaxLocal * cells;
    TrackStore& st = t->st;
    st.S = n_streams; st.R = (int)R; st.cells = (int)cells; st.W = g.W; st.H = g.H;
    st.fx = K[0]; st.fy = K[1]; st.cx = K[2]; st.cy = K[3];
    int rc = YGZB_OK;
    {
        Carver sz(nullptr);
        sz.take<double>(E * 12); sz.take<int32_t>(E); sz.take<int32_t>(E); sz.take<long long>(E); sz.take<double>(E * cells * 2);
        sz.take<uint8_t>(E * cells); sz.take<double>(E * cells); sz.take<double>(E * cells * 3); sz.take<int32_t>(E);
        sz.take<long long>(E * cap); sz.take<double>(E * cap * 2);
        rc = check_cuda(ctx, cudaMalloc(&t->d_store, sz.bytes()), "cudaMalloc(tracker store)");
        if (rc == YGZB_OK) rc = check_cuda(ctx, cudaMemsetAsync(t->d_store, 0, sz.bytes(), ctx->stream), "memset");
        if (rc == YGZB_OK) {
            Carver c(t->d_store);
            st.kf_T = c.take<double>(E * 12); st.kf_n = c.take<int32_t>(E); st.kf_slot = c.take<int32_t>(E); st.kf_mp0 = c.take<long long>(E);
            st.kf_px = c.take<double>(E * cells * 2); st.kf_level = c.take<uint8_t>(E * cells); st.kf_depth = c.take<double>(E * cells);
            st.kf_pw = c.take<double>(E * cells * 3); st.kf_nobs = c.take<int32_t>(E); st.kf_obs_id = c.take<long long>(E * cap);
            st.kf_obs_px = c.take<double>(E * cap * 2);
        }
    }
    if (rc == YGZB_OK) rc = dalloc(ctx, &t->d_depth, S * g.W * g.H);
    st.depth_map = t->d_depth;
    if (rc == YGZB_OK) {
        const size_t J = (size_t)max_jobs, F = J * cells, Cn = J * cap;
        TrackBatch& b = t->b;
        b.J = 0;
        b.cap = (int)cap;
        auto carve = [&](Carver& c) {
            b.jobs = c.take<ygzb_track_job>(J);
            b.ref_slot = c.take<int32_t>(J); b.cur_slot = c.take<int32_t>(J); b.offsets = c.take<int32_t>(J + 1); b.in_off = c.take<int32_t>(J);
            b.n_feat = c.take<int32_t>(J); b.n_meas = c.take<int32_t>(J);
            b.T_ref = c.take<double>(J * 12); b.T_cur = c.take<double>(J * 12);
            b.feat_scratch = c.take<uint8_t>(sparse_align_scratch_bytes(F));
            b.aligned = c.take<int32_t>(J); b.rel = c.take<double>(J * kTrackMaxLocal * 12);
            b.cand_ok = c.take<uint8_t>(Cn); b.cand_px = c.take<double>(Cn * 2); b.n_cand = c.take<int32_t>(J);
            b.c_cnt = c.take<int32_t>(J); b.c_off = c.take<int32_t>(J + 1); b.c_src = c.take<int32_t>(Cn);
            b.c_pw = c.take<double>(Cn * 3); b.c_px = c.take<double>(Cn * 2); b.c_depth = c.take<double>(Cn);
            b.inlier = c.take<uint8_t>(Cn); b.enable = c.take<uint8_t>(Cn); b.n_inl = c.take<int32_t>(J);
            b.pose_ws = c.take<double>(pose_only_ws_doubles((int)J));
            b.results = c.take<ygzb_track_result>(J);
        };
        Carver sz(nullptr);
        carve(sz);
        rc = check_cuda(ctx, cudaMalloc(&t->d_batch, sz.bytes()), "cudaMalloc(tracker batch)");
        if (rc == YGZB_OK) rc = check_cuda(ctx, cudaMemsetAsync(t->d_batch, 0, sz.bytes(), ctx->stream), "memset");
        if (rc == YGZB_OK) {
            Carver c(t->d_batch);
            carve(c);
        }
    }
    if (rc == YGZB_OK) rc = check_cuda(ctx, cudaMallocHost((void**)&t->h_jobs, sizeof(ygzb_track_job) * (size_t)max_jobs), "cudaMallocHost");
    if (rc == YGZB_OK) rc = check_cuda(ctx, cudaMallocHost((void**)&t->h_kfjobs, sizeof(ygzb_keyframe_job) * S), "cudaMallocHost");
    if (rc == YGZB_OK) rc = dalloc(ctx, &t->d_kfjobs, S);
    if (rc == YGZB_OK) rc = dalloc(ctx, &t->d_kfres, S);
    // (a result record carries YGZB_TRACK_RING pose slots and only the first n_local are written by a job: the whole record is
    //  copied back, so start from zeros rather than from whatever cudaMalloc returned)
    if (rc == YGZB_OK) rc = check_cuda(ctx, cudaMemsetAsync(t->d_kfres, 0, sizeof(ygzb_keyframe_result) * S, ctx->stream), "memset");
    if (rc == YGZB_OK) rc = check_cuda(ctx, cudaEventCreateWithFlags(&t->staged, cudaEventDisableTiming), "cudaEventCreate");
    if (rc == YGZB_OK) rc = check_cuda(ctx, cudaStreamCreateWithFlags(&t->front, cudaStreamNonBlocking), "cudaStreamCreate");
    for (cudaEvent_t* e : {&t->e_fill, &t->e_front, &t->e_main, &t->e_up})
        if (rc == YGZB_OK) rc = check_cuda(ctx, cudaEventCreateWithFlags(e, cudaEventDisableTiming), "cudaEventCreate");
    if (rc == YGZB_OK) {   // (events start out "completed": recorded once on an idle stream)
        rc = check_cuda(ctx, cudaEventRecord(t->e_fill, ctx->stream), "cudaEventRecord");
        if (rc == YGZB_OK) rc = check_cuda(ctx, cudaEventRecord(t->e_main, ctx->stream), "cudaEventRecord");
        if (rc == YGZB_OK) rc = check_cuda(ctx, cudaEventRecord(t->e_up, ctx->stream), "cudaEventRecord");
    }
    if (rc == YGZB_OK) {
        t->pcap = (int)(kTrackMaxLocal * cells + 1);
        t->ocap = (int)(kTrackMaxLocal * kTrackMaxLocal * cells);
        BABuild B{};
        B.pcap = t->pcap;
        B.ocap = t->ocap;
        Carver sz(nullptr);
        const size_t head = babuild_carve(sz, B, S, (int)cells, (int)S);
        t->ba_bytes = head + ba2_scratch_bytes(S * t->pcap, S * t->ocap, S) + 512;
        rc = check_cuda(ctx, cudaMalloc(&t->d_ba, t->ba_bytes), "cudaMalloc(tracker BA)");
    }
    if (rc != YGZB_OK) {
        ygzb_tracker_destroy(t);
        return rc;
    }
    *out = t;
    return YGZB_OK;
}

void ygzb_tracker_destroy(ygzb_tracker* t) {
    if (!t) return;
    cudaSetDevice(t->ctx->device);
    cudaStreamSynchronize(t->ctx->stream);
    if (t->d_store) cudaFree(t->d_store);
    if (t->d_batch) cudaFree(t->d_batch);
    if (t->d_depth) cudaFree(t->d_depth);
    if (t->h_jobs) cudaFreeHost(t->h_jobs);
    if (t->h_kfjobs) cudaFreeHost(t->h_kfjobs);
    if (t->d_kfjobs) cudaFree(t->d_kfjobs);
    if (t->d_kfres) cudaFree(t->d_kfres);
    if (t->d_ba) cudaFree(t->d_ba);
    if (t->staged) cudaEventDestroy(t->staged);
    if (t->front) {
        cudaStreamSynchronize(t->front);
        cudaStreamDestroy(t->front);
    }
    for (cudaEvent_t e : {t->e_fill, t->e_front, t->e_main, t->e_up})
        if (e) cudaEventDestroy(e);
    delete t;
}

int ygzb_tracker_set_depth(ygzb_tracker* t, int stream, const double* depth) {
    if (!t || !depth || stream < 0 || stream >= t->st.S) return YGZB_ERR_INVALID;
    ygzb_ctx* ctx = t->ctx;
    cudaSetDevice(ctx->device);
    const size_t n = (size_t)t->st.W * t->st.H;
    YGZB_CUDA(ctx, cudaMemcpyAsync(t->d_depth + (size_t)stream * n, depth, n * sizeof(double), cudaMemcpyDefault, ctx->stream));
    return YGZB_OK;
}

int ygzb_tracker_upload(ygzb_tracker* t, int first, int count, const uint8_t* host, size_t frame_stride) {
    if (!t) return YGZB_ERR_INVALID;
    ygzb_ctx* ctx = t->ctx;
    cudaSetDevice(ctx->device);
    // on the front stream, behind the last key-frame insertion (which still reads the frame slots of the previous window) and
    // behind the last tracking chain (ditto); NOT behind a local BA in flight
    YGZB_CUDA(ctx, cudaStreamWaitEvent(t->front, t->e_fill, 0));
    YGZB_CUDA(ctx, cudaStreamWaitEvent(t->front, t->e_main, 0));
    cudaStream_t main = ctx->stream;
    ctx->stream = t->front;
    int rc = ygzb_frames_upload(t->f, first, count, host, 1, frame_stride);
    if (rc == YGZB_OK) rc = check_cuda(ctx, cudaEventRecord(t->e_up, ctx->stream), "cudaEventRecord");
    ctx->stream = main;
    return rc;
}

int ygzb_tracker_track(ygzb_tracker* t, int n_jobs, const ygzb_track_job* jobs, ygzb_track_result* results) {
    if (!t || n_jobs < 0 || (n_jobs && (!jobs || !results))) return YGZB_ERR_INVALID;
    if (n_jobs == 0) return YGZB_OK;
    ygzb_ctx* ctx = t->ctx;
    cudaSetDevice(ctx->device);
    if (n_jobs > t->max_jobs) return set_error(ctx, YGZB_ERR_CAPACITY, "%d jobs exceed the tracker's max_jobs %d", n_jobs, t->max_jobs);
    for (int j = 0; j < n_jobs; ++j) {
        const ygzb_track_job& q = jobs[j];
        if (q.stream < 0 || q.stream >= t->st.S || q.cur_slot < 0 || q.cur_slot >= t->f->capacity || q.n_local < 1 || q.n_local > kTrackMaxLocal - 1)
            return set_error(ctx, YGZB_ERR_INVALID, "track job %d: stream / slot / n_local out of range", j);
        for (int k = 0; k < q.n_local; ++k)
            if (q.entry[k] < 0 || q.entry[k] >= YGZB_TRACK_RING) return set_error(ctx, YGZB_ERR_INVALID, "track job %d: ring entry out of range", j);
    }
    YGZB_CUDA(ctx, cudaEventSynchronize(t->staged));   // the previous copy out of the staging buffer has finished
    memcpy(t->h_jobs, jobs, sizeof(ygzb_track_job) * (size_t)n_jobs);
    TrackBatch b = t->b;
    b.J = n_jobs;
    t->last_J = n_jobs;
    const int cl = t->cluster;
    int rc;
    {   // part 1 on the front stream: behind the key-frame insertion (new reference features, and the batch arrays it still
        // reads) and the previous chain, concurrent with a local BA on the main stream
        cudaStream_t main = ctx->stream;
        YGZB_CUDA(ctx, cudaStreamWaitEvent(t->front, t->e_fill, 0));
        YGZB_CUDA(ctx, cudaStreamWaitEvent(t->front, t->e_main, 0));
        ctx->stream = t->front;
        cudaError_t ce = cudaMemcpyAsync(const_cast<ygzb_track_job*>(t->b.jobs), t->h_jobs, sizeof(ygzb_track_job) * (size_t)n_jobs,
                                         cudaMemcpyHostToDevice, ctx->stream);
        if (ce == cudaSuccess) ce = cudaEventRecord(t->staged, ctx->stream);
        rc = ce == cudaSuccess ? launch_track_chain_front(t->f, t->st, b, cl) : check_cuda(ctx, ce, "H2D(track jobs)");
        if (rc == YGZB_OK) rc = check_cuda(ctx, cudaEventRecord(t->e_front, ctx->stream), "cudaEventRecord");
        ctx->stream = main;
        if (rc != YGZB_OK) return rc;
        YGZB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, t->e_front, 0));
    }
    rc = launch_track_chain_mid(t->f, t->st, b);
    if (rc != YGZB_OK) return rc;
    rc = launch_pose_only_dev(ctx, n_jobs, b.c_off, b.c_cnt, b.c_pw, b.c_px, b.T_cur, b.inlier, b.c_depth, b.n_inl, b.enable, b.pose_ws, cl, b.cap);
    if (rc != YGZB_OK) return rc;
    {
        ProfScope ps(ctx, kStageOther);
        track_finish_kernel<<<(n_jobs + 63) / 64, 64, 0, ctx->stream>>>(b);
        YGZB_LAUNCHED(ctx);
    }
    YGZB_CUDA(ctx, cudaMemcpyAsync(results, b.results, sizeof(ygzb_track_result) * (size_t)n_jobs, cudaMemcpyDeviceToHost, ctx->stream));
    YGZB_CUDA(ctx, cudaEventRecord(t->e_main, ctx->stream));
    return YGZB_OK;
}

int ygzb_tracker_make_keyframes(ygzb_tracker* t, int n, const ygzb_keyframe_job* jobs, const ygzb_ba_params* ba,
                                ygzb_keyframe_result* results) {
    if (!t || n < 0 || (n && (!jobs || !results || !ba))) return YGZB_ERR_INVALID;
    if (n == 0) return YGZB_OK;
    ygzb_ctx* ctx = t->ctx;
    ygzb_frames* f = t->f;
    cudaSetDevice(ctx->device);
    if (n > t->st.S) return set_error(ctx, YGZB_ERR_CAPACITY, "%d key-frame jobs for %d streams", n, t->st.S);
    std::vector<int32_t> slots(n), prob_of(n);
    int P = 0;
    for (int i = 0; i < n; ++i) {
        const ygzb_keyframe_job& q = jobs[i];
        if (q.stream < 0 || q.stream >= t->st.S || q.frame_slot < 0 || q.frame_slot >= f->capacity || q.kf_slot < 0 || q.kf_slot >= f->capacity ||
            q.entry < 0 || q.entry >= YGZB_TRACK_RING || q.track_job >= t->last_J || q.n_local < 1 || q.n_local > kTrackMaxLocal - 1)
            return set_error(ctx, YGZB_ERR_INVALID, "key-frame job %d: field out of range", i);
        for (int k = 0; k < q.n_local; ++k)
            if (q.local_entry[k] < 0 || q.local_entry[k] >= YGZB_TRACK_RING) return set_error(ctx, YGZB_ERR_INVALID, "key-frame job %d: ring entry out of range", i);
        if (q.local_entry[q.n_local - 1] != q.entry) return set_error(ctx, YGZB_ERR_INVALID, "key-frame job %d: the newest local key-frame must be the inserted one", i);
        for (int i2 = 0; i2 < i; ++i2)
            if (jobs[i2].stream == q.stream) return set_error(ctx, YGZB_ERR_INVALID, "two key-frame jobs for stream %d", q.stream);
        slots[i] = q.frame_slot;
        prob_of[i] = (q.run_ba && q.n_local >= 2) ? P++ : -1;
    }
    // FeatureDetector::Detect on the frames (results stay in the slots' feature store); the frames may have been uploaded on
    // the front stream without a tracking chain behind them (first frame of a stream)
    YGZB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, t->e_up, 0));
    int rc = ygzb_detect(f, slots.data(), n, nullptr, nullptr);
    if (rc != YGZB_OK) return rc;
    for (int i = 0; i < n; ++i)
        if (jobs[i].frame_slot != jobs[i].kf_slot) {
            rc = ygzb_frames_copy(f, jobs[i].frame_slot, jobs[i].kf_slot);   // the key-frame keeps its pyramid (Frame.h:138)
            if (rc != YGZB_OK) return rc;
        }
    YGZB_CUDA(ctx, cudaEventSynchronize(t->staged));
    memcpy(t->h_kfjobs, jobs, sizeof(ygzb_keyframe_job) * (size_t)n);
    YGZB_CUDA(ctx, cudaMemcpyAsync(t->d_kfjobs, t->h_kfjobs, sizeof(ygzb_keyframe_job) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    BABuild B{};
    B.pcap = t->pcap;
    B.ocap = t->ocap;
    Carver c(t->d_ba);
    const size_t head = babuild_carve(c, B, (size_t)t->st.S, t->st.cells, t->st.S);
    // the problem indices travel behind the jobs in the same staging buffer's lifetime: small synchronous-safe copy from a
    // host vector is fine because the stream is synchronised on `staged` before the vector dies (cudaMemcpyAsync from pageable
    // memory returns after the data has been staged)
    YGZB_CUDA(ctx, cudaMemcpyAsync(B.prob_of, prob_of.data(), sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    YGZB_CUDA(ctx, cudaEventRecord(t->staged, ctx->stream));
    TrackBatch b = t->b;
    b.J = t->last_J;
    {
        ProfScope ps(ctx, kStageOther);
        kf_fill_kernel<<<(unsigned)n, 1024, 0, ctx->stream>>>(t->st, b, t->d_kfjobs, f->d_count, f->d_fx, f->d_fy, f->d_flevel, ctx->geo.n_cells,
                                                             t->d_kfres);
        YGZB_LAUNCHED(ctx);
    }
    YGZB_CUDA(ctx, cudaEventRecord(t->e_fill, ctx->stream));   // from here on only the BA runs: the next batch's front part may start
    double* d_ba_stats = nullptr;
    if (P > 0) {
        {
            ProfScope ps(ctx, kStageOther);
            ba_build_kernel<<<(unsigned)n, 1024, 0, ctx->stream>>>(t->st, t->d_kfjobs, B, b.cap);
            YGZB_LAUNCHED(ctx);
        }
        BA2Problem in{};
        in.n_problems = P;
        in.kf_off = B.kf_off; in.pt_off = B.pt_off; in.obs_off = B.obs_off;
        in.n_kf = B.n_kf; in.n_pt = B.n_pt;
        in.poses = B.poses; in.fixed = B.fixed; in.pts = B.pts;
        in.kf_idx = B.so_kf; in.pt_idx = nullptr; in.obs = B.so_uv; in.lm_start = B.lm_start;
        in.total_pts = (size_t)P * t->pcap;
        in.total_obs = (size_t)P * t->ocap;
        int max_local = 1;
        for (int i = 0; i < n; ++i) max_local = std::max(max_local, jobs[i].n_local);
        in.max_pts = (size_t)(max_local - 1) * t->st.cells;   // the newest key-frame's own points have one observation: never in the BA
        in.max_obs = (size_t)max_local * in.max_pts;
        in.max_free = max_local - 1;
        in.max_kf = max_local;
        void* scratch = static_cast<uint8_t*>(t->d_ba) + ((head + 255) & ~(size_t)255);
        rc = launch_local_ba2(ctx, in, scratch, ba, nullptr, &d_ba_stats);
        if (rc != YGZB_OK) return rc;
    }
    {
        ProfScope ps(ctx, kStageOther);
        ba_writeback_kernel<<<(unsigned)n, 256, 0, ctx->stream>>>(t->st, t->d_kfjobs, B, d_ba_stats, t->d_kfres);
        YGZB_LAUNCHED(ctx);
    }
    YGZB_CUDA(ctx, cudaMemcpyAsync(results, t->d_kfres, sizeof(ygzb_keyframe_result) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    return YGZB_OK;
}

}  // extern "C"
