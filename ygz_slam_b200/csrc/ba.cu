// ba.cu -- local bundle adjustment of the Ceres twin (trust-region LM + Schur complement) and pose-only refinement
// (Ceres-style trust-region LM), each as ONE persistent CTA cluster per problem: the whole optimisation loop runs
// on the device, the host sees one launch per batch of problems.  ba::LocalBAG2O runs in ba2.cu; its C ABI
// marshalling is here.
//
// Replaces:
//   ba::LocalBA, ba::TwoViewBACeres  reference src/Algorithm/BA.cpp:324-385, 11-89
//   ba::OptimizeCurrentPoseOnly      reference src/Algorithm/BA.cpp:188-264
//   CeresReprojectionErrorPoseOnly   reference include/ygz/Ceres/CeresReprojectionErrorPoseOnly.h:27-58
// g2o / Ceres themselves are outside the reference tree: the optimiser logic follows the published
// algorithms as pinned in oracle/ba.cpp (SURVEY.md appendix A.3 / A.4).
//
// Local BA, per LM trial (C4: 10 keyframes, 2000 landmarks, ~8000 observations):
//   linearise      thread per observation : error, Huber weight, 2x3 / 2x6 Jacobians by forward-mode jets
//   Hll, bl        thread per landmark    : sum over its observations (CSR by landmark)
//   Hpp, bp        warp per free pose     : warp-shuffle reduction of J^T J (21+6 terms) over its observations
//   Schur S, b_s   warp per 6x6 block pair: S(f1,f2) -= Hpl Hll^-1 Hpl^T over the landmarks seen by both poses,
//                                           36 partial sums per lane reduced with warp shuffles, no atomics
//   solve          dense Cholesky of S (<= 96x96) in shared memory by the whole CTA
//   back-subst     thread per landmark
// Roofline class: FP64 ALU / latency (0.3 MB of unique data per iteration, ~1.1e7 FLOP): bench.py reports
// achieved FLOP/s for the reduce, not HBM bytes.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <mutex>
#include <utility>
#include <vector>

#include <cooperative_groups.h>

#include "ba2.cuh"
#include "common.cuh"
#include "se3.cuh"
#include "track.cuh"

namespace ygzb {

namespace {

constexpr int kBAThreads = 256;
constexpr int kMaxFreePoses = 16;             // S is at most 96 x 96 doubles = 72 KB of shared memory
constexpr int kMaxPoses = 64;

struct BAArgs {
    // problem p owns poses [kf_off[p], kf_off[p+1]), points [pt_off[p], ..), observations [obs_off[p], ..)
    const int32_t *kf_off, *pt_off, *obs_off;
    double* poses;            // [t; angle-axis], in/out
    const uint8_t* fixed;
    double* pts;              // in/out
    const int32_t* kf_idx;    // per obs, LOCAL pose index inside the problem
    const int32_t* pt_idx;    // per obs, LOCAL point index
    const double* obs;        // per obs (u, v)
    // structure built on the host (index bookkeeping only)
    const int32_t* lm_start;  // per point (global index): range in lm_obs
    const int32_t* lm_obs;    // observation ids (global) grouped by landmark
    const int32_t* ps_start;  // per pose (global index): range in ps_obs
    const int32_t* ps_obs;    // observation ids grouped by pose
    const int32_t* pair_off;  // per problem: offset into pair_start (n_free*(n_free+1)/2 + 1 entries per problem)
    const int32_t* pair_start;
    const int32_t* pair_o1;   // entries: observation on pose f1, observation on pose f2 (same landmark)
    const int32_t* pair_o2;
    // per-observation / per-landmark scratch
    double* lin;              // [n_obs][21]: e(2) w Jl(6) Jp(12)
    double* Hll;              // [n_pt][9]
    double* bl;               // [n_pt][3]
    double* Dinv;             // [n_pt][9]
    double* xl;               // [n_pt][3]
    double* pts_backup;       // [n_pt][3]
    double* scale_l;          // [n_pt][3]  Ceres twin: Jacobi scaling of the landmark columns
    double* stats;            // [n_problems][8]: trials, successful steps, cost_first, cost_last, radius, termination
    float fx, fy, cx, cy;
    int max_iters;
    double huber_delta;
    const uint8_t* loss_mask;   // residual blocks that carry the HuberLoss (null = all of them)
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, o);
    return v;
}

// block-wide sum, result valid in every thread
__device__ double block_sum(double v, double* s_tmp /* 33 doubles */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) s_tmp[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double t = (lane < (int)(blockDim.x >> 5)) ? s_tmp[lane] : 0.0;
        t = warp_sum(t);
        if (lane == 0) s_tmp[32] = t;
    }
    __syncthreads();
    return s_tmp[32];
}

__device__ double block_max(double v, double* s_tmp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_down_sync(0xFFFFFFFFu, v, o));
    __syncthreads();
    if (lane == 0) s_tmp[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double t = (lane < (int)(blockDim.x >> 5)) ? s_tmp[lane] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t = fmax(t, __shfl_down_sync(0xFFFFFFFFu, t, o));
        if (lane == 0) s_tmp[32] = t;
    }
    __syncthreads();
    return s_tmp[32];
}

__device__ __forceinline__ void inverse3d(const double* H /* row major 3x3 */, double* inv) {
#define COF(i, j) (H[((i + 1) % 3) * 3 + (j + 1) % 3] * H[((i + 2) % 3) * 3 + (j + 2) % 3] - H[((i + 1) % 3) * 3 + (j + 2) % 3] * H[((i + 2) % 3) * 3 + (j + 1) % 3])
    const double c00 = COF(0, 0), c10 = COF(1, 0), c20 = COF(2, 0);
    const double det = (c00 * H[0] + c10 * H[3]) + c20 * H[6];
    const double invdet = 1.0 / det;
    inv[0] = c00 * invdet; inv[1] = c10 * invdet; inv[2] = c20 * invdet;
    inv[3] = COF(0, 1) * invdet; inv[4] = COF(1, 1) * invdet; inv[5] = COF(2, 1) * invdet;
    inv[6] = COF(0, 2) * invdet; inv[7] = COF(1, 2) * invdet; inv[8] = COF(2, 2) * invdet;
#undef COF
}

// Hpl = w * Jp^T Jl (6x3) from the linearisation record
__device__ __forceinline__ void make_hpl(const double* __restrict__ rec, double Hpl[6][3]) {
    const double w = rec[2];
    const double* Jl = rec + 3;
    const double* Jp = rec + 9;
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) Hpl[a][b] = w * (Jp[a] * Jl[b] + Jp[6 + a] * Jl[3 + b]);
}

// ---- ba::LocalBA (Ceres twin): residual of CeresReprojectionError with forward-mode jets ---------------------------
// pose = [t; angle-axis], X = world point, (c0, c1) = normalised observation.  9 partials: 0..5 pose, 6..8 point --
// what ceres::AutoDiffCostFunction<CeresReprojectionError, 2, 6, 3> evaluates (reference
// include/ygz/Ceres/CeresReprojectionError.h:33-69, ceres/rotation.h AngleAxisRotatePoint).  The operation order
// follows oracle/ba.cpp so that the two agree to rounding.
struct Jet9 {
    double a;
    double v[9];
};
__device__ __forceinline__ Jet9 j9c(double c) {
    Jet9 r;
    r.a = c;
#pragma unroll
    for (int i = 0; i < 9; ++i) r.v[i] = 0.0;
    return r;
}
__device__ __forceinline__ Jet9 operator+(const Jet9& x, const Jet9& y) {
    Jet9 r;
    r.a = x.a + y.a;
#pragma unroll
    for (int i = 0; i < 9; ++i) r.v[i] = x.v[i] + y.v[i];
    return r;
}
__device__ __forceinline__ Jet9 operator-(const Jet9& x, const Jet9& y) {
    Jet9 r;
    r.a = x.a - y.a;
#pragma unroll
    for (int i = 0; i < 9; ++i) r.v[i] = x.v[i] - y.v[i];
    return r;
}
__device__ __forceinline__ Jet9 operator*(const Jet9& x, const Jet9& y) {
    Jet9 r;
    r.a = x.a * y.a;
#pragma unroll
    for (int i = 0; i < 9; ++i) r.v[i] = x.a * y.v[i] + x.v[i] * y.a;
    return r;
}
__device__ __forceinline__ Jet9 operator/(const Jet9& x, const Jet9& y) {
    const double inv = 1.0 / y.a, q = x.a * inv;
    Jet9 r;
    r.a = q;
#pragma unroll
    for (int i = 0; i < 9; ++i) r.v[i] = (x.v[i] - q * y.v[i]) * inv;
    return r;
}

// value only: p = AngleAxisRotatePoint(aa, X) + t
__device__ __forceinline__ void ceres_project(const double* __restrict__ pose, double X0, double X1, double X2, double p[3]) {
    const double a0 = pose[3], a1 = pose[4], a2 = pose[5];
    const double theta2 = a0 * a0 + a1 * a1 + a2 * a2;
    if (theta2 > 2.2204460492503131e-16) {
        const double theta = sqrt(theta2), costheta = cos(theta), sintheta = sin(theta), inv = 1.0 / theta;
        const double w0 = a0 * inv, w1 = a1 * inv, w2 = a2 * inv;
        const double c0 = w1 * X2 - w2 * X1, c1 = w2 * X0 - w0 * X2, c2 = w0 * X1 - w1 * X0;
        const double tmp = (w0 * X0 + w1 * X1 + w2 * X2) * (1.0 - costheta);
        p[0] = X0 * costheta + c0 * sintheta + w0 * tmp;
        p[1] = X1 * costheta + c1 * sintheta + w1 * tmp;
        p[2] = X2 * costheta + c2 * sintheta + w2 * tmp;
    } else {
        p[0] = X0 + (a1 * X2 - a2 * X1);
        p[1] = X1 + (a2 * X0 - a0 * X2);
        p[2] = X2 + (a0 * X1 - a1 * X0);
    }
    p[0] += pose[0];
    p[1] += pose[1];
    p[2] += pose[2];
}

// residual + Jacobians into a linearisation record: rec = e(2) w(=1) Jl(2x3) Jp(2x6)
__device__ __noinline__ void ceres_linearise(const double* __restrict__ pose, double X0, double X1, double X2, double c0, double c1,
                                             double* __restrict__ rec) {
    Jet9 T[6], Xj[3];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        T[i] = j9c(pose[i]);
        T[i].v[i] = 1.0;
    }
    Xj[0] = j9c(X0); Xj[1] = j9c(X1); Xj[2] = j9c(X2);
    Xj[0].v[6] = 1.0; Xj[1].v[7] = 1.0; Xj[2].v[8] = 1.0;
    Jet9 p[3];
    const Jet9 theta2 = T[3] * T[3] + T[4] * T[4] + T[5] * T[5];
    if (theta2.a > 2.2204460492503131e-16) {
        const double th = sqrt(theta2.a), dth = 1.0 / (2.0 * th);
        Jet9 theta, costheta, sintheta;
        theta.a = th; costheta.a = cos(th); sintheta.a = sin(th);
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            theta.v[i] = theta2.v[i] * dth;
            costheta.v[i] = -sintheta.a * theta.v[i];
            sintheta.v[i] = costheta.a * theta.v[i];
        }
        const Jet9 inv = j9c(1.0) / theta;
        const Jet9 w0 = T[3] * inv, w1 = T[4] * inv, w2 = T[5] * inv;
        const Jet9 x0 = w1 * Xj[2] - w2 * Xj[1], x1 = w2 * Xj[0] - w0 * Xj[2], x2 = w0 * Xj[1] - w1 * Xj[0];
        const Jet9 tmp = (w0 * Xj[0] + w1 * Xj[1] + w2 * Xj[2]) * (j9c(1.0) - costheta);
        p[0] = Xj[0] * costheta + x0 * sintheta + w0 * tmp;
        p[1] = Xj[1] * costheta + x1 * sintheta + w1 * tmp;
        p[2] = Xj[2] * costheta + x2 * sintheta + w2 * tmp;
    } else {
        p[0] = Xj[0] + (T[4] * Xj[2] - T[5] * Xj[1]);
        p[1] = Xj[1] + (T[5] * Xj[0] - T[3] * Xj[2]);
        p[2] = Xj[2] + (T[3] * Xj[1] - T[4] * Xj[0]);
    }
    p[0] = p[0] + T[0];
    p[1] = p[1] + T[1];
    p[2] = p[2] + T[2];
    const Jet9 r0 = j9c(c0) - p[0] / p[2], r1 = j9c(c1) - p[1] / p[2];
    rec[0] = r0.a; rec[1] = r1.a; rec[2] = 1.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        rec[3 + k] = r0.v[6 + k];
        rec[6 + k] = r1.v[6 + k];
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        rec[9 + k] = r0.v[k];
        rec[15 + k] = r1.v[k];
    }
}

// ---- local BA: one thread-block CLUSTER (kClusterSize CTAs on kClusterSize SMs) per problem ---------------------
// The observation / landmark / pair-entry loops stride over the whole cluster, the per-pose and per-block-pair sums
// are warp-reduced and combined with f64 global atomics (RED.ADD.F64) into a small L2-resident workspace, scalar
// reductions go through per-CTA partials + barrier.cluster, and CTA 0 factorises the reduced system in shared memory.
// Every CTA keeps its own replica of the poses and of the LM scalars and takes the same (deterministic) decisions.
constexpr int kClusterSize = 8;
constexpr int kMaxCluster = 16;           // non-portable cluster size (opt-in attribute)

struct ClusterWs {            // per problem, in global memory
    double red[4][kMaxCluster][4];
    double Hpp[kMaxFreePoses * 36];
    double bp[kMaxFreePoses * 6];
    double S[kMaxFreePoses * 6 * kMaxFreePoses * 6];
    double bs[kMaxFreePoses * 6];
    double xp[kMaxFreePoses * 6];
    int ok;
};

// ba::LocalBA (Ceres trust-region LM with Jacobi scaling, normalised residuals, optional per-block Huber loss, poses as
// [t; angle-axis] with additive updates): Schur complement with per-parameter damping
// d_k = clamp(s_k^2 H_kk, 1e-6, 1e32) / (radius s_k^2)
__global__ void __launch_bounds__(kBAThreads) local_ba_kernel(const BAArgs a, ClusterWs* __restrict__ ws_all) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ double s_mem[];          // CTA 0: S (dimp x dimp) + rhs
    __shared__ double s_tmp[33];
    __shared__ double s_pose[kMaxPoses][6];    // replica of the pose estimates [t; angle-axis]
    __shared__ double s_backup[kMaxPoses][6];
    __shared__ double s_xp[kMaxFreePoses * 6];
    __shared__ double s_sp[kMaxFreePoses * 6];   // Jacobi scaling of the pose columns
    __shared__ int s_free[kMaxPoses];
    __shared__ int s_np;

    const int rank = (int)cluster.block_rank(), C = (int)cluster.num_blocks();
    const int prob = blockIdx.x / C, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int T = kBAThreads, CT = C * T, ct = rank * T + tid;       // cluster-wide thread id
    const int GW = C * (T / 32), gw = rank * (T / 32) + warp;        // cluster-wide warp id
    ClusterWs& ws = ws_all[prob];
    const int k0 = a.kf_off[prob], n_kf = a.kf_off[prob + 1] - k0;
    const int p0 = a.pt_off[prob], n_pt = a.pt_off[prob + 1] - p0;
    const int o0 = a.obs_off[prob], n_obs = a.obs_off[prob + 1] - o0;
    if (tid == 0) {
        int nf = 0;
        for (int k = 0; k < n_kf; ++k) s_free[k] = a.fixed[k0 + k] ? -1 : nf++;
        s_np = nf;
    }
    if (tid < n_kf)
        for (int c = 0; c < 6; ++c) s_pose[tid][c] = a.poses[6 * (size_t)(k0 + tid) + c];
    __syncthreads();
    const int np = s_np, dimp = 6 * np;
    double* s_S = s_mem;
    double* s_bs = s_S + dimp * dimp;
    const double fx = a.fx, fy = a.fy, cx = a.cx, cy = a.cy;
    const double dsqr = a.huber_delta * a.huber_delta;
    const int32_t* pair_start = a.pair_start + a.pair_off[prob];
    const int n_pairs = np * (np + 1) / 2;
    int red_slot = 0;

    // cluster-wide sum of up to 2 values (identical result in every thread of every CTA); contains a cluster barrier
    auto cluster_sum2 = [&](double v0, double v1, double* out0, double* out1) {
        v0 = block_sum(v0, s_tmp);
        v1 = block_sum(v1, s_tmp);
        const int slot = red_slot;
        red_slot = (red_slot + 1) & 3;
        if (tid == 0) {
            ws.red[slot][rank][0] = v0;
            ws.red[slot][rank][1] = v1;
        }
        cluster.sync();
        double s0 = 0, s1 = 0;
        for (int r = 0; r < C; ++r) {
            s0 += __ldcg(&ws.red[slot][r][0]);
            s1 += __ldcg(&ws.red[slot][r][1]);
        }
        *out0 = s0;
        *out1 = s1;
    };
    auto reproject = [&](int o, double* e0, double* e1, double* px, double* py, double* pz) {
        const double* X = a.pts + 3 * (size_t)(p0 + a.pt_idx[o0 + o]);
        const double X0 = __ldcg(X), X1 = __ldcg(X + 1), X2 = __ldcg(X + 2);
        double p[3];
        ceres_project(s_pose[a.kf_idx[o0 + o]], X0, X1, X2, p);
        const double iz = 1.0 / p[2];
        // PinholeCamera::Pixel2Camera2D: float intrinsics, double maths
        *e0 = (a.obs[2 * (size_t)(o0 + o)] - cx) / fx - p[0] * iz;
        *e1 = (a.obs[2 * (size_t)(o0 + o) + 1] - cy) / fy - p[1] * iz;
        *px = p[0]; *py = p[1]; *pz = p[2];
    };
    // LM damping of one parameter from its Hessian diagonal and Jacobi scale
    double radius = 1e4, decrease_factor = 2.0;
    auto damp = [&](double hkk, double sk) { return fmin(fmax(sk * sk * hkk, 1e-6), 1e32) / radius / (sk * sk); };
    int term = 0, n_success = 0;   // termination code (see ygz_b200.h), accepted steps

    int trials_total = 0;
    double chi_first = 0, chi_last = 0, rho = 0, currentChi = 0;

    for (int iteration = 0; iteration < a.max_iters; ++iteration) {
        // ---- computeActiveErrors + buildSystem -------------------------------------------------------------------
        for (int i = ct; i < np * 36; i += CT) ws.Hpp[i] = 0.0;
        for (int i = ct; i < dimp; i += CT) ws.bp[i] = 0.0;
        double acc = 0;
        for (int o = ct; o < n_obs; o += CT) {
            const double* X = a.pts + 3 * (size_t)(p0 + a.pt_idx[o0 + o]);
            double* rec = a.lin + 21 * (size_t)(o0 + o);
            ceres_linearise(s_pose[a.kf_idx[o0 + o]], __ldcg(X), __ldcg(X + 1), __ldcg(X + 2),
                            (a.obs[2 * (size_t)(o0 + o)] - cx) / fx, (a.obs[2 * (size_t)(o0 + o) + 1] - cy) / fy, rec);
            // ceres::HuberLoss through the Corrector: rho'' <= 0, so the block is weighted by rho' = a / |r| beyond a
            const double e2 = rec[0] * rec[0] + rec[1] * rec[1];
            if (a.huber_delta > 0 && e2 > dsqr && (!a.loss_mask || a.loss_mask[o0 + o])) {
                const double rt = sqrt(e2);
                rec[2] = a.huber_delta / rt;
                acc += 2 * a.huber_delta * rt - dsqr;
            } else {
                acc += e2;
            }
        }
        double dummy;
        cluster_sum2(acc, 0.0, &currentChi, &dummy);   // (barrier: lin[] and the zeroed Hpp/bp are visible cluster-wide)
        if (iteration == 0) chi_first = currentChi;
        // Hll, bl : thread per landmark
        double mx = 0;
        for (int j = ct; j < n_pt; j += CT) {
            double H[6] = {0, 0, 0, 0, 0, 0}, b[3] = {0, 0, 0};
            for (int q = a.lm_start[p0 + j]; q < a.lm_start[p0 + j + 1]; ++q) {
                const double* rec = a.lin + 21 * (size_t)a.lm_obs[q];
                const double w = rec[2];
                const double* J0 = rec + 3;
                const double* J1 = rec + 6;
                H[0] += w * (J0[0] * J0[0] + J1[0] * J1[0]); H[1] += w * (J0[0] * J0[1] + J1[0] * J1[1]);
                H[2] += w * (J0[0] * J0[2] + J1[0] * J1[2]); H[3] += w * (J0[1] * J0[1] + J1[1] * J1[1]);
                H[4] += w * (J0[1] * J0[2] + J1[1] * J1[2]); H[5] += w * (J0[2] * J0[2] + J1[2] * J1[2]);
#pragma unroll
                for (int c = 0; c < 3; ++c) b[c] += -w * (J0[c] * rec[0] + J1[c] * rec[1]);
            }
            double* Hj = a.Hll + 9 * (size_t)(p0 + j);
            Hj[0] = H[0]; Hj[1] = H[1]; Hj[2] = H[2]; Hj[3] = H[1]; Hj[4] = H[3]; Hj[5] = H[4]; Hj[6] = H[2]; Hj[7] = H[4]; Hj[8] = H[5];
            double* bj = a.bl + 3 * (size_t)(p0 + j);
            bj[0] = b[0]; bj[1] = b[1]; bj[2] = b[2];
            mx = fmax(mx, fmax(fabs(b[0]), fmax(fabs(b[1]), fabs(b[2]))));   // gradient max norm
            if (iteration == 0) {  // Jacobi scaling from the initial Jacobian: 1 / (1 + ||column||)
                double* sj = a.scale_l + 3 * (size_t)(p0 + j);
                sj[0] = 1.0 / (1.0 + sqrt(H[0])); sj[1] = 1.0 / (1.0 + sqrt(H[3])); sj[2] = 1.0 / (1.0 + sqrt(H[5]));
            }
        }
        // Hpp, bp : (free pose, chunk) tasks over all warps of the cluster, f64 atomics into the workspace
        if (np > 0) {
            const int CH = max(1, GW / np);
            for (int task = gw; task < np * CH; task += GW) {
                const int fi = task % np, chunk = task / np;
                int k = 0;
                while (s_free[k] != fi) ++k;
                double h[21], g[6];
#pragma unroll
                for (int t = 0; t < 21; ++t) h[t] = 0;
#pragma unroll
                for (int t = 0; t < 6; ++t) g[t] = 0;
                for (int q = a.ps_start[k0 + k] + chunk * 32 + lane; q < a.ps_start[k0 + k + 1]; q += CH * 32) {
                    const double* rec = a.lin + 21 * (size_t)a.ps_obs[q];
                    const double w = rec[2];
                    const double* J0 = rec + 9;
                    const double* J1 = rec + 15;
                    int t = 0;
#pragma unroll
                    for (int r = 0; r < 6; ++r) {
#pragma unroll
                        for (int c = r; c < 6; ++c) h[t++] += w * (J0[r] * J0[c] + J1[r] * J1[c]);
                        g[r] += -w * (J0[r] * rec[0] + J1[r] * rec[1]);
                    }
                }
                int t = 0;
#pragma unroll
                for (int r = 0; r < 6; ++r) {
#pragma unroll
                    for (int c = r; c < 6; ++c) {
                        const double v = warp_sum(h[t++]);
                        if (lane == 0) {
                            atomicAdd(&ws.Hpp[fi * 36 + r * 6 + c], v);
                            if (c != r) atomicAdd(&ws.Hpp[fi * 36 + c * 6 + r], v);
                        }
                    }
                    const double gv = warp_sum(g[r]);
                    if (lane == 0) atomicAdd(&ws.bp[fi * 6 + r], gv);
                }
            }
        }
        {
            // gradient max norm: a max reduction through the partial slots of cluster_sum2
            const double bm = block_max(mx, s_tmp);
            const int slot = red_slot;
            red_slot = (red_slot + 1) & 3;
            if (tid == 0) ws.red[slot][rank][0] = bm;
            cluster.sync();                                   // also publishes Hll/bl and the Hpp/bp atomics
            double m0 = 0;
            for (int r = 0; r < C; ++r) m0 = fmax(m0, __ldcg(&ws.red[slot][r][0]));
            for (int i = 0; i < dimp; ++i) m0 = fmax(m0, fabs(__ldcg(&ws.bp[i])));
            if (iteration == 0) {
                if (tid < dimp) s_sp[tid] = 1.0 / (1.0 + sqrt(__ldcg(&ws.Hpp[(tid / 6) * 36 + (tid % 6) * 7])));
                __syncthreads();
            }
            if (m0 <= 1e-10) term = 1;   // gradient tolerance
        }
        if (term) break;

        do {
            // _optimizer->push(): pose replica in shared memory, landmarks per owner thread
            if (tid < n_kf)
                for (int c = 0; c < 6; ++c) s_backup[tid][c] = s_pose[tid][c];
            for (int j = ct; j < n_pt; j += CT) {
                double D[9];
                const double* Hj = a.Hll + 9 * (size_t)(p0 + j);
#pragma unroll
                for (int t = 0; t < 9; ++t) D[t] = Hj[t];
                const double* sj = a.scale_l + 3 * (size_t)(p0 + j);
                D[0] += damp(Hj[0], sj[0]); D[4] += damp(Hj[4], sj[1]); D[8] += damp(Hj[8], sj[2]);
                inverse3d(D, a.Dinv + 9 * (size_t)(p0 + j));
#pragma unroll
                for (int c = 0; c < 3; ++c) a.pts_backup[3 * (size_t)(p0 + j) + c] = a.pts[3 * (size_t)(p0 + j) + c];
            }
            for (int i = ct; i < dimp * dimp; i += CT) ws.S[i] = 0.0;
            for (int i = ct; i < dimp; i += CT) ws.bs[i] = 0.0;
            cluster.sync();
            // Schur complement: (block pair, chunk) tasks over all warps of the cluster
            if (n_pairs > 0) {
                const int CH = max(1, GW / n_pairs);
                for (int task = gw; task < n_pairs * CH; task += GW) {
                    const int pr = task % n_pairs, chunk = task / n_pairs;
                    int f1 = 0, rem = pr;
                    while (rem >= np - f1) {
                        rem -= np - f1;
                        ++f1;
                    }
                    const int f2 = f1 + rem;
                    double accS[36], accb[6];
#pragma unroll
                    for (int t = 0; t < 36; ++t) accS[t] = 0;
#pragma unroll
                    for (int t = 0; t < 6; ++t) accb[t] = 0;
                    for (int q = pair_start[pr] + chunk * 32 + lane; q < pair_start[pr + 1]; q += CH * 32) {
                        const int o1 = a.pair_o1[q], o2 = a.pair_o2[q];
                        const int j = p0 + a.pt_idx[o1];
                        const double* Di = a.Dinv + 9 * (size_t)j;
                        double H1[6][3], BD[6][3];
                        make_hpl(a.lin + 21 * (size_t)o1, H1);
#pragma unroll
                        for (int r = 0; r < 6; ++r)
#pragma unroll
                            for (int c = 0; c < 3; ++c) BD[r][c] = H1[r][0] * Di[c] + H1[r][1] * Di[3 + c] + H1[r][2] * Di[6 + c];
                        if (o1 == o2) {
                            const double* bj = a.bl + 3 * (size_t)j;
#pragma unroll
                            for (int r = 0; r < 6; ++r) accb[r] += BD[r][0] * bj[0] + BD[r][1] * bj[1] + BD[r][2] * bj[2];
#pragma unroll
                            for (int r = 0; r < 6; ++r)
#pragma unroll
                                for (int c = 0; c < 6; ++c) accS[r * 6 + c] += BD[r][0] * H1[c][0] + BD[r][1] * H1[c][1] + BD[r][2] * H1[c][2];
                        } else {
                            double H2[6][3];
                            make_hpl(a.lin + 21 * (size_t)o2, H2);
#pragma unroll
                            for (int r = 0; r < 6; ++r)
#pragma unroll
                                for (int c = 0; c < 6; ++c) accS[r * 6 + c] += BD[r][0] * H2[c][0] + BD[r][1] * H2[c][1] + BD[r][2] * H2[c][2];
                        }
                    }
#pragma unroll
                    for (int t = 0; t < 36; ++t) {
                        const double v = warp_sum(accS[t]);
                        if (lane == 0) {
                            const int r = t / 6, c = t - r * 6;
                            atomicAdd(&ws.S[(6 * f1 + r) * dimp + 6 * f2 + c], -v);
                            if (f1 != f2) atomicAdd(&ws.S[(6 * f2 + c) * dimp + 6 * f1 + r], -v);
                        }
                    }
                    if (f1 == f2) {
#pragma unroll
                        for (int r = 0; r < 6; ++r) {
                            const double v = warp_sum(accb[r]);
                            if (lane == 0) atomicAdd(&ws.bs[6 * f1 + r], -v);
                        }
                    }
                }
            }
            cluster.sync();
            // CTA 0: S = Hpp + D - sum, dense Cholesky in shared memory, triangular solves by warp 0
            if (rank == 0) {
                for (int i = tid; i < dimp * dimp; i += T) {
                    const int r = i / dimp, c = i - r * dimp;
                    double v = __ldcg(&ws.S[i]);
                    if (r / 6 == c / 6) {
                        const double h = __ldcg(&ws.Hpp[(r / 6) * 36 + (r % 6) * 6 + (c % 6)]);
                        v += h + (r == c ? damp(h, s_sp[r]) : 0.0);
                    }
                    s_S[i] = v;
                }
                if (tid < dimp) s_bs[tid] = __ldcg(&ws.bs[tid]) + __ldcg(&ws.bp[tid]);
                __shared__ int s_ok;
                if (tid == 0) s_ok = 1;
                __syncthreads();
                for (int j = 0; j < dimp; ++j) {
                    if (tid == 0) {
                        const double d = s_S[j * dimp + j];
                        if (!(d > 0)) s_ok = 0;
                        s_S[j * dimp + j] = sqrt(d);
                    }
                    __syncthreads();
                    if (!s_ok) break;
                    const double djj = s_S[j * dimp + j];
                    const int rem = dimp - j - 1;
                    // column scale fused into the trailing update: L(i,j) = S(i,j)/djj is recomputed by the readers
                    for (int e = tid; e < rem * rem; e += T) {
                        const int r = j + 1 + e / rem, c = j + 1 + e % rem;
                        if (c <= r) s_S[r * dimp + c] -= (s_S[r * dimp + j] / djj) * (s_S[c * dimp + j] / djj);
                    }
                    __syncthreads();
                    // column j is final after this scaling and is not read again before the solves
                    for (int i = j + 1 + tid; i < dimp; i += T) s_S[i * dimp + j] /= djj;
                }
                __syncthreads();
                if (s_ok && warp == 0) {
                    // forward then backward substitution, one row at a time, the dot product split over the lanes
                    for (int i = 0; i < dimp; ++i) {
                        double s = 0;
                        for (int k = lane; k < i; k += 32) s += s_S[i * dimp + k] * s_bs[k];
                        s = warp_sum(s);
                        if (lane == 0) s_bs[i] = (s_bs[i] - s) / s_S[i * dimp + i];
                        __syncwarp();
                    }
                    for (int i = dimp - 1; i >= 0; --i) {
                        double s = 0;
                        for (int k = i + 1 + lane; k < dimp; k += 32) s += s_S[k * dimp + i] * s_bs[k];
                        s = warp_sum(s);
                        if (lane == 0) s_bs[i] = (s_bs[i] - s) / s_S[i * dimp + i];
                        __syncwarp();
                    }
                }
                __syncthreads();
                if (tid < dimp) ws.xp[tid] = s_bs[tid];
                if (tid == 0) ws.ok = s_ok;
            }
            cluster.sync();
            const bool ok2 = __ldcg(&ws.ok) != 0;
            if (tid < dimp) s_xp[tid] = __ldcg(&ws.xp[tid]);
            __syncthreads();
            // landmark back-substitution + update (owner thread), pose update (replicated), scale term
            double scale = 0, xnorm2 = 0;
            for (int j = ct; j < n_pt; j += CT) {
                const double* bj = a.bl + 3 * (size_t)(p0 + j);
                double r[3] = {bj[0], bj[1], bj[2]};
                for (int q = a.lm_start[p0 + j]; q < a.lm_start[p0 + j + 1]; ++q) {
                    const int o = a.lm_obs[q];
                    const int fi = s_free[a.kf_idx[o]];
                    if (fi < 0) continue;
                    double H1[6][3];
                    make_hpl(a.lin + 21 * (size_t)o, H1);
#pragma unroll
                    for (int c = 0; c < 3; ++c)
#pragma unroll
                        for (int rr = 0; rr < 6; ++rr) r[c] -= H1[rr][c] * s_xp[6 * fi + rr];
                }
                const double* Di = a.Dinv + 9 * (size_t)(p0 + j);
                double* X = a.pts + 3 * (size_t)(p0 + j);
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const double x = Di[3 * c] * r[0] + Di[3 * c + 1] * r[1] + Di[3 * c + 2] * r[2];
                    a.xl[3 * (size_t)(p0 + j) + c] = x;   // the model cost change needs J delta per observation
                    scale += x * x;                      // |step|^2
                    xnorm2 += X[c] * X[c];
                    X[c] += x;
                }
            }
            if (rank == 0 && tid < n_kf && s_free[tid] >= 0) {
                const double* u = s_xp + 6 * s_free[tid];
#pragma unroll
                for (int c = 0; c < 6; ++c) {
                    scale += u[c] * u[c];
                    xnorm2 += s_pose[tid][c] * s_pose[tid][c];
                }
            }
            if (tid < n_kf && s_free[tid] >= 0) {  // plain Euclidean parameter block: x + delta
                const double* u = s_xp + 6 * s_free[tid];
#pragma unroll
                for (int c = 0; c < 6; ++c) s_pose[tid][c] += u[c];
            }
            __syncthreads();
            double step2, x2;
            cluster_sum2(scale, xnorm2, &step2, &x2);   // (barrier: updated landmarks and xl visible cluster-wide)
            // candidate cost and model cost change -(J delta)^T (r + J delta / 2), one pass over the observations
            double newc = 0, model = 0;
            for (int o = ct; o < n_obs; o += CT) {
                double e0, e1, x, y, z;
                reproject(o, &e0, &e1, &x, &y, &z);
                const double e2n = e0 * e0 + e1 * e1;
                newc += (a.huber_delta > 0 && e2n > dsqr && (!a.loss_mask || a.loss_mask[o0 + o])) ? 2 * a.huber_delta * sqrt(e2n) - dsqr : e2n;
                const double* rec = a.lin + 21 * (size_t)(o0 + o);
                const int fi = s_free[a.kf_idx[o0 + o]];
                const double* dl = a.xl + 3 * (size_t)(p0 + a.pt_idx[o0 + o]);
                const double d0 = __ldcg(dl), d1 = __ldcg(dl + 1), d2 = __ldcg(dl + 2);
#pragma unroll
                for (int row = 0; row < 2; ++row) {
                    double jy = 0;
                    if (fi >= 0) {
#pragma unroll
                        for (int k = 0; k < 6; ++k) jy += rec[9 + 6 * row + k] * s_xp[6 * fi + k];
                    }
                    jy += rec[3 + 3 * row] * d0;
                    jy += rec[4 + 3 * row] * d1;
                    jy += rec[5 + 3 * row] * d2;
                    model -= rec[2] * jy * (rec[row] + jy / 2);
                }
            }
            double newc_tot, model_tot;
            cluster_sum2(newc, model, &newc_tot, &model_tot);
            const double cost = 0.5 * currentChi, new_cost = 0.5 * newc_tot;
            bool accepted = false;
            double relative_decrease = 0;
            if (ok2 && model_tot > 0) {
                relative_decrease = (cost - new_cost) / model_tot;
                accepted = relative_decrease > 1e-3;
            }
            bool accept = accepted;
            if (accepted) {
                if (sqrt(step2) <= 1e-8 * (sqrt(x2) + 1e-8)) {  // parameter tolerance: checked before the step is taken
                    term = 2;
                    accept = false;
                } else {
                    ++n_success;
                    currentChi = newc_tot;
                    if (fabs(cost - new_cost) <= 1e-6 * cost) {
                        term = 3;   // function tolerance
                    } else {
                        const double t3 = 2.0 * relative_decrease - 1.0;
                        radius = radius / fmax(1.0 / 3.0, 1.0 - t3 * t3 * t3);
                        radius = fmin(1e16, radius);
                        decrease_factor = 2.0;
                    }
                }
            } else {
                radius = radius / decrease_factor;
                decrease_factor *= 2.0;
                if (radius < 1e-32) term = 4;
            }
            rho = accepted ? 1.0 : -1.0;
            if (!accept) {  // _optimizer->pop()
                if (tid < n_kf)
                    for (int c = 0; c < 6; ++c) s_pose[tid][c] = s_backup[tid][c];
                for (int j = ct; j < n_pt; j += CT)
#pragma unroll
                    for (int c = 0; c < 3; ++c) a.pts[3 * (size_t)(p0 + j) + c] = a.pts_backup[3 * (size_t)(p0 + j) + c];
                __syncthreads();
            }
            ++trials_total;
        } while (rho < 0 && !term && trials_total < a.max_iters);
        chi_last = currentChi;
        if (term || trials_total >= a.max_iters) break;
    }
    if (rank == 0) {
        if (tid < n_kf)
            for (int c = 0; c < 6; ++c) a.poses[6 * (size_t)(k0 + tid) + c] = s_pose[tid][c];
        if (tid == 0) {
            double* st = a.stats + 8 * (size_t)prob;
            st[0] = trials_total; st[1] = n_success; st[2] = 0.5 * chi_first; st[3] = 0.5 * chi_last; st[4] = radius; st[5] = term;
            st[6] = 0.0; st[7] = 0.0;   // (unused by this kernel; the host copies all 8 slots)
        }
    }
}

// ---- pose-only refinement ----------------------------------------------------------------------------------
// value + partials with respect to the angle-axis only: the rotation of the pose, differentiated ONCE per evaluation instead
// of once per point (round 1's six-partial jets spent two thirds of the kernel's FP64 instructions re-deriving it per point)
struct Jet3 {
    double a;
    double v[3];
};
__device__ __forceinline__ Jet3 j3c(double c) { return Jet3{c, {0, 0, 0}}; }
__device__ __forceinline__ Jet3 operator+(const Jet3& x, const Jet3& y) { return Jet3{x.a + y.a, {x.v[0] + y.v[0], x.v[1] + y.v[1], x.v[2] + y.v[2]}}; }
__device__ __forceinline__ Jet3 operator-(const Jet3& x, const Jet3& y) { return Jet3{x.a - y.a, {x.v[0] - y.v[0], x.v[1] - y.v[1], x.v[2] - y.v[2]}}; }
__device__ __forceinline__ Jet3 operator*(const Jet3& x, const Jet3& y) {
    return Jet3{x.a * y.a, {x.a * y.v[0] + x.v[0] * y.a, x.a * y.v[1] + x.v[1] * y.a, x.a * y.v[2] + x.v[2] * y.a}};
}
__device__ __forceinline__ Jet3 operator/(const Jet3& x, const Jet3& y) {
    const double inv = 1.0 / y.a, q = x.a * inv;
    return Jet3{q, {(x.v[0] - q * y.v[0]) * inv, (x.v[1] - q * y.v[1]) * inv, (x.v[2] - q * y.v[2]) * inv}};
}

// column k of R(angle-axis) and of dR/d(angle-axis): ceres::AngleAxisRotatePoint (both branches) applied to the basis vector e_k
__device__ void rotate_basis(const double aa[3], int k, double col[3], double dcol[3][3]) {
    Jet3 P[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        P[i] = j3c(aa[i]);
        P[i].v[i] = 1.0;
    }
    const Jet3 pt[3] = {j3c(k == 0 ? 1.0 : 0.0), j3c(k == 1 ? 1.0 : 0.0), j3c(k == 2 ? 1.0 : 0.0)};
    const Jet3 theta2 = P[0] * P[0] + P[1] * P[1] + P[2] * P[2];
    Jet3 out[3];
    if (theta2.a > 2.2204460492503131e-16) {
        Jet3 theta, costheta, sintheta;
        const double s = sqrt(theta2.a), d = 1.0 / (2.0 * s);
        theta.a = s;
        const double c = cos(s), sn = sin(s);
        costheta.a = c;
        sintheta.a = sn;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            theta.v[i] = theta2.v[i] * d;
            costheta.v[i] = -sn * theta.v[i];
            sintheta.v[i] = c * theta.v[i];
        }
        const Jet3 inv = j3c(1.0) / theta;
        const Jet3 w[3] = {P[0] * inv, P[1] * inv, P[2] * inv};
        const Jet3 wxp[3] = {w[1] * pt[2] - w[2] * pt[1], w[2] * pt[0] - w[0] * pt[2], w[0] * pt[1] - w[1] * pt[0]};
        const Jet3 tmp = (w[0] * pt[0] + w[1] * pt[1] + w[2] * pt[2]) * (j3c(1.0) - costheta);
#pragma unroll
        for (int i = 0; i < 3; ++i) out[i] = pt[i] * costheta + wxp[i] * sintheta + w[i] * tmp;
    } else {
        const Jet3 wxp[3] = {P[1] * pt[2] - P[2] * pt[1], P[2] * pt[0] - P[0] * pt[2], P[0] * pt[1] - P[1] * pt[0]};
#pragma unroll
        for (int i = 0; i < 3; ++i) out[i] = pt[i] + wxp[i];
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        col[i] = out[i].a;
#pragma unroll
        for (int m = 0; m < 3; ++m) dcol[i][m] = out[i].v[m];
    }
}

struct PoseOnlyArgs {
    const int32_t* offsets;   // per problem range of points
    const int32_t* counts;    // optional: points of problem p (default offsets[p + 1] - offsets[p])
    const double* pw;         // [total][3]
    const double* px;         // [total][2]
    double* T_cw;             // [n_problems][12] in/out
    uint8_t* inlier;          // [total]
    double* depth;            // [total]
    int32_t* n_inlier;        // [n_problems]
    uint8_t* enable;          // scratch [total]
    double* ws;               // (unused since the partial sums travel through distributed shared memory; kept for the scratch layout)
    float fx, fy, cx, cy;
    int stage_k;              // points per thread the dynamic shared memory can stage (0: read the points from global memory)
};

// One 8-CTA cluster per frame: the forward-mode jets are FP64 and a single SM's FP64 pipe bounded the one-CTA version.
// The points are strided over the cluster; every reduction publishes per-CTA partials, meets at barrier.cluster and is
// summed in rank order by every CTA, so all CTAs take identical trust-region decisions on their replica of the pose.
constexpr int kPoseThreads = 256;
constexpr int kPoseCluster = 8;
constexpr int kPoseRed = 32;

// A y = b for the 6 x 6 SPD system of a trust-region step (b in y on entry): LDL^T with one reciprocal per pivot instead of the
// square roots and 33 divisions of a textbook Cholesky -- every thread runs this between two reductions, so its dependent chain
// is on the critical path of every LM iteration.  false if a pivot is not positive (Ceres: the linear solver failed).
__device__ bool cholesky6(double A[36], double y[6]) {
    double rd[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        double d = A[j * 6 + j];
#pragma unroll
        for (int k = 0; k < j; ++k) d -= A[j * 6 + k] * A[j * 6 + k] * A[k * 6 + k];
        if (!(d > 0)) return false;
        A[j * 6 + j] = d;
        rd[j] = 1.0 / d;
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            double s = A[i * 6 + j];
#pragma unroll
            for (int k = 0; k < j; ++k) s -= A[i * 6 + k] * A[j * 6 + k] * A[k * 6 + k];
            A[i * 6 + j] = s * rd[j];
        }
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        double s = y[i];
#pragma unroll
        for (int k = 0; k < i; ++k) s -= A[i * 6 + k] * y[k];
        y[i] = s;
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) y[i] *= rd[i];
#pragma unroll
    for (int i = 5; i >= 0; --i) {
        double s = y[i];
#pragma unroll
        for (int k = i + 1; k < 6; ++k) s -= A[k * 6 + i] * y[k];
        y[i] = s;
    }
    return true;
}

__global__ void __launch_bounds__(kPoseThreads) pose_only_kernel(const PoseOnlyArgs a) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ double s_pts[];                        // staged points: [(k * 5 + c) * kPoseThreads + tid], c = X Y Z u_n v_n
    __shared__ double s_red[kPoseThreads / 32][kPoseRed];
    __shared__ double s_pub[4][kPoseRed];                    // this CTA's partial sums of the last four reductions (read by the peers)
    __shared__ double s_pose[6], s_cand[6], s_scale[6], s_sum[kPoseRed];
    __shared__ double s_R[9], s_dR[27], s_Rpose[6];          // rotation (row major), dR[3 * (3 j + k) + m] = d R_jk / d aa_m, and their pose
    const int rank = (int)cluster.block_rank(), C = (int)cluster.num_blocks();
    const int prob = blockIdx.x / C, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int CT = C * kPoseThreads, ct = rank * kPoseThreads + tid;   // cluster-wide thread id
    const int i0 = a.offsets[prob], n = a.counts ? a.counts[prob] : a.offsets[prob + 1] - i0;
    const double fx = a.fx, fy = a.fy, cx = a.cx, cy = a.cy;
    const int K = (n + CT - 1) / CT;                         // points per thread: i = ct + k * CT
    const bool staged = K <= a.stage_k && K <= 32;
    unsigned en_mask = 0;                                    // (staged) enable flag of this thread's k-th point
    int slot = 0;

    // cluster-wide sums of the per-thread partials `part[0 .. cnt)` into s_sum (identical in every thread of every CTA afterwards):
    // warp level, CTA level through shared memory, cluster level through distributed shared memory (one cluster barrier)
    auto finish_reduce = [&](int cnt) {
        __syncthreads();
        if (tid < cnt) {
            double s = 0;
            for (int w = 0; w < kPoseThreads / 32; ++w) s += s_red[w][tid];
            s_pub[slot][tid] = s;
        }
        cluster.sync();
        if (tid < cnt) {
            double s = 0;
            for (int r = 0; r < C; ++r) s += cluster.map_shared_rank(&s_pub[slot][0], r)[tid];
            s_sum[tid] = s;
        }
        slot = (slot + 1) & 3;
        __syncthreads();
    };
    auto reduce_few = [&](const double* part, int cnt) {
        for (int t = 0; t < cnt; ++t) {
            const double v = warp_sum(part[t]);
            if (lane == 0) s_red[warp][t] = v;
        }
        finish_reduce(cnt);
    };
    auto reduce32 = [&](double* part) {   // 32 values: a reduce-scatter butterfly, lane l ends with the warp total of part[l]
        int off = 16;
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1, off >>= 1) {
            const bool up = (lane & off) != 0;
#pragma unroll
            for (int i = 0; i < m; ++i) {
                const double keep = up ? part[i + m] : part[i];
                const double send = up ? part[i] : part[i + m];
                part[i] = keep + __shfl_xor_sync(0xFFFFFFFFu, send, off);
            }
        }
        s_red[warp][lane] = part[0];
        finish_reduce(32);
    };
    // R(aa) and dR / d aa of `pose` into shared memory (three threads, a column each); skipped when they are already there
    auto rotation_of = [&](const double* pose) {
        bool same = true;
        for (int k = 0; k < 6; ++k) same = same && s_Rpose[k] == pose[k];
        if (same) return;   // (uniform: shared memory values)
        __syncthreads();
        if (tid < 3) {
            double col[3], dcol[3][3];
            const double aa[3] = {pose[3], pose[4], pose[5]};
            rotate_basis(aa, tid, col, dcol);
            for (int j = 0; j < 3; ++j) {
                s_R[3 * j + tid] = col[j];
                for (int m = 0; m < 3; ++m) s_dR[3 * (3 * j + tid) + m] = dcol[j][m];
            }
        }
        if (tid >= 32 && tid < 38) s_Rpose[tid - 32] = pose[tid - 32];
        __syncthreads();
    };
    auto point = [&](int k, double* X, double* o) {   // world point and normalised observation of this thread's k-th point
        if (staged) {
#pragma unroll
            for (int c = 0; c < 3; ++c) X[c] = s_pts[(k * 5 + c) * kPoseThreads + tid];
            o[0] = s_pts[(k * 5 + 3) * kPoseThreads + tid];
            o[1] = s_pts[(k * 5 + 4) * kPoseThreads + tid];
        } else {
            const size_t i = (size_t)(i0 + ct + k * CT);
#pragma unroll
            for (int c = 0; c < 3; ++c) X[c] = a.pw[3 * i + c];
            o[0] = (a.px[2 * i] - cx) / fx;
            o[1] = (a.px[2 * i + 1] - cy) / fy;
        }
    };
    auto enabled = [&](int k) { return staged ? (en_mask >> k & 1u) != 0 : a.enable[i0 + ct + k * CT] != 0; };
    // J^T J (21), J^T r (6), cost (27), failed blocks (28) at `pose`: the derivative of ceres' angle-axis residual, with the rotation
    // differentiated once (rotation_of) and pushed through the projection analytically
    auto eval_normal = [&](const double* pose) {
        rotation_of(pose);
        double part[32];
#pragma unroll
        for (int t = 0; t < 32; ++t) part[t] = 0;
        const double t0 = pose[0], t1 = pose[1], t2 = pose[2];
        for (int k = 0; k < K; ++k) {
            if (ct + k * CT >= n || !enabled(k)) continue;
            double X[3], o[2];
            point(k, X, o);
            const double p2 = s_R[6] * X[0] + s_R[7] * X[1] + s_R[8] * X[2] + t2;
            if (p2 < 0) {
                part[28] += 1;
                continue;
            }
            const double p0 = s_R[0] * X[0] + s_R[1] * X[1] + s_R[2] * X[2] + t0, p1 = s_R[3] * X[0] + s_R[4] * X[1] + s_R[5] * X[2] + t1;
            const double inv = 1.0 / p2, q0 = p0 * inv, q1 = p1 * inv, r0 = o[0] - q0, r1 = o[1] - q1;
            double dp[3][3];   // d p_j / d aa_m
#pragma unroll
            for (int j = 0; j < 3; ++j)
#pragma unroll
                for (int m = 0; m < 3; ++m)
                    dp[j][m] = s_dR[3 * (3 * j) + m] * X[0] + s_dR[3 * (3 * j + 1) + m] * X[1] + s_dR[3 * (3 * j + 2) + m] * X[2];
            // residual = observation - p / p_z: d r0 = -(d p0 - q0 d p2) / p_z
            double j0[6], j1[6];
            j0[0] = -inv; j0[1] = 0.0; j0[2] = q0 * inv;
            j1[0] = 0.0; j1[1] = -inv; j1[2] = q1 * inv;
#pragma unroll
            for (int m = 0; m < 3; ++m) {
                j0[3 + m] = -(dp[0][m] - q0 * dp[2][m]) * inv;
                j1[3 + m] = -(dp[1][m] - q1 * dp[2][m]) * inv;
            }
            int t = 0;
#pragma unroll
            for (int r = 0; r < 6; ++r) {
#pragma unroll
                for (int c = r; c < 6; ++c) part[t++] += j0[r] * j0[c] + j1[r] * j1[c];
            }
#pragma unroll
            for (int q = 0; q < 6; ++q) part[21 + q] += j0[q] * r0 + j1[q] * r1;
            part[27] += r0 * r0 + r1 * r1;
        }
        reduce32(part);
    };

    // initial pose = [t; so3.log()]
    SE3d T = se3_from_mat(a.T_cw + 12 * (size_t)prob);
    double backup[6];
    {
        double th;
        const V3d rl = so3_log(T.q, &th);
        backup[0] = T.t.x; backup[1] = T.t.y; backup[2] = T.t.z; backup[3] = rl.x; backup[4] = rl.y; backup[5] = rl.z;
    }
    for (int k = 0; k < K; ++k) {   // (per-point flags are written and later read by the same thread)
        const int i = ct + k * CT;
        if (i >= n) break;
        a.enable[i0 + i] = 1;
        a.inlier[i0 + i] = 1;
        a.depth[i0 + i] = -1;
        if (staged) {
            en_mask |= 1u << k;
#pragma unroll
            for (int c = 0; c < 3; ++c) s_pts[(k * 5 + c) * kPoseThreads + tid] = a.pw[3 * (size_t)(i0 + i) + c];
            s_pts[(k * 5 + 3) * kPoseThreads + tid] = (a.px[2 * (size_t)(i0 + i)] - cx) / fx;
            s_pts[(k * 5 + 4) * kPoseThreads + tid] = (a.px[2 * (size_t)(i0 + i) + 1] - cy) / fy;
        }
    }
    if (tid < 6) s_Rpose[tid] = __longlong_as_double(0x7FF8000000000000LL);   // NaN: no rotation cached yet
    __syncthreads();
    int cntInlier = 0;
    for (int round = 0; round < 4; ++round) {
        if (tid < 6) s_pose[tid] = backup[tid];
        __syncthreads();
        // ---- Ceres trust-region LM (default options) ----
        eval_normal(s_pose);
        bool run = !(s_sum[28] > 0);
        double cost = 0.5 * s_sum[27];
        if (run) {
            if (tid < 6) {
                // diagonal index of column tid in the packed upper triangle
                int t = 0;
                for (int r = 0; r < tid; ++r) t += 6 - r;
                s_scale[tid] = 1.0 / (1.0 + sqrt(s_sum[t]));
            }
            double gmax = 0;
            for (int k = 0; k < 6; ++k) gmax = fmax(gmax, fabs(s_sum[21 + k]));
            if (gmax <= 1e-10) run = false;
        }
        __syncthreads();
        double radius = 1e4, decrease_factor = 2.0;
        // unscaled normal equations J^T J / J^T r at the current point (s_sum holds them after eval_normal(.., false)); the Jacobi
        // scaled system Ceres solves is D J^T J D / D J^T r, formed here from the same sums instead of a second pass over the points
        double U[27];
        for (int t = 0; t < 27; ++t) U[t] = s_sum[t];
        __syncthreads();
        for (int iter = 0; run && iter < 50; ++iter) {
            double A[36], g[6], y[6];
            {
                int t = 0;
                for (int r = 0; r < 6; ++r)
                    for (int c = r; c < 6; ++c) {
                        A[r * 6 + c] = A[c * 6 + r] = U[t++] * s_scale[r] * s_scale[c];
                    }
                for (int k = 0; k < 6; ++k) g[k] = U[21 + k] * s_scale[k];
            }
            double An[36];
            for (int t = 0; t < 36; ++t) An[t] = A[t];
            for (int k = 0; k < 6; ++k) {
                const double d = fmin(fmax(A[k * 6 + k], 1e-6), 1e32);
                An[k * 6 + k] += d / radius;
                y[k] = -g[k];
            }
            bool step_ok = cholesky6(An, y);
            double model_cost_change = 0;
            if (step_ok) {
                // -(Js y)^T (r + Js y / 2) = -(y^T g) - y^T A y / 2
                double yg = 0, yAy = 0;
                for (int r = 0; r < 6; ++r) {
                    yg += y[r] * g[r];
                    double s = 0;
                    for (int c = 0; c < 6; ++c) s += A[r * 6 + c] * y[c];
                    yAy += y[r] * s;
                }
                model_cost_change = -yg - 0.5 * yAy;
                step_ok = model_cost_change > 0;
            }
            bool accepted = false;
            if (step_ok) {  // uniform across the CTA: every thread computed the same numbers from s_sum
                double step_norm = 0, x_norm = 0;
                if (tid < 6) s_cand[tid] = s_pose[tid] + y[tid] * s_scale[tid];
                for (int k = 0; k < 6; ++k) {
                    const double d = y[k] * s_scale[k];
                    step_norm += d * d;
                    x_norm += s_pose[k] * s_pose[k];
                }
                step_norm = sqrt(step_norm);
                x_norm = sqrt(x_norm);
                __syncthreads();
                // ONE pass at the candidate: its cost decides the step, and if the step is accepted the same sums are the normal
                // equations of the next iteration (a rejected step wastes the Jacobian part of the pass, not a second reduction)
                eval_normal(s_cand);
                const double new_cost = 0.5 * s_sum[27];
                if (!(s_sum[28] > 0)) {
                    const double relative_decrease = (cost - new_cost) / model_cost_change;
                    if (relative_decrease > 1e-3) {
                        accepted = true;
                        if (step_norm <= 1e-8 * (x_norm + 1e-8)) break;  // parameter tolerance: stop before taking the step
                        const double cost_change = cost - new_cost;
                        __syncthreads();
                        if (tid < 6) s_pose[tid] = s_cand[tid];
                        __syncthreads();
                        const double old_cost = cost;
                        cost = new_cost;
                        if (fabs(cost_change) <= 1e-6 * old_cost) break;  // function tolerance
                        double gmax = 0;
                        for (int k = 0; k < 6; ++k) gmax = fmax(gmax, fabs(s_sum[21 + k]));
                        for (int t = 0; t < 27; ++t) U[t] = s_sum[t];
                        __syncthreads();
                        if (gmax <= 1e-10) break;                         // gradient tolerance
                        radius = radius / fmax(1.0 / 3.0, 1.0 - pow(2.0 * relative_decrease - 1.0, 3));
                        radius = fmin(1e16, radius);
                        decrease_factor = 2.0;
                    }
                }
            }
            if (!accepted) {
                radius = radius / decrease_factor;
                decrease_factor *= 2.0;
                if (radius < 1e-32) break;
            }
            __syncthreads();
        }
        __syncthreads();
        // ---- classification with the pose of the PREVIOUS round (BA.cpp:231-251) ----
        double cnt = 0;
        for (int k = 0; k < K; ++k) {
            const int i = ct + k * CT;
            if (i >= n) break;
            const double* X = a.pw + 3 * (size_t)(i0 + i);
            const V3d pc = transform(T, V3d{X[0], X[1], X[2]});
            const double u = fx * pc.x / pc.z + cx, v = fy * pc.y / pc.z + cy;
            const double dx = u - a.px[2 * (size_t)(i0 + i)], dy = v - a.px[2 * (size_t)(i0 + i) + 1];
            const double error2 = dx * dx + dy * dy;
            if (error2 > (double)5.991f) {
                a.inlier[i0 + i] = 0;
                a.enable[i0 + i] = 0;
                en_mask &= ~(1u << (k & 31));
            } else {
                a.depth[i0 + i] = pc.z;
                a.inlier[i0 + i] = 1;
                a.enable[i0 + i] = 1;
                en_mask |= 1u << (k & 31);
                cnt += 1;
            }
        }
        reduce_few(&cnt, 1);
        cntInlier = (int)s_sum[0];
        if (cntInlier < 10) break;
        double th;
        T.q = so3_exp(V3d{s_pose[3], s_pose[4], s_pose[5]}, &th);
        T.t = V3d{s_pose[0], s_pose[1], s_pose[2]};
        __syncthreads();
    }
    cluster.sync();   // no CTA may exit while another still reads its partials
    if (rank == 0 && tid == 0) {
        se3_to_mat(T, a.T_cw + 12 * (size_t)prob);
        a.n_inlier[prob] = cntInlier;
    }
}

}  // namespace

size_t pose_only_ws_doubles(int n_problems) { return (size_t)n_problems * 4 * kPoseCluster * kPoseRed; }

// ba::OptimizeCurrentPoseOnly on device-resident problems (the tracking engine): problem p owns points
// [d_offsets[p], d_offsets[p] + d_counts[p]); cluster = CTAs per problem (1, 2, 4 or 8)
// points per thread the kernel may stage in shared memory for problems of at most max_points points on `cluster` CTAs
// (0 = more than fits: the kernel then reads the points from global memory); sets the kernel's shared-memory opt-in once
static int pose_only_stage_k(int max_points, int cluster) {
    static std::once_flag once;
    static int max_k = 0;
    std::call_once(once, [] {
        int dev = 0, optin = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        const int budget = std::max(0, optin - 8 * 1024);   // the kernel's static arrays use ~4 KB
        cudaFuncSetAttribute(pose_only_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, budget);
        max_k = std::min(32, budget / (int)(5 * kPoseThreads * sizeof(double)));
    });
    const int k = (std::max(max_points, 1) + cluster * kPoseThreads - 1) / (cluster * kPoseThreads);
    return k <= max_k ? k : 0;
}

int launch_pose_only_dev(ygzb_ctx* ctx, int n_problems, const int32_t* d_offsets, const int32_t* d_counts, const double* d_pw,
                         const double* d_px, double* d_T_cw, uint8_t* d_inlier, double* d_depth, int32_t* d_n_inlier, uint8_t* d_enable,
                         double* d_ws, int cluster, int max_points) {
    if (n_problems <= 0) return YGZB_OK;
    PoseOnlyArgs a;
    a.offsets = d_offsets; a.counts = d_counts; a.pw = d_pw; a.px = d_px; a.T_cw = d_T_cw; a.inlier = d_inlier; a.depth = d_depth;
    a.n_inlier = d_n_inlier; a.enable = d_enable; a.ws = d_ws;
    a.fx = ctx->prm.fx; a.fy = ctx->prm.fy; a.cx = ctx->prm.cx; a.cy = ctx->prm.cy;
    cluster = std::max(1, std::min(cluster, kPoseCluster));
    a.stage_k = pose_only_stage_k(max_points, cluster);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(n_problems * cluster));
    cfg.blockDim = dim3(kPoseThreads);
    cfg.dynamicSmemBytes = (size_t)a.stage_k * 5 * kPoseThreads * sizeof(double);
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    ProfScope ps(ctx, kStagePoseOnly);
    YGZB_CUDA(ctx, cudaLaunchKernelEx(&cfg, pose_only_kernel, a));
    YGZB_LAUNCHED(ctx);
    return YGZB_OK;
}

}  // namespace ygzb

// ---- extern "C" entry points (marshalling + index bookkeeping only) ---------------------------------------
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
#define TRY(x)                          \
    do {                                \
        int _rc = (x);                  \
        if (_rc != YGZB_OK) return _rc; \
    } while (0)
}  // namespace

extern "C" {

void ygzb_default_ba_params(ygzb_ba_params* p) {
    p->max_iters = 20;        // optimizer.optimize(20), BA.cpp:502
    p->huber_delta = 5.991;   // rk->setDelta(5.991), BA.cpp:451
    p->chi2_outlier = 5.991;  // BA.cpp:508
    p->tau = 1e-5;            // g2o OptimizationAlgorithmLevenberg
    p->max_trials = 10;
}

}  // extern "C"

namespace {
// ba::LocalBAG2O through the second-generation kernel (ba2.cu): validation and ONE staged host-to-device copy here, the
// landmark-major observation lists and everything else on the device
int run_local_ba2(ygzb_ctx* ctx, int n_problems, const int32_t* kf_off, const int32_t* pt_off, const int32_t* obs_off, double* poses,
                  const uint8_t* fixed, double* pts, const int32_t* kf_idx, const int32_t* pt_idx, const double* obs_px,
                  const ygzb_ba_params* prm, uint8_t* outlier, std::vector<double>& hst) {
    const size_t P = (size_t)n_problems, NK = (size_t)kf_off[n_problems], NP = (size_t)pt_off[n_problems], NO = (size_t)obs_off[n_problems];
    BA2Problem in{};
    in.n_problems = n_problems;
    for (size_t p = 0; p < P; ++p) {
        const int k0 = kf_off[p], nk = kf_off[p + 1] - k0, npt = pt_off[p + 1] - pt_off[p], o0 = obs_off[p], no = obs_off[p + 1] - o0;
        if (nk < 1 || nk > kBA2MaxPoses) return set_error(ctx, YGZB_ERR_INVALID, "problem %zu: %d poses (1..%d supported)", p, nk, kBA2MaxPoses);
        int nf = 0;
        for (int k = 0; k < nk; ++k) nf += fixed[k0 + k] ? 0 : 1;
        if (nf > kBA2MaxFree) return set_error(ctx, YGZB_ERR_INVALID, "problem %zu: %d free poses (max %d)", p, nf, kBA2MaxFree);
        for (int o = 0; o < no; ++o)
            if (kf_idx[o0 + o] < 0 || kf_idx[o0 + o] >= nk || pt_idx[o0 + o] < 0 || pt_idx[o0 + o] >= npt)
                return set_error(ctx, YGZB_ERR_INVALID, "observation %d: index out of range", o0 + o);
        in.max_free = std::max(in.max_free, nf);
        in.max_kf = std::max(in.max_kf, nk);
        in.max_pts = std::max(in.max_pts, (size_t)npt);
        in.max_obs = std::max(in.max_obs, (size_t)no);
    }
    in.total_pts = NP;
    in.total_obs = NO;
    Carver sz(nullptr);
    sz.take<int32_t>(3 * (P + 1)); sz.take<double>(6 * NK); sz.take<uint8_t>(NK); sz.take<double>(3 * NP); sz.take<int32_t>(2 * NO);
    sz.take<double>(2 * NO);
    const size_t in_span = sz.bytes();
    void* buf = dev_scratch(ctx, 7, in_span + ba2_scratch_bytes(NP, NO, P) + 256);
    if (!buf) return YGZB_ERR_CUDA;
    Carver c(buf);
    int32_t* d_off = c.take<int32_t>(3 * (P + 1));
    double* d_poses = c.take<double>(6 * NK);
    uint8_t* d_fixed = c.take<uint8_t>(NK);
    double* d_pts = c.take<double>(3 * NP);
    int32_t* d_idx = c.take<int32_t>(2 * NO);
    double* d_obs = c.take<double>(2 * NO);
    const size_t in_bytes = (size_t)(reinterpret_cast<uint8_t*>(d_obs + 2 * NO) - static_cast<uint8_t*>(buf));
    uint8_t* stage = static_cast<uint8_t*>(host_scratch(ctx, 1, in_bytes));
    if (!stage) return YGZB_ERR_CUDA;
    YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // an earlier copy may still read the staging buffer
    auto put = [&](const void* dev_ptr, const void* src, size_t bytes) {
        if (bytes) memcpy(stage + (static_cast<const uint8_t*>(dev_ptr) - static_cast<uint8_t*>(buf)), src, bytes);
    };
    put(d_off, kf_off, (P + 1) * 4);
    put(d_off + (P + 1), pt_off, (P + 1) * 4);
    put(d_off + 2 * (P + 1), obs_off, (P + 1) * 4);
    put(d_poses, poses, 6 * NK * 8);
    put(d_fixed, fixed, NK);
    put(d_pts, pts, 3 * NP * 8);
    put(d_idx, kf_idx, NO * 4);
    put(d_idx + NO, pt_idx, NO * 4);
    put(d_obs, obs_px, 2 * NO * 8);
    YGZB_CUDA(ctx, cudaMemcpyAsync(buf, stage, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    in.kf_off = d_off; in.pt_off = d_off + (P + 1); in.obs_off = d_off + 2 * (P + 1);
    in.poses = d_poses; in.fixed = d_fixed; in.pts = d_pts; in.kf_idx = d_idx; in.pt_idx = d_idx + NO; in.obs = d_obs;
    in.lm_start = nullptr;
    uint8_t* d_outl = nullptr;
    double* d_stats = nullptr;
    void* scratch = static_cast<uint8_t*>(buf) + ((in_span + 255) & ~(size_t)255);
    TRY(launch_local_ba2(ctx, in, scratch, prm, &d_outl, &d_stats));
    TRY(d2h(ctx, poses, d_poses, 6 * NK));
    TRY(d2h(ctx, pts, d_pts, 3 * NP));
    if (outlier) TRY(d2h(ctx, outlier, d_outl, NO));
    hst.resize(8 * P);
    TRY(d2h(ctx, hst.data(), d_stats, 8 * P));
    YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (size_t p = 0; p < P; ++p)
        if (hst[8 * p + 6] != 0)
            return set_error(ctx, YGZB_ERR_INVALID, "problem %zu: a point is observed twice by one key-frame (not a SLAM graph)", p);
    return YGZB_OK;
}

// shared body of ygzb_local_ba_ceres and ygzb_two_view_ba: index bookkeeping on the host, one cluster launch, results
// back.  hst receives the 8 raw statistics of every problem.
int run_local_ba(ygzb_ctx* ctx, int n_problems, const int32_t* kf_off, const int32_t* pt_off, const int32_t* obs_off,
                 double* poses, const uint8_t* fixed, double* pts, const int32_t* kf_idx, const int32_t* pt_idx,
                 const double* obs_px, const ygzb_ba_params* prm, std::vector<double>& hst, const uint8_t* loss_mask = nullptr) {
    cudaSetDevice(ctx->device);
    for (const auto& oc : {std::make_pair(kf_off, "kf_off"), std::make_pair(pt_off, "pt_off"), std::make_pair(obs_off, "obs_off")}) {
        const int rc = check_offsets(ctx, oc.first, n_problems, oc.second);
        if (rc != YGZB_OK) return rc;
    }
    const size_t P = (size_t)n_problems, NK = (size_t)kf_off[n_problems], NP = (size_t)pt_off[n_problems], NO = (size_t)obs_off[n_problems];
    // ---- structure: observations grouped by landmark, by pose, and landmark-sharing observation pairs per block pair
    std::vector<int32_t> lm_start(NP + 1, 0), lm_obs(NO), ps_start(NK + 1, 0), ps_obs(NO), pair_off(P + 1, 0), pair_start, pair_o1, pair_o2;
    int max_free = 0;
    for (size_t p = 0; p < P; ++p) {
        const int k0 = kf_off[p], nk = kf_off[p + 1] - k0, p0 = pt_off[p], npt = pt_off[p + 1] - p0, o0 = obs_off[p], no = obs_off[p + 1] - o0;
        if (nk < 1 || nk > kMaxPoses) return set_error(ctx, YGZB_ERR_INVALID, "problem %zu: %d poses (1..%d supported)", p, nk, kMaxPoses);
        std::vector<int> free_index(nk, -1);
        int nf = 0;
        for (int k = 0; k < nk; ++k)
            if (!fixed[k0 + k]) free_index[k] = nf++;
        if (nf > kMaxFreePoses) return set_error(ctx, YGZB_ERR_INVALID, "problem %zu: %d free poses (max %d)", p, nf, kMaxFreePoses);
        max_free = std::max(max_free, nf);
        for (int o = 0; o < no; ++o) {
            if (kf_idx[o0 + o] < 0 || kf_idx[o0 + o] >= nk || pt_idx[o0 + o] < 0 || pt_idx[o0 + o] >= npt)
                return set_error(ctx, YGZB_ERR_INVALID, "observation %d: index out of range", o0 + o);
            lm_start[p0 + pt_idx[o0 + o] + 1]++;
            ps_start[k0 + kf_idx[o0 + o] + 1]++;
        }
        (void)npt;
    }
    for (size_t i = 0; i < NP; ++i) lm_start[i + 1] += lm_start[i];
    for (size_t i = 0; i < NK; ++i) ps_start[i + 1] += ps_start[i];
    {
        std::vector<int32_t> lc(lm_start.begin(), lm_start.end() - 1), pc(ps_start.begin(), ps_start.end() - 1);
        for (size_t p = 0; p < P; ++p)
            for (int o = obs_off[p]; o < obs_off[p + 1]; ++o) {
                lm_obs[lc[pt_off[p] + pt_idx[o]]++] = o;
                ps_obs[pc[kf_off[p] + kf_idx[o]]++] = o;
            }
    }
    // landmark-sharing observation pairs per (free pose f1 <= f2) block pair, as CSR: two passes (count, fill), no
    // per-problem allocations.  pair_start holds n_pairs + 1 entries per problem.
    std::vector<int32_t> free_of(NK, -1), nfree(P, 0);
    for (size_t p = 0; p < P; ++p) {
        int nf = 0;
        for (int k = kf_off[p]; k < kf_off[p + 1]; ++k)
            if (!fixed[k]) free_of[k] = nf++;
        nfree[p] = nf;
        pair_off[p + 1] = pair_off[p] + nf * (nf + 1) / 2 + 1;
    }
    pair_start.assign((size_t)pair_off[P], 0);
    auto for_each_pair = [&](auto&& visit) {
        for (size_t p = 0; p < P; ++p) {
            const int k0 = kf_off[p], p0 = pt_off[p], npt = pt_off[p + 1] - p0, nf = nfree[p];
            if (nf == 0) continue;
            for (int j = 0; j < npt; ++j) {
                const int qa = lm_start[p0 + j], qb = lm_start[p0 + j + 1];
                for (int q1 = qa; q1 < qb; ++q1) {
                    const int f1 = free_of[k0 + kf_idx[lm_obs[q1]]];
                    if (f1 < 0) continue;
                    for (int q2 = qa; q2 < qb; ++q2) {
                        const int f2 = free_of[k0 + kf_idx[lm_obs[q2]]];
                        if (f2 < f1 || (f2 == f1 && q2 != q1)) continue;
                        visit(pair_off[p] + f1 * nf - f1 * (f1 - 1) / 2 + (f2 - f1), lm_obs[q1], lm_obs[q2]);
                    }
                }
            }
        }
    };
    for_each_pair([&](int slot, int32_t, int32_t) { pair_start[slot + 1]++; });   // every problem owns n_pairs + 1 entries
    // the counts sit one entry to the right: a running sum over the whole array turns them into start offsets (the extra
    // entry of every problem carries the total across the problem boundary)
    {
        int32_t run = 0;
        for (size_t i = 0; i < pair_start.size(); ++i) {
            run += pair_start[i];
            pair_start[i] = run;
        }
    }
    pair_o1.assign((size_t)(pair_start.empty() ? 0 : pair_start.back()), 0);
    pair_o2.assign(pair_o1.size(), 0);
    {
        std::vector<int32_t> cursor(pair_start);
        for_each_pair([&](int slot, int32_t o1, int32_t o2) {
            const int32_t at = cursor[slot]++;
            pair_o1[at] = o1;
            pair_o2[at] = o2;
        });
    }
    const size_t NPAIR = pair_o1.size(), NPS = pair_start.size();

    Carver sz(nullptr);
    sz.take<int32_t>(3 * (P + 1)); sz.take<double>(6 * NK); sz.take<uint8_t>(NK); sz.take<double>(3 * NP); sz.take<int32_t>(2 * NO);
    sz.take<double>(2 * NO); sz.take<int32_t>(NP + 1 + NO + NK + 1 + NO); sz.take<int32_t>(P + 1 + NPS + 2 * NPAIR);
    sz.take<double>(21 * NO); sz.take<double>(9 * NP); sz.take<double>(3 * NP); sz.take<double>(9 * NP); sz.take<double>(3 * NP);
    sz.take<double>(3 * NP); sz.take<double>(3 * NP); sz.take<double>(8 * P);
    void* buf = dev_scratch(ctx, 7, sz.bytes());
    if (!buf) return YGZB_ERR_CUDA;
    Carver c(buf);
    int32_t* d_off = c.take<int32_t>(3 * (P + 1));
    double* d_poses = c.take<double>(6 * NK);
    uint8_t* d_fixed = c.take<uint8_t>(NK);
    double* d_pts = c.take<double>(3 * NP);
    int32_t* d_idx = c.take<int32_t>(2 * NO);
    double* d_obs = c.take<double>(2 * NO);
    int32_t* d_csr = c.take<int32_t>(NP + 1 + NO + NK + 1 + NO);
    int32_t* d_pairs = c.take<int32_t>(P + 1 + NPS + 2 * NPAIR);
    BAArgs a;
    a.lin = c.take<double>(21 * NO);
    a.Hll = c.take<double>(9 * NP);
    a.bl = c.take<double>(3 * NP);
    a.Dinv = c.take<double>(9 * NP);
    a.xl = c.take<double>(3 * NP);
    a.pts_backup = c.take<double>(3 * NP);
    a.scale_l = c.take<double>(3 * NP);
    a.stats = c.take<double>(8 * P);
    // kf_idx / pt_idx stay LOCAL to the problem; lm_obs / ps_obs / pair entries are GLOBAL observation ids.
    // All inputs sit at the front of the device buffer in one contiguous run: they are assembled in a pinned staging
    // buffer with the same layout and travel as ONE host-to-device copy (instead of 17 pageable ones).
    const size_t in_bytes = (size_t)(reinterpret_cast<uint8_t*>(d_pairs + P + 1 + NPS + 2 * NPAIR) - static_cast<uint8_t*>(buf));
    uint8_t* stage = static_cast<uint8_t*>(host_scratch(ctx, 1, in_bytes));
    if (!stage) return YGZB_ERR_CUDA;
    YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // an earlier copy may still read the staging buffer
    auto put = [&](const void* dev_ptr, const void* src, size_t bytes) {
        if (bytes) memcpy(stage + (static_cast<const uint8_t*>(dev_ptr) - static_cast<uint8_t*>(buf)), src, bytes);
    };
    put(d_off, kf_off, (P + 1) * 4);
    put(d_off + (P + 1), pt_off, (P + 1) * 4);
    put(d_off + 2 * (P + 1), obs_off, (P + 1) * 4);
    put(d_poses, poses, 6 * NK * 8);
    put(d_fixed, fixed, NK);
    put(d_pts, pts, 3 * NP * 8);
    put(d_idx, kf_idx, NO * 4);
    put(d_idx + NO, pt_idx, NO * 4);
    put(d_obs, obs_px, 2 * NO * 8);
    put(d_csr, lm_start.data(), (NP + 1) * 4);
    put(d_csr + NP + 1, lm_obs.data(), NO * 4);
    put(d_csr + NP + 1 + NO, ps_start.data(), (NK + 1) * 4);
    put(d_csr + NP + 1 + NO + NK + 1, ps_obs.data(), NO * 4);
    put(d_pairs, pair_off.data(), (P + 1) * 4);
    put(d_pairs + P + 1, pair_start.data(), NPS * 4);
    put(d_pairs + P + 1 + NPS, pair_o1.data(), NPAIR * 4);
    put(d_pairs + P + 1 + NPS + NPAIR, pair_o2.data(), NPAIR * 4);
    YGZB_CUDA(ctx, cudaMemcpyAsync(buf, stage, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    a.kf_off = d_off; a.pt_off = d_off + (P + 1); a.obs_off = d_off + 2 * (P + 1);
    a.poses = d_poses; a.fixed = d_fixed; a.pts = d_pts; a.kf_idx = d_idx; a.pt_idx = d_idx + NO; a.obs = d_obs;
    a.lm_start = d_csr; a.lm_obs = d_csr + NP + 1; a.ps_start = d_csr + NP + 1 + NO; a.ps_obs = d_csr + NP + 1 + NO + NK + 1;
    a.pair_off = d_pairs; a.pair_start = d_pairs + P + 1; a.pair_o1 = d_pairs + P + 1 + NPS; a.pair_o2 = d_pairs + P + 1 + NPS + NPAIR;
    a.fx = ctx->prm.fx; a.fy = ctx->prm.fy; a.cx = ctx->prm.cx; a.cy = ctx->prm.cy;
    a.max_iters = prm->max_iters; a.huber_delta = prm->huber_delta;
    a.loss_mask = nullptr;
    if (loss_mask && NO) {
        uint8_t* d_mask = static_cast<uint8_t*>(dev_scratch(ctx, 4, NO));
        if (!d_mask) return YGZB_ERR_CUDA;
        YGZB_CUDA(ctx, cudaMemcpyAsync(d_mask, loss_mask, NO, cudaMemcpyHostToDevice, ctx->stream));
        a.loss_mask = d_mask;
    }
    const int dimp = 6 * std::max(max_free, 1);
    const size_t smem = sizeof(double) * ((size_t)dimp * dimp + (size_t)dimp);
    ClusterWs* d_ws = static_cast<ClusterWs*>(dev_scratch(ctx, 5, sizeof(ClusterWs) * P));
    if (!d_ws) return YGZB_ERR_CUDA;
    {
        // opt in to the largest reduced system (16 free poses: 74.5 KB) once: a per-call value would race between the
        // contexts of several host threads
        static std::once_flag smem_once;
        std::call_once(smem_once, [] {
            const int max_smem = (int)(sizeof(double) * ((size_t)(6 * kMaxFreePoses) * (6 * kMaxFreePoses) + 6 * kMaxFreePoses));
            cudaFuncSetAttribute(local_ba_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
        });
    }
    {
        // one cluster of CTAs (= SMs) per problem.  Every LM trial crosses ~8 cluster barriers, so small problems (a few
        // thousand observations: the local BA of the tracking loop) are faster on fewer CTAs; large ones want all eight
        size_t max_obs = 0;
        for (size_t p = 0; p < P; ++p) max_obs = std::max(max_obs, (size_t)(obs_off[p + 1] - obs_off[p]));
        int cluster = kClusterSize;
        (void)max_obs;   // size-dependent choice pending measurement (tools/ba_cluster_sweep.py)
        if (const char* e = getenv("YGZB_BA_CLUSTER")) {   // tuning knob: 1, 2, 4 or 8
            const int v = atoi(e);
            if (v == 1 || v == 2 || v == 4 || v == 8 || v == 16) cluster = v;
        }
        if (cluster > 8) YGZB_CUDA(ctx, cudaFuncSetAttribute(local_ba_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)(n_problems * cluster));
        cfg.blockDim = dim3(kBAThreads);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = ctx->stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = cluster;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        ProfScope ps(ctx, kStageLocalBA);
        YGZB_CUDA(ctx, cudaLaunchKernelEx(&cfg, local_ba_kernel, a, d_ws));
    }
    YGZB_LAUNCHED(ctx);
    TRY(d2h(ctx, poses, d_poses, 6 * NK));
    TRY(d2h(ctx, pts, d_pts, 3 * NP));
    hst.resize(8 * P);
    TRY(d2h(ctx, hst.data(), a.stats, 8 * P));
    YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return YGZB_OK;
}
}  // namespace

extern "C" {

int ygzb_local_ba(ygzb_ctx* ctx, int n_problems, const int32_t* kf_off, const int32_t* pt_off, const int32_t* obs_off,
                  double* poses, const uint8_t* fixed, double* pts, const int32_t* kf_idx, const int32_t* pt_idx,
                  const double* obs_px, const ygzb_ba_params* prm, uint8_t* outlier, ygzb_ba_stats* stats) {
    if (!ctx || n_problems < 1 || !kf_off || !pt_off || !obs_off || !poses || !fixed || !pts || !kf_idx || !pt_idx || !obs_px ||
        !prm || !outlier)
        return YGZB_ERR_INVALID;
    cudaSetDevice(ctx->device);
    for (const auto& oc : {std::make_pair(kf_off, "kf_off"), std::make_pair(pt_off, "pt_off"), std::make_pair(obs_off, "obs_off")}) {
        const int rc = check_offsets(ctx, oc.first, n_problems, oc.second);
        if (rc != YGZB_OK) return rc;
    }
    std::vector<double> hst;
    try {   // the header promises that calls never throw: allocation failures of the host-side bookkeeping become an error code
        TRY(run_local_ba2(ctx, n_problems, kf_off, pt_off, obs_off, poses, fixed, pts, kf_idx, pt_idx, obs_px, prm, outlier, hst));
    } catch (const std::exception& e) {
        return set_error(ctx, YGZB_ERR_INVALID, "ygzb_local_ba: %s", e.what());
    }
    if (stats)
        for (size_t p = 0; p < (size_t)n_problems; ++p) {
            stats[p].iters = (int)hst[8 * p];
            stats[p].lm_trials = (int)hst[8 * p + 1];
            stats[p].chi2_initial = hst[8 * p + 2];
            stats[p].chi2_final = hst[8 * p + 3];
            stats[p].lambda_final = hst[8 * p + 4];
            stats[p].n_outliers = (int)hst[8 * p + 5];
        }
    return YGZB_OK;
}

int ygzb_local_ba_ceres(ygzb_ctx* ctx, int n_problems, const int32_t* kf_off, const int32_t* pt_off, const int32_t* obs_off,
                        double* poses, const uint8_t* fixed, double* pts, const int32_t* kf_idx, const int32_t* pt_idx,
                        const double* obs_px, int max_iters, double huber_a, ygzb_ceres_stats* stats) {
    if (!ctx || n_problems < 1 || !kf_off || !pt_off || !obs_off || !poses || !fixed || !pts || !kf_idx || !pt_idx || !obs_px ||
        max_iters < 0 || !(huber_a >= 0))
        return YGZB_ERR_INVALID;
    ygzb_ba_params prm;
    ygzb_default_ba_params(&prm);
    prm.max_iters = max_iters;   // ceres::Solver::Options::max_num_iterations (50 by default)
    prm.huber_delta = huber_a;   // 0: no loss function (nullptr in AddResidualBlock, BA.cpp:346,364); 0.1: BA.cpp:108-135
    std::vector<double> hst;
    try {
        TRY(run_local_ba(ctx, n_problems, kf_off, pt_off, obs_off, poses, fixed, pts, kf_idx, pt_idx, obs_px, &prm, hst));
    } catch (const std::exception& e) {
        return set_error(ctx, YGZB_ERR_INVALID, "ygzb_local_ba_ceres: %s", e.what());
    }
    if (stats)
        for (size_t p = 0; p < (size_t)n_problems; ++p) {
            stats[p].iters = (int)hst[8 * p];
            stats[p].successful_steps = (int)hst[8 * p + 1];
            stats[p].cost_initial = hst[8 * p + 2];
            stats[p].cost_final = hst[8 * p + 3];
            stats[p].radius_final = hst[8 * p + 4];
            stats[p].termination = (int)hst[8 * p + 5];
        }
    return YGZB_OK;
}

// ba::TwoViewBACeres (reference src/Algorithm/BA.cpp:11-89) for a batch of two-view problems, on the Ceres-flavoured
// cluster kernel: reference pose fixed (point-only blocks), current pose and points free, HuberLoss(0.1) on the blocks of the
// non-inlier points, then the reference's inlier test (classification kernel below)
__global__ void two_view_classify_kernel(int n, const int32_t* __restrict__ prob_of, const double* __restrict__ T_ref,
                                         const double* __restrict__ poses, const double* __restrict__ pts, const double* __restrict__ px_ref,
                                         const double* __restrict__ px_cur, float fx, float fy, float cx, float cy, uint8_t* __restrict__ inlier,
                                         double* __restrict__ T_cur_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int p = prob_of[i];
    const double* Tr = T_ref + 12 * (size_t)p;
    const double* pc = poses + 12 * (size_t)p + 6;   // [t; angle-axis] of the current frame
    double th;
    SE3d Tc;
    Tc.q = so3_exp(V3d{pc[3], pc[4], pc[5]}, &th);
    Tc.t = V3d{pc[0], pc[1], pc[2]};
    double Tm[12];
    se3_to_mat(Tc, Tm);
    if (i == 0 || prob_of[i - 1] != p)
        for (int c = 0; c < 12; ++c) T_cur_out[12 * (size_t)p + c] = Tm[c];
    const double X = pts[3 * (size_t)i], Y = pts[3 * (size_t)i + 1], Z = pts[3 * (size_t)i + 2];
    const double x1 = Tr[0] * X + Tr[1] * Y + Tr[2] * Z + Tr[3], y1 = Tr[4] * X + Tr[5] * Y + Tr[6] * Z + Tr[7], z1 = Tr[8] * X + Tr[9] * Y + Tr[10] * Z + Tr[11];
    const double x2 = Tm[0] * X + Tm[1] * Y + Tm[2] * Z + Tm[3], y2 = Tm[4] * X + Tm[5] * Y + Tm[6] * Z + Tm[7], z2 = Tm[8] * X + Tm[9] * Y + Tm[10] * Z + Tm[11];
    const double e1x = px_ref[2 * (size_t)i] - (fx * x1 / z1 + cx), e1y = px_ref[2 * (size_t)i + 1] - (fy * y1 / z1 + cy);
    const double e2x = px_cur[2 * (size_t)i] - (fx * x2 / z2 + cx), e2y = px_cur[2 * (size_t)i + 1] - (fy * y2 / z2 + cy);
    uint8_t in = 1;
    if (e1x * e1x + e1y * e1y > 5.991 || e2x * e2x + e2y * e2y > 5.991) in = 0;   // BA.cpp:70-77
    else if (z1 < 0 || z2 < 0) in = 0;                                            // :78-81
    inlier[i] = in;
}

int ygzb_two_view_ba(ygzb_ctx* ctx, int n_problems, const int32_t* offsets, const double* T_cw_ref, double* T_cw_cur, const double* px_ref,
                     const double* px_cur, uint8_t* inlier, double* pts, ygzb_ceres_stats* stats) {
    if (!ctx || n_problems < 1 || !offsets || !T_cw_ref || !T_cw_cur) return YGZB_ERR_INVALID;
    cudaSetDevice(ctx->device);
    {
        const int rc = check_offsets(ctx, offsets, n_problems, "offsets");
        if (rc != YGZB_OK) return rc;
    }
    const size_t P = (size_t)n_problems, N = (size_t)offsets[n_problems];
    if (N && (!px_ref || !px_cur || !inlier || !pts)) return YGZB_ERR_INVALID;
    try {
        std::vector<int32_t> kf_off(P + 1), pt_off(offsets, offsets + P + 1), obs_off(P + 1), kf_idx(2 * N), pt_idx(2 * N), prob_of(N);
        std::vector<double> poses(12 * P), obs(4 * N), X(pts, pts + 3 * N);
        std::vector<uint8_t> fixed(2 * P), mask(2 * N);
        for (size_t p = 0; p < P; ++p) {
            kf_off[p] = (int32_t)(2 * p);
            obs_off[p] = 2 * offsets[p];
            fixed[2 * p] = 1;   // the reference frame: CeresReprojectionErrorPointOnly blocks (BA.cpp:33-43)
            fixed[2 * p + 1] = 0;
            for (int k = 0; k < 2; ++k) {   // pose = [translation; so3 log] (BA.cpp:24-26)
                const SE3d T = se3_from_mat((k ? T_cw_cur : T_cw_ref) + 12 * p);
                double th;
                const V3d l = so3_log(T.q, &th);
                double* o = &poses[12 * p + 6 * k];
                o[0] = T.t.x; o[1] = T.t.y; o[2] = T.t.z; o[3] = l.x; o[4] = l.y; o[5] = l.z;
            }
            for (int i = offsets[p]; i < offsets[p + 1]; ++i) {
                const int li = i - offsets[p];
                prob_of[i] = (int32_t)p;
                if (!inlier[i]) {   // BA.cpp:35-37
                    X[3 * (size_t)i] = 0; X[3 * (size_t)i + 1] = 0; X[3 * (size_t)i + 2] = 1;
                }
                kf_idx[2 * (size_t)i] = 0; kf_idx[2 * (size_t)i + 1] = 1;
                pt_idx[2 * (size_t)i] = pt_idx[2 * (size_t)i + 1] = li;
                obs[4 * (size_t)i] = px_ref[2 * (size_t)i]; obs[4 * (size_t)i + 1] = px_ref[2 * (size_t)i + 1];
                obs[4 * (size_t)i + 2] = px_cur[2 * (size_t)i]; obs[4 * (size_t)i + 3] = px_cur[2 * (size_t)i + 1];
                mask[2 * (size_t)i] = mask[2 * (size_t)i + 1] = inlier[i] ? 0 : 1;
            }
        }
        kf_off[P] = (int32_t)(2 * P);
        obs_off[P] = 2 * offsets[P];
        ygzb_ba_params prm;
        ygzb_default_ba_params(&prm);
        prm.max_iters = 50;
        prm.huber_delta = 0.1;
        std::vector<double> hst;
        TRY(run_local_ba(ctx, n_problems, kf_off.data(), pt_off.data(), obs_off.data(), poses.data(), fixed.data(), X.data(),
                         kf_idx.data(), pt_idx.data(), obs.data(), &prm, hst, mask.data()));
        if (stats)
            for (size_t p = 0; p < P; ++p) {
                stats[p].iters = (int)hst[8 * p]; stats[p].successful_steps = (int)hst[8 * p + 1]; stats[p].cost_initial = hst[8 * p + 2];
                stats[p].cost_final = hst[8 * p + 3]; stats[p].radius_final = hst[8 * p + 4]; stats[p].termination = (int)hst[8 * p + 5];
            }
        std::memcpy(pts, X.data(), 3 * N * sizeof(double));
        // inlier classification + pose conversion on the device
        Carver sz(nullptr);
        sz.take<int32_t>(N); sz.take<double>(12 * P); sz.take<double>(12 * P); sz.take<double>(3 * N); sz.take<double>(2 * N); sz.take<double>(2 * N);
        sz.take<uint8_t>(N); sz.take<double>(12 * P);
        void* buf = dev_scratch(ctx, 6, sz.bytes());
        if (!buf) return YGZB_ERR_CUDA;
        Carver c(buf);
        int32_t* d_prob = c.take<int32_t>(N);
        double* d_Tref = c.take<double>(12 * P);
        double* d_poses = c.take<double>(12 * P);
        double* d_pts = c.take<double>(3 * N);
        double* d_pr = c.take<double>(2 * N);
        double* d_pc = c.take<double>(2 * N);
        uint8_t* d_in = c.take<uint8_t>(N);
        double* d_Tcur = c.take<double>(12 * P);
        TRY(h2d(ctx, d_prob, prob_of.data(), N));
        TRY(h2d(ctx, d_Tref, T_cw_ref, 12 * P));
        TRY(h2d(ctx, d_poses, poses.data(), 12 * P));
        TRY(h2d(ctx, d_pts, X.data(), 3 * N));
        TRY(h2d(ctx, d_pr, px_ref, 2 * N));
        TRY(h2d(ctx, d_pc, px_cur, 2 * N));
        if (N) {
            two_view_classify_kernel<<<(unsigned)((N + 127) / 128), 128, 0, ctx->stream>>>((int)N, d_prob, d_Tref, d_poses, d_pts, d_pr, d_pc, ctx->prm.fx,
                                                                                       ctx->prm.fy, ctx->prm.cx, ctx->prm.cy, d_in, d_Tcur);
            YGZB_LAUNCHED(ctx);
            TRY(d2h(ctx, inlier, d_in, N));
            TRY(d2h(ctx, T_cw_cur, d_Tcur, 12 * P));
        }
        YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    } catch (const std::exception& e) {
        return set_error(ctx, YGZB_ERR_INVALID, "ygzb_two_view_ba: %s", e.what());
    }
    return YGZB_OK;
}

int ygzb_pose_only(ygzb_ctx* ctx, int n_problems, const int32_t* offsets, const double* pt_world, const double* px, double* T_cw,
                   uint8_t* inlier, double* depth, int32_t* n_inlier) {
    if (!ctx || n_problems < 1 || !offsets || !T_cw || !n_inlier) return YGZB_ERR_INVALID;
    cudaSetDevice(ctx->device);
    {
        const int rc = check_offsets(ctx, offsets, n_problems, "offsets");
        if (rc != YGZB_OK) return rc;
    }
    const size_t P = (size_t)n_problems, N = (size_t)offsets[n_problems];
    if (N && (!pt_world || !px || !inlier || !depth)) return YGZB_ERR_INVALID;
    Carver sz(nullptr);
    sz.take<int32_t>(P + 1); sz.take<double>(3 * N); sz.take<double>(2 * N); sz.take<double>(12 * P); sz.take<uint8_t>(N);
    sz.take<double>(N); sz.take<int32_t>(P); sz.take<uint8_t>(N); sz.take<double>(P * 4 * kPoseCluster * kPoseRed);
    void* buf = dev_scratch(ctx, 7, sz.bytes());
    if (!buf) return YGZB_ERR_CUDA;
    Carver c(buf);
    PoseOnlyArgs a;
    int32_t* d_off = c.take<int32_t>(P + 1);
    double* d_pw = c.take<double>(3 * N);
    double* d_px = c.take<double>(2 * N);
    a.T_cw = c.take<double>(12 * P);
    a.inlier = c.take<uint8_t>(N);
    a.depth = c.take<double>(N);
    a.n_inlier = c.take<int32_t>(P);
    a.enable = c.take<uint8_t>(N);
    a.ws = c.take<double>(P * 4 * kPoseCluster * kPoseRed);
    a.offsets = d_off; a.counts = nullptr; a.pw = d_pw; a.px = d_px;
    a.fx = ctx->prm.fx; a.fy = ctx->prm.fy; a.cx = ctx->prm.cx; a.cy = ctx->prm.cy;
    {   // the four inputs are the first sub-buffers of `buf`: one pinned staging copy instead of four pageable ones
        const size_t in_bytes = (size_t)(reinterpret_cast<uint8_t*>(a.T_cw + 12 * P) - static_cast<uint8_t*>(buf));
        uint8_t* stage = static_cast<uint8_t*>(host_scratch(ctx, 1, in_bytes));
        if (!stage) return YGZB_ERR_CUDA;
        YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        auto put = [&](const void* dev_ptr, const void* src, size_t bytes) {
            if (bytes) memcpy(stage + (static_cast<const uint8_t*>(dev_ptr) - static_cast<uint8_t*>(buf)), src, bytes);
        };
        put(d_off, offsets, (P + 1) * 4);
        put(d_pw, pt_world, 3 * N * 8);
        put(d_px, px, 2 * N * 8);
        put(a.T_cw, T_cw, 12 * P * 8);
        YGZB_CUDA(ctx, cudaMemcpyAsync(buf, stage, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    {
        int max_points = 0;
        for (size_t q = 0; q < P; ++q) max_points = std::max(max_points, offsets[q + 1] - offsets[q]);
        a.stage_k = pose_only_stage_k(max_points, kPoseCluster);
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)(n_problems * kPoseCluster));
        cfg.blockDim = dim3(kPoseThreads);
        cfg.dynamicSmemBytes = (size_t)a.stage_k * 5 * kPoseThreads * sizeof(double);
        cfg.stream = ctx->stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = kPoseCluster;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        ProfScope ps(ctx, kStagePoseOnly);
        YGZB_CUDA(ctx, cudaLaunchKernelEx(&cfg, pose_only_kernel, a));
    }
    YGZB_LAUNCHED(ctx);
    TRY(d2h(ctx, T_cw, a.T_cw, 12 * P));
    TRY(d2h(ctx, inlier, a.inlier, N));
    TRY(d2h(ctx, depth, a.depth, N));
    TRY(d2h(ctx, n_inlier, a.n_inlier, P));
    YGZB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return YGZB_OK;
}

}  // extern "C"
