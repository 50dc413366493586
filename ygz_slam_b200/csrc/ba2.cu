// ba2.cu -- ba::LocalBAG2O, second generation: a landmark-partitioned thread-block cluster per problem.
//
// Replaces:
//   ba::LocalBAG2O                   reference src/Algorithm/BA.cpp:386-543
//   VertexSE3Sophus::oplusImpl       reference include/ygz/G2oTypes.h:38-45
//   EdgeSophusSE3ProjectXYZ          reference include/ygz/G2oTypes.h:84-132 (computeError, linearizeOplus)
// g2o itself is outside the reference tree: the Levenberg schedule follows oracle/ba.cpp (SURVEY.md appendix A.3).
//
// Why a second generation: the first one strides observations over the cluster, keeps a 21-double linearisation record
// per observation in global memory that every CTA reads through L2 (__ldcg), combines partial sums with f64 atomics and
// crosses ~13 cluster barriers per LM trial; ncu showed 5 % issue-slot utilisation (profiles/r1_final2_local_ba.txt).
// Here
//   * the LANDMARKS are partitioned over the CTAs of the cluster (contiguous ranges of the landmark-major observation
//     list), so everything a landmark needs -- its observations, Hll, bl, (Hll + lambda I)^-1, the 6-double
//     linearisation record (x, y, z, e0, e1, w) of each observation from which the 2x3 / 2x6 Jacobians are rebuilt in
//     ~30 flops -- is private to ONE CTA and staged in its shared memory (global scratch only when a problem is too big);
//   * the reduced system is accumulated by warp tasks (block pair of free poses x stripe of landmarks) that keep their 36+6
//     sums in registers across the whole stripe and shuffle-reduce once; no atomics anywhere: partial sums are combined
//     in a fixed order inside the CTA and with a reduce-scatter / all-gather over distributed shared memory across the
//     cluster, so the result is bit-reproducible run to run;
//   * an LM trial crosses 3 cluster barriers (2 for the reduced system, 1 for chi2 / gain ratio) and 6 CTA barriers;
//     a rejected trial re-uses the linearisation and only re-inverts (Hll + lambda I).
// The observation lists arrive landmark-major (CSR): csr_* kernels below build that order on the device from the
// (kf_idx, pt_idx) arrays of the C ABI, deterministic (observations of a landmark sorted by their original index).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include <cooperative_groups.h>

#include "ba2.cuh"
#include "common.cuh"
#include "se3.cuh"

namespace ygzb {

namespace {

namespace cg = cooperative_groups;

constexpr int kT = kBA2Threads;
constexpr int kW = kT / 32;
constexpr int kPairW = 42;   // record of a block-pair task: 36 (Hpl D Hpl^T) + 6 (Hpl D bl, diagonal pairs only)
constexpr int kPoseW = 27;   // record of a pose task: 21 (upper triangle of Hpp) + 6 (bp)

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, o);
    return v;
}

// block-wide sum of two values (result valid in every thread); s_tmp: 2 * (kW + 1) doubles
// Sums of N per-lane values over the warp, all at once (a "reduce-scatter" butterfly): at every step a lane keeps one half of
// its values and hands the other half to its partner, so N values cost N - 1 (+ log2(32 / N)) shuffles instead of 5 N.
// N = 32: lane l returns the total of v[l]; N = 16: lanes 2 i and 2 i + 1 return the total of v[i].  (A warp flushes 42
// sums per block pair: 420 32-bit shuffles with one butterfly per value was a quarter of the accumulate phase.)
template <int N>
__device__ __forceinline__ double warp_reduce_scatter(double* v, int lane) {
    int off = 16;
#pragma unroll
    for (int n = N / 2; n >= 1; n >>= 1, off >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < n; ++i) {
            const double keep = up ? v[i + n] : v[i];
            const double send = up ? v[i] : v[i + n];
            v[i] = keep + __shfl_xor_sync(0xFFFFFFFFu, send, off);
        }
    }
#pragma unroll
    for (; off >= 1; off >>= 1) v[0] += __shfl_xor_sync(0xFFFFFFFFu, v[0], off);
    return v[0];
}

__device__ void block_sum2(double& v0, double& v1, double* s_tmp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v0 = warp_sum(v0);
    v1 = warp_sum(v1);
    __syncthreads();
    if (lane == 0) {
        s_tmp[warp] = v0;
        s_tmp[kW + 1 + warp] = v1;
    }
    __syncthreads();
    if (warp == 0) {
        double t0 = lane < kW ? s_tmp[lane] : 0.0, t1 = lane < kW ? s_tmp[kW + 1 + lane] : 0.0;
        t0 = warp_sum(t0);
        t1 = warp_sum(t1);
        if (lane == 0) {
            s_tmp[kW] = t0;
            s_tmp[2 * kW + 1] = t1;
        }
    }
    __syncthreads();
    v0 = s_tmp[kW];
    v1 = s_tmp[2 * kW + 1];
}

__device__ double block_max(double v, double* s_tmp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_down_sync(0xFFFFFFFFu, v, o));
    __syncthreads();
    if (lane == 0) s_tmp[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double t = lane < kW ? s_tmp[lane] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t = fmax(t, __shfl_down_sync(0xFFFFFFFFu, t, o));
        if (lane == 0) s_tmp[kW] = t;
    }
    __syncthreads();
    return s_tmp[kW];
}

// 1 / x for positive, normal x: hardware seed (MUFU.RCP64H, ~20 bits) + two Newton steps; within 1-2 ulp of the IEEE
// quotient at a fraction of the latency of the division sequence (the serial solve of an LM trial is latency bound)
constexpr int kCtaSolveMinDim = 24;   // reduced systems above this size are factorised by the whole CTA

__device__ __forceinline__ double fast_rcp(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(r, fma(-x, r, 1.0), r);
    r = fma(r, fma(-x, r, 1.0), r);
    return r;
}

__device__ __forceinline__ SE3d pose_from_g2o(const double* est) {
    const double v[6] = {est[3], est[4], est[5], est[0], est[1], est[2]};
    return se3_exp(v);
}

// Jacobians of EdgeSophusSE3ProjectXYZ::linearizeOplus (G2oTypes.h:108-131) rebuilt from the camera-frame point (x, y, 1/z)
// and the rotation rows of the pose at the linearisation point (the record keeps 1/z: no division when they are rebuilt)
struct Jac {
    double l0[3], l1[3];   // d e / d landmark, rows u and v
    double p0[6], p1[6];   // d e / d pose ([omega; upsilon] order of VertexSE3Sophus)
};
__device__ __forceinline__ void pose_jac(double x, double y, double iz, double fx, double fy, double* p0, double* p1) {
    const double iz2 = iz * iz;
    p0[0] = x * y * iz2 * fx; p0[1] = -(1.0 + x * x * iz2) * fx; p0[2] = y * iz * fx;
    p0[3] = -iz * fx; p0[4] = 0.0; p0[5] = x * iz2 * fx;
    p1[0] = (1.0 + y * y * iz2) * fy; p1[1] = -x * y * iz2 * fy; p1[2] = -x * iz * fy;
    p1[3] = 0.0; p1[4] = -iz * fy; p1[5] = y * iz2 * fy;
}
__device__ __forceinline__ void point_jac(double x, double y, double iz_pos, double fx, double fy, const double* R /* 12: [R|t] rows */,
                                          double* l0, double* l1) {
    const double iz = -iz_pos;
    const double t02 = x * iz * fx, t12 = y * iz * fy;   // -x/z fx, -y/z fy
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        l0[c] = iz * (fx * R[c] + t02 * R[8 + c]);
        l1[c] = iz * (fy * R[4 + c] + t12 * R[8 + c]);
    }
}
// Hpl = w Jp^T Jl (6 x 3)
__device__ __forceinline__ void make_hpl(const double* rec /* x y 1/z e0 e1 w */, const double* R, double fx, double fy, double H[6][3]) {
    double p0[6], p1[6], l0[3], l1[3];
    pose_jac(rec[0], rec[1], rec[2], fx, fy, p0, p1);
    point_jac(rec[0], rec[1], rec[2], fx, fy, R, l0, l1);
    const double w = rec[5];
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) H[a][b] = w * (p0[a] * l0[b] + p1[a] * l1[b]);
}

// symmetric 3x3 stored as (00, 01, 02, 11, 12, 22)
__device__ __forceinline__ void sym_inverse3(const double* h, double lambda, double* inv) {
    const double h0 = h[0] + lambda, h1 = h[1], h2 = h[2], h3 = h[3] + lambda, h4 = h[4], h5 = h[5] + lambda;
    const double c00 = h3 * h5 - h4 * h4, c01 = h2 * h4 - h1 * h5, c02 = h1 * h4 - h2 * h3;
    const double det = (c00 * h0 + c01 * h1) + c02 * h2;
    const double id = 1.0 / det;
    inv[0] = c00 * id; inv[1] = c01 * id; inv[2] = c02 * id;
    inv[3] = (h0 * h5 - h2 * h2) * id; inv[4] = (h1 * h2 - h0 * h4) * id; inv[5] = (h0 * h3 - h1 * h1) * id;
}
__device__ __forceinline__ void sym_mul3(const double* s, const double* v, double* out) {
    out[0] = s[0] * v[0] + s[1] * v[1] + s[2] * v[2];
    out[1] = s[1] * v[0] + s[3] * v[1] + s[4] * v[2];
    out[2] = s[2] * v[0] + s[4] * v[1] + s[5] * v[2];
}

// doubles of the CTA-private staging area for nl landmarks with no observations (see Stage): 14 per observation (two
// 6-double records + pixel) + 30 per landmark + the int / byte tables, rounded up
__host__ __device__ inline size_t ba2_stage_doubles(size_t nl, size_t no) {
    return 14 * no + 30 * nl + ((nl + 1) * 4 + ((no + 7) & ~(size_t)7) + nl * kBA2MaxFree + 7) / 8 + 1;
}

struct Stage {   // CTA-private per-landmark / per-observation state: shared memory when it fits, else global scratch
    double* lin[2];  // [no][6]  x y z e0 e1 w   (double buffered: accepted state / trial state)
    double* Hll[2];  // [nl][6]
    double* bl[2];   // [nl][3]
    double* X[2];    // [nl][3]  landmark positions of the accepted state / of the trial
    double* Dinv;    // [nl][6]  (Hll + lambda I)^-1 of the accepted state at the trial's lambda
    double* uv;      // [no][2]  measured pixels (copy of so_uv: read every trial)
    int32_t* qa;     // [nl + 1] first observation of every landmark, relative to the CTA's first observation
    uint8_t* kf;     // [no]     pose index of every observation
    uint8_t* slot;   // [nl][kBA2MaxFree]  position of the landmark's observation on free pose f inside its list, 0xFF = none
    uint32_t* ent;   // [ba2_entry_cap] dense (landmark, slot on f1, slot on f2) entries sorted by block pair, or null (see accumulate)
};

// upper bound of the block-pair entries of a CTA with nl landmarks and no observations on np free poses: a landmark seen by d
// free poses contributes d (d + 1) / 2 <= d (np + 1) / 2 entries
__host__ __device__ inline size_t ba2_entry_cap(size_t nl, size_t no, size_t np) {
    const size_t a = (no * (np + 1) + 1) / 2, b = nl * (np * (np + 1) / 2);
    return a < b ? a : b;
}

// L D L^T x = b by one warp with the factor of ldlt_factor_rl in S (unit lower triangle) and rd = 1 / D; b is overwritten with x
__device__ void warp_ldlt_subst(const double* S, double* b, const double* rd, int dimp, int lane) {
    // L z = b (unit diagonal), column oriented: the lane that owns row i publishes z_i, every lane updates its later rows
    double r[3];
#pragma unroll
    for (int m = 0; m < 3; ++m) r[m] = (lane + 32 * m < dimp) ? b[lane + 32 * m] : 0.0;
    for (int i = 0; i < dimp; ++i) {
        const int mi = i >> 5;
        const double mine = mi == 0 ? r[0] : (mi == 1 ? r[1] : r[2]);
        const double z = __shfl_sync(0xFFFFFFFFu, mine, i & 31);
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            const int k = lane + 32 * m;
            if (k > i && k < dimp) r[m] -= S[k * dimp + i] * z;
        }
    }
    // D y = z, then L^T x = y
#pragma unroll
    for (int m = 0; m < 3; ++m)
        if (lane + 32 * m < dimp) r[m] *= rd[lane + 32 * m];
    for (int i = dimp - 1; i >= 0; --i) {
        const int mi = i >> 5;
        const double mine = mi == 0 ? r[0] : (mi == 1 ? r[1] : r[2]);
        const double x = __shfl_sync(0xFFFFFFFFu, mine, i & 31);
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            const int k = lane + 32 * m;
            if (k < i) r[m] -= S[i * dimp + k] * x;
        }
    }
#pragma unroll
    for (int m = 0; m < 3; ++m)
        if (lane + 32 * m < dimp) b[lane + 32 * m] = r[m];
    __syncwarp();
}

// Right-looking LDL^T by a group of TI x TK threads (one warp as 4 x 8 for the small systems of the tracking loop, the whole
// CTA as 16 x 16 for the larger ones): per column the rank-1 update of the trailing triangle is one INDEPENDENT multiply-add
// per element (operands loaded first, then the arithmetic, then the stores -- no dependent chain longer than one operation;
// the left-looking version's dot product of length j per lane cost 88k cycles per LM trial at 54 x 54 and 12k at 12 x 12, a
// dependent FP64 operation being ~40 cycles), the thread that updates the next pivot also publishes its reciprocal, and there is
// ONE barrier per column.  Column j is scaled by 1 / D_j after the barrier (nothing reads it again before the substitution).
// S keeps D on the diagonal and the unit lower factor below it, rd = 1 / D (0 marks a non-positive pivot: the condition under
// which g2o's dense Cholesky fails).  Rows up to TI * A, i.e. n <= TI * A (+ the column itself).  Uniform return value.
template <int TI, int TK, int A, int B, bool kCta>
__device__ __forceinline__ bool ldlt_factor_rl(double* S, double* rd, int n, int t) {
    const int ti = t / TK, tk = t % TK;
    auto sync = [] {
        if (kCta) __syncthreads();
        else __syncwarp();
    };
    if (t == 0) {
        const double d = S[0];
        rd[0] = d > 0 ? fast_rcp(d) : 0.0;
    }
    sync();
    for (int j = 0; j < n; ++j) {
        const double r = rd[j];
        if (r == 0.0) return false;
        const int base = j + 1;
        double li[A], cj[B], v[A][B];
#pragma unroll
        for (int a = 0; a < A; ++a) {
            const int i = base + ti + TI * a;
            li[a] = i < n ? S[i * n + j] * r : 0.0;
        }
#pragma unroll
        for (int b = 0; b < B; ++b) {
            const int k = base + tk + TK * b;
            cj[b] = k < n ? S[k * n + j] : 0.0;
        }
#pragma unroll
        for (int a = 0; a < A; ++a)
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const int i = base + ti + TI * a, k = base + tk + TK * b;
                v[a][b] = (i < n && k <= i) ? S[i * n + k] : 0.0;
            }
#pragma unroll
        for (int a = 0; a < A; ++a)
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const int i = base + ti + TI * a, k = base + tk + TK * b;
                if (i < n && k <= i) {
                    const double u = v[a][b] - li[a] * cj[b];
                    S[i * n + k] = u;
                    if (a == 0 && b == 0 && t == 0) rd[base] = u > 0 ? fast_rcp(u) : 0.0;   // the next pivot
                }
            }
        sync();
        for (int q = t; q < n - base; q += TI * TK) S[(base + q) * n + j] *= r;
    }
    sync();
    return true;
}

// ---- 6 x 6 BLOCK LDL^T (right-looking).  Measured on the scalar version: a column costs ~900 cycles, of which only ~200 are
// the six dependent FP64 operations of the pivot chain -- the rest is the barrier and the shared-memory round trip around it.
// The dimension of the reduced system is a multiple of 6 (one block per free pose), so a pivot BLOCK is factorised by every
// thread itself in registers (same loads, same bits everywhere: nothing to publish), the rows of the block column are pushed
// through that factor (W = C Lb^-T = L D, L = W D^-1), the trailing triangle gets its rank-6 update, and there is ONE barrier per
// six columns.  The arithmetic is that of the scalar LDL^T (same pivots, no explicit inverse), the storage too: unit lower
// factor below the diagonal, D on it, rd = 1 / D -- warp_ldlt_subst applies it.  A non-positive pivot (the condition under which
// g2o's dense Cholesky fails) returns false, uniformly.  n <= TI * A + 6.
template <int TI, int TK, int A, int B, bool kCta>
__device__ __forceinline__ bool ldlt6_factor(double* S, double* rd, int n, int t) {
    const int ti = t / TK, tk = t % TK;
    auto sync = [] {
        if (kCta) __syncthreads();
        else __syncwarp();
    };
    sync();
    for (int J = 0; J < n; J += 6) {
        double P[6][6], rp[6];   // pivot block: lower triangle in, unit lower factor (below the diagonal) + D (diagonal) out
#pragma unroll
        for (int r = 0; r < 6; ++r)
#pragma unroll
            for (int c = 0; c <= r; ++c) P[r][c] = S[(J + r) * n + J + c];
        bool pd = true;
#pragma unroll
        for (int p = 0; p < 6; ++p) {
            const double d = P[p][p];
            pd = pd && d > 0;
            rp[p] = fast_rcp(d);
            double u[6];   // the unscaled column below the pivot
#pragma unroll
            for (int r = p + 1; r < 6; ++r) u[r] = P[r][p];
#pragma unroll
            for (int r = p + 1; r < 6; ++r) {
                const double l = u[r] * rp[p];
#pragma unroll
                for (int c = p + 1; c <= r; ++c) P[r][c] -= l * u[c];
                P[r][p] = l;
            }
        }
        if (!pd) return false;
        const int base = J + 6;
        double Wr[A][6], Lc[B][6], v[A][B];
#pragma unroll
        for (int a = 0; a < A; ++a) {
            const int i = base + ti + TI * a;
            if (i < n) {
                double X[6];
#pragma unroll
                for (int c = 0; c < 6; ++c) X[c] = S[i * n + J + c];
                // S_iJ = L_i D Lb^T  ->  (L_i D)_c = X_c - sum_{q<c} (L_i D)_q Lb[c][q]
#pragma unroll
                for (int c = 0; c < 6; ++c) {
                    double w = X[c];
#pragma unroll
                    for (int q = 0; q < c; ++q) w -= Wr[a][q] * P[c][q];
                    Wr[a][c] = w;
                }
            } else {
#pragma unroll
                for (int c = 0; c < 6; ++c) Wr[a][c] = 0.0;
            }
        }
#pragma unroll
        for (int b = 0; b < B; ++b) {
            const int k = base + tk + TK * b;
            if (k < n) {
                double X[6], W[6];
#pragma unroll
                for (int c = 0; c < 6; ++c) X[c] = S[k * n + J + c];
#pragma unroll
                for (int c = 0; c < 6; ++c) {
                    double w = X[c];
#pragma unroll
                    for (int q = 0; q < c; ++q) w -= W[q] * P[c][q];
                    W[c] = w;
                    Lc[b][c] = w * rp[c];
                }
            } else {
#pragma unroll
                for (int c = 0; c < 6; ++c) Lc[b][c] = 0.0;
            }
        }
#pragma unroll
        for (int a = 0; a < A; ++a)
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const int i = base + ti + TI * a, k = base + tk + TK * b;
                v[a][b] = (i < n && k <= i) ? S[i * n + k] : 0.0;
            }
#pragma unroll
        for (int a = 0; a < A; ++a)
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const int i = base + ti + TI * a, k = base + tk + TK * b;
                if (i < n && k <= i) {
                    const double s0 = Wr[a][0] * Lc[b][0] + Wr[a][1] * Lc[b][1] + Wr[a][2] * Lc[b][2];
                    const double s1 = Wr[a][3] * Lc[b][3] + Wr[a][4] * Lc[b][4] + Wr[a][5] * Lc[b][5];
                    S[i * n + k] = v[a][b] - (s0 + s1);
                }
            }
        sync();
        // the factor replaces the block column (everybody has read the unscaled values before the barrier)
        if (tk == 0) {
#pragma unroll
            for (int a = 0; a < A; ++a) {
                const int i = base + ti + TI * a;
                if (i < n) {
#pragma unroll
                    for (int c = 0; c < 6; ++c) S[i * n + J + c] = Wr[a][c] * rp[c];
                }
            }
        }
        if (t == 0) {
#pragma unroll
            for (int r = 0; r < 6; ++r) {
#pragma unroll
                for (int c = 0; c <= r; ++c) S[(J + r) * n + J + c] = P[r][c];
                rd[J + r] = rp[r];
            }
        }
    }
    sync();
    return true;
}

// The whole solve of a small system (N = 12: two free poses, the local BA of the tracking loop; N = 6) by ONE lane with the
// lower triangle in registers and every loop unrolled (static indices only): no shuffles, no barriers, no shared-memory round
// trips between dependent steps -- the dependent-FMA latency (8.7 cycles) is the only chain.  Same arithmetic as the scalar
// LDL^T.  x overwrites b; false if a pivot is not positive.
template <int N>
__device__ __forceinline__ bool lane_ldlt_solve(const double* __restrict__ S, double* __restrict__ b) {
    double L[N * (N + 1) / 2], rd[N], z[N];
#define LT(i, j) L[(i) * ((i) + 1) / 2 + (j)]
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = 0; j <= i; ++j) LT(i, j) = S[i * N + j];
        z[i] = b[i];
    }
    bool pd = true;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        const double d = LT(j, j);
        pd = pd && d > 0;
        rd[j] = fast_rcp(d);
        double u[N];
#pragma unroll
        for (int i = j + 1; i < N; ++i) u[i] = LT(i, j);
#pragma unroll
        for (int i = j + 1; i < N; ++i) {
            const double l = u[i] * rd[j];
#pragma unroll
            for (int k = j + 1; k <= i; ++k) LT(i, k) -= l * u[k];
            LT(i, j) = l;
        }
    }
    if (!pd) return false;
#pragma unroll
    for (int i = 1; i < N; ++i) {
        double s = z[i];
#pragma unroll
        for (int k = 0; k < i; ++k) s -= LT(i, k) * z[k];
        z[i] = s;
    }
#pragma unroll
    for (int i = 0; i < N; ++i) z[i] *= rd[i];
#pragma unroll
    for (int i = N - 2; i >= 0; --i) {
        double s = z[i];
#pragma unroll
        for (int k = i + 1; k < N; ++k) s -= LT(k, i) * z[k];
        z[i] = s;
    }
#pragma unroll
    for (int i = 0; i < N; ++i) b[i] = z[i];
#undef LT
    return true;
}

__global__ void __launch_bounds__(kT) local_ba2_kernel(const BA2Args a) {
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(16) double s_dyn[];
    __shared__ double s_Rlin[kBA2MaxPoses][12];   // poses of the accepted state as [R|t] (the Jacobians are rebuilt from these)
    __shared__ double s_Rtry[kBA2MaxPoses][12];   // poses of the trial
    __shared__ SE3d s_T[kBA2MaxPoses];            // accepted poses (the estimate of VertexSE3Sophus is their logarithm)
    __shared__ SE3d s_Ttry[kBA2MaxPoses];         // trial poses
    __shared__ double s_xp[6 * kBA2MaxFree], s_rd[6 * kBA2MaxFree];
    __shared__ double s_tmp[2 * (kW + 1)];
    __shared__ double s_small[4];                 // per-CTA scalars offered to the cluster: chi2, scale, max |diag|, flag
    __shared__ double s_bc[4];                    // cluster totals of the same
    __shared__ int s_free[kBA2MaxPoses], s_kfof[kBA2MaxFree];
    __shared__ int s_np, s_ok, s_dup;
    __shared__ int s_estart[kBA2MaxFree * (kBA2MaxFree + 1) / 2 + 1];   // entry list: first entry of every block pair
    __shared__ int s_gstart[kBA2MaxFree * (kBA2MaxFree + 1) / 2 + kBA2MaxFree + 1];   // first 32-lane work group of every task

    const int rank = (int)cluster.block_rank(), C = (int)cluster.num_blocks();
    const int prob = blockIdx.x / C, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int k0 = a.kf_off[prob], n_kf = a.n_kf ? a.n_kf[prob] : a.kf_off[prob + 1] - k0;
    const int p0 = a.pt_off[prob], n_pt = a.n_pt ? a.n_pt[prob] : a.pt_off[prob + 1] - p0;
    const double fx = a.fx, fy = a.fy, cx = a.cx, cy = a.cy;
    const double dsqr = a.huber_delta * a.huber_delta;

    if (tid == 0) {
        int nf = 0;
        for (int k = 0; k < n_kf; ++k) {
            s_free[k] = a.fixed[k0 + k] ? -1 : nf;
            if (!a.fixed[k0 + k]) s_kfof[nf++] = k;
        }
        s_np = nf;
        s_dup = 0;
    }
    if (tid < n_kf) {
        s_T[tid] = pose_from_g2o(a.poses + 6 * (size_t)(k0 + tid));
        se3_to_mat(s_T[tid], s_Rlin[tid]);
    }
    __syncthreads();
    const int np = s_np, dimp = 6 * np, n_pairs = np * (np + 1) / 2;
    const int V = kPairW * n_pairs + kPoseW * np, poseBase = kPairW * n_pairs;

    // this CTA's landmarks [j_lo, j_hi) and their observations [q_lo, q_hi) of the landmark-major list
    const int per_cta = (n_pt + C - 1) / C;
    const int j_lo = min(n_pt, rank * per_cta), j_hi = min(n_pt, j_lo + per_cta), nl = j_hi - j_lo;
    const int q_lo = a.lm_start[p0 + j_lo], q_hi = a.lm_start[p0 + j_hi], no = q_hi - q_lo;

    // ---- dynamic shared memory: [S | bs] aliased with the task slots, the exchange vectors, then the staging area
    const int n_tasks_all = n_pairs + np;
    const int sysDoubles = max(dimp * dimp + dimp, (n_tasks_all + kW) * kPairW);
    double* s_S = s_dyn;
    double* s_bs = s_S + dimp * dimp;
    double* s_part = s_dyn;                 // (task + warp) slots of kPairW doubles; consumed before S is assembled
    double* s_x = s_dyn + sysDoubles;       // [V] CTA partial, after the exchange the cluster totals
    double* s_tot = s_x + V;                // [V] totals of the slice this CTA owns
    double* s_stage = s_tot + V;
    Stage st;
    {
        const size_t need = ba2_stage_doubles((size_t)nl, (size_t)no);
        const size_t have = (size_t)a.dyn_doubles - (size_t)(sysDoubles + 2 * V);
        // global fall-back: disjoint regions because the size is monotone and 8 extra "landmarks" per preceding CTA cover its rounding
        double* base = need <= have ? s_stage : a.lin + ba2_stage_doubles((size_t)(p0 + j_lo) + 8 * ((size_t)rank + 16 * (size_t)prob), (size_t)q_lo);
        st.lin[0] = base;
        st.lin[1] = st.lin[0] + (size_t)6 * no;
        st.Hll[0] = st.lin[1] + (size_t)6 * no;
        st.Hll[1] = st.Hll[0] + (size_t)6 * nl;
        st.bl[0] = st.Hll[1] + (size_t)6 * nl;
        st.bl[1] = st.bl[0] + (size_t)3 * nl;
        st.X[0] = st.bl[1] + (size_t)3 * nl;
        st.X[1] = st.X[0] + (size_t)3 * nl;
        st.Dinv = st.X[1] + (size_t)3 * nl;
        st.uv = st.Dinv + (size_t)6 * nl;
        st.qa = reinterpret_cast<int32_t*>(st.uv + (size_t)2 * no);
        st.kf = reinterpret_cast<uint8_t*>(st.qa + nl + 1);
        st.slot = st.kf + ((no + 7) & ~7);
        const size_t ent_doubles = (ba2_entry_cap((size_t)nl, (size_t)no, (size_t)np) + 1) / 2;
        st.ent = (need + ent_doubles <= have && nl < 65536) ? reinterpret_cast<uint32_t*>(s_stage + need) : nullptr;
    }
    // slot table: which observation of a landmark sits on which free pose; landmark positions into the staging area
    for (int i = tid; i < nl * kBA2MaxFree; i += kT) st.slot[i] = 0xFF;
    for (int i = tid; i < 3 * nl; i += kT) st.X[0][i] = a.pts[3 * (size_t)(p0 + j_lo) + i];
    for (int i = tid; i < 2 * no; i += kT) st.uv[i] = a.so_uv[2 * (size_t)q_lo + i];
    for (int i = tid; i < no; i += kT) st.kf[i] = (uint8_t)a.so_kf[q_lo + i];
    for (int i = tid; i <= nl; i += kT) st.qa[i] = a.lm_start[p0 + j_lo + i] - q_lo;
    __syncthreads();
    for (int jj = tid; jj < nl; jj += kT) {
        const int qa = a.lm_start[p0 + j_lo + jj], qb = a.lm_start[p0 + j_lo + jj + 1];
        for (int q = qa; q < qb; ++q) {
            const int f = s_free[a.so_kf[q]];
            if (f < 0) continue;
            if (st.slot[jj * kBA2MaxFree + f] != 0xFF || q - qa >= 255) s_dup = 1;   // two observations of a point in one key-frame
            st.slot[jj * kBA2MaxFree + f] = (uint8_t)(q - qa);
        }
    }
    // ---- work list of the reduced system.  With few key-frames per landmark most (landmark, block pair) combinations are empty
    // (C4: a landmark is seen by 4 of 10 key-frames -> 16 % of the lanes of a 32-landmark chunk had work): the non-empty ones are
    // listed once, sorted by block pair (counting sort; inside a pair ascending landmark, so the order is deterministic), and a
    // task's work groups are 32 consecutive entries.  Without room for the list a work group is a 32-landmark chunk.
    __syncthreads();
    const int n_chunks = (nl + 31) / 32;
    auto pair_index = [&](int f1, int f2) { return f1 * np - f1 * (f1 - 1) / 2 + (f2 - f1); };
    if (st.ent) {
        for (int t = tid; t <= n_pairs; t += kT) s_estart[t] = 0;
        __syncthreads();
        for (int jj = tid; jj < nl; jj += kT)
            for (int f1 = 0; f1 < np; ++f1) {
                if (st.slot[jj * kBA2MaxFree + f1] == 0xFF) continue;
                for (int f2 = f1; f2 < np; ++f2)
                    if (st.slot[jj * kBA2MaxFree + f2] != 0xFF) atomicAdd(&s_estart[pair_index(f1, f2) + 1], 1);
            }
        __syncthreads();
        if (tid == 0)
            for (int t = 0; t < n_pairs; ++t) s_estart[t + 1] += s_estart[t];
        __syncthreads();
        for (int f1 = 0, t = 0; f1 < np; ++f1)
            for (int f2 = f1; f2 < np; ++f2, ++t) {
                if (t % kW != warp) continue;
                int pos = s_estart[t];
                for (int base = 0; base < nl; base += 32) {
                    const int jj = base + lane;
                    const int s1 = jj < nl ? st.slot[jj * kBA2MaxFree + f1] : 0xFF, s2 = jj < nl ? st.slot[jj * kBA2MaxFree + f2] : 0xFF;
                    const bool has = s1 != 0xFF && s2 != 0xFF;
                    const unsigned m = __ballot_sync(0xFFFFFFFFu, has);
                    if (has) st.ent[pos + __popc(m & ((1u << lane) - 1u))] = (unsigned)jj | ((unsigned)s1 << 16) | ((unsigned)s2 << 24);
                    pos += __popc(m);
                }
            }
    }
    if (tid == 0) {
        int g = 0;
        for (int t = 0; t < n_pairs + np; ++t) {
            s_gstart[t] = g;
            const int tb = t < n_pairs ? t : pair_index(t - n_pairs, t - n_pairs);
            g += st.ent ? (s_estart[tb + 1] - s_estart[tb] + 31) / 32 : n_chunks;
        }
        s_gstart[n_pairs + np] = g;
    }
    __syncthreads();
    int cur = 0;   // index of the accepted state in the double buffers

    auto robust = [&](double e2, double* w) {   // RobustKernelHuber (delta in pixels, BA.cpp:450-452)
        *w = 1.0;
        if (a.huber_delta > 0 && e2 > dsqr) {
            const double e = sqrt(e2);
            *w = a.huber_delta / e;
            return 2 * e * a.huber_delta - dsqr;
        }
        return e2;
    };
    // cluster totals of the per-CTA scalars in s_small (sum for [0], [1], [3]; max for [2]); contains a cluster barrier
    auto exchange_small = [&]() {
        cluster.sync();
        if (tid == 0) {
            double t0 = 0, t1 = 0, t2 = 0, t3 = 0;
            for (int r = 0; r < C; ++r) {
                const double* rs = cluster.map_shared_rank(s_small, r);
                t0 += rs[0];
                t1 += rs[1];
                t2 = fmax(t2, rs[2]);
                t3 += rs[3];
            }
            s_bc[0] = t0; s_bc[1] = t1; s_bc[2] = t2; s_bc[3] = t3;
        }
        __syncthreads();
    };
    // cluster totals of s_x[lo, hi): reduce-scatter (every CTA sums one slice over the ranks, in rank order) + all-gather
    // over distributed shared memory; two cluster barriers; s_x holds the totals afterwards in every CTA
    auto exchange_vector = [&](int lo, int hi) {
        const int len = hi - lo, sl = (len + C - 1) / C;
        cluster.sync();
        for (int i = lo + rank * sl + tid; i < min(hi, lo + (rank + 1) * sl); i += kT) {
            double t = 0;
            for (int r = 0; r < C; ++r) t += cluster.map_shared_rank(s_x, r)[i];
            s_tot[i] = t;
        }
        cluster.sync();
        for (int i = lo + tid; i < hi; i += kT) s_x[i] = cluster.map_shared_rank(s_tot, (i - lo) / max(sl, 1))[i];
        __syncthreads();
    };

    // ---- linearisation of this CTA's landmarks at (poses R, positions X) into buffer `buf`: the record (x, y, z, e, w) of every
    // observation, Hll and bl of every landmark; returns the CTA-partial robust chi2 and max |diag Hll| per thread
    auto linearise = [&](int buf, const double (*R)[12], const double* X, double* chi_out, double* mx_out) {
        double chi = 0, mx = 0;
        for (int jj = tid; jj < nl; jj += kT) {
            const double X0 = X[3 * jj], X1 = X[3 * jj + 1], X2 = X[3 * jj + 2];
            double H[6] = {0, 0, 0, 0, 0, 0}, b[3] = {0, 0, 0};
            for (int q = q_lo + st.qa[jj]; q < q_lo + st.qa[jj + 1]; ++q) {
                const double* Tm = R[st.kf[q - q_lo]];
                const double x = Tm[0] * X0 + Tm[1] * X1 + Tm[2] * X2 + Tm[3];
                const double y = Tm[4] * X0 + Tm[5] * X1 + Tm[6] * X2 + Tm[7];
                const double z = Tm[8] * X0 + Tm[9] * X1 + Tm[10] * X2 + Tm[11];
                const double iz = 1.0 / z;
                const double e0 = st.uv[2 * (size_t)(q - q_lo)] - (x * iz * fx + cx), e1 = st.uv[2 * (size_t)(q - q_lo) + 1] - (y * iz * fy + cy);
                double w;
                chi += robust(e0 * e0 + e1 * e1, &w);
                double* rec = st.lin[buf] + 6 * (size_t)(q - q_lo);
                rec[0] = x; rec[1] = y; rec[2] = iz; rec[3] = e0; rec[4] = e1; rec[5] = w;
                double l0[3], l1[3];
                point_jac(x, y, iz, fx, fy, Tm, l0, l1);
                H[0] += w * (l0[0] * l0[0] + l1[0] * l1[0]); H[1] += w * (l0[0] * l0[1] + l1[0] * l1[1]);
                H[2] += w * (l0[0] * l0[2] + l1[0] * l1[2]); H[3] += w * (l0[1] * l0[1] + l1[1] * l1[1]);
                H[4] += w * (l0[1] * l0[2] + l1[1] * l1[2]); H[5] += w * (l0[2] * l0[2] + l1[2] * l1[2]);
#pragma unroll
                for (int c = 0; c < 3; ++c) b[c] += -w * (l0[c] * e0 + l1[c] * e1);
            }
#pragma unroll
            for (int t = 0; t < 6; ++t) st.Hll[buf][6 * jj + t] = H[t];
            st.bl[buf][3 * jj] = b[0]; st.bl[buf][3 * jj + 1] = b[1]; st.bl[buf][3 * jj + 2] = b[2];
            mx = fmax(mx, fmax(fabs(H[0]), fmax(fabs(H[3]), fabs(H[5]))));
        }
        *chi_out = chi;
        *mx_out = mx;
    };

    // ---- warp tasks.  Task t < n_pairs: block pair (f1 <= f2) of the reduced system; t >= n_pairs: Hpp / bp of free
    // pose t - n_pairs.  The (task, 32-landmark chunk) items of [t_lo, t_hi) are dealt to the warps in contiguous runs, a
    // warp keeps its sums in registers while the task stays the same and leaves them in slot (task + warp).
    auto accumulate = [&](int t_lo, int t_hi, double lambda) {
        const int g0 = s_gstart[t_lo], items = s_gstart[t_hi] - g0, per = (items + kW - 1) / kW;
        const double* lin = st.lin[cur];
        int it = g0 + warp * per, task = t_lo;
        const int end = min(g0 + items, it + per);
        while (it < end) {
            while (s_gstart[task + 1] <= it) ++task;   // tasks without work groups are skipped (their slots are never read)
            const int c_lo = it - s_gstart[task], c_hi = min(s_gstart[task + 1], end) - s_gstart[task];
            double* out = s_part + (size_t)(task + warp) * kPairW;
            if (task < n_pairs) {
                int f1 = 0, rem = task;
                while (rem >= np - f1) {
                    rem -= np - f1;
                    ++f1;
                }
                const int f2 = f1 + rem;
                const double* R1 = s_Rlin[s_kfof[f1]];
                const double* R2 = s_Rlin[s_kfof[f2]];
                const int e_lo = st.ent ? s_estart[task] : 0, e_hi = st.ent ? s_estart[task + 1] : 0;
                double acc[48];   // [0, 36) the 6 x 6 block, [36, 42) the right-hand side (diagonal pairs), the rest stays zero
                double* accS = acc;
                double* accb = acc + 36;
#pragma unroll
                for (int t = 0; t < 48; ++t) acc[t] = 0;
                for (int ch = c_lo; ch < c_hi; ++ch) {
                    int jj, s1, s2;
                    if (st.ent) {
                        const int idx = e_lo + ch * 32 + lane;
                        if (idx >= e_hi) continue;
                        const unsigned e = st.ent[idx];
                        jj = (int)(e & 0xFFFFu);
                        s1 = (int)((e >> 16) & 0xFFu);
                        s2 = (int)(e >> 24);
                    } else {
                        jj = ch * 32 + lane;
                        if (jj >= nl) continue;
                        s1 = st.slot[jj * kBA2MaxFree + f1];
                        s2 = st.slot[jj * kBA2MaxFree + f2];
                        if (s1 == 0xFF || s2 == 0xFF) continue;
                    }
                    const int qa = st.qa[jj];
                    const double* Di = st.Dinv + 6 * jj;
                    double H1[6][3], BD[6][3];
                    make_hpl(lin + 6 * (size_t)(qa + s1), R1, fx, fy, H1);
#pragma unroll
                    for (int r = 0; r < 6; ++r) sym_mul3(Di, H1[r], BD[r]);   // (Hpl D)_r = D Hpl_r (D symmetric)
                    if (f1 == f2) {
                        const double* bj = st.bl[cur] + 3 * jj;
#pragma unroll
                        for (int r = 0; r < 6; ++r) accb[r] += BD[r][0] * bj[0] + BD[r][1] * bj[1] + BD[r][2] * bj[2];
#pragma unroll
                        for (int r = 0; r < 6; ++r)
#pragma unroll
                            for (int c = 0; c < 6; ++c) accS[r * 6 + c] += BD[r][0] * H1[c][0] + BD[r][1] * H1[c][1] + BD[r][2] * H1[c][2];
                    } else {
                        double H2[6][3];
                        make_hpl(lin + 6 * (size_t)(qa + s2), R2, fx, fy, H2);
#pragma unroll
                        for (int r = 0; r < 6; ++r)
#pragma unroll
                            for (int c = 0; c < 6; ++c) accS[r * 6 + c] += BD[r][0] * H2[c][0] + BD[r][1] * H2[c][1] + BD[r][2] * H2[c][2];
                    }
                }
                {
                    const double lo = warp_reduce_scatter<32>(acc, lane), hi = warp_reduce_scatter<16>(acc + 32, lane);
                    out[lane] = lo;
                    if (!(lane & 1) && 32 + (lane >> 1) < kPairW) out[32 + (lane >> 1)] = hi;
                }
            } else {
                const int f = task - n_pairs, td = pair_index(f, f);
                const int e_lo = st.ent ? s_estart[td] : 0, e_hi = st.ent ? s_estart[td + 1] : 0;
                double acc[32];   // [0, 21) upper triangle of Hpp, [21, 27) bp
                double* h = acc;
                double* g = acc + 21;
#pragma unroll
                for (int t = 0; t < 32; ++t) acc[t] = 0;
                for (int ch = c_lo; ch < c_hi; ++ch) {
                    int jj, s1;
                    if (st.ent) {
                        const int idx = e_lo + ch * 32 + lane;
                        if (idx >= e_hi) continue;
                        const unsigned e = st.ent[idx];
                        jj = (int)(e & 0xFFFFu);
                        s1 = (int)((e >> 16) & 0xFFu);
                    } else {
                        jj = ch * 32 + lane;
                        if (jj >= nl) continue;
                        s1 = st.slot[jj * kBA2MaxFree + f];
                        if (s1 == 0xFF) continue;
                    }
                    const double* rec = lin + 6 * (size_t)(st.qa[jj] + s1);
                    double q0[6], q1[6];
                    pose_jac(rec[0], rec[1], rec[2], fx, fy, q0, q1);
                    const double w = rec[5];
                    int t = 0;
#pragma unroll
                    for (int r = 0; r < 6; ++r) {
#pragma unroll
                        for (int c = r; c < 6; ++c) h[t++] += w * (q0[r] * q0[c] + q1[r] * q1[c]);
                        g[r] += -w * (q0[r] * rec[3] + q1[r] * rec[4]);
                    }
                }
                {
                    const double tot = warp_reduce_scatter<32>(acc, lane);
                    if (lane < kPoseW) out[lane] = tot;
                }
            }
            it += c_hi - c_lo;
        }
        __syncthreads();
        // slots -> CTA partial vector: the warps that worked on a task are a contiguous range, added in warp order
        for (int i = tid; i < (t_hi - t_lo) * kPairW; i += kT) {
            const int trel = i / kPairW, e = i - trel * kPairW, tk = t_lo + trel;
            const bool pose = tk >= n_pairs;
            if (pose && e >= kPoseW) continue;
            double v = 0;
            const int ga = s_gstart[tk] - g0, gb = s_gstart[tk + 1] - g0;
            if (per > 0 && gb > ga) {
                const int w_lo = ga / per, w_hi = min(kW - 1, (gb - 1) / per);
                for (int w = w_lo; w <= w_hi; ++w) v += s_part[(size_t)(tk + w) * kPairW + e];
            }
            s_x[pose ? poseBase + (tk - n_pairs) * kPoseW + e : tk * kPairW + e] = v;
        }
        __syncthreads();
    };

    // ---- prologue: first linearisation, lambda_0 = tau * max |diag H| (computeLambdaInit) ------------------------------
    __syncthreads();
    int iters = 0, trials_total = 0;
    double chi_first = 0, chi_last = 0, lambda = 0, ni = 2, rho = 0, currentChi = 0;
    {
        double chi, mx;
        linearise(0, s_Rlin, st.X[0], &chi, &mx);
        double dummy = 0;
        block_sum2(chi, dummy, s_tmp);
        mx = block_max(mx, s_tmp);
        accumulate(n_pairs, n_pairs + np, 0.0);
        exchange_vector(poseBase, V);
        if (tid == 0) {
            s_small[0] = chi;
            s_small[1] = 0;
            s_small[2] = mx;
            s_small[3] = s_dup;
        }
        exchange_small();
        currentChi = chi_first = chi_last = s_bc[0];
        double m0 = s_bc[2];
        for (int f = 0; f < np; ++f) {
            const double* h = s_x + poseBase + f * kPoseW;
            const int diag[6] = {0, 6, 11, 15, 18, 20};
            for (int c = 0; c < 6; ++c) m0 = fmax(m0, fabs(h[diag[c]]));
        }
        lambda = a.tau * m0;
    }
    const bool dup = s_bc[3] > 0;   // unsupported input: reported through stats, nothing is optimised

    // optional phase timing (a.debug != null): cycles of CTA 0 / thread 0 per phase, summed over the trials
    long long tph[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tlast = clock64();
    auto tick = [&](int ph) {
        if (a.debug) {
            const long long now = clock64();
            tph[ph] += now - tlast;
            tlast = now;
        }
    };
    bool fresh = false;   // Hpp / bp of the accepted state are in s_x (the prologue computed them for iteration 0)
    for (int iteration = 0; iteration < a.max_iters && !dup; ++iteration) {
        int qmax = 0;
        do {
            // ---- reduced system of the accepted state at the current lambda: (Hll + lambda I)^-1 is rebuilt per use
            tick(6);
            for (int jj = tid; jj < nl; jj += kT) sym_inverse3(st.Hll[cur] + 6 * jj, lambda, st.Dinv + 6 * jj);
            __syncthreads();
            accumulate(0, fresh ? n_pairs + np : n_pairs, lambda);
            tick(0);
            exchange_vector(0, fresh ? V : poseBase);
            tick(1);
            fresh = false;
            // S = Hpp + lambda I - sum Hpl D Hpl^T, b_s = bp - sum Hpl D bl (every CTA: same bits)
            for (int i = tid; i < dimp * dimp; i += kT) {
                const int r = i / dimp, c = i - r * dimp, fr = r / 6, fc = c / 6, rr = r - 6 * fr, cc = c - 6 * fc;
                double v;
                if (fr <= fc) v = -s_x[(fr * np - fr * (fr - 1) / 2 + (fc - fr)) * kPairW + rr * 6 + cc];
                else v = -s_x[(fc * np - fc * (fc - 1) / 2 + (fr - fc)) * kPairW + cc * 6 + rr];
                if (fr == fc) {
                    const int lo = min(rr, cc), hi = max(rr, cc);
                    v += s_x[poseBase + fr * kPoseW + (lo * 6 - lo * (lo - 1) / 2 + (hi - lo))] + (r == c ? lambda : 0.0);
                }
                s_S[i] = v;
            }
            if (tid < dimp) {
                const int f = tid / 6, r = tid - 6 * f;
                s_bs[tid] = s_x[poseBase + f * kPoseW + 21 + r] - s_x[(f * np - f * (f - 1) / 2) * kPairW + 36 + r];
            }
            __syncthreads();
            tick(2);
            // ---- dense LDL^T + triangular solves (small systems: warp 0 alone; larger ones: factorisation by the whole CTA),
            // then VertexSE3Sophus::oplusImpl for the trial poses
            if (a.solver == 0 && dimp > kCtaSolveMinDim) {
                // (more than 11 free poses: the scalar version; its 6 x 6 tile per thread would not fit the registers in block form)
                const bool ok = dimp <= 70 ? ldlt6_factor<16, 16, 4, 4, true>(s_S, s_rd, dimp, tid)
                                           : ldlt_factor_rl<16, 16, 6, 6, true>(s_S, s_rd, dimp, tid);
                tick(7);
                if (warp == 0) {
                    if (ok) warp_ldlt_subst(s_S, s_bs, s_rd, dimp, lane);
                    if (lane == 0) s_ok = ok ? 1 : 0;
                    for (int i = lane; i < dimp; i += 32) s_xp[i] = ok ? s_bs[i] : 0.0;
                }
            } else if (a.solver == 0 && warp == 0 && (dimp == 12 || dimp == 6)) {
                // one or two free poses (the local BA of the tracking loop): one lane, everything in registers -- measured in
                // isolation (tools/microbench_ldlt.cu) 2.1k cycles against 8.0k for the warp version (4.6k block factorisation +
                // 3.4k substitution, each dependent step paying a shuffle or a shared-memory round trip)
                bool ok = true;
                if (lane == 0) ok = dimp == 12 ? lane_ldlt_solve<12>(s_S, s_bs) : lane_ldlt_solve<6>(s_S, s_bs);
                ok = __shfl_sync(0xFFFFFFFFu, ok ? 1 : 0, 0) != 0;
                tick(7);
                if (lane == 0) s_ok = ok ? 1 : 0;
                __syncwarp();
                for (int i = lane; i < dimp; i += 32) s_xp[i] = ok ? s_bs[i] : 0.0;
            } else if (a.solver == 0 && warp == 0 && dimp > 0) {
                const bool ok = ldlt6_factor<4, 8, 5, 3, false>(s_S, s_rd, dimp, lane);
                tick(7);
                if (ok) warp_ldlt_subst(s_S, s_bs, s_rd, dimp, lane);
                if (lane == 0) s_ok = ok ? 1 : 0;
                for (int i = lane; i < dimp; i += 32) s_xp[i] = ok ? s_bs[i] : 0.0;
            } else if (a.solver == 0) {
                if (warp == 0 && lane == 0) s_ok = 1;   // no free pose: nothing to solve
            } else if (dimp > kCtaSolveMinDim) {
                const bool ok = dimp <= 64 ? ldlt_factor_rl<16, 16, 4, 4, true>(s_S, s_rd, dimp, tid)
                                           : ldlt_factor_rl<16, 16, 6, 6, true>(s_S, s_rd, dimp, tid);
                tick(7);
                if (warp == 0) {
                    if (ok) warp_ldlt_subst(s_S, s_bs, s_rd, dimp, lane);
                    if (lane == 0) s_ok = ok ? 1 : 0;
                    for (int i = lane; i < dimp; i += 32) s_xp[i] = ok ? s_bs[i] : 0.0;
                }
            } else if (warp == 0 && dimp > 0) {
                const bool ok = ldlt_factor_rl<4, 8, 6, 3, false>(s_S, s_rd, dimp, lane);
                tick(7);
                if (ok) warp_ldlt_subst(s_S, s_bs, s_rd, dimp, lane);
                if (lane == 0) s_ok = ok ? 1 : 0;
                for (int i = lane; i < dimp; i += 32) s_xp[i] = ok ? s_bs[i] : 0.0;
            } else if (warp == 0) {   // no free pose: nothing to solve
                if (lane == 0) s_ok = 1;
            }
            __syncthreads();
            const bool ok2 = s_ok != 0;
            tick(3);
            double chi_part = 0, scale = 0;
            if (warp == 0) {
                for (int k = lane; k < n_kf; k += 32) {
                    if (s_free[k] >= 0) {
                        // VertexSE3Sophus::oplusImpl: estimate <- log(exp(update) * exp(estimate)); the replica keeps the group
                        // element itself (the logarithm is taken once, for the result), which skips a log / exp round trip per trial
                        const double* u = s_xp + 6 * s_free[k];
                        const double v[6] = {u[3], u[4], u[5], u[0], u[1], u[2]};
                        s_Ttry[k] = se3_mul(se3_exp(v), s_T[k]);
                        se3_to_mat(s_Ttry[k], s_Rtry[k]);
                    } else {
                        s_Ttry[k] = s_T[k];
                        for (int c = 0; c < 12; ++c) s_Rtry[k][c] = s_Rlin[k][c];
                    }
                }
                if (rank == 0)
                    for (int i = lane; i < dimp; i += 32) {
                        const int f = i / 6, rr = i - 6 * f;
                        scale += s_xp[i] * (lambda * s_xp[i] + s_x[poseBase + f * kPoseW + 21 + rr]);
                    }
            } else {
                // ---- the other warps meanwhile: landmark back-substitution, trial positions, gain-ratio denominator
                for (int jj = tid - 32; jj < nl; jj += kT - 32) {
                    const double* bj = st.bl[cur] + 3 * jj;
                    double r[3] = {bj[0], bj[1], bj[2]};
                    for (int q = st.qa[jj]; q < st.qa[jj + 1]; ++q) {
                        const int kf = st.kf[q], fi = s_free[kf];
                        if (fi < 0) continue;
                        double H1[6][3];
                        make_hpl(st.lin[cur] + 6 * (size_t)q, s_Rlin[kf], fx, fy, H1);
#pragma unroll
                        for (int c = 0; c < 3; ++c)
#pragma unroll
                            for (int rr = 0; rr < 6; ++rr) r[c] -= H1[rr][c] * s_xp[6 * fi + rr];
                    }
                    double xl[3];
                    sym_mul3(st.Dinv + 6 * jj, r, xl);
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        scale += xl[c] * (lambda * xl[c] + bj[c]);
                        st.X[cur ^ 1][3 * jj + c] = st.X[cur][3 * jj + c] + xl[c];
                    }
                }
            }
            __syncthreads();
            tick(4);
            // ---- chi2 at the trial point = linearisation of the next iteration if the step is accepted
            {
                double mx;
                linearise(cur ^ 1, s_Rtry, st.X[cur ^ 1], &chi_part, &mx);
            }
            tick(5);
            block_sum2(chi_part, scale, s_tmp);
            if (tid == 0) {
                s_small[0] = chi_part;
                s_small[1] = scale;
                s_small[2] = 0;
                s_small[3] = 0;
            }
            exchange_small();
            tick(6);
            double tempChi = s_bc[0];
            const double scale_tot = s_bc[1] + 1e-3;
            if (!ok2) tempChi = 1.7976931348623157e308;
            rho = (currentChi - tempChi) / scale_tot;
            if (rho > 0 && isfinite(tempChi)) {
                const double t2 = 2 * rho - 1;
                double alpha = 1. - t2 * t2 * t2;
                alpha = fmin(alpha, 2. / 3.);
                lambda *= fmax(1. / 3., alpha);
                ni = 2;
                currentChi = tempChi;
                // the trial becomes the accepted state: swap the double buffers, take over the poses
                cur ^= 1;
                fresh = true;
                if (tid < n_kf) {
                    s_T[tid] = s_Ttry[tid];
                    for (int c = 0; c < 12; ++c) s_Rlin[tid][c] = s_Rtry[tid][c];
                }
                __syncthreads();
            } else {   // _optimizer->pop(): the accepted state was never touched
                lambda *= ni;
                ni *= 2;
            }
            ++qmax;
            ++trials_total;
        } while (rho < 0 && qmax < a.max_trials);
        ++iters;
        chi_last = currentChi;
        if (qmax == a.max_trials || rho == 0) break;
    }
    // ---- results: landmark positions, outlier flags (BA.cpp:505-515: plain chi2 > 5.991 at the final estimate), poses
    cluster.sync();   // the last exchange_small may still be read by a neighbour: s_small is rewritten below
    double n_out = 0, zero = 0;
    for (int jj = tid; jj < nl; jj += kT) {
        const int gj = p0 + j_lo + jj;
        for (int c = 0; c < 3; ++c) a.pts[3 * (size_t)gj + c] = st.X[cur][3 * jj + c];
        for (int q = q_lo + st.qa[jj]; q < q_lo + st.qa[jj + 1]; ++q) {
            const double* rec = st.lin[cur] + 6 * (size_t)(q - q_lo);
            const int out = (rec[3] * rec[3] + rec[4] * rec[4] > a.chi2_outlier) ? 1 : 0;
            a.outlier[a.so_orig ? a.so_orig[q] : q] = (uint8_t)out;
            n_out += out;
        }
    }
    block_sum2(n_out, zero, s_tmp);
    if (tid == 0) {
        s_small[0] = n_out;
        s_small[1] = s_small[2] = s_small[3] = 0;
    }
    exchange_small();
    if (rank == 0) {
        if (tid < n_kf && s_free[tid] >= 0) {   // fixed vertices keep their input bits
            double lg[6];
            se3_log(s_T[tid], lg);
            double* o = a.poses + 6 * (size_t)(k0 + tid);
            o[0] = lg[3]; o[1] = lg[4]; o[2] = lg[5]; o[3] = lg[0]; o[4] = lg[1]; o[5] = lg[2];
        }
        if (tid == 0) {
            double* stt = a.stats + 8 * (size_t)prob;
            stt[0] = iters; stt[1] = trials_total; stt[2] = chi_first; stt[3] = chi_last; stt[4] = lambda; stt[5] = s_bc[0];
            stt[6] = dup ? 1.0 : 0.0; stt[7] = 0;
            if (a.debug)
                for (int k = 0; k < 8; ++k) a.debug[8 * (size_t)prob + k] = (double)tph[k];
        }
    }
    cluster.sync();   // no CTA may exit while another still reads its shared memory
}

// ---- landmark-major observation lists built on the device ---------------------------------------------------------
__global__ void csr_count_kernel(int n_problems, const int32_t* __restrict__ obs_off, const int32_t* __restrict__ pt_off,
                                 const int32_t* __restrict__ pt_idx, int32_t* __restrict__ cnt) {
    const int p = blockIdx.y;
    const int o0 = obs_off[p], no = obs_off[p + 1] - o0;
    for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < no; o += gridDim.x * blockDim.x) atomicAdd(&cnt[pt_off[p] + pt_idx[o0 + o]], 1);
}

// one CTA per problem: exclusive scan of the counts -> lm_start, scatter of the observation ids, sort of every landmark's
// short list by original id (deterministic order), gather of (pose index, pixel)
__global__ void __launch_bounds__(1024) csr_build_kernel(const int32_t* __restrict__ obs_off, const int32_t* __restrict__ pt_off,
                                                         const int32_t* __restrict__ kf_idx, const int32_t* __restrict__ pt_idx,
                                                         const double* __restrict__ obs, int32_t* __restrict__ cnt,
                                                         int32_t* __restrict__ lm_start, int32_t* __restrict__ so_orig,
                                                         int32_t* __restrict__ so_kf, double* __restrict__ so_uv, int last) {
    __shared__ int s_scan[1024];
    __shared__ int s_carry;
    const int p = blockIdx.x, tid = threadIdx.x;
    const int o0 = obs_off[p], no = obs_off[p + 1] - o0, p0 = pt_off[p], npt = pt_off[p + 1] - p0;
    if (tid == 0) s_carry = o0;
    __syncthreads();
    for (int base = 0; base < npt; base += 1024) {
        const int j = base + tid;
        const int c = j < npt ? cnt[p0 + j] : 0;
        s_scan[tid] = c;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {   // Hillis-Steele inclusive scan
            const int v = tid >= o ? s_scan[tid - o] : 0;
            __syncthreads();
            s_scan[tid] += v;
            __syncthreads();
        }
        const int start = s_carry + s_scan[tid] - c;
        if (j < npt) {
            lm_start[p0 + j] = start;
            cnt[p0 + j] = start;   // becomes the fill cursor
        }
        __syncthreads();
        if (tid == 1023) s_carry += s_scan[1023];
        __syncthreads();
    }
    // end of the problem's last list; for all but the last problem this is also the first start of the next problem (same
    // value, written by both CTAs)
    if (tid == 0) lm_start[p0 + npt] = o0 + no;
    (void)last;
    for (int o = tid; o < no; o += 1024) so_orig[atomicAdd(&cnt[p0 + pt_idx[o0 + o]], 1)] = o0 + o;
    __syncthreads();
    for (int j = tid; j < npt; j += 1024) {
        const int qa = lm_start[p0 + j], qb = cnt[p0 + j];   // the cursor ended at the end of the list
        for (int i = qa + 1; i < qb; ++i) {
            const int v = so_orig[i];
            int k = i - 1;
            while (k >= qa && so_orig[k] > v) {
                so_orig[k + 1] = so_orig[k];
                --k;
            }
            so_orig[k + 1] = v;
        }
        for (int i = qa; i < qb; ++i) {
            const int o = so_orig[i];
            so_kf[i] = kf_idx[o];
            so_uv[2 * (size_t)i] = obs[2 * (size_t)o];
            so_uv[2 * (size_t)i + 1] = obs[2 * (size_t)o + 1];
        }
    }
}

}  // namespace

size_t ba2_scratch_bytes(size_t NP, size_t NO, size_t P) {
    Carver sz(nullptr);
    sz.take<int32_t>(NP + 1); sz.take<int32_t>(NP + 1); sz.take<int32_t>(NO); sz.take<int32_t>(NO); sz.take<double>(2 * NO);
    sz.take<double>(ba2_stage_doubles(NP + 8 * 16 * P, NO));   // global fall-back of the staging areas (+ per-CTA rounding slack)
    sz.take<uint8_t>(NP * kBA2MaxFree); sz.take<uint8_t>(NO); sz.take<double>(8 * P); sz.take<double>(8 * P);
    return sz.bytes();
}

// Device-to-device entry: everything in `in` is a device pointer.  Builds the landmark-major lists, runs the cluster
// kernel, leaves poses / pts / outlier / stats on the device.  max_pts / max_free bound the problems of the batch.
int launch_local_ba2(ygzb_ctx* ctx, const BA2Problem& in, void* scratch, const ygzb_ba_params* prm, uint8_t** d_outlier_out,
                     double** d_stats_out) {
    const size_t P = (size_t)in.n_problems, NP = in.total_pts, NO = in.total_obs;
    Carver c(scratch);
    int32_t* d_cnt = c.take<int32_t>(NP + 1);
    int32_t* d_lm_start = c.take<int32_t>(NP + 1);
    int32_t* d_so_orig = c.take<int32_t>(NO);
    int32_t* d_so_kf = c.take<int32_t>(NO);
    double* d_so_uv = c.take<double>(2 * NO);
    BA2Args a;
    a.lin = c.take<double>(ba2_stage_doubles(NP + 8 * 16 * P, NO));   // global fall-back of the CTA-private staging areas
    a.slot = c.take<uint8_t>(NP * kBA2MaxFree);
    a.outlier = c.take<uint8_t>(NO);
    a.stats = c.take<double>(8 * P);
    a.debug = getenv("YGZB_BA_DEBUG") ? c.take<double>(8 * P) : nullptr;
    {
        const char* e = getenv("YGZB_BA_SOLVER");
        a.solver = e && atoi(e) == 1 ? 1 : 0;
    }
    if (in.lm_start) {   // the caller already has landmark-major lists (the tracking engine builds them itself)
        a.lm_start = in.lm_start; a.so_kf = in.kf_idx; a.so_uv = in.obs; a.so_orig = nullptr;
    } else {
        YGZB_CUDA(ctx, cudaMemsetAsync(d_cnt, 0, (NP + 1) * sizeof(int32_t), ctx->stream));
        if (NO) {
            ProfScope ps(ctx, kStageOther);
            const dim3 grid((unsigned)std::min<size_t>((in.max_obs + 255) / 256, 64), (unsigned)P);
            csr_count_kernel<<<grid, 256, 0, ctx->stream>>>((int)P, in.obs_off, in.pt_off, in.pt_idx, d_cnt);
            YGZB_LAUNCHED(ctx);
        }
        {
            ProfScope ps(ctx, kStageOther);
            csr_build_kernel<<<(unsigned)P, 1024, 0, ctx->stream>>>(in.obs_off, in.pt_off, in.kf_idx, in.pt_idx, in.obs, d_cnt, d_lm_start,
                                                                    d_so_orig, d_so_kf, d_so_uv, (int)P - 1);
            YGZB_LAUNCHED(ctx);
        }
        a.lm_start = d_lm_start; a.so_kf = d_so_kf; a.so_uv = d_so_uv; a.so_orig = d_so_orig;
    }
    a.kf_off = in.kf_off; a.pt_off = in.pt_off; a.obs_off = in.obs_off;
    a.n_kf = in.n_kf; a.n_pt = in.n_pt;
    a.poses = in.poses; a.fixed = in.fixed; a.pts = in.pts;
    a.fx = ctx->prm.fx; a.fy = ctx->prm.fy; a.cx = ctx->prm.cx; a.cy = ctx->prm.cy;
    a.max_iters = prm->max_iters; a.max_trials = prm->max_trials; a.huber_delta = prm->huber_delta;
    a.chi2_outlier = prm->chi2_outlier; a.tau = prm->tau;

    // cluster size: ~300 landmarks per CTA keep a problem's per-landmark state in shared memory and its FP64 work spread
    int cluster = 1;
    while (cluster < 8 && in.max_pts > (size_t)cluster * 320) cluster *= 2;
    {   // many block pairs (free poses) per landmark chunk: the warp tasks of the reduced system dominate a trial, and their
        // number per warp is (pairs + poses) * chunks / warps -- spread such problems over a 16-CTA cluster (non-portable size)
        const size_t tasks = (size_t)std::max(in.max_free, 0) * (std::max(in.max_free, 0) + 1) / 2 + std::max(in.max_free, 0);
        auto items_per_warp = [&](int c) { return tasks * (((in.max_pts + c - 1) / c + 31) / 32) / (kT / 32); };
        while (cluster < 16 && items_per_warp(cluster) > 24) cluster *= 2;
    }
    if (const char* e = getenv("YGZB_BA_CLUSTER")) {   // tuning knob: 1, 2, 4 or 8
        const int v = atoi(e);
        if (v == 1 || v == 2 || v == 4 || v == 8 || v == 16) cluster = v;
    }
    if (cluster > 8) cudaFuncSetAttribute(local_ba2_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    const int np = std::max(in.max_free, 0), dimp = 6 * np, n_pairs = np * (np + 1) / 2;
    const int V = kPairW * n_pairs + kPoseW * np;
    const size_t sys = std::max<size_t>((size_t)dimp * dimp + dimp, (size_t)(n_pairs + np + kW) * kPairW);
    const size_t nl = (in.max_pts + cluster - 1) / cluster;
    const size_t no = std::min<size_t>(in.max_obs, nl * (size_t)std::max(in.max_kf, 1));
    const size_t stage = ba2_stage_doubles(nl, no) + 2 + (ba2_entry_cap(nl, no, (size_t)np) + 1) / 2;   // + the block-pair entry list
    static int max_optin = 0;
    static std::once_flag once;
    std::call_once(once, [&] {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        cudaFuncSetAttribute(local_ba2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - 24 * 1024);
    });
    const size_t cap = (size_t)std::max(0, max_optin - 24 * 1024) / sizeof(double);   // the kernel's static arrays use ~22 KB
    if (sys + 2 * (size_t)V > cap) return set_error(ctx, YGZB_ERR_CAPACITY, "local BA: %d free poses do not fit shared memory", np);
    const size_t dyn = std::min(cap, sys + 2 * (size_t)V + stage);
    a.dyn_doubles = (long long)dyn;

    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(P * cluster));
    cfg.blockDim = dim3(kT);
    cfg.dynamicSmemBytes = dyn * sizeof(double);
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    {
        ProfScope ps(ctx, kStageLocalBA);
        YGZB_CUDA(ctx, cudaLaunchKernelEx(&cfg, local_ba2_kernel, a));
    }
    YGZB_LAUNCHED(ctx);
    if (a.debug) {   // YGZB_BA_DEBUG: phase cycles of problem 0 (blocking; diagnostics only)
        double h[16];
        double hs[8];
        cudaStreamSynchronize(ctx->stream);
        cudaMemcpy(h, a.debug, sizeof(double) * 8, cudaMemcpyDeviceToHost);
        cudaMemcpy(hs, a.stats, sizeof(double) * 8, cudaMemcpyDeviceToHost);
        fprintf(stderr, "[ba2] P=%zu cluster=%d iters=%.0f trials=%.0f cycles/trial: accumulate %.0f exchange %.0f assemble %.0f substitution %.0f "
                        "pose+backsubst %.0f linearise %.0f reduce+exchange+decide %.0f factorisation %.0f\n",
                P, cluster, hs[0], hs[1], h[0] / hs[1], h[1] / hs[1], h[2] / hs[1], h[3] / hs[1], h[4] / hs[1], h[5] / hs[1], h[6] / hs[1],
                h[7] / hs[1]);
    }
    if (d_outlier_out) *d_outlier_out = a.outlier;
    if (d_stats_out) *d_stats_out = a.stats;
    return YGZB_OK;
}

}  // namespace ygzb
