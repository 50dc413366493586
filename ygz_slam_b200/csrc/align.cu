// align.cu -- 8x8 patch alignment, direct projection (affine warp + alignment) and SVO-style sparse
// image alignment.  Compiled with -fmad=false: every f32/f64 operation below is evaluated exactly as
// written, in the reference's order, so the per-patch results are bit-identical to an unfused CPU build.
//
// Replaces:
//   cvutils::Align2D                     reference src/Algorithm/CVUtils.cpp:186-318
//   cvutils::GetBilateralInterpUchar     reference include/ygz/Algorithm/CVUtils.h:59-71
//   Matcher::FindDirectProjection        reference src/Algorithm/Matcher.cpp:356-417
//   Matcher::GetWarpAffineMatrix         reference src/Algorithm/Matcher.cpp:420-436  (incl. the world/ref-camera mix-up)
//   Matcher::WarpAffine                  reference src/Algorithm/Matcher.cpp:438-466
//   Matcher::GetBestSearchLevel          reference include/ygz/Algorithm/Matcher.h:123-134
//   SparseImgAlign::{run,precomputeReferencePatches,computeResiduals,solve,update}
//                                        reference src/Algorithm/SparseImageAlign.cpp:21-238
//   NLLSSolver::optimizeGaussNewton      reference include/ygz/Algorithm/NLSSolver_impl.hpp:16-88
//   cvutils::JacobXYZ2Cam                reference include/ygz/Algorithm/CVUtils.h:77-99
//
// Parallel mapping
//   Align2D / FindDirectProjection: ONE THREAD PER PATCH.  The inverse-compositional loop is a chain of
//     sequential f32 sums whose rounding decides the convergence flag; keeping the reference's summation
//     order makes (u, v, ok) bit-exact.  A patch touches <= 1 kB, so thousands of patches per launch keep
//     the SMs busy through thread-level parallelism (latency-bound, L1/L2-resident; HBM traffic negligible).
//   SparseImgAlign: ONE CTA PER (ref, cur) PAIR, the whole coarse-to-fine Gauss-Newton loop runs on the
//     device (no host round trip per iteration): threads stride over features, 16 residuals each; the
//     6x6 normal equations (21 + 6 doubles) are reduced with warp shuffles + shared memory; thread 0
//     solves LDL^T and applies T <- T * exp(-x).
#include <algorithm>
#include <cstdlib>
#include <mutex>

#include <cooperative_groups.h>

#include "common.cuh"
#include "se3.cuh"
#include "track.cuh"

namespace ygzb {

namespace {

struct LevelImg {
    const uint8_t* d;
    int w, h, pitch;
};

__device__ __forceinline__ LevelImg level_img(const uint8_t* pyr, size_t slot_stride, int slot, const Geometry& g, int L) {
    return LevelImg{pyr + (size_t)slot * slot_stride + g.lv[L].off, g.lv[L].w, g.lv[L].h, g.lv[L].pitch};
}

// Eigen's fixed-size 3x3 inverse: cofactors, determinant from column 0, multiply by 1/det
__device__ void inverse3f(const float H[3][3], float inv[3][3]) {
#define COF(i, j) (H[(i + 1) % 3][(j + 1) % 3] * H[(i + 2) % 3][(j + 2) % 3] - H[(i + 1) % 3][(j + 2) % 3] * H[(i + 2) % 3][(j + 1) % 3])
    const float c00 = COF(0, 0), c10 = COF(1, 0), c20 = COF(2, 0);
    const float det = (c00 * H[0][0] + c10 * H[1][0]) + c20 * H[2][0];
    const float invdet = 1.0f / det;
    inv[0][0] = c00 * invdet; inv[0][1] = c10 * invdet; inv[0][2] = c20 * invdet;
    inv[1][0] = COF(0, 1) * invdet; inv[1][1] = COF(1, 1) * invdet; inv[1][2] = COF(2, 1) * invdet;
    inv[2][0] = COF(0, 2) * invdet; inv[2][1] = COF(1, 2) * invdet; inv[2][2] = COF(2, 2) * invdet;
#undef COF
}

// cvutils::Align2D.  pwb = 10x10 template with border, ref = 8x8 template.  Returns success.
__device__ bool align2d_dev(const LevelImg& im, const uint8_t* __restrict__ pwb, const uint8_t* __restrict__ ref, int n_iter,
                            double* pu, double* pv) {
    const int halfpatch = 4, patch = 8, ref_step = 10;
    bool converged = false;
    float H[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    for (int y = 0; y < patch; ++y) {
        const uint8_t* it = pwb + (y + 1) * ref_step + 1;
        for (int x = 0; x < patch; ++x, ++it) {
            float J[3];
            J[0] = (float)(0.5 * ((int)it[1] - (int)it[-1]));
            J[1] = (float)(0.5 * ((int)it[ref_step] - (int)it[-ref_step]));
            J[2] = 1.f;
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int b = 0; b < 3; ++b) H[a][b] += J[a] * J[b];
        }
    }
    float Hinv[3][3];
    inverse3f(H, Hinv);
    float mean_diff = 0.f;
    float u = (float)*pu, v = (float)*pv;
    const float min_update_squared = (float)(0.03 * 0.03);
    float chi2 = 0.f;
    for (int iter = 0; iter < n_iter; ++iter) {
        chi2 = 0.f;
        const int u_r = (int)floorf(u), v_r = (int)floorf(v);
        if (u_r < halfpatch || v_r < halfpatch || u_r >= im.w - halfpatch || v_r >= im.h - halfpatch) break;
        if (isnan(u) || isnan(v)) return false;
        const float sx = u - (float)u_r, sy = v - (float)v_r;
        const float wTL = (float)((1.0 - sx) * (1.0 - sy));
        const float wTR = (float)(sx * (1.0 - sy));
        const float wBL = (float)((1.0 - sx) * sy);
        const float wBR = sx * sy;
        float J0 = 0.f, J1 = 0.f, J2 = 0.f;
        for (int y = 0; y < patch; ++y) {
            const uint8_t* it = im.d + (size_t)(v_r + y - halfpatch) * im.pitch + (u_r - halfpatch);
            const uint8_t* tb = pwb + (y + 1) * ref_step + 1;
#pragma unroll
            for (int x = 0; x < patch; ++x) {
                const float search_pixel = wTL * (float)it[x] + wTR * (float)it[x + 1] + wBL * (float)it[x + im.pitch] +
                                           wBR * (float)it[x + im.pitch + 1];
                const float res = search_pixel - (float)ref[y * patch + x] + mean_diff;
                const float dx = (float)(0.5 * ((int)tb[x + 1] - (int)tb[x - 1]));
                const float dy = (float)(0.5 * ((int)tb[x + ref_step] - (int)tb[x - ref_step]));
                J0 -= res * dx;
                J1 -= res * dy;
                J2 -= res;
                chi2 += res * res;
            }
        }
        const float up0 = (Hinv[0][0] * J0 + Hinv[0][1] * J1) + Hinv[0][2] * J2;
        const float up1 = (Hinv[1][0] * J0 + Hinv[1][1] * J1) + Hinv[1][2] * J2;
        const float up2 = (Hinv[2][0] * J0 + Hinv[2][1] * J1) + Hinv[2][2] * J2;
        u += up0;
        v += up1;
        mean_diff += up2;
        if (up0 * up0 + up1 * up1 < min_update_squared) {
            converged = true;
            break;
        }
    }
    *pu = (double)u;
    *pv = (double)v;
    return converged && chi2 < 20000.f;
}

__global__ void __launch_bounds__(128) align2d_kernel(const uint8_t* __restrict__ pyr, size_t slot_stride, Geometry g, int n,
                                                      const int32_t* __restrict__ slot, const uint8_t* __restrict__ level,
                                                      const uint8_t* __restrict__ ref_border, const uint8_t* __restrict__ ref,
                                                      int n_iter, double* __restrict__ uv, uint8_t* __restrict__ ok) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t pwb[100], rp[64];
    for (int k = 0; k < 100; ++k) pwb[k] = ref_border[(size_t)i * 100 + k];
    if (ref) {
        for (int k = 0; k < 64; ++k) rp[k] = ref[(size_t)i * 64 + k];
    } else {
        for (int y = 1; y < 9; ++y)
            for (int x = 0; x < 8; ++x) rp[(y - 1) * 8 + x] = pwb[y * 10 + 1 + x];
    }
    const LevelImg im = level_img(pyr, slot_stride, slot[i], g, level[i]);
    double u = uv[2 * i], v = uv[2 * i + 1];
    const bool s = align2d_dev(im, pwb, rp, n_iter, &u, &v);
    uv[2 * i] = u;
    uv[2 * i + 1] = v;
    ok[i] = s ? 1 : 0;
}

// cvutils::Align1D (reference src/Algorithm/CVUtils.cpp:64-184): 1-D search along `dir` (epipolar direction)
__device__ bool align1d_dev(const LevelImg& im, float dirx, float diry, const uint8_t* __restrict__ pwb, const uint8_t* __restrict__ ref,
                            int n_iter, double* pu, double* pv, double* h_inv) {
    const int halfpatch = 4, patch = 8, ref_step = 10;
    bool converged = false;
    float H00 = 0.f, H01 = 0.f, H10 = 0.f, H11 = 0.f;
    for (int y = 0; y < patch; ++y) {
        const uint8_t* it = pwb + (y + 1) * ref_step + 1;
        for (int x = 0; x < patch; ++x, ++it) {
            const float J0 = (float)(0.5 * (dirx * (float)((int)it[1] - (int)it[-1]) + diry * (float)((int)it[ref_step] - (int)it[-ref_step])));
            H00 += J0 * J0;
            H01 += J0 * 1.f;
            H10 += 1.f * J0;
            H11 += 1.f;
        }
    }
    *h_inv = 1.0 / H00 * patch * patch;
    const float invdet = 1.0f / (H00 * H11 - H10 * H01);
    const float I00 = H11 * invdet, I01 = -H01 * invdet, I10 = -H10 * invdet, I11 = H00 * invdet;
    float mean_diff = 0.f;
    float u = (float)*pu, v = (float)*pv;
    const float min_update_squared = (float)(0.03 * 0.03);
    float chi2 = 0.f, up0 = 0.f, up1 = 0.f;
    for (int iter = 0; iter < n_iter; ++iter) {
        const int u_r = (int)floorf(u), v_r = (int)floorf(v);
        if (u_r < halfpatch || v_r < halfpatch || u_r >= im.w - halfpatch || v_r >= im.h - halfpatch) break;
        if (isnan(u) || isnan(v)) return false;
        const float sx = u - (float)u_r, sy = v - (float)v_r;
        const float wTL = (float)((1.0 - sx) * (1.0 - sy));
        const float wTR = (float)(sx * (1.0 - sy));
        const float wBL = (float)((1.0 - sx) * sy);
        const float wBR = sx * sy;
        float new_chi2 = 0.f, J0 = 0.f, J1 = 0.f;
        for (int y = 0; y < patch; ++y) {
            const uint8_t* it = im.d + (size_t)(v_r + y - halfpatch) * im.pitch + (u_r - halfpatch);
            const uint8_t* tb = pwb + (y + 1) * ref_step + 1;
            for (int x = 0; x < patch; ++x) {
                const float search_pixel = wTL * (float)it[x] + wTR * (float)it[x + 1] + wBL * (float)it[x + im.pitch] +
                                           wBR * (float)it[x + im.pitch + 1];
                const float res = search_pixel - (float)ref[y * patch + x] + mean_diff;
                const float dv = (float)(0.5 * (dirx * (float)((int)tb[x + 1] - (int)tb[x - 1]) + diry * (float)((int)tb[x + ref_step] - (int)tb[x - ref_step])));
                J0 -= res * dv;
                J1 -= res;
                new_chi2 += res * res;
            }
        }
        if (iter > 0 && new_chi2 > chi2) {
            u -= up0;
            v -= up1;
            break;
        }
        chi2 = new_chi2;
        up0 = I00 * J0 + I01 * J1;
        up1 = I10 * J0 + I11 * J1;
        u += up0 * dirx;
        v += up0 * diry;
        mean_diff += up1;
        if (up0 * up0 + up1 * up1 < min_update_squared) {
            converged = true;
            break;
        }
    }
    *pu = (double)u;
    *pv = (double)v;
    return converged;
}

__global__ void __launch_bounds__(128) align1d_kernel(const uint8_t* __restrict__ pyr, size_t slot_stride, Geometry g, int n,
                                                      const int32_t* __restrict__ slot, const uint8_t* __restrict__ level,
                                                      const float* __restrict__ dir, const uint8_t* __restrict__ ref_border,
                                                      const uint8_t* __restrict__ ref, int n_iter, double* __restrict__ uv,
                                                      uint8_t* __restrict__ ok, double* __restrict__ h_inv) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t pwb[100], rp[64];
    for (int k = 0; k < 100; ++k) pwb[k] = ref_border[(size_t)i * 100 + k];
    if (ref) {
        for (int k = 0; k < 64; ++k) rp[k] = ref[(size_t)i * 64 + k];
    } else {
        for (int y = 1; y < 9; ++y)
            for (int x = 0; x < 8; ++x) rp[(y - 1) * 8 + x] = pwb[y * 10 + 1 + x];
    }
    const LevelImg im = level_img(pyr, slot_stride, slot[i], g, level[i]);
    double u = uv[2 * i], v = uv[2 * i + 1], hi = 0;
    const bool s = align1d_dev(im, dir[2 * i], dir[2 * i + 1], pwb, rp, n_iter, &u, &v, &hi);
    uv[2 * i] = u;
    uv[2 * i + 1] = v;
    ok[i] = s ? 1 : 0;
    h_inv[i] = hi;
}

struct CamF {
    float fx, fy, cx, cy;
};
__device__ __forceinline__ V3d pixel2camera(const CamF& c, double px, double py, double depth) {
    return V3d{(px - c.cx) * depth / c.fx, (py - c.cy) * depth / c.fy, depth};
}
__device__ __forceinline__ void camera2pixel(const CamF& c, V3d p, double* u, double* v) {
    *u = c.fx * p.x / p.z + c.cx;
    *v = c.fy * p.y / p.z + c.cy;
}

// cvutils::GetBilateralInterpUchar (f64 weights, truncating cast)
__device__ __forceinline__ uint8_t interp_uchar(double x, double y, const LevelImg& im) {
    const double xx = x - floor(x), yy = y - floor(y);
    const uint8_t* d = im.d + (size_t)(int)y * im.pitch + (int)x;
    return (uint8_t)((1 - xx) * (1 - yy) * d[0] + xx * (1 - yy) * d[1] + (1 - xx) * yy * d[im.pitch] + xx * yy * d[im.pitch + 1]);
}

// Matcher::FindDirectProjection(ref, curr, Feature*, px, level) for one candidate: poses as 3x4 matrices, (cu, cv) = predicted
// full-resolution pixel in, aligned pixel out.  Returns the function's bool.
__device__ bool find_direct_projection_dev(const uint8_t* __restrict__ pyr, size_t slot_stride, const Geometry& g, const CamF& cam,
                                           int ref_slot, int cur_slot, const double* __restrict__ Tr_mat, const double* __restrict__ Tc_mat,
                                           double pxr, double pyr_, double ref_depth, int lvl, double* cu_io, double* cv_io,
                                           uint8_t* search_level) {
    *search_level = 0;
    if (ref_depth < 0) return false;
    const int half = 4;
    const SE3d Tr = se3_from_mat(Tr_mat), Tc = se3_from_mat(Tc_mat);
    const SE3d Tr_inv = se3_inverse(Tr);
    const SE3d TCR = se3_mul(Tc, Tr_inv);
    const V3d pt_ref = pixel2camera(cam, pxr, pyr_, ref_depth);
    const V3d pt_ref_world = transform(Tr_inv, pt_ref);
    const V3d pt_du = pixel2camera(cam, pxr + (double)half * (1 << lvl), pyr_, pt_ref.z);
    const V3d pt_dv = pixel2camera(cam, pxr, pyr_ + (double)half * (1 << lvl), pt_ref.z);
    double cu, cv, duu, duv, dvu, dvv;
    camera2pixel(cam, transform(TCR, pt_ref_world), &cu, &cv);  // sic: world point through T_CR (Matcher.cpp:425-430)
    camera2pixel(cam, transform(TCR, pt_du), &duu, &duv);
    camera2pixel(cam, transform(TCR, pt_dv), &dvu, &dvv);
    const double A00 = (duu - cu) / half, A10 = (duv - cv) / half, A01 = (dvu - cu) / half, A11 = (dvv - cv) / half;
    int sl = 0;
    double D = A00 * A11 - A01 * A10;
    while (D > 3.0 && sl < g.n_levels - 1) {
        sl += 1;
        D *= 0.25;
    }
    *search_level = (uint8_t)sl;
    const double det = A00 * A11 - A10 * A01;
    const double invdet = 1.0 / det;
    const double R00 = A11 * invdet, R01 = -A01 * invdet, R10 = -A10 * invdet, R11 = A00 * invdet;
    const LevelImg rim = level_img(pyr, slot_stride, ref_slot, g, lvl);
    uint8_t pwb[100], patch[64];
    const double rx = pxr / (1 << lvl), ry = pyr_ / (1 << lvl);
    for (int y = 0, k = 0; y < 10; ++y)
        for (int x = 0; x < 10; ++x, ++k) {
            const double ppx = (double)(x - 5) * (1 << sl), ppy = (double)(y - 5) * (1 << sl);
            const double qx = (R00 * ppx + R01 * ppy) + rx, qy = (R10 * ppx + R11 * ppy) + ry;
            // NaN (singular warp) fails every comparison in the reference and would index out of range there;
            // it is mapped to 0 here
            if (!(qx >= 0 && qy >= 0 && qx < rim.w - 1 && qy < rim.h - 1)) pwb[k] = 0;
            else pwb[k] = interp_uchar(qx, qy, rim);
        }
    for (int y = 1; y < 9; ++y)
        for (int x = 0; x < 8; ++x) patch[(y - 1) * 8 + x] = pwb[y * 10 + 1 + x];
    double su = *cu_io / (1 << sl), sv = *cv_io / (1 << sl);
    const LevelImg cim = level_img(pyr, slot_stride, cur_slot, g, sl);
    const bool success = align2d_dev(cim, pwb, patch, 10, &su, &sv);
    const double ou = su * (1 << sl), ov = sv * (1 << sl);
    *cu_io = ou;
    *cv_io = ov;
    const bool in = ou >= 10 && ou < g.W - 10 && ov >= 10 && ov < g.H - 10;  // curr->InFrame(px_curr), border 10
    return in && success;
}

__global__ void __launch_bounds__(128) project_align_kernel(const uint8_t* __restrict__ pyr, size_t slot_stride, Geometry g, CamF cam,
                                                            int n, const int32_t* __restrict__ ref_slot,
                                                            const int32_t* __restrict__ cur_slot, const double* __restrict__ poses,
                                                            const int32_t* __restrict__ ref_pose, const int32_t* __restrict__ cur_pose,
                                                            const double* __restrict__ ref_px, const double* __restrict__ ref_depth,
                                                            const uint8_t* __restrict__ ref_level, double* __restrict__ cur_px,
                                                            uint8_t* __restrict__ search_level, uint8_t* __restrict__ ok) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double cu = cur_px[2 * i], cv = cur_px[2 * i + 1];
    uint8_t sl = 0;
    const bool good = find_direct_projection_dev(pyr, slot_stride, g, cam, ref_slot[i], cur_slot[i], poses + 12 * (size_t)ref_pose[i],
                                                 poses + 12 * (size_t)cur_pose[i], ref_px[2 * i], ref_px[2 * i + 1], ref_depth[i],
                                                 ref_level[i], &cu, &cv, &sl);
    search_level[i] = sl;
    ok[i] = good ? 1 : 0;
    if (ref_depth[i] < 0) return;   // (the reference returns before touching px_curr)
    cur_px[2 * i] = cu;
    cur_px[2 * i + 1] = cv;
}

// ---- SparseImgAlign -----------------------------------------------------------------------------------
struct SparseArgs {
    const uint8_t* pyr;
    size_t slot_stride;
    Geometry g;
    CamF cam;
    const int32_t* ref_slot;
    const int32_t* cur_slot;
    const int32_t* offsets;     // [n_problems + 1] into the per-feature arrays
    const int32_t* in_off;      // optional: px / depth / has_mp of problem p start at in_off[p] (default: offsets[p])
    const int32_t* n_feat;      // optional: feature count of problem p (default: offsets[p + 1] - offsets[p])
    const double* px;           // [2 total]
    const double* depth;
    const uint8_t* has_mp;
    const double* T_ref;        // [12 n_problems]
    double* T_cur;              // [12 n_problems] in/out
    int max_level, min_level, n_iter;
    double eps;
    int32_t* n_meas_out;        // [n_problems]  (n_meas / 16)
    int32_t* iters_out;         // [n_problems][kMaxLevels] or null
    void* feat_scratch;         // [offsets[n_problems]] SparseFeat: global fall-back of the per-feature staging
};

// One thread-block CLUSTER per (ref, cur) pair: the normal equations are FP64 (as in the reference), and one SM's FP64
// pipe would bound a single CTA.  The Gauss-Newton of the reference is reorganised around the FP64 work:
//   * J_px = (dx FJ0 + dy FJ1) * s  (FJ0/FJ1 = the two 6-vectors of the feature, dx/dy = reference gradients, s = f / 2^level),
//     so  sum_px J J^T = s^2 (Gxx FJ0 FJ0^T + Gxy (FJ0 FJ1^T + FJ1 FJ0^T) + Gyy FJ1 FJ1^T)  with per-feature constants
//     G = sum_px (dx^2, dx dy, dy^2), and  sum_px J res = s (FJ0 sum dx res + FJ1 sum dy res): an iteration costs 3 FP64 FMAs per
//     pixel + ~75 per feature instead of 27 per pixel;
//   * the features are partitioned over the CTAs of the cluster and staged in shared memory (reference patch, gradients, FJ,
//     G, camera-frame point), or in global memory when a CTA's share does not fit; 4 lanes share a feature (one patch row each);
//   * per-iteration partial sums are exchanged through distributed shared memory (one cluster barrier), every CTA adds them
//     in rank order and takes the same step (LDL^T with hardware-seeded reciprocals).
constexpr int kSparseThreads = 256;
constexpr int kSparseCluster = 8;          // CTAs per problem of ygzb_sparse_align (the tracker chooses its own)
constexpr int kNormalTerms = 21 + 6 + 1;   // H upper triangle, Jres, chi2 (+ the measurement count in a separate integer)

struct SparseFeat {           // 4-byte fields first: arrays of structs in shared memory, one per feature of the CTA
    float patch[16], gdx[16], gdy[16];
    double FJ[12];
    double G[3];
    double xyz[3];
    float u, v;            // projection into the current level at the current pose (phase A of an iteration)
    int ui, vi;
    int state;             // bit 0: visible (sticky across levels), bit 1: inside the current image at this iteration
    int pad;
};

__device__ __forceinline__ double rcp_f64(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(r, fma(-x, r, 1.0), r);
    r = fma(r, fma(-x, r, 1.0), r);
    return r;
}

__device__ bool ldlt_solve6(const double H[6][6], const double b[6], double x[6]) {
    double L[6][6], D[6], rD[6];
    for (int j = 0; j < 6; ++j) {
        double d = H[j][j];
        for (int k = 0; k < j; ++k) d -= L[j][k] * L[j][k] * D[k];
        D[j] = d;
        if (!(fabs(d) > 0)) return false;
        rD[j] = rcp_f64(fabs(d));
        if (d < 0) rD[j] = -rD[j];
        L[j][j] = 1;
        for (int i = j + 1; i < 6; ++i) {
            double s = H[i][j];
            for (int k = 0; k < j; ++k) s -= L[i][k] * L[j][k] * D[k];
            L[i][j] = s * rD[j];
        }
    }
    double y[6];
    for (int i = 0; i < 6; ++i) {
        double s = b[i];
        for (int k = 0; k < i; ++k) s -= L[i][k] * y[k];
        y[i] = s;
    }
    for (int i = 0; i < 6; ++i) y[i] *= rD[i];
    for (int i = 5; i >= 0; --i) {
        double s = y[i];
        for (int k = i + 1; k < 6; ++k) s -= L[k][i] * x[k];
        x[i] = s;
    }
    return true;
}

__global__ void __launch_bounds__(kSparseThreads) sparse_align_kernel(const SparseArgs a, int feat_cap /* features per CTA that fit shared memory */) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ double s_red[kSparseThreads / 32][kNormalTerms];
    __shared__ unsigned s_nm[kSparseThreads / 32];
    __shared__ double s_part[2][kNormalTerms + 1];   // this CTA's partial sums of an iteration (double buffered), [kNormalTerms] = count
    __shared__ SE3d s_T, s_old;
    __shared__ double s_Tm[12];
    __shared__ int s_flag;
    __shared__ double s_chi2;
    __shared__ unsigned long long s_last_nmeas;

    const int rank = (int)cluster.block_rank(), C = (int)cluster.num_blocks();
    const int prob = blockIdx.x / C, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int f0 = a.offsets[prob];
    const int nf = a.n_feat ? a.n_feat[prob] : a.offsets[prob + 1] - f0;
    const long din = a.in_off ? (long)a.in_off[prob] - f0 : 0;
    const Geometry& g = a.g;
    if (nf == 0) {
        if (rank == 0 && tid == 0) a.n_meas_out[prob] = 0;
        return;
    }
    // this CTA's features: a contiguous share, staged in shared memory (the launcher sizes the cluster so that it fits)
    const int per = (nf + C - 1) / C;
    const int j_lo = min(nf, rank * per), nl = min(nf, j_lo + per) - j_lo;
    SparseFeat* F = nl <= feat_cap ? reinterpret_cast<SparseFeat*>(s_raw) : static_cast<SparseFeat*>(a.feat_scratch) + f0 + j_lo;
    if (tid == 0) {
        const SE3d Tref = se3_from_mat(a.T_ref + 12 * (size_t)prob);
        s_T = se3_mul(se3_from_mat(a.T_cur + 12 * (size_t)prob), se3_inverse(Tref));
        s_chi2 = 1e10;
        s_last_nmeas = 0;
    }
    for (int j = tid; j < nl; j += kSparseThreads) {
        SparseFeat& ft = F[j];
        const long gi = f0 + j_lo + j + din;
        ft.state = 0;
        const V3d xyz = pixel2camera(a.cam, a.px[2 * gi], a.px[2 * gi + 1], a.depth[gi]);
        ft.xyz[0] = xyz.x; ft.xyz[1] = xyz.y; ft.xyz[2] = xyz.z;
        for (int k = 0; k < 16; ++k) ft.patch[k] = 0.f;
    }
    __syncthreads();
    int slot = 0;

    for (int lvl = a.max_level; lvl >= a.min_level; --lvl) {
        const LevelImg rim = level_img(a.pyr, a.slot_stride, a.ref_slot[prob], g, lvl);
        const LevelImg cim = level_img(a.pyr, a.slot_stride, a.cur_slot[prob], g, lvl);
        const float scale = 1.0f / (float)(1 << lvl);
        const double focal = (double)(float)((a.cam.fx + a.cam.fy) / 2);  // PinholeCamera::_f is a float
        const double jscale = focal / (1 << lvl);
        // precomputeReferencePatches (features that are not cached at this level keep their stale patch with a zero Jacobian)
        for (int j = tid; j < nl; j += kSparseThreads) {
            SparseFeat& ft = F[j];
            const long gi = f0 + j_lo + j + din;
            for (int k = 0; k < 16; ++k) ft.gdx[k] = ft.gdy[k] = 0.f;
            ft.G[0] = ft.G[1] = ft.G[2] = 0.0;
            const float u_ref = (float)(a.px[2 * gi] * scale), v_ref = (float)(a.px[2 * gi + 1] * scale);
            const int ui = (int)floorf(u_ref), vi = (int)floorf(v_ref);
            if ((a.has_mp && !a.has_mp[gi]) || ui - 3 < 0 || vi - 3 < 0 || ui + 3 >= rim.w || vi + 3 >= rim.h) continue;
            ft.state |= 1;
            const double X = ft.xyz[0], Y = ft.xyz[1], zi = 1. / ft.xyz[2], zi2 = zi * zi;
            double* J = ft.FJ;
            J[0] = -zi; J[1] = 0; J[2] = X * zi2; J[3] = Y * J[2]; J[4] = -(1.0 + X * J[2]); J[5] = Y * zi;
            J[6] = 0; J[7] = -zi; J[8] = Y * zi2; J[9] = 1.0 + Y * J[8]; J[10] = -J[3]; J[11] = -X * zi;
            const float su = u_ref - (float)ui, sv = v_ref - (float)vi;
            const float wtl = (float)((1.0 - su) * (1.0 - sv)), wtr = (float)(su * (1.0 - sv)), wbl = (float)((1.0 - su) * sv), wbr = su * sv;
            const int st = rim.pitch;
            int pc = 0;
            double gxx = 0, gxy = 0, gyy = 0;
            for (int y = 0; y < 4; ++y) {
                const uint8_t* p = rim.d + (size_t)(vi + y - 2) * st + (ui - 2);
                for (int xx = 0; xx < 4; ++xx, ++p, ++pc) {
                    ft.patch[pc] = wtl * (float)p[0] + wtr * (float)p[1] + wbl * (float)p[st] + wbr * (float)p[st + 1];
                    const float dx = 0.5f * ((wtl * (float)p[1] + wtr * (float)p[2] + wbl * (float)p[st + 1] + wbr * (float)p[st + 2]) -
                                             (wtl * (float)p[-1] + wtr * (float)p[0] + wbl * (float)p[st - 1] + wbr * (float)p[st]));
                    const float dy = 0.5f * ((wtl * (float)p[st] + wtr * (float)p[1 + st] + wbl * (float)p[st * 2] + wbr * (float)p[st * 2 + 1]) -
                                             (wtl * (float)p[-st] + wtr * (float)p[1 - st] + wbl * (float)p[0] + wbr * (float)p[1]));
                    ft.gdx[pc] = dx;
                    ft.gdy[pc] = dy;
                    gxx += (double)dx * (double)dx;
                    gxy += (double)dx * (double)dy;
                    gyy += (double)dy * (double)dy;
                }
            }
            ft.G[0] = gxx; ft.G[1] = gxy; ft.G[2] = gyy;
        }
        if (tid == 0) {
            s_old = s_T;
            s_flag = 0;
            se3_to_mat(s_T, s_Tm);
        }
        __syncthreads();

        int it = 0;
        for (it = 0; it < a.n_iter; ++it) {
            // phase A: projection of every visible feature at the current pose
            for (int j = tid; j < nl; j += kSparseThreads) {
                SparseFeat& ft = F[j];
                if (!(ft.state & 1)) continue;
                ft.state &= ~2;
                const double x = s_Tm[0] * ft.xyz[0] + s_Tm[1] * ft.xyz[1] + s_Tm[2] * ft.xyz[2] + s_Tm[3];
                const double y = s_Tm[4] * ft.xyz[0] + s_Tm[5] * ft.xyz[1] + s_Tm[6] * ft.xyz[2] + s_Tm[7];
                const double z = s_Tm[8] * ft.xyz[0] + s_Tm[9] * ft.xyz[1] + s_Tm[10] * ft.xyz[2] + s_Tm[11];
                double pu, pv;
                camera2pixel(a.cam, V3d{x, y, z}, &pu, &pv);
                const float u_cur = (float)pu * scale, v_cur = (float)pv * scale;
                const int ui = (int)floorf(u_cur), vi = (int)floorf(v_cur);
                if (ui < 0 || vi < 0 || ui - 3 < 0 || vi - 3 < 0 || ui + 3 >= cim.w || vi + 3 >= cim.h) continue;
                ft.u = u_cur; ft.v = v_cur; ft.ui = ui; ft.vi = vi;
                ft.state |= 2;
            }
            __syncthreads();
            // phase B: (feature, patch row) items over the threads
            double acc[kNormalTerms];
#pragma unroll
            for (int k = 0; k < kNormalTerms; ++k) acc[k] = 0.0;
            unsigned nm = 0;
            for (int item = tid; item < nl * 4; item += kSparseThreads) {
                const SparseFeat& ft = F[item >> 2];
                if ((ft.state & 3) != 3) continue;
                const int y = item & 3;
                const float su = ft.u - (float)ft.ui, sv = ft.v - (float)ft.vi;
                const float wtl = (float)((1.0 - su) * (1.0 - sv)), wtr = (float)(su * (1.0 - sv)), wbl = (float)((1.0 - su) * sv), wbr = su * sv;
                const int st = cim.pitch;
                const uint8_t* p = cim.d + (size_t)(ft.vi + y - 2) * st + (ft.ui - 2);
                double sa = 0, sb = 0;
#pragma unroll
                for (int xx = 0; xx < 4; ++xx, ++p) {
                    const int pc = 4 * y + xx;
                    const float inten = wtl * (float)p[0] + wtr * (float)p[1] + wbl * (float)p[st] + wbr * (float)p[st + 1];
                    const float res = inten - ft.patch[pc];
                    acc[27] += (double)(res * res);
                    sa += (double)ft.gdx[pc] * (double)res;
                    sb += (double)ft.gdy[pc] * (double)res;
                }
                nm += 4;
#pragma unroll
                for (int k = 0; k < 6; ++k) acc[21 + k] -= (ft.FJ[k] * sa + ft.FJ[6 + k] * sb) * jscale;
                if (y == 0) {
                    const double s2 = jscale * jscale, gxx = ft.G[0] * s2, gxy = ft.G[1] * s2, gyy = ft.G[2] * s2;
                    int t = 0;
#pragma unroll
                    for (int r = 0; r < 6; ++r)
#pragma unroll
                        for (int c = r; c < 6; ++c, ++t)
                            acc[t] += gxx * (ft.FJ[r] * ft.FJ[c]) + gxy * (ft.FJ[r] * ft.FJ[6 + c] + ft.FJ[6 + r] * ft.FJ[c]) + gyy * (ft.FJ[6 + r] * ft.FJ[6 + c]);
                }
            }
#pragma unroll
            for (int k = 0; k < kNormalTerms; ++k) {
                double v = acc[k];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, o);
                if (lane == 0) s_red[warp][k] = v;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) nm += __shfl_down_sync(0xFFFFFFFFu, nm, o);
            if (lane == 0) s_nm[warp] = nm;
            __syncthreads();
            if (tid <= kNormalTerms) {
                double v = 0;
                if (tid < kNormalTerms) {
                    for (int w = 0; w < kSparseThreads / 32; ++w) v += s_red[w][tid];
                } else {
                    unsigned n = 0;
                    for (int w = 0; w < kSparseThreads / 32; ++w) n += s_nm[w];
                    v = (double)n;
                }
                s_part[slot][tid] = v;
            }
            cluster.sync();
            if (tid == 0) {
                double tot[kNormalTerms];
                unsigned long long n_meas = 0;
                for (int k = 0; k < kNormalTerms; ++k) tot[k] = 0;
                for (int r = 0; r < C; ++r) {
                    const double* pr = cluster.map_shared_rank(&s_part[slot][0], r);
                    for (int k = 0; k < kNormalTerms; ++k) tot[k] += pr[k];
                    n_meas += (unsigned long long)pr[kNormalTerms];
                }
                s_last_nmeas = n_meas;
                double H[6][6], b[6], x[6];
                int t = 0;
                for (int r = 0; r < 6; ++r)
                    for (int c = r; c < 6; ++c) H[r][c] = H[c][r] = tot[t++];
                for (int k = 0; k < 6; ++k) b[k] = tot[21 + k];
                const double new_chi2 = (double)((float)tot[27] / (float)n_meas);
                bool stop = !ldlt_solve6(H, b, x) || isnan(x[0]);
                if ((it > 0 && new_chi2 > s_chi2) || stop) {
                    s_T = s_old;  // rollback
                    s_flag = 1;
                } else {
                    double mx[6];
                    for (int k = 0; k < 6; ++k) mx[k] = -x[k];
                    const SE3d Tn = se3_mul(s_T, se3_exp(mx));
                    s_old = s_T;
                    s_T = Tn;
                    s_chi2 = new_chi2;
                    double nmx = -1;
                    for (int k = 0; k < 6; ++k) nmx = fabs(x[k]) > nmx ? fabs(x[k]) : nmx;
                    if (nmx <= a.eps) s_flag = 1;
                }
                se3_to_mat(s_T, s_Tm);
            }
            slot ^= 1;
            __syncthreads();
            if (s_flag) break;
        }
        if (rank == 0 && tid == 0 && a.iters_out) a.iters_out[prob * kMaxLevels + lvl] = it;
        __syncthreads();
    }
    cluster.sync();   // no CTA may exit while another still reads its partials
    if (rank == 0 && tid == 0) {
        const SE3d Tref = se3_from_mat(a.T_ref + 12 * (size_t)prob);
        se3_to_mat(se3_mul(s_T, Tref), a.T_cur + 12 * (size_t)prob);
        a.n_meas_out[prob] = (int32_t)(s_last_nmeas / 16);
    }
}

// ---- device-resident tracking chain (track.cuh): the caller-side steps between the kernels above -----------------------
// plain 3x4 matrix products exactly as the host drivers write them (host/vo_driver.cpp: mul / inv of Mat34)
__device__ __forceinline__ void mat34_mul(const double* A, const double* B, double* C) {
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) C[4 * r + c] = A[4 * r] * B[c] + A[4 * r + 1] * B[4 + c] + A[4 * r + 2] * B[8 + c];
        C[4 * r + 3] = A[4 * r] * B[3] + A[4 * r + 1] * B[7] + A[4 * r + 2] * B[11] + A[4 * r + 3];
    }
}
__device__ __forceinline__ void mat34_inv(const double* A, double* C) {
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) C[4 * r + c] = A[4 * c + r];
        C[4 * r + 3] = -(A[r] * A[3] + A[4 + r] * A[7] + A[8 + r] * A[11]);
    }
}

// per job: problem description of the sparse alignment from the ring entry of the reference key-frame
__global__ void track_prep_kernel(TrackStore st, TrackBatch b) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= b.J) return;
    const ygzb_track_job job = b.jobs[j];
    const int e = job.stream * st.R + job.entry[job.n_local - 1];
    b.ref_slot[j] = st.kf_slot[e];
    b.cur_slot[j] = job.cur_slot;
    b.offsets[j] = j * st.cells;
    if (j == 0) b.offsets[b.J] = b.J * st.cells;
    b.in_off[j] = e * st.cells;
    b.n_feat[j] = st.kf_n[e];
    // the alignment runs RELATIVE to the reference key-frame (cur._TCW = ref._TCW, VisualOdometry.cpp:66: the start is the
    // identity in the key-frame's frame); track_compose_kernel applies the key-frame's pose afterwards, so this part of the
    // chain does not depend on a local BA that may still be refining that pose
    for (int c = 0; c < 12; ++c) b.T_ref[12 * (size_t)j + c] = b.T_cur[12 * (size_t)j + c] = (c == 0 || c == 5 || c == 10) ? 1.0 : 0.0;
    b.n_cand[j] = 0;
    b.c_off[j] = j * b.cap;
    if (j == 0) b.c_off[b.J] = b.J * b.cap;
}

// per job: T_cw of the aligned frame = (pose relative to the reference key-frame) * (pose of the key-frame, after its BA)
__global__ void track_compose_kernel(TrackStore st, TrackBatch b) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= b.J) return;
    const ygzb_track_job job = b.jobs[j];
    const double* Tk = st.kf_T + 12 * (size_t)(job.stream * st.R + job.entry[job.n_local - 1]);
    const SE3d Trel = se3_from_mat(b.T_cur + 12 * (size_t)j), Tref = se3_from_mat(Tk);
    se3_to_mat(se3_mul(Trel, Tref), b.T_cur + 12 * (size_t)j);
    for (int c = 0; c < 12; ++c) b.T_ref[12 * (size_t)j + c] = Tk[c];
}

// per job: Matcher::SparseImageAlignment's motion check (Matcher.cpp:482-488) and the current pose relative to every
// local key-frame (GetWarpAffineMatrix is only correct for an identity reference pose, Matcher.cpp:425-430)
__global__ void track_motion_kernel(TrackStore st, TrackBatch b) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= b.J) return;
    const ygzb_track_job job = b.jobs[j];
    const double* Tc = b.T_cur + 12 * (size_t)j;
    double inv_ref[12], tcr[12], lg[6];
    mat34_inv(b.T_ref + 12 * (size_t)j, inv_ref);
    mat34_mul(Tc, inv_ref, tcr);
    se3_log(se3_from_mat(tcr), lg);
    double nrm = 0;
    for (int k = 0; k < 6; ++k) nrm += lg[k] * lg[k];
    b.aligned[j] = sqrt(nrm) <= 0.2 ? 1 : 0;
    for (int k = 0; k < job.n_local; ++k) {
        double inv_k[12];
        mat34_inv(st.kf_T + 12 * (size_t)(job.stream * st.R + job.entry[k]), inv_k);
        mat34_mul(Tc, inv_k, b.rel + 12 * ((size_t)j * kTrackMaxLocal + k));
    }
}

// LocalMapping::FindCandidates (LocalMapping.cpp:47-80) + Matcher::FindDirectProjection (:82-111) for dense candidate
// c = local key-frame k * cells + feature g of job blockIdx.y
__global__ void __launch_bounds__(128) track_project_kernel(const uint8_t* __restrict__ pyr, size_t slot_stride, Geometry g, CamF cam,
                                                            TrackStore st, TrackBatch b) {
    const int j = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= b.cap) return;
    const size_t at = (size_t)j * b.cap + c;
    b.cand_ok[at] = 0;
    if (!b.aligned[j]) return;
    const ygzb_track_job job = b.jobs[j];
    const int k = c / st.cells, f = c - k * st.cells;
    if (k >= job.n_local) return;
    const int e = job.stream * st.R + job.entry[k];
    if (f >= st.kf_n[e]) return;
    const double* X = st.kf_pw + 3 * ((size_t)e * st.cells + f);
    const double* T = b.T_cur + 12 * (size_t)j;
    const double x = T[0] * X[0] + T[1] * X[1] + T[2] * X[2] + T[3];
    const double y = T[4] * X[0] + T[5] * X[1] + T[6] * X[2] + T[7];
    const double z = T[8] * X[0] + T[9] * X[1] + T[10] * X[2] + T[11];
    double u = st.fx * x / z + st.cx, v = st.fy * y / z + st.cy;
    if (!(z > 0 && u >= 20 && u < st.W - 20 && v >= 20 && v < st.H - 20)) return;
    atomicAdd(&b.n_cand[j], 1);
    const double eye[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
    uint8_t sl;
    const size_t fe = (size_t)e * st.cells + f;
    const bool ok = find_direct_projection_dev(pyr, slot_stride, g, cam, st.kf_slot[e], job.cur_slot, eye,
                                               b.rel + 12 * ((size_t)j * kTrackMaxLocal + k), st.kf_px[2 * fe], st.kf_px[2 * fe + 1],
                                               st.kf_depth[fe], st.kf_level[fe], &u, &v, &sl);
    b.cand_px[2 * at] = u;
    b.cand_px[2 * at + 1] = v;
    b.cand_ok[at] = ok ? 1 : 0;
}

// ordered compaction of the successfully projected candidates of job blockIdx.x (candidate order = local key-frame, then
// feature: the order in which the reference's caller loops hand them to OptimizeCurrentPoseOnly)
// inclusive scan of one int per thread over a 1024-thread CTA (shuffles + one pass over the 32 warp totals: two barriers
// instead of the twenty of a shared-memory Hillis-Steele scan); s_w = 33 ints; *total = the CTA total
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
    __syncthreads();
    return out;
}

__global__ void __launch_bounds__(1024) track_compact_kernel(TrackStore st, TrackBatch b) {
    __shared__ int s_scan[33];
    __shared__ int s_carry;
    const int j = blockIdx.x, tid = threadIdx.x;
    const ygzb_track_job job = b.jobs[j];
    const int total = job.n_local * st.cells;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < total; base += 1024) {
        const int c = base + tid;
        const int flag = (c < total && b.cand_ok[(size_t)j * b.cap + c]) ? 1 : 0;
        int chunk_total;
        const int incl = block_scan_1024(flag, s_scan, &chunk_total);
        if (flag) {
            const size_t dst = (size_t)j * b.cap + s_carry + incl - 1;
            const int k = c / st.cells, f = c - k * st.cells;
            const size_t fe = (size_t)(job.stream * st.R + job.entry[k]) * st.cells + f;
            b.c_src[dst] = c;
            b.c_px[2 * dst] = b.cand_px[2 * ((size_t)j * b.cap + c)];
            b.c_px[2 * dst + 1] = b.cand_px[2 * ((size_t)j * b.cap + c) + 1];
            b.c_pw[3 * dst] = st.kf_pw[3 * fe];
            b.c_pw[3 * dst + 1] = st.kf_pw[3 * fe + 1];
            b.c_pw[3 * dst + 2] = st.kf_pw[3 * fe + 2];
        }
        __syncthreads();
        if (tid == 0) s_carry += chunk_total;
        __syncthreads();
    }
    if (tid == 0) b.c_cnt[j] = s_carry;
}

// One cluster of `cluster` CTAs per problem.  A CTA stages its share of a problem's features, at most
// ceil(max_feat / cluster), in dynamic shared memory, or in a.feat_scratch when that share exceeds what a CTA can opt in to.
// Fills the frame fields of `a` (pyramids, geometry, camera) from f.
int launch_sparse_align_kernel(ygzb_frames* f, SparseArgs a, int n_problems, int max_feat, int cluster) {
    ygzb_ctx* ctx = f->ctx;
    a.pyr = f->d_pyr;
    a.slot_stride = ctx->slot_stride;
    a.g = ctx->geo;
    a.cam = CamF{ctx->prm.fx, ctx->prm.fy, ctx->prm.cx, ctx->prm.cy};
    static std::once_flag once;
    static int max_dyn = 0;
    std::call_once(once, [] {
        int dev = 0, optin = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        max_dyn = optin - 8 * 1024;   // the kernel's static arrays
        cudaFuncSetAttribute(sparse_align_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn);
    });
    const int feat_cap = max_dyn / (int)sizeof(SparseFeat);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(n_problems * cluster));
    cfg.blockDim = dim3(kSparseThreads);
    cfg.dynamicSmemBytes = (size_t)std::min(feat_cap, (max_feat + cluster - 1) / cluster) * sizeof(SparseFeat);
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    ProfScope ps(ctx, kStageSparseAlign);
    YGZB_CUDA(ctx, cudaLaunchKernelEx(&cfg, sparse_align_kernel, a, feat_cap));
    YGZB_LAUNCHED(ctx);
    return YGZB_OK;
}

}  // namespace

size_t sparse_align_scratch_bytes(size_t n_features) { return n_features * sizeof(SparseFeat); }

int launch_align2d(ygzb_frames* f, int n, const int32_t* d_slot, const uint8_t* d_level, const uint8_t* d_ref_border,
                   const uint8_t* d_ref, int n_iter, double* d_uv, uint8_t* d_ok) {
    ygzb_ctx* ctx = f->ctx;
    if (n <= 0) return YGZB_OK;
    ProfScope ps(ctx, kStageAlign2D);
    align2d_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(f->d_pyr, ctx->slot_stride, ctx->geo, n, d_slot, d_level, d_ref_border,
                                                             d_ref, n_iter, d_uv, d_ok);
    YGZB_LAUNCHED(ctx);
    return YGZB_OK;
}

int launch_align1d(ygzb_frames* f, int n, const int32_t* d_slot, const uint8_t* d_level, const float* d_dir, const uint8_t* d_ref_border,
                   const uint8_t* d_ref, int n_iter, double* d_uv, uint8_t* d_ok, double* d_hinv) {
    ygzb_ctx* ctx = f->ctx;
    if (n <= 0) return YGZB_OK;
    ProfScope ps(ctx, kStageAlign2D);
    align1d_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(f->d_pyr, ctx->slot_stride, ctx->geo, n, d_slot, d_level, d_dir, d_ref_border,
                                                             d_ref, n_iter, d_uv, d_ok, d_hinv);
    YGZB_LAUNCHED(ctx);
    return YGZB_OK;
}

int launch_project_align(ygzb_frames* f, int n, const int32_t* d_ref_slot, const int32_t* d_cur_slot, const double* d_poses,
                         const int32_t* d_ref_pose, const int32_t* d_cur_pose, const double* d_ref_px, const double* d_ref_depth,
                         const uint8_t* d_ref_level, double* d_cur_px, uint8_t* d_search_level, uint8_t* d_ok) {
    ygzb_ctx* ctx = f->ctx;
    if (n <= 0) return YGZB_OK;
    const CamF cam{ctx->prm.fx, ctx->prm.fy, ctx->prm.cx, ctx->prm.cy};
    ProfScope ps(ctx, kStageProjectAlign);
    project_align_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(f->d_pyr, ctx->slot_stride, ctx->geo, cam, n, d_ref_slot,
                                                                   d_cur_slot, d_poses, d_ref_pose, d_cur_pose, d_ref_px,
                                                                   d_ref_depth, d_ref_level, d_cur_px, d_search_level, d_ok);
    YGZB_LAUNCHED(ctx);
    return YGZB_OK;
}

int launch_sparse_align(ygzb_frames* f, int n_problems, const int32_t* d_ref_slot, const int32_t* d_cur_slot,
                        const int32_t* d_offsets, int max_feat, const double* d_px, const double* d_depth, const uint8_t* d_has_mp,
                        const double* d_T_ref, double* d_T_cur, int max_level, int min_level, int n_iter, double eps,
                        int32_t* d_n_meas, int32_t* d_iters, void* d_feat_scratch) {
    if (n_problems <= 0) return YGZB_OK;
    SparseArgs a{};
    a.ref_slot = d_ref_slot;
    a.cur_slot = d_cur_slot;
    a.offsets = d_offsets;
    a.px = d_px;
    a.depth = d_depth;
    a.has_mp = d_has_mp;
    a.T_ref = d_T_ref;
    a.T_cur = d_T_cur;
    a.max_level = max_level;
    a.min_level = min_level;
    a.n_iter = n_iter;
    a.eps = eps;
    a.n_meas_out = d_n_meas;
    a.iters_out = d_iters;
    a.feat_scratch = d_feat_scratch;
    return launch_sparse_align_kernel(f, a, n_problems, max_feat, kSparseCluster);
}

// Tracking chain of a batch, part 1 (on whatever stream ctx->stream currently is: the tracker points it at its second
// stream): prep -> sparse alignment relative to the reference key-frame.  Needs the key-frame's features, not its pose.
int launch_track_chain_front(ygzb_frames* f, const TrackStore& st, const TrackBatch& b, int sparse_cluster) {
    ygzb_ctx* ctx = f->ctx;
    if (b.J <= 0) return YGZB_OK;
    {
        ProfScope ps(ctx, kStageOther);
        track_prep_kernel<<<(b.J + 127) / 128, 128, 0, ctx->stream>>>(st, b);
        YGZB_LAUNCHED(ctx);
    }
    SparseArgs a{};
    a.ref_slot = b.ref_slot;
    a.cur_slot = b.cur_slot;
    a.offsets = b.offsets;
    a.in_off = b.in_off;
    a.n_feat = b.n_feat;
    a.px = st.kf_px;
    a.depth = st.kf_depth;
    a.has_mp = nullptr;            // every feature of a key-frame has its map point (depth-initialised)
    a.T_ref = b.T_ref;
    a.T_cur = b.T_cur;
    a.max_level = 2;               // Matcher's SparseImgAlign(2, 0, 30, GaussNewton) (Matcher.cpp:18)
    a.min_level = 0;
    a.n_iter = 30;
    a.eps = 1e-6;
    a.n_meas_out = b.n_meas;
    a.iters_out = nullptr;
    a.feat_scratch = b.feat_scratch;
    return launch_sparse_align_kernel(f, a, b.J, st.cells, sparse_cluster);
}

// part 2 (main stream, behind a local BA in flight): key-frame pose applied -> motion check / relative poses -> candidate
// projection + direct projection -> ordered compaction.  The pose-only refinement (ba.cu) follows on the same stream.
int launch_track_chain_mid(ygzb_frames* f, const TrackStore& st, const TrackBatch& b) {
    ygzb_ctx* ctx = f->ctx;
    if (b.J <= 0) return YGZB_OK;
    {
        ProfScope ps(ctx, kStageOther);
        track_compose_kernel<<<(b.J + 63) / 64, 64, 0, ctx->stream>>>(st, b);
        YGZB_LAUNCHED(ctx);
    }
    {
        ProfScope ps(ctx, kStageOther);
        track_motion_kernel<<<(b.J + 63) / 64, 64, 0, ctx->stream>>>(st, b);
        YGZB_LAUNCHED(ctx);
    }
    {
        const CamF cam{ctx->prm.fx, ctx->prm.fy, ctx->prm.cx, ctx->prm.cy};
        ProfScope ps(ctx, kStageProjectAlign);
        track_project_kernel<<<dim3((unsigned)((b.cap + 127) / 128), (unsigned)b.J), 128, 0, ctx->stream>>>(f->d_pyr, ctx->slot_stride, ctx->geo,
                                                                                                          cam, st, b);
        YGZB_LAUNCHED(ctx);
    }
    {
        ProfScope ps(ctx, kStageOther);
        track_compact_kernel<<<(unsigned)b.J, 1024, 0, ctx->stream>>>(st, b);
        YGZB_LAUNCHED(ctx);
    }
    return YGZB_OK;
}

}  // namespace ygzb
