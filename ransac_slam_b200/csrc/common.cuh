// common.cuh -- device-side data layout and camera-model math shared by all kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/rslam.h"

namespace rslam {

constexpr int kPatch = 13;            // 2*6+1 matching patch (src/Map.cpp:294)
constexpr int kPatchPix = 169;
constexpr int kHalfPatch = 6;
constexpr int kNB = 64;               // block size of the blocked Cholesky / TRSM

struct CamDev {
    double k1, k2, Cx, Cy, f, dx, dy, fku, fkv;
    int nRows, nCols;
};

struct ParDev {
    double std_z, chi2, corr_thr, p_free, max_eig, la, aa;  // la/aa: (std_a*dt)^2, (std_alpha*dt)^2
    int n_hyp0;
    unsigned quirks;
};

// per-filter device descriptor (array of `batch` of these lives in HBM; kernels index it with blockIdx.y / .z)
struct DevFilter {
    // dimensions
    int n;       // state dimension 13 + sum(feature sizes)
    int N;       // number of features
    int ldp;     // leading dimension of P (multiple of 16)
    int ldw;     // leading dimension of W (>= n+1, multiple of 16)
    int lds;     // leading dimension of the innovation matrix S (multiple of 16)
    int kmax;    // 2 * Nmax
    int mwords;  // words per inlier mask row
    int pad0;
    // state
    double* P;
    double* x_kk;
    double* x_km1;
    // per-feature SoA
    int* ftype;   // 0 inverse depth / 1 cartesian
    int* foff;    // offset of the feature block in x
    double* h;    // 2N
    double* Hc;   // 14N  row-major 2x7  (d h / d r, d h / d q)
    double* Hf;   // 12N  row-major 2x6
    double* S;    // 4N   row-major 2x2 (includes +R)
    double* z;    // 2N
    unsigned char* has_h;
    unsigned char* ic;
    unsigned char* li;
    unsigned char* hi;
    int* times_predicted;
    int* times_measured;
    float* patch;  // N x 169 row-major (r*13+c) predicted appearance
    // appearance at initialisation (only needed when the predicted patch is warped on the device, pred_patch_fc)
    unsigned char* patch_init;  // N x 41 x 41 row-major
    double* init_pose;          // N x 14: r_wc(3), R_wc row-major(9), uv(2)
    double* pp_geom;            // N x 12: per-feature warp geometry of the current frame (k_pred_patch_setup): Hm (9), xs, ys, ok
    int* last_id;               // N: index of the latest inverse-depth feature <= i (-1 if none): XYZ_w actually used (quirk Q3)
    // image (may be shared between filters)
    const unsigned char* image;
    int img_rows, img_cols, img_stride, pad1;
    // RANSAC workspace
    int* ic_list;      // [N]  features with individually_compatible, feature order
    int* id_list;      // [N]  matched inverse-depth features, feature order (z_id columns)
    int* sup_rows;     // [6 * round_up(N, 64)]  state rows of the support-scoring tiles, tile order (k_ransac_compact)
    int* id_pos;       // [N]  feature -> column in z_id (or -1)
    double* hyp_ab;    // [N x 16]  a_p (7) = Hc_p^T g_p, b_p (6) = Hf_p^T g_p, [13] element offset of column y_p in P (as bits), [14] feature size
    double* hyp_xcam;  // [N x 7]   hypothesised r, q
    int* support;      // [N]
    unsigned* masks;   // [N x mwords]
    const double* u01; // n_u01 draws for this filter
    int n_u01, pad2;
    int* ctl;          // control block, see CTL_* below
    // update workspace
    int* upd_list;     // [N]
    double* W;         // ldw x kmax : P H^T, then V = W L^-T; row n holds the innovation (then y = L^-1 nu)
    double* Sm;        // lds x kmax : innovation covariance, then its Cholesky factor (lower)
    double* Jn;        // 16 + scratch
    double* Linv;      // [ceil(kmax/64)][64 x 64] inverses of the Cholesky factor's diagonal blocks (column-major)
};

enum CtlSlot {
    CTL_NIC = 0,      // number of individually compatible matches
    CTL_MID = 1,      // number of matched inverse-depth features (z_id columns)
    CTL_NCART = 2,    // matched cartesian features (reference UB, Q2)
    CTL_M = 3,        // measurements in the current joint update
    CTL_K = 4,        // 2*m
    CTL_STATUS = 5,   // ransac status
    CTL_HYPRUN = 6,
    CTL_BEST = 7,
    CTL_NHYP = 8,
    CTL_WINNER = 9,   // winning hypothesis index in the u01 sequence
    CTL_WINNER_T = 10,// winning distinct hypothesis (index into ic_list)
    CTL_JN_DONE = 11, // k_upd_jnorm_wide: CTAs that have finished (reset to 0 by the last one)
    CTL_SIZE = 16
};

// src/ExtendKF.cpp:91-102 (map_prep_add_dev in kernels_map.cuh has an unfused copy, kept in step by hand: change both)
__device__ __forceinline__ void q2r_dev(const double* q, double R[9]) {
    const double r = q[0], x = q[1], y = q[2], z = q[3];
    R[0] = r * r + x * x - y * y - z * z;
    R[1] = 2 * (x * y - r * z);
    R[2] = 2 * (z * x + r * y);
    R[3] = 2 * (x * y + r * z);
    R[4] = r * r - x * x + y * y - z * z;
    R[5] = 2 * (y * z - r * x);
    R[6] = 2 * (z * x - r * y);
    R[7] = 2 * (y * z + r * x);
    R[8] = r * r - x * x - y * y + z * z;
}

// closed-form 3x3 inverse by cofactors (Eigen fixed-size inverse, used at src/Tracking.cpp:136)
__device__ __forceinline__ void inv3_dev(const double* m, double* o) {
    const double c00 = m[4] * m[8] - m[5] * m[7];
    const double c10 = m[7] * m[2] - m[8] * m[1];  // cofactor(1,0)
    const double c20 = m[1] * m[5] - m[2] * m[4];
    const double det = c00 * m[0] + c10 * m[3] + c20 * m[6];
    const double id = 1.0 / det;
    o[0] = c00 * id;
    o[1] = c10 * id;
    o[2] = c20 * id;
    o[3] = (m[5] * m[6] - m[3] * m[8]) * id;
    o[4] = (m[8] * m[0] - m[6] * m[2]) * id;
    o[5] = (m[2] * m[3] - m[0] * m[5]) * id;
    o[6] = (m[3] * m[7] - m[4] * m[6]) * id;
    o[7] = (m[6] * m[1] - m[7] * m[0]) * id;
    o[8] = (m[0] * m[4] - m[1] * m[3]) * id;
}

// radial distortion, exactly 10 Newton steps (src/ExtendKF.cpp:175-204)
__device__ __forceinline__ void distort_dev(const CamDev& cam, double u, double v, double& ud, double& vd) {
    const double xu = (u - cam.Cx) * cam.dx;
    const double yu = (v - cam.Cy) * cam.dy;
    const double ru = sqrt(xu * xu + yu * yu);
    const double ru2 = ru * ru;
    double rd = ru / (1 + cam.k1 * ru2 + cam.k2 * (ru2 * ru2));
#pragma unroll
    for (int k = 0; k < 10; k++) {
        const double rd2 = rd * rd;
        const double rd3 = rd2 * rd;
        const double rd4 = rd2 * rd2;
        const double f = rd + cam.k1 * rd3 + cam.k2 * (rd4 * rd) - ru;
        const double fp = 1 + 3 * cam.k1 * rd2 + 5 * cam.k2 * rd4;
        rd = rd - f / fp;
    }
    const double rd2 = rd * rd;
    const double D = 1 + cam.k1 * rd2 + cam.k2 * (rd2 * rd2);
    ud = xu / D / cam.dx + cam.Cx;
    vd = yu / D / cam.dy + cam.Cy;
}

// Throughput variant for support scoring (hundreds of millions of calls per sweep): the same 10 Newton steps, but the step
// f / f' uses a refined single-precision reciprocal seed (rel. error ~1e-14) instead of an IEEE division -- Newton is
// self-correcting, so the converged rd agrees with distort_dev to the last bits -- and the final divisions share one reciprocal.
__device__ __forceinline__ double fast_rcp(double v) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(v));  // MUFU.RCP64H: ~20-bit seed, no float round trip
    r = r * fma(-v, r, 2.0);
    r = r * fma(-v, r, 2.0);
    return r;
}
// sin and cos together for support scoring: three-constant Cody-Waite reduction by pi/2 (exact enough for |a| < 1e5, like the fast
// path of the CUDA math library) + the classic degree-13 / degree-14 minimax kernels on [-pi/4, pi/4] (errors < 2^-57), ~30
// instructions instead of ~77 for the library sincos().  Larger arguments (and only those) take the library path.
__device__ __forceinline__ void sincos_fast(double a, double* sn, double* cs) {
    if (fabs(a) > 1.0e5) {
        sincos(a, sn, cs);
        return;
    }
    const double kf = rint(a * 6.36619772367581382433e-01);
    double r = fma(-kf, 1.57079632679489655800e+00, a);
    r = fma(-kf, 6.12323399573676603587e-17, r);
    r = fma(-kf, -1.49738490485916983378e-33, r);  // pi/2 - hi - mid
    const double z = r * r;
    double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
    ps = fma(z, ps, 2.75573137070700676789e-06);
    ps = fma(z, ps, -1.98412698298579493134e-04);
    ps = fma(z, ps, 8.33333333332248946124e-03);
    ps = fma(z, ps, -1.66666666666666324348e-01);
    const double s = fma(z * r, ps, r);
    double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
    pc = fma(z, pc, -2.75573143513906633035e-07);
    pc = fma(z, pc, 2.48015872894767294178e-05);
    pc = fma(z, pc, -1.38888888888741095749e-03);
    pc = fma(z, pc, 4.16666666666666019037e-02);
    const double c = fma(z * z, pc, fma(z, -0.5, 1.0));
    const int q = (int)kf;
    const double ss = (q & 1) ? c : s, cc = (q & 1) ? s : c;
    *sn = (q & 2) ? -ss : ss;
    *cs = ((q + 1) & 2) ? -cc : cc;
}
__device__ __forceinline__ void distort_fast_dev(const CamDev& cam, double u, double v, double& ud, double& vd) {
    const double xu = (u - cam.Cx) * cam.dx;
    const double yu = (v - cam.Cy) * cam.dy;
    const double ru = sqrt(xu * xu + yu * yu);
    const double ru2 = ru * ru;
    double rd = ru / (1 + cam.k1 * ru2 + cam.k2 * (ru2 * ru2));
#pragma unroll
    for (int k = 0; k < 10; k++) {
        const double rd2 = rd * rd;
        const double rd4 = rd2 * rd2;
        const double f = rd + cam.k1 * (rd2 * rd) + cam.k2 * (rd4 * rd) - ru;
        const double fp = 1 + 3 * cam.k1 * rd2 + 5 * cam.k2 * rd4;
        rd = fma(-f, fast_rcp(fp), rd);
    }
    const double rd2 = rd * rd;
    const double iD = 1.0 / (1 + cam.k1 * rd2 + cam.k2 * (rd2 * rd2));
    ud = xu * iD / cam.dx + cam.Cx;
    vd = yu * iD / cam.dy + cam.Cy;
}

// distort_fm for the latency path (one call per feature, on a kernel that is a single dependent chain per thread): the Newton
// iteration of src/ExtendKF.cpp:191-196 converges to a fixed point of its update in 3-5 steps and the reference's remaining steps
// leave rd unchanged, so iterating until rd stops changing (at most the reference's 10 steps) returns the same rd -- up to the last
// bit where the reciprocal-based step and the reference's division round differently (|d rd| <= 1 ulp, far inside the 1e-9 bar).
// The final undistorted -> distorted scaling keeps the reference's exact divisions.
__device__ __forceinline__ void distort_fixpoint_dev(const CamDev& cam, double u, double v, double& ud, double& vd) {
    const double xu = (u - cam.Cx) * cam.dx;
    const double yu = (v - cam.Cy) * cam.dy;
    const double ru = sqrt(xu * xu + yu * yu);
    const double ru2 = ru * ru;
    double rd = ru * fast_rcp(1 + cam.k1 * ru2 + cam.k2 * (ru2 * ru2));
#pragma unroll 1
    for (int k = 0; k < 10; k++) {
        const double rd2 = rd * rd;
        const double rd4 = rd2 * rd2;
        const double f = rd + cam.k1 * (rd2 * rd) + cam.k2 * (rd4 * rd) - ru;
        const double fp = 1 + 3 * cam.k1 * rd2 + 5 * cam.k2 * rd4;
        const double rn = fma(-f, fast_rcp(fp), rd);
        const bool same = !(rn != rd);
        rd = rn;
        if (same) break;
    }
    const double rd2 = rd * rd;
    const double D = 1 + cam.k1 * rd2 + cam.k2 * (rd2 * rd2);
    ud = xu / D / cam.dx + cam.Cx;
    vd = yu / D / cam.dy + cam.Cy;
}

// Jacobian of the undistortion (src/ExtendKF.cpp:312-332), row-major 2x2 (map_prep_add_dev in kernels_map.cuh has an unfused copy, kept in step by hand: change both)
__device__ __forceinline__ void jacob_undistort_dev(const CamDev& cam, double ud, double vd, double J[4]) {
    const double a = ud - cam.Cx, b = vd - cam.Cy;
    const double adx = a * cam.dx, bdy = b * cam.dy;
    const double rd2 = adx * adx + bdy * bdy;
    const double g = cam.k1 + 2 * cam.k2 * rd2;
    const double c = 1 + cam.k1 * rd2 + cam.k2 * rd2 * rd2;
    J[0] = c + a * g * (2 * a * cam.dx * cam.dx);
    J[1] = a * g * (2 * b * cam.dy * cam.dy);
    J[2] = b * g * (2 * a * cam.dx * cam.dx);
    J[3] = c + b * g * (2 * b * cam.dy * cam.dy);
}

// d(R(q) a)/dq, 3x4 row-major (src/ExtendKF.cpp:286-311) (map_prep_add_dev in kernels_map.cuh has an unfused copy, kept in step by hand: change both)
__device__ __forceinline__ void dRq_times_a_by_dq_dev(const double* q, const double* a, double o[12]) {
    const double q0 = q[0], q1 = q[1], q2 = q[2], q3 = q[3];
    // column 0
    o[0] = 2 * (q0 * a[0] - q3 * a[1] + q2 * a[2]);
    o[4] = 2 * (q3 * a[0] + q0 * a[1] - q1 * a[2]);
    o[8] = 2 * (-q2 * a[0] + q1 * a[1] + q0 * a[2]);
    // column 1
    o[1] = 2 * (q1 * a[0] + q2 * a[1] + q3 * a[2]);
    o[5] = 2 * (q2 * a[0] - q1 * a[1] - q0 * a[2]);
    o[9] = 2 * (q3 * a[0] + q0 * a[1] - q1 * a[2]);
    // column 2
    o[2] = 2 * (-q2 * a[0] + q1 * a[1] + q0 * a[2]);
    o[6] = 2 * (q1 * a[0] + q2 * a[1] + q3 * a[2]);
    o[10] = 2 * (-q0 * a[0] + q3 * a[1] - q2 * a[2]);
    // column 3
    o[3] = 2 * (-q3 * a[0] - q0 * a[1] + q1 * a[2]);
    o[7] = 2 * (q0 * a[0] - q3 * a[1] + q2 * a[2]);
    o[11] = 2 * (q1 * a[0] + q2 * a[1] + q3 * a[2]);
}

__device__ __forceinline__ int warp_sum_int(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace rslam
