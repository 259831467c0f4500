// oracle/rslam_oracle.cpp -- TEST INFRASTRUCTURE ONLY.  PARITY UNPINNED (see below).
//
// CPU restatement of the reference's 1-point-RANSAC EKF measurement-update path, written from the reference's
// algorithm (plumewind/ransac_slam, /root/reference) with an owned dense-matrix type instead of Eigen/OpenCV.
// Every function cites the reference file:line it follows.  It is the CHECKER for the CUDA path: only tests/,
// __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load it.  The shipped product
// (ransac_slam_b200/) never includes, links or calls anything in oracle/.
//
// PARITY UNPINNED: the reference has no tests, golden vectors or fixtures for this path (test/odometry.cpp is a
// ROS TF relay) and cannot be compiled here (needs ROS + OpenCV C++ + Eigen, all absent).  The oracle is pinned
// only by (i) the source text it follows, (ii) cv2 4.13 cross-checks of the two OpenCV primitives it restates
// (cv::remap, cv::calcCovarMatrix; tests/golden/), (iii) dense-vs-sparse self consistency and (iv) an
// independent numpy restatement of the update/S_i algebra (oracle/np_oracle.py).
//
// Modes:  dense  = reference-faithful operation order (dense 2 x n H_i, (H*P)*H^T, LU inverse, (K*S)*K^T, full
//                  (ncand+1)^2 covariance matrix in matching) -- this is what is timed as the CPU baseline;
//         sparse = same quantities, skipping the structural zeros of H_i and the unused covariance rows, so
//                  that test vectors at larger N finish in seconds.  Both modes must agree to <=1e-12.
//
// Quirks of the reference that change results are reproduced (SURVEY.md A.3) behind named switches that default
// to reference behaviour.
#include <cfenv>
#include <climits>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <string>

#include "omat.h"

namespace orc {

enum Quirk : unsigned {
    Q1_ANGLES_FROM_POSITIONS = 1u << 0,  // src/Tracking.cpp:448
    Q4_JNORM_INT_EXPONENT = 1u << 1,     // src/ExtendKF.cpp:627
    Q6_RESCUE_WITHOUT_R = 1u << 2,       // src/Tracking.cpp:589
    Q11_PATCH_OFFSET_MINUS1 = 1u << 3,   // src/Tracking.cpp:264-265
    Q_ALL = 0xFu
};

struct Cam {  // include/ransac_slam/System.h:69-82, filled at src/System.cpp:34-58
    double k1, k2;
    int nRows, nCols;
    double Cx, Cy, f, dx, dy;
    Mat K;  // 3x3: [f/d 0 Cx; 0 f/d Cy; 0 0 1]
};

struct Feature {  // include/ransac_slam/ExtendKF.h:14-42
    Mat patch_when_initialized;  // 41x41
    Mat patch_when_matching;     // 13x13
    Mat patch_template;          // 13x13, caller-supplied predicted appearance used when warp_patches == false
    double r_wc_when_initialized[3] = {0, 0, 0};
    Mat R_wc_when_initialized;  // 3x3
    double uv_when_initialized[2] = {0, 0};
    int half_patch_size_when_initialized = 20;
    int half_patch_size_when_matching = 6;
    int times_predicted = 0, times_measured = 0;
    int type = 0;  // 0 = "inversedepth", 1 = "cartesian"
    bool individually_compatible = false, low_innovation_inlier = false, high_innovation_inlier = false;
    bool has_z = false;
    double z[2] = {0, 0};
    bool has_h = false;
    double h[2] = {0, 0};
    Mat H;  // dense 2 x n (dense mode) -- always kept so tests can read it
    Mat S;  // 2x2
    Mat R;  // 2x2 identity (src/Map.cpp:310)
};

struct Filter {
    Cam cam;
    double std_a = 0.007, std_alpha = 0.007, std_z = 1.0;
    double eps = 2.220446049250313e-16;
    unsigned quirks = Q_ALL;
    bool sparse = false;     // false: dense reference-faithful mode
    bool fast_corr = false;  // true: only row 0 + diagonal of the correlation matrix
    bool warp_patches = true;
    std::vector<Feature> fi;
    Mat x_k_k, p_k_k, x_k_km1, p_k_km1;
    // diagnostics of the last ransac call
    int last_hyp_run = 0, last_best_support = 0, last_nhyp_final = 0, last_num_ic = 0;
    std::string err;
};

static int state_offset(const Filter& F, int idx) {  // 13 + sizes of preceding features (src/Tracking.cpp:153)
    int off = 13;
    for (int i = 0; i < idx; i++) off += F.fi[i].type == 0 ? 6 : 3;
    return off;
}
static int state_dim(const Filter& F) { return state_offset(F, (int)F.fi.size()); }

// ---------------------------------------------------------------------------------------------------------
// camera model helpers
// ---------------------------------------------------------------------------------------------------------
// src/ExtendKF.cpp:91-102
static Mat q2r(const double* q) {
    double x = q[1], y = q[2], z = q[3], r = q[0];
    Mat R(3, 3);
    R(0, 0) = r * r + x * x - y * y - z * z;
    R(0, 1) = 2 * (x * y - r * z);
    R(0, 2) = 2 * (z * x + r * y);
    R(1, 0) = 2 * (x * y + r * z);
    R(1, 1) = r * r - x * x + y * y - z * z;
    R(1, 2) = 2 * (y * z - r * x);
    R(2, 0) = 2 * (z * x - r * y);
    R(2, 1) = 2 * (y * z + r * x);
    R(2, 2) = r * r - x * x - y * y + z * z;
    return R;
}
// src/ExtendKF.cpp:153-174
static void hu(const Cam& cam, const double* yi, double* uv) {
    double u0 = cam.Cx, v0 = cam.Cy, f = cam.f;
    double ku = 1.0 / cam.dx, kv = 1.0 / cam.dy;
    uv[0] = u0 + (yi[0] / yi[2]) * f * ku;
    uv[1] = v0 + (yi[1] / yi[2]) * f * kv;
}
// src/ExtendKF.cpp:175-204 (vectorised over columns; uv is 2 x m)
static Mat distort_fm(const Cam& cam, const Mat& uv) {
    const double Cx = cam.Cx, Cy = cam.Cy, k1 = cam.k1, k2 = cam.k2, dx = cam.dx, dy = cam.dy;
    int m = uv.cols();
    Mat uvd(2, m);
    for (int c = 0; c < m; c++) {
        double xu = (uv(0, c) - Cx) * dx;
        double yu = (uv(1, c) - Cy) * dy;
        double ru = std::sqrt(std::pow(xu, 2) + std::pow(yu, 2));
        double rd = ru / (1 + k1 * std::pow(ru, 2) + k2 * std::pow(ru, 4));
        for (int k = 0; k < 10; k++) {
            double f = rd + k1 * std::pow(rd, 3) + k2 * std::pow(rd, 5) - ru;
            double f_p = 1 + 3 * k1 * std::pow(rd, 2) + 5 * k2 * std::pow(rd, 4);
            rd = rd - f / f_p;
        }
        double D = 1 + k1 * std::pow(rd, 2) + k2 * std::pow(rd, 4);
        uvd(0, c) = xu / D / dx + Cx;
        uvd(1, c) = yu / D / dy + Cy;
    }
    return uvd;
}
// src/ExtendKF.cpp:266-285
static Mat undistort_fm(const Cam& cam, const Mat& uvd) {
    const double Cx = cam.Cx, Cy = cam.Cy, k1 = cam.k1, k2 = cam.k2, dx = cam.dx, dy = cam.dy;
    int m = uvd.cols();
    Mat uvu(2, m);
    for (int c = 0; c < m; c++) {
        double xd = (uvd(0, c) - Cx) * dx;
        double yd = (uvd(1, c) - Cy) * dy;
        double rd = std::sqrt(std::pow(xd, 2) + std::pow(yd, 2));
        double D = 1 + k1 * std::pow(rd, 2) + k2 * std::pow(rd, 4);
        uvu(0, c) = xd * D / dx + Cx;
        uvu(1, c) = yd * D / dy + Cy;
    }
    return uvu;
}
// src/ExtendKF.cpp:312-332
static Mat jacob_undistor_fm(const Cam& cam, const double* uvd) {
    const double Cx = cam.Cx, Cy = cam.Cy, k1 = cam.k1, k2 = cam.k2, dx = cam.dx, dy = cam.dy;
    double rd2 = std::pow((uvd[0] - Cx) * dx, 2) + std::pow((uvd[1] - Cy) * dy, 2);
    double uu_ud = (1 + k1 * rd2 + k2 * rd2 * rd2) + (uvd[0] - Cx) * (k1 + 2 * k2 * rd2) * (2 * (uvd[0] - Cx) * dx * dx);
    double vu_vd = (1 + k1 * rd2 + k2 * rd2 * rd2) + (uvd[1] - Cy) * (k1 + 2 * k2 * rd2) * (2 * (uvd[1] - Cy) * dy * dy);
    double uu_vd = (uvd[0] - Cx) * (k1 + 2 * k2 * rd2) * (2 * (uvd[1] - Cy) * dy * dy);
    double vu_ud = (uvd[1] - Cy) * (k1 + 2 * k2 * rd2) * (2 * (uvd[0] - Cx) * dx * dx);
    Mat J(2, 2);
    J(0, 0) = uu_ud;
    J(0, 1) = uu_vd;
    J(1, 0) = vu_ud;
    J(1, 1) = vu_vd;
    return J;
}
// src/ExtendKF.cpp:286-311
static Mat dRq_times_a_by_dq(const double* q, const double* a) {
    Mat res(3, 4);
    double T[4][9] = {
        {2 * q[0], -2 * q[3], 2 * q[2], 2 * q[3], 2 * q[0], -2 * q[1], -2 * q[2], 2 * q[1], 2 * q[0]},
        {2 * q[1], 2 * q[2], 2 * q[3], 2 * q[2], -2 * q[1], -2 * q[0], 2 * q[3], 2 * q[0], -2 * q[1]},
        {-2 * q[2], 2 * q[1], 2 * q[0], 2 * q[1], 2 * q[2], 2 * q[3], -2 * q[0], 2 * q[3], -2 * q[2]},
        {-2 * q[3], -2 * q[0], 2 * q[1], 2 * q[0], -2 * q[3], 2 * q[2], 2 * q[1], 2 * q[2], 2 * q[3]}};
    for (int k = 0; k < 4; k++)
        for (int i = 0; i < 3; i++) res(i, k) = T[k][3 * i] * a[0] + T[k][3 * i + 1] * a[1] + T[k][3 * i + 2] * a[2];
    return res;
}
// src/ExtendKF.cpp:137-152
static void inversedepth2cartesian(const double* id, double* xyz) {
    double theta = id[3], phi = id[4], rho = id[5];
    double m[3] = {std::cos(phi) * std::sin(theta), -std::sin(phi), std::cos(phi) * std::cos(theta)};
    for (int i = 0; i < 3; i++) xyz[i] = id[i] + (1.0 / rho) * m[i];
}
// src/ExtendKF.cpp:103-132 ; returns false when the reference leaves zi empty
static bool hi_cartesian(const Cam& cam, const double* hrl, double* zi) {
    if ((std::atan2(hrl[0], hrl[2]) * 180 / M_PI < -60) || (std::atan2(hrl[0], hrl[2]) * 180 / M_PI > 60) ||
        (std::atan2(hrl[1], hrl[2]) * 180 / M_PI < -60) || (std::atan2(hrl[1], hrl[2]) * 180 / M_PI > 60))
        return false;
    Mat uv_u(2, 1);
    hu(cam, hrl, uv_u.data());
    Mat uv_d = distort_fm(cam, uv_u);
    if ((uv_d(0, 0) > 0) && (uv_d(0, 0) < cam.nCols) && (uv_d(1, 0) > 0) && (uv_d(1, 0) < cam.nRows)) {
        zi[0] = uv_d(0, 0);
        zi[1] = uv_d(1, 0);
        return true;
    }
    return false;
}
// src/ExtendKF.cpp:56-90
static void predict_camera_measurements(Filter& F, const Mat& xkk) {
    const double* t_wc = &xkk.a[0];
    Mat r_wc = q2r(&xkk.a[3]);
    int index = 13;
    for (size_t i = 0; i < F.fi.size(); i++) {
        Feature& ft = F.fi[i];
        double hrl[3], hi[2];
        if (ft.type == 0) {
            const double* yi = &xkk.a[index];
            double mi[3] = {std::cos(yi[4]) * std::sin(yi[3]), -std::sin(yi[4]), std::cos(yi[4]) * std::cos(yi[3])};
            double v[3];
            for (int k = 0; k < 3; k++) v[k] = (yi[k] - t_wc[k]) * yi[5] + mi[k];
            for (int k = 0; k < 3; k++) hrl[k] = r_wc(0, k) * v[0] + r_wc(1, k) * v[1] + r_wc(2, k) * v[2];  // r_wc^T * v
            if (hi_cartesian(F.cam, hrl, hi)) {
                ft.h[0] = hi[0];
                ft.h[1] = hi[1];
                ft.has_h = true;
            }
            index += 6;
        } else {
            const double* yi = &xkk.a[index];
            Mat rinv = inv3_fixed(r_wc);
            double v[3] = {yi[0] - t_wc[0], yi[1] - t_wc[1], yi[2] - t_wc[2]};
            for (int k = 0; k < 3; k++) hrl[k] = rinv(k, 0) * v[0] + rinv(k, 1) * v[1] + rinv(k, 2) * v[2];
            if (hi_cartesian(F.cam, hrl, hi)) {
                ft.h[0] = hi[0];
                ft.h[1] = hi[1];
                ft.has_h = true;
            }
            index += 3;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Jacobians  (src/Tracking.cpp:71-163, 540-573)
// ---------------------------------------------------------------------------------------------------------
static Mat mat3x1(const double* v) {
    Mat m(3, 1);
    m[0] = v[0];
    m[1] = v[1];
    m[2] = v[2];
    return m;
}
// src/Tracking.cpp:113-163
static void calculate_Hi_inverse_depth(Filter& F, const double* x_v, const double* yi, int order, int ncols, Mat& Hi) {
    const Cam& cam = F.cam;
    Hi.resize(2, ncols);
    Mat a1 = inv2_fixed(jacob_undistor_fm(cam, F.fi[order].h));
    double f = cam.f, ku = 1 / cam.dx, kv = 1 / cam.dy;
    Mat Rrw = inv3_fixed(q2r(&x_v[3]));
    double mi[3] = {std::cos(yi[4]) * std::sin(yi[3]), -std::sin(yi[4]), std::cos(yi[4]) * std::cos(yi[3])};
    double d[3];
    for (int k = 0; k < 3; k++) d[k] = (yi[k] - x_v[k]) * yi[5] + mi[k];
    Mat hc = Rrw * mat3x1(d);
    Mat a2(2, 3);
    a2(0, 0) = f * ku / (hc[2]);
    a2(0, 1) = 0;
    a2(0, 2) = -hc[0] * f * ku / (hc[2] * hc[2]);
    a2(1, 0) = 0;
    a2(1, 1) = f * kv / (hc[2]);
    a2(1, 2) = -hc[1] * f * kv / (hc[2] * hc[2]);
    Mat a12 = a1 * a2;
    Mat a30 = (a12 * neg(Rrw)) * yi[5];
    double b1[4] = {x_v[3], -x_v[4], -x_v[5], -x_v[6]};
    Mat dRq = dRq_times_a_by_dq(b1, d);
    Mat b0(3, 4);
    const double b2[4] = {1, -1, -1, -1};
    for (int j = 0; j < 4; j++)
        for (int i = 0; i < 3; i++) b0(i, j) = dRq(i, j) * b2[j];
    Mat a31 = a12 * b0;
    Hi.set_block(0, 0, a30);
    Hi.set_block(0, 3, a31);
    int ins = state_offset(F, order);
    Mat c0(3, 6);
    Mat c1 = yi[5] * Rrw;
    double c2[3] = {std::cos(yi[4]) * std::cos(yi[3]), 0, -std::cos(yi[4]) * std::sin(yi[3])};
    double c3[3] = {-std::sin(yi[4]) * std::sin(yi[3]), -std::cos(yi[4]), -std::sin(yi[4]) * std::cos(yi[3])};
    double dr[3] = {yi[0] - x_v[0], yi[1] - x_v[1], yi[2] - x_v[2]};
    c0.set_block(0, 0, c1);
    c0.set_block(0, 3, Rrw * mat3x1(c2));
    c0.set_block(0, 4, Rrw * mat3x1(c3));
    c0.set_block(0, 5, Rrw * mat3x1(dr));
    Hi.set_block(0, ins, a12 * c0);
}
// src/Tracking.cpp:71-112
static void calculate_Hi_cartesian(Filter& F, const double* x_v, const double* yi, int order, int ncols, Mat& Hi) {
    const Cam& cam = F.cam;
    Hi.resize(2, ncols);
    Mat a1 = inv2_fixed(jacob_undistor_fm(cam, F.fi[order].h));
    Mat Rrw = inv3_fixed(q2r(&x_v[3]));
    double f = cam.f, ku = 1 / cam.dx, kv = 1 / cam.dy;
    double d[3] = {yi[0] - x_v[0], yi[1] - x_v[1], yi[2] - x_v[2]};
    Mat hrl = Rrw * mat3x1(d);
    Mat a2(2, 3);
    a2(0, 0) = f * ku / (hrl[2]);
    a2(0, 1) = 0;
    a2(0, 2) = -hrl[0] * f * ku / (hrl[2] * hrl[2]);
    a2(1, 0) = 0;
    a2(1, 1) = f * kv / (hrl[2]);
    a2(1, 2) = -hrl[1] * f * kv / (hrl[2] * hrl[2]);
    Mat a12 = a1 * a2;
    Mat a30 = a12 * neg(Rrw);
    double b1[4] = {x_v[3], -x_v[4], -x_v[5], -x_v[6]};
    Mat dRq = dRq_times_a_by_dq(b1, d);
    Mat b0(3, 4);
    const double b2[4] = {1, -1, -1, -1};
    for (int j = 0; j < 4; j++)
        for (int i = 0; i < 3; i++) b0(i, j) = dRq(i, j) * b2[j];
    Mat a31 = a12 * b0;
    Hi.set_block(0, 0, a30);
    Hi.set_block(0, 3, a31);
    int ins = state_offset(F, order);
    Hi.set_block(0, ins, a12 * Rrw);
}
// src/Tracking.cpp:540-573
static void calculate_derivatives(Filter& F, const Mat& xk) {
    int ncols = state_dim(F);
    int index = 13;
    for (size_t i = 0; i < F.fi.size(); i++) {
        Feature& ft = F.fi[i];
        if (ft.has_h) {
            if (ft.type == 1)
                calculate_Hi_cartesian(F, &xk.a[0], &xk.a[index], (int)i, ncols, ft.H);
            else
                calculate_Hi_inverse_depth(F, &xk.a[0], &xk.a[index], (int)i, ncols, ft.H);
        }
        index += ft.type == 0 ? 6 : 3;
    }
}

// column indices where H_i can be non-zero (camera 0..12, own feature block)
static std::vector<int> nz_cols(const Filter& F, int i) {
    std::vector<int> c;
    for (int k = 0; k < 13; k++) c.push_back(k);
    int off = state_offset(F, i), sz = F.fi[i].type == 0 ? 6 : 3;
    for (int k = 0; k < sz; k++) c.push_back(off + k);
    return c;
}
// H_i * P * H_i^T, left to right (src/Tracking.cpp:42, :420, :589)
static Mat HPHt(const Filter& F, int i, const Mat& P) {
    const Mat& H = F.fi[i].H;
    if (!F.sparse) return mul_nt(H * P, H);
    std::vector<int> nz = nz_cols(F, i);
    int n = P.rows();
    Mat T(2, n);  // (H*P) restricted to the needed columns
    for (int jj : nz)
        for (int a = 0; a < 2; a++) {
            double s = 0;
            for (int kk : nz) s += H(a, kk) * P(kk, jj);
            T(a, jj) = s;
        }
    Mat S(2, 2);
    for (int a = 0; a < 2; a++)
        for (int b = 0; b < 2; b++) {
            double s = 0;
            for (int jj : nz) s += T(a, jj) * H(b, jj);
            S(a, b) = s;
        }
    return S;
}
// P * H_i^T  (n x 2)
static Mat PHt(const Filter& F, int i, const Mat& P) {
    const Mat& H = F.fi[i].H;
    if (!F.sparse) return mul_nt(P, H);
    std::vector<int> nz = nz_cols(F, i);
    int n = P.rows();
    Mat W(n, 2);
    for (int a = 0; a < 2; a++)
        for (int kk : nz) {
            double hv = H(a, kk);
            const double* pc = &P.a[(size_t)kk * n];
            for (int r = 0; r < n; r++) W(r, a) += pc[r] * hv;
        }
    return W;
}

// ---------------------------------------------------------------------------------------------------------
// OpenCV primitives restated (OpenCV 3.2 pinned by CMakeLists.txt:28-29; cross-checked against cv2 4.13,
// tests/golden/make_cv_fixtures.py)
// ---------------------------------------------------------------------------------------------------------
// cv::remap(src CV_32F, map1/map2 CV_32F, INTER_LINEAR, BORDER_CONSTANT, 0): map coordinates are quantised to 1/32 px
// (sx = cvRound(32*x) round-half-even, ix = sx>>5, fx = sx&31), weights (1-fx/32)(1-fy/32) ... as float; out-of-range
// taps read the border value 0.
// default rounding mode: to nearest even.  NaN and values outside int give INT_MIN, what cvRound's cvtsd2si returns on x86 (the
// cast alone would be undefined behaviour); remap then reads the border value
static inline int cv_round(double v) { return (v >= -2147483648.0 && v < 2147483648.0) ? (int)std::nearbyint(v) : INT_MIN; }
static Mat cv_remap_linear_const0(const Mat& src, const Mat& mapx, const Mat& mapy) {
    int orow = mapx.rows(), ocol = mapx.cols();
    Mat dst(orow, ocol);
    for (int i = 0; i < orow; i++)
        for (int j = 0; j < ocol; j++) {
            float mx = (float)mapx(i, j), my = (float)mapy(i, j);
            int sx = cv_round((double)(mx * 32.0f)), sy = cv_round((double)(my * 32.0f));
            int ix = sx >> 5, iy = sy >> 5;
            float fx = (float)(sx & 31) / 32.0f, fy = (float)(sy & 31) / 32.0f;
            float w00 = (1.f - fy) * (1.f - fx), w01 = (1.f - fy) * fx, w10 = fy * (1.f - fx), w11 = fy * fx;
            auto tap = [&](int yy, int xx) -> float {
                if (xx < 0 || yy < 0 || xx >= src.cols() || yy >= src.rows()) return 0.f;
                return (float)src(yy, xx);
            };
            float v = tap(iy, ix) * w00 + tap(iy, ix + 1) * w01 + tap(iy + 1, ix) * w10 + tap(iy + 1, ix + 1) * w11;
            dst(i, j) = (double)v;
        }
    return dst;
}
// Converter::corrcoef_opencv, src/Converter.cpp:188-209: cv::calcCovarMatrix(float in, CV_COVAR_NORMAL|CV_COVAR_ROWS)
// -> double (n_vars x n_vars) scatter matrix about the per-column mean, then /(cols-1), then normalised.
// M is (npix x nvar) with float-exact entries.  row0_only: compute just row 0 and the diagonal (same values).
static Mat corrcoef_opencv(const Mat& M, bool row0_only) {
    int np = M.rows(), nv = M.cols();
    std::vector<double> mean(nv);
    for (int j = 0; j < nv; j++) {
        double s = 0;
        for (int p = 0; p < np; p++) s += (double)(float)M(p, j);
        mean[j] = s * (1.0 / np);
    }
    Mat D(np, nv);
    for (int j = 0; j < nv; j++)
        for (int p = 0; p < np; p++) D(p, j) = (double)(float)M(p, j) - mean[j];
    Mat cov(nv, nv);
    if (!row0_only) {
        cov = D.t() * D;
    } else {
        for (int j = 0; j < nv; j++) {
            double s0 = 0, sd = 0;
            for (int p = 0; p < np; p++) {
                s0 += D(p, 0) * D(p, j);
                sd += D(p, j) * D(p, j);
            }
            cov(0, j) = s0;
            cov(j, 0) = s0;
            cov(j, j) = sd;
        }
    }
    double scale = (double)(nv - 1);  // M_cov = M_cov/(M_cov.cols - 1)   (src/Converter.cpp:196)
    for (size_t i = 0; i < cov.a.size(); i++) cov.a[i] = cov.a[i] / scale;
    Mat out(nv, nv);
    if (!row0_only) {
        for (int i = 0; i < nv; i++)
            for (int j = 0; j < nv; j++) out(i, j) = cov(i, j) / std::sqrt(cov(i, i) * cov(j, j));
    } else {
        for (int j = 0; j < nv; j++) out(0, j) = cov(0, j) / std::sqrt(cov(0, 0) * cov(j, j));
    }
    return out;
}

// ---------------------------------------------------------------------------------------------------------
// predicted appearance (src/Tracking.cpp:164-278)
// ---------------------------------------------------------------------------------------------------------
static Mat homog4(const Mat& R, const double* r) {  // [R 0;0 1]*[I r;0 1]   (src/Tracking.cpp:188-194, quirk Q12)
    Mat a = Mat::Identity(4), b = Mat::Identity(4);
    a.set_block(0, 0, R);
    for (int i = 0; i < 3; i++) b(i, 3) = r[i];
    return a * b;
}
static void pred_patch_fc(Filter& F, int order, const double* XYZ_w) {
    Feature& ft = F.fi[order];
    const Cam& cam = F.cam;
    const double* r_wc = &F.x_k_km1.a[0];
    Mat R_wc = q2r(&F.x_k_km1.a[3]);
    const double* uv_p_pred = ft.h;
    int halfW_pred = ft.half_patch_size_when_matching;
    int uv_len = halfW_pred * 2 + 1;
    Mat patch_pred;
    if ((uv_p_pred[0] > halfW_pred) && (uv_p_pred[0] < (cam.nCols - halfW_pred)) && (uv_p_pred[1] > halfW_pred) &&
        (uv_p_pred[1] < (cam.nRows - halfW_pred))) {
        if (!F.warp_patches) {  // synthetic configs: predicted appearance supplied by the caller
            ft.patch_when_matching = ft.patch_template;
            return;
        }
        const double* uv_p_f = ft.uv_when_initialized;
        int halfW_fea = ft.half_patch_size_when_initialized;
        double dx = cam.dx, f = cam.f, cx = cam.Cx, cy = cam.Cy;
        const Mat& K = cam.K;
        Mat H_Wk_p_f = homog4(ft.R_wc_when_initialized, ft.r_wc_when_initialized);
        Mat H_Wk = homog4(R_wc, r_wc);
        Mat H_kpf_k = inv4_fixed(H_Wk_p_f) * H_Wk;

        double n1[3] = {uv_p_f[0] - cx, uv_p_f[1] - cy, -f / dx};
        double nn = std::sqrt(n1[0] * n1[0] + n1[1] * n1[1] + n1[2] * n1[2]);
        double n[3] = {n1[0] / nn, n1[1] / nn, n1[2] / nn};
        Mat n2(4, 1);
        n2[0] = uv_p_pred[0] - cx;
        n2[1] = uv_p_pred[1] - cy;
        n2[2] = -f / dx;
        n2[3] = 1;
        Mat n_temp = H_kpf_k * n2;
        double nt[3] = {n_temp[0] / n_temp[3], n_temp[1] / n_temp[3], n_temp[2] / n_temp[3]};
        double ntn = std::sqrt(nt[0] * nt[0] + nt[1] * nt[1] + nt[2] * nt[2]);
        double ns[3] = {n[0] + nt[0] / ntn, n[1] + nt[1] / ntn, n[2] + nt[2] / ntn};
        double nsn = std::sqrt(ns[0] * ns[0] + ns[1] * ns[1] + ns[2] * ns[2]);
        for (int i = 0; i < 3; i++) n[i] = ns[i] / nsn;

        Mat XYZ_temp(4, 1);
        for (int i = 0; i < 3; i++) XYZ_temp[i] = XYZ_w[i];
        XYZ_temp[3] = 1;
        Mat XYZ_kpf = inv4_fixed(H_Wk_p_f) * XYZ_temp;
        double X3[3] = {XYZ_kpf[0] / XYZ_kpf[3], XYZ_kpf[1] / XYZ_kpf[3], XYZ_kpf[2] / XYZ_kpf[3]};
        double d = -(n[0] * X3[0] + n[1] * X3[1] + n[2] * X3[2]);

        // K * (R12 - t12 * n^T / d) * K^-1        (src/Tracking.cpp:226, :255)
        Mat R12 = H_kpf_k.block(0, 0, 3, 3);
        Mat tn(3, 3);
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++) tn(i, j) = (H_kpf_k(i, 3) * n[j]) / d;
        Mat Hm = (K * (R12 - tn)) * inv3_fixed(K);
        Mat Hm_inv = inv3_fixed(Hm);

        Mat uvf(2, 1);
        uvf[0] = uv_p_f[0];
        uvf[1] = uv_p_f[1];
        Mat uv_c1_und = undistort_fm(cam, uvf);
        Mat hom(3, 1);
        hom[0] = uv_c1_und[0];
        hom[1] = uv_c1_und[1];
        hom[2] = 1;
        Mat uv_temp = Hm_inv * hom;
        Mat uc_c2_und(2, 1);
        uc_c2_und[0] = uv_temp[0] / uv_temp[2];
        uc_c2_und[1] = uv_temp[1] / uv_temp[2];
        Mat uv_c2 = distort_fm(cam, uc_c2_und);

        // cv::Range(double,double) truncates toward zero (Q13); meshgrid_opencv is end-inclusive (src/Converter.cpp:30-47)
        int xs = (int)(uv_c2[0] - halfW_pred), xe = (int)(uv_c2[0] + halfW_pred);
        int ys = (int)(uv_c2[1] - halfW_pred), ye = (int)(uv_c2[1] + halfW_pred);
        std::vector<int> t_x, t_y;
        for (int i = xs; i <= xe; i++) t_x.push_back(i);
        for (int j = ys; j <= ye; j++) t_y.push_back(j);
        if ((int)t_x.size() != uv_len || (int)t_y.size() != uv_len) {
            // reference maps a 169-element view onto a differently sized grid here (UB); treat as "no prediction"
            ft.patch_when_matching = Mat::Zero(uv_len, uv_len);
            return;
        }
        int np = uv_len * uv_len;
        Mat uv_pred(2, np);  // column-major flatten of the meshgrid: idx = j*13 + i -> (t_x[j], t_y[i])
        for (int j = 0; j < uv_len; j++)
            for (int i = 0; i < uv_len; i++) {
                uv_pred(0, j * uv_len + i) = t_x[j];
                uv_pred(1, j * uv_len + i) = t_y[i];
            }
        Mat uv_c2_und = undistort_fm(cam, uv_pred);
        Mat homs(3, np);
        for (int c = 0; c < np; c++) {
            homs(0, c) = uv_c2_und(0, c);
            homs(1, c) = uv_c2_und(1, c);
            homs(2, c) = 1;
        }
        Mat uv_c1_h = Hm * homs;
        Mat uv_c1_u(2, np);
        for (int c = 0; c < np; c++) {
            uv_c1_u(0, c) = uv_c1_h(0, c) / uv_c1_h(2, c);
            uv_c1_u(1, c) = uv_c1_h(1, c) / uv_c1_h(2, c);
        }
        Mat uv_c1 = distort_fm(cam, uv_c1_u);
        double off = (F.quirks & Q11_PATCH_OFFSET_MINUS1) ? 1.0 : 0.0;
        Mat mapx(uv_len, uv_len), mapy(uv_len, uv_len);
        for (int j = 0; j < uv_len; j++)
            for (int i = 0; i < uv_len; i++) {
                mapx(i, j) = uv_c1(0, j * uv_len + i) - (uv_p_f[0] - halfW_fea - off);
                mapy(i, j) = uv_c1(1, j * uv_len + i) - (uv_p_f[1] - halfW_fea - off);
            }
        patch_pred = cv_remap_linear_const0(ft.patch_when_initialized, mapx, mapy);
    } else {
        patch_pred = Mat::Zero(uv_len, uv_len);
    }
    ft.patch_when_matching = patch_pred;
}

// ---------------------------------------------------------------------------------------------------------
// active search (src/Tracking.cpp:279-351)
// ---------------------------------------------------------------------------------------------------------
static void matching(Filter& F, const uint8_t* image, int rows, int cols, int stride) {
    (void)rows;
    (void)cols;
    const double correlation_threshold = 0.80;
    const double chi_095_2 = 5.9915;
    const Cam& cam = F.cam;
    for (size_t fidx = 0; fidx < F.fi.size(); fidx++) {
        Feature& ft = F.fi[fidx];
        if (!ft.has_h) continue;
        const double* h = ft.h;
        const Mat& S = ft.S;
        int hps = ft.half_patch_size_when_matching;
        int pix = (2 * hps + 1) * (2 * hps + 1);
        // SelfAdjointEigenSolver on 2x2 (lower triangle): largest eigenvalue
        double a = S(0, 0), b = S(1, 0), dd = S(1, 1);
        double lmax = 0.5 * (a + dd) + std::sqrt(0.25 * (a - dd) * (a - dd) + b * b);
        if (!(lmax < 100)) continue;
        const Mat& predicted_patch = ft.patch_when_matching;
        int hsx = (int)std::ceil(2 * std::sqrt(S(0, 0)));
        int hsy = (int)std::ceil(2 * std::sqrt(S(1, 1)));
        int maxc = (2 * hsx + 1) * (2 * hsy + 1) + 1;
        Mat patches(pix, maxc);
        std::vector<int> cand_x, cand_y;
        for (int p = 0; p < pix; p++) patches(p, 0) = predicted_patch[p];
        int idx = 0;
        int x_end = (int)std::round(h[0]) + hsx;
        int y_end = (int)std::round(h[1]) + hsy;
        Mat Sinv = lu_inverse(S);
        for (int j = (int)std::round(h[0]) - hsx; j <= x_end; j++) {
            for (int i = (int)std::round(h[1]) - hsy; i <= y_end; i++) {
                double nu0 = j - h[0], nu1 = i - h[1];
                // nu^T * S^-1 * nu, left to right
                double t0 = nu0 * Sinv(0, 0) + nu1 * Sinv(1, 0);
                double t1 = nu0 * Sinv(0, 1) + nu1 * Sinv(1, 1);
                double chi = t0 * nu0 + t1 * nu1;
                if (chi < chi_095_2) {
                    if ((j > hps) && (j < (cam.nCols - hps)) && (i > hps) && (i < (cam.nRows - hps))) {
                        idx++;
                        // image(Range(i-6,i+7), Range(j-6,j+7)) -> 13x13, flattened column-major
                        for (int c = 0; c < 2 * hps + 1; c++)
                            for (int r = 0; r < 2 * hps + 1; r++)
                                patches(c * (2 * hps + 1) + r, idx) = (double)image[(size_t)(i - hps + r) * stride + (j - hps + c)];
                        cand_x.push_back(j);
                        cand_y.push_back(i);
                    }
                }
            }
        }
        if (idx == 0) continue;  // Q10: reference divides by zero / maxCoeff on empty -> treated as "no match"
        Mat used = patches.block(0, 0, pix, idx + 1);
        Mat corr = corrcoef_opencv(used, F.fast_corr || F.sparse);
        // Eigen maxCoeff(&index): first maximum; NaN in slot 0 is sticky (visitor uses '>')
        double best = corr(0, 1);
        int bidx = 0;
        for (int c = 1; c < idx; c++) {
            double v = corr(0, c + 1);
            if (v > best) {
                best = v;
                bidx = c;
            }
        }
        if (best > correlation_threshold) {
            ft.individually_compatible = true;
            ft.z[0] = cand_x[bidx];
            ft.z[1] = cand_y[bidx];
            ft.has_z = true;
        }
    }
}

// src/Tracking.cpp:32-70
static void search_IC_matches(Filter& F, const uint8_t* image, int rows, int cols, int stride) {
    predict_camera_measurements(F, F.x_k_km1);
    calculate_derivatives(F, F.x_k_km1);
    for (size_t i = 0; i < F.fi.size(); i++)
        if (F.fi[i].has_h) F.fi[i].S = HPHt(F, (int)i, F.p_k_km1) + F.fi[i].R;
    int index = 13;
    double XYZ_w[3] = {0, 0, 0};
    for (size_t i = 0; i < F.fi.size(); i++) {
        if (F.fi[i].type == 1) {
            index += 3;  // Q3: XYZ_w not recomputed for cartesian features
        } else {
            inversedepth2cartesian(&F.x_k_km1.a[index], XYZ_w);
            index += 6;
        }
        if (F.fi[i].has_h) pred_patch_fc(F, (int)i, XYZ_w);
    }
    if (image) matching(F, image, rows, cols, stride);
}

// ---------------------------------------------------------------------------------------------------------
// 1-point RANSAC (src/Tracking.cpp:352-539).  u01: explicit uniform draws replacing ExtendKF::rand (Q8).
// returns 0 ok, 1 no IC matches (Q9), 2 cartesian matches present (Q2, reference UB), 3 u01 exhausted
// ---------------------------------------------------------------------------------------------------------
static int ransac_hypotheses(Filter& F, const double* u01, int n_u01) {
    const double p_at_least_one_spurious_free = 0.99;
    const double threshold = F.std_z;
    int n_hyp = 1000;
    int max_hypothesis_support = 0;
    const int n = F.x_k_km1.rows();
    const int feat_len = (int)F.fi.size();
    F.last_hyp_run = 0;
    F.last_best_support = 0;

    // state_vector_pattern + z_id / z_euc  (:361-397)
    std::vector<int> pos_r, pos_ang, pos_rho, pos_xyz;  // row indices selected by pattern columns 0..3
    std::vector<double> z_id, z_euc;
    int position = 13;
    for (int i = 0; i < feat_len; i++) {
        const Feature& ft = F.fi[i];
        if (ft.type == 0) {
            if (ft.has_z) {
                for (int k = 0; k < 3; k++) pos_r.push_back(position + k);
                pos_ang.push_back(position + 3);
                pos_ang.push_back(position + 4);
                pos_rho.push_back(position + 5);
                z_id.push_back(ft.z[0]);
                z_id.push_back(ft.z[1]);
            }
            position += 6;
        } else {
            if (ft.has_z) {
                for (int k = 0; k < 3; k++) pos_xyz.push_back(position + k);
                z_euc.push_back(ft.z[0]);
                z_euc.push_back(ft.z[1]);
            }
            position += 3;
        }
    }
    const int z_id_len = (int)z_id.size() / 2;
    const int z_euc_len = (int)z_euc.size() / 2;
    if (z_euc_len) return 2;  // Q2: nu = z_id - h_distorted with mismatched sizes in the reference

    std::vector<int> ic_pos;
    for (int j = 0; j < feat_len; j++)
        if (F.fi[j].individually_compatible) ic_pos.push_back(j);
    const int num_IC_matches = (int)ic_pos.size();
    F.last_num_ic = num_IC_matches;
    if (num_IC_matches == 0) return 1;  // Q9

    const Cam& cam = F.cam;
    int rc = 0;
    int i = 0;
    for (i = 0; i < n_hyp; i++) {
        if (i >= n_u01) {
            rc = 3;
            break;
        }
        double t = u01[i];
        int random_match_position = (int)std::floor(t * num_IC_matches);
        int pos = ic_pos[random_match_position];
        const Feature& fp = F.fi[pos];
        // S = Hi*P*Hi^T + R ; K = P*Hi^T*S^-1 ; xi = x + K*(zi - h^T)     (:419-422)
        Mat S = HPHt(F, pos, F.p_k_km1) + fp.R;
        Mat K = PHt(F, pos, F.p_k_km1) * lu_inverse(S);
        double innov[2] = {fp.z[0] - fp.h[0], fp.z[1] - fp.h[1]};
        std::vector<double> xi(n);
        for (int r = 0; r < n; r++) xi[r] = F.x_k_km1[r] + (K(r, 0) * innov[0] + K(r, 1) * innov[1]);
        F.last_hyp_run = i + 1;

        // compute_hypothesis_support_fast, inlined (:424-503)
        int hypothesis_support = 0;
        std::vector<char> inl_id(z_id_len, 0);
        Mat Rq = q2r(&xi[3]);  // rotcw = Rq^T
        double ku = 1 / cam.dx, f = cam.f, u0 = cam.Cx, v0 = cam.Cy;
        if (z_id_len) {
            std::vector<double> ri_v(3 * z_id_len), ang_v(2 * z_id_len), rho_v(z_id_len);
            for (int k = 0; k < 3 * z_id_len; k++) ri_v[k] = xi[pos_r[k]];
            for (int k = 0; k < 2 * z_id_len; k++) ang_v[k] = xi[pos_ang[k]];
            for (int k = 0; k < z_id_len; k++) rho_v[k] = xi[pos_rho[k]];
            // anglesi = Map(ri_v.data(), 2, m)   <- Q1 (reference)   |   Map(anglesi_v.data(), 2, m) (intended)
            const double* ang_src = (F.quirks & Q1_ANGLES_FROM_POSITIONS) ? ri_v.data() : ang_v.data();
            Mat himg(2, z_id_len);
            for (int c = 0; c < z_id_len; c++) {
                double a0 = ang_src[2 * c], a1 = ang_src[2 * c + 1];
                double mi[3] = {std::cos(a1) * std::sin(a0), -std::sin(a1), std::cos(a1) * std::cos(a0)};
                double v[3];
                for (int k = 0; k < 3; k++) {
                    double rm = ri_v[3 * c + k] - xi[k];
                    double byrho;
                    if (!F.sparse) {
                        // row * dense diag(rho): sum over all rows of the diagonal matrix (:449,:458-460)
                        byrho = 0.0;
                        for (int kk = 0; kk < z_id_len; kk++)
                            byrho += (ri_v[3 * kk + k] - xi[k]) * (kk == c ? rho_v[kk] : 0.0);
                    } else {
                        byrho = rm * rho_v[c];
                    }
                    v[k] = byrho + mi[k];
                }
                double hc[3];
                for (int k = 0; k < 3; k++) hc[k] = Rq(0, k) * v[0] + Rq(1, k) * v[1] + Rq(2, k) * v[2];
                double hn0 = hc[0] / hc[2], hn1 = hc[1] / hc[2];
                himg(0, c) = f * ku * hn0 + u0;
                himg(1, c) = f * ku * hn1 + v0;  // ku for both rows (:471)
            }
            Mat hd = distort_fm(cam, himg);
            for (int c = 0; c < z_id_len; c++) {
                double nu0 = z_id[2 * c] - hd(0, c), nu1 = z_id[2 * c + 1] - hd(1, c);
                double residual = std::sqrt(std::pow(nu0, 2) + std::pow(nu1, 2));
                if (residual < threshold) {
                    inl_id[c] = 1;
                    hypothesis_support++;
                }
            }
        }
        if (hypothesis_support > max_hypothesis_support) {  // (:507-535)
            max_hypothesis_support = hypothesis_support;
            int j_id = 0;
            for (int j = 0; j < feat_len; j++)
                if (F.fi[j].has_z) {
                    if (F.fi[j].type == 0) {
                        F.fi[j].low_innovation_inlier = inl_id[j_id] != 0;
                        j_id++;
                    }
                }
            double epsilon = 1 - ((double)hypothesis_support / (double)num_IC_matches);
            n_hyp = (int)std::ceil((std::log(1 - p_at_least_one_spurious_free)) / (std::log(1 - (1 - epsilon))));
            if (n_hyp == 0) break;
        }
        if (i > n_hyp) break;
    }
    F.last_best_support = max_hypothesis_support;
    F.last_nhyp_final = n_hyp;
    return rc;
}

// ---------------------------------------------------------------------------------------------------------
// joint EKF update (src/ExtendKF.cpp:559-678)
// ---------------------------------------------------------------------------------------------------------
// src/ExtendKF.cpp:597-639
static void update(Filter& F, const Mat& x_km_k, const Mat& p_km_k, const std::vector<int>& feats, const Mat& z, const Mat& h) {
    if (z.rows()) {
        const int n = p_km_k.rows(), k = z.rows();
        Mat R = Mat::Identity(k);
        Mat S, PHt_;
        if (!F.sparse) {
            Mat H(k, n);
            for (size_t t = 0; t < feats.size(); t++) H.set_block(2 * (int)t, 0, F.fi[feats[t]].H);
            S = mul_nt(H * p_km_k, H) + R;
            PHt_ = mul_nt(p_km_k, H);
        } else {
            // same quantities using only the structurally non-zero columns of each H_i
            PHt_ = Mat(n, k);
            for (size_t t = 0; t < feats.size(); t++) {
                Mat w = PHt(F, feats[t], p_km_k);
                PHt_.set_block(0, 2 * (int)t, w);
            }
            Mat HP(k, n);
            for (size_t t = 0; t < feats.size(); t++) {
                const Mat& Hi = F.fi[feats[t]].H;
                std::vector<int> nz = nz_cols(F, feats[t]);
                for (int a = 0; a < 2; a++)
                    for (int kk : nz) {
                        double hv = Hi(a, kk);
                        for (int c = 0; c < n; c++) HP(2 * (int)t + a, c) += hv * p_km_k(kk, c);
                    }
            }
            S = Mat(k, k);
            for (size_t t = 0; t < feats.size(); t++) {
                const Mat& Hi = F.fi[feats[t]].H;
                std::vector<int> nz = nz_cols(F, feats[t]);
                for (int b = 0; b < 2; b++)
                    for (int r = 0; r < k; r++) {
                        double s = 0;
                        for (int kk : nz) s += HP(r, kk) * Hi(b, kk);
                        S(r, 2 * (int)t + b) = s;
                    }
            }
            S = S + R;
        }
        Mat K = PHt_ * lu_inverse(S);
        Mat xkk = x_km_k + K * (z - h);
        Mat pkk_temp = p_km_k - mul_nt(K * S, K);
        Mat pkk(n, n);
        for (int j = 0; j < n; j++)
            for (int i = 0; i < n; i++) pkk(i, j) = 0.5 * pkk_temp(i, j) + 0.5 * pkk_temp(j, i);

        double r = xkk[3], x = xkk[4], y = xkk[5], zq = xkk[6];
        double nrm = std::sqrt(xkk[3] * xkk[3] + xkk[4] * xkk[4] + xkk[5] * xkk[5] + xkk[6] * xkk[6]);
        for (int i = 3; i < 7; i++) xkk[i] = xkk[i] / nrm;
        F.x_k_k = xkk;

        Mat temp(4, 4);
        double tv[16] = {x * x + y * y + zq * zq, -r * x, -r * y, -r * zq, -x * r, r * r + y * y + zq * zq, -x * y, -x * zq,
                         -y * r, -y * x, r * r + x * x + zq * zq, -y * zq, -zq * r, -zq * x, -zq * y, r * r + x * x + y * y};
        for (int i = 0; i < 4; i++)
            for (int j = 0; j < 4; j++) temp(i, j) = tv[4 * i + j];
        double s = (r * r + x * x + y * y + zq * zq);
        double scale = (F.quirks & Q4_JNORM_INT_EXPONENT) ? std::pow(s, (double)(-3 / 2)) : std::pow(s, -1.5);
        Mat Jnorm = scale * temp;
        Mat JnT = Jnorm.t();
        // (:629-634)
        Mat out = pkk;
        out.set_block(0, 3, pkk.block(0, 3, 3, 4) * JnT);
        out.set_block(3, 0, Jnorm * pkk.block(3, 0, 4, 3));
        out.set_block(3, 3, (Jnorm * pkk.block(3, 3, 4, 4)) * JnT);
        out.set_block(3, 7, Jnorm * pkk.block(3, 7, 4, n - 7));
        out.set_block(7, 3, pkk.block(7, 3, n - 7, 4) * JnT);
        F.p_k_k = out;
    } else {
        F.x_k_k = x_km_k;
        F.p_k_k = p_km_k;
    }
}
static void stack_and_update(Filter& F, bool hi, const Mat& x0, const Mat& P0) {  // :559-596 / :640-678
    std::vector<int> feats;
    for (size_t i = 0; i < F.fi.size(); i++)
        if (hi ? F.fi[i].high_innovation_inlier : F.fi[i].low_innovation_inlier) feats.push_back((int)i);
    Mat z(2 * (int)feats.size(), 1), h(2 * (int)feats.size(), 1);
    for (size_t t = 0; t < feats.size(); t++) {
        z[2 * t] = F.fi[feats[t]].z[0];
        z[2 * t + 1] = F.fi[feats[t]].z[1];
        h[2 * t] = F.fi[feats[t]].h[0];
        h[2 * t + 1] = F.fi[feats[t]].h[1];
    }
    update(F, x0, P0, feats, z, h);
}
static void ekf_update_li_inliers(Filter& F) {
    Mat x0 = F.x_k_km1, P0 = F.p_k_km1;  // by-value args at :597
    stack_and_update(F, false, x0, P0);
}
static void ekf_update_hi_inliers(Filter& F) {
    Mat x0 = F.x_k_k, P0 = F.p_k_k;
    stack_and_update(F, true, x0, P0);
}
// src/Tracking.cpp:574-597
static void rescue_hi_inliers(Filter& F) {
    const double chi2inv_2_95 = 5.9915;
    predict_camera_measurements(F, F.x_k_k);
    calculate_derivatives(F, F.x_k_k);
    for (size_t i = 0; i < F.fi.size(); i++) {
        Feature& ft = F.fi[i];
        if (ft.individually_compatible && !ft.low_innovation_inlier) {
            Mat Si = HPHt(F, (int)i, F.p_k_k);
            if (!(F.quirks & Q6_RESCUE_WITHOUT_R)) Si = Si + ft.R;
            double nu0 = ft.z[0] - ft.h[0], nu1 = ft.z[1] - ft.h[1];
            Mat Sinv = lu_inverse(Si);
            double t0 = nu0 * Sinv(0, 0) + nu1 * Sinv(1, 0);
            double t1 = nu0 * Sinv(0, 1) + nu1 * Sinv(1, 1);
            double chi = t0 * nu0 + t1 * nu1;
            ft.high_innovation_inlier = chi < chi2inv_2_95;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// constant-velocity prediction (src/ExtendKF.cpp:333-529)  -- SURVEY 8(f) "next" row 2
// ---------------------------------------------------------------------------------------------------------
static void v2q(const Filter& F, const double* v, double* q) {  // :428-443 (Q14: zero quaternion below eps)
    double theta = std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
    if (theta < F.eps) {
        q[0] = q[1] = q[2] = q[3] = 0;
    } else {
        double vn[3] = {v[0] / theta, v[1] / theta, v[2] / theta};
        double vnn = std::sqrt(vn[0] * vn[0] + vn[1] * vn[1] + vn[2] * vn[2]);
        q[0] = std::cos(theta / 2.0);
        for (int i = 0; i < 3; i++) q[i + 1] = std::sin(theta / 2.0) * (vn[i] / vnn);
    }
}
static void qprod(const Filter& F, const double* q, const double* wW, double dt, double* qp) {  // :416-427
    double v[3] = {wW[0] * dt, wW[1] * dt, wW[2] * dt};
    double p[4];
    v2q(F, v, p);
    const double* qv = q + 1;
    const double* pu = p + 1;
    double cr[3] = {qv[1] * pu[2] - qv[2] * pu[1], qv[2] * pu[0] - qv[0] * pu[2], qv[0] * pu[1] - qv[1] * pu[0]};
    qp[0] = q[0] * p[0] - (qv[0] * pu[0] + qv[1] * pu[1] + qv[2] * pu[2]);
    for (int i = 0; i < 3; i++) qp[i + 1] = (q[0] * pu[i] + p[0] * qv[i]) + cr[i];
}
static Mat dq3_by_dq1(const double* q) {  // :482-490
    Mat m(4, 4);
    double v[16] = {q[0], -q[1], -q[2], -q[3], q[1], q[0], -q[3], q[2], q[2], q[3], q[0], -q[1], q[3], -q[2], q[1], q[0]};
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) m(i, j) = v[4 * i + j];
    return m;
}
static double dq0_by_domegaA(double oA, double o, double dt) { return (-dt / 2.0) * (oA / o) * std::sin(o * dt / 2.0); }
static double dqA_by_domegaA(double oA, double o, double dt) {
    return (dt / 2.0) * oA * oA / (o * o) * std::cos(o * dt / 2.0) + (1.0 / o) * (1.0 - oA * oA / (o * o)) * std::sin(o * dt / 2.0);
}
static double dqA_by_domegaB(double oA, double oB, double o, double dt) {
    return (oA * oB / (o * o)) * ((dt / 2.0) * std::cos(o * dt / 2.0) - (1.0 / o) * std::sin(o * dt / 2.0));
}
static Mat dqomegadt_by_domega(const double* w, double dt) {  // :491-512
    double om = std::sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
    Mat m(4, 3);
    for (int j = 0; j < 3; j++) m(0, j) = dq0_by_domegaA(w[j], om, dt);
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) m(i + 1, j) = (i == j) ? dqA_by_domegaA(w[i], om, dt) : dqA_by_domegaB(w[i], w[j], om, dt);
    return m;
}
static void ekf_prediction(Filter& F) {  // :333-388, filter_type == "constant_velocity" (src/System.cpp:63)
    const double dt = 1;
    const int n = F.x_k_k.rows();
    const double* x = F.x_k_k.data();
    F.x_k_km1 = F.x_k_k;
    double qn[4];
    qprod(F, x + 3, x + 10, dt, qn);
    for (int i = 0; i < 3; i++) F.x_k_km1[i] = x[i] + x[7 + i] * dt;
    for (int i = 0; i < 4; i++) F.x_k_km1[3 + i] = qn[i];
    // dfv_by_dxv (:444-481)
    Mat Fm = Mat::Identity(13);
    double wdt[3] = {x[10] * dt, x[11] * dt, x[12] * dt}, qwt[4];
    v2q(F, wdt, qwt);
    double qd[16] = {qwt[0], -qwt[1], -qwt[2], -qwt[3], qwt[1], qwt[0], qwt[3], -qwt[2],
                     qwt[2], -qwt[3], qwt[0], qwt[1], qwt[3], qwt[2], -qwt[1], qwt[0]};
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) Fm(3 + i, 3 + j) = qd[4 * i + j];
    for (int i = 0; i < 3; i++) Fm(i, 7 + i) = dt;
    Mat ab = dq3_by_dq1(x + 3) * dqomegadt_by_domega(x + 10, dt);
    Fm.set_block(3, 10, ab);
    // Q = G*Pn*G^T (:347-376)
    double la = std::pow(F.std_a * dt, 2), aa = std::pow(F.std_alpha * dt, 2);
    Mat Pn(6, 6);
    for (int i = 0; i < 3; i++) {
        Pn(i, i) = la;
        Pn(3 + i, 3 + i) = aa;
    }
    Mat G(13, 6);
    for (int i = 0; i < 3; i++) {
        G(7 + i, i) = 1;
        G(10 + i, 3 + i) = 1;
        G(i, i) = dt;
    }
    G.set_block(3, 3, ab);
    Mat Q = mul_nt(G * Pn, G);
    const Mat& P = F.p_k_k;
    Mat out = P;  // pk_km5: bottom-right block copied (:382)
    Mat Pxx = P.block(0, 0, 13, 13);
    out.set_block(0, 0, mul_nt(Fm * Pxx, Fm) + Q);
    if (n > 13) {
        out.set_block(0, 13, Fm * P.block(0, 13, 13, n - 13));
        out.set_block(13, 0, mul_nt(P.block(13, 0, n - 13, 13), Fm));
    }
    F.p_k_km1 = out;
}
// Map::map_management step 2 (src/Map.cpp:34-55): per-frame counter update + flag reset
static void map_reset_flags(Filter& F) {
    for (auto& ft : F.fi) {
        if (ft.has_h) ft.times_predicted += 1;
        if (ft.low_innovation_inlier || ft.high_innovation_inlier) ft.times_measured += 1;
        ft.individually_compatible = false;
        ft.low_innovation_inlier = false;
        ft.high_innovation_inlier = false;
        ft.has_h = false;
        ft.has_z = false;
        ft.H.resize(0, 0);
        ft.S.resize(0, 0);
    }
}


// ---------------------------------------------------------------------------------------------------------
// Map management (src/Map.cpp) -- SURVEY 8f row 3
// ---------------------------------------------------------------------------------------------------------
// Map::delete_a_feature (src/Map.cpp:69-104).  feature_id is 1-based and the type is read from features_info[feature_id-1] as it
// stands at call time (map_management has already erased the record, src/Map.cpp:27-28).  Returns -4 where the reference reads out
// of range.
static int delete_a_feature(Filter& F, int feature_id) {
    if (feature_id - 1 < 0 || feature_id - 1 >= (int)F.fi.size()) return -4;
    int parToDelete = F.fi[feature_id - 1].type == 1 ? 3 : 6;
    int indexFromWichDelete = 14 - 1;
    for (int i = 0; i < feature_id - 1; i++) indexFromWichDelete += F.fi[i].type == 0 ? 6 : 3;
    const int n = F.x_k_k.rows();
    int delete_surplus = n - (indexFromWichDelete + parToDelete);
    if (delete_surplus < 0) return -4;
    Mat x_temp(n - parToDelete, 1);
    Mat p_temp(n - parToDelete, n - parToDelete);
    for (int i = 0; i < indexFromWichDelete; i++) x_temp[i] = F.x_k_k[i];
    for (int i = 0; i < delete_surplus; i++) x_temp[indexFromWichDelete + i] = F.x_k_k[n - delete_surplus + i];
    F.x_k_k = x_temp;
    const int a = indexFromWichDelete, d = delete_surplus;
    p_temp.set_block(0, 0, F.p_k_k.block(0, 0, a, a));
    p_temp.set_block(0, a, F.p_k_k.block(0, n - d, a, d));
    p_temp.set_block(a, 0, F.p_k_k.block(n - d, 0, d, a));
    p_temp.set_block(a, a, F.p_k_k.block(n - d, n - d, d, d));
    F.p_k_k = p_temp;
    return 0;
}

// Map::map_management step 1 (src/Map.cpp:19-32).  reference_indexing: pass the loop counter i to delete_a_feature exactly like the
// reference (it runs ahead of the iterator after the first erase); otherwise delete the state block of the erased record.
static int map_delete_pass(Filter& F, bool reference_indexing, int* n_deleted) {
    int i = 1, deleted = 0;
    for (size_t pos = 0; pos < F.fi.size(); i++) {
        const Feature& ft = F.fi[pos];
        if (ft.times_measured < ft.times_predicted * 0.5 && ft.times_predicted > 5) {
            if (reference_indexing) {
                F.fi.erase(F.fi.begin() + pos);
                int rc = delete_a_feature(F, i);
                if (rc) return rc;
            } else {
                // consistent variant: delete_a_feature reads the type at [id-1], so call it with the record's own id, then erase
                int rc = delete_a_feature(F, (int)pos + 1);
                if (rc) return rc;
                F.fi.erase(F.fi.begin() + pos);
            }
            deleted++;
        } else {
            pos++;
        }
    }
    if (n_deleted) *n_deleted = deleted;
    return state_dim(F) == F.x_k_k.rows() ? 0 : -4;
}

// Map::inversedepth_2_cartesian (src/Map.cpp:105-196): converts the first inverse-depth feature whose linearity index is below 0.1
// (dense J_all * P * J_all^T like the reference); returns its index or -1.
static int inversedepth_2_cartesian_map(Filter& F) {
    const double linearity_index_threshold = 0.1;
    Mat X = F.x_k_k, P = F.p_k_k;
    for (size_t i = 0; i < F.fi.size(); i++) {
        if (F.fi[i].type != 0) continue;
        int ip = state_offset(F, (int)i);
        double std_rho = std::sqrt(P(ip + 5, ip + 5));
        double rho = X[ip + 5];
        double std_d = std_rho / (rho * rho);
        double theta = X[ip + 3], phi = X[ip + 4];
        double mi[3] = {std::cos(phi) * std::sin(theta), -std::sin(phi), std::cos(phi) * std::cos(theta)};
        double X_out[3];
        inversedepth2cartesian(&X.a[ip], X_out);
        double a = 0, n1 = 0, n2 = 0;
        for (int k = 0; k < 3; k++) {
            a += (X_out[k] - X[ip + k]) * (X_out[k] - X[k]);
            n1 += (X_out[k] - X[ip + k]) * (X_out[k] - X[ip + k]);
            n2 += (X_out[k] - X[k]) * (X_out[k] - X[k]);
        }
        double d_c2p = std::sqrt(n2);
        double cos_alpha = a / (std::sqrt(n1) * std::sqrt(n2));
        double linearity_index = 4 * std_d * cos_alpha / d_c2p;
        if (linearity_index < linearity_index_threshold) {
            const int size_X_old = X.rows();
            Mat Xe(size_X_old - 3, 1);
            for (int k = 0; k < ip; k++) Xe[k] = X[k];
            for (int k = 0; k < 3; k++) Xe[ip + k] = X_out[k];
            for (int k = ip + 6; k < size_X_old; k++) Xe[k - 3] = X[k];
            F.x_k_k = Xe;
            double dmt[3] = {std::cos(phi) * std::cos(theta), 0, -std::cos(phi) * std::sin(theta)};
            double dmp[3] = {-std::sin(phi) * std::sin(theta), -std::cos(phi), -std::sin(phi) * std::cos(theta)};
            Mat J_all(size_X_old - 3, size_X_old);
            for (int k = 0; k < ip; k++) J_all(k, k) = 1.0;
            for (int r = 0; r < 3; r++) {
                J_all(ip + r, ip + r) = 1.0;
                J_all(ip + r, ip + 3) = (1 / rho) * dmt[r];
                J_all(ip + r, ip + 4) = (1 / rho) * dmp[r];
                J_all(ip + r, ip + 5) = -mi[r] / (rho * rho);
            }
            for (int k = ip + 6; k < size_X_old; k++) J_all(k - 3, k) = 1.0;
            F.p_k_k = mul_nt(J_all * P, J_all);
            F.fi[i].type = 1;
            return (int)i;
        }
    }
    return -1;
}

// ExtendKF::hinv (src/ExtendKF.cpp:236-265)
static void hinv(const Filter& F, const double* uvd, const double* Xv, double initial_rho, double* newFeature) {
    const Cam& cam = F.cam;
    double fku = cam.K(0, 0), fkv = cam.K(1, 1), U0 = cam.K(0, 2), V0 = cam.K(1, 2);
    Mat uvdm(2, 1);
    uvdm[0] = uvd[0];
    uvdm[1] = uvd[1];
    Mat uv = undistort_fm(cam, uvdm);
    double h_LR[3] = {-(U0 - uv[0]) / fku, -(V0 - uv[1]) / fkv, 1};
    Mat R = q2r(Xv + 3);
    double n[3];
    for (int r = 0; r < 3; r++) n[r] = R(r, 0) * h_LR[0] + R(r, 1) * h_LR[1] + R(r, 2) * h_LR[2];
    newFeature[0] = Xv[0];
    newFeature[1] = Xv[1];
    newFeature[2] = Xv[2];
    newFeature[3] = std::atan2(n[0], n[2]);
    newFeature[4] = std::atan2(-n[1], std::sqrt(n[0] * n[0] + n[2] * n[2]));
    newFeature[5] = initial_rho;
}

// Map::add_a_feature_covariance_inverse_depth (src/Map.cpp:339-400)
static Mat add_a_feature_covariance_inverse_depth(const Filter& F, const Mat& P, const double* uvd, const double* Xv) {
    const Cam& cam = F.cam;
    double fku = cam.K(0, 0), fkv = cam.K(1, 1), U0 = cam.K(0, 2), V0 = cam.K(1, 2);
    Mat R_wc = q2r(Xv + 3);
    Mat uvdm(2, 1);
    uvdm[0] = uvd[0];
    uvdm[1] = uvd[1];
    Mat uvu = undistort_fm(cam, uvdm);
    double XYZ_c[3] = {-(U0 - uvu[0]) / fku, -(V0 - uvu[1]) / fkv, 1};
    double XYZ_w[3];
    for (int r = 0; r < 3; r++) XYZ_w[r] = R_wc(r, 0) * XYZ_c[0] + R_wc(r, 1) * XYZ_c[1] + R_wc(r, 2) * XYZ_c[2];
    double X_w = XYZ_w[0], Y_w = XYZ_w[1], Z_w = XYZ_w[2];
    Mat dgw_dqwr = dRq_times_a_by_dq(Xv + 3, XYZ_c);
    Mat dtheta_dgw(1, 3), dphi_dgw(1, 3);
    dtheta_dgw[0] = Z_w / (X_w * X_w + Z_w * Z_w);
    dtheta_dgw[1] = 0;
    dtheta_dgw[2] = -X_w / (X_w * X_w + Z_w * Z_w);
    dphi_dgw[0] = (X_w * Y_w) / ((X_w * X_w + Y_w * Y_w + Z_w * Z_w) * std::sqrt(X_w * X_w + Z_w * Z_w));
    dphi_dgw[1] = -std::sqrt(X_w * X_w + Z_w * Z_w) / (X_w * X_w + Y_w * Y_w + Z_w * Z_w);
    dphi_dgw[2] = (Z_w * Y_w) / ((X_w * X_w + Y_w * Y_w + Z_w * Z_w) * std::sqrt(X_w * X_w + Z_w * Z_w));
    Mat dy_dxv(6, 13);
    for (int k = 0; k < 3; k++) dy_dxv(k, k) = 1.0;
    dy_dxv.set_block(3, 3, dtheta_dgw * dgw_dqwr);
    dy_dxv.set_block(4, 3, dphi_dgw * dgw_dqwr);
    Mat dyprima_dgw(5, 3);
    dyprima_dgw.set_block(3, 0, dtheta_dgw);
    dyprima_dgw.set_block(4, 0, dphi_dgw);
    // src/Map.cpp:375-379: `Eigen::Matrix<double,3,2> dgc_dhu; dgc_dhu << 1/fku, 0, 0, 0, 1/fkv, 0;` -- the comma initialiser fills
    // ROW BY ROW, so the matrix is [1/fku 0; 0 0; 1/fkv 0] (the MATLAB original had the transpose of a 2 x 3).  Quirk Q16, found by
    // running the reference's own Map.cpp (oracle/_ref); reproduced.
    Mat dgc_dhu(3, 2);
    dgc_dhu(0, 0) = 1 / fku;
    dgc_dhu(2, 0) = 1 / fkv;
    Mat dhu_dhd = jacob_undistor_fm(cam, uvd);
    Mat dyprima_dhd = dyprima_dgw * R_wc * dgc_dhu * dhu_dhd;
    Mat dy_dhd(6, 3);
    dy_dhd.set_block(0, 0, dyprima_dhd);
    dy_dhd(5, 2) = 1;
    Mat Padd(3, 3);
    Padd(0, 0) = Padd(1, 1) = std::pow(F.std_z, 2);
    Padd(2, 2) = std::pow(1, 2);
    const int P_len = P.rows();
    Mat P_xv = P.block(0, 0, 13, 13);
    Mat P_yxv = P.block(13, 0, P_len - 13, 13);
    Mat P_y = P.block(13, 13, P_len - 13, P_len - 13);
    Mat P_xvy = P.block(0, 13, 13, P_len - 13);
    Mat P_RES1 = mul_nt(P_xv, dy_dxv);
    Mat P_RES2 = mul_nt(P_yxv, dy_dxv);
    Mat P_RES3 = mul_nt(dy_dxv * P_xv, dy_dxv) + mul_nt(dy_dhd * Padd, dy_dhd);
    Mat P_RES(P_len + 6, P_len + 6);
    P_RES.set_block(0, 0, P_xv);
    P_RES.set_block(0, 13, P_xvy);
    P_RES.set_block(0, P_len, P_RES1);
    P_RES.set_block(13, 0, P_yxv);
    P_RES.set_block(13, 13, P_y);
    P_RES.set_block(13, P_len, P_RES2);
    P_RES.set_block(P_len, 0, dy_dxv * P_xv);
    P_RES.set_block(P_len, 13, dy_dxv * P_xvy);
    P_RES.set_block(P_len, P_len, P_RES3);
    return P_RES;
}

// step 4 of Map::initialize_a_features (src/Map.cpp:268-311) for a given corner uv: state, covariance and the feature record
static int map_add_feature(Filter& F, const double* uv, const uint8_t* image, int rows, int cols, int stride) {
    const int initial_rho = 1;
    Mat X_RES = F.x_k_k, P_RES = F.p_k_k;
    double Xv[13];
    for (int k = 0; k < 13; k++) Xv[k] = F.x_k_k[k];
    double newFeature[6];
    hinv(F, uv, Xv, initial_rho, newFeature);
    Mat Xn(X_RES.rows() + 6, 1);
    for (int k = 0; k < X_RES.rows(); k++) Xn[k] = X_RES[k];
    for (int k = 0; k < 6; k++) Xn[X_RES.rows() + k] = newFeature[k];
    F.p_k_k = add_a_feature_covariance_inverse_depth(F, P_RES, uv, Xv);
    F.x_k_k = Xn;
    Feature nf;
    nf.patch_when_initialized = Mat(41, 41);
    const int u0 = (int)(uv[0] - 20), v0 = (int)(uv[1] - 20);  // cv::Range(double) truncates (src/Map.cpp:286)
    for (int r = 0; r < 41; r++)
        for (int c = 0; c < 41; c++) {
            int gy = v0 + r, gx = u0 + c;
            nf.patch_when_initialized(r, c) = (image && gx >= 0 && gx < cols && gy >= 0 && gy < rows) ? image[(size_t)gy * stride + gx] : 0;
        }
    nf.patch_when_matching = Mat(13, 13);
    nf.patch_template = Mat(13, 13);
    for (int k = 0; k < 3; k++) nf.r_wc_when_initialized[k] = Xn[k];
    nf.R_wc_when_initialized = q2r(&Xn.a[3]);
    nf.uv_when_initialized[0] = uv[0];
    nf.uv_when_initialized[1] = uv[1];
    nf.type = 0;
    nf.R = Mat::Identity(2);
    F.fi.push_back(nf);
    return (int)F.fi.size() - 1;
}


// ---------------------------------------------------------------------------------------------------------
// Feature initialisation: cv::FAST + Map::initialize_features (src/Map.cpp:198-338) -- SURVEY 8f row 4
// ---------------------------------------------------------------------------------------------------------
// cv::FAST(image, keypoints, threshold, nonmaxSuppression = true) with the default TYPE_9_16, restated from the published
// algorithm (OpenCV 3.2, pinned by CMakeLists.txt:28-29; modules/features2d/src/fast.cpp FAST_t<16> + fast_score.cpp
// cornerScore<16>): a pixel is a corner iff 9 contiguous pixels of the 16-pixel Bresenham circle of radius 3 are all darker than
// v - t or all brighter than v + t; its score is the largest t for which that still holds; with non-maximum suppression a corner is
// kept iff its score is strictly greater than the scores of its 8 neighbours (non-corners count 0).  Keypoints come out row by row,
// left to right; the 3-pixel border is never tested.  Pinned against cv2 4.13 by tests/golden/fast_fixtures.npz.
static const int kFastRing[16][2] = {{0, 3},  {1, 3},   {2, 2},   {3, 1},   {3, 0},  {3, -1}, {2, -2}, {1, -3},
                                     {0, -3}, {-1, -3}, {-2, -2}, {-3, -1}, {-3, 0}, {-3, 1}, {-2, 2}, {-1, 3}};  // (dx, dy)
static int fast9_strength(const uint8_t* img, int stride, int x, int y) {
    // max over the 16 arcs of 9 contiguous ring pixels of min(v - ring) ("darker" arc) and of min(ring - v) ("brighter" arc)
    const int v = img[(size_t)y * stride + x];
    int d[25];
    for (int k = 0; k < 25; k++) d[k] = v - img[(size_t)(y + kFastRing[k % 16][1]) * stride + (x + kFastRing[k % 16][0])];
    int best = -256;
    for (int s0 = 0; s0 < 16; s0++) {
        int a = 256, b = 256;
        for (int j = 0; j < 9; j++) {
            a = std::min(a, d[s0 + j]);
            b = std::min(b, -d[s0 + j]);
        }
        best = std::max(best, std::max(a, b));
    }
    return best;
}
static void fast9(const uint8_t* img, int rows, int cols, int stride, int threshold, bool nonmax, std::vector<int>& xs, std::vector<int>& ys) {
    xs.clear();
    ys.clear();
    threshold = std::min(std::max(threshold, 0), 255);
    if (rows < 7 || cols < 7) return;
    std::vector<int> score((size_t)rows * cols, 0);
    for (int y = 3; y < rows - 3; y++)
        for (int x = 3; x < cols - 3; x++) {
            int sgth = fast9_strength(img, stride, x, y);
            if (sgth > threshold) score[(size_t)y * cols + x] = nonmax ? sgth - 1 : 1;
        }
    for (int y = 3; y < rows - 3; y++)
        for (int x = 3; x < cols - 3; x++) {
            const int sc = score[(size_t)y * cols + x];
            if (!sc) continue;
            bool keep = true;
            if (nonmax)
                for (int dy = -1; dy <= 1 && keep; dy++)
                    for (int dx = -1; dx <= 1; dx++)
                        if ((dx || dy) && !(sc > score[(size_t)(y + dy) * cols + (x + dx)])) {
                            keep = false;
                            break;
                        }
            if (keep) {
                xs.push_back(x);
                ys.push_back(y);
            }
        }
}

// Map::initialize_a_features (src/Map.cpp:212-323) with the two uniform draws of `rand(2,1,0,1)` (:231) supplied by the caller.
// Returns 1 if a feature was added.
static int initialize_a_features(Filter& F, int step, const uint8_t* image, int rows, int cols, int stride, const double* u2) {
    (void)step;
    const int excluded_band = 21;
    const int semi[2] = {30, 20};
    predict_camera_measurements(F, F.x_k_k);
    std::vector<std::pair<double, double>> h_pred;
    for (auto& ft : F.fi)
        if (ft.has_h) h_pred.push_back({ft.h[0], ft.h[1]});
    double cx = std::round(u2[0] * (F.cam.nCols - 2 * excluded_band - 2 * semi[0])) + excluded_band + semi[0];
    double cy = std::round(u2[1] * (F.cam.nRows - 2 * excluded_band - 2 * semi[1])) + excluded_band + semi[1];
    const int x0 = (int)(cx - semi[0]), y0 = (int)(cy - semi[1]);  // cv::Range truncation
    const int wr = (int)(cy + semi[1] + 1) - y0, wc = (int)(cx + semi[0] + 1) - x0;
    (void)rows;
    (void)cols;
    std::vector<int> kx, ky;
    fast9(image + (size_t)y0 * stride + x0, wr, wc, stride, 100, true, kx, ky);
    int added = 0;
    int features_in_the_box = 0;
    for (auto& h : h_pred)
        if (h.first > (cx - semi[0]) && h.first < (cx + semi[0]) && h.second > (cy - semi[1]) && h.second < (cy + semi[1])) features_in_the_box++;
    if (!kx.empty() && !features_in_the_box) {
        // MATLAB-style "- 1" kept by the port (src/Map.cpp:243-244): the corner is shifted one pixel up and left
        double uv[2] = {kx[0] + (-semi[0] + cx - 1), ky[0] + (-semi[1] + cy - 1)};
        map_add_feature(F, uv, image, F.cam.nRows, F.cam.nCols, stride);
        added = 1;
    }
    for (auto& ft : F.fi) ft.has_h = false;  // :320-322
    return added;
}

// Map::initialize_features (src/Map.cpp:198-211): u01 holds 2 draws per attempt; returns the number of features initialised, or -1
// if the draws ran out before the loop ended
static int initialize_features(Filter& F, int step, int min_features_to_init, const uint8_t* image, int rows, int cols, int stride, const double* u01,
                               int n_pairs, int* attempts_out) {
    const int max_attempts = 50;
    int attempts = 0, initialized = 0;
    while (initialized < min_features_to_init && attempts < max_attempts) {
        if (attempts >= n_pairs) {
            if (attempts_out) *attempts_out = attempts;
            return -1;
        }
        initialized += initialize_a_features(F, step, image, rows, cols, stride, u01 + 2 * attempts);
        attempts++;
    }
    if (attempts_out) *attempts_out = attempts;
    return initialized;
}

// Map::map_management (src/Map.cpp:16-67)
static int map_management(Filter& F, const uint8_t* image, int rows, int cols, int stride, int step, int min_features, bool reference_indexing,
                          const double* u01, int n_pairs, int* info3) {
    int nd = 0;
    int rc = map_delete_pass(F, reference_indexing, &nd);
    if (rc) return rc;
    int measured = 0;
    for (auto& ft : F.fi)
        if (ft.low_innovation_inlier || ft.high_innovation_inlier) measured++;
    map_reset_flags(F);
    int conv = inversedepth_2_cartesian_map(F);
    int attempts = 0, init = 0;
    if (measured == 0)
        init = initialize_features(F, step, min_features, image, rows, cols, stride, u01, n_pairs, &attempts);
    else if (measured < min_features)
        init = initialize_features(F, step, min_features - measured, image, rows, cols, stride, u01, n_pairs, &attempts);
    if (info3) {
        info3[0] = nd;
        info3[1] = conv;
        info3[2] = init;
        info3[3] = attempts;
    }
    return init < 0 ? -5 : 0;
}

}  // namespace orc

// ---------------------------------------------------------------------------------------------------------
// C interface for ctypes (tests / bench cpu_baseline only)
// ---------------------------------------------------------------------------------------------------------
using namespace orc;
extern "C" {

void* orc_create(const double* cam9, double std_a, double std_alpha, double std_z) {
    Filter* F = new Filter();
    F->cam.k1 = cam9[0];
    F->cam.k2 = cam9[1];
    F->cam.nRows = (int)cam9[2];
    F->cam.nCols = (int)cam9[3];
    F->cam.Cx = cam9[4];
    F->cam.Cy = cam9[5];
    F->cam.f = cam9[6];
    F->cam.dx = cam9[7];
    F->cam.dy = cam9[8];
    F->cam.K = Mat::Identity(3);
    F->cam.K(0, 0) = F->cam.f / F->cam.dx;  // cam.K << (cam.f/d), 0, Cx ... with d == dx (src/System.cpp:58)
    F->cam.K(1, 1) = F->cam.f / F->cam.dx;
    F->cam.K(0, 2) = F->cam.Cx;
    F->cam.K(1, 2) = F->cam.Cy;
    F->std_a = std_a;
    F->std_alpha = std_alpha;
    F->std_z = std_z;
    return F;
}
void orc_destroy(void* h) { delete (Filter*)h; }
void orc_set_options(void* h, unsigned quirks, int sparse, int fast_corr, int warp_patches) {
    Filter* F = (Filter*)h;
    F->quirks = quirks;
    F->sparse = sparse != 0;
    F->fast_corr = fast_corr != 0;
    F->warp_patches = warp_patches != 0;
}
void orc_set_threads(int n) { set_threads(n); }
int orc_num_features(void* h) { return (int)((Filter*)h)->fi.size(); }
int orc_state_dim(void* h) { return state_dim(*(Filter*)h); }
// which: 0 = x_k_k/p_k_k, 1 = x_k_km1/p_k_km1.  P column-major n x n, contiguous.
void orc_set_state(void* h, int which, const double* x, const double* P, int n) {
    Filter* F = (Filter*)h;
    Mat& xv = which ? F->x_k_km1 : F->x_k_k;
    Mat& Pm = which ? F->p_k_km1 : F->p_k_k;
    xv.resize(n, 1);
    std::memcpy(xv.data(), x, sizeof(double) * n);
    Pm.resize(n, n);
    std::memcpy(Pm.data(), P, sizeof(double) * (size_t)n * n);
}
void orc_get_state(void* h, int which, double* x, double* P) {
    Filter* F = (Filter*)h;
    const Mat& xv = which ? F->x_k_km1 : F->x_k_k;
    const Mat& Pm = which ? F->p_k_km1 : F->p_k_k;
    if (x) std::memcpy(x, xv.data(), sizeof(double) * xv.size());
    if (P) std::memcpy(P, Pm.data(), sizeof(double) * Pm.size());
}
// patch_init: 41x41 row-major uint8 (as cut from the image) or NULL; patch_match: 13x13 row-major float-exact doubles or NULL
int orc_add_feature(void* h, int type, const uint8_t* patch_init, const double* patch_match, const double* r_wc, const double* R_wc_rowmajor,
                    const double* uv) {
    Filter* F = (Filter*)h;
    Feature ft;
    ft.type = type;
    ft.patch_when_initialized = Mat(41, 41);
    if (patch_init)
        for (int r = 0; r < 41; r++)
            for (int c = 0; c < 41; c++) ft.patch_when_initialized(r, c) = patch_init[r * 41 + c];
    ft.patch_when_matching = Mat(13, 13);
    if (patch_match)
        for (int r = 0; r < 13; r++)
            for (int c = 0; c < 13; c++) ft.patch_when_matching(r, c) = patch_match[r * 13 + c];
    ft.patch_template = ft.patch_when_matching;
    ft.R_wc_when_initialized = Mat::Identity(3);
    if (R_wc_rowmajor)
        for (int r = 0; r < 3; r++)
            for (int c = 0; c < 3; c++) ft.R_wc_when_initialized(r, c) = R_wc_rowmajor[3 * r + c];
    if (r_wc)
        for (int k = 0; k < 3; k++) ft.r_wc_when_initialized[k] = r_wc[k];
    if (uv) {
        ft.uv_when_initialized[0] = uv[0];
        ft.uv_when_initialized[1] = uv[1];
    }
    ft.R = Mat::Identity(2);
    F->fi.push_back(ft);
    return (int)F->fi.size() - 1;
}
void orc_set_patch_matching(void* h, int i, const double* patch_rowmajor13) {
    Filter* F = (Filter*)h;
    for (int r = 0; r < 13; r++)
        for (int c = 0; c < 13; c++) F->fi[i].patch_when_matching(r, c) = patch_rowmajor13[r * 13 + c];
}
void orc_get_patch_matching(void* h, int i, double* patch_rowmajor13) {
    Filter* F = (Filter*)h;
    for (int r = 0; r < 13; r++)
        for (int c = 0; c < 13; c++) patch_rowmajor13[r * 13 + c] = F->fi[i].patch_when_matching(r, c);
}
// direct injection of matches (skips active search): z (2N), ic flags (N)
void orc_set_matches(void* h, const double* z, const uint8_t* ic) {
    Filter* F = (Filter*)h;
    for (size_t i = 0; i < F->fi.size(); i++) {
        F->fi[i].individually_compatible = ic[i] != 0;
        F->fi[i].has_z = ic[i] != 0;
        F->fi[i].z[0] = z[2 * i];
        F->fi[i].z[1] = z[2 * i + 1];
    }
}
void orc_map_reset_flags(void* h) { map_reset_flags(*(Filter*)h); }
void orc_ekf_prediction(void* h) { ekf_prediction(*(Filter*)h); }
void orc_search_ic_matches(void* h, const uint8_t* image, int rows, int cols, int stride) {
    search_IC_matches(*(Filter*)h, image, rows, cols, stride);
}
int orc_ransac_hypotheses(void* h, const double* u01, int n_u01) { return ransac_hypotheses(*(Filter*)h, u01, n_u01); }
void orc_ransac_info(void* h, int* out4) {
    Filter* F = (Filter*)h;
    out4[0] = F->last_hyp_run;
    out4[1] = F->last_best_support;
    out4[2] = F->last_nhyp_final;
    out4[3] = F->last_num_ic;
}
void orc_update_li(void* h) { ekf_update_li_inliers(*(Filter*)h); }
void orc_rescue_hi(void* h) { rescue_hi_inliers(*(Filter*)h); }
void orc_update_hi(void* h) { ekf_update_hi_inliers(*(Filter*)h); }

// per-feature outputs: h[2N], S[4N] (row-major 2x2), z[2N], flags[4N] = {has_h, ic, li, hi}, counters[2N]
void orc_get_features(void* hd, double* h, double* S, double* z, uint8_t* flags, int* counters) {
    Filter* F = (Filter*)hd;
    for (size_t i = 0; i < F->fi.size(); i++) {
        const Feature& ft = F->fi[i];
        if (h) {
            h[2 * i] = ft.h[0];
            h[2 * i + 1] = ft.h[1];
        }
        if (S) {
            for (int a = 0; a < 2; a++)
                for (int b = 0; b < 2; b++) S[4 * i + 2 * a + b] = (ft.S.rows() == 2) ? ft.S(a, b) : 0.0;
        }
        if (z) {
            z[2 * i] = ft.z[0];
            z[2 * i + 1] = ft.z[1];
        }
        if (flags) {
            flags[4 * i] = ft.has_h;
            flags[4 * i + 1] = ft.individually_compatible;
            flags[4 * i + 2] = ft.low_innovation_inlier;
            flags[4 * i + 3] = ft.high_innovation_inlier;
        }
        if (counters) {
            counters[2 * i] = ft.times_predicted;
            counters[2 * i + 1] = ft.times_measured;
        }
    }
}
// dense H of feature i: 2 x n row-major into out (zeros if not computed)
void orc_get_H(void* hd, int i, double* out) {
    Filter* F = (Filter*)hd;
    int n = state_dim(*F);
    const Mat& H = F->fi[i].H;
    for (int a = 0; a < 2; a++)
        for (int c = 0; c < n; c++) out[(size_t)a * n + c] = (H.rows() == 2 && H.cols() == n) ? H(a, c) : 0.0;
}
// stand-alone primitives for the cv2 cross-check fixtures
void orc_cv_remap(const double* src, int srows, int scols, const double* mapx, const double* mapy, int orows, int ocols, double* dst) {
    Mat s(srows, scols), mx(orows, ocols), my(orows, ocols);
    for (int r = 0; r < srows; r++)
        for (int c = 0; c < scols; c++) s(r, c) = src[r * scols + c];
    for (int r = 0; r < orows; r++)
        for (int c = 0; c < ocols; c++) {
            mx(r, c) = mapx[r * ocols + c];
            my(r, c) = mapy[r * ocols + c];
        }
    Mat d = cv_remap_linear_const0(s, mx, my);
    for (int r = 0; r < orows; r++)
        for (int c = 0; c < ocols; c++) dst[r * ocols + c] = d(r, c);
}
void orc_corrcoef(const double* M_rowmajor, int np, int nv, int row0_only, double* out_rowmajor) {
    Mat M(np, nv);
    for (int r = 0; r < np; r++)
        for (int c = 0; c < nv; c++) M(r, c) = M_rowmajor[r * nv + c];
    Mat o = corrcoef_opencv(M, row0_only != 0);
    for (int r = 0; r < nv; r++)
        for (int c = 0; c < nv; c++) out_rowmajor[r * nv + c] = o(r, c);
}
void orc_distort(void* h, const double* uv, int m, double* out) {
    Filter* F = (Filter*)h;
    Mat u(2, m);
    for (int c = 0; c < m; c++) {
        u(0, c) = uv[2 * c];
        u(1, c) = uv[2 * c + 1];
    }
    Mat d = distort_fm(F->cam, u);
    for (int c = 0; c < m; c++) {
        out[2 * c] = d(0, c);
        out[2 * c + 1] = d(1, c);
    }
}
void orc_undistort(void* h, const double* uv, int m, double* out) {
    Filter* F = (Filter*)h;
    Mat u(2, m);
    for (int c = 0; c < m; c++) {
        u(0, c) = uv[2 * c];
        u(1, c) = uv[2 * c + 1];
    }
    Mat d = undistort_fm(F->cam, u);
    for (int c = 0; c < m; c++) {
        out[2 * c] = d(0, c);
        out[2 * c + 1] = d(1, c);
    }
}
void orc_lu_inverse(const double* A_colmajor, int n, double* out_colmajor) {
    Mat A(n, n);
    std::memcpy(A.data(), A_colmajor, sizeof(double) * (size_t)n * n);
    Mat X = lu_inverse(A);
    std::memcpy(out_colmajor, X.data(), sizeof(double) * (size_t)n * n);
}
void orc_dgemm(int tA, int tB, int M, int N, int K, const double* A, int lda, const double* B, int ldb, double* C, int ldc) {
    dgemm(tA != 0, tB != 0, M, N, K, A, lda, B, ldb, C, ldc);
}

// --- map management -------------------------------------------------------------------------------------------------------
int orc_map_delete_pass(void* h, int reference_indexing, int* n_deleted) { return map_delete_pass(*(Filter*)h, reference_indexing != 0, n_deleted); }
int orc_map_delete_feature(void* h, int index) {
    Filter& F = *(Filter*)h;
    if (index < 0 || index >= (int)F.fi.size()) return -1;
    int rc = delete_a_feature(F, index + 1);
    if (rc) return rc;
    F.fi.erase(F.fi.begin() + index);
    return 0;
}
int orc_map_inversedepth_to_cartesian(void* h) { return inversedepth_2_cartesian_map(*(Filter*)h); }
int orc_map_add_feature(void* h, const double* uv, const uint8_t* image, int rows, int cols, int stride) {
    return map_add_feature(*(Filter*)h, uv, image, rows, cols, stride);
}
void orc_set_counters(void* h, const int* times_predicted, const int* times_measured) {
    Filter& F = *(Filter*)h;
    for (size_t i = 0; i < F.fi.size(); i++) {
        F.fi[i].times_predicted = times_predicted[i];
        F.fi[i].times_measured = times_measured[i];
    }
}
void orc_get_types(void* h, int* types) {
    Filter& F = *(Filter*)h;
    for (size_t i = 0; i < F.fi.size(); i++) types[i] = F.fi[i].type;
}
void orc_get_feature_init(void* h, int i, uint8_t* patch41, double* pose14) {
    Filter& F = *(Filter*)h;
    const Feature& ft = F.fi[i];
    for (int r = 0; r < 41; r++)
        for (int c = 0; c < 41; c++) patch41[r * 41 + c] = (uint8_t)ft.patch_when_initialized(r, c);
    for (int k = 0; k < 3; k++) pose14[k] = ft.r_wc_when_initialized[k];
    for (int r = 0; r < 3; r++)
        for (int c = 0; c < 3; c++) pose14[3 + 3 * r + c] = ft.R_wc_when_initialized(r, c);
    pose14[12] = ft.uv_when_initialized[0];
    pose14[13] = ft.uv_when_initialized[1];
}

// --- FAST + feature initialisation + full map management ---------------------------------------------------------------------
int orc_fast9(const uint8_t* img, int rows, int cols, int stride, int threshold, int nonmax, int max_kp, int* xy) {
    std::vector<int> xs, ys;
    fast9(img, rows, cols, stride, threshold, nonmax != 0, xs, ys);
    for (size_t i = 0; i < xs.size() && (int)i < max_kp; i++) {
        xy[2 * i] = xs[i];
        xy[2 * i + 1] = ys[i];
    }
    return (int)xs.size();
}
int orc_initialize_features(void* h, int step, int n, const uint8_t* image, int rows, int cols, int stride, const double* u01, int n_pairs, int* attempts) {
    return initialize_features(*(Filter*)h, step, n, image, rows, cols, stride, u01, n_pairs, attempts);
}
int orc_map_management(void* h, const uint8_t* image, int rows, int cols, int stride, int step, int min_features, int reference_indexing, const double* u01,
                       int n_pairs, int* info4) {
    return map_management(*(Filter*)h, image, rows, cols, stride, step, min_features, reference_indexing != 0, u01, n_pairs, info4);
}
// ExtendKF::initialize_x_and_p (src/ExtendKF.cpp:32-54): 13-state start, no features
void orc_initialize_x_and_p(void* h, double v0, double w0, double std_v0, double std_w0) {
    Filter& F = *(Filter*)h;
    F.fi.clear();
    F.x_k_k.resize(13, 1);
    F.x_k_k[3] = 1;
    F.x_k_k[7] = F.x_k_k[8] = F.x_k_k[9] = v0;
    F.x_k_k[10] = F.x_k_k[11] = F.x_k_k[12] = w0;
    F.p_k_k.resize(13, 13);
    const double eps = F.eps;
    for (int i = 0; i < 7; i++)
        if (i != 5) F.p_k_k(i, i) = eps;  // Q7: index 5 is skipped by the reference (src/ExtendKF.cpp:42-47)
    for (int i = 7; i < 10; i++) F.p_k_k(i, i) = std_v0 * std_v0;
    for (int i = 10; i < 13; i++) F.p_k_k(i, i) = std_w0 * std_w0;
    F.x_k_km1 = F.x_k_k;
    F.p_k_km1 = F.p_k_k;
}
}
