// kernels_map.cuh -- Map state surgery on the device (SURVEY 8f row 3): the covariance never leaves HBM while the map changes.
//
//   Map::delete_a_feature                         (src/Map.cpp:69-104)    remove a 3/6-wide block of rows and columns
//   Map::inversedepth_2_cartesian                 (src/Map.cpp:105-196)   linearity test, then P <- J P J^T with J = blockdiag(I, J_3x6, I)
//   Map::add_a_feature_covariance_inverse_depth   (src/Map.cpp:339-400) + ExtendKF::hinv (src/ExtendKF.cpp:236-265)
//
// All three are the same shape of work:  P' = T P T^T (+ E),  x' = T x,  where T copies most rows and forms a few "special" rows as
// small linear combinations of a contiguous range of old rows (none for delete, 3 rows from 6 for the conversion, 6 rows from the 13
// camera rows for a new feature).  The reference multiplies dense n x n matrices for this (J_all * P * J_all^T, src/Map.cpp:171-188);
// here one out-of-place pass writes P' into a scratch covariance (thread per output entry, coalesced down the columns) and the
// handle swaps the two buffers: 16 n^2 bytes of HBM traffic, no flops to speak of.
#pragma once
#include "common.cuh"
#include "kernels_track.cuh"

namespace rslam {

struct MapXform {
    int mode;      // 0 delete, 1 inverse depth -> cartesian, 2 add inverse-depth feature
    int n_old, n_new;
    int cut_at;    // first old row that is dropped (delete / convert); n_old for add
    int cut_cnt;   // number of old rows dropped (3 or 6 / 6 / 0)
    int sp_at;     // first special row of the new state (n_new if none)
    int sp_cnt;    // special rows: 0 / 3 / 6
    int src_at;    // first old row the special rows combine
    int src_cnt;   // 6 / 13
};

// scratch layout (doubles) written by the prep kernels: coefficient matrix C[sp_cnt][src_cnt] row-major at 0, additive block
// E[6][6] at 96, special entries of x' at 132
constexpr int kMapC = 0, kMapE = 96, kMapX = 132, kMapScratch = 160;

__device__ __forceinline__ int map_old_row(const MapXform& xf, int r) {  // new copy-row -> old row
    if (r < xf.cut_at) return r;
    return r + xf.cut_cnt - xf.sp_cnt;  // delete: r + cut_cnt ; convert: r + 3 ; add: never reached for r >= n_old (special)
}

// linearity test of the inverse-depth feature y[6] (src/Map.cpp:113-148) at camera position xc[3]; var_rho = its P(rho, rho)
// __noinline__: the batched map management calls this too, and its threshold decision must come out the same there; inlined into
// different kernels, the same source can be contracted into different FMAs (one compiled body gives the same bits for the same inputs)
__device__ __noinline__ bool map_is_linear_dev(const double* xc, const double* y, double var_rho, double threshold) {
    const double std_rho = sqrt(var_rho);
    const double rho = y[5];
    const double std_d = std_rho / (rho * rho);
    const double theta = y[3], phi = y[4];
    const double mi[3] = {cos(phi) * sin(theta), -sin(phi), cos(phi) * cos(theta)};
    double a = 0, n1 = 0, n2 = 0;
    for (int k = 0; k < 3; k++) {
        const double xo = y[k] + mi[k] / rho;  // inversedepth2cartesian (src/ExtendKF.cpp:137-152)
        const double d1 = xo - y[k], d2 = xo - xc[k];
        a += d1 * d2;
        n1 += d1 * d1;
        n2 += d2 * d2;
    }
    const double d_c2p = sqrt(n2);
    const double cos_alpha = a / (sqrt(n1) * sqrt(n2));
    const double linearity_index = 4 * std_d * cos_alpha / d_c2p;
    return linearity_index < threshold;
}

// linearity index of every inverse-depth feature (src/Map.cpp:113-148); the first feature (feature order) below the threshold is
// the one the reference converts (it returns after one conversion).  result[0] = that feature index or INT_MAX.
__global__ void k_map_linearity(DevFilter* Fs, int b, double threshold, int* result) {
    const DevFilter& F = Fs[b];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F.N || F.ftype[i] != 0) return;
    const int ip = F.foff[i];
    if (map_is_linear_dev(F.x_kk, F.x_kk + ip, F.P[(ip + 5) + (size_t)(ip + 5) * F.ldp], threshold)) atomicMin(result, i);
}

// coefficients of the conversion of the inverse-depth feature y[6] (src/Map.cpp:150-169): J = [I3, dm/dtheta / rho, dm/dphi / rho,
// -m / rho^2] into C[3][6], E[6][6] = 0, the cartesian point into xs[3]
__device__ __forceinline__ void map_prep_convert_dev(const double* y, double* C, double* E, double* xs) {
    const double theta = y[3], phi = y[4], rho = y[5];
    const double mi[3] = {cos(phi) * sin(theta), -sin(phi), cos(phi) * cos(theta)};
    const double dmt[3] = {cos(phi) * cos(theta), 0.0, -cos(phi) * sin(theta)};
    const double dmp[3] = {-sin(phi) * sin(theta), -cos(phi), -sin(phi) * cos(theta)};
    for (int r = 0; r < 3; r++) {
        for (int c = 0; c < 3; c++) C[r * 6 + c] = (r == c) ? 1.0 : 0.0;
        C[r * 6 + 3] = (1 / rho) * dmt[r];
        C[r * 6 + 4] = (1 / rho) * dmp[r];
        C[r * 6 + 5] = -mi[r] / (rho * rho);
        xs[r] = y[r] + mi[r] / rho;
    }
    for (int e = 0; e < 36; e++) E[e] = 0.0;
}

// the conversion of the feature at state offset ip
__global__ void k_map_prep_convert(DevFilter* Fs, int b, int ip, double* scratch) {
    const DevFilter& F = Fs[b];
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    map_prep_convert_dev(F.x_kk + ip, scratch + kMapC, scratch + kMapE, scratch + kMapX);
}

// new inverse-depth feature from the distorted pixel uvd at the camera state Xv[13]: hinv (src/ExtendKF.cpp:236-265) into xs[6], the
// Jacobians dy/dxv (6 x 13, into C row-major) and dy/dhd (6 x 3) and E = dy/dhd * diag(std_z^2, std_z^2, std_rho^2) * dy/dhd^T
// (src/Map.cpp:339-386), and the pose and pixel at initialisation into pose14.
// Every product and sum is an explicit round-to-nearest operation in the reference's order (no FMA contraction): the per-filter
// kernel and the batched one inline this into different code, where nvcc would fuse different products, and both must give the
// same bits.
__device__ __forceinline__ void map_prep_add_dev(const double* Xv, const CamDev& cam, double ud, double vd, double initial_rho, double std_pxl,
                                                 double std_rho, double* C, double* E, double* xs, double* pose14) {
    auto mul = [](double a, double b) { return __dmul_rn(a, b); };
    auto add = [](double a, double b) { return __dadd_rn(a, b); };
    auto sub = [](double a, double b) { return __dsub_rn(a, b); };
    // q2r (src/ExtendKF.cpp:91-102)
    const double qr = Xv[3], qx = Xv[4], qy = Xv[5], qz = Xv[6];
    double R[9];
    R[0] = sub(sub(add(mul(qr, qr), mul(qx, qx)), mul(qy, qy)), mul(qz, qz));
    R[1] = mul(2, sub(mul(qx, qy), mul(qr, qz)));
    R[2] = mul(2, add(mul(qz, qx), mul(qr, qy)));
    R[3] = mul(2, add(mul(qx, qy), mul(qr, qz)));
    R[4] = sub(add(sub(mul(qr, qr), mul(qx, qx)), mul(qy, qy)), mul(qz, qz));
    R[5] = mul(2, sub(mul(qy, qz), mul(qr, qx)));
    R[6] = mul(2, sub(mul(qz, qx), mul(qr, qy)));
    R[7] = mul(2, add(mul(qy, qz), mul(qr, qx)));
    R[8] = add(sub(sub(mul(qr, qr), mul(qx, qx)), mul(qy, qy)), mul(qz, qz));
    // undistort_fm (src/ExtendKF.cpp:266-285)
    const double xd = mul(sub(ud, cam.Cx), cam.dx), yd = mul(sub(vd, cam.Cy), cam.dy);
    const double rd = sqrt(add(mul(xd, xd), mul(yd, yd)));
    const double D = add(add(1.0, mul(mul(cam.k1, rd), rd)), mul(mul(mul(mul(cam.k2, rd), rd), rd), rd));
    const double uu = add(mul(xd, D) / cam.dx, cam.Cx), vu = add(mul(yd, D) / cam.dy, cam.Cy);
    const double gc[3] = {-sub(cam.Cx, uu) / cam.fku, -sub(cam.Cy, vu) / cam.fkv, 1.0};
    double gw[3];
    for (int k = 0; k < 3; k++) gw[k] = add(add(mul(R[3 * k], gc[0]), mul(R[3 * k + 1], gc[1])), mul(R[3 * k + 2], gc[2]));
    const double Xw = gw[0], Yw = gw[1], Zw = gw[2];
    const double xz2 = add(mul(Xw, Xw), mul(Zw, Zw)), n2 = add(xz2, mul(Yw, Yw)), sxz = sqrt(xz2);
    xs[0] = Xv[0];
    xs[1] = Xv[1];
    xs[2] = Xv[2];
    xs[3] = atan2(Xw, Zw);
    xs[4] = atan2(-Yw, sxz);
    xs[5] = initial_rho;
    // dRq_times_a_by_dq(q, gc), 3 x 4 row-major (src/ExtendKF.cpp:286-311)
    const double* a = gc;
    double dgw_dq[12];
    dgw_dq[0] = mul(2, add(sub(mul(qr, a[0]), mul(qz, a[1])), mul(qy, a[2])));
    dgw_dq[4] = mul(2, sub(add(mul(qz, a[0]), mul(qr, a[1])), mul(qx, a[2])));
    dgw_dq[8] = mul(2, add(add(mul(-qy, a[0]), mul(qx, a[1])), mul(qr, a[2])));
    dgw_dq[1] = mul(2, add(add(mul(qx, a[0]), mul(qy, a[1])), mul(qz, a[2])));
    dgw_dq[5] = mul(2, sub(sub(mul(qy, a[0]), mul(qx, a[1])), mul(qr, a[2])));
    dgw_dq[9] = mul(2, sub(add(mul(qz, a[0]), mul(qr, a[1])), mul(qx, a[2])));
    dgw_dq[2] = mul(2, add(add(mul(-qy, a[0]), mul(qx, a[1])), mul(qr, a[2])));
    dgw_dq[6] = mul(2, add(add(mul(qx, a[0]), mul(qy, a[1])), mul(qz, a[2])));
    dgw_dq[10] = mul(2, sub(add(mul(-qr, a[0]), mul(qz, a[1])), mul(qy, a[2])));
    dgw_dq[3] = mul(2, add(sub(mul(-qz, a[0]), mul(qr, a[1])), mul(qx, a[2])));
    dgw_dq[7] = mul(2, add(sub(mul(qr, a[0]), mul(qz, a[1])), mul(qy, a[2])));
    dgw_dq[11] = mul(2, add(add(mul(qx, a[0]), mul(qy, a[1])), mul(qz, a[2])));
    const double dth[3] = {Zw / xz2, 0.0, -Xw / xz2};
    const double dph[3] = {mul(Xw, Yw) / mul(n2, sxz), -sxz / n2, mul(Zw, Yw) / mul(n2, sxz)};
    for (int e = 0; e < 78; e++) C[e] = 0.0;
    C[0 * 13 + 0] = C[1 * 13 + 1] = C[2 * 13 + 2] = 1.0;
    for (int c = 0; c < 4; c++) {
        C[3 * 13 + 3 + c] = add(add(mul(dth[0], dgw_dq[c]), mul(dth[1], dgw_dq[4 + c])), mul(dth[2], dgw_dq[8 + c]));
        C[4 * 13 + 3 + c] = add(add(mul(dph[0], dgw_dq[c]), mul(dph[1], dgw_dq[4 + c])), mul(dph[2], dgw_dq[8 + c]));
    }
    // dyprima_dhd = dyprima_dgw * R_wc * dgc_dhu * dhu_dhd (left to right, src/Map.cpp:371); jacob_undistort_fm
    // (src/ExtendKF.cpp:312-332) first
    const double ja = sub(ud, cam.Cx), jb = sub(vd, cam.Cy);
    const double adx = mul(ja, cam.dx), bdy = mul(jb, cam.dy);
    const double rd2 = add(mul(adx, adx), mul(bdy, bdy));
    const double g = add(cam.k1, mul(mul(2, cam.k2), rd2));
    const double cc = add(add(1.0, mul(cam.k1, rd2)), mul(mul(cam.k2, rd2), rd2));
    double J[4];
    J[0] = add(cc, mul(mul(ja, g), mul(mul(mul(2, ja), cam.dx), cam.dx)));
    J[1] = mul(mul(ja, g), mul(mul(mul(2, jb), cam.dy), cam.dy));
    J[2] = mul(mul(jb, g), mul(mul(mul(2, ja), cam.dx), cam.dx));
    J[3] = add(cc, mul(mul(jb, g), mul(mul(mul(2, jb), cam.dy), cam.dy)));
    double tR[2][3];  // rows theta, phi of dyprima_dgw * R_wc
    for (int c = 0; c < 3; c++) {
        tR[0][c] = add(add(mul(dth[0], R[c]), mul(dth[1], R[3 + c])), mul(dth[2], R[6 + c]));
        tR[1][c] = add(add(mul(dph[0], R[c]), mul(dph[1], R[3 + c])), mul(dph[2], R[6 + c]));
    }
    // * dgc_dhu.  The reference comma-initialises the 3 x 2 matrix with "1/fku, 0, 0, 0, 1/fkv, 0" (src/Map.cpp:375-379); Eigen
    // fills row by row, so what it multiplies by is [1/fku 0; 0 0; 1/fkv 0], not the [1/fku 0; 0 1/fkv; 0 0] of the MATLAB
    // original (quirk Q16, found by compiling and running the reference's own Map.cpp).  Reproduced: the new feature's
    // (theta, phi) covariance block is rank one.
    double tg[2][2];
    for (int r = 0; r < 2; r++) {
        tg[r][0] = add(mul(tR[r][0], 1 / cam.fku), mul(tR[r][2], 1 / cam.fkv));
        tg[r][1] = 0.0;
    }
    double dy_dhd[6][3];
    for (int r = 0; r < 6; r++)
        for (int c = 0; c < 3; c++) dy_dhd[r][c] = 0.0;
    for (int r = 0; r < 2; r++)
        for (int c = 0; c < 2; c++) dy_dhd[3 + r][c] = add(mul(tg[r][0], J[c]), mul(tg[r][1], J[2 + c]));
    dy_dhd[5][2] = 1.0;
    const double pad[3] = {mul(std_pxl, std_pxl), mul(std_pxl, std_pxl), mul(std_rho, std_rho)};
    for (int r = 0; r < 6; r++)
        for (int c = 0; c < 6; c++) {
            double s = 0;
            for (int k = 0; k < 3; k++) s = add(s, mul(mul(dy_dhd[r][k], pad[k]), dy_dhd[c][k]));
            E[r * 6 + c] = s;
        }
    double* ip = pose14;
    ip[0] = Xv[0];
    ip[1] = Xv[1];
    ip[2] = Xv[2];
    for (int e = 0; e < 9; e++) ip[3 + e] = R[e];
    ip[12] = ud;
    ip[13] = vd;
}

// the rest of the features_info record of a new feature i_new at state offset off (src/Map.cpp:286-311)
__device__ __forceinline__ void map_new_record_dev(const DevFilter& F, int i_new, int off) {
    F.ftype[i_new] = 0;
    F.foff[i_new] = off;
    F.times_predicted[i_new] = 0;
    F.times_measured[i_new] = 0;
    F.has_h[i_new] = F.ic[i_new] = F.li[i_new] = F.hi[i_new] = 0;
    F.last_id[i_new] = i_new;
}

// its 41 x 41 patch around the pixel, cut from the filter's image (cv::Range truncates the double bounds toward zero,
// src/Map.cpp:286), and its zeroed predicted patch; entries t0, t0 + nt, ... of each
__device__ __forceinline__ void map_new_patch_dev(const DevFilter& F, int i_new, double ud, double vd, int t0, int nt) {
    const int u0 = (int)(ud - 20), v0 = (int)(vd - 20);
    for (int e = t0; e < 1681; e += nt) {
        const int r = e / 41, c = e % 41;
        const int gy = v0 + r, gx = u0 + c;
        unsigned char v = 0;
        if (F.image && gx >= 0 && gx < F.img_cols && gy >= 0 && gy < F.img_rows) v = F.image[(size_t)gy * F.img_stride + gx];
        F.patch_init[(size_t)i_new * 1681 + e] = v;
    }
    for (int e = t0; e < kPatchPix; e += nt) F.patch[(size_t)i_new * kPatchPix + e] = 0.f;
}

// one new feature at the end of filter b's state: coefficients into scratch and the features_info record
__global__ void k_map_prep_add(DevFilter* Fs, int b, CamDev cam, double ud, double vd, double initial_rho, double std_pxl, double std_rho,
                               double* scratch) {
    const DevFilter& F = Fs[b];
    const int i_new = F.N;  // the descriptor still holds the old N
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        map_prep_add_dev(F.x_kk, cam, ud, vd, initial_rho, std_pxl, std_rho, scratch + kMapC, scratch + kMapE, scratch + kMapX, F.init_pose + (size_t)i_new * 14);
        map_new_record_dev(F, i_new, F.n);
    }
    map_new_patch_dev(F, i_new, ud, vd, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}

// The entry arithmetic of every P' = T P T^T (+ E) pass, shared by the single-edit passes and the batched pass, so that a batch of
// edits gives the same bits as the sequence of single passes: a special entry against a copied one is sum_k c[k] * v(k) from
// s = 0 in k order; a special x special entry is (C P) C^T, left to right like the reference's products.
template <class V>
__device__ __forceinline__ double map_comb(const double* c, int cnt, V v) {
    double s = 0;
    for (int k = 0; k < cnt; k++) s += c[k] * v(k);
    return s;
}
template <class V>
__device__ __forceinline__ double map_quad(const double* cr, const double* cc, int cnt, V p) {
    double v = 0;
    for (int k = 0; k < cnt; k++) {
        double t = 0;
        for (int l = 0; l < cnt; l++) t += cr[l] * p(l, k);
        v += t * cc[k];
    }
    return v;
}

// P' = T P T^T + E and x' = T x, out of place.  grid (ceil(n_new / 256), min(n_new, 65535)): thread per entry; a CTA row takes
// columns blockIdx.y, blockIdx.y + gridDim.y, ... (gridDim.y is capped at 65535, and a map may have more state rows than that).
__global__ void __launch_bounds__(256) k_map_xform(DevFilter* Fs, int b, MapXform xf, const double* scratch, double* Pdst, double* xdst) {
    const DevFilter& F = Fs[b];
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= xf.n_new) return;
    const size_t ld = F.ldp;
    const double* P = F.P;
    const double* C = scratch + kMapC;
    const bool rs = r >= xf.sp_at && r < xf.sp_at + xf.sp_cnt;
    for (int c = blockIdx.y; c < xf.n_new; c += gridDim.y) {
        const bool cs = c >= xf.sp_at && c < xf.sp_at + xf.sp_cnt;
        double v;
        if (!rs && !cs) {
            v = P[map_old_row(xf, r) + (size_t)map_old_row(xf, c) * ld];
        } else if (rs && !cs) {
            const double* col = P + (size_t)map_old_row(xf, c) * ld + xf.src_at;
            v = map_comb(C + (r - xf.sp_at) * xf.src_cnt, xf.src_cnt, [&](int k) { return col[k]; });
        } else if (!rs && cs) {
            const double* row = P + map_old_row(xf, r) + (size_t)xf.src_at * ld;
            v = map_comb(C + (c - xf.sp_at) * xf.src_cnt, xf.src_cnt, [&](int k) { return row[(size_t)k * ld]; });
        } else {
            // evaluated for the lower-triangle position and mirrored, so that P stays exactly symmetric (the library's invariant)
            const int rr = r > c ? r : c, c2 = r > c ? c : r;
            const double* S = P + xf.src_at + (size_t)xf.src_at * ld;
            v = map_quad(C + (rr - xf.sp_at) * xf.src_cnt, C + (c2 - xf.sp_at) * xf.src_cnt, xf.src_cnt, [&](int l, int k) { return S[l + (size_t)k * ld]; });
            v += scratch[kMapE + (rr - xf.sp_at) * 6 + (c2 - xf.sp_at)];
        }
        Pdst[r + (size_t)c * ld] = v;
        if (c == 0) xdst[r] = rs ? scratch[kMapX + (r - xf.sp_at)] : F.x_kk[map_old_row(xf, r)];
    }
}

// ---- feature initialisation (SURVEY 8f row 4): cv::FAST (TYPE_9_16, non-maximum suppression) + the "features in the box" test ----
// cv::FAST as the reference calls it (src/Map.cpp:324-338: cv::FAST(im, keypoints, 100, true)), from the published algorithm
// (OpenCV 3.2 modules/features2d/src/fast.cpp, fast_score.cpp): corner iff 9 contiguous pixels of the radius-3 Bresenham circle are
// all darker than v - t or all brighter than v + t; score = the largest t for which that holds; a corner survives iff its score is
// strictly greater than its 8 neighbours' (non-corners score 0); the 3-pixel border is never tested; output row by row, left to right.
// pass 1: score of every pixel of the window (x0, y0, w, h) of the filter's image; thread per pixel
// score of the pixel at img (stride bytes per row); the caller keeps the 3-pixel border at 0
__device__ __forceinline__ int fast9_score_dev(const unsigned char* img, int stride, int threshold) {
    const int v = img[0];
    const int RX[16] = {0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1};
    const int RY[16] = {3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3};
    int d[16];
#pragma unroll 1
    for (int k = 0; k < 16; k++) d[k] = v - (int)img[RY[k] * stride + RX[k]];
    // NOTE: written with plain compare-and-assign loops that are NOT unrolled on purpose.  The obvious fully unrolled
    // min()/max() form of this arc search is miscompiled by nvcc 12.9 for sm_100a (the fused three-input VIMNMX3 chain returns
    // wrong strengths, e.g. 36 instead of 117; reproduced in isolation by tools/ubench/fast_dbg.cu), so keep it this way.
    int best = -256;
#pragma unroll 1
    for (int s0 = 0; s0 < 16; s0++) {
        int a = 256, bb = 256;
#pragma unroll 1
        for (int j = 0; j < 9; j++) {
            const int t = d[(s0 + j) & 15];
            if (t < a) a = t;
            if (-t < bb) bb = -t;
        }
        const int m = a > bb ? a : bb;
        if (m > best) best = m;
    }
    return best > threshold ? best - 1 : 0;
}

// pass 1: score of every pixel of the window (x0, y0, w, h) of the filter's image; thread per pixel
__global__ void __launch_bounds__(256) k_fast9_score(DevFilter* Fs, int b, int x0, int y0, int w, int h, int threshold, int* score) {
    const DevFilter& F = Fs[b];
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= w * h) return;
    const int x = e % w, y = e / w;
    int out = 0;
    if (x >= 3 && x < w - 3 && y >= 3 && y < h - 3) out = fast9_score_dev(F.image + (size_t)(y0 + y) * F.img_stride + (x0 + x), F.img_stride, threshold);
    score[e] = out;
}

// a corner survives iff its score is strictly greater than its 8 neighbours' (a positive score lies inside the tested area, so all
// 8 neighbours exist)
__device__ __forceinline__ bool fast9_keep_dev(const int* score, int e, int w) {
    const int sc = score[e];
    return sc > 0 && sc > score[e - 1] && sc > score[e + 1] && sc > score[e - w - 1] && sc > score[e - w] && sc > score[e - w + 1] &&
           sc > score[e + w - 1] && sc > score[e + w] && sc > score[e + w + 1];
}

// pass 2: non-maximum suppression and ORDERED compaction (row-major) by one CTA: res[0] = number of keypoints, xy[2 i] = (x, y)
__global__ void __launch_bounds__(1024) k_fast9_nms(const int* score, int w, int h, int max_kp, int* res, int* xy) {
    __shared__ int s_warp[32];
    __shared__ int s_base;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int e0 = 0; e0 < w * h; e0 += 1024) {
        const int e = e0 + threadIdx.x;
        bool keep = false;
        int x = 0, y = 0;
        if (e < w * h) {
            x = e % w;
            y = e / w;
            keep = fast9_keep_dev(score, e, w);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[wid] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
        for (int k = 0; k < 32; k++) {
            const int c = s_warp[k];
            if (k < wid) before += c;
            total += c;
        }
        if (keep) {
            const int pos = s_base + before + __popc(bal & ((1u << lane) - 1));
            if (pos < max_kp) {
                xy[2 * pos] = x;
                xy[2 * pos + 1] = y;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) s_base += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) res[0] = s_base;
}

// predicted (distorted) pixel of feature i at state x, with the reference's two visibility gates (src/ExtendKF.cpp:56-135)
// __noinline__: the batched map management calls this too, and its threshold decision must come out the same there; inlined into
// different kernels, the same source can be contracted into different FMAs (one compiled body gives the same bits for the same inputs)
__device__ __noinline__ bool predict_pixel_dev(const CamDev& cam, const double* x, int off, int type, double& hx, double& hy) {
    double R[9];
    q2r_dev(x + 3, R);
    double d[3];
    if (type == 0) {
        const double th = x[off + 3], ph = x[off + 4], rho = x[off + 5];
        const double mi[3] = {cos(ph) * sin(th), -sin(ph), cos(ph) * cos(th)};
        for (int k = 0; k < 3; k++) d[k] = (x[off + k] - x[k]) * rho + mi[k];
    } else {
        for (int k = 0; k < 3; k++) d[k] = x[off + k] - x[k];
    }
    double hrl[3];
    if (type == 0) {
        for (int k = 0; k < 3; k++) hrl[k] = R[k] * d[0] + R[3 + k] * d[1] + R[6 + k] * d[2];  // R^T d (:75)
    } else {
        double Ri[9];
        inv3_dev(R, Ri);
        for (int k = 0; k < 3; k++) hrl[k] = Ri[3 * k] * d[0] + Ri[3 * k + 1] * d[1] + Ri[3 * k + 2] * d[2];  // R^-1 d (:83)
    }
    const double ax = atan2(hrl[0], hrl[2]) * 180 / M_PI, ay = atan2(hrl[1], hrl[2]) * 180 / M_PI;
    if (ax < -60 || ax > 60 || ay < -60 || ay > 60) return false;
    const double uu = cam.Cx + (hrl[0] / hrl[2]) * cam.f * (1.0 / cam.dx);
    const double vu = cam.Cy + (hrl[1] / hrl[2]) * cam.f * (1.0 / cam.dy);
    distort_dev(cam, uu, vu, hx, hy);
    return (hx > 0) && (hx < cam.nCols) && (hy > 0) && (hy < cam.nRows);
}

__device__ __forceinline__ bool map_in_box(double hx, double hy, double cx, double cy, double sx, double sy) {
    return hx > (cx - sx) && hx < (cx + sx) && hy > (cy - sy) && hy < (cy + sy);
}

// step 3 of Map::initialize_a_features (src/Map.cpp:248-261): how many features predicted at x_k_k fall inside the sampling box
__global__ void k_map_box_count(DevFilter* Fs, int b, CamDev cam, double cx, double cy, double sx, double sy, int* res) {
    const DevFilter& F = Fs[b];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F.N) return;
    double hx, hy;
    if (!predict_pixel_dev(cam, F.x_kk, F.foff[i], F.ftype[i], hx, hy)) return;
    if (map_in_box(hx, hy, cx, cy, sx, sy)) atomicAdd(res, 1);
}

// ---- Map::map_management for every filter of a batch (rslam_map_management_batch) ---------------------------------------------
// Three launches whatever the batch and the edits: k_mmb_plan (delete pass, step 2, conversion choice; CTA per filter),
// k_mmb_init (the reference's sequential initialisation attempts; CTA per filter) and k_mmb_xform (one out-of-place pass over P per
// filter, batched over blockIdx.z).  The new state vector is built in the spare x by the first two.  Every entry of the final P is
// a fixed-depth expression of the P before the call; k_mmb_xform evaluates it with the same arithmetic (map_comb / map_quad) and
// from the same intermediate doubles as the sequence of single k_map_xform passes would, so the result is the same bits.

// per-filter slots of the plan, read back by the host at the end of the call
enum MbSlot {
    MB_STATUS = 0,    // RSLAM_OK / RSLAM_ERR_REFERENCE_UB / RSLAM_ERR_CAPACITY / RSLAM_ERR_INVALID
    MB_DELETED = 1,   // features deleted (before the failure, for a REFERENCE_UB filter)
    MB_CONVERTED = 2, // index of the converted feature or -1
    MB_INIT = 3,      // features initialised
    MB_ATTEMPTS = 4,  // initialisation attempts
    MB_N = 5,         // features after the call
    MB_NS = 6,        // state dimension after the call
    MB_EDIT = 7,      // 1: P and x change (the host swaps in the spare buffers)
    MB_N_CV = 8,      // features after the delete pass
    MB_NS_CV = 9,     // state dimension after the delete pass and the conversion
    MB_CONV_AT = 10,  // post-delete state offset of the converted feature or -1
    MB_TARGET = 11,   // features to initialise
    MB_CSRC = 16,     // [6] rows of the old state that the converted feature's rows combine
    MB_INTS = 32
};
// per-filter coefficient block: conversion C[3][6] at 0, E[6][6] at 18, x[3] at 54; addition a at kMbAdd + a * kMbAddStride:
// C[6][13] at 0, E[6][6] at 78 (its x goes straight into the spare state vector)
constexpr int kMbAdd = 64, kMbAddStride = 114, kMbMaxAttempts = 50;
constexpr int kMbSx = 30, kMbSy = 20, kMbBand = 21;  // sampling box half-sizes and excluded band (src/Map.cpp:200, 215-216)
constexpr int kMbWin = (2 * kMbSx + 1) * (2 * kMbSy + 1);
constexpr int kMbCols = 8;  // columns per CTA of k_mmb_xform

struct MapBatchWs {
    int* plan;     // [B][MB_INTS]
    int* rowmap;   // [B][nmax]: post-delete state row -> row of the state before the call
    int* recsrc;   // [B][Nmax]: record slot after the delete pass -> slot before it
    int* rectail;  // [B][Nmax]
    int* types;    // [B][Nmax]
    int* vis;      // [B][Nmax]: feature predicted inside the image at x_k_k
    double* pix;   // [B][2 Nmax]: its predicted pixel
    double* coef;  // [B][coef_stride]
    double* const* Pdst;  // [B] spare covariance of each filter
    double* const* xdst;  // [B] spare state vector of each filter
    const double* u01;    // [B][2 n_pairs]
    int n_pairs, Nmax, nmax, coef_stride;
};

// in-place forward compaction of a per-feature array (per T units a record): slot j <- slot cmap[j] for j in [first, N0), cmap[j] >= j.
// Staged through shared memory a chunk at a time, so no slot is overwritten before it has been read.  32-bit indices: an array holds
// max_features * 1681 units at most, below 2^31 for any map whose covariance fits in device memory.
template <class T>
__device__ void mb_compact(T* base, int per, int first, int N0, const int* cmap, unsigned char* stage_bytes, int stage_cap_bytes) {
    T* stage = (T*)stage_bytes;
    const int cap = stage_cap_bytes / (int)sizeof(T);
    const int e1 = N0 * per;
    for (int c0 = first * per; c0 < e1; c0 += cap) {
        const int m = e1 - c0 < cap ? e1 - c0 : cap;
#pragma unroll 8
        for (int t = threadIdx.x; t < m; t += blockDim.x) {
            const int e = c0 + t;
            const int j = e / per;
            stage[t] = base[cmap[j] * per + (e - j * per)];
        }
        __syncthreads();
        for (int t = threadIdx.x; t < m; t += blockDim.x) base[c0 + t] = stage[t];
        __syncthreads();
    }
}

// the `k`-th row (0-based) of the old state that is not yet removed; gone = one bit per old row
__device__ __forceinline__ int mb_select_kept(const unsigned* gone, int words, int k) {
    for (int w = 0; w < words; w++) {
        const unsigned kept = ~gone[w];
        const int c = __popc(kept);
        if (k < c) {
            unsigned m = kept;
            for (int i = 0; i < k; i++) m &= m - 1;
            return w * 32 + __ffs(m) - 1;
        }
        k -= c;
    }
    return -1;
}

// Steps 1-3 of Map::map_management and the choice of the conversion, per filter (CTA per filter).  A filter on which the delete
// pass is undefined in the reference is left exactly as it was.  dynamic smem: 2 * ceil(n / 32) words.
__global__ void __launch_bounds__(256, 1) k_mmb_plan(DevFilter* Fs, MapBatchWs ws, int min_features, int reference_indexing) {
    const int b = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const DevFilter& F = Fs[b];
    int* pl = ws.plan + (size_t)b * MB_INTS;
    int* dm = ws.rowmap + (size_t)b * ws.nmax;
    int* src = ws.recsrc + (size_t)b * ws.Nmax;
    int* tail = ws.rectail + (size_t)b * ws.Nmax;
    int* ty = ws.types + (size_t)b * ws.Nmax;
    double* cf = ws.coef + (size_t)b * ws.coef_stride;
    double* xn = ws.xdst[b];
    const double* x0 = F.x_kk;
    const double* P0 = F.P;
    const size_t ld = F.ldp;
    const int N0 = F.N, n0 = F.n, words = (n0 + 31) / 32;
    extern __shared__ unsigned s_gone[];  // removed rows of the old state; then the kept rows before each word
    unsigned* s_pre = s_gone + words;
    __shared__ int s_res[4];
    __shared__ int s_meas, s_conv;
    __shared__ __align__(16) unsigned char s_stage[16384];
    for (int w = tid; w < words; w += nt) s_gone[w] = 0;
    for (int i = tid; i < N0; i += nt) {
        src[i] = i;
        tail[i] = i;
        ty[i] = F.ftype[i];
    }
    if (tid == 0) {
        s_meas = 0;
        s_conv = 0x7fffffff;
    }
    __syncthreads();
    if (tid == 0) {
        // the delete loop of src/Map.cpp:19-32 exactly as rslam_map_delete_features runs it, on the counters only
        int pos = 0, cnt = N0, cur_n = n0, deleted = 0, status = RSLAM_OK;
        for (int i = 1; pos < cnt; i++) {
            const int tp = F.times_predicted[src[pos]], tm = F.times_measured[src[pos]];
            if (tm < tp * 0.5 && tp > 5) {
                const int erased_type = ty[pos];
                // features_info.erase: slot cnt - 1 keeps the last record of the list it had, which a later feature may inherit
                tail[cnt - 1] = src[cnt - 1];
                for (int k = pos; k < cnt - 1; k++) {
                    src[k] = src[k + 1];
                    ty[k] = ty[k + 1];
                }
                cnt--;
                int size, off = 13;
                if (reference_indexing) {
                    if (i - 1 >= cnt) {
                        status = RSLAM_ERR_REFERENCE_UB;
                        break;
                    }
                    size = ty[i - 1] == 0 ? 6 : 3;
                    for (int k = 0; k < i - 1; k++) off += ty[k] == 0 ? 6 : 3;
                } else {
                    size = erased_type == 0 ? 6 : 3;
                    for (int k = 0; k < pos; k++) off += ty[k] == 0 ? 6 : 3;
                }
                if (off + size > cur_n) {
                    status = RSLAM_ERR_REFERENCE_UB;
                    break;
                }
                for (int k = 0; k < size; k++) {  // rows off .. off + size - 1 of the current state
                    const int o = mb_select_kept(s_gone, words, off);
                    s_gone[o >> 5] |= 1u << (o & 31);
                }
                cur_n -= size;
                deleted++;
            } else {
                pos++;
            }
        }
        if (status == RSLAM_OK) {
            int total = 13;
            for (int k = 0; k < cnt; k++) total += ty[k] == 0 ? 6 : 3;
            if (total != cur_n) status = RSLAM_ERR_REFERENCE_UB;  // the reference would assert
        }
        s_res[0] = status;
        s_res[1] = deleted;
        s_res[2] = cnt;
        s_res[3] = cur_n;
        unsigned acc = 0;
        for (int w = 0; w < words; w++) {
            s_pre[w] = acc;
            acc += __popc(~s_gone[w]);
        }
    }
    __syncthreads();
    const int status = s_res[0], deleted = s_res[1], N1 = s_res[2], nd = s_res[3];
    if (status != RSLAM_OK) {
        if (tid == 0) {
            for (int k = 0; k < MB_INTS; k++) pl[k] = 0;
            pl[MB_STATUS] = status;
            pl[MB_DELETED] = deleted;
            pl[MB_CONVERTED] = -1;
            pl[MB_N] = N0;
            pl[MB_NS] = n0;
        }
        return;
    }
    // post-delete row -> old row
    for (int o = tid; o < n0; o += nt) {
        const unsigned g = s_gone[o >> 5];
        if (!((g >> (o & 31)) & 1u)) dm[s_pre[o >> 5] + __popc(~g & ((1u << (o & 31)) - 1u))] = o;
    }
    // records: survivors in order, then what features_info.erase leaves behind in the freed slots
    for (int j = N1 + tid; j < N0; j += nt) src[j] = tail[j];
    __syncthreads();
    if (deleted) {
        int first = N0;
        for (int j = 0; j < N0; j++)
            if (src[j] != j) {
                first = j;
                break;
            }
        mb_compact(F.times_predicted, 1, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.times_measured, 1, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.patch, kPatchPix, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.patch_init, 1681, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.init_pose, 14, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.has_h, 1, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.ic, 1, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.li, 1, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.hi, 1, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.h, 2, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.z, 2, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.S, 4, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.Hc, 14, first, N0, src, s_stage, sizeof(s_stage));
        mb_compact(F.Hf, 12, first, N0, src, s_stage, sizeof(s_stage));
    }
    // the `measured` count of src/Map.cpp:57-66, then step 2 (src/Map.cpp:34-55)
    int meas = 0;
    for (int j = tid; j < N1; j += nt) meas += begin_frame_dev(F, j) ? 1 : 0;
    if (meas) atomicAdd(&s_meas, meas);
    if (tid == 0) {
        for (int j = 0, off = 13; j < N1; j++) {
            F.ftype[j] = ty[j];
            F.foff[j] = off;
            off += ty[j] == 0 ? 6 : 3;
        }
    }
    __syncthreads();
    // Map::inversedepth_2_cartesian: the first inverse-depth feature whose linearity index is below 0.1, on the post-delete state
    for (int j = tid; j < N1; j += nt) {
        if (ty[j] != 0) continue;
        const int ip = F.foff[j];
        double y[6];
        for (int l = 0; l < 6; l++) y[l] = x0[dm[ip + l]];
        const int r5 = dm[ip + 5];
        if (map_is_linear_dev(x0, y, P0[r5 + (size_t)r5 * ld], 0.1)) atomicMin(&s_conv, j);
    }
    __syncthreads();
    const int conv = s_conv == 0x7fffffff ? -1 : s_conv;
    const int conv_at = conv >= 0 ? F.foff[conv] : -1;
    const int n_cv = conv >= 0 ? nd - 3 : nd;
    if (tid == 0) {
        if (conv >= 0) {
            double y[6];
            for (int l = 0; l < 6; l++) {
                pl[MB_CSRC + l] = dm[conv_at + l];
                y[l] = x0[dm[conv_at + l]];
            }
            map_prep_convert_dev(y, cf, cf + 18, cf + 54);
            ty[conv] = 1;
        }
        for (int j = 0, off = 13, last = -1; j < N1; j++) {
            F.ftype[j] = ty[j];
            F.foff[j] = off;
            off += ty[j] == 0 ? 6 : 3;
            if (ty[j] == 0) last = j;
            F.last_id[j] = last;
        }
        const int measured = s_meas;
        pl[MB_STATUS] = RSLAM_OK;
        pl[MB_DELETED] = deleted;
        pl[MB_CONVERTED] = conv;
        pl[MB_INIT] = 0;
        pl[MB_ATTEMPTS] = 0;
        pl[MB_N] = N1;
        pl[MB_NS] = n_cv;
        pl[MB_EDIT] = (deleted > 0 || conv >= 0) ? 1 : 0;
        pl[MB_N_CV] = N1;
        pl[MB_NS_CV] = n_cv;
        pl[MB_CONV_AT] = conv_at;
        pl[MB_TARGET] = measured == 0 ? min_features : (measured < min_features ? min_features - measured : 0);
    }
    __syncthreads();
    // the state vector after the delete pass and the conversion
    for (int r = tid; r < n_cv; r += nt) {
        if (conv >= 0 && r >= conv_at && r < conv_at + 3)
            xn[r] = cf[54 + r - conv_at];
        else
            xn[r] = x0[dm[(conv >= 0 && r >= conv_at + 3) ? r + 3 : r]];
    }
}

// Map::initialize_features (src/Map.cpp:198-323), the reference's sequential attempt loop, one CTA per filter: each attempt's box
// test sees the features this call has already added.
__global__ void __launch_bounds__(128, 1) k_mmb_init(DevFilter* Fs, MapBatchWs ws, CamDev cam, double initial_rho, double std_pxl, double std_rho) {
    const int b = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const DevFilter& F = Fs[b];
    int* pl = ws.plan + (size_t)b * MB_INTS;
    if (pl[MB_STATUS] != RSLAM_OK) return;
    const int target = pl[MB_TARGET];
    if (target <= 0) return;
    int* vis = ws.vis + (size_t)b * ws.Nmax;
    double* pix = ws.pix + (size_t)b * 2 * ws.Nmax;
    double* cf = ws.coef + (size_t)b * ws.coef_stride;
    double* xn = ws.xdst[b];
    const double* u = ws.u01 + (size_t)2 * ws.n_pairs * b;
    __shared__ int s_score[kMbWin];
    __shared__ int s_first;
    int N = pl[MB_N_CV], n = pl[MB_NS_CV];
    for (int j = tid; j < N; j += nt) vis[j] = predict_pixel_dev(cam, xn, F.foff[j], F.ftype[j], pix[2 * j], pix[2 * j + 1]) ? 1 : 0;
    if (tid == 0) s_first = 0x7fffffff;
    __syncthreads();
    int attempts = 0, init = 0, status = RSLAM_OK;
    const int sx = kMbSx, sy = kMbSy, excluded_band = kMbBand;
    while (init < target && attempts < kMbMaxAttempts) {
        const double cx = round(u[2 * attempts] * (cam.nCols - 2 * excluded_band - 2 * sx)) + excluded_band + sx;
        const double cy = round(u[2 * attempts + 1] * (cam.nRows - 2 * excluded_band - 2 * sy)) + excluded_band + sy;
        attempts++;
        bool in_box = false;
        for (int j = tid; j < N; j += nt) in_box |= vis[j] && map_in_box(pix[2 * j], pix[2 * j + 1], cx, cy, (double)sx, (double)sy);
        const bool any_in_box = __syncthreads_or(in_box);
        const int x0 = (int)(cx - sx), y0 = (int)(cy - sy);
        const int w = (int)(cx + sx + 1) - x0, h = (int)(cy + sy + 1) - y0;
        if (!F.image || x0 < 0 || y0 < 0 || w < 1 || h < 1 || w * h > kMbWin || x0 + w > F.img_cols || y0 + h > F.img_rows) {
            status = RSLAM_ERR_INVALID;  // the window leaves the image (uniforms outside [0, 1) or an image smaller than the camera)
            break;
        }
        // cv::FAST(window, 100, nonmax) and the first keypoint in its row-major output order
        for (int e = tid; e < w * h; e += nt) {
            const int x = e % w, y = e / w;
            int out = 0;
            if (x >= 3 && x < w - 3 && y >= 3 && y < h - 3) out = fast9_score_dev(F.image + (size_t)(y0 + y) * F.img_stride + (x0 + x), F.img_stride, 100);
            s_score[e] = out;
        }
        __syncthreads();
        for (int e = tid; e < w * h; e += nt)
            if (fast9_keep_dev(s_score, e, w)) atomicMin(&s_first, e);
        __syncthreads();
        const int first = s_first;
        __syncthreads();
        if (tid == 0) s_first = 0x7fffffff;
        if (first != 0x7fffffff && !any_in_box) {
            if (N + 1 > ws.Nmax || n + 6 > ws.nmax) {
                status = RSLAM_ERR_CAPACITY;
                break;
            }
            // the port keeps MATLAB's "- 1" (src/Map.cpp:243-244): the corner lands one pixel up and left of where FAST found it
            const double ud = (first % w) + (-sx + cx - 1), vd = (first / w) + (-sy + cy - 1);
            if (tid == 0) {
                double* ca = cf + kMbAdd + (size_t)init * kMbAddStride;
                map_prep_add_dev(xn, cam, ud, vd, initial_rho, std_pxl, std_rho, ca, ca + 78, xn + n, F.init_pose + (size_t)N * 14);
                map_new_record_dev(F, N, n);
                vis[N] = predict_pixel_dev(cam, xn, n, 0, pix[2 * N], pix[2 * N + 1]) ? 1 : 0;
            }
            map_new_patch_dev(F, N, ud, vd, tid, nt);
            N++;
            n += 6;
            init++;
        }
        __syncthreads();
    }
    if (tid == 0) {
        pl[MB_STATUS] = status;
        pl[MB_INIT] = init;
        pl[MB_ATTEMPTS] = attempts;
        pl[MB_N] = N;
        pl[MB_NS] = n;
        if (init) pl[MB_EDIT] = 1;
    }
}

// one index of the final state: a copy of an old row, row k of the conversion, or row k of added feature a
struct MbIdx {
    int kind, k, a, old;
};
__device__ __forceinline__ MbIdx mb_classify(int i, const int* dm, int n_cv, int conv_at) {
    if (i >= n_cv) {
        const int a = (i - n_cv) / 6;
        return MbIdx{2, i - n_cv - 6 * a, a, 0};
    }
    if (conv_at >= 0 && i >= conv_at && i < conv_at + 3) return MbIdx{1, i - conv_at, 0, 0};
    return MbIdx{0, 0, 0, dm[(conv_at >= 0 && i >= conv_at + 3) ? i + 3 : i]};
}

// entry of P after the delete pass and the conversion (rows / columns that are not additions): what k_map_xform's conversion pass
// writes, on the post-delete P
__device__ __forceinline__ double mb_p_cv(const double* P0, size_t ld, const MbIdx& r, const MbIdx& c, const int* csrc, const double* cc) {
    if (r.kind == 0 && c.kind == 0) return P0[r.old + c.old * ld];
    if (r.kind == 1 && c.kind == 0) return map_comb(cc + r.k * 6, 6, [&](int l) { return P0[csrc[l] + c.old * ld]; });
    if (r.kind == 0 && c.kind == 1) return map_comb(cc + c.k * 6, 6, [&](int l) { return P0[r.old + csrc[l] * ld]; });
    const int kr = r.k > c.k ? r.k : c.k, kc = r.k > c.k ? c.k : r.k;
    return map_quad(cc + kr * 6, cc + kc * 6, 6, [&](int l, int k) { return P0[csrc[l] + csrc[k] * ld]; }) + cc[18 + kr * 6 + kc];
}

// entry (r, c) of the final P where r or c is a row of the conversion or of an addition
__device__ __forceinline__ double mb_entry_special(const double* P0, size_t ld, MbIdx ri, MbIdx ci, const int* csrc, const double* cf) {
    auto add_c = [&](int a) { return cf + kMbAdd + (size_t)a * kMbAddStride; };
    auto cam_of = [](int k) { return MbIdx{0, 0, 0, k}; };
    // P before addition pass a, camera row k x column c (c not an addition >= a) and row r x camera column k (r likewise)
    auto colcam = [&](int k, const MbIdx& c) {
        if (c.kind == 2) return map_comb(add_c(c.a) + c.k * 13, 13, [&](int l) { return P0[k + l * ld]; });
        return mb_p_cv(P0, ld, cam_of(k), c, csrc, cf);
    };
    auto rowcam = [&](const MbIdx& rr, int k) {
        if (rr.kind == 2) return map_comb(add_c(rr.a) + rr.k * 13, 13, [&](int l) { return P0[l + k * ld]; });
        return mb_p_cv(P0, ld, rr, cam_of(k), csrc, cf);
    };
    const int ar = ri.kind == 2 ? ri.a : -1, ac = ci.kind == 2 ? ci.a : -1;
    if (ar < 0 && ac < 0) return mb_p_cv(P0, ld, ri, ci, csrc, cf);
    if (ar == ac) {
        // evaluated for the lower-triangle position and mirrored, like k_map_xform
        const int kr = ri.k > ci.k ? ri.k : ci.k, kc = ri.k > ci.k ? ci.k : ri.k;
        const double* C = add_c(ar);
        double v = map_quad(C + kr * 13, C + kc * 13, 13, [&](int l, int k) { return P0[l + k * ld]; });
        v += C[78 + kr * 6 + kc];
        return v;
    }
    if (ar > ac) return map_comb(add_c(ar) + ri.k * 13, 13, [&](int k) { return colcam(k, ci); });
    return map_comb(add_c(ac) + ci.k * 13, 13, [&](int k) { return rowcam(ri, k); });
}

// P' for every edited filter, out of place into its spare buffer.  grid (ceil(nb / 256), ceil(nb / kMbCols), B), nb >= every n'.
// An addition pass reads the 13 camera rows / columns of the P before it: camera x camera entries are never edited, and the
// camera entries of earlier additions and of the conversion are re-evaluated here exactly as their own pass stored them.  Copied
// entries (all but O(n) of them) are plain loads, kMbCols of them in flight per thread.
__global__ void __launch_bounds__(256) k_mmb_xform(DevFilter* Fs, MapBatchWs ws) {
    const int b = blockIdx.z;
    const int* pl = ws.plan + (size_t)b * MB_INTS;
    if (pl[MB_STATUS] == RSLAM_ERR_REFERENCE_UB || !pl[MB_EDIT]) return;
    const int n_new = pl[MB_NS];
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    const int c0 = blockIdx.y * kMbCols;
    if (r >= n_new || c0 >= n_new) return;
    const DevFilter& F = Fs[b];
    const double* P0 = F.P;
    const size_t ld = F.ldp;
    double* Pd = ws.Pdst[b];
    const int* dm = ws.rowmap + (size_t)b * ws.nmax;
    const double* cf = ws.coef + (size_t)b * ws.coef_stride;
    const int n_cv = pl[MB_NS_CV], conv_at = pl[MB_CONV_AT];
    const MbIdx ri = mb_classify(r, dm, n_cv, conv_at);
    int oc[kMbCols];
    double v[kMbCols];
#pragma unroll
    for (int j = 0; j < kMbCols; j++) {
        const MbIdx cj = mb_classify(c0 + j < n_new ? c0 + j : n_new - 1, dm, n_cv, conv_at);
        oc[j] = (ri.kind == 0 && cj.kind == 0) ? cj.old : -1;
        v[j] = oc[j] >= 0 ? P0[ri.old + oc[j] * ld] : 0.0;
    }
#pragma unroll
    for (int j = 0; j < kMbCols; j++)
        if (c0 + j < n_new && oc[j] >= 0) Pd[r + (size_t)(c0 + j) * ld] = v[j];
#pragma unroll 1
    for (int c = c0; c < c0 + kMbCols && c < n_new; c++) {
        const MbIdx cj = mb_classify(c, dm, n_cv, conv_at);
        if (ri.kind != 0 || cj.kind != 0) Pd[r + (size_t)c * ld] = mb_entry_special(P0, ld, ri, cj, pl + MB_CSRC, cf);
    }
}

}  // namespace rslam
