// kernels_track.cuh -- prediction, measurement prediction + Jacobians + S_i, ZNCC active search, 1-point RANSAC.
// Every kernel takes the array of per-filter descriptors and uses blockIdx.y as the filter index.
#pragma once
#include "common.cuh"

namespace rslam {

// ---------------------------------------------------------------------------------------------------------------
// Map::map_management step 2 (src/Map.cpp:34-55): counters + per-frame flag reset.  One thread per feature.
// ---------------------------------------------------------------------------------------------------------------
// for feature i; returns whether it was measured (li or hi) in the last frame
__device__ __forceinline__ bool begin_frame_dev(const DevFilter& F, int i) {
    const bool measured = F.li[i] || F.hi[i];
    if (F.has_h[i]) F.times_predicted[i] += 1;
    if (measured) F.times_measured[i] += 1;
    F.ic[i] = 0;
    F.li[i] = 0;
    F.hi[i] = 0;
    F.has_h[i] = 0;
    return measured;
}

__global__ void k_begin_frame(DevFilter* Fs) {
    DevFilter& F = Fs[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F.N) return;
    begin_frame_dev(F, i);
}

// ---------------------------------------------------------------------------------------------------------------
// ExtendKF::ekf_prediction (src/ExtendKF.cpp:333-388), constant velocity, dt = 1.
//   x_k_km1 = [fv(x_v); y],  P_cc <- F P_cc F^T + Q,  P_cf <- F P_cf,  P_fc <- P_fc F^T,  P_ff untouched (in place).
// Every CTA recomputes the 13x13 F (cheap); CTA 0 also does the camera block.  Thread j >= 13 owns column/row j.
// ---------------------------------------------------------------------------------------------------------------
__device__ void v2q_dev(const double* v, double* q) {  // src/ExtendKF.cpp:428-443 (Q14: zero quaternion below eps)
    const double theta = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
    if (theta < 2.220446049250313e-16) {
        q[0] = q[1] = q[2] = q[3] = 0.0;
    } else {
        const double vn0 = v[0] / theta, vn1 = v[1] / theta, vn2 = v[2] / theta;
        const double vnn = sqrt(vn0 * vn0 + vn1 * vn1 + vn2 * vn2);
        const double s = sin(theta / 2.0);
        q[0] = cos(theta / 2.0);
        q[1] = s * (vn0 / vnn);
        q[2] = s * (vn1 / vnn);
        q[3] = s * (vn2 / vnn);
    }
}

// F = dfv/dxv, Q = G Pn G^T and the predicted camera state, CTA-collective: thread 0 does the short serial part (quaternion
// product, the 4 x 3 block dq3_by_dq1 * dqomegadt_by_domega) into shared memory, then every thread fills its entries of F and Q
// (the serial version cost a fifth of the kernel on the single-filter path: 169 x 6 products out of a locally indexed array).
__device__ void build_F_Q(const double* x, const ParDev& par, double* Fm /*13x13 row-major*/, double* Q /*13x13*/, double* xv_new /*13*/,
                          double* sG /*13x6 scratch*/) {
    const double dt = 1.0;
    __shared__ double s_qd[16], s_ab[12];
    if (threadIdx.x == 0) {
        double wdt[3] = {x[10] * dt, x[11] * dt, x[12] * dt}, qwt[4];
        v2q_dev(wdt, qwt);
        // qprod (src/ExtendKF.cpp:416-427)
        const double* q = x + 3;
        const double cr0 = q[2] * qwt[3] - q[3] * qwt[2], cr1 = q[3] * qwt[1] - q[1] * qwt[3], cr2 = q[1] * qwt[2] - q[2] * qwt[1];
        for (int i = 0; i < 3; i++) xv_new[i] = x[i] + x[7 + i] * dt;
        xv_new[3] = q[0] * qwt[0] - (q[1] * qwt[1] + q[2] * qwt[2] + q[3] * qwt[3]);
        xv_new[4] = (q[0] * qwt[1] + qwt[0] * q[1]) + cr0;
        xv_new[5] = (q[0] * qwt[2] + qwt[0] * q[2]) + cr1;
        xv_new[6] = (q[0] * qwt[3] + qwt[0] * q[3]) + cr2;
        for (int i = 7; i < 13; i++) xv_new[i] = x[i];
        // dfv_by_dxv (src/ExtendKF.cpp:444-481)
        const double qd[16] = {qwt[0], -qwt[1], -qwt[2], -qwt[3], qwt[1], qwt[0], qwt[3], -qwt[2],
                               qwt[2], -qwt[3], qwt[0], qwt[1], qwt[3], qwt[2], -qwt[1], qwt[0]};
#pragma unroll
        for (int i = 0; i < 16; i++) s_qd[i] = qd[i];
        // dq3_by_dq1(qOld) * dqomegadt_by_domega(omegaOld, dt)   (src/ExtendKF.cpp:482-529)
        const double a[16] = {q[0], -q[1], -q[2], -q[3], q[1], q[0], -q[3], q[2], q[2], q[3], q[0], -q[1], q[3], -q[2], q[1], q[0]};
        const double* w = x + 10;
        const double om = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
        double b[12];
        const double sh = sin(om * dt / 2.0), ch = cos(om * dt / 2.0);
#pragma unroll
        for (int j = 0; j < 3; j++) b[j] = (-dt / 2.0) * (w[j] / om) * sh;
#pragma unroll
        for (int i = 0; i < 3; i++)
#pragma unroll
            for (int j = 0; j < 3; j++) {
                if (i == j)
                    b[(i + 1) * 3 + j] = (dt / 2.0) * w[i] * w[i] / (om * om) * ch + (1.0 / om) * (1.0 - w[i] * w[i] / (om * om)) * sh;
                else
                    b[(i + 1) * 3 + j] = (w[i] * w[j] / (om * om)) * ((dt / 2.0) * ch - (1.0 / om) * sh);
            }
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 3; j++) {
                double sacc = 0;
#pragma unroll
                for (int k = 0; k < 4; k++) sacc += a[4 * i + k] * b[3 * k + j];
                s_ab[3 * i + j] = sacc;
            }
    }
    __syncthreads();
    // G(7:10,0:3)=I, G(10:13,3:6)=I, G(0:3,0:3)=I*dt, G(3:7,3:6)=ab  (src/ExtendKF.cpp:347-376)
    for (int e = threadIdx.x; e < 78; e += blockDim.x) {
        const int i = e / 6, k = e % 6;
        double g = 0.0;
        if (i < 3) g = (k == i) ? dt : 0.0;
        else if (i < 7) g = (k >= 3) ? s_ab[3 * (i - 3) + (k - 3)] : 0.0;
        else if (i < 10) g = (k == i - 7) ? 1.0 : 0.0;
        else g = (k == 3 + (i - 10)) ? 1.0 : 0.0;
        sG[e] = g;
    }
    for (int e = threadIdx.x; e < 169; e += blockDim.x) {
        const int i = e / 13, j = e % 13;
        double f = (i == j) ? 1.0 : 0.0;
        if (i >= 3 && i < 7 && j >= 3 && j < 7) f = s_qd[4 * (i - 3) + (j - 3)];
        if (i < 3 && j == 7 + i) f = dt;
        if (i >= 3 && i < 7 && j >= 10) f = s_ab[3 * (i - 3) + (j - 10)];
        Fm[e] = f;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 169; e += blockDim.x) {
        const int i = e / 13, j = e % 13;
        double sacc = 0;
#pragma unroll
        for (int k = 0; k < 6; k++) sacc += (sG[i * 6 + k] * (k < 3 ? par.la : par.aa)) * sG[j * 6 + k];
        Q[e] = sacc;
    }
}

__global__ void __launch_bounds__(128) k_ekf_prediction(DevFilter* Fs, ParDev par, int with_begin) {
    DevFilter& F = Fs[blockIdx.y];
    __shared__ double sF[169], sQ[169], sX[13], sP[169], sT[169];
    const int n = F.n;
    if (blockIdx.x * blockDim.x >= (unsigned)n && blockIdx.x != 0) return;
    // everything this thread reads from P is fetched before F and Q are built (none of it depends on them): the loads fly while
    // thread 0 runs the serial quaternion part
    const int ld = F.ldp;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    double v[13];
#pragma unroll
    for (int c = 0; c < 13; c++) v[c] = (j >= 13 && j < n) ? F.P[j + (size_t)c * ld] : 0.0;  // row j (== column j by symmetry), coalesced
    double pcam[2] = {0.0, 0.0};
    if (blockIdx.x == 0) {
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int e = threadIdx.x + u * 128;
            if (e < 169) pcam[u] = F.P[(e / 13) + (size_t)(e % 13) * ld];
        }
    }
    build_F_Q(F.x_kk, par, sF, sQ, sX, sT);  // sT doubles as the 13 x 6 scratch for G (free until the camera block below)
    __syncthreads();
    if (blockIdx.x == 0) {
        // camera block: F Pcc F^T + Q  (left to right)
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int e = threadIdx.x + u * 128;
            if (e < 169) sP[e] = pcam[u];
        }
        __syncthreads();
        for (int e = threadIdx.x; e < 169; e += blockDim.x) {
            const int i = e / 13, j = e % 13;
            double s = 0;
            for (int k = 0; k < 13; k++) s += sF[i * 13 + k] * sP[k * 13 + j];
            sT[e] = s;
        }
        __syncthreads();
        for (int e = threadIdx.x; e < 169; e += blockDim.x) {
            const int i = e / 13, j = e % 13;
            double s = 0;
            for (int k = 0; k < 13; k++) s += sT[i * 13 + k] * sF[j * 13 + k];
            if (i >= j) {  // lower triangle is authoritative; mirror so that P stays exactly symmetric
                F.P[i + (size_t)j * ld] = s + sQ[e];
                F.P[j + (size_t)i * ld] = s + sQ[e];
            }
        }
        if (threadIdx.x < 13) F.x_km1[threadIdx.x] = sX[threadIdx.x];
    }
    if (with_begin && j < F.N) {  // Map::map_management step 2 (src/Map.cpp:34-55): counters + per-frame flag reset
        if (F.has_h[j]) F.times_predicted[j] += 1;
        if (F.li[j] || F.hi[j]) F.times_measured[j] += 1;
        F.ic[j] = 0;
        F.li[j] = 0;
        F.hi[j] = 0;
        F.has_h[j] = 0;
    }
    if (j >= 13 && j < n) {
        F.x_km1[j] = F.x_kk[j];
        double o[13];
#pragma unroll
        for (int i = 0; i < 13; i++) {
            double s = 0;
#pragma unroll
            for (int k = 0; k < 13; k++) s += sF[i * 13 + k] * v[k];
            o[i] = s;
        }
#pragma unroll
        for (int c = 0; c < 13; c++) {
            F.P[j + (size_t)c * ld] = o[c];
            F.P[c + (size_t)j * ld] = o[c];
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// (a) measurement prediction h_i, sparse Jacobian H_i and S_i = H_i P H_i^T + R_i.  One thread per feature.
//   mode 0 : Tracking::search_IC_matches first half (src/Tracking.cpp:35-44) at x_k_km1
//   mode 1 : Tracking::rescue_hi_inliers (src/Tracking.cpp:574-597) at x_k_k: refresh h/H where visible, then chi2 gate
// References: ExtendKF::predict_camera_measurements / hi_cartesian / hu / distort_fm (src/ExtendKF.cpp:56-204),
// Tracking::calculate_Hi_inverse_depth / calculate_Hi_cartesian (src/Tracking.cpp:71-163).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mul_2x2_2x3(const double* a1, const double* a2, double* o) {
#pragma unroll
    for (int i = 0; i < 2; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) o[i * 3 + j] = a1[i * 2] * a2[j] + a1[i * 2 + 1] * a2[3 + j];
}

__device__ __forceinline__ void gather_inliers(DevFilter& F, int which, int* s_scan, int* s_base);  // kernels_update.cuh
__device__ __forceinline__ void predict_feature(DevFilter& F, const CamDev& cam, const ParDev& par, int mode, int i, const double* sPcc);

// fuse_gather (mode 1, single-CTA grids only): the ordered high-innovation inlier list + innovation (gather_inliers, the first step
// of ekf_update_hi_inliers) is built by the same CTA right behind the gate, saving a dependent launch on the single-filter path.
__device__ __forceinline__ void upd_jnorm_cta(DevFilter& F, const ParDev& par);  // kernels_update.cuh
// fuse_jnorm (mode 1, single-CTA grids only): the quaternion normalisation that closes the preceding low-innovation update
// (src/ExtendKF.cpp:611-634) runs at the head of this launch instead of as its own.
__global__ void __launch_bounds__(128) k_predict(DevFilter* Fs, CamDev cam, ParDev par, int mode, int fuse_gather, int fuse_jnorm) {
    DevFilter& F = Fs[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    __shared__ double sPcc[49];
    __shared__ int s_scan[32], s_base;
    if (fuse_jnorm) {
        upd_jnorm_cta(F, par);
        __syncthreads();  // P rows / columns 3..6 and the normalised quaternion are visible to this CTA
    }
    const int ld = F.ldp;
    if (threadIdx.x < 49) sPcc[threadIdx.x] = F.P[(threadIdx.x / 7) + (size_t)(threadIdx.x % 7) * ld];
    __syncthreads();
    if (i < F.N) predict_feature(F, cam, par, mode, i, sPcc);
    if (fuse_gather) {
        __syncthreads();  // the hi flags of this CTA's features are written
        gather_inliers(F, 1, s_scan, &s_base);
    }
}

__device__ __forceinline__ void predict_feature(DevFilter& F, const CamDev& cam, const ParDev& par, int mode, int i, const double* sPcc) {
    const int ld = F.ldp;
    const double* x = mode == 0 ? F.x_km1 : F.x_kk;
    const int off = F.foff[i];
    const int type = F.ftype[i];
    const int fs = type == 0 ? 6 : 3;
    double t[3] = {x[0], x[1], x[2]};
    double q[4] = {x[3], x[4], x[5], x[6]};
    double R[9];
    q2r_dev(q, R);
    double Rrw[9];
    inv3_dev(R, Rrw);
    double y[6];
#pragma unroll
    for (int k = 0; k < 6; k++) y[k] = (k < fs) ? x[off + k] : 0.0;
    double d[3], rho = 1.0, mi[3] = {0, 0, 0}, sth = 0, cth = 0, sph = 0, cph = 0;
    if (type == 0) {
        sincos(y[3], &sth, &cth);
        sincos(y[4], &sph, &cph);
        rho = y[5];
        mi[0] = cph * sth;
        mi[1] = -sph;
        mi[2] = cph * cth;
#pragma unroll
        for (int k = 0; k < 3; k++) d[k] = (y[k] - t[k]) * rho + mi[k];
    } else {
#pragma unroll
        for (int k = 0; k < 3; k++) d[k] = y[k] - t[k];
    }
    // predict_camera_measurements: hrl = R^T d (inverse depth, :75) / R^-1 d (cartesian, :83)
    double hrl[3];
    if (type == 0) {
#pragma unroll
        for (int k = 0; k < 3; k++) hrl[k] = R[k] * d[0] + R[3 + k] * d[1] + R[6 + k] * d[2];
    } else {
#pragma unroll
        for (int k = 0; k < 3; k++) hrl[k] = Rrw[3 * k] * d[0] + Rrw[3 * k + 1] * d[1] + Rrw[3 * k + 2] * d[2];
    }
    bool vis = true;
    {
        // the reference's gate is |atan2(x, z)| <= 60 deg and |atan2(y, z)| <= 60 deg (src/ExtendKF.cpp:106-109); for z > 0 that is
        // |x| <= tan(60 deg) z, and z <= 0 is never inside it (the degenerate x = z = 0 passes atan2 but yields NaN pixels, which
        // the image gate below rejects either way).  Two multiplications instead of two atan2 (~285 instructions on a kernel that is
        // one dependent instruction chain per thread).
        const double t60 = 1.7320508075688772;
        if (!(hrl[2] > 0 && fabs(hrl[0]) <= t60 * hrl[2] && fabs(hrl[1]) <= t60 * hrl[2])) vis = false;
    }
    double hd[2] = {0, 0};
    if (vis) {
        const double uu = cam.Cx + (hrl[0] / hrl[2]) * cam.f * (1.0 / cam.dx);
        const double vu = cam.Cy + (hrl[1] / hrl[2]) * cam.f * (1.0 / cam.dy);
        distort_fixpoint_dev(cam, uu, vu, hd[0], hd[1]);
        vis = (hd[0] > 0) && (hd[0] < cam.nCols) && (hd[1] > 0) && (hd[1] < cam.nRows);
    }
    // calculate_derivatives (src/Tracking.cpp:540-573) rebuilds H_i at THIS state for every feature whose h is non-empty -- also for a
    // feature that fails the gates now but still carries the h of an earlier prediction (predict_camera_measurements leaves it in
    // place, src/ExtendKF.cpp:77-78): its Jacobian is taken at the new state with zi = the stale h.
    const bool have = vis || F.has_h[i];
    if (!vis && have) {
        hd[0] = F.h[2 * i];
        hd[1] = F.h[2 * i + 1];
    }
    double Hc[14], Hf[12];
    if (have) {
        // Jacobian at zi = h
        double Ju[4];
        jacob_undistort_dev(cam, hd[0], hd[1], Ju);
        const double idet = 1.0 / (Ju[0] * Ju[3] - Ju[2] * Ju[1]);
        const double a1[4] = {Ju[3] * idet, -Ju[1] * idet, -Ju[2] * idet, Ju[0] * idet};
        double hc[3];
#pragma unroll
        for (int k = 0; k < 3; k++) hc[k] = Rrw[3 * k] * d[0] + Rrw[3 * k + 1] * d[1] + Rrw[3 * k + 2] * d[2];
        const double fku = cam.f * (1.0 / cam.dx), fkv = cam.f * (1.0 / cam.dy);
        const double a2[6] = {fku / hc[2], 0, -hc[0] * fku / (hc[2] * hc[2]), 0, fkv / hc[2], -hc[1] * fkv / (hc[2] * hc[2])};
        double A[6];
        mul_2x2_2x3(a1, a2, A);
        // d h / d r = A * (-Rrw) [* rho]
#pragma unroll
        for (int a = 0; a < 2; a++)
#pragma unroll
            for (int c = 0; c < 3; c++) {
                double s = A[a * 3] * (-Rrw[c]) + A[a * 3 + 1] * (-Rrw[3 + c]) + A[a * 3 + 2] * (-Rrw[6 + c]);
                Hc[a * 7 + c] = (type == 0) ? s * rho : s;
            }
        // d h / d q = A * dRq_times_a_by_dq(qconj, d) * diag(1,-1,-1,-1)
        const double qb[4] = {q[0], -q[1], -q[2], -q[3]};
        double dR[12];
        dRq_times_a_by_dq_dev(qb, d, dR);
#pragma unroll
        for (int a = 0; a < 2; a++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const double sg = (c == 0) ? 1.0 : -1.0;
                Hc[a * 7 + 3 + c] = A[a * 3] * (dR[c] * sg) + A[a * 3 + 1] * (dR[4 + c] * sg) + A[a * 3 + 2] * (dR[8 + c] * sg);
            }
        // d h / d y
        double c0[18];  // 3 x 6 row-major
        if (type == 0) {
            const double c2[3] = {cph * cth, 0.0, -cph * sth};
            const double c3[3] = {-sph * sth, -cph, -sph * cth};
            const double dr[3] = {y[0] - t[0], y[1] - t[1], y[2] - t[2]};
#pragma unroll
            for (int r = 0; r < 3; r++) {
                c0[r * 6 + 0] = rho * Rrw[3 * r];
                c0[r * 6 + 1] = rho * Rrw[3 * r + 1];
                c0[r * 6 + 2] = rho * Rrw[3 * r + 2];
                c0[r * 6 + 3] = Rrw[3 * r] * c2[0] + Rrw[3 * r + 1] * c2[1] + Rrw[3 * r + 2] * c2[2];
                c0[r * 6 + 4] = Rrw[3 * r] * c3[0] + Rrw[3 * r + 1] * c3[1] + Rrw[3 * r + 2] * c3[2];
                c0[r * 6 + 5] = Rrw[3 * r] * dr[0] + Rrw[3 * r + 1] * dr[1] + Rrw[3 * r + 2] * dr[2];
            }
        } else {
#pragma unroll
            for (int r = 0; r < 3; r++) {
                c0[r * 6 + 0] = Rrw[3 * r];
                c0[r * 6 + 1] = Rrw[3 * r + 1];
                c0[r * 6 + 2] = Rrw[3 * r + 2];
                c0[r * 6 + 3] = c0[r * 6 + 4] = c0[r * 6 + 5] = 0.0;
            }
        }
#pragma unroll
        for (int a = 0; a < 2; a++)
#pragma unroll
            for (int c = 0; c < 6; c++) Hf[a * 6 + c] = A[a * 3] * c0[c] + A[a * 3 + 1] * c0[6 + c] + A[a * 3 + 2] * c0[12 + c];
        if (vis) {
            F.has_h[i] = 1;
            F.h[2 * i] = hd[0];
            F.h[2 * i + 1] = hd[1];
        }
#pragma unroll
        for (int e = 0; e < 14; e++) F.Hc[14 * i + e] = Hc[e];
#pragma unroll
        for (int e = 0; e < 12; e++) F.Hf[12 * i + e] = Hf[e];
    }
    bool need_S;
    if (mode == 0) {
        need_S = have;  // every feature with a non-empty h (src/Tracking.cpp:41)
    } else {
        need_S = F.ic[i] && !F.li[i];
        if (need_S && !have) {  // a match injected without any prediction (rslam_set_matches): whatever the arrays hold
#pragma unroll
            for (int e = 0; e < 14; e++) Hc[e] = F.Hc[14 * i + e];
#pragma unroll
            for (int e = 0; e < 12; e++) Hf[e] = F.Hf[12 * i + e];
            hd[0] = F.h[2 * i];
            hd[1] = F.h[2 * i + 1];
        }
    }
    if (!need_S) return;
    // S = H P H^T over the 7 + fs structurally non-zero columns; T = H * P first (left to right).
    // All 13 x 6 + 6 x 7 loads have compile-time trip counts (columns beyond fs are predicated to 0) so that they are issued as
    // one batch: on the single-filter path this kernel is pure memory latency.
    const double* P = F.P;
    double Pfc[6][7];  // P[off+k, j]   (feature rows, camera columns)
    double Pff[6][6];  // P[off+k, off+j]
#pragma unroll
    for (int k = 0; k < 6; k++) {
#pragma unroll
        for (int j = 0; j < 7; j++) Pfc[k][j] = (k < fs) ? P[(off + k) + (size_t)j * ld] : 0.0;
#pragma unroll
        for (int j = 0; j < 6; j++) Pff[k][j] = (k < fs && j < fs) ? P[(off + k) + (size_t)(off + j) * ld] : 0.0;
    }
    double T[2][13];
#pragma unroll
    for (int j = 0; j < 7; j++) {
        double s0 = 0, s1 = 0;
#pragma unroll
        for (int k = 0; k < 7; k++) {
            const double p = sPcc[k * 7 + j];
            s0 += Hc[k] * p;
            s1 += Hc[7 + k] * p;
        }
#pragma unroll
        for (int k = 0; k < 6; k++) {
            s0 += Hf[k] * Pfc[k][j];
            s1 += Hf[6 + k] * Pfc[k][j];
        }
        T[0][j] = s0;
        T[1][j] = s1;
    }
#pragma unroll
    for (int j = 0; j < 6; j++) {
        double s0 = 0, s1 = 0;
#pragma unroll
        for (int k = 0; k < 7; k++) {
            const double p = Pfc[j][k];  // P[k, off+j] == P[off+j, k] (exactly symmetric storage)
            s0 += Hc[k] * p;
            s1 += Hc[7 + k] * p;
        }
#pragma unroll
        for (int k = 0; k < 6; k++) {
            s0 += Hf[k] * Pff[k][j];
            s1 += Hf[6 + k] * Pff[k][j];
        }
        T[0][7 + j] = s0;
        T[1][7 + j] = s1;
    }
    double S[4];
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
        for (int b = 0; b < 2; b++) {
            double s = 0;
#pragma unroll
            for (int j = 0; j < 7; j++) s += T[a][j] * Hc[b * 7 + j];
#pragma unroll
            for (int j = 0; j < 6; j++) s += T[a][7 + j] * Hf[b * 6 + j];
            S[a * 2 + b] = s;
        }
    if (mode == 0) {
        S[0] += 1.0;  // R_i = I_2 (src/Map.cpp:310), not scaled by std_z (Q5)
        S[3] += 1.0;
#pragma unroll
        for (int e = 0; e < 4; e++) F.S[4 * i + e] = S[e];
    } else {
        if (!(par.quirks & RSLAM_Q6_RESCUE_WITHOUT_R)) {
            S[0] += 1.0;
            S[3] += 1.0;
        }
        const double nu0 = F.z[2 * i] - hd[0], nu1 = F.z[2 * i + 1] - hd[1];
        const double idet = 1.0 / (S[0] * S[3] - S[1] * S[2]);
        const double i00 = S[3] * idet, i01 = -S[1] * idet, i10 = -S[2] * idet, i11 = S[0] * idet;
        const double t0 = nu0 * i00 + nu1 * i10, t1 = nu0 * i01 + nu1 * i11;
        const double chi = t0 * nu0 + t1 * nu1;
        F.hi[i] = (chi < par.chi2) ? 1 : 0;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// (a4) predicted appearance: Tracking::pred_patch_fc (src/Tracking.cpp:164-278) -- SURVEY 8(f) next row 1.
// One CTA per feature, one thread per pixel of the 13 x 13 predicted patch.  The 41 x 41 initial patch is warped by the
// plane-induced homography K (R12 - t12 n^T / d) K^-1 between the initialisation camera and the predicted camera, through the
// undistort / distort model, and sampled exactly like cv::remap(INTER_LINEAR, BORDER_CONSTANT 0) on CV_32F data: map coordinates
// cast to float, quantised to 1/32 px with round-half-even, float weights, out-of-range taps = 0.  Geometry in fp64.
// Reference quirks kept: Q11 (MATLAB -1 in the patch offset), Q12 (translation R*r), Q13 (truncating cv::Range), Q3 (stale XYZ_w
// for cartesian features).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void undistort_dev(const CamDev& cam, double ud, double vd, double& uu, double& vu) {  // src/ExtendKF.cpp:266-285
    const double xd = (ud - cam.Cx) * cam.dx, yd = (vd - cam.Cy) * cam.dy;
    const double rd = sqrt(xd * xd + yd * yd);
    const double rd2 = rd * rd;
    const double D = 1 + cam.k1 * rd2 + cam.k2 * (rd2 * rd2);
    uu = xd * D / cam.dx + cam.Cx;
    vu = yd * D / cam.dy + cam.Cy;
}
__device__ __forceinline__ void inv4_dev(const double* m, double* o) {  // closed-form 4x4 inverse, row-major
    const double a00 = m[0], a01 = m[1], a02 = m[2], a03 = m[3], a10 = m[4], a11 = m[5], a12 = m[6], a13 = m[7];
    const double a20 = m[8], a21 = m[9], a22 = m[10], a23 = m[11], a30 = m[12], a31 = m[13], a32 = m[14], a33 = m[15];
    const double s0 = a00 * a11 - a10 * a01, s1 = a00 * a12 - a10 * a02, s2 = a00 * a13 - a10 * a03;
    const double s3 = a01 * a12 - a11 * a02, s4 = a01 * a13 - a11 * a03, s5 = a02 * a13 - a12 * a03;
    const double c5 = a22 * a33 - a32 * a23, c4 = a21 * a33 - a31 * a23, c3 = a21 * a32 - a31 * a22;
    const double c2 = a20 * a33 - a30 * a23, c1 = a20 * a32 - a30 * a22, c0 = a20 * a31 - a30 * a21;
    const double id = 1.0 / (s0 * c5 - s1 * c4 + s2 * c3 + s3 * c2 - s4 * c1 + s5 * c0);
    o[0] = (a11 * c5 - a12 * c4 + a13 * c3) * id;
    o[1] = (-a01 * c5 + a02 * c4 - a03 * c3) * id;
    o[2] = (a31 * s5 - a32 * s4 + a33 * s3) * id;
    o[3] = (-a21 * s5 + a22 * s4 - a23 * s3) * id;
    o[4] = (-a10 * c5 + a12 * c2 - a13 * c1) * id;
    o[5] = (a00 * c5 - a02 * c2 + a03 * c1) * id;
    o[6] = (-a30 * s5 + a32 * s2 - a33 * s1) * id;
    o[7] = (a20 * s5 - a22 * s2 + a23 * s1) * id;
    o[8] = (a10 * c4 - a11 * c2 + a13 * c0) * id;
    o[9] = (-a00 * c4 + a01 * c2 - a03 * c0) * id;
    o[10] = (a30 * s4 - a31 * s2 + a33 * s0) * id;
    o[11] = (-a20 * s4 + a21 * s2 - a23 * s0) * id;
    o[12] = (-a10 * c3 + a11 * c1 - a12 * c0) * id;
    o[13] = (a00 * c3 - a01 * c1 + a02 * c0) * id;
    o[14] = (-a30 * s3 + a31 * s1 - a32 * s0) * id;
    o[15] = (a20 * s3 - a21 * s1 + a22 * s0) * id;
}
__device__ __forceinline__ void homog4_dev(const double* R, const double* r, double* H) {  // [R 0;0 1] * [I r;0 1] = [R, R r; 0 1]
#pragma unroll
    for (int i = 0; i < 3; i++) {
        H[4 * i] = R[3 * i];
        H[4 * i + 1] = R[3 * i + 1];
        H[4 * i + 2] = R[3 * i + 2];
        H[4 * i + 3] = R[3 * i] * r[0] + R[3 * i + 1] * r[1] + R[3 * i + 2] * r[2];
    }
    H[12] = H[13] = H[14] = 0.0;
    H[15] = 1.0;
}
__device__ __forceinline__ void mat3_mul(const double* A, const double* B, double* C) {
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}

// distort_fm with the reference's arithmetic (IEEE divisions, same operation order as distort_dev) that stops at the fixed point of
// the Newton update: once a step returns rd unchanged every later step returns it unchanged too, so the result is bit-identical to
// the reference's ten steps (src/ExtendKF.cpp:191-196) -- typically after 4-6 of them.
__device__ __forceinline__ void distort_exact_dev(const CamDev& cam, double u, double v, double& ud, double& vd) {
    const double xu = (u - cam.Cx) * cam.dx;
    const double yu = (v - cam.Cy) * cam.dy;
    const double ru = sqrt(xu * xu + yu * yu);
    const double ru2 = ru * ru;
    double rd = ru / (1 + cam.k1 * ru2 + cam.k2 * (ru2 * ru2));
#pragma unroll 1
    for (int k = 0; k < 10; k++) {
        const double rd2 = rd * rd;
        const double rd3 = rd2 * rd;
        const double rd4 = rd2 * rd2;
        const double f = rd + cam.k1 * rd3 + cam.k2 * (rd4 * rd) - ru;
        const double fp = 1 + 3 * cam.k1 * rd2 + 5 * cam.k2 * rd4;
        const double rn = rd - f / fp;
        const bool same = !(rn != rd);
        rd = rn;
        if (same) break;
    }
    const double rd2 = rd * rd;
    const double D = 1 + cam.k1 * rd2 + cam.k2 * (rd2 * rd2);
    ud = xu / D / cam.dx + cam.Cx;
    vd = yu / D / cam.dy + cam.Cy;
}

// Per-feature geometry of the warp, ONE THREAD PER FEATURE (it is a serial chain of ~1.5 k fp64 operations; as thread 0 of a
// per-feature CTA it kept 191 threads waiting and was 35 % of the batched-filter frame): the homography Hm, the integer origin of the
// 13 x 13 window in the current image and the validity of that window -> F.pp_geom[12 i .. 12 i + 11] = Hm (9), xs, ys, ok.
constexpr int kPPGeom = 12;
__global__ void __launch_bounds__(64) k_pred_patch_setup(DevFilter* Fs, CamDev cam) {
    DevFilter& F = Fs[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F.N || !F.has_h[i] || F.patch_init == nullptr) return;
    double* out = F.pp_geom + (size_t)i * kPPGeom;
    const double h0 = F.h[2 * i], h1 = F.h[2 * i + 1];
    const bool inside = (h0 > kHalfPatch) && (h0 < (cam.nCols - kHalfPatch)) && (h1 > kHalfPatch) && (h1 < (cam.nRows - kHalfPatch));
    if (!inside) {  // src/Tracking.cpp:275: zero patch
        out[11] = -1.0;
        return;
    }
    const double* ip = F.init_pose + (size_t)i * 14;
    const double uvf0 = ip[12], uvf1 = ip[13];
    const double* x = F.x_km1;
    double Rwc[9], Hpf[16], Hk[16], Hpfi[16], Hkk[16];
    q2r_dev(x + 3, Rwc);
    homog4_dev(ip + 3, ip, Hpf);
    homog4_dev(Rwc, x, Hk);
    inv4_dev(Hpf, Hpfi);
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) {
            double sacc = 0;
#pragma unroll
            for (int k = 0; k < 4; k++) sacc += Hpfi[4 * a + k] * Hk[4 * k + b];
            Hkk[4 * a + b] = sacc;
        }
    const double fz = -cam.f / cam.dx;
    const double n1[3] = {uvf0 - cam.Cx, uvf1 - cam.Cy, fz};
    const double nn = sqrt(n1[0] * n1[0] + n1[1] * n1[1] + n1[2] * n1[2]);
    double n[3] = {n1[0] / nn, n1[1] / nn, n1[2] / nn};
    const double n2[4] = {h0 - cam.Cx, h1 - cam.Cy, fz, 1.0};
    double nt4[4];
#pragma unroll
    for (int a = 0; a < 4; a++) nt4[a] = Hkk[4 * a] * n2[0] + Hkk[4 * a + 1] * n2[1] + Hkk[4 * a + 2] * n2[2] + Hkk[4 * a + 3] * n2[3];
    const double nt[3] = {nt4[0] / nt4[3], nt4[1] / nt4[3], nt4[2] / nt4[3]};
    const double ntn = sqrt(nt[0] * nt[0] + nt[1] * nt[1] + nt[2] * nt[2]);
    const double ns[3] = {n[0] + nt[0] / ntn, n[1] + nt[1] / ntn, n[2] + nt[2] / ntn};
    const double nsn = sqrt(ns[0] * ns[0] + ns[1] * ns[1] + ns[2] * ns[2]);
#pragma unroll
    for (int a = 0; a < 3; a++) n[a] = ns[a] / nsn;
    // XYZ_w of the feature (Q3: cartesian features reuse the value of the previous inverse-depth feature)
    double X[3] = {0, 0, 0};
    const int li = F.last_id[i];
    if (li >= 0) {
        const double* y = x + F.foff[li];
        double st, ct, sph, cph;
        sincos(y[3], &st, &ct);
        sincos(y[4], &sph, &cph);
        const double m3[3] = {cph * st, -sph, cph * ct};
#pragma unroll
        for (int a = 0; a < 3; a++) X[a] = y[a] + (1.0 / y[5]) * m3[a];
    }
    double Xk[4];
#pragma unroll
    for (int a = 0; a < 4; a++) Xk[a] = Hpfi[4 * a] * X[0] + Hpfi[4 * a + 1] * X[1] + Hpfi[4 * a + 2] * X[2] + Hpfi[4 * a + 3];
    const double d = -(n[0] * (Xk[0] / Xk[3]) + n[1] * (Xk[1] / Xk[3]) + n[2] * (Xk[2] / Xk[3]));
    const double fk = cam.f / cam.dx;  // cam.K << f/d, 0, Cx ; 0, f/d, Cy ; 0 0 1 (src/System.cpp:58)
    const double K[9] = {fk, 0, cam.Cx, 0, fk, cam.Cy, 0, 0, 1};
    double Ki[9], M[9], T[9], Hm[9], Hmi[9];
    inv3_dev(K, Ki);
#pragma unroll
    for (int a = 0; a < 3; a++)
#pragma unroll
        for (int b = 0; b < 3; b++) M[3 * a + b] = Hkk[4 * a + b] - (Hkk[4 * a + 3] * n[b]) / d;
    mat3_mul(K, M, T);
    mat3_mul(T, Ki, Hm);
    inv3_dev(Hm, Hmi);
    double uu, vu;
    undistort_dev(cam, uvf0, uvf1, uu, vu);
    const double w0 = Hmi[0] * uu + Hmi[1] * vu + Hmi[2], w1 = Hmi[3] * uu + Hmi[4] * vu + Hmi[5], w2 = Hmi[6] * uu + Hmi[7] * vu + Hmi[8];
    double c2u, c2v;
    distort_exact_dev(cam, w0 / w2, w1 / w2, c2u, c2v);
    const int xs = (int)(c2u - kHalfPatch), xe = (int)(c2u + kHalfPatch), ys = (int)(c2v - kHalfPatch), ye = (int)(c2v + kHalfPatch);
#pragma unroll
    for (int a = 0; a < 9; a++) out[a] = Hm[a];
    out[9] = (double)xs;
    out[10] = (double)ys;
    out[11] = ((xe - xs + 1 == kPatch) && (ye - ys + 1 == kPatch)) ? 1.0 : 0.0;
}

// The 169 pixels of one predicted patch: one CTA per feature, one thread per pixel (the first 169 of 192).
__global__ void __launch_bounds__(192) k_pred_patch(DevFilter* Fs, CamDev cam) {
    DevFilter& F = Fs[blockIdx.y];
    const int i = blockIdx.x;
    if (i >= F.N || !F.has_h[i] || F.patch_init == nullptr) return;
    __shared__ unsigned int spw[(41 * 41 + 3) / 4 + 2];
    const int tid = threadIdx.x;
    float* out = F.patch + (size_t)i * kPatchPix;
    const double* geo = F.pp_geom + (size_t)i * kPPGeom;
    const double ok = geo[11];
    if (!(ok > 0.0)) {  // h within half a patch of the border (ok < 0), or a window that is not 13 x 13 (ok == 0): zero patch
        if (tid < kPatchPix) out[tid] = 0.f;
        return;
    }
    // 41 x 41 bytes; a feature's block starts 1681 i bytes into the array, i.e. at any byte alignment: the aligned words that cover it are
    // copied (three loads per thread instead of nine byte loads) and the patch is addressed at the same misalignment in shared memory
    // (the array is allocated with 4 spare bytes)
    const unsigned char* sp;
    {
        const unsigned char* src = F.patch_init + (size_t)i * 1681;
        const int mis = (int)((size_t)src & 3);
        const unsigned int* wsrc = reinterpret_cast<const unsigned int*>(src - mis);
        const int nwords = (mis + 41 * 41 + 3) >> 2;
        for (int e = tid; e < nwords; e += blockDim.x) spw[e] = wsrc[e];
        sp = reinterpret_cast<const unsigned char*>(spw) + mis;
    }
    const double* ip = F.init_pose + (size_t)i * 14;
    const double uvf0 = ip[12], uvf1 = ip[13];
    double Hm[9];
#pragma unroll
    for (int a = 0; a < 9; a++) Hm[a] = geo[a];
    const int xs = (int)geo[9], ys = (int)geo[10];
    __syncthreads();
    if (tid >= kPatchPix) return;
    const int r = tid / kPatch, c = tid % kPatch;
    double uu, vu;
    undistort_dev(cam, (double)(xs + c), (double)(ys + r), uu, vu);
    const double w0 = Hm[0] * uu + Hm[1] * vu + Hm[2], w1 = Hm[3] * uu + Hm[4] * vu + Hm[5], w2 = Hm[6] * uu + Hm[7] * vu + Hm[8];
    double c1u, c1v;
    distort_exact_dev(cam, w0 / w2, w1 / w2, c1u, c1v);
    const float mx = (float)(c1u - (uvf0 - 20 - 1)), my = (float)(c1v - (uvf1 - 20 - 1));
    const int sx = __float2int_rn(mx * 32.0f), sy = __float2int_rn(my * 32.0f);
    const int ix = sx >> 5, iy = sy >> 5;
    const float fx = (float)(sx & 31) / 32.0f, fy = (float)(sy & 31) / 32.0f;
    const float w00 = (1.f - fy) * (1.f - fx), w01 = (1.f - fy) * fx, w10 = fy * (1.f - fx), w11 = fy * fx;
    auto tap = [&](int yy, int xx) -> float { return (xx < 0 || yy < 0 || xx >= 41 || yy >= 41) ? 0.f : (float)sp[yy * 41 + xx]; };
    out[tid] = tap(iy, ix) * w00 + tap(iy, ix + 1) * w01 + tap(iy + 1, ix) * w10 + tap(iy + 1, ix + 1) * w11;
}

// ---------------------------------------------------------------------------------------------------------------
// (b) active search: Tracking::matching (src/Tracking.cpp:279-351) + Converter::corrcoef_opencv (src/Converter.cpp:188-209).
// One CTA per feature.  The search window and the predicted 13x13 patch are staged in shared memory; each thread scores
// candidates with one-pass sums (sum b, sum b^2 exact in integers; sum a*b in fp64); block arg-max keeps the FIRST maximum in
// the reference's (x outer, y inner) visiting order; a NaN score on the first visited candidate is sticky (Eigen maxCoeff).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kMaxHalfSearch = 20;                           // ceil(2*sqrt(S_ii)) with S_ii < 100
constexpr int kWinMax = 2 * kMaxHalfSearch + 1 + 2 * kHalfPatch;  // 53
constexpr int kSearchThreads = 64;
constexpr int kStrip = 4;  // vertically adjacent candidates scored by one thread

// Scoring is register-tiled: a thread owns a strip of kStrip vertically adjacent candidates (same x), walks the 13 patch columns
// and for each loads the 16 window pixels the strip touches once; every predicted-patch value is then used for kStrip candidates.
// The window is converted to fp64 once when it is staged (an int->double conversion per candidate pixel saturated the XU pipe);
// sum b and sum b^2 are exact integer-valued doubles built with a sliding column sum.  Per candidate pixel this is ~0.56 shared
// loads and ~1.7 DFMA instead of 2 loads + 1 conversion + 1 DFMA + 2 IMAD.
__global__ void __launch_bounds__(kSearchThreads) k_search(DevFilter* Fs, CamDev cam, ParDev par) {
    DevFilter& F = Fs[blockIdx.y];
    const int i = blockIdx.x;
    if (i >= F.N) return;
    if (!F.has_h[i] || F.image == nullptr) return;
    __shared__ double win[(kWinMax + kStrip - 1) * kWinMax];  // rows padded to whole strips
    __shared__ double pa[kPatchPix];  // predicted patch minus its mean
    __shared__ double s_part[kPatch];
    __shared__ double red_c[2], red_firstc[2];
    __shared__ int red_i[2], red_first[2];
    __shared__ double s_stats[2];
    const double h0 = F.h[2 * i], h1 = F.h[2 * i + 1];
    const double S00 = F.S[4 * i], S01 = F.S[4 * i + 1], S10 = F.S[4 * i + 2], S11 = F.S[4 * i + 3];
    // largest eigenvalue of the symmetric 2x2 (lower triangle, as SelfAdjointEigenSolver)
    const double lmax = 0.5 * (S00 + S11) + sqrt(0.25 * (S00 - S11) * (S00 - S11) + S10 * S10);
    if (!(lmax < par.max_eig)) return;
    // predicted patch is zero when h is within half a patch of the border (src/Tracking.cpp:174-175,275) -> NaN scores -> no match
    if (!((h0 > kHalfPatch) && (h0 < (cam.nCols - kHalfPatch)) && (h1 > kHalfPatch) && (h1 < (cam.nRows - kHalfPatch)))) return;
    const int hsx = (int)ceil(2 * sqrt(S00)), hsy = (int)ceil(2 * sqrt(S11));
    if (hsx > kMaxHalfSearch || hsy > kMaxHalfSearch) return;  // cannot happen while lmax < max_eig <= 100 (rslam_create checks it)
    const int cx = (int)round(h0), cy = (int)round(h1);
    const int x_lo = cx - hsx, y_lo = cy - hsy;
    const int ncx = 2 * hsx + 1, ncy = 2 * hsy + 1;
    const int nsy = (ncy + kStrip - 1) / kStrip;
    const int ww = ncx + 2 * kHalfPatch, wh = nsy * kStrip + 2 * kHalfPatch;  // rows padded to whole strips (zeros)
    const int wx0 = x_lo - kHalfPatch, wy0 = y_lo - kHalfPatch;
    {   // window load: a warp per row, lanes along x (coalesced bytes, no integer divisions), four rows x two 32-pixel chunks in flight
        const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5, nwrp = blockDim.x >> 5;
        const unsigned char* img = F.image;
        const int icols = F.img_cols, irows = F.img_rows, istride = F.img_stride;
        for (int wyb = wrp * 4; wyb < wh; wyb += 4 * nwrp) {
            unsigned char v[4][2];
#pragma unroll
            for (int u = 0; u < 4; u++)
#pragma unroll
                for (int hh = 0; hh < 2; hh++) {
                    const int wy = wyb + u, wx = lane + 32 * hh;
                    const int gx = wx0 + wx, gy = wy0 + wy;
                    v[u][hh] = 0;
                    if (wy < wh && wx < ww && gx >= 0 && gx < icols && gy >= 0 && gy < irows) v[u][hh] = img[(size_t)gy * istride + gx];
                }
#pragma unroll
            for (int u = 0; u < 4; u++)
#pragma unroll
                for (int hh = 0; hh < 2; hh++) {
                    const int wy = wyb + u, wx = lane + 32 * hh;
                    if (wy < wh && wx < ww) win[wy * ww + wx] = (double)v[u][hh];
                }
        }
    }
    for (int e = threadIdx.x; e < kPatchPix; e += blockDim.x) pa[e] = (double)F.patch[(size_t)i * kPatchPix + e];
    __syncthreads();
    // mean and centred energy of the predicted patch: per-row partial sums, then a fixed-order sum of the 13 partials
    if (threadIdx.x < kPatch) {
        double sa = 0;
        for (int c = 0; c < kPatch; c++) sa += pa[threadIdx.x * kPatch + c];
        s_part[threadIdx.x] = sa;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double sa = 0;
        for (int r = 0; r < kPatch; r++) sa += s_part[r];
        s_stats[0] = sa * (1.0 / kPatchPix);
    }
    __syncthreads();
    const double mean_a = s_stats[0];
    for (int e = threadIdx.x; e < kPatchPix; e += blockDim.x) pa[e] -= mean_a;
    __syncthreads();
    if (threadIdx.x < kPatch) {
        double va = 0;
        for (int c = 0; c < kPatch; c++) va += pa[threadIdx.x * kPatch + c] * pa[threadIdx.x * kPatch + c];
        s_part[threadIdx.x] = va;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double va = 0;
        for (int r = 0; r < kPatch; r++) va += s_part[r];
        s_stats[1] = va;  // sum (a - mean)^2, exactly 0 for a constant (e.g. zeroed) patch
    }
    __syncthreads();
    const double var_a = s_stats[1];
    const double idet = 1.0 / (S00 * S11 - S01 * S10);
    const double i00 = S11 * idet, i01 = -S01 * idet, i10 = -S10 * idet, i11 = S00 * idet;
    double best_c = -INFINITY;   // best finite score seen by this thread
    int best_idx = 0x7fffffff;   // its visiting-order index jx*ncy + iy
    int first_idx = 0x7fffffff;  // first accepted candidate seen by this thread
    double first_c = 0.0;
    for (int strip = threadIdx.x; strip < ncx * nsy; strip += blockDim.x) {
        const int jx = strip % ncx, iy0 = (strip / ncx) * kStrip;
        const int j = x_lo + jx;
        bool ok[kStrip];
        bool any = false;
#pragma unroll
        for (int t = 0; t < kStrip; t++) {
            const int iy = iy0 + t, ii = y_lo + iy;
            const double nu0 = j - h0, nu1 = ii - h1;
            const double t0 = nu0 * i00 + nu1 * i10, t1 = nu0 * i01 + nu1 * i11;
            ok[t] = iy < ncy && ((t0 * nu0 + t1 * nu1) < par.chi2) && (j > kHalfPatch) && (j < (cam.nCols - kHalfPatch)) && (ii > kHalfPatch) &&
                    (ii < (cam.nRows - kHalfPatch));
            any |= ok[t];
        }
        if (!any) continue;
        double sab[kStrip], sb[kStrip], sbb[kStrip];
#pragma unroll
        for (int t = 0; t < kStrip; t++) sab[t] = sb[t] = sbb[t] = 0.0;
        const double* wp = &win[iy0 * ww + jx];
#pragma unroll 1
        for (int c = 0; c < kPatch; c++) {
            double wv[kPatch + kStrip - 1];
#pragma unroll
            for (int r = 0; r < kPatch + kStrip - 1; r++) wv[r] = wp[r * ww + c];
            // column sums of b and b^2 for the first candidate, then slide down
            double cs = 0.0, cq = 0.0;
#pragma unroll
            for (int r = 0; r < kPatch; r++) {
                cs += wv[r];
                cq = fma(wv[r], wv[r], cq);
            }
            sb[0] += cs;
            sbb[0] += cq;
#pragma unroll
            for (int t = 1; t < kStrip; t++) {
                cs += wv[t + kPatch - 1] - wv[t - 1];
                cq += wv[t + kPatch - 1] * wv[t + kPatch - 1] - wv[t - 1] * wv[t - 1];
                sb[t] += cs;
                sbb[t] += cq;
            }
#pragma unroll
            for (int r = 0; r < kPatch; r++) {
                const double a = pa[r * kPatch + c];
#pragma unroll
                for (int t = 0; t < kStrip; t++) sab[t] = fma(a, wv[r + t], sab[t]);  // sum (a - mean_a) * b == sum (a - mean_a)(b - mean_b)
            }
        }
#pragma unroll
        for (int t = 0; t < kStrip; t++) {
            if (!ok[t]) continue;
            const int cand = jx * ncy + iy0 + t;  // reference visiting order: x outer, y inner
            const double var_b = ((double)kPatchPix * sbb[t] - sb[t] * sb[t]) / kPatchPix;  // exact: integer-valued operands < 2^53
            // a constant candidate window (saturated image regions) has centred b == 0 exactly in the reference's covariance
            // (cv::calcCovarMatrix centres both variables, src/Converter.cpp:195): 0 / 0 = NaN there, and NaN matters (it is sticky in
            // slot 0, Q10).  The uncentred sum here would give +-inf instead, so the exact integer test decides.
            const double corr = (var_b == 0.0 || var_a == 0.0) ? __longlong_as_double(0x7ff8000000000000LL) : sab[t] / sqrt(var_a * var_b);
            if (cand < first_idx) {
                first_idx = cand;
                first_c = corr;
            }
            if (corr == corr && (corr > best_c || (corr == best_c && cand < best_idx))) {  // NaN never wins; ties keep the earlier index
                best_c = corr;
                best_idx = cand;
            }
        }
    }
    // block reduce: maximum finite corr, ties -> smaller visiting index ; and the globally first accepted candidate
    const unsigned fm = 0xffffffffu;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double oc = __shfl_xor_sync(fm, best_c, o);
        const int oi = __shfl_xor_sync(fm, best_idx, o);
        if (oc > best_c || (oc == best_c && oi < best_idx)) {
            best_c = oc;
            best_idx = oi;
        }
        const int of = __shfl_xor_sync(fm, first_idx, o);
        const double ofc = __shfl_xor_sync(fm, first_c, o);
        if (of < first_idx) {
            first_idx = of;
            first_c = ofc;
        }
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        red_c[w] = best_c;
        red_i[w] = best_idx;
        red_first[w] = first_idx;
        red_firstc[w] = first_c;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < kSearchThreads / 32; k++) {
            if (red_c[k] > best_c || (red_c[k] == best_c && red_i[k] < best_idx)) {
                best_c = red_c[k];
                best_idx = red_i[k];
            }
            if (red_first[k] < first_idx) {
                first_idx = red_first[k];
                first_c = red_firstc[k];
            }
        }
        if (first_idx == 0x7fffffff) return;  // no candidate pixel (Q10: reference divides by zero here)
        if (first_c != first_c) return;        // NaN in slot 0 is sticky in Eigen's maxCoeff -> unmatched (Q10)
        if (best_c > par.corr_thr) {
            F.ic[i] = 1;
            const int jx = best_idx / ncy, iy = best_idx % ncy;
            F.z[2 * i] = (double)(x_lo + jx);
            F.z[2 * i + 1] = (double)(y_lo + iy);
        }
    }
}

// one (match, hypothesis) pair of compute_hypothesis_support_fast (src/Tracking.cpp:443-477): re-projection of the hypothesised feature,
// Newton distortion, squared residual against the squared threshold.  xi: the hypothesis' x_i rows of the tile (SJT matches, tile
// layout of sup_rows).  Dead lanes run the arithmetic on zeros (it converges at once) so that the warp-uniform early exit stays uniform.
constexpr int kSupTile = 64;  // matches per scoring tile
__device__ __forceinline__ bool support_pair_inlier(const DevFilter& F, const CamDev& cam, bool q1, bool live, const double* xi, int jl, int jj,
                                                    const double* xc, const double* Rm, double fku, double idx, double idy, double thr2) {
    double r3[3] = {0, 0, 0}, a0 = 0, a1 = 0, rho = 0;
    if (live) {
        if (q1) {
            r3[0] = xi[4 * jl];
            r3[1] = xi[4 * jl + 1];
            r3[2] = xi[4 * jl + 2];
            rho = xi[4 * jl + 3];
            a0 = xi[4 * kSupTile + 2 * jl];
            a1 = xi[4 * kSupTile + 2 * jl + 1];
        } else {
            r3[0] = xi[6 * jl];
            r3[1] = xi[6 * jl + 1];
            r3[2] = xi[6 * jl + 2];
            a0 = xi[6 * jl + 3];
            a1 = xi[6 * jl + 4];
            rho = xi[6 * jl + 5];
        }
    }
    double s0, c0, s1, c1;
    sincos_fast(a0, &s0, &c0);
    sincos_fast(a1, &s1, &c1);
    const double mi[3] = {c1 * s0, -s1, c1 * c0};
    double v3[3];
#pragma unroll
    for (int k = 0; k < 3; k++) v3[k] = (r3[k] - xc[k]) * rho + mi[k];
    double hc[3];
#pragma unroll
    for (int k = 0; k < 3; k++) hc[k] = Rm[k] * v3[0] + Rm[3 + k] * v3[1] + Rm[6 + k] * v3[2];  // R^T v
    const double ihz = fast_rcp(hc[2]);
    const double u = fku * (hc[0] * ihz) + cam.Cx;
    const double v = fku * (hc[1] * ihz) + cam.Cy;  // ku for both rows (src/Tracking.cpp:471)
    // distort_fm (src/ExtendKF.cpp:175-204) with the refined-reciprocal Newton step of distort_fast_dev
    const double xu = (u - cam.Cx) * cam.dx;
    const double yu = (v - cam.Cy) * cam.dy;
    const double ru = sqrt(xu * xu + yu * yu);
    const double ru2 = ru * ru;
    double rd = ru * fast_rcp(1 + cam.k1 * ru2 + cam.k2 * (ru2 * ru2));
#pragma unroll 1
    for (int it = 0; it < 10; it++) {
        const double rd2 = rd * rd;
        const double rd4 = rd2 * rd2;
        const double f = rd + cam.k1 * (rd2 * rd) + cam.k2 * (rd4 * rd) - ru;
        const double fp = 1 + 3 * cam.k1 * rd2 + 5 * cam.k2 * rd4;
        const double rn = fma(-f, fast_rcp(fp), rd);
        const bool same = !(rn != rd) || !live;  // a NaN lane never settles: rn != rd is true for NaN, so it runs all 10 steps
        rd = rn;
        if (__all_sync(0xffffffffu, same)) break;
    }
    const double rdd = rd * rd;
    const double iD = fast_rcp(1 + cam.k1 * rdd + cam.k2 * (rdd * rdd));
    const double ud = xu * iD * idx + cam.Cx;
    const double vd = yu * iD * idy + cam.Cy;
    bool inl = false;
    if (live) {
        const int fj = F.id_list[jj];
        const double n0 = F.z[2 * fj] - ud, n1 = F.z[2 * fj + 1] - vd;
        inl = n0 * n0 + n1 * n1 < thr2;
    }
    return inl;
}

// ---------------------------------------------------------------------------------------------------------------
// (c) 1-point RANSAC (src/Tracking.cpp:352-539)
// ---------------------------------------------------------------------------------------------------------------
// c.1 ordered compaction of the individually-compatible list and the matched inverse-depth list (z_id columns, :361-397)
__device__ __forceinline__ void ransac_compact_cta(DevFilter& F) {  // CTA-collective, any block size that is a multiple of 32 (<= 1024)
    // flags are 0 / 1: ordered positions from one ballot per warp + the warp totals (three barriers per block of features instead of the
    // 34 of a shared-memory scan)
    __shared__ int s_wa[32], s_wb[32], s_wc[32];
    __shared__ int s_base[3];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if (threadIdx.x == 0) s_base[0] = s_base[1] = s_base[2] = 0;
    __syncthreads();
    for (int base = 0; base < F.N; base += blockDim.x) {
        const int i = base + threadIdx.x;
        bool a = false, b = false, c = false;
        if (i < F.N) {
            a = F.ic[i] != 0;
            const bool idp = F.ftype[i] == 0;
            b = a && idp;
            c = a && !idp;
        }
        const unsigned ba = __ballot_sync(0xffffffffu, a), bb = __ballot_sync(0xffffffffu, b), bc = __ballot_sync(0xffffffffu, c);
        if (lane == 0) {
            s_wa[wid] = __popc(ba);
            s_wb[wid] = __popc(bb);
            s_wc[wid] = __popc(bc);
        }
        __syncthreads();
        int pa = s_base[0], pb = s_base[1];
        for (int w2 = 0; w2 < wid; w2++) {
            pa += s_wa[w2];
            pb += s_wb[w2];
        }
        const unsigned lt = (1u << lane) - 1u;
        pa += __popc(ba & lt);
        pb += __popc(bb & lt);
        if (i < F.N) {
            if (a) F.ic_list[pa] = i;
            if (b) {
                F.id_list[pb] = i;
                F.id_pos[i] = pb;
            } else {
                F.id_pos[i] = -1;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int ta = 0, tb = 0, tc = 0;
            for (int w2 = 0; w2 < nw; w2++) {
                ta += s_wa[w2];
                tb += s_wb[w2];
                tc += s_wc[w2];
            }
            s_base[0] += ta;
            s_base[1] += tb;
            s_base[2] += tc;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        F.ctl[CTL_NIC] = s_base[0];
        F.ctl[CTL_MID] = s_base[1];
        F.ctl[CTL_NCART] = s_base[2];
    }
    for (int i = threadIdx.x; i < F.N; i += blockDim.x) F.support[i] = 0;  // accumulated with atomics by k_ransac_support
}
__global__ void __launch_bounds__(1024) k_ransac_compact(DevFilter* Fs) { ransac_compact_cta(Fs[blockIdx.y]); }

// c.2 one thread per distinct 1-point hypothesis t (match p = ic_list[t]): partial EKF state update restricted to the camera
//     (src/Tracking.cpp:419-422):  g = S_p^-1 (z_p - h_p);  a = Hc_p^T g;  b = Hf_p^T g;  x_i[0..6] = x[0..6] + P[0..6,nz] [a;b]
// tid / nthreads index the tile-ordered row table (always built in full); the hypothesis handled by this thread is t_lo + tid,
// restricted to [t_lo, t_hi) -- a sweep sharded by match index only needs the constants of its own distinct hypotheses.
__device__ __forceinline__ void ransac_hyp_thread(DevFilter& F, int q1, int tid_, int nthreads, int t_lo = 0, int t_hi = 0x7fffffff) {
    int t = tid_;
    // state rows read by the support-scoring tiles, in tile order (one coalesced load per thread there instead of a dependent
    // id_list -> foff chain): kSupTile matches per tile, 6 rows per match, spread over the whole grid.  Quirk Q1 (reference): 3
    // position rows + rho per match, and the two "angle" rows are entries (2jj, 2jj+1) of the stacked POSITION vector of all matches.
    {
        const int m = F.ctl[CTL_MID];
        const int ntile = (m + kSupTile - 1) / kSupTile;
        const int total = ntile * 6 * kSupTile, stride = nthreads;
        for (int e0 = t; e0 < total; e0 += 4 * stride) {  // four entries per pass: their two dependent index loads overlap
            int feat[4], add[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int e = e0 + u * stride;
                feat[u] = -1;
                add[u] = 0;
                if (e >= total) continue;
                const int J0 = (e / (6 * kSupTile)) * kSupTile, k = e % (6 * kSupTile);
                if (q1) {
                    if (k < 4 * kSupTile) {
                        const int jj = J0 + (k >> 2), c = k & 3;
                        if (jj < m) {
                            feat[u] = jj;
                            add[u] = c < 3 ? c : 5;
                        }
                    } else {
                        const int tt = 2 * J0 + (k - 4 * kSupTile);  // index into the stacked position vector ri_v
                        if (tt / 3 < m && (tt >> 1) < m) {
                            feat[u] = tt / 3;
                            add[u] = tt % 3;
                        }
                    }
                } else {
                    const int jj = J0 + k / 6;
                    if (jj < m) {
                        feat[u] = jj;
                        add[u] = k % 6;
                    }
                }
            }
            int idf[4];
#pragma unroll
            for (int u = 0; u < 4; u++) idf[u] = feat[u] >= 0 ? F.id_list[feat[u]] : 0;
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int e = e0 + u * stride;
                if (e < total) F.sup_rows[e] = feat[u] >= 0 ? F.foff[idf[u]] + add[u] : -1;
            }
        }
    }
    t = t_lo + tid_;
    if (t >= F.ctl[CTL_NIC] || t >= t_hi) return;
    const int p = F.ic_list[t];
    const int off = F.foff[p];
    const int fs = F.ftype[p] == 0 ? 6 : 3;
    const double S0 = F.S[4 * p], S1 = F.S[4 * p + 1], S2 = F.S[4 * p + 2], S3 = F.S[4 * p + 3];
    const double idet = 1.0 / (S0 * S3 - S1 * S2);
    const double nu0 = F.z[2 * p] - F.h[2 * p], nu1 = F.z[2 * p + 1] - F.h[2 * p + 1];
    const double g0 = (S3 * nu0 - S1 * nu1) * idet, g1 = (-S2 * nu0 + S0 * nu1) * idet;
    double ab[13];
#pragma unroll
    for (int c = 0; c < 7; c++) ab[c] = F.Hc[14 * p + c] * g0 + F.Hc[14 * p + 7 + c] * g1;
#pragma unroll
    for (int c = 0; c < 6; c++) ab[7 + c] = (c < fs) ? (F.Hf[12 * p + c] * g0 + F.Hf[12 * p + 6 + c] * g1) : 0.0;
#pragma unroll
    for (int c = 0; c < 13; c++) F.hyp_ab[(size_t)t * 16 + c] = ab[c];
    const int ld = F.ldp;
    // the scoring kernel's per-hypothesis constants ride in the same 128-byte record: element offset of column y_p in P, feature size
    F.hyp_ab[(size_t)t * 16 + 13] = __longlong_as_double((long long)off * ld);
    F.hyp_ab[(size_t)t * 16 + 14] = (double)fs;
    F.hyp_ab[(size_t)t * 16 + 15] = 0.0;
    // all 7 x 13 entries of P are fetched as one batch (compile-time trip counts, columns beyond fs predicated off): on the
    // single-filter path this kernel is nothing but memory latency
    double pc[7][13];
#pragma unroll
    for (int r = 0; r < 7; r++) {
#pragma unroll
        for (int c = 0; c < 7; c++) pc[r][c] = F.P[r + (size_t)c * ld];
#pragma unroll
        for (int c = 0; c < 6; c++) pc[r][7 + c] = c < fs ? F.P[r + (size_t)(off + c) * ld] : 0.0;
    }
    double xr[7];
#pragma unroll
    for (int r = 0; r < 7; r++) xr[r] = F.x_km1[r];
#pragma unroll
    for (int r = 0; r < 7; r++) {
        double s = 0;
#pragma unroll
        for (int c = 0; c < 7; c++) s += pc[r][c] * ab[c];
#pragma unroll
        for (int c = 0; c < 6; c++)
            if (c < fs) s += pc[r][7 + c] * ab[7 + c];
        F.hyp_xcam[(size_t)t * 7 + r] = xr[r] + s;
    }
}
__global__ void __launch_bounds__(128) k_ransac_hyp(DevFilter* Fs, int q1) {
    ransac_hyp_thread(Fs[blockIdx.y], q1, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}
// single-CTA fusion of the two for maps of up to 256 features (one dependent launch less on the single-filter path)
__global__ void __launch_bounds__(256) k_ransac_compact_hyp(DevFilter* Fs, int q1) {
    DevFilter& F = Fs[blockIdx.y];
    ransac_compact_cta(F);
    __syncthreads();  // lists and counts written by this CTA are visible to it
    ransac_hyp_thread(F, q1, threadIdx.x, blockDim.x);
}

// c.3 support scoring (compute_hypothesis_support_fast, inlined at src/Tracking.cpp:424-503).
//     CTA = tile of SJT = 64 matched inverse-depth features x batch of SHB = 6 distinct hypotheses, 192 threads, 5 CTAs per SM.
//     The hypothesised feature rows are formed on the fly,      x_i[row] = x[row] + P[row, 0..6] a_p + P[row, y_p] b_p ,
//     so K (n x 2) is never materialised; the only pair-unique HBM traffic is the 6x6 block P[y_j, y_p] (288 B).
//       phase 1: exactly two state rows per thread (384 rows per tile, coalesced down the columns of P); per row the 7 camera
//                columns are read once and reused for the 6 hypotheses, whose 36 pair-unique entries are fetched 12 at a time.
//       phase 2: exactly two (match, hypothesis) pairs per thread: re-projection, Newton distortion, residual < std_z; a warp
//                covers 32 consecutive matches of one hypothesis, so its ballot IS the mask word.
//     ncu (profiles/r01_s2a_support_c4.md) showed the previous version of this kernel ISSUE bound, not HBM bound: 44 warp
//     instructions per pair at 53 % issue-slot utilisation with DRAM at 49 %, while a pure-load kernel with the same access pattern
//     runs at the streaming-copy peak (tools/ubench/pblock_read.cu: 6.9-7.5 TB/s for every tile shape).  Hence the instruction diet:
//     column pointers advanced by one 64-bit add per load instead of re-derived, hypothesis constants as 16-byte shared loads,
//     read-only loads through the non-coherent path, balanced 2 + 2 work per thread, Newton iterations stopped as soon as a whole
//     warp has reached its fixed point (bit-identical to running all 10: a step that leaves rd unchanged leaves it unchanged for
//     good), one shared reciprocal instead of four divisions, squared residual against the squared threshold.
//     Quirk Q1 (reference): the angles of match jj are entries (2jj, 2jj+1) of the stacked POSITION vector of all matches; those
//     two extra rows replace the (unused) theta / phi rows, so the row count per pair is 6 either way.
#ifdef RSLAM_SUP_CLOCKS
__device__ unsigned long long g_sup_clk[8];
#endif
constexpr int SJT = kSupTile, SHB = 6;
constexpr int SUP_THREADS = 192;
constexpr int kSupSmemBytes = 0;
static_assert(6 * SJT == 2 * SUP_THREADS && SHB * SJT == 2 * SUP_THREADS, "two rows and two pairs per thread");
#ifndef RSLAM_SUP_MINB
#define RSLAM_SUP_MINB 5
#endif
__global__ void __launch_bounds__(SUP_THREADS, RSLAM_SUP_MINB) k_ransac_support(DevFilter* Fs, CamDev cam, ParDev par, const int* t_indirect, int t_begin, int t_end,
                                                                  int t_lo, int t_hi, const int* used, int* sup_alt, unsigned long long* pair_counter) {
#ifdef RSLAM_SUP_CLOCKS
    const long long ck0 = clock64();
#endif
    DevFilter& F = Fs[blockIdx.z];
    const int nIC = F.ctl[CTL_NIC];
    const int m = F.ctl[CTL_MID];
    const int J0 = blockIdx.x * SJT;
    if (J0 >= m) return;
    __shared__ int s_t[SHB], s_slot[SHB], s_fsp[SHB];
    __shared__ long long s_colbase[SHB];  // element offset of column y_p in P
    __shared__ __align__(16) double s_ab[SHB][14];
    __shared__ double s_xc[SHB][7], s_R[SHB][9];
    __shared__ double xi[SHB][6 * SJT];
    const int tid = threadIdx.x;
    const bool q1 = (par.quirks & RSLAM_Q1_ANGLES_FROM_POSITIONS) != 0;
    const int ld = F.ldp;
    // Set-up is pure latency (no pair-unique bytes in flight), so its dependent loads are kept to two round trips: every thread that
    // fetches a hypothesis constant resolves the hypothesis itself (slot -> t), and the 128-byte record written by k_ransac_hyp
    // carries a_p, b_p, the column offset of y_p and the feature size together.
    int my_t = -1;
    if (tid < SHB * 16 + SHB * 7) {
        const int pl = tid < SHB * 16 ? (tid >> 4) : (tid - SHB * 16) / 7;
        const int slot = t_begin + blockIdx.y * SHB + pl;
        int t = -1;
        if (slot < t_end) {
            t = t_indirect ? t_indirect[slot] : slot;
            if (t < t_lo || t >= t_hi || t >= nIC) t = -1;
            if (t >= 0 && used && !used[t]) t = -1;
        }
        my_t = t;
        if (tid < SHB * 16) {
            const int c = tid & 15;
            const double v = t >= 0 ? F.hyp_ab[(size_t)t * 16 + c] : 0.0;
            if (c < 13) s_ab[pl][c] = v;
            if (c == 13) {
                s_ab[pl][13] = 0.0;
                s_colbase[pl] = t >= 0 ? __double_as_longlong(v) : 0;
            }
            if (c == 14) s_fsp[pl] = t >= 0 ? (int)v : 0;
            if (c == 15) {
                s_t[pl] = t;
                s_slot[pl] = slot;
            }
        } else {
            const int c = (tid - SHB * 16) % 7;
            s_xc[pl][c] = t >= 0 ? F.hyp_xcam[(size_t)t * 7 + c] : 0.0;
        }
    }
    // the two state rows this thread owns, from the table k_ransac_compact laid out in tile order
    int rows[2];
#pragma unroll
    for (int rr = 0; rr < 2; rr++) rows[rr] = F.sup_rows[(size_t)blockIdx.x * (6 * SJT) + tid + rr * SUP_THREADS];
    const int nv = __syncthreads_count(tid < SHB * 16 && (tid & 15) == 15 && my_t >= 0);
    if (nv == 0) return;
    if (pair_counter && tid == 0) atomicAdd(pair_counter, (unsigned long long)nv * (unsigned long long)min(SJT, m - J0));
    if (tid < SHB && s_t[tid] >= 0) q2r_dev(&s_xc[tid][3], s_R[tid]);  // consumed behind the barrier that separates the two phases
#ifdef RSLAM_SUP_CLOCKS
    const long long ck1 = clock64();
#endif
    // ---- phase 1 ----
    const double* __restrict__ P = F.P;
    const double* __restrict__ x = F.x_km1;
#pragma unroll 1
    for (int rr = 0; rr < 2; rr++) {
        const int k = tid + rr * SUP_THREADS;
        const int row = rows[rr];
        if (row < 0) {
#pragma unroll
            for (int pl = 0; pl < SHB; pl++) xi[pl][k] = 0.0;
            continue;
        }
        const double* prow = P + row;
        double pc[7];
        {
            const double* q = prow;
#pragma unroll
            for (int c = 0; c < 7; c++) {
                pc[c] = __ldg(q);
                q += ld;
            }
        }
        const double xr = __ldg(x + row);
#pragma unroll
        for (int g = 0; g < SHB; g += 2) {  // 2 hypotheses = 12 independent loads in flight per thread (x 960 threads per SM)
            double pv[2][6];
#pragma unroll
            for (int q = 0; q < 2; q++) {
                const double* col = prow + s_colbase[g + q];
                const int fs = s_fsp[g + q];
#pragma unroll
                for (int c = 0; c < 6; c++) {
                    pv[q][c] = (c < 3 ? fs > 0 : fs > 3) ? __ldg(col) : 0.0;
                    col += ld;
                }
            }
#pragma unroll
            for (int q = 0; q < 2; q++) {
                const double2* ab = reinterpret_cast<const double2*>(s_ab[g + q]);
                double a[14];
#pragma unroll
                for (int c = 0; c < 7; c++) {
                    const double2 v = ab[c];
                    a[2 * c] = v.x;
                    a[2 * c + 1] = v.y;
                }
                double sacc = xr;
#pragma unroll
                for (int c = 0; c < 7; c++) sacc += pc[c] * a[c];
#pragma unroll
                for (int c = 0; c < 6; c++) sacc += pv[q][c] * a[7 + c];
                xi[g + q][k] = sacc;
            }
        }
    }
#ifdef RSLAM_SUP_CLOCKS
    const long long ck2a = clock64();
#endif
    __syncthreads();
#ifdef RSLAM_SUP_CLOCKS
    const long long ck2 = clock64();
#endif
    // ---- phase 2 ----
    const double fku = cam.f * (1.0 / cam.dx);
    const double idx = 1.0 / cam.dx, idy = 1.0 / cam.dy;
    const double thr2 = par.std_z * par.std_z;
#pragma unroll 1
    for (int e = tid; e < SHB * SJT; e += SUP_THREADS) {
        const int pl = e / SJT, jl = e % SJT;
        const int jj = J0 + jl;
        const int t = s_t[pl];
        const bool live = t >= 0 && jj < m;
        const bool inl = support_pair_inlier(F, cam, q1, live, xi[pl], jl, jj, s_xc[pl], s_R[pl], fku, idx, idy, thr2);
        const unsigned bal = __ballot_sync(0xffffffffu, inl);
        if ((tid & 31) == 0 && t >= 0 && (jj >> 5) < F.mwords) {
            F.masks[(size_t)t * F.mwords + (jj >> 5)] = bal;
            const int cnt = __popc(bal);
            if (cnt) atomicAdd(sup_alt ? &sup_alt[s_slot[pl]] : &F.support[t], cnt);
        }
    }
#ifdef RSLAM_SUP_CLOCKS
    if (tid == 0) {
        const long long ck3 = clock64();
        atomicAdd(&g_sup_clk[0], (unsigned long long)(ck1 - ck0));
        atomicAdd(&g_sup_clk[1], (unsigned long long)(ck2a - ck1));
        atomicAdd(&g_sup_clk[2], (unsigned long long)(ck2 - ck2a));
        atomicAdd(&g_sup_clk[3], (unsigned long long)(ck3 - ck2));
        atomicAdd(&g_sup_clk[4], 1ull);
    }
#endif
}

__device__ __forceinline__ void gather_inliers(DevFilter& F, int which, int* s_scan, int* s_base);  // kernels_update.cuh

// c.4 replay of the reference's sequential, adaptive control flow (src/Tracking.cpp:403-415, 506-537) over the uniform draws,
//     then write-back of the winner's low_innovation_inlier flags.  One CTA per filter; warp 0 walks the draws 32 at a time:
//     a chunk without a new record (support > best so far) only has to be checked against the current budget n_hyp, so the
//     scalar loop body runs only for the (rare) record-setting hypotheses.
// cond != 0 (rslam_frame's graph, large batches): the low-innovation update that follows sits in an IF node of the graph;
// any filter that has low-innovation inliers arms it, otherwise its launches (every CTA of which would exit at once) are skipped
__global__ void __launch_bounds__(256) k_ransac_select(DevFilter* Fs, ParDev par, int gather_li, unsigned long long cond) {
    DevFilter& F = Fs[blockIdx.y];
    __shared__ int s_state[8];  // 1 max, 2 n_hyp, 3 winner i, 5 hyp_run, 6 status
    constexpr int kResolved = 8192;  // draws resolved to supports up front
    __shared__ int s_sup[kResolved];
    const int nIC = F.ctl[CTL_NIC];
    const int n_u01 = F.n_u01;
    const double* u01 = F.u01;
    const int* support = F.support;
    // the first min(n_u01, 8192) draws are resolved to supports by the whole CTA up front (parallel, latency paid once per batch of 2048:
    // beyond that the warp below pays two dependent round trips per 32 draws -- 86 us of this kernel's 90 at N = 2000, 4800 hypotheses)
    for (int b0 = 0; b0 < kResolved && (b0 == 0 || b0 < n_u01); b0 += 2048) {
        // 8 draws per thread (256 threads): all uniforms first, then all supports -- two round trips instead of sixteen
        double u[8];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int i = b0 + threadIdx.x + k * 256;
            u[k] = (i < n_u01 && nIC > 0) ? u01[i] : -1.0;
        }
        int sv[8];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            sv[k] = -1;
            if (u[k] >= 0.0) {
                const int pos = (int)floor(u[k] * (double)nIC);
                sv[k] = support[pos < nIC ? pos : nIC - 1];
            }
        }
#pragma unroll
        for (int k = 0; k < 8; k++) s_sup[b0 + threadIdx.x + k * 256] = sv[k];
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        int mx = 0, n_hyp = par.n_hyp0, win = -1, run = 0, status = 0;
        bool done = false;
        if (nIC == 0) {
            done = true;
            status = 1;  // Q9
        }
        for (int base = 0; !done; base += 32) {
            const int i = base + lane;
            int s = -1;
            if (i < kResolved && i < ((n_u01 + 2047) & ~2047)) {
                s = s_sup[i];
            } else if (i < n_u01) {
                const int pos = (int)floor(u01[i] * (double)nIC);
                s = support[pos < nIC ? pos : nIC - 1];
            }
            // lanes that would stop the loop if no record happens before them
            const bool over = !(i < n_hyp);           // for-condition fails at i
            const bool exhausted = (i < n_hyp) && s < 0;  // ran out of draws
            const unsigned m_rec = __ballot_sync(0xffffffffu, s > mx);
            const unsigned m_stop = __ballot_sync(0xffffffffu, over || exhausted);
            const int first_rec = m_rec ? __ffs(m_rec) - 1 : 32;
            const int first_stop = m_stop ? __ffs(m_stop) - 1 : 32;
            if (first_rec == 32 && first_stop == 32) {
                run = base + 32;  // whole chunk evaluated, nothing changed
                continue;
            }
            if (first_stop <= first_rec) {  // loop ends before any new record in this chunk
                const bool ex = __shfl_sync(0xffffffffu, (int)exhausted, first_stop) != 0;
                run = base + first_stop;
                if (ex) status = 3;
                done = true;
                continue;
            }
            // a record inside the chunk: replay the chunk sequentially (all lanes run the same scalar code on shuffled values)
            for (int e = 0; e < 32 && !done; e++) {
                const int ie = base + e;
                const int se = __shfl_sync(0xffffffffu, s, e);
                if (!(ie < n_hyp)) {
                    done = true;
                    break;
                }
                if (se < 0) {
                    done = true;
                    status = 3;
                    break;
                }
                run = ie + 1;
                if (se > mx) {
                    mx = se;
                    win = ie;
                    const double epsilon = 1 - ((double)se / (double)nIC);
                    n_hyp = (int)ceil(log(1 - par.p_free) / log(1 - (1 - epsilon)));
                    if (n_hyp == 0) {
                        done = true;
                        break;
                    }
                }
                if (ie > n_hyp) {
                    done = true;
                    break;
                }
            }
        }
        if (lane == 0) {
            s_state[1] = mx;
            s_state[2] = n_hyp;
            s_state[3] = win;
            s_state[5] = run;
            s_state[6] = status;
        }
    }
    __syncthreads();
    const int win = s_state[3];
    int wt = -1;
    if (win >= 0) {
        const int pos = (int)floor(u01[win] * (double)nIC);
        wt = pos < nIC ? pos : nIC - 1;
        const int m = F.ctl[CTL_MID];
        for (int jj = threadIdx.x; jj < m; jj += blockDim.x) {
            const unsigned wbits = F.masks[(size_t)wt * F.mwords + (jj >> 5)];
            F.li[F.id_list[jj]] = (wbits >> (jj & 31)) & 1u;
        }
    }
    if (threadIdx.x == 0) {
        F.ctl[CTL_STATUS] = s_state[6];
        F.ctl[CTL_HYPRUN] = s_state[5];
        F.ctl[CTL_BEST] = s_state[1];
        F.ctl[CTL_NHYP] = s_state[2];
        F.ctl[CTL_WINNER] = win;
        F.ctl[CTL_WINNER_T] = wt;
    }
    if (gather_li) {  // fused first step of ekf_update_li_inliers: ordered inlier list + innovation (saves a launch on the latency path)
        __shared__ int s_scan[256];
        __shared__ int s_base;
        __syncthreads();
        gather_inliers(F, 0, s_scan, &s_base);
        if (cond != 0ull && threadIdx.x == 0 && s_base > 0) cudaGraphSetConditional((cudaGraphConditionalHandle)cond, 1u);
    }
}

// sweep (config C4): reduce key = (support << 32) | (0xFFFFFFFF - hypothesis id) over hypotheses [h0, h1)
__global__ void __launch_bounds__(256) k_sweep_reduce(DevFilter* Fs, const int* hyp_idx, int h0, int h1, int t_lo, int t_hi, const int* sup_alt,
                                                      unsigned long long* out_key) {
    DevFilter& F = Fs[0];
    unsigned long long best = 0ull;
    const int nIC = min(F.ctl[CTL_NIC], t_hi);
    for (int i = h0 + blockIdx.x * blockDim.x + threadIdx.x; i < h1; i += gridDim.x * blockDim.x) {
        const int t = hyp_idx[i];
        if (t < t_lo || t >= nIC) continue;
        const unsigned long long key = ((unsigned long long)(unsigned)(sup_alt ? sup_alt[i] : F.support[t]) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)i);
        best = key > best ? key : best;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long ob = __shfl_xor_sync(0xffffffffu, best, o);
        best = ob > best ? ob : best;
    }
    if ((threadIdx.x & 31) == 0 && best) atomicMax(out_key, best);
}

// sweep set-up in two launches instead of five (the fixed per-sweep cost is what limits the sharded sweep's scaling):
//   k_sweep_compact : ordered match lists (k_ransac_compact) + zeroing of the dedupe marks and of the key / pair counter
//   k_sweep_prep    : blocks [0, nb_hyp) build the hypothesis constants of the distinct hypotheses [t_lo, t_hi) and the row table;
//                     the remaining blocks mark which distinct hypotheses the id range [h0, h1) references (k_sweep_mark)
__global__ void __launch_bounds__(1024) k_sweep_compact(DevFilter* Fs, int* used, int n_used, unsigned long long* key2) {
    ransac_compact_cta(Fs[0]);
    for (int i = threadIdx.x; i < n_used; i += blockDim.x) used[i] = 0;
    if (threadIdx.x < 2) key2[threadIdx.x] = 0ull;
}
__global__ void __launch_bounds__(128) k_sweep_prep(DevFilter* Fs, int q1, int t_lo, int t_hi, int nb_hyp, const int* hyp_idx, int h0, int h1, int m_lo, int m_hi,
                                                    int* used) {
    DevFilter& F = Fs[0];
    if ((int)blockIdx.x < nb_hyp) {
        ransac_hyp_thread(F, q1, blockIdx.x * blockDim.x + threadIdx.x, nb_hyp * blockDim.x, t_lo, t_hi);
        return;
    }
    if (!used) return;
    const int nIC = min(F.ctl[CTL_NIC], m_hi);
    const int nb = gridDim.x - nb_hyp;
    for (int i = h0 + (blockIdx.x - nb_hyp) * blockDim.x + threadIdx.x; i < h1; i += nb * blockDim.x) {
        const int t = hyp_idx[i];
        if (t >= m_lo && t < nIC) used[t] = 1;
    }
}
// After the MAX all-reduce of the key every rank knows the winner; the rank that scored it (its inlier mask row is valid) publishes the
// mask words, every other rank zeros -- a MAX all-reduce of the words then hands the mask to everybody without a host round trip
// (the "broadcast from the owner" of SURVEY 8e with the root resolved on the device).
__global__ void k_sweep_winner_mask(DevFilter* Fs, const unsigned long long* key, const int* hyp_idx, int h0, int h1, int m_lo, int m_hi, unsigned* out_words, int nwords) {
    DevFilter& F = Fs[0];
    const unsigned long long k = *key;
    bool mine = false;
    int t = -1;
    if (k != 0ull) {
        const int id = (int)(0xFFFFFFFFu - (unsigned)(k & 0xFFFFFFFFull));
        t = hyp_idx[id];
        mine = id >= h0 && id < h1 && t >= m_lo && t < min(F.ctl[CTL_NIC], m_hi);
    }
    for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < nwords; w += gridDim.x * blockDim.x)
        out_words[w] = (mine && w < F.mwords) ? F.masks[(size_t)t * F.mwords + w] : 0u;
}

}  // namespace rslam
