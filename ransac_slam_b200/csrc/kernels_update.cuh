// kernels_update.cuh -- (d) joint EKF update of ExtendKF::update (src/ExtendKF.cpp:597-639) for the low- / high-innovation
// inlier sets (src/ExtendKF.cpp:559-596, 640-678), re-formulated for the GPU:
//
//     W = P H^T                      (gather product over the 7 + 6 structurally non-zero columns of each H_i)
//     S = H W + I                    (k x k, k = 2m)
//     S = L L^T                      (blocked right-looking Cholesky, NB = 64, trailing updates on fp64 tensor cores)
//     V = W L^-T ,  y = L^-1 nu      (blocked TRSM; nu rides along as row n of W)
//     x+ = x + V y
//     P+ = P - V V^T                 (SYRK on DMMA tiles, lower triangle + mirrored store => exactly symmetric, which is what
//                                     the reference's 0.5*(P + P^T) produces from its K S K^T form)
//     quaternion normalisation + Jnorm fix-up of rows/cols 3..6 (with the reference's pow(s,-3/2) -> s^-1 quirk, Q4)
//
// In exact arithmetic this equals the reference's K = P H^T S^-1, P - K S K^T.  All fp64.  P stays resident in HBM and is
// updated in place.  m (and therefore k) is data dependent and lives in device memory; grids are sized for the worst case and
// surplus CTAs exit immediately, so the whole frame is a fixed launch sequence (CUDA-graph friendly, no host round trip).
#pragma once
#include "common.cuh"

namespace rslam {

// ---- U1: ordered list of the inlier set + innovation ----------------------------------------------------------------
// which = 0: low_innovation_inlier, prior state x_k_km1 (:559-596); which = 1: high_innovation_inlier, state x_k_k (:640-678).
// CTA-collective, any block size that is a multiple of 32 (every thread of the CTA must call it).  Flags are 0 / 1, so the ordered
// positions come from one ballot per warp + the warp totals (two barriers per chunk instead of a 16-barrier shared-memory scan).
// With an empty low-innovation set the reference copies the prior (src/ExtendKF.cpp:635-638).
__device__ __forceinline__ void gather_inliers(DevFilter& F, int which, int* s_scan /*[>= 32]*/, int* s_base) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if (threadIdx.x == 0) *s_base = 0;
    __syncthreads();
    const unsigned char* flag = which == 0 ? F.li : F.hi;
    for (int base = 0; base < F.N; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const bool a = i < F.N && flag[i];
        const unsigned bal = __ballot_sync(0xffffffffu, a);
        if (lane == 0) s_scan[wid] = __popc(bal);
        __syncthreads();
        int t = *s_base;
        for (int w2 = 0; w2 < wid; w2++) t += s_scan[w2];
        if (a) {
            t += __popc(bal & ((1u << lane) - 1u));
            F.upd_list[t] = i;
            // innovation z - h rides along as row n of W
            F.W[F.n + (size_t)(2 * t) * F.ldw] = F.z[2 * i] - F.h[2 * i];
            F.W[F.n + (size_t)(2 * t + 1) * F.ldw] = F.z[2 * i + 1] - F.h[2 * i + 1];
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int tot = 0;
            for (int w2 = 0; w2 < nw; w2++) tot += s_scan[w2];
            *s_base += tot;
        }
        __syncthreads();
    }
    const int m = *s_base;
    if (threadIdx.x == 0) {
        F.ctl[CTL_M] = m;
        F.ctl[CTL_K] = 2 * m;
    }
    if (which == 0 && m == 0)
        for (int r = threadIdx.x; r < F.n; r += blockDim.x) F.x_kk[r] = F.x_km1[r];
}

__global__ void __launch_bounds__(256) k_upd_gather(DevFilter* Fs, int which) {
    __shared__ int s_scan[256];
    __shared__ int s_base;
    gather_inliers(Fs[blockIdx.y], which, s_scan, &s_base);
}

// ---- U2: W = P H^T.  Thread per state row r, CTA handles a chunk of measurements. ---------------------------------------
constexpr int kWChunk = 8;   // measurements (features) per CTA in y
__global__ void __launch_bounds__(256) k_upd_W(DevFilter* Fs) {
    DevFilter& F = Fs[blockIdx.z];
    const int m = F.ctl[CTL_M];
    const int t0 = blockIdx.y * kWChunk;
    if (t0 >= m) return;
    const int t1 = min(m, t0 + kWChunk);
    __shared__ double sH[kWChunk][26];
    __shared__ int sOff[kWChunk], sFs[kWChunk];
    for (int e = threadIdx.x; e < (t1 - t0) * 26; e += blockDim.x) {
        const int tt = e / 26, c = e % 26;
        const int f = F.upd_list[t0 + tt];
        sH[tt][c] = c < 14 ? F.Hc[14 * f + c] : F.Hf[12 * f + (c - 14)];
    }
    for (int e = threadIdx.x; e < (t1 - t0); e += blockDim.x) {
        const int f = F.upd_list[t0 + e];
        sOff[e] = F.foff[f];
        sFs[e] = F.ftype[f] == 0 ? 6 : 3;
    }
    __syncthreads();
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= F.n) return;
    const int ld = F.ldp;
    const double* P = F.P;
    double pc[7];
#pragma unroll
    for (int c = 0; c < 7; c++) pc[c] = P[r + (size_t)c * ld];
    // two measurements per pass, feature columns with compile-time trip counts (columns beyond fs predicated off): 12 independent
    // loads in flight per thread instead of one (same summation order as before)
    for (int tt0 = 0; tt0 < t1 - t0; tt0 += 2) {
        double pf[2][6];
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int tt = tt0 + u;
            const bool live = tt < t1 - t0;
            const int off = live ? sOff[tt] : 0, fs = live ? sFs[tt] : 0;
#pragma unroll
            for (int c = 0; c < 6; c++) pf[u][c] = c < fs ? P[r + (size_t)(off + c) * ld] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int tt = tt0 + u;
            if (tt >= t1 - t0) break;
            double w0 = 0, w1 = 0;
#pragma unroll
            for (int c = 0; c < 7; c++) {
                w0 += pc[c] * sH[tt][c];
                w1 += pc[c] * sH[tt][7 + c];
            }
            const int fs = sFs[tt];
#pragma unroll
            for (int c = 0; c < 6; c++)
                if (c < fs) {
                    w0 += pf[u][c] * sH[tt][14 + c];
                    w1 += pf[u][c] * sH[tt][20 + c];
                }
            F.W[r + (size_t)(2 * (t0 + tt)) * F.ldw] = w0;
            F.W[r + (size_t)(2 * (t0 + tt) + 1) * F.ldw] = w1;
        }
    }
}

// ---- U3: S = H W + I (lower block triangle only). Thread per (ti >= tj) measurement pair. ------------------------------
__global__ void __launch_bounds__(256) k_upd_S(DevFilter* Fs) {
    DevFilter& F = Fs[blockIdx.z];
    const int m = F.ctl[CTL_M];
    const int tj = blockIdx.y * 16 + (threadIdx.x >> 4);
    const int ti = blockIdx.x * 16 + (threadIdx.x & 15);
    if (ti >= m || tj >= m || ti < tj) return;
    const int f = F.upd_list[ti];
    const int off = F.foff[f], fs = F.ftype[f] == 0 ? 6 : 3;
    const double* Hc = F.Hc + 14 * f;
    const double* Hf = F.Hf + 12 * f;
    const double* w0 = F.W + (size_t)(2 * tj) * F.ldw;
    const double* w1 = w0 + F.ldw;
    double s00 = 0, s01 = 0, s10 = 0, s11 = 0;
#pragma unroll
    for (int c = 0; c < 7; c++) {
        const double a = w0[c], b = w1[c];
        s00 += Hc[c] * a;
        s01 += Hc[c] * b;
        s10 += Hc[7 + c] * a;
        s11 += Hc[7 + c] * b;
    }
    for (int c = 0; c < fs; c++) {
        const double a = w0[off + c], b = w1[off + c];
        s00 += Hf[c] * a;
        s01 += Hf[c] * b;
        s10 += Hf[6 + c] * a;
        s11 += Hf[6 + c] * b;
    }
    if (ti == tj) {
        s00 += 1.0;  // R = I (src/ExtendKF.cpp:594,676)
        s11 += 1.0;
        // keep the diagonal block exactly symmetric: use the lower entry for both
        s01 = s10;
    }
    double* S = F.Sm;
    const int ld = F.lds;
    S[(2 * ti) + (size_t)(2 * tj) * ld] = s00;
    S[(2 * ti + 1) + (size_t)(2 * tj) * ld] = s10;
    S[(2 * ti) + (size_t)(2 * tj + 1) * ld] = s01;
    S[(2 * ti + 1) + (size_t)(2 * tj + 1) * ld] = s11;
}

// ---- U3d: S = H P H^T + I straight from P, for the latency path of a single small filter: with no dependency on W it lets
//           W = P H^T (side stream) run concurrently with S and its single-CTA Cholesky factorisation.  Warp per (ti >= tj)
//           measurement pair; lane l < 7 + fs_i owns one of the state rows H_i touches, forms (P H_j^T)[row, 0..1] in the same
//           order as k_upd_W, multiplies by H_i's two coefficients for that row, and a fixed shuffle tree adds the lanes.
__global__ void __launch_bounds__(256) k_upd_S_direct(DevFilter* Fs) {
    DevFilter& F = Fs[blockIdx.z];
    const int m = F.ctl[CTL_M];
    const int lane = threadIdx.x & 31;
    const int pr = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (pr >= m * (m + 1) / 2) return;
    int ti = (int)((sqrt(8.0 * (double)pr + 1.0) - 1.0) * 0.5);  // pr = ti (ti + 1) / 2 + tj, tj <= ti
    while (ti * (ti + 1) / 2 > pr) ti--;
    while ((ti + 1) * (ti + 2) / 2 <= pr) ti++;
    const int tj = pr - ti * (ti + 1) / 2;
    const int fi = F.upd_list[ti], fj = F.upd_list[tj];
    const int offi = F.foff[fi], fsi = F.ftype[fi] == 0 ? 6 : 3;
    const int offj = F.foff[fj], fsj = F.ftype[fj] == 0 ? 6 : 3;
    double p00 = 0, p01 = 0, p10 = 0, p11 = 0;
    if (lane < 7 + fsi) {
        const int ld = F.ldp;
        const double* prow = F.P + (lane < 7 ? lane : offi + lane - 7);
        const double* Hcj = F.Hc + 14 * fj;
        const double* Hfj = F.Hf + 12 * fj;
        double pc[7], pf[6];
#pragma unroll
        for (int c = 0; c < 7; c++) pc[c] = prow[(size_t)c * ld];
#pragma unroll
        for (int c = 0; c < 6; c++) pf[c] = c < fsj ? prow[(size_t)(offj + c) * ld] : 0.0;
        double w0 = 0, w1 = 0;
#pragma unroll
        for (int c = 0; c < 7; c++) {
            w0 += pc[c] * Hcj[c];
            w1 += pc[c] * Hcj[7 + c];
        }
#pragma unroll
        for (int c = 0; c < 6; c++)
            if (c < fsj) {
                w0 += pf[c] * Hfj[c];
                w1 += pf[c] * Hfj[6 + c];
            }
        const double h0 = lane < 7 ? F.Hc[14 * fi + lane] : F.Hf[12 * fi + lane - 7];
        const double h1 = lane < 7 ? F.Hc[14 * fi + 7 + lane] : F.Hf[12 * fi + 6 + lane - 7];
        p00 = h0 * w0;
        p01 = h0 * w1;
        p10 = h1 * w0;
        p11 = h1 * w1;
    }
#pragma unroll
    for (int o = 8; o >= 1; o >>= 1) {
        p00 += __shfl_down_sync(0xffffffffu, p00, o);
        p01 += __shfl_down_sync(0xffffffffu, p01, o);
        p10 += __shfl_down_sync(0xffffffffu, p10, o);
        p11 += __shfl_down_sync(0xffffffffu, p11, o);
    }
    if (lane == 0) {
        if (ti == tj) {
            p00 += 1.0;  // R = I (src/ExtendKF.cpp:594,676)
            p11 += 1.0;
            p01 = p10;   // keep the diagonal block exactly symmetric: use the lower entry for both
        }
        double* S = F.Sm;
        const int lds = F.lds;
        S[(2 * ti) + (size_t)(2 * tj) * lds] = p00;
        S[(2 * ti + 1) + (size_t)(2 * tj) * lds] = p10;
        S[(2 * ti) + (size_t)(2 * tj + 1) * lds] = p01;
        S[(2 * ti + 1) + (size_t)(2 * tj + 1) * lds] = p11;
    }
}

// ---- async-copy / DMMA primitives ------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool valid) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    const int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}
__device__ __forceinline__ void dmma8x8x4(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// ---- Cholesky of the innovation covariance: 64-wide panels factorised in shared memory -------------------------------------------
// fp64 sqrt / divide / dependent-FMA chains cost ~80-130 cycles each on this part and a CTA barrier ~30, so the panel code keeps
// the per-column serial chain as short as possible and does everything else as wide, independent work:
//   * a 64-wide panel (diagonal block + the rows below it, all in smem) is processed in four 16-column sub-blocks, right-looking;
//   * the 16 x 16 diagonal sub-block is factorised by ONE warp entirely in registers (lane = row, column loop unrolled, pivots and
//     column entries exchanged with shuffles): no barrier and no smem round trip inside the 16 dependent columns
//     (~140 cycles per column: shuffle + rsqrt + multiply + shuffle + FMA);
//   * the rows below are solved one thread per row by forward substitution against that sub-block (running updates, the 120
//     multipliers are broadcast loads), which also writes a k-major copy of the 16 new columns;
//   * the remaining columns of the panel are updated from that copy on the fp64 tensor cores (DMMA m8n8k4, K = 16);
//   * the explicit inverse of the 64 x 64 diagonal block (the TRSM kernels multiply by it on tensor cores) is built one thread
//     per column by forward substitution in registers, by two warps, WHILE the other warps run the trailing update.
constexpr int kSB = 16;
constexpr int kTld = 260;          // panel storage is k-major: entry (row i, column c) at sT[c * kTld + i]; 260 == 4 (mod 16), so DMMA
                                   // fragment loads, thread-per-row accesses and column stores are all bank-conflict free
constexpr int kPanRowsMax = 256;   // diagonal block (rows 0..63) + up to 192 rows below it
// smem carve-up shared by the panel kernels: sT[64][260] panel, sX[64][65] inverse of the diagonal block, sRd[64] (1 / l_jj)
constexpr int kInvLd = 33;  // leading dimension of the 32 x 32 scratch of the blocked triangular inverse
constexpr int kPanelDoubles = kNB * kTld + kNB * (kNB + 1) + kNB + 32 * kInvLd;
constexpr int kPanelSmemBytes = kPanelDoubles * (int)sizeof(double);
constexpr int kCholSmallMaxK = 256;
constexpr int kCholSmallSmemBytes = kPanelSmemBytes;

struct PanelSmem {
    double* sT;
    double (*sX)[kNB + 1];
    double* sRd;
    double* sW;  // [32][kInvLd]
};
template <int LD = kTld>
__device__ __forceinline__ PanelSmem panel_carve(double* base) {
    PanelSmem p;
    p.sT = base;
    p.sX = reinterpret_cast<double(*)[kNB + 1]>(base + kNB * LD);
    p.sRd = base + kNB * LD + kNB * (kNB + 1);
    p.sW = p.sRd + kNB;
    return p;
}

// lanes 0..15 hold row `lane` of a 16 x 16 SPD block (lower triangle in a[0..lane]); on exit a[] is row `lane` of L and rd[j] =
// 1 / l_jj on every lane.  Upper entries are garbage and must be ignored by the caller.
__device__ __forceinline__ void warp_potrf16(double (&a)[kSB], double (&rd)[kSB]) {
    // Per column the serial chain is  pivot shuffle -> 1 / d -> one FMA:  the column entries a_cj are shuffled UNSCALED together with
    // the pivot, the products a_ij a_cj are formed while the reciprocal is in flight, and the update is a_ic -= (a_ij a_cj) (1 / d).
    // The reciprocal is a MUFU.RCP64H seed + two Newton steps (~50 cycles); rsqrt(d) (77 cycles), needed only to scale the finished
    // column and for rd, runs beside the chain.  (Scaling first and shuffling l_ij, as before, put shuffle -> rsqrt -> multiply ->
    // shuffle -> FMA = ~143 cycles on the chain; this is ~85.)
    const unsigned fm = 0xffffffffu;
#pragma unroll
    for (int j = 0; j < kSB; j++) {
        const double aj = a[j];
        const double d = __shfl_sync(fm, aj, j);
        double t[kSB];
#pragma unroll
        for (int c = j + 1; c < kSB; c++) t[c] = aj * __shfl_sync(fm, aj, c);
        double q;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(q) : "d"(d));
        q = q * fma(-d, q, 2.0);
        q = q * fma(-d, q, 2.0);
#pragma unroll
        for (int c = j + 1; c < kSB; c++) a[c] = fma(-t[c], q, a[c]);
        const double r = rsqrt(d);
        rd[j] = r;
        a[j] = aj * r;  // l_ij (lane j: d * rsqrt(d) = sqrt(d))
    }
}

// In-place factorisation of the panel in sT: rows 0..63 = diagonal block (lower triangle valid, identity padding beyond w), rows
// 64..R-1 = the rows below it.  On exit rows 0..63 hold L_jj (lower, zeros above), rows >= 64 hold A L_jj^-T, sRd the reciprocal
// diagonal.  CTA-collective (256 threads).
template <int LD = kTld>
__device__ __forceinline__ void smem_panel_factor(const PanelSmem& ps, int R, int w) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double* sT = ps.sT;
    if (tid < kNB) ps.sRd[tid] = 1.0;
    __syncthreads();
    // not unrolled: the body is ~3 k straight-line instructions (register-resident 16 x 16 potrf); four copies of it made the single-CTA
    // kernel 260 KB of code, i.e. an instruction-cache miss stream on a path that runs every section once or twice per launch
#pragma unroll 1
    for (int c0 = 0; c0 < kNB && c0 < w; c0 += kSB) {
        if (warp == 0) {  // (a) diagonal sub-block, in registers
            double a[kSB], rd[kSB];
            const int l16 = lane & 15, r = c0 + l16;
#pragma unroll
            for (int c = 0; c < kSB; c++) a[c] = (c <= l16) ? sT[(c0 + c) * LD + r] : 0.0;
            warp_potrf16(a, rd);
            if (lane < kSB) {
#pragma unroll
                for (int c = 0; c < kSB; c++) sT[(c0 + c) * LD + r] = (c <= lane) ? a[c] : 0.0;
                double myrd = 1.0;
#pragma unroll
                for (int c = 0; c < kSB; c++)
                    if (c == lane) myrd = rd[c];
                ps.sRd[r] = myrd;
            }
        }
        __syncthreads();
        const int base = c0 + kSB;  // first row / column behind the sub-block
        {  // (b) rows behind the sub-block: x = a L_ss^-T by forward substitution, one thread per row (multipliers are broadcast loads)
            const int i = base + tid;
            if (i < R) {
                double a[kSB];
#pragma unroll
                for (int c = 0; c < kSB; c++) a[c] = sT[(c0 + c) * LD + i];
#pragma unroll
                for (int c = 0; c < kSB; c++) {
                    const double x = a[c] * ps.sRd[c0 + c];
                    a[c] = x;
#pragma unroll
                    for (int c2 = c + 1; c2 < kSB; c2++) a[c2] = fma(-x, sT[(c0 + c) * LD + c0 + c2], a[c2]);
                }
#pragma unroll
                for (int c = 0; c < kSB; c++) sT[(c0 + c) * LD + i] = a[c];
            }
        }
        __syncthreads();
        const int ncol = kNB - base;  // 48, 32, 16, 0 columns of the panel still to update
        if (ncol > 0) {               // (c) A[i][c] -= sum_t x_it x_ct on DMMA tiles (rows i >= base, cols base <= c < 64, c <= i)
            const int nrow = R - base;
            const int MT = (nrow + 15) >> 4, NT = ncol >> 3;  // warp tile 16 x 8
            for (int tile = warp; tile < MT * NT; tile += 8) {
                const int mt = tile / NT, nt = tile - mt * NT;
                if (mt * 16 + 15 < nt * 8) continue;  // entirely above the diagonal
                double c00 = 0.0, c01 = 0.0, c10 = 0.0, c11 = 0.0;
#pragma unroll
                for (int ks = 0; ks < kSB / 4; ks++) {
                    const double* kr = sT + (c0 + ks * 4 + (lane & 3)) * LD + base;
                    const double bf = kr[nt * 8 + (lane >> 2)];
                    dmma8x8x4(c00, c01, kr[mt * 16 + (lane >> 2)], bf);
                    dmma8x8x4(c10, c11, kr[mt * 16 + 8 + (lane >> 2)], bf);
                }
                const int i = base + mt * 16 + (lane >> 2), cc = base + nt * 8 + 2 * (lane & 3);
                if (i < R) {
                    if (cc <= i) sT[cc * LD + i] -= c00;
                    if (cc + 1 <= i) sT[(cc + 1) * LD + i] -= c01;
                }
                if (i + 8 < R) {
                    if (cc <= i + 8) sT[cc * LD + i + 8] -= c10;
                    if (cc + 1 <= i + 8) sT[(cc + 1) * LD + i + 8] -= c11;
                }
            }
            __syncthreads();
        }
    }
}

// explicit inverse of the 64 x 64 lower-triangular diagonal block (rows 0..63 of sT, identity padded) -> sX (full 64 x 64, zeros
// above the diagonal), BLOCKED:  inv [A 0; B C] = [inv A 0; -inv C * (B * inv A)  inv C].
//   level 0: the four 16 x 16 diagonal blocks, concurrently.  Column c of a block's inverse solves L x = e_c by forward
//            substitution with running updates of the right-hand side; FOUR adjacent lanes share a column (two warps per block, all
//            8 warps busy): lane part p keeps rows 4 q + p, the owner of row t forms x_t = b_t / l_tt and hands it to its three
//            neighbours with a shuffle.  The chain is multiply -> shuffle -> FMA, ~180 cycles per step: 16 steps here instead of the
//            64 of an unblocked substitution (which cost 11.6 k cycles, a quarter of the single-CTA factorisation).
//   level 1 / 2: the off-diagonal 16 x 16 and 32 x 32 blocks from two small products each on the fp64 tensor cores.
// CTA-collective (256 threads).
template <int LD = kTld>
__device__ __forceinline__ void smem_trinv64(const PanelSmem& ps) {
    const unsigned fm = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double* sT = ps.sT;
    {   // level 0
        const int r0 = 16 * (warp >> 1), cl = (warp & 1) * 8 + (lane >> 2), p = lane & 3;
        double b[4];
#pragma unroll
        for (int q = 0; q < 4; q++) b[q] = (4 * q + p == cl) ? 1.0 : 0.0;
#pragma unroll
        for (int t = 0; t < 16; t++) {
            const double x = __shfl_sync(fm, b[t / 4] * ps.sRd[r0 + t], (lane & ~3) | (t & 3));
            if (p == (t & 3)) ps.sX[r0 + t][r0 + cl] = x;
            // rows 4 q + p behind t; entries of rows <= t are already final (or were stored above) and may be clobbered
#pragma unroll
            for (int q = t / 4; q < 4; q++) b[q] = fma(-sT[(r0 + t) * LD + r0 + 4 * q + p], x, b[q]);
        }
        // blocks above the block diagonal are zero
        for (int e = tid; e < 6 * 256; e += 256) {
            const int blk = e >> 8, i = (e >> 4) & 15, j = e & 15;
            const int bi = blk < 3 ? 0 : (blk < 5 ? 1 : 2), bj = blk < 3 ? blk + 1 : (blk < 5 ? blk - 1 : 3);
            ps.sX[16 * bi + i][16 * bj + j] = 0.0;
        }
    }
    __syncthreads();
    // C (8 x 8 per warp) = A * B with A(i, k) = a_at(i, k), B(k, j) = b_at(k, j), K a multiple of 4
    const int fr = lane >> 2, fk = lane & 3;
    {   // level 1: for each 32 x 32 half h: X21 = -X22 * (L21 * X11), 16 x 16 blocks; 2 halves x 4 output tiles = one tile per warp
        const int h = warp >> 2, mi = (warp >> 1) & 1, ni = warp & 1, base = 32 * h;
        double c0 = 0.0, c1 = 0.0;
#pragma unroll
        for (int ks = 0; ks < 4; ks++) {  // T = L21 * X11
            const int k = base + ks * 4 + fk;
            dmma8x8x4(c0, c1, sT[k * LD + base + 16 + mi * 8 + fr], ps.sX[k][base + ni * 8 + fr]);
        }
        double* T = ps.sW + h * 16 * kInvLd;  // [16][kInvLd] per half
        T[(mi * 8 + fr) * kInvLd + ni * 8 + 2 * fk] = c0;
        T[(mi * 8 + fr) * kInvLd + ni * 8 + 2 * fk + 1] = c1;
        __syncthreads();
        c0 = c1 = 0.0;
#pragma unroll
        for (int ks = 0; ks < 4; ks++) {  // X21 = -X22 * T
            const int k = ks * 4 + fk;
            dmma8x8x4(c0, c1, ps.sX[base + 16 + mi * 8 + fr][base + 16 + k], T[k * kInvLd + ni * 8 + fr]);
        }
        ps.sX[base + 16 + mi * 8 + fr][base + ni * 8 + 2 * fk] = -c0;
        ps.sX[base + 16 + mi * 8 + fr][base + ni * 8 + 2 * fk + 1] = -c1;
    }
    __syncthreads();
    {   // level 2: X21 (rows 32..63, cols 0..31) = -X22 * (L21 * X11), 32 x 32 blocks; 16 output tiles, two per warp
        const int mi = warp >> 1, nj = (warp & 1) * 2;
        double c[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
#pragma unroll
        for (int ks = 0; ks < 8; ks++) {  // T = L21 * X11
            const int k = ks * 4 + fk;
            const double a = sT[k * LD + 32 + mi * 8 + fr];
#pragma unroll
            for (int u = 0; u < 2; u++) dmma8x8x4(c[u][0], c[u][1], a, ps.sX[k][(nj + u) * 8 + fr]);
        }
        __syncthreads();  // level 1 is done reading sW
#pragma unroll
        for (int u = 0; u < 2; u++) {
            ps.sW[(mi * 8 + fr) * kInvLd + (nj + u) * 8 + 2 * fk] = c[u][0];
            ps.sW[(mi * 8 + fr) * kInvLd + (nj + u) * 8 + 2 * fk + 1] = c[u][1];
            c[u][0] = c[u][1] = 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int ks = 0; ks < 8; ks++) {  // X21 = -X22 * T
            const int k = ks * 4 + fk;
            const double a = ps.sX[32 + mi * 8 + fr][32 + k];
#pragma unroll
            for (int u = 0; u < 2; u++) dmma8x8x4(c[u][0], c[u][1], a, ps.sW[k * kInvLd + (nj + u) * 8 + fr]);
        }
#pragma unroll
        for (int u = 0; u < 2; u++) {
            ps.sX[32 + mi * 8 + fr][(nj + u) * 8 + 2 * fk] = -c[u][0];
            ps.sX[32 + mi * 8 + fr][(nj + u) * 8 + 2 * fk + 1] = -c[u][1];
        }
    }
    __syncthreads();
}

__device__ __forceinline__ void store_linv(const double (*sX)[kNB + 1], double* out, int t0, int nt) {  // 64 x 64 column-major
    for (int e = t0; e < kNB * kNB; e += nt) out[e] = sX[e % kNB][e / kNB];
}

// load the diagonal block at (j0, j0) (identity padded beyond w) and `nr` rows starting at global row r0 into the panel.
// Warp `wp` takes columns wp, wp + 8, ...; a lane takes rows lane, lane + 32, ...: no integer divisions, and all of a thread's loads
// of a column batch are issued before the first store (the element-indexed loop this replaces kept one load in flight per
// thread and cost ~8.7 k cycles per 64 x 128 panel, a fifth of the single-CTA factorisation).
template <int LD = kTld>
__device__ __forceinline__ void panel_load(const PanelSmem& ps, const double* S, int ld, int j0, int w, int r0, int nr) {
    // plain (coherent) loads: k_chol_small re-reads entries of S that its own trailing update has just written.
    // 256 threads: warp wp owns columns wp + 8 cs; all (up to 64) loads of a thread are issued before its first store.
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    double v[8][8];
#pragma unroll
    for (int cs = 0; cs < 8; cs++) {
        const int c = wp + 8 * cs;
        const double* col = S + (size_t)(j0 + c) * ld;
#pragma unroll
        for (int q = 0; q < 2; q++) {
            const int i = lane + 32 * q;
            v[cs][q] = (i == c) ? 1.0 : 0.0;
            if (i < w && c < w && i >= c) v[cs][q] = col[j0 + i];
        }
#pragma unroll
        for (int q = 0; q < 6; q++) {
            const int i = lane + 32 * q;
            v[cs][2 + q] = (c < w && i < nr) ? col[r0 + i] : 0.0;
        }
    }
#pragma unroll
    for (int cs = 0; cs < 8; cs++) {
        double* dst = ps.sT + (wp + 8 * cs) * LD;
        dst[lane] = v[cs][0];
        dst[lane + 32] = v[cs][1];
#pragma unroll
        for (int q = 0; q < 6; q++) {
            const int i = lane + 32 * q;
            if (i < nr) dst[kNB + i] = v[cs][2 + q];
        }
    }
}

// ---- U4a: Cholesky panel at block column `step` (multi-launch path, k > 256).  Every CTA owns one 64-row block of the panel and
//           factors the diagonal block redundantly (cheaper than a dependent launch).  LEFT-LOOKING inside a 256-wide outer block:
//           before factoring, the CTA subtracts from its 128 x 64 slice (diagonal block + own rows) the contribution of the earlier
//           panels of the same outer block (K <= 192, DMMA, staged through the unused rows of the panel buffer), so a frame has one
//           launch per panel plus one K = 256 trailing update per outer block -- 78 launches at k = 4000 instead of 250, and no thin
//           K = 64 GEMMs.  The inverses of the diagonal blocks are built afterwards, all at once (k_chol_trinv).
constexpr int kOB = 4;  // panels per outer block
__global__ void __launch_bounds__(256) k_chol_panel(DevFilter* Fs, int step) {
    DevFilter& F = Fs[blockIdx.y];
    const int kk = F.ctl[CTL_K];
    const int j0 = kNB * step;
    if (j0 >= kk) return;
    const int r0 = j0 + kNB * blockIdx.x;
    if (r0 >= kk) return;
    const int w = min(kNB, kk - j0);
    extern __shared__ __align__(16) double psm[];
    const PanelSmem ps = panel_carve(psm);
    double* S = F.Sm;
    const int ld = F.lds;
    const int nr = blockIdx.x == 0 ? 0 : min(kNB, kk - r0);
#ifdef RSLAM_PHASE_CLOCKS
    long long tprev = clock64();
#define PPH(i) do { __syncthreads(); if (blockIdx.x == 1 && threadIdx.x == 0) { const long long now__ = clock64(); F.Jn[16 + (i)] += (double)(now__ - tprev); tprev = now__; } } while (0)
#else
#define PPH(i)
#endif
    panel_load(ps, S, ld, j0, w, r0, nr);
    PPH(0);
    const int ob0 = kNB * kOB * (step / kOB);  // first column of the outer block
    if (ob0 < j0) {
        // pending update: [D; A] -= [Ld; La] Ld^T over the columns [ob0, j0) already factored in this outer block
        const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
        const bool active = wp < 4 || nr > 0;  // warp wp owns rows 16 wp .. 16 wp + 15 of the 128-row slice
        double acc[2][8][2];
#pragma unroll
        for (int a2 = 0; a2 < 2; a2++)
#pragma unroll
            for (int b2 = 0; b2 < 8; b2++) acc[a2][b2][0] = acc[a2][b2][1] = 0.0;
        double* U = ps.sT + 2 * kNB;  // staging: entry (k, row) at U[k * kTld + row], rows 0..63 = diagonal rows, 64..127 = own rows
        // chunk c0: 64 columns x 128 rows, 32 values per thread, fetched into registers one chunk ahead (in flight during the DMMA work)
        double v[8][4];
        auto fetch = [&](int c0) {
#pragma unroll
            for (int cs = 0; cs < 8; cs++) {
                const double* col = S + (size_t)(c0 + wp + 8 * cs) * ld;
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const int r = lane + 32 * q;
                    const int grow = r < kNB ? j0 + r : r0 + (r - kNB);
                    const bool ok = r < kNB ? (r < w) : (r - kNB < nr);
                    v[cs][q] = ok ? col[grow] : 0.0;
                }
            }
        };
        fetch(ob0);
        for (int c0 = ob0; c0 < j0; c0 += kNB) {
            __syncthreads();  // the previous chunk has been consumed
#pragma unroll
            for (int cs = 0; cs < 8; cs++)
#pragma unroll
                for (int q = 0; q < 4; q++) U[(wp + 8 * cs) * kTld + lane + 32 * q] = v[cs][q];
            __syncthreads();
            if (c0 + kNB < j0) fetch(c0 + kNB);
            if (active) {
#pragma unroll 4
                for (int ks = 0; ks < kNB / 4; ks++) {
                    const double* kr = U + (ks * 4 + (lane & 3)) * kTld;
                    double af[2], bf[8];
#pragma unroll
                    for (int a2 = 0; a2 < 2; a2++) af[a2] = kr[wp * 16 + a2 * 8 + (lane >> 2)];
#pragma unroll
                    for (int b2 = 0; b2 < 8; b2++) bf[b2] = kr[b2 * 8 + (lane >> 2)];
#pragma unroll
                    for (int a2 = 0; a2 < 2; a2++)
#pragma unroll
                        for (int b2 = 0; b2 < 8; b2++) dmma8x8x4(acc[a2][b2][0], acc[a2][b2][1], af[a2], bf[b2]);
                }
            }
        }
        if (active) {
#pragma unroll
            for (int a2 = 0; a2 < 2; a2++)
#pragma unroll
                for (int b2 = 0; b2 < 8; b2++)
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int i = wp * 16 + a2 * 8 + (lane >> 2), cc = b2 * 8 + 2 * (lane & 3) + e;
                        // identity padding of the diagonal block (rows / columns >= w) must stay untouched: its staged rows were zero
                        ps.sT[cc * kTld + i] -= acc[a2][b2][e];
                    }
        }
    }
    __syncthreads();
    PPH(1);
    smem_panel_factor(ps, kNB + nr, w);
    PPH(2);
    if (blockIdx.x == 0) {
        for (int e = threadIdx.x; e < kNB * kNB; e += blockDim.x) {
            const int i = e % kNB, c = e / kNB;
            if (i < w && c < w) S[(j0 + i) + (size_t)(j0 + c) * ld] = ps.sT[c * kTld + i];
        }
        return;
    }
    for (int e = threadIdx.x; e < nr * kNB; e += blockDim.x) {
        const int i = e % nr, c = e / nr;
        if (c < w) S[(r0 + i) + (size_t)(j0 + c) * ld] = ps.sT[c * kTld + kNB + i];
    }
    PPH(3);
#ifdef RSLAM_PHASE_CLOCKS
    if (threadIdx.x == 0 && blockIdx.x == 1) F.Jn[16 + 4] += 1.0;
#endif
#undef PPH
}

// ---- U4b: explicit inverses of ALL 64 x 64 diagonal blocks of the finished factor, one CTA per block (the TRSM kernel multiplies by
//           them on tensor cores).  Built after the factorisation so that the 63 serial panel steps do not each carry one.
constexpr int kTrinvLd = 68;  // 64 rows are enough here; == 4 (mod 16) like kTld, so the same access patterns stay conflict free
constexpr int kTrinvSmemBytes = (kNB * kTrinvLd + kNB * (kNB + 1) + kNB + 32 * kInvLd) * (int)sizeof(double);  // 77 KB: 2 CTAs per SM
__global__ void __launch_bounds__(256) k_chol_trinv(DevFilter* Fs) {
    DevFilter& F = Fs[blockIdx.y];
    const int kk = F.ctl[CTL_K];
    const int j0 = kNB * blockIdx.x;
    if (j0 >= kk) return;
    const int w = min(kNB, kk - j0);
    extern __shared__ __align__(16) double psm[];
    const PanelSmem ps = panel_carve<kTrinvLd>(psm);
    panel_load<kTrinvLd>(ps, F.Sm, F.lds, j0, w, j0, 0);
    __syncthreads();
    if (threadIdx.x < kNB) ps.sRd[threadIdx.x] = 1.0 / ps.sT[threadIdx.x * kTrinvLd + threadIdx.x];
    // panel_load leaves the strict upper triangle of the block zero and the padding identity: exactly what smem_trinv64 expects
    __syncthreads();
    smem_trinv64<kTrinvLd>(ps);
    store_linv(ps.sX, F.Linv + (size_t)blockIdx.x * kNB * kNB, threadIdx.x, blockDim.x);
}

// ---- U4s: whole Cholesky (+ inverses of the diagonal blocks) in ONE CTA for small systems (k <= 256): the launch-latency
//           path of the 100-feature configuration.
// LD: panel row capacity (k-major leading dimension, == 4 mod 16); MINB: CTAs per SM asked of the compiler.  <kTld, 1> serves any k <= 256;
// <212, 2> (k <= 200: the 100-feature filters) fits two CTAs per SM -- 109 KB of shared memory each, no scratch for the inverse (that is
// k_chol_trinv's) -- so that one filter's serial column chain runs beside another's.
constexpr int kCholSmallLd2 = 212;
constexpr int kCholSmall2SmemBytes = (kNB * kCholSmallLd2 + kNB) * (int)sizeof(double);
template <int LD, int MINB>
__global__ void __launch_bounds__(256, MINB) k_chol_small(DevFilter* Fs) {
    DevFilter& F = Fs[blockIdx.y];
    const int kk = F.ctl[CTL_K];
    if (kk <= 0) return;
    extern __shared__ __align__(16) double psm[];
    PanelSmem ps = panel_carve<LD>(psm);
    if (LD != kTld) {  // compact carve-up: panel + reciprocal diagonal only
        ps.sRd = psm + kNB * LD;
        ps.sX = nullptr;
        ps.sW = nullptr;
    }
    double* S = F.Sm;
    const int ld = F.lds;
#ifdef RSLAM_PHASE_CLOCKS
    long long tc[6] = {0, 0, 0, 0, 0, 0};
#define PH(i) do { __syncthreads(); const long long now__ = clock64(); tc[i] += now__ - tprev; tprev = now__; } while (0)
    long long tprev = clock64();
#else
#define PH(i)
#endif
    for (int j0 = 0; j0 < kk; j0 += kNB) {
        const int w = min(kNB, kk - j0);
        const int rem = max(0, kk - (j0 + kNB));
        panel_load<LD>(ps, S, ld, j0, w, j0 + kNB, rem);
        __syncthreads();
        PH(0);
        smem_panel_factor<LD>(ps, kNB + rem, w);
        PH(1);
        // store the panel and run the trailing update on DMMA tiles (the inverses of the diagonal blocks, which the TRSM kernel
        // multiplies by, are built afterwards by k_chol_trinv for all blocks at once: ~10 k cycles less on this serial chain per panel)
        {
            {
                const int ln = threadIdx.x & 31, wp = threadIdx.x >> 5;
                for (int c = wp; c < w; c += 8) {  // warp per column, lanes down the rows: coalesced, no divisions
                    double* col = S + (size_t)(j0 + c) * ld + j0;
                    const double* src = ps.sT + c * LD;
                    for (int i = ln; i < w; i += 32) col[i] = src[i];
                    for (int i = ln; i < rem; i += 32) col[kNB + i] = src[kNB + i];
                }
            }
            // trailing update S[a, b] -= sum_c X[a, c] X[b, c] (lower triangle), warp tiles 16 x 32 straight from the k-major panel
            const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
            const int MT = (rem + 15) >> 4, NT = (rem + 31) >> 5;
            for (int tile = wrp; tile < MT * NT; tile += 8) {
                const int mt = tile / NT, nt2 = tile - mt * NT;
                if (mt * 16 + 15 < nt2 * 32) continue;
                double acc[2][4][2];
#pragma unroll
                for (int a = 0; a < 2; a++)
#pragma unroll
                    for (int b = 0; b < 4; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
#pragma unroll 4
                for (int ks = 0; ks < kNB / 4; ks++) {
                    const double* kr = ps.sT + (ks * 4 + (lane & 3)) * LD + kNB;
                    double af[2], bf[4];
#pragma unroll
                    for (int a = 0; a < 2; a++) af[a] = kr[mt * 16 + a * 8 + (lane >> 2)];
#pragma unroll
                    for (int b = 0; b < 4; b++) bf[b] = kr[nt2 * 32 + b * 8 + (lane >> 2)];
#pragma unroll
                    for (int a = 0; a < 2; a++)
#pragma unroll
                        for (int b = 0; b < 4; b++) dmma8x8x4(acc[a][b][0], acc[a][b][1], af[a], bf[b]);
                }
#pragma unroll
                for (int a = 0; a < 2; a++)
#pragma unroll
                    for (int b = 0; b < 4; b++)
#pragma unroll
                        for (int e = 0; e < 2; e++) {
                            const int ar = mt * 16 + a * 8 + (lane >> 2), bc = nt2 * 32 + b * 8 + 2 * (lane & 3) + e;
                            if (ar < rem && bc <= ar) S[(j0 + kNB + ar) + (size_t)(j0 + kNB + bc) * ld] -= acc[a][b][e];
                        }
            }
        }
        __syncthreads();  // the trailing update must have landed before the next panel is loaded; sT is reused
        PH(2);
    }
#ifdef RSLAM_PHASE_CLOCKS
    if (threadIdx.x == 0)
        for (int i = 0; i < 6; i++) F.Jn[16 + i] = (double)tc[i];
#endif
#undef PH
}

// ---- U5: TRSM  V = W L^-T  for all n+1 rows of W (row n: the innovation, which becomes y = L^-1 nu), ONE launch ---------------
// Left-looking over 64-wide column blocks, a CTA owns R rows for the whole solve (no inter-CTA dependency):
//     V_j = ( W_j - sum_{i<j} V_i L_ji^T ) * inv(L_jj)^T
// Both products run on fp64 tensor cores (DMMA m8n8k4); the K = 64 j accumulation streams V (own rows, written earlier by this
// CTA) and L through a 3-stage cp.async pipeline; the diagonal step multiplies by the explicit inverse of the 64 x 64 diagonal
// block produced by the Cholesky kernels, so there is no serial substitution on the n-row side.
constexpr int GBK_T = 16, GSTAGES_T = 3;
template <int R, int WM>
struct TrsmCfg {
    static constexpr int kThreads = WM * 2 * 32;
    static constexpr int kMT = R / (8 * WM);       // m8 tiles per warp
    static constexpr int kLdA = R + 4;             // doubles per k-row of the A / T staging (== 8 mod 32 words -> conflict free)
    static constexpr int kLdB = kNB + 4;
    static constexpr int kSmemBytes = (GSTAGES_T * GBK_T * (kLdA + kLdB) + kNB * kLdA + kNB * kLdB) * (int)sizeof(double);
};

// Two-level like the Cholesky: the launch covers the 64-wide column blocks [jb0, jb1) of one 256-wide outer block and accumulates only over
// the blocks of that outer block (K <= 192); the contribution of every earlier outer block has already been subtracted from W by a
// K = 256 GEMM (GEMM_TRSM_OUTER) that runs at the SYRK kernel's efficiency instead of this kernel's (58 % of the fp64 tensor rate when it
// carried the whole K = 64 j accumulation).
template <int R, int WM>
__global__ void __launch_bounds__(WM * 64) k_trsm_ll(DevFilter* Fs, int jb0, int jb1) {
    using Cfg = TrsmCfg<R, WM>;
    constexpr int MT = Cfg::kMT, LDA = Cfg::kLdA, LDB = Cfg::kLdB, NT = 4;
    static_assert(R % (8 * WM) == 0 && (LDA % 2) == 0, "tile shape");
    DevFilter& F = Fs[blockIdx.y];
    const int kk = F.ctl[CTL_K];
    if (kk <= 0) return;
    const int M = F.n + 1;
    const int r0 = blockIdx.x * R;
    if (r0 >= M) return;
    extern __shared__ __align__(16) double tsm[];
    double* As = tsm;                                   // [stage][GBK][LDA]
    double* Bs = As + GSTAGES_T * GBK_T * LDA;          // [stage][GBK][LDB]
    double* Ts = Bs + GSTAGES_T * GBK_T * LDB;          // [64][LDA]   T = W_j - acc   (k-major, like an A tile)
    double* Ls = Ts + kNB * LDA;                        // [64][LDB]   Ls[k][n] = inv(L_jj)[n][k]
    double* W = F.W;
    const double* Sm = F.Sm;
    const int ldw = F.ldw, lds = F.lds;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm0 = (warp % WM) * (MT * 8), wn0 = (warp / WM) * 32;
    const int nb = min((kk + kNB - 1) / kNB, jb1);
    if (jb0 * kNB >= kk) return;
    constexpr int A_CHUNKS = GBK_T * (R / 2), B_CHUNKS = GBK_T * (kNB / 2);
    const int kbase = jb0 * kNB;  // first column of the outer block

    for (int j = jb0; j < nb; j++) {
        const int c0 = j * kNB;
        const int w = min(kNB, kk - c0);
        // inverse of the diagonal block -> Ls (async, overlaps the accumulation)
        {
            const double* Li = F.Linv + (size_t)j * kNB * kNB;
            for (int ch = tid; ch < kNB * (kNB / 2); ch += Cfg::kThreads) {
                const int kc = ch / (kNB / 2), r2 = ch % (kNB / 2);
                cp_async16(&Ls[kc * LDB + 2 * r2], Li + 2 * r2 + (size_t)kc * kNB, true);
            }
            cp_async_commit();
        }
        double acc[MT][NT][2];
#pragma unroll
        for (int a = 0; a < MT; a++)
#pragma unroll
            for (int b = 0; b < NT; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
        // this thread's entries of W_j, fetched now: they are needed only after the accumulation (ncu: long-scoreboard 1.56 warps per
        // issue with the loads placed at the point of use), and nothing in this launch writes block j before its own diagonal step
        double wpre[MT][NT][2];
#pragma unroll
        for (int mt = 0; mt < MT; mt++) {
            const int row = r0 + wm0 + mt * 8 + (lane >> 2);
#pragma unroll
            for (int nt = 0; nt < NT; nt++)
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    const int cl = wn0 + nt * 8 + 2 * (lane & 3) + e;
                    wpre[mt][nt][e] = (row < M && cl < w) ? W[row + (size_t)(c0 + cl) * ldw] : 0.0;
                }
        }
        const int nkt = (c0 - kbase) / GBK_T;  // K = 64 (j - jb0)
        auto load_stage = [&](int stage, int kt) {
            const int k0 = kbase + kt * GBK_T;
            for (int ch = tid; ch < A_CHUNKS; ch += Cfg::kThreads) {
                const int kc = ch / (R / 2), r2 = ch % (R / 2);
                const int row = r0 + 2 * r2;
                const bool v = row < M;
                cp_async16(&As[(stage * GBK_T + kc) * LDA + 2 * r2], v ? (W + row + (size_t)(k0 + kc) * ldw) : W, v);
            }
            for (int ch = tid; ch < B_CHUNKS; ch += Cfg::kThreads) {
                const int kc = ch / (kNB / 2), r2 = ch % (kNB / 2);
                const int row = c0 + 2 * r2;
                const bool v = row < kk;
                cp_async16(&Bs[(stage * GBK_T + kc) * LDB + 2 * r2], v ? (Sm + row + (size_t)(k0 + kc) * lds) : Sm, v);
            }
        };
#pragma unroll
        for (int s = 0; s < GSTAGES_T - 1; s++) {
            if (s < nkt) load_stage(s, s);
            cp_async_commit();
        }
        for (int kt = 0; kt < nkt; kt++) {
            cp_async_wait<GSTAGES_T - 2>();
            __syncthreads();
            {
                const int nk = kt + GSTAGES_T - 1;
                if (nk < nkt) load_stage(nk % GSTAGES_T, nk);
                cp_async_commit();
            }
            const double* as = As + (kt % GSTAGES_T) * GBK_T * LDA;
            const double* bs = Bs + (kt % GSTAGES_T) * GBK_T * LDB;
#pragma unroll
            for (int ks = 0; ks < GBK_T / 4; ks++) {
                const int krow = ks * 4 + (lane & 3);
                double af[MT], bf[NT];
#pragma unroll
                for (int mt = 0; mt < MT; mt++) af[mt] = as[krow * LDA + wm0 + mt * 8 + (lane >> 2)];
#pragma unroll
                for (int nt = 0; nt < NT; nt++) bf[nt] = bs[krow * LDB + wn0 + nt * 8 + (lane >> 2)];
#pragma unroll
                for (int mt = 0; mt < MT; mt++)
#pragma unroll
                    for (int nt = 0; nt < NT; nt++) dmma8x8x4(acc[mt][nt][0], acc[mt][nt][1], af[mt], bf[nt]);
            }
        }
        cp_async_wait<0>();
        __syncthreads();
        // T = W_j - acc  -> Ts[col][row]
#pragma unroll
        for (int mt = 0; mt < MT; mt++) {
            const int rl = wm0 + mt * 8 + (lane >> 2);
            const int row = r0 + rl;
#pragma unroll
            for (int nt = 0; nt < NT; nt++) {
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    const int cl = wn0 + nt * 8 + 2 * (lane & 3) + e;
                    double v = 0.0;
                    if (row < M && cl < w) v = wpre[mt][nt][e] - acc[mt][nt][e];
                    Ts[cl * LDA + rl] = v;
                }
            }
        }
        __syncthreads();
        // V_j = T * inv(L_jj)^T
#pragma unroll
        for (int a = 0; a < MT; a++)
#pragma unroll
            for (int b = 0; b < NT; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
#pragma unroll 4
        for (int ks = 0; ks < kNB / 4; ks++) {
            const int krow = ks * 4 + (lane & 3);
            double af[MT], bf[NT];
#pragma unroll
            for (int mt = 0; mt < MT; mt++) af[mt] = Ts[krow * LDA + wm0 + mt * 8 + (lane >> 2)];
#pragma unroll
            for (int nt = 0; nt < NT; nt++) bf[nt] = Ls[krow * LDB + wn0 + nt * 8 + (lane >> 2)];
#pragma unroll
            for (int mt = 0; mt < MT; mt++)
#pragma unroll
                for (int nt = 0; nt < NT; nt++) dmma8x8x4(acc[mt][nt][0], acc[mt][nt][1], af[mt], bf[nt]);
        }
#pragma unroll
        for (int mt = 0; mt < MT; mt++) {
            const int row = r0 + wm0 + mt * 8 + (lane >> 2);
#pragma unroll
            for (int nt = 0; nt < NT; nt++) {
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    const int cl = wn0 + nt * 8 + 2 * (lane & 3) + e;
                    if (row < M && cl < w) W[row + (size_t)(c0 + cl) * ldw] = acc[mt][nt][e];
                }
            }
        }
        __threadfence();  // the V_j stores must have reached L2 before the next block's cp.async (L2 path) reads them
        __syncthreads();  // V_j visible to this CTA's next accumulation; Ts / Ls free for reuse
    }
}

// ---- U5s: TRSM for SMALL innovation dimension (k <= 256).  The left-looking kernel above re-reads its own V rows from L2 for every
// column block and waits on each of those round trips (26 % tensor-pipe utilisation, long-scoreboard bound, on the batched
// configuration).  Here the CTA's 32 rows of W are loaded ONCE into shared memory and turned into V in place; the only streamed
// operand is L (off-diagonal blocks, then the inverse of the diagonal block), through a two-stage cp.async ring of 32-deep k-chunks (the same bytes as
// four stages of 16, half the chunk barriers) flattened over the whole (column block, k-chunk) sequence, so the next chunk is always in flight.
constexpr int TS_R = 32, TS_THREADS = 128, TS_LDA = TS_R + 4, TS_LDB = kNB + 4, TS_STAGES = 2, TS_BK = 32, TS_CPB = kNB / TS_BK;  // chunks per 64-column block
inline int trsm_small_smem_bytes(int kmax) { return (((kmax + kNB - 1) / kNB * kNB) * TS_LDA + TS_STAGES * TS_BK * TS_LDB) * (int)sizeof(double); }

__global__ void __launch_bounds__(TS_THREADS, 2) k_trsm_small(DevFilter* Fs, int krows) {
    DevFilter& F = Fs[blockIdx.y];
    const int kk = F.ctl[CTL_K];
    if (kk <= 0) return;
    const int M = F.n + 1;
    const int r0 = blockIdx.x * TS_R;
    if (r0 >= M) return;
    extern __shared__ __align__(16) double tsm2[];
    double* Vs = tsm2;                    // [krows][TS_LDA]  k-major: W rows on entry, V rows on exit
    double* Bs = tsm2 + krows * TS_LDA;   // [stage][TS_BK][TS_LDB]
    double* W = F.W;
    const double* Sm = F.Sm;
    const int ldw = F.ldw, lds = F.lds;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm0 = (warp & 1) * 16, wn0 = (warp >> 1) * 32;  // warp grid 2 x 2, warp tile 16 x 32
    const int nb = (kk + kNB - 1) / kNB;
    const int total = TS_CPB * nb * (nb + 1) / 2;  // sum_j (CPB j + CPB) chunks

    for (int ch = tid; ch < nb * kNB * (TS_R / 2); ch += TS_THREADS) {
        const int kc = ch / (TS_R / 2), r2 = ch % (TS_R / 2);
        const int row = r0 + 2 * r2;
        const bool v = row < M && kc < kk;
        cp_async16(&Vs[kc * TS_LDA + 2 * r2], v ? (W + row + (size_t)kc * ldw) : W, v);
    }
    int lj = 0, lc = 0;  // loader cursor (column block, chunk within it)
    auto load_next = [&](int stage) {
        double* bs = Bs + stage * TS_BK * TS_LDB;
        const int c0 = lj * kNB;
        if (lc < TS_CPB * lj) {  // off-diagonal: Bs[k][col] = L[c0 + col, 16 lc + k]
            const int k0 = lc * TS_BK;
#pragma unroll
            for (int it = 0; it < TS_BK * (kNB / 2) / TS_THREADS; it++) {
                const int ch = tid + it * TS_THREADS;
                const int kc = ch / (kNB / 2), r2 = ch % (kNB / 2);
                const int row = c0 + 2 * r2;
                const bool v = row < kk;
                cp_async16(&bs[kc * TS_LDB + 2 * r2], v ? (Sm + row + (size_t)(k0 + kc) * lds) : Sm, v);
            }
        } else {  // diagonal: Bs[k][col] = inv(L_jj)[col, 16 d + k]
            const int d = lc - TS_CPB * lj;
            const double* Li = F.Linv + (size_t)lj * kNB * kNB + (size_t)d * TS_BK * kNB;
#pragma unroll
            for (int it = 0; it < TS_BK * (kNB / 2) / TS_THREADS; it++) {
                const int ch = tid + it * TS_THREADS;
                const int kc = ch / (kNB / 2), r2 = ch % (kNB / 2);
                cp_async16(&bs[kc * TS_LDB + 2 * r2], Li + 2 * r2 + (size_t)kc * kNB, true);
            }
        }
        if (++lc == TS_CPB * lj + TS_CPB) {
            lc = 0;
            lj++;
        }
    };
#pragma unroll
    for (int s = 0; s < TS_STAGES - 1; s++) {
        if (s < total) load_next(s);
        cp_async_commit();
    }
    double acc[2][4][2];
    int j = 0, c = 0;
    for (int q = 0; q < total; q++) {
        const int c0 = j * kNB;
        if (c == 0 || c == TS_CPB * j) {
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
                for (int b = 0; b < 4; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
        }
        cp_async_wait<TS_STAGES - 2>();
        __syncthreads();
        {
            const int nq = q + TS_STAGES - 1;
            if (nq < total) load_next(nq % TS_STAGES);
            cp_async_commit();
        }
        const bool diag = c >= TS_CPB * j;
        const double* as = Vs + (diag ? (c0 + (c - TS_CPB * j) * TS_BK) : c * TS_BK) * TS_LDA;
        const double* bs = Bs + (q % TS_STAGES) * TS_BK * TS_LDB;
#pragma unroll
        for (int ks = 0; ks < TS_BK / 4; ks++) {
            const int krow = ks * 4 + (lane & 3);
            double af[2], bf[4];
#pragma unroll
            for (int mt = 0; mt < 2; mt++) af[mt] = as[krow * TS_LDA + wm0 + mt * 8 + (lane >> 2)];
#pragma unroll
            for (int nt = 0; nt < 4; nt++) bf[nt] = bs[krow * TS_LDB + wn0 + nt * 8 + (lane >> 2)];
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int nt = 0; nt < 4; nt++) dmma8x8x4(acc[mt][nt][0], acc[mt][nt][1], af[mt], bf[nt]);
        }
        if (!diag && c == TS_CPB * j - 1) {
            // T = W_j - acc, in place (each thread touches only its own elements; the accumulation never reads rows >= c0)
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int nt = 0; nt < 4; nt++)
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int rl = wm0 + mt * 8 + (lane >> 2), cl = wn0 + nt * 8 + 2 * (lane & 3) + e;
                        Vs[(c0 + cl) * TS_LDA + rl] -= acc[mt][nt][e];
                    }
        } else if (diag && c == TS_CPB * j + TS_CPB - 1) {
            // V_j = T inv(L_jj)^T : everybody must be done reading T before it is overwritten
            __syncthreads();
            const int w = min(kNB, kk - c0);
#pragma unroll
            for (int mt = 0; mt < 2; mt++) {
                const int rl = wm0 + mt * 8 + (lane >> 2);
                const int row = r0 + rl;
#pragma unroll
                for (int nt = 0; nt < 4; nt++)
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int cl = wn0 + nt * 8 + 2 * (lane & 3) + e;
                        Vs[(c0 + cl) * TS_LDA + rl] = acc[mt][nt][e];
                        if (row < M && cl < w) W[row + (size_t)(c0 + cl) * ldw] = acc[mt][nt][e];
                    }
            }
        }
        if (++c == TS_CPB * j + TS_CPB) {
            c = 0;
            j++;
        }
    }
    cp_async_wait<0>();
}

// ---- fp64 tensor-core GEMM:  C -= A * B^T  (A: M x K, B: N x K, C: M x N, all column-major) ------------------------------
// DMMA m8n8k4 (mma.sync.aligned.m8n8k4.row.col.f64): tcgen05 has no fp64 kind, so mma.sync DMMA is the fp64 tensor path on
// sm_100a.  3-stage cp.async pipeline, padded smem (+4 doubles per k-row) so that the fragment loads are bank-conflict free.
// Two tile shapes: 128 x 128 (8 warps, warp tile 64 x 32) for large problems, 64 x 64 (4 warps, 32 x 32) when the large tiling
// would leave most SMs idle (the 100-feature configuration).
constexpr int GBK = 16, GSTAGES = 4, GPAD = 4;
template <int BM, int BN>
struct GemmCfg {
    static constexpr int kBM = BM, kBN = BN;
    static constexpr int kWM = 2, kWN = BN / 32;            // warp grid; every warp owns (BM/2) x 32
    static constexpr int kThreads = kWM * kWN * 32;
    static constexpr int kMT = BM / (8 * kWM), kNT = 4;
    static constexpr int kLdA = BM + GPAD, kLdB = BN + GPAD;  // == 8 (mod 32) words per k-row -> conflict-free fragment loads
    static constexpr int kSmemBytes = GSTAGES * GBK * (kLdA + kLdB) * (int)sizeof(double);
    // 128 x 64 tiles with 4 warps: two CTAs are resident per SM, so one CTA's prologue / epilogue / barrier bubbles are
    // covered by the other CTA's DMMA stream (the single 128 x 128 CTA left the tensor pipe ~20 % idle)
    static constexpr int kMinBlocks = (BM == 128 && BN == 64) ? 2 : 1;
};

// Cholesky trailing updates are two-level: inside a 256-wide outer block the panel kernels are left-looking (k_chol_panel); after the
// last panel of an outer block the rest of the matrix gets one K = 256 update (GEMM_CHOL_OUTER).  Same flops as a K = 64 update after
// every panel, but 4x fewer passes over the trailing matrix and DMMA tiles with a 4x longer k-loop.
enum GemmMode { GEMM_SYRK_P = 0, GEMM_CHOL_OUTER = 2, GEMM_TRSM_OUTER = 3 };

struct GemmProb {
    const double* A;
    const double* B;
    double* C;
    int lda, ldb, ldc, M, N, K;
    bool lower, mirror;
};

__device__ __forceinline__ bool gemm_setup(const DevFilter& F, int mode, int step, int ob, GemmProb& g) {
    const int kk = F.ctl[CTL_K];
    if (mode == GEMM_SYRK_P) {
        if (kk <= 0) return false;
        g.A = g.B = F.W;
        g.lda = g.ldb = F.ldw;
        g.C = F.P;
        g.ldc = F.ldp;
        g.M = g.N = F.n + 1;  // row n of W is y = L^-1 nu: row n of V V^T is V y, i.e. the state correction (fused x update)
        g.K = kk;
        g.lower = g.mirror = true;
        return true;
    }
    g.mirror = false;
    if (mode == GEMM_TRSM_OUTER) {  // W[:, o:] -= V_J L[o:, J]^T after the outer block J = step of the TRSM is solved; `ob` 64-blocks wide
        const int wob = kNB * ob;
        const int o = wob * (step + 1);
        if (kk <= o) return false;
        g.A = F.W + (size_t)(o - wob) * F.ldw;
        g.lda = F.ldw;
        g.B = F.Sm + o + (size_t)(o - wob) * F.lds;
        g.ldb = F.lds;
        g.C = F.W + (size_t)o * F.ldw;
        g.ldc = F.ldw;
        g.M = F.n + 1;
        g.N = kk - o;
        g.K = wob;
        g.lower = false;
        return true;
    }
    g.lda = g.ldb = g.ldc = F.lds;
    const int o = kNB * kOB * (step + 1);  // step = outer block index
    if (kk <= o) return false;
    g.A = g.B = F.Sm + o + (size_t)(o - kNB * kOB) * F.lds;
    g.C = F.Sm + o + (size_t)o * F.lds;
    g.M = g.N = kk - o;
    g.K = kNB * kOB;
    g.lower = true;
    return true;
}

#ifdef RSLAM_PHASE_CLOCKS
// Per-CTA timeline of filter 0's last syrk_P launch (record 0) and of its first trsm_outer launch (record 1), read by
// rslam_debug_gemm_stamps: globaltimer at start and end, clock64 at start, after the first chunk has landed, after the main loop and
// at the end, %smid, and the number of k-chunks.
constexpr int kGemmStampCtas = 16384, kGemmStampFields = 8;
__device__ unsigned long long g_gemm_stamps[2][kGemmStampCtas][kGemmStampFields];
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ unsigned smid() {
    unsigned s;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(s));
    return s;
}
#define GEMM_STAMP(field, value) do { if (stamp__) stamp__[field] = (value); } while (0)
#else
#define GEMM_STAMP(field, value)
#endif

// In SYRK mode the product is taken over the n+1 rows of W: entries (n, c) of V V^T are (V y)[c] and update the state,
//   x_k_k[c] = x0[c] + (V y)[c]   (x0 = x_k_km1 for the low-innovation update, x_k_k for the high-innovation one),
// everything else is the covariance downdate P -= V V^T.
template <int BM, int BN>
__global__ void __launch_bounds__(GemmCfg<BM, BN>::kThreads, GemmCfg<BM, BN>::kMinBlocks) k_gemm_dmma(DevFilter* Fs, int mode, int step) {
    using Cfg = GemmCfg<BM, BN>;
    constexpr int LDA = Cfg::kLdA, LDB = Cfg::kLdB, MT = Cfg::kMT, NT = Cfg::kNT, THREADS = Cfg::kThreads;
    const DevFilter& F = Fs[blockIdx.z];
    GemmProb g;
    if (!gemm_setup(F, mode & 0xff, step, mode >> 16, g)) return;
    int ti, tj;
    const int tm = (g.M + BM - 1) / BM, tn = (g.N + BN - 1) / BN;
    if (g.lower) {
        // tile row i needs column tiles 0 .. min(R*(i+1), tn) - 1 with R = BM / BN; rows are enumerated back to back
        constexpr int RT = BM / BN;
        const long long t = blockIdx.x;
        int i = (int)((sqrt(1.0 + 8.0 * (double)t / RT) - 1.0) * 0.5);
        if (i < 0) i = 0;
        while (i > 0 && (long long)RT * i * (i + 1) / 2 > t) i--;
        while ((long long)RT * (i + 1) * (i + 2) / 2 <= t) i++;
        if (i >= tm) return;
        ti = i;
        tj = (int)(t - (long long)RT * i * (i + 1) / 2);
        if (tj >= tn) return;
    } else {
        if ((long long)blockIdx.x >= (long long)tm * tn) return;
        ti = blockIdx.x % tm;
        tj = blockIdx.x / tm;
    }
#ifdef RSLAM_PHASE_CLOCKS
    const int rec__ = (mode & 0xff) == GEMM_SYRK_P ? 0 : ((mode & 0xff) == GEMM_TRSM_OUTER && step == 0 ? 1 : -1);
    unsigned long long* stamp__ = rec__ >= 0 && blockIdx.z == 0 && blockIdx.x < kGemmStampCtas && threadIdx.x == 0 ? g_gemm_stamps[rec__][blockIdx.x] : nullptr;
    GEMM_STAMP(0, globaltimer_ns());
    GEMM_STAMP(2, clock64());
    GEMM_STAMP(6, smid());
    GEMM_STAMP(7, (g.K + GBK - 1) / GBK);
#endif
    extern __shared__ __align__(16) double gsm[];
    double* As = gsm;                          // [stage][GBK][LDA]
    double* Bs = gsm + GSTAGES * GBK * LDA;    // [stage][GBK][LDB]
    const int m0 = ti * BM, n0 = tj * BN;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm0 = (warp % Cfg::kWM) * (MT * 8), wn0 = (warp / Cfg::kWM) * (NT * 8);
    const int nkt = (g.K + GBK - 1) / GBK, nfull = g.K / GBK;  // k-chunks; those with all GBK columns inside K
    constexpr int A_CHUNKS = GBK * (BM / 2), B_CHUNKS = GBK * (BN / 2);
    constexpr int A_PER = A_CHUNKS / THREADS, B_PER = B_CHUNKS / THREADS, KSTEPS = GBK / 4, CP_PER_KS = (A_PER + B_PER) / KSTEPS;
    static_assert(A_CHUNKS % THREADS == 0 && B_CHUNKS % THREADS == 0, "tile loads must divide evenly");
    static_assert(THREADS % (BM / 2) == 0 && THREADS % (BN / 2) == 0, "a thread copies the same rows in every k-row it serves");
    static_assert((A_PER + B_PER) % KSTEPS == 0, "copies spread evenly over the k-steps of a chunk");
    constexpr int A_KSTRIDE = THREADS / (BM / 2), B_KSTRIDE = THREADS / (BN / 2);  // k-rows between a thread's successive copies

    // Copy slots: a thread's 16-byte copies of a chunk all read the same two rows of A (of B), in k-rows kc0, kc0 + KSTRIDE, ...
    // The row test and the source pointers are set up once per tile; per chunk the pointers advance by GBK columns.  A row past
    // M (N) is zero-filled from a pointer kept on row 0, which stays inside the operand on every chunk that is not the last.
    const int a_kc = tid / (BM / 2), a_r = 2 * (tid % (BM / 2));
    const int b_kc = tid / (BN / 2), b_r = 2 * (tid % (BN / 2));
    const bool a_ok = m0 + a_r < g.M, b_ok = n0 + b_r < g.N;
    const double* pa = g.A + (a_ok ? m0 + a_r : 0) + (size_t)a_kc * g.lda;  // the next chunk to load
    const double* pb = g.B + (b_ok ? n0 + b_r : 0) + (size_t)b_kc * g.ldb;
    const size_t a_step = (size_t)A_KSTRIDE * g.lda, b_step = (size_t)B_KSTRIDE * g.ldb;
    const size_t a_chunk = (size_t)GBK * g.lda, b_chunk = (size_t)GBK * g.ldb;
    double* const a_dst = As + a_kc * LDA + a_r;
    double* const b_dst = Bs + b_kc * LDB + b_r;
    auto copy = [&](int stage, int i) {  // copy i of this thread for the chunk at pa / pb, a full chunk
        if (i < A_PER)
            cp_async16(a_dst + (stage * GBK + i * A_KSTRIDE) * LDA, pa + i * a_step, a_ok);
        else
            cp_async16(b_dst + (stage * GBK + (i - A_PER) * B_KSTRIDE) * LDB, pb + (i - A_PER) * b_step, b_ok);
    };
    auto copy_last = [&](int stage, int kleft) {  // the chunk that ends past K: columns >= K zero-filled, like rows >= M
#pragma unroll
        for (int i = 0; i < A_PER; i++) {
            const bool v = a_ok && a_kc + i * A_KSTRIDE < kleft;
            cp_async16(a_dst + (stage * GBK + i * A_KSTRIDE) * LDA, v ? pa + i * a_step : g.A, v);
        }
#pragma unroll
        for (int i = 0; i < B_PER; i++) {
            const bool v = b_ok && b_kc + i * B_KSTRIDE < kleft;
            cp_async16(b_dst + (stage * GBK + i * B_KSTRIDE) * LDB, v ? pb + i * b_step : g.B, v);
        }
    };
    auto load_stage = [&](int stage, int kt) {  // whole chunk kt at once (prologue, and the last chunk when it ends past K)
        if (kt < nfull) {
#pragma unroll
            for (int i = 0; i < A_PER + B_PER; i++) copy(stage, i);
        } else if (kt < nkt) {
            copy_last(stage, g.K - kt * GBK);
        }
        pa += a_chunk;
        pb += b_chunk;
    };

    double acc[MT][NT][2];
#pragma unroll
    for (int a = 0; a < MT; a++)
#pragma unroll
        for (int b = 0; b < NT; b++) acc[a][b][0] = acc[a][b][1] = 0.0;

    // One chunk of DMMA work.  The fragments of k-step ks + 1 are loaded while the DMMAs of k-step ks issue, and `copies(ks)` issues
    // that k-step's share of the next stage's copies between them, so neither the copy issue nor the first fragment loads of a
    // k-step sit in front of the tensor pipe as one block.  Every accumulator still takes its DMMAs in ascending k.
    const int frag_a = (lane & 3) * LDA + wm0 + (lane >> 2), frag_b = (lane & 3) * LDB + wn0 + (lane >> 2);
    auto compute = [&](const double* as, const double* bs, auto&& copies) {
        double af[2][MT], bf[2][NT];
#pragma unroll
        for (int mt = 0; mt < MT; mt++) af[0][mt] = as[frag_a + mt * 8];
#pragma unroll
        for (int nt = 0; nt < NT; nt++) bf[0][nt] = bs[frag_b + nt * 8];
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ks++) {
            const int cur = ks & 1;
            if (ks + 1 < KSTEPS) {
#pragma unroll
                for (int mt = 0; mt < MT; mt++) af[cur ^ 1][mt] = as[frag_a + (ks + 1) * 4 * LDA + mt * 8];
#pragma unroll
                for (int nt = 0; nt < NT; nt++) bf[cur ^ 1][nt] = bs[frag_b + (ks + 1) * 4 * LDB + nt * 8];
            }
            copies(ks);
#pragma unroll
            for (int mt = 0; mt < MT; mt++)
#pragma unroll
                for (int nt = 0; nt < NT; nt++) dmma8x8x4(acc[mt][nt][0], acc[mt][nt][1], af[cur][mt], bf[cur][nt]);
        }
    };

#pragma unroll
    for (int s = 0; s < GSTAGES - 1; s++) {
        load_stage(s, s);
        cp_async_commit();
    }
    for (int kt = 0; kt < nkt; kt++) {
        cp_async_wait<GSTAGES - 2>();
        __syncthreads();
#ifdef RSLAM_PHASE_CLOCKS
        if (kt == 0) GEMM_STAMP(3, clock64());
#endif
        const int nk = kt + GSTAGES - 1, ns = nk % GSTAGES;  // the chunk loaded during this one, into the stage read last time
        const double* as = As + (kt % GSTAGES) * GBK * LDA;
        const double* bs = Bs + (kt % GSTAGES) * GBK * LDB;
        if (nk < nfull) {
            compute(as, bs, [&](int ks) {
#pragma unroll
                for (int c = 0; c < CP_PER_KS; c++) copy(ns, ks * CP_PER_KS + c);
            });
            pa += a_chunk;
            pb += b_chunk;
        } else {
            load_stage(ns, nk);
            compute(as, bs, [](int) {});
        }
        cp_async_commit();
    }
    cp_async_wait<0>();
    GEMM_STAMP(4, clock64());
    const bool syrk = (mode & 0xff) == GEMM_SYRK_P;
    const int xrow = syrk ? F.n : -1;
    const double* x0 = ((mode >> 8) & 0xff) ? F.x_kk : F.x_km1;
    // epilogue: C -= acc ; lower: only row >= col ; mirror: also store the transposed element.  The C entries of two m8 tile rows (16
    // per thread) are fetched as one batch before any of them is stored: issued one by one behind the stores of the previous entry
    // (the compiler cannot move a load of C above a store to C) the 64 dependent round trips cost ~30 us per tile -- as much as the
    // whole k-loop of a K = 256 update (ncu / event timing: the K = 256 GEMMs ran at 45 % of the rate of the K = 3300 SYRK).
    constexpr int EB = 2;
    static_assert(MT % EB == 0, "epilogue batches");
#pragma unroll
    for (int mt0 = 0; mt0 < MT; mt0 += EB) {
        double cv[EB][NT][2];
#pragma unroll
        for (int u = 0; u < EB; u++) {
            const int row = m0 + wm0 + (mt0 + u) * 8 + (lane >> 2);
#pragma unroll
            for (int nt = 0; nt < NT; nt++)
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    const int cc = n0 + wn0 + nt * 8 + 2 * (lane & 3) + e;
                    const bool ok = row < g.M && cc < g.N && !(g.lower && row < cc) && row != xrow;
                    cv[u][nt][e] = ok ? g.C[row + (size_t)cc * g.ldc] : 0.0;
                }
        }
#pragma unroll
        for (int u = 0; u < EB; u++) {
            const int row = m0 + wm0 + (mt0 + u) * 8 + (lane >> 2);
            if (row >= g.M) continue;
#pragma unroll
            for (int nt = 0; nt < NT; nt++)
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    const int cc = n0 + wn0 + nt * 8 + 2 * (lane & 3) + e;
                    if (cc >= g.N) continue;
                    if (g.lower && row < cc) continue;
                    if (row == xrow) {
                        if (cc < xrow) F.x_kk[cc] = x0[cc] + acc[mt0 + u][nt][e];
                        continue;
                    }
                    const double v = cv[u][nt][e] - acc[mt0 + u][nt][e];
                    g.C[row + (size_t)cc * g.ldc] = v;
                    if (g.mirror && row != cc) g.C[cc + (size_t)row * g.ldc] = v;
                }
        }
    }
    GEMM_STAMP(5, clock64());
    GEMM_STAMP(1, globaltimer_ns());
}
#undef GEMM_STAMP

// ---- U6s: covariance downdate for SMALL innovation dimension (k <= 256: the 100-feature and batched-filter configurations) -----
// With K this small a 64 x 64 tile is a handful of k-steps, so the one-tile-per-CTA GEMM above spends most of its life in the
// prologue (first loads) and the epilogue (read-modify-write of the P tile from HBM) -- 35 % tensor-pipe utilisation on the
// 4096-filter batch.  Here a CTA owns a SEGMENT of one 64-row tile row of P:
//   * its 64 x K block of V (the A operand) is loaded once and stays in shared memory for all tiles of the segment,
//   * the tiles of the segment are dealt alternately to TWO independent warp groups (4 warps each, one warp per SM sub-partition,
//     warp tile 32 x 32); each group streams its B operand through its own two-stage cp.async ring of 32-deep k-chunks, FLATTENED over
//     (tile, k-chunk) so that the pipeline never drains, and synchronises on its own named barrier -- the groups drift apart, and
//     one group's barrier / fragment-load bubbles are covered by the other group's DMMA stream (what two co-resident CTAs would
//     do, without paying for the resident A twice),
//   * the P tile is fetched into registers at the first k-chunk of its tile and consumed in the epilogue, which hides its HBM
//     latency behind the tile's DMMA work.
// seg_len = 1 gives one CTA per tile (single filter: maximum parallelism, minimum latency); seg_len = tiles-per-row gives one CTA
// per tile row (large batches: minimum traffic).  Same row-n convention as k_gemm_dmma: row n of V V^T is the state correction.
#ifndef RSLAM_SR_STAGES
#define RSLAM_SR_STAGES 2
#endif
constexpr int SR_BM = 64, SR_THREADS = 256, SR_LD = SR_BM + 4, SR_STAGES = RSLAM_SR_STAGES, SR_BK = 32, SR_KMAX = 256;
inline int syrk_rows_smem_bytes(int kmax) { return (((kmax + SR_BK - 1) / SR_BK * SR_BK) * SR_LD + 2 * SR_STAGES * SR_BK * SR_LD) * (int)sizeof(double); }

__device__ __forceinline__ void group_barrier(int g) { asm volatile("bar.sync %0, 128;\n" ::"r"(1 + g) : "memory"); }

__global__ void __launch_bounds__(SR_THREADS, 1) k_syrk_rows(DevFilter* Fs, int which, int seg_len, int kpad) {
    const DevFilter& F = Fs[blockIdx.z];
    const int kk = F.ctl[CTL_K];
    if (kk <= 0) return;
    const int n = F.n, M = n + 1;
    const int tm = (M + SR_BM - 1) / SR_BM;
    // blockIdx.x -> (tile row ti, segment): long rows first
    int t = blockIdx.x, ti = tm - 1;
    for (;; ti--) {
        if (ti < 0) return;
        const int ns = (ti + seg_len) / seg_len;  // ceil((ti + 1) / seg_len)
        if (t < ns) break;
        t -= ns;
    }
    const int tj0 = t * seg_len, tj1 = min(ti + 1, tj0 + seg_len);
    extern __shared__ __align__(16) double rsm[];
    const int tid = threadIdx.x, grp = tid >> 7, gt = tid & 127, lane = tid & 31, gw = (tid >> 5) & 3;
    double* As = rsm;                                                         // [kpad][SR_LD]   the CTA's 64 rows of V, k-major
    double* Bs = rsm + kpad * SR_LD + grp * (SR_STAGES * SR_BK * SR_LD);      // this group's ring [stage][SR_BK][SR_LD]
    const double* W = F.W;
    const int ldw = F.ldw, ldp = F.ldp;
    double* P = F.P;
    const int wm0 = (gw & 1) * 32, wn0 = (gw >> 1) * 32;  // warp grid 2 x 2 inside the group, warp tile 32 x 32
    const int m0 = ti * SR_BM;
    const int nkt = (kk + SR_BK - 1) / SR_BK;
    // the segment's tiles are dealt alternately to the two groups; an odd last tile is SPLIT between them by columns (group g takes columns
    // 32 g .. 32 g + 31 with 32 x 16 warp tiles) instead of leaving one group idle for a whole tile
    const int nfull = (tj1 - tj0) >> 1, ntile = nfull + ((tj1 - tj0) & 1);
    auto tile_col = [&](int tile) { return tile < nfull ? tj0 + grp + 2 * tile : tj1 - 1; };
    const int total = ntile * nkt;
    const double* x0 = which ? F.x_kk : F.x_km1;

    // A: all of K, once, by the whole CTA
    for (int ch = tid; ch < nkt * SR_BK * (SR_BM / 2); ch += SR_THREADS) {
        const int kc = ch / (SR_BM / 2), r2 = ch % (SR_BM / 2);
        const int row = m0 + 2 * r2;
        const bool v = row < M && kc < kk;
        cp_async16(&As[kc * SR_LD + 2 * r2], v ? (W + row + (size_t)kc * ldw) : W, v);
    }
    auto load_B = [&](int q) {
        const int tile = q / nkt, kt = q - tile * nkt;
        const int n0 = tile_col(tile) * SR_BM, k0 = kt * SR_BK;
        double* bs = Bs + (q % SR_STAGES) * SR_BK * SR_LD;
#pragma unroll
        for (int it = 0; it < SR_BK * (SR_BM / 2) / 128; it++) {
            const int ch = gt + it * 128;
            const int kc = ch / (SR_BM / 2), r2 = ch % (SR_BM / 2);
            const int row = n0 + 2 * r2, col = k0 + kc;
            const bool v = row < M && col < kk;
            cp_async16(&bs[kc * SR_LD + 2 * r2], v ? (W + row + (size_t)col * ldw) : W, v);
        }
    };
#pragma unroll
    for (int s = 0; s < SR_STAGES - 1; s++) {
        if (s < total) load_B(s);
        cp_async_commit();
    }
    // the resident A block was loaded by both groups: one CTA-wide barrier, after that the groups run on their own
    cp_async_wait<SR_STAGES - 2>();
    __syncthreads();
    double acc[4][4][2], cpre[4][4][2];
    for (int q = 0; q < total; q++) {
        const int tile = q / nkt, kt = q - tile * nkt;
        const int n0 = tile_col(tile) * SR_BM;
        const bool half = tile >= nfull;
        const int wn = half ? grp * 32 + (gw >> 1) * 16 : wn0;  // first column of this warp's block inside the tile
        const int ntl = half ? 2 : 4;                          // m8n8 tiles across
        if (kt == 0) {
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    acc[a][b][0] = acc[a][b][1] = 0.0;
                    const int row = m0 + wm0 + a * 8 + (lane >> 2);
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int cc = n0 + wn + b * 8 + 2 * (lane & 3) + e;
                        cpre[a][b][e] = (b < ntl && row < n && cc <= row) ? P[row + (size_t)cc * ldp] : 0.0;
                    }
                }
        }
        if (q > 0) {
            cp_async_wait<SR_STAGES - 2>();
            group_barrier(grp);
        }
        {
            const int nq = q + SR_STAGES - 1;
            if (nq < total) load_B(nq);
            cp_async_commit();
        }
        const double* as = As + kt * SR_BK * SR_LD;
        const double* bs = Bs + (q % SR_STAGES) * SR_BK * SR_LD;
        // a warp whose 32 x 32 block lies entirely above the diagonal of a diagonal tile, or entirely below the last state row, only
        // produces entries that are never stored: it keeps the pipeline protocol (loads, barriers) and skips the arithmetic, which leaves
        // its scheduler's tensor pipe to the other warp group.  (Predicating single m8 tiles inside the unrolled DMMA stream was tried
        // and LOST 6 %: the predicate breaks the back-to-back issue of the 16 DMMAs.)
        const bool dead = (n0 == m0 && wn > wm0 + 31) || (m0 + wm0 >= M);
        if (!dead && !half) {
#pragma unroll
            for (int ks = 0; ks < SR_BK / 4; ks++) {
                const int krow = ks * 4 + (lane & 3);
                double af[4], bf[4];
#pragma unroll
                for (int mt = 0; mt < 4; mt++) af[mt] = as[krow * SR_LD + wm0 + mt * 8 + (lane >> 2)];
#pragma unroll
                for (int nt = 0; nt < 4; nt++) bf[nt] = bs[krow * SR_LD + wn0 + nt * 8 + (lane >> 2)];
#pragma unroll
                for (int mt = 0; mt < 4; mt++)
#pragma unroll
                    for (int nt = 0; nt < 4; nt++) dmma8x8x4(acc[mt][nt][0], acc[mt][nt][1], af[mt], bf[nt]);
            }
        } else if (!dead) {
#pragma unroll
            for (int ks = 0; ks < SR_BK / 4; ks++) {
                const int krow = ks * 4 + (lane & 3);
                double af[4], bf[2];
#pragma unroll
                for (int mt = 0; mt < 4; mt++) af[mt] = as[krow * SR_LD + wm0 + mt * 8 + (lane >> 2)];
#pragma unroll
                for (int nt = 0; nt < 2; nt++) bf[nt] = bs[krow * SR_LD + wn + nt * 8 + (lane >> 2)];
#pragma unroll
                for (int mt = 0; mt < 4; mt++)
#pragma unroll
                    for (int nt = 0; nt < 2; nt++) dmma8x8x4(acc[mt][nt][0], acc[mt][nt][1], af[mt], bf[nt]);
            }
        }
        if (kt == nkt - 1) {  // epilogue of this tile: P -= acc (lower part, mirrored), row n -> state correction
#pragma unroll
            for (int mt = 0; mt < 4; mt++) {
                const int row = m0 + wm0 + mt * 8 + (lane >> 2);
                if (row >= M) continue;
#pragma unroll
                for (int nt = 0; nt < 4; nt++)
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int cc = n0 + wn + nt * 8 + 2 * (lane & 3) + e;
                        if (nt >= ntl || cc > row || cc >= n) continue;
                        if (row == n) {
                            F.x_kk[cc] = x0[cc] + acc[mt][nt][e];
                            continue;
                        }
                        const double v = cpre[mt][nt][e] - acc[mt][nt][e];
                        P[row + (size_t)cc * ldp] = v;
                        if (row != cc) P[cc + (size_t)row * ldp] = v;
                    }
            }
        }
    }
    cp_async_wait<0>();
}

// ---- U7: x+ = x + V y is fused into the SYRK kernel (row n of V V^T); the empty-set copy of the prior happens in gather_inliers ----

// ---- U9: quaternion normalisation and its Jacobian applied to P (src/ExtendKF.cpp:611-634).  One CTA per filter. -----------
// CTA-collective, any block size (every thread of the CTA must call it)
__device__ __forceinline__ void upd_jnorm_cta(DevFilter& F, const ParDev& par) {
    if (F.ctl[CTL_K] <= 0) return;  // no measurements: x_k_k = x, p_k_k = P untouched (:635-638); uniform over the CTA
    __shared__ double sJ[16];
    __shared__ double sB[16], sT[16];
    const int ld = F.ldp;
    double* P = F.P;
    const double r = F.x_kk[3], x = F.x_kk[4], y = F.x_kk[5], z = F.x_kk[6];
    // rows 3..6 of the first 3 * blockDim columns are fetched now (they do not depend on Jn): their latency hides behind the serial part
    double v0[3][4];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const int c = threadIdx.x + (int)blockDim.x * k;
#pragma unroll
        for (int l = 0; l < 4; l++) v0[k][l] = (c < F.n && !(c >= 3 && c < 7)) ? P[(3 + l) + (size_t)c * ld] : 0.0;
    }
    __syncthreads();  // everybody has read the un-normalised quaternion
    if (threadIdx.x == 0) {
        const double s = r * r + x * x + y * y + z * z;
        const double scale = (par.quirks & RSLAM_Q4_JNORM_INT_EXPONENT) ? 1.0 / s : 1.0 / (s * sqrt(s));
        const double tv[16] = {x * x + y * y + z * z, -r * x, -r * y, -r * z, -x * r, r * r + y * y + z * z, -x * y, -x * z,
                               -y * r, -y * x, r * r + x * x + z * z, -y * z, -z * r, -z * x, -z * y, r * r + x * x + y * y};
        for (int e = 0; e < 16; e++) sJ[e] = scale * tv[e];
        const double nrm = sqrt(s);
        F.x_kk[3] = r / nrm;
        F.x_kk[4] = x / nrm;
        F.x_kk[5] = y / nrm;
        F.x_kk[6] = z / nrm;
    }
    if (threadIdx.x < 16) sB[threadIdx.x] = P[(3 + threadIdx.x / 4) + (size_t)(3 + threadIdx.x % 4) * ld];
    __syncthreads();
    if (threadIdx.x < 16) {  // (Jn * B)
        const int i = threadIdx.x / 4, j = threadIdx.x % 4;
        double s = 0;
        for (int l = 0; l < 4; l++) s += sJ[i * 4 + l] * sB[l * 4 + j];
        sT[threadIdx.x] = s;
    }
    __syncthreads();
    if (threadIdx.x < 16) {  // (Jn * B) * Jn^T
        const int i = threadIdx.x / 4, j = threadIdx.x % 4;
        double s = 0;
        for (int l = 0; l < 4; l++) s += sT[i * 4 + l] * sJ[j * 4 + l];
        if (i >= j) {  // lower triangle is authoritative; mirror so that P stays exactly symmetric
            P[(3 + i) + (size_t)(3 + j) * ld] = s;
            P[(3 + j) + (size_t)(3 + i) * ld] = s;
        }
    }
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const int c = threadIdx.x + (int)blockDim.x * k;
        if (c >= F.n || (c >= 3 && c < 7)) continue;
        double o[4];
#pragma unroll
        for (int i = 0; i < 4; i++) o[i] = sJ[i * 4] * v0[k][0] + sJ[i * 4 + 1] * v0[k][1] + sJ[i * 4 + 2] * v0[k][2] + sJ[i * 4 + 3] * v0[k][3];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            P[(3 + i) + (size_t)c * ld] = o[i];
            P[c + (size_t)(3 + i) * ld] = o[i];
        }
    }
    for (int c = threadIdx.x + 3 * (int)blockDim.x; c < F.n; c += blockDim.x) {
        double v[4], o[4];
#pragma unroll
        for (int l = 0; l < 4; l++) v[l] = P[(3 + l) + (size_t)c * ld];
#pragma unroll
        for (int i = 0; i < 4; i++) o[i] = sJ[i * 4] * v[0] + sJ[i * 4 + 1] * v[1] + sJ[i * 4 + 2] * v[2] + sJ[i * 4 + 3] * v[3];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            P[(3 + i) + (size_t)c * ld] = o[i];
            P[c + (size_t)(3 + i) * ld] = o[i];
        }
    }
}
__global__ void __launch_bounds__(256) k_upd_jnorm(DevFilter* Fs, ParDev par) { upd_jnorm_cta(Fs[blockIdx.y], par); }

// The same for large maps: one CTA over 12013 columns of 4 strided rows is a 125 us latency chain (N = 2000); here CTA b takes columns
// [256 b, 256 b + 256), every CTA forms Jn from the un-normalised quaternion, and the CTA that finishes LAST (a counter in the control
// block) writes the normalised quaternion back -- nobody can read it after that.  CTA 0 also does the 4 x 4 block.
__global__ void __launch_bounds__(256) k_upd_jnorm_wide(DevFilter* Fs, ParDev par) {
    DevFilter& F = Fs[blockIdx.y];
    if (F.ctl[CTL_K] <= 0) return;
    __shared__ double sJ[16], sB[16], sT[16];
    __shared__ int s_last;
    const int ld = F.ldp;
    double* P = F.P;
    const double r = F.x_kk[3], x = F.x_kk[4], y = F.x_kk[5], z = F.x_kk[6];
    const double s = r * r + x * x + y * y + z * z;
    const int c = blockIdx.x * 256 + threadIdx.x;
    const bool mine = c < F.n && !(c >= 3 && c < 7);
    double v[4];
#pragma unroll
    for (int l = 0; l < 4; l++) v[l] = mine ? P[(3 + l) + (size_t)c * ld] : 0.0;
    if (threadIdx.x == 0) {
        const double scale = (par.quirks & RSLAM_Q4_JNORM_INT_EXPONENT) ? 1.0 / s : 1.0 / (s * sqrt(s));
        const double tv[16] = {x * x + y * y + z * z, -r * x, -r * y, -r * z, -x * r, r * r + y * y + z * z, -x * y, -x * z,
                               -y * r, -y * x, r * r + x * x + z * z, -y * z, -z * r, -z * x, -z * y, r * r + x * x + y * y};
        for (int e = 0; e < 16; e++) sJ[e] = scale * tv[e];
    }
    if (blockIdx.x == 0 && threadIdx.x < 16) sB[threadIdx.x] = P[(3 + threadIdx.x / 4) + (size_t)(3 + threadIdx.x % 4) * ld];
    __syncthreads();
    if (blockIdx.x == 0) {
        if (threadIdx.x < 16) {  // (Jn * B)
            const int i = threadIdx.x / 4, j = threadIdx.x % 4;
            double t = 0;
            for (int l = 0; l < 4; l++) t += sJ[i * 4 + l] * sB[l * 4 + j];
            sT[threadIdx.x] = t;
        }
        __syncthreads();
        if (threadIdx.x < 16) {  // (Jn * B) * Jn^T
            const int i = threadIdx.x / 4, j = threadIdx.x % 4;
            double t = 0;
            for (int l = 0; l < 4; l++) t += sT[i * 4 + l] * sJ[j * 4 + l];
            if (i >= j) {
                P[(3 + i) + (size_t)(3 + j) * ld] = t;
                P[(3 + j) + (size_t)(3 + i) * ld] = t;
            }
        }
    }
    if (mine) {
        double o[4];
#pragma unroll
        for (int i = 0; i < 4; i++) o[i] = sJ[i * 4] * v[0] + sJ[i * 4 + 1] * v[1] + sJ[i * 4 + 2] * v[2] + sJ[i * 4 + 3] * v[3];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            P[(3 + i) + (size_t)c * ld] = o[i];
            P[c + (size_t)(3 + i) * ld] = o[i];
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(&F.ctl[CTL_JN_DONE], 1) == (int)gridDim.x - 1;
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {  // every CTA has read the un-normalised quaternion
        const double nrm = sqrt(s);
        F.x_kk[3] = r / nrm;
        F.x_kk[4] = x / nrm;
        F.x_kk[5] = y / nrm;
        F.x_kk[6] = z / nrm;
        F.ctl[CTL_JN_DONE] = 0;
    }
}


}  // namespace rslam
