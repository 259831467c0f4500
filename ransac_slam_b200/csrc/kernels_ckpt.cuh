// kernels_ckpt.cuh -- checkpoint / resume of whole filters (rslam_checkpoint_save / rslam_checkpoint_load, sm_100a).
//
// A snapshot (layout: include/rslam.h) holds, per filter, a record block (x_k_k, x_k_km1 and every per-feature array, each
// 16-byte aligned) followed by the lower triangle of P in LAPACK packed storage (UPLO = 'L': column j holds rows j..n-1).  The
// host cuts the stream of blocks into chunks (a filter's records, or a range of whole 64-column tile columns of its triangle)
// and builds per chunk a flat list of work items, so one launch of each kernel serves every filter of the chunk whatever B is
// and heterogeneous n costs no empty CTAs.
#pragma once
#include "common.cuh"

namespace rslam {

constexpr int kCkTile = 64;   // covariance tile edge
constexpr int kCkSegs = 17;   // record segments: 0 = head {n, N}, 1..16 the arrays below

// one 64 x 64 lower tile (I, J), I >= J, of filter `slot`; pbase: element offset of the filter's packed triangle from the chunk
// base (negative when the chunk starts inside the triangle)
struct CkptTile {
    int slot, n, I, J;
    long long pbase;
};
// the record block of filter `slot` (n, N of the snapshot) at byte offset `off` from the chunk base
struct CkptRec {
    int slot, n, N, pad;
    long long off;
};

__host__ __device__ inline size_t ck_al16(size_t v) { return (v + 15) & ~(size_t)15; }
// first element of packed column j of an n x n lower triangle
__host__ __device__ inline long long ck_colstart(long long j, long long n) { return j * n - j * (j - 1) / 2; }

// bytes of record segment k for a filter with state dimension n and N features (k >= 1)
__host__ __device__ inline size_t ck_seg_bytes(int k, long long n, long long N) {
    switch (k) {
        case 1: case 2: return 8 * n;                    // x_k_k, x_k_km1
        case 3: case 4: return 4 * N;                    // times_predicted, times_measured
        case 5: case 6: case 7: case 8: return N;        // has_h, ic, li, hi
        case 9: case 11: return 16 * N;                  // h, z (2 per feature)
        case 10: return 32 * N;                          // S (2 x 2)
        case 12: return 112 * N;                         // Hc (2 x 7)
        case 13: return 96 * N;                          // Hf (2 x 6)
        case 14: return 4 * (size_t)kPatchPix * N;       // predicted patch (float)
        case 15: return 1681 * N;                        // patch_init (41 x 41 u8)
        default: return 112 * N;                         // 16: init_pose (14 doubles)
    }
}
// byte offset of segment k inside the record block
__host__ __device__ inline size_t ck_seg_off(int k, long long n, long long N) {
    size_t o = 16;
    for (int s = 1; s < k; s++) o += ck_al16(ck_seg_bytes(s, n, N));
    return o;
}
__host__ __device__ inline size_t ck_rec_bytes(long long n, long long N) { return ck_seg_off(kCkSegs, n, N); }
__host__ __device__ inline size_t ck_tri_bytes(long long n) { return ck_al16(8 * (size_t)(n * (n + 1) / 2)); }

__device__ __forceinline__ unsigned char* ck_seg_ptr(const DevFilter& F, int k) {
    switch (k) {
        case 1: return (unsigned char*)F.x_kk;
        case 2: return (unsigned char*)F.x_km1;
        case 3: return (unsigned char*)F.times_predicted;
        case 4: return (unsigned char*)F.times_measured;
        case 5: return F.has_h;
        case 6: return F.ic;
        case 7: return F.li;
        case 8: return F.hi;
        case 9: return (unsigned char*)F.h;
        case 10: return (unsigned char*)F.S;
        case 11: return (unsigned char*)F.z;
        case 12: return (unsigned char*)F.Hc;
        case 13: return (unsigned char*)F.Hf;
        case 14: return (unsigned char*)F.patch;
        case 15: return F.patch_init;
        default: return (unsigned char*)F.init_pose;
    }
}

// dst[0, len) = src[0, len), in the widest word both pointers allow (the per-slot arrays of a handle are only as aligned as
// their element size times the slot index)
template <typename W>
__device__ __forceinline__ void ck_copy_w(unsigned char* dst, const unsigned char* src, size_t len) {
    const size_t nw = len / sizeof(W);
    for (size_t e = threadIdx.x; e < nw; e += blockDim.x) ((W*)dst)[e] = ((const W*)src)[e];
    for (size_t e = nw * sizeof(W) + threadIdx.x; e < len; e += blockDim.x) dst[e] = src[e];
}
__device__ __forceinline__ void ck_copy(unsigned char* dst, const unsigned char* src, size_t len) {
    const uintptr_t a = (uintptr_t)dst | (uintptr_t)src;
    if ((a & 15) == 0)
        ck_copy_w<uint4>(dst, src, len);
    else if ((a & 7) == 0)
        ck_copy_w<unsigned long long>(dst, src, len);
    else if ((a & 3) == 0)
        ck_copy_w<unsigned>(dst, src, len);
    else
        ck_copy_w<unsigned char>(dst, src, len);
}
__device__ __forceinline__ void ck_zero(unsigned char* p, size_t len) {
    for (size_t e = threadIdx.x; e < len; e += blockDim.x) p[e] = 0;
}

// grid (records in the chunk, kCkSegs): CTA (r, k) writes segment k of record r and its zero padding
__global__ void __launch_bounds__(256) k_ckpt_records_pack(const DevFilter* __restrict__ Fs, const CkptRec* __restrict__ recs, unsigned char* __restrict__ dst) {
    const CkptRec R = recs[blockIdx.x];
    const int k = blockIdx.y;
    unsigned char* d = dst + R.off;
    if (k == 0) {
        if (threadIdx.x < 4) ((int*)d)[threadIdx.x] = threadIdx.x == 0 ? R.n : (threadIdx.x == 1 ? R.N : 0);
        return;
    }
    const size_t len = ck_seg_bytes(k, R.n, R.N);
    d += ck_seg_off(k, R.n, R.N);
    ck_copy(d, ck_seg_ptr(Fs[R.slot], k), len);
    ck_zero(d + len, ck_al16(len) - len);
}

// the reverse; the slot's entries past the snapshot's n / N (up to nmax / Nmax) are cleared
__global__ void __launch_bounds__(256) k_ckpt_records_unpack(const DevFilter* __restrict__ Fs, const CkptRec* __restrict__ recs, const unsigned char* __restrict__ src, int nmax, int Nmax) {
    const CkptRec R = recs[blockIdx.x];
    const int k = blockIdx.y + 1;
    const size_t len = ck_seg_bytes(k, R.n, R.N), cap = ck_seg_bytes(k, nmax, Nmax);
    unsigned char* d = ck_seg_ptr(Fs[R.slot], k);
    ck_copy(d, src + R.off + ck_seg_off(k, R.n, R.N), len);
    ck_zero(d + len, cap - len);
}

// CTA per lower tile (I, J): loads the tile and its mirror (J, I), both coalesced; any bit difference between P[i, j] and P[j, i]
// raises bad[slot - b0]; then writes the tile's column segments to their packed positions (64 rows of one column = one
// contiguous 512-byte run).  The CTA of the last diagonal tile also zeroes the triangle's 8-byte padding when n(n+1)/2 is odd.
__global__ void __launch_bounds__(256) k_ckpt_pack(const DevFilter* __restrict__ Fs, const CkptTile* __restrict__ tiles, double* __restrict__ dst, int* __restrict__ bad, int b0) {
    __shared__ double sM[kCkTile][kCkTile + 1];
    const CkptTile t = tiles[blockIdx.x];
    const DevFilter& F = Fs[t.slot];
    const double* __restrict__ P = F.P;
    const size_t ldp = F.ldp;
    const int n = t.n, i0 = kCkTile * t.I, j0 = kCkTile * t.J;
    const int r = threadIdx.x & 63, c0 = threadIdx.x >> 6;
    double v[16];
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const int i = i0 + r, j = j0 + c0 + 4 * k;
        v[k] = (i < n && j < n) ? P[i + j * ldp] : 0.0;
    }
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const int rr = c0 + 4 * k, row = j0 + r, col = i0 + rr;  // sM[rr][cc] = P[j0 + cc, i0 + rr], cc = r
        sM[rr][r] = (row < n && col < n) ? P[row + col * ldp] : 0.0;
    }
    __syncthreads();
    bool diff = false;
#pragma unroll
    for (int k = 0; k < 16; k++) diff |= __double_as_longlong(v[k]) != __double_as_longlong(sM[r][c0 + 4 * k]);
    if (__syncthreads_or(diff) && threadIdx.x == 0) bad[t.slot - b0] = 1;
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const int i = i0 + r, j = j0 + c0 + 4 * k;
        if (j < n && i < n && i >= j) dst[t.pbase + ck_colstart(j, n) + (i - j)] = v[k];
    }
    const long long tri = (long long)n * (n + 1) / 2;
    if (threadIdx.x == 0 && t.I == t.J && i0 + kCkTile >= n && (tri & 1)) dst[t.pbase + tri] = 0.0;
}

// CTA per lower tile: reads the packed tile once and stores (I, J) and, transposed through shared memory, (J, I), both coalesced,
// into the slot's P at its own leading dimension (a diagonal tile's upper half comes from the transposed store)
__global__ void __launch_bounds__(256) k_ckpt_unpack(const DevFilter* __restrict__ Fs, const CkptTile* __restrict__ tiles, const double* __restrict__ src) {
    __shared__ double sT[kCkTile][kCkTile + 1];
    const CkptTile t = tiles[blockIdx.x];
    const DevFilter& F = Fs[t.slot];
    double* __restrict__ P = F.P;
    const size_t ldp = F.ldp;
    const int n = t.n, i0 = kCkTile * t.I, j0 = kCkTile * t.J;
    const int r = threadIdx.x & 63, c0 = threadIdx.x >> 6;
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const int c = c0 + 4 * k, i = i0 + r, j = j0 + c;
        double v = 0.0;
        if (j < n && i < n && i >= j) {
            v = src[t.pbase + ck_colstart(j, n) + (i - j)];
            P[i + j * ldp] = v;
        }
        sT[r][c] = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const int rr = c0 + 4 * k, i = i0 + rr, j = j0 + r;  // element (i, j) of the lower tile goes to P[j, i]
        if (j < n && i < n && i >= j) P[j + i * ldp] = sT[rr][r];
    }
}

}  // namespace rslam
