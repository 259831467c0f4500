// rslam_api.cu -- host side of the C ABI declared in include/rslam.h: handle lifecycle, state transfer and the launch
// sequences of the per-frame path.  No CPU fallback: every entry point needs a CUDA device.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <string>
#include <vector>

#include "common.cuh"
#include "kernels_ckpt.cuh"
#include "kernels_map.cuh"
#include "kernels_track.cuh"
#include "kernels_update.cuh"

using namespace rslam;

namespace {
thread_local std::string g_err;
int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define CK(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e__ = (call);                                                                             \
        if (e__ != cudaSuccess) return fail(RSLAM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }
inline int cdiv(int a, int b) { return (a + b - 1) / b; }
}  // namespace

struct rslam_filter {
    int device = 0, B = 1, Nmax = 0, nmax = 0, ldp = 0, ldw = 0, lds = 0, kmax = 0, mwords = 0;
    rslam_camera cam{};
    rslam_params par{};
    CamDev camd{};
    ParDev pard{};
    cudaStream_t stream = nullptr;
    long long launches = 0;
    std::vector<DevFilter> hF;  // host mirror of the device descriptors
    std::vector<std::vector<int>> htype;  // host mirror of the feature types (the map-management entry points edit the feature list)
    // map surgery scratch (allocated on first use): one spare covariance / state vector that is swapped with the filter's own
    double* map_P = nullptr;
    double* map_x = nullptr;
    double* map_coef = nullptr;
    int* map_res = nullptr;
    unsigned char* map_tmp = nullptr;  // staging for erasing one entry of the per-feature arrays
    // rslam_map_management_batch (allocated on its first call): a spare covariance / state vector PER FILTER (B x ldp x nmax
    // doubles more), swapped with the filter's own on every edit; per-filter plans and coefficients; pinned staging of its inputs
    // (spare pointers, uniforms) and of its one read-back (plans)
    std::vector<double*> mb_P, mb_x;
    MapBatchWs mb{};
    bool mb_ready = false;
    void* mb_h_in = nullptr;   // pinned: [2B] spare pointers, then the uniforms
    void* mb_d_in = nullptr;   // device copy of it
    size_t mb_in_cap = 0;
    int* mb_h_plan = nullptr;  // pinned: [B][MB_INTS] plans, then [B][Nmax] feature types
    // rslam_checkpoint_save / _load: the device staging buffer of host-memory snapshots (<= 256 MB, allocated by the first such
    // call) and the work lists of the current call (chunk records and tiles, then the per-filter symmetry flags)
    unsigned char* ck_stage = nullptr;
    size_t ck_stage_cap = 0;
    unsigned char* ck_list = nullptr;
    size_t ck_list_cap = 0;
    int* fast_score = nullptr;         // FAST scores of the window under test
    size_t fast_cap = 0;
    int* fast_xy = nullptr;
    int fast_xy_cap = 0;
    DevFilter* dF = nullptr;
    std::vector<void*> allocs;
    // shared buffers
    unsigned char* d_images = nullptr;  // rslam_frame's host images (every call rebinds every filter)
    size_t image_cap = 0;
    // rslam_set_image's host images: one buffer per filter and one for the image shared by the batch.  No call writes, moves or frees
    // a buffer that a filter other than the one(s) it binds still reads.
    std::vector<unsigned char*> si_img;
    std::vector<size_t> si_cap;
    unsigned char* si_shared = nullptr;
    size_t si_shared_cap = 0;
    double* d_u01 = nullptr;
    size_t u01_cap = 0;
    // second staging set: rslam_prefetch_inputs copies the NEXT frame's host inputs into it on the copy stream while the current
    // frame computes; the rslam_frame that is handed the same host pointers swaps the two sets instead of copying
    unsigned char* pf_images = nullptr;
    size_t pf_image_cap = 0;
    double* pf_u01 = nullptr;
    size_t pf_u01_cap = 0;
    cudaStream_t copy = nullptr;
    cudaEvent_t ev_staged = nullptr, ev_free_cur = nullptr, ev_free_pf = nullptr;  // copy done; last frame that read the current / the other set done
    bool staged = false;
    const void* staged_img = nullptr;
    const void* staged_u01 = nullptr;
    long long staged_geom[5] = {0, 0, 0, 0, 0};  // rows, cols, stride, share, n_u01
    int* d_hyp_idx = nullptr;
    size_t hyp_cap = 0;
    int* d_used = nullptr;
    int* d_support_all = nullptr;  // base of the per-filter support arrays (zeroed before every scoring pass)
    int* d_sup_h = nullptr;        // per-hypothesis supports of a brute-force sweep
    size_t sup_h_cap = 0;
    unsigned long long* d_key = nullptr;  // [0] key, [1] pair counter
    bool have_image = false;
    bool warp_patches = false;  // run pred_patch_fc on the device before the search
    bool upd_ws = false;
    bool chol2 = true;  // batches of small filters: k_chol_small with two CTAs per SM (RSLAM_CHOL2=0: one)
    bool chol_outer_small = true;  // 64 x 64 tiles for the K = 256 trailing updates of the Cholesky (RSLAM_CHOL_OUTER_SMALL=0: 128 x 64)
    int trsm_ob = 16;  // outer-block width of the large-k TRSM in 64-column blocks (0: one left-looking launch); RSLAM_TRSM_OB overrides
    int hN = 0, hn = 0;  // max over filters of the uploaded N / n
    bool descr_dirty = false;
    // CUDA-graph replay of the per-frame launch sequence
    bool graph_enabled = true;
    bool capturing = false;
    bool li_conditional = true;  // RSLAM_LI_CONDITIONAL=0 keeps the low-innovation update's launches unconditional in the graph
    long long cond_nodes = 0;    // launches inside the IF node (not counted as launches: they run only when armed)
    // side stream for work that is independent of the critical path of a single small filter (W = P H^T beside S + Cholesky)
    bool jnorm_pending = false;  // rslam_frame only: the li update's k_upd_jnorm was deferred into the next rescue launch
    bool hi_gathered = false;  // the last rslam_rescue_hi also built the hi inlier list (single-CTA grids)
    cudaStream_t side = nullptr;
    // what k_set_inputs last wrote into the device descriptors (rslam_frame skips the launch when unchanged)
    const unsigned char* bound_img = nullptr;
    long long bound_iper = -1;
    int bound_geom[3] = {-1, -1, -1};
    const double* bound_u01 = nullptr;
    int bound_nu = -1;
    bool bound_has_img = false;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaGraphExec_t graph_exec = nullptr;
    long long graph_key = -1;
    long long graph_nodes = 0;
    // optional per-launch event timing (diagnostics only; never enabled inside a timed region)
    bool prof = false;
    struct ProfRec {
        const char* name;
        cudaEvent_t e0, e1;
    };
    std::vector<ProfRec> prof_recs;
    std::vector<cudaEvent_t> prof_pool;
};

namespace {

template <typename T>
int dev_alloc(rslam_filter* f, T** p, size_t count, bool zero = true) {
    void* q = nullptr;
    size_t bytes = count * sizeof(T);
    if (bytes == 0) bytes = 16;
    CK(cudaMalloc(&q, bytes));
    if (zero) CK(cudaMemsetAsync(q, 0, bytes, f->stream));
    f->allocs.push_back(q);
    *p = (T*)q;
    return 0;
}

// give back a buffer obtained from dev_alloc (regrown scratch); stream-ordered work that still uses it has been issued on f->stream
void dev_release(rslam_filter* f, void* p) {
    if (!p) return;
    for (size_t i = 0; i < f->allocs.size(); i++)
        if (f->allocs[i] == p) {
            f->allocs.erase(f->allocs.begin() + i);
            break;
        }
    cudaStreamSynchronize(f->stream);
    cudaFree(p);
}

int push_descr(rslam_filter* f) {
    CK(cudaMemcpyAsync(f->dF, f->hF.data(), sizeof(DevFilter) * f->B, cudaMemcpyHostToDevice, f->stream));
    // hF is pageable: the copy is staged before the call returns, so later host edits are safe
    f->descr_dirty = false;
    f->bound_iper = -1;  // the pushed descriptors carry their own image / u01 bindings: rslam_frame must re-bind
    f->bound_nu = -1;
    return 0;
}

int ensure_update_ws(rslam_filter* f) {
    if (f->upd_ws) return 0;
    const size_t wsz = (size_t)f->ldw * f->kmax, ssz = (size_t)f->lds * f->kmax, lsz = (size_t)cdiv(f->kmax, kNB) * kNB * kNB;
    double *W = nullptr, *S = nullptr, *Li = nullptr;
    int rc;
    if ((rc = dev_alloc(f, &W, wsz * f->B))) return rc;
    if ((rc = dev_alloc(f, &S, ssz * f->B))) return rc;
    if ((rc = dev_alloc(f, &Li, lsz * f->B))) return rc;
    for (int b = 0; b < f->B; b++) {
        f->hF[b].W = W + wsz * b;
        f->hF[b].Sm = S + ssz * b;
        f->hF[b].Linv = Li + lsz * b;
    }
    f->upd_ws = true;
    return push_descr(f);
}

bool is_device_ptr(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

__global__ void k_set_inputs(DevFilter* Fs, int B, const unsigned char* img, long long img_stride_per_filter, int rows, int cols, int stride,
                             int set_img, const double* u01, int n_u01, int set_u01) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    if (set_img) {
        Fs[b].image = img ? img + img_stride_per_filter * b : nullptr;
        Fs[b].img_rows = rows;
        Fs[b].img_cols = cols;
        Fs[b].img_stride = stride;
    }
    if (set_u01) {
        Fs[b].u01 = u01 + (size_t)n_u01 * b;
        Fs[b].n_u01 = n_u01;
    }
}

cudaEvent_t prof_event(rslam_filter* f) {
    if (!f->prof_pool.empty()) {
        cudaEvent_t e = f->prof_pool.back();
        f->prof_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

#define LAUNCH(f, kern, grid, block, smem, ...) LAUNCH_N(f, #kern, kern, grid, block, smem, __VA_ARGS__)
#define LAUNCH_N(f, name, kern, grid, block, smem, ...) LAUNCH_ON(f, (f)->stream, name, kern, grid, block, smem, __VA_ARGS__)
#define LAUNCH_ON(f, strm, name, kern, grid, block, smem, ...)                \
    do {                                                                      \
        const bool prof__ = (f)->prof && !(f)->capturing;                     \
        cudaEvent_t e0__ = nullptr, e1__ = nullptr;                           \
        if (prof__) {                                                         \
            e0__ = prof_event(f);                                             \
            e1__ = prof_event(f);                                             \
            cudaEventRecord(e0__, (strm));                                    \
        }                                                                     \
        kern<<<grid, block, smem, (strm)>>>(__VA_ARGS__);                     \
        if (prof__) {                                                         \
            cudaEventRecord(e1__, (strm));                                    \
            (f)->prof_recs.push_back(rslam_filter::ProfRec{name, e0__, e1__}); \
        }                                                                     \
        (f)->launches++;                                                      \
    } while (0)

int check_launch() {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(RSLAM_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
    return 0;
}

int run_update(rslam_filter* f, int which, bool gathered = false, bool defer_jnorm = false) {
    int rc = ensure_update_ws(f);
    if (rc) return rc;
    const int B = f->B, N = f->hN, n = f->hn;
    if (N == 0) return 0;
    const int kmax = 2 * N;
    const int nsteps = cdiv(kmax, kNB);
    // k_upd_W is a thread per state row: 128-thread CTAs when they leave fewer idle rows (n = 613: 640 threads instead of 768)
    const int wbs = round_up(n, 128) < round_up(n, 256) ? 128 : 256;
    if (!gathered) LAUNCH(f, k_upd_gather, dim3(1, B), 256, 0, f->dF, which);
    if (kmax <= kCholSmallMaxK && B == 1) {
        // latency path of one small filter: S comes straight from P, so W = P H^T (needed only by the TRSM) runs on the side stream
        // next to S and its Cholesky factorisation (a fork / join that the frame graph captures as parallel branches).  Under
        // per-launch profiling everything stays on the one stream so that the events bracket single kernels.
        const bool fork = !(f->prof && !f->capturing);
        cudaStream_t ws = fork ? f->side : f->stream;
        if (fork) {
            CK(cudaEventRecord(f->ev_fork, f->stream));
            CK(cudaStreamWaitEvent(f->side, f->ev_fork, 0));
        }
        LAUNCH_ON(f, ws, "k_upd_W", k_upd_W, dim3(cdiv(n, wbs), cdiv(N, kWChunk), B), wbs, 0, f->dF);
        if (fork) CK(cudaEventRecord(f->ev_join, f->side));
        LAUNCH_N(f, "k_upd_S", k_upd_S_direct, dim3(cdiv(N * (N + 1) / 2, 8), 1, B), 256, 0, f->dF);
        LAUNCH_N(f, "k_chol_small", (k_chol_small<kTld, 1>), dim3(1, B), 256, kCholSmallSmemBytes, f->dF);
        LAUNCH(f, k_chol_trinv, dim3(nsteps, B), 256, kTrinvSmemBytes, f->dF);
        if (fork) CK(cudaStreamWaitEvent(f->stream, f->ev_join, 0));
    } else if (kmax <= kCholSmallMaxK) {
        LAUNCH(f, k_upd_W, dim3(cdiv(n, wbs), cdiv(N, kWChunk), B), wbs, 0, f->dF);
        LAUNCH(f, k_upd_S, dim3(cdiv(N, 16), cdiv(N, 16), B), 256, 0, f->dF);
        if (f->chol2 && kmax + kNB <= kCholSmallLd2 + kNB && kmax <= 200 && B >= 2 * 148) {  // two CTAs per SM
            LAUNCH_N(f, "k_chol_small", (k_chol_small<kCholSmallLd2, 2>), dim3(1, B), 256, kCholSmall2SmemBytes, f->dF);
        } else {
            LAUNCH_N(f, "k_chol_small", (k_chol_small<kTld, 1>), dim3(1, B), 256, kCholSmallSmemBytes, f->dF);
        }
        LAUNCH(f, k_chol_trinv, dim3(nsteps, B), 256, kTrinvSmemBytes, f->dF);
    } else {
        LAUNCH(f, k_upd_W, dim3(cdiv(n, wbs), cdiv(N, kWChunk), B), wbs, 0, f->dF);
        LAUNCH(f, k_upd_S, dim3(cdiv(N, 16), cdiv(N, 16), B), 256, 0, f->dF);
        for (int s = 0; s < nsteps; s++) {
            LAUNCH(f, k_chol_panel, dim3(nsteps - s, B), 256, kPanelSmemBytes, f->dF, s);
            const int o = kNB * (s + 1);
            if (kmax <= o) break;
            if ((s + 1) % kOB == 0) {  // end of a 256-wide outer block: everything beyond it gets one K = 256 update
                // the trailing matrix of a K = 256 update is a few hundred 128 x 64 tiles -- one to three waves of 296 slots, the last one mostly
                // empty; 64 x 64 tiles (three CTAs per SM, 444 slots, half the work each) waste less of the machine on these sizes
                const int tm = cdiv(kmax - o, 128), ts = cdiv(kmax - o, 64);
                if (f->chol_outer_small && (long long)ts * (ts + 1) / 2 * B <= 8 * 444) {
                    LAUNCH_N(f, "k_gemm_dmma/chol_outer", (k_gemm_dmma<64, 64>), dim3(ts * (ts + 1) / 2, 1, B), (GemmCfg<64, 64>::kThreads), (GemmCfg<64, 64>::kSmemBytes), f->dF,
                             (int)GEMM_CHOL_OUTER, s / kOB);
                } else {
                    LAUNCH_N(f, "k_gemm_dmma/chol_outer", (k_gemm_dmma<128, 64>), dim3(tm * (tm + 1), 1, B), (GemmCfg<128, 64>::kThreads), (GemmCfg<128, 64>::kSmemBytes), f->dF,
                             (int)GEMM_CHOL_OUTER, s / kOB);
                }
            }
        }
        LAUNCH(f, k_chol_trinv, dim3(nsteps, B), 256, kTrinvSmemBytes, f->dF);
    }
    if (kmax <= SR_KMAX) {  // small systems: W rows resident in smem, L streamed once
        LAUNCH(f, k_trsm_small, dim3(cdiv(n + 1, TS_R), B), TS_THREADS, trsm_small_smem_bytes(kmax), f->dF, round_up(kmax, kNB));
    } else {
        // two-level: the 64-wide blocks of one outer block (f->trsm_ob blocks wide) are solved left-looking by k_trsm_ll (a CTA owns its
        // rows), then one GEMM with K = 64 trsm_ob subtracts that outer block's contribution from all remaining columns of W.
        // trsm_ob == 0: the whole solve in one left-looking launch.
        const int ob = f->trsm_ob > 0 ? f->trsm_ob : nsteps;
        const int nouter = cdiv(nsteps, ob);
        for (int J = 0; J < nouter; J++) {
            if (cdiv(n + 1, 48) * B >= 200) {  // 48-row CTAs, two resident per SM: one CTA's barriers / diagonal step hide behind the other's DMMA stream
                LAUNCH_N(f, "k_trsm_ll", (k_trsm_ll<48, 2>), dim3(cdiv(n + 1, 48), B), 128, (TrsmCfg<48, 2>::kSmemBytes), f->dF, J * ob, (J + 1) * ob);
            } else {
                LAUNCH_N(f, "k_trsm_ll", (k_trsm_ll<32, 2>), dim3(cdiv(n + 1, 32), B), 128, (TrsmCfg<32, 2>::kSmemBytes), f->dF, J * ob, (J + 1) * ob);
            }
            const int o = kNB * ob * (J + 1);
            if (kmax > o) {
                const int tm = cdiv(n + 1, 128), tn = cdiv(kmax - o, 64);
                LAUNCH_N(f, "k_gemm_dmma/trsm_outer", (k_gemm_dmma<128, 64>), dim3(tm * tn, 1, B), (GemmCfg<128, 64>::kThreads), (GemmCfg<128, 64>::kSmemBytes), f->dF,
                         (int)GEMM_TRSM_OUTER | (ob << 16), J);
            }
        }
    }
    if (kmax <= SR_KMAX) {
        // small innovation dimension: row-segment SYRK (A resident, flattened B pipeline, P tile prefetched).  Segment length: whole
        // tile rows when the batch alone fills the machine, single tiles for one filter (latency).
        const int tm = cdiv(n + 1, SR_BM);
        int seg = tm;
        auto ctas = [&](int L) { long long c = 0; for (int i = 0; i < tm; i++) c += (i + L) / L; return c * B; };
        while (seg > 1 && ctas(seg) < 2 * 148) seg = (seg + 1) / 2;
        const int kpad = round_up(kmax, SR_BK);
        LAUNCH_N(f, "k_syrk_rows", k_syrk_rows, dim3((unsigned)(ctas(seg) / B), 1, B), SR_THREADS, syrk_rows_smem_bytes(kmax), f->dF, which, seg, kpad);
    } else {
        const int tm = cdiv(n + 1, 128);
        const int smode = (int)GEMM_SYRK_P | (which << 8);
        if ((long long)tm * (tm + 1) * B >= 192) {
            LAUNCH_N(f, "k_gemm_dmma/syrk_P", (k_gemm_dmma<128, 64>), dim3(tm * (tm + 1), 1, B), (GemmCfg<128, 64>::kThreads), (GemmCfg<128, 64>::kSmemBytes), f->dF, smode, 0);
        } else {
            const int ts = cdiv(n + 1, 64);
            LAUNCH_N(f, "k_gemm_dmma/syrk_P", (k_gemm_dmma<64, 64>), dim3(ts * (ts + 1) / 2, 1, B), (GemmCfg<64, 64>::kThreads), (GemmCfg<64, 64>::kSmemBytes), f->dF, smode, 0);
        }
    }
    if (!defer_jnorm) {  // deferred: fused into the head of the rescue kernel
        if (n >= 4096) {
            LAUNCH_N(f, "k_upd_jnorm", k_upd_jnorm_wide, dim3(cdiv(n, 256), B), 256, 0, f->dF, f->pard);
        } else {
            LAUNCH(f, k_upd_jnorm, dim3(1, B), 256, 0, f->dF, f->pard);
        }
    }
    return check_launch();
}

int run_ransac_core(rslam_filter* f, bool select, bool gather_li = false, unsigned long long cond = 0ull) {
    const int B = f->B, N = f->hN;
    if (N == 0) return 0;
    const int q1 = (int)((f->par.quirks & RSLAM_Q1_ANGLES_FROM_POSITIONS) != 0);
    if (N <= 256) {
        LAUNCH(f, k_ransac_compact_hyp, dim3(1, B), 256, 0, f->dF, q1);
    } else {
        LAUNCH(f, k_ransac_compact, dim3(1, B), N > 1024 ? 1024 : 256, 0, f->dF);
        LAUNCH(f, k_ransac_hyp, dim3(cdiv(N, 128), B), 128, 0, f->dF, q1);
    }
    if (select) {
        LAUNCH(f, k_ransac_support, dim3(cdiv(N, SJT), cdiv(N, SHB), B), SUP_THREADS, kSupSmemBytes, f->dF, f->camd, f->pard, (const int*)nullptr, 0, N, 0, N, (const int*)nullptr,
               (int*)nullptr, (unsigned long long*)nullptr);
        LAUNCH(f, k_ransac_select, dim3(1, B), 256, 0, f->dF, f->pard, gather_li ? 1 : 0, cond);
    }
    return check_launch();
}

}  // namespace

extern "C" {

void rslam_default_params(rslam_params* p) {
    p->std_a = 0.007;
    p->std_alpha = 0.007;
    p->std_z = 1.0;
    p->chi2_095_2 = 5.9915;
    p->corr_threshold = 0.80;
    p->p_spurious_free = 0.99;
    p->n_hyp_initial = 1000;
    p->max_ellipse_eig = 100.0;
    p->quirks = RSLAM_Q_ALL;
    p->dedupe_hypotheses = 1;
}

const char* rslam_last_error(void) { return g_err.c_str(); }
const char* rslam_version(void) { return "rslam-b200 0.1 (sm_100a)"; }

int rslam_create(const rslam_camera* cam, const rslam_params* par, int max_features, int batch, int device, rslam_filter** out) {
    if (!cam || !out || max_features < 1 || batch < 1) return fail(RSLAM_ERR_INVALID, "rslam_create: bad arguments");
    // k_search stages windows of half-width <= kMaxHalfSearch = ceil(2 sqrt(100)); a larger gate would drop the features it lets through
    if (par && !(par->max_ellipse_eig > 0.0 && par->max_ellipse_eig <= 100.0))
        return fail(RSLAM_ERR_INVALID, "rslam_create: max_ellipse_eig = %g is not in (0, 100]", par->max_ellipse_eig);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(RSLAM_ERR_CUDA, "rslam_create: no CUDA device (this library has no CPU fallback)");
    }
    if (device < 0 || device >= ndev) return fail(RSLAM_ERR_INVALID, "rslam_create: device %d out of range (%d devices)", device, ndev);
    CK(cudaSetDevice(device));
    rslam_filter* f = new rslam_filter();
    f->device = device;
    f->B = batch;
    f->Nmax = max_features;
    f->nmax = 13 + 6 * max_features;
    f->ldp = round_up(f->nmax, 16);
    f->ldw = round_up(f->nmax + 1, 16);
    f->kmax = 2 * max_features;
    f->lds = round_up(f->kmax, 16);
    f->mwords = cdiv(max_features, 32);
    if (const char* e = getenv("RSLAM_TRSM_OB")) f->trsm_ob = atoi(e);
    if (const char* e = getenv("RSLAM_CHOL_OUTER_SMALL")) f->chol_outer_small = atoi(e) != 0;
    if (const char* e = getenv("RSLAM_CHOL2")) f->chol2 = atoi(e) != 0;
    if (const char* e = getenv("RSLAM_LI_CONDITIONAL")) f->li_conditional = atoi(e) != 0;
    f->cam = *cam;
    if (par)
        f->par = *par;
    else
        rslam_default_params(&f->par);
    f->camd = CamDev{cam->k1, cam->k2, cam->Cx, cam->Cy, cam->f, cam->dx, cam->dy, cam->f * (1.0 / cam->dx), cam->f * (1.0 / cam->dy), cam->nRows, cam->nCols};
    f->pard = ParDev{f->par.std_z, f->par.chi2_095_2, f->par.corr_threshold, f->par.p_spurious_free, f->par.max_ellipse_eig,
                     (f->par.std_a * 1.0) * (f->par.std_a * 1.0), (f->par.std_alpha * 1.0) * (f->par.std_alpha * 1.0), f->par.n_hyp_initial, f->par.quirks};
    // a failure from here on releases the handle, its streams and its events (rslam_destroy copes with a half-built handle)
#define CKF(call)                                                                                                         \
    do {                                                                                                                  \
        cudaError_t e__ = (call);                                                                                         \
        if (e__ != cudaSuccess) {                                                                                         \
            rslam_destroy(f);                                                                                             \
            return fail(RSLAM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__);     \
        }                                                                                                                 \
    } while (0)
    CKF(cudaStreamCreateWithFlags(&f->stream, cudaStreamNonBlocking));
    CKF(cudaStreamCreateWithFlags(&f->side, cudaStreamNonBlocking));
    CKF(cudaEventCreateWithFlags(&f->ev_fork, cudaEventDisableTiming));
    CKF(cudaEventCreateWithFlags(&f->ev_join, cudaEventDisableTiming));
    CKF(cudaStreamCreateWithFlags(&f->copy, cudaStreamNonBlocking));
    CKF(cudaEventCreateWithFlags(&f->ev_staged, cudaEventDisableTiming));
    CKF(cudaEventCreateWithFlags(&f->ev_free_cur, cudaEventDisableTiming));
    CKF(cudaEventCreateWithFlags(&f->ev_free_pf, cudaEventDisableTiming));
    CKF(cudaFuncSetAttribute(k_gemm_dmma<128, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmCfg<128, 64>::kSmemBytes));
    CKF(cudaFuncSetAttribute(k_gemm_dmma<64, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmCfg<64, 64>::kSmemBytes));
    CKF(cudaFuncSetAttribute(k_trsm_ll<48, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, TrsmCfg<48, 2>::kSmemBytes));
    CKF(cudaFuncSetAttribute(k_trsm_ll<32, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, TrsmCfg<32, 2>::kSmemBytes));
    CKF(cudaFuncSetAttribute(k_ransac_support, cudaFuncAttributeMaxDynamicSharedMemorySize, kSupSmemBytes));
    CKF(cudaFuncSetAttribute(k_chol_panel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPanelSmemBytes));
    CKF(cudaFuncSetAttribute(k_chol_trinv, cudaFuncAttributeMaxDynamicSharedMemorySize, kTrinvSmemBytes));
    CKF(cudaFuncSetAttribute(k_chol_small<kTld, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kCholSmallSmemBytes));
    CKF(cudaFuncSetAttribute(k_chol_small<kCholSmallLd2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kCholSmall2SmemBytes));
    CKF(cudaFuncSetAttribute(k_trsm_small, cudaFuncAttributeMaxDynamicSharedMemorySize, trsm_small_smem_bytes(SR_KMAX)));
    CKF(cudaFuncSetAttribute(k_syrk_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, syrk_rows_smem_bytes(SR_KMAX)));

    const int B = batch, N = max_features, n = f->nmax;
    f->hF.assign(B, DevFilter{});
    f->htype.assign(B, std::vector<int>());
    int rc = 0;
    double *P, *xkk, *xkm1, *h, *Hc, *Hf, *S, *z, *hyp_ab, *hyp_xcam, *Jn;
    int *ftype, *foff, *tp, *tm, *ic_list, *id_list, *id_pos, *support, *ctl, *upd_list, *sup_rows;
    unsigned char *has_h, *ic, *li, *hi;
    float* patch;
    unsigned* masks;
    unsigned char* patch_init;
    double *init_pose, *pp_geom;
    int* last_id;
    const size_t psz = (size_t)f->ldp * n;
#define A(ptr, cnt)                                       \
    if ((rc = dev_alloc(f, &ptr, (size_t)(cnt)*B))) {    \
        rslam_destroy(f);                                 \
        return rc;                                        \
    }
    A(P, psz) A(xkk, n) A(xkm1, n) A(h, 2 * N) A(Hc, 14 * N) A(Hf, 12 * N) A(S, 4 * N) A(z, 2 * N) A(hyp_ab, 16 * N) A(hyp_xcam, 7 * N) A(Jn, 32)
    A(ftype, N) A(foff, N) A(tp, N) A(tm, N) A(ic_list, N) A(id_list, N) A(id_pos, N) A(support, N) A(ctl, CTL_SIZE) A(upd_list, N) A(sup_rows, 6 * (size_t)round_up(N, 64))
    A(has_h, N) A(ic, N) A(li, N) A(hi, N) A(patch, (size_t)N * kPatchPix) A(masks, (size_t)N * f->mwords)
    A(patch_init, (size_t)N * 1681 + 4) A(init_pose, (size_t)N * 14) A(pp_geom, (size_t)N * 12) A(last_id, N)
#undef A
    if ((rc = dev_alloc(f, &f->dF, (size_t)B))) {
        rslam_destroy(f);
        return rc;
    }
    if ((rc = dev_alloc(f, &f->d_used, (size_t)N)) || (rc = dev_alloc(f, &f->d_key, (size_t)2))) {
        rslam_destroy(f);
        return rc;
    }
    for (int b = 0; b < B; b++) {
        DevFilter& D = f->hF[b];
        D.n = 13;
        D.N = 0;
        D.ldp = f->ldp;
        D.ldw = f->ldw;
        D.lds = f->lds;
        D.kmax = f->kmax;
        D.mwords = f->mwords;
        D.P = P + psz * b;
        D.x_kk = xkk + (size_t)n * b;
        D.x_km1 = xkm1 + (size_t)n * b;
        D.ftype = ftype + (size_t)N * b;
        D.foff = foff + (size_t)N * b;
        D.h = h + (size_t)2 * N * b;
        D.Hc = Hc + (size_t)14 * N * b;
        D.Hf = Hf + (size_t)12 * N * b;
        D.S = S + (size_t)4 * N * b;
        D.z = z + (size_t)2 * N * b;
        D.has_h = has_h + (size_t)N * b;
        D.ic = ic + (size_t)N * b;
        D.li = li + (size_t)N * b;
        D.hi = hi + (size_t)N * b;
        D.times_predicted = tp + (size_t)N * b;
        D.times_measured = tm + (size_t)N * b;
        D.patch = patch + (size_t)N * kPatchPix * b;
        D.image = nullptr;
        D.patch_init = patch_init + (size_t)N * 1681 * b;
        D.init_pose = init_pose + (size_t)N * 14 * b;
        D.pp_geom = pp_geom + (size_t)N * 12 * b;
        D.last_id = last_id + (size_t)N * b;
        D.ic_list = ic_list + (size_t)N * b;
        D.id_list = id_list + (size_t)N * b;
        D.sup_rows = sup_rows + 6 * (size_t)round_up(N, 64) * b;
        D.id_pos = id_pos + (size_t)N * b;
        D.hyp_ab = hyp_ab + (size_t)16 * N * b;
        D.hyp_xcam = hyp_xcam + (size_t)7 * N * b;
        D.support = support + (size_t)N * b;
        f->d_support_all = support;
        D.masks = masks + (size_t)N * f->mwords * b;
        D.u01 = nullptr;
        D.n_u01 = 0;
        D.ctl = ctl + (size_t)CTL_SIZE * b;
        D.upd_list = upd_list + (size_t)N * b;
        D.W = nullptr;
        D.Sm = nullptr;
        D.Jn = Jn + (size_t)32 * b;
        D.Linv = nullptr;
    }
    if ((rc = push_descr(f))) {
        rslam_destroy(f);
        return rc;
    }
    CKF(cudaStreamSynchronize(f->stream));
#undef CKF
    *out = f;
    return RSLAM_OK;
}

int rslam_destroy(rslam_filter* f) {
    if (!f) return RSLAM_OK;
    cudaSetDevice(f->device);
    if (f->stream) cudaStreamSynchronize(f->stream);
    if (f->graph_exec) cudaGraphExecDestroy(f->graph_exec);
    for (auto& r : f->prof_recs) {
        cudaEventDestroy(r.e0);
        cudaEventDestroy(r.e1);
    }
    for (auto e : f->prof_pool) cudaEventDestroy(e);
    for (void* p : f->allocs) cudaFree(p);
    if (f->d_images) cudaFree(f->d_images);
    for (unsigned char* p : f->si_img)
        if (p) cudaFree(p);
    if (f->si_shared) cudaFree(f->si_shared);
    if (f->d_u01) cudaFree(f->d_u01);
    if (f->pf_images) cudaFree(f->pf_images);
    if (f->pf_u01) cudaFree(f->pf_u01);
    if (f->ev_staged) cudaEventDestroy(f->ev_staged);
    if (f->ev_free_cur) cudaEventDestroy(f->ev_free_cur);
    if (f->ev_free_pf) cudaEventDestroy(f->ev_free_pf);
    if (f->copy) cudaStreamDestroy(f->copy);
    if (f->mb_h_in) cudaFreeHost(f->mb_h_in);
    if (f->mb_d_in) cudaFree(f->mb_d_in);
    if (f->mb_h_plan) cudaFreeHost(f->mb_h_plan);
    if (f->ck_stage) cudaFree(f->ck_stage);
    if (f->ck_list) cudaFree(f->ck_list);
    if (f->d_hyp_idx) cudaFree(f->d_hyp_idx);
    if (f->d_sup_h) cudaFree(f->d_sup_h);
    if (f->ev_fork) cudaEventDestroy(f->ev_fork);
    if (f->ev_join) cudaEventDestroy(f->ev_join);
    if (f->side) cudaStreamDestroy(f->side);
    if (f->stream) cudaStreamDestroy(f->stream);
    delete f;
    return RSLAM_OK;
}

int rslam_sync(rslam_filter* f) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    CK(cudaStreamSynchronize(f->stream));
    CK(cudaStreamSynchronize(f->copy));  // an outstanding rslam_prefetch_inputs copy
    return RSLAM_OK;
}
void* rslam_stream(rslam_filter* f) { return f ? (void*)f->stream : nullptr; }
long long rslam_launch_count(rslam_filter* f) { return f ? f->launches : 0; }
int rslam_num_features(rslam_filter* f, int b) { return (f && b >= 0 && b < f->B) ? f->hF[b].N : -1; }
int rslam_state_dim(rslam_filter* f, int b) { return (f && b >= 0 && b < f->B) ? f->hF[b].n : -1; }

int rslam_upload_state(rslam_filter* f, int b, int which, const double* x, const double* P, int n, int ldp, const int* feat_types, int N) {
    if (!f || b < 0 || b >= f->B || !x || n < 13 || N < 0) return fail(RSLAM_ERR_INVALID, "rslam_upload_state: bad arguments");
    if (N > f->Nmax) return fail(RSLAM_ERR_CAPACITY, "rslam_upload_state: %d features > max_features %d", N, f->Nmax);
    CK(cudaSetDevice(f->device));
    std::vector<int> types(N, 0), offs(N, 0);
    int off = 13;
    for (int i = 0; i < N; i++) {
        types[i] = feat_types ? feat_types[i] : 0;
        if (types[i] != 0 && types[i] != 1) return fail(RSLAM_ERR_INVALID, "rslam_upload_state: feature type must be 0 or 1");
        offs[i] = off;
        off += types[i] == 0 ? 6 : 3;
    }
    if (off != n) return fail(RSLAM_ERR_INVALID, "rslam_upload_state: n = %d does not match 13 + sum(feature sizes) = %d", n, off);
    if (P && ldp < n) return fail(RSLAM_ERR_INVALID, "rslam_upload_state: ldp < n");
    if (which != 0 && which != 1) return fail(RSLAM_ERR_INVALID, "rslam_upload_state: which must be 0 (x_k_k) or 1 (x_k_km1)");
    DevFilter& D = f->hF[b];
    f->htype[b] = types;
    const bool shape_changed = (D.n != n) || (D.N != N);
    D.n = n;
    D.N = N;
    std::vector<int> lastid(N, -1);
    for (int i = 0, last = -1; i < N; i++) {
        if (types[i] == 0) last = i;
        lastid[i] = last;
    }
    if (N) {
        CK(cudaMemcpyAsync(D.ftype, types.data(), sizeof(int) * N, cudaMemcpyHostToDevice, f->stream));
        CK(cudaMemcpyAsync(D.foff, offs.data(), sizeof(int) * N, cudaMemcpyHostToDevice, f->stream));
        CK(cudaMemcpyAsync(D.last_id, lastid.data(), sizeof(int) * N, cudaMemcpyHostToDevice, f->stream));
    }
    CK(cudaMemcpyAsync(which ? D.x_km1 : D.x_kk, x, sizeof(double) * n, cudaMemcpyDefault, f->stream));
    if (P) {
        CK(cudaMemcpy2DAsync(D.P, sizeof(double) * f->ldp, P, sizeof(double) * ldp, sizeof(double) * n, n, cudaMemcpyDefault, f->stream));
    }
    if (shape_changed) {
        // a new map: clear per-feature state
        CK(cudaMemsetAsync(D.has_h, 0, f->Nmax, f->stream));
        CK(cudaMemsetAsync(D.ic, 0, f->Nmax, f->stream));
        CK(cudaMemsetAsync(D.li, 0, f->Nmax, f->stream));
        CK(cudaMemsetAsync(D.hi, 0, f->Nmax, f->stream));
        CK(cudaMemsetAsync(D.times_predicted, 0, sizeof(int) * f->Nmax, f->stream));
        CK(cudaMemsetAsync(D.times_measured, 0, sizeof(int) * f->Nmax, f->stream));
    }
    f->hN = 0;
    f->hn = 0;
    for (int k = 0; k < f->B; k++) {
        f->hN = f->hF[k].N > f->hN ? f->hF[k].N : f->hN;
        f->hn = f->hF[k].n > f->hn ? f->hF[k].n : f->hn;
    }
    CK(cudaStreamSynchronize(f->stream));  // types/offs are stack vectors
    return push_descr(f);
}

int rslam_download_state(rslam_filter* f, int b, int which, double* x, double* P, int ldp) {
    if (!f || b < 0 || b >= f->B) return fail(RSLAM_ERR_INVALID, "rslam_download_state: bad arguments");
    CK(cudaSetDevice(f->device));
    DevFilter& D = f->hF[b];
    if (x) CK(cudaMemcpyAsync(x, which ? D.x_km1 : D.x_kk, sizeof(double) * D.n, cudaMemcpyDefault, f->stream));
    if (P) {
        if (ldp < D.n) return fail(RSLAM_ERR_INVALID, "rslam_download_state: ldp < n");
        CK(cudaMemcpy2DAsync(P, sizeof(double) * ldp, D.P, sizeof(double) * f->ldp, sizeof(double) * D.n, D.n, cudaMemcpyDefault, f->stream));
    }
    CK(cudaStreamSynchronize(f->stream));
    return RSLAM_OK;
}

int rslam_download_pose(rslam_filter* f, int b, double* x13) {
    if (!f || b < 0 || b >= f->B || !x13) return fail(RSLAM_ERR_INVALID, "rslam_download_pose: bad arguments");
    CK(cudaSetDevice(f->device));
    CK(cudaMemcpyAsync(x13, f->hF[b].x_kk, sizeof(double) * 13, cudaMemcpyDefault, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    return RSLAM_OK;
}

int rslam_upload_patches(rslam_filter* f, int b, const double* patches, int N) {
    if (!f || b < 0 || b >= f->B || !patches || N < 0 || N > f->Nmax) return fail(RSLAM_ERR_INVALID, "rslam_upload_patches: bad arguments");
    CK(cudaSetDevice(f->device));
    std::vector<float> tmp((size_t)N * kPatchPix);
    for (size_t i = 0; i < tmp.size(); i++) tmp[i] = (float)patches[i];  // Converter::toCvMat_f (src/Converter.cpp:83-94)
    CK(cudaMemcpyAsync(f->hF[b].patch, tmp.data(), sizeof(float) * tmp.size(), cudaMemcpyHostToDevice, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    return RSLAM_OK;
}

int rslam_upload_feature_init(rslam_filter* f, int b, const uint8_t* patches41, const double* r_wc, const double* R_wc, const double* uv, int N) {
    if (!f || b < 0 || b >= f->B || !patches41 || !r_wc || !R_wc || !uv || N < 0 || N > f->Nmax) return fail(RSLAM_ERR_INVALID, "rslam_upload_feature_init: bad arguments");
    CK(cudaSetDevice(f->device));
    std::vector<double> pose((size_t)N * 14);
    for (int i = 0; i < N; i++) {
        for (int k = 0; k < 3; k++) pose[(size_t)i * 14 + k] = r_wc[3 * i + k];
        for (int k = 0; k < 9; k++) pose[(size_t)i * 14 + 3 + k] = R_wc[9 * i + k];
        pose[(size_t)i * 14 + 12] = uv[2 * i];
        pose[(size_t)i * 14 + 13] = uv[2 * i + 1];
    }
    CK(cudaMemcpyAsync(f->hF[b].patch_init, patches41, (size_t)N * 1681, cudaMemcpyHostToDevice, f->stream));
    CK(cudaMemcpyAsync(f->hF[b].init_pose, pose.data(), sizeof(double) * pose.size(), cudaMemcpyHostToDevice, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    return RSLAM_OK;
}

int rslam_set_patch_warp(rslam_filter* f, int enable) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    f->warp_patches = enable != 0;
    f->graph_key = -1;
    return RSLAM_OK;
}

int rslam_download_patches(rslam_filter* f, int b, float* patches, int N) {
    if (!f || b < 0 || b >= f->B || !patches || N < 0 || N > f->Nmax) return fail(RSLAM_ERR_INVALID, "rslam_download_patches: bad arguments");
    CK(cudaSetDevice(f->device));
    CK(cudaMemcpyAsync(patches, f->hF[b].patch, sizeof(float) * (size_t)N * kPatchPix, cudaMemcpyDeviceToHost, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    return RSLAM_OK;
}

int rslam_download_features(rslam_filter* f, int b, double* h, double* S, double* z, uint8_t* flags, int* counters) {
    if (!f || b < 0 || b >= f->B) return fail(RSLAM_ERR_INVALID, "rslam_download_features: bad arguments");
    CK(cudaSetDevice(f->device));
    DevFilter& D = f->hF[b];
    const int N = D.N;
    if (N == 0) return RSLAM_OK;
    if (h) CK(cudaMemcpyAsync(h, D.h, sizeof(double) * 2 * N, cudaMemcpyDeviceToHost, f->stream));
    if (S) CK(cudaMemcpyAsync(S, D.S, sizeof(double) * 4 * N, cudaMemcpyDeviceToHost, f->stream));
    if (z) CK(cudaMemcpyAsync(z, D.z, sizeof(double) * 2 * N, cudaMemcpyDeviceToHost, f->stream));
    std::vector<unsigned char> a(N), bb(N), c(N), d(N);
    std::vector<int> tp(N), tm(N);
    if (flags) {
        CK(cudaMemcpyAsync(a.data(), D.has_h, N, cudaMemcpyDeviceToHost, f->stream));
        CK(cudaMemcpyAsync(bb.data(), D.ic, N, cudaMemcpyDeviceToHost, f->stream));
        CK(cudaMemcpyAsync(c.data(), D.li, N, cudaMemcpyDeviceToHost, f->stream));
        CK(cudaMemcpyAsync(d.data(), D.hi, N, cudaMemcpyDeviceToHost, f->stream));
    }
    if (counters) {
        CK(cudaMemcpyAsync(tp.data(), D.times_predicted, sizeof(int) * N, cudaMemcpyDeviceToHost, f->stream));
        CK(cudaMemcpyAsync(tm.data(), D.times_measured, sizeof(int) * N, cudaMemcpyDeviceToHost, f->stream));
    }
    CK(cudaStreamSynchronize(f->stream));
    for (int i = 0; i < N; i++) {
        if (flags) {
            flags[4 * i] = a[i];
            flags[4 * i + 1] = bb[i];
            flags[4 * i + 2] = c[i];
            flags[4 * i + 3] = d[i];
        }
        if (counters) {
            counters[2 * i] = tp[i];
            counters[2 * i + 1] = tm[i];
        }
    }
    return RSLAM_OK;
}

int rslam_download_H(rslam_filter* f, int b, double* Hc, double* Hf) {
    if (!f || b < 0 || b >= f->B) return fail(RSLAM_ERR_INVALID, "rslam_download_H: bad arguments");
    CK(cudaSetDevice(f->device));
    DevFilter& D = f->hF[b];
    if (Hc) CK(cudaMemcpyAsync(Hc, D.Hc, sizeof(double) * 14 * D.N, cudaMemcpyDeviceToHost, f->stream));
    if (Hf) CK(cudaMemcpyAsync(Hf, D.Hf, sizeof(double) * 12 * D.N, cudaMemcpyDeviceToHost, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    return RSLAM_OK;
}

int rslam_upload_linearisation(rslam_filter* f, int b, const double* h, const double* Hc, const double* Hf, const double* z, const uint8_t* flags) {
    if (!f || b < 0 || b >= f->B) return fail(RSLAM_ERR_INVALID, "rslam_upload_linearisation: bad arguments");
    CK(cudaSetDevice(f->device));
    DevFilter& D = f->hF[b];
    const int N = D.N;
    if (N == 0) return RSLAM_OK;
    if (h) CK(cudaMemcpyAsync(D.h, h, sizeof(double) * 2 * N, cudaMemcpyDefault, f->stream));
    if (Hc) CK(cudaMemcpyAsync(D.Hc, Hc, sizeof(double) * 14 * N, cudaMemcpyDefault, f->stream));
    if (Hf) CK(cudaMemcpyAsync(D.Hf, Hf, sizeof(double) * 12 * N, cudaMemcpyDefault, f->stream));
    if (z) CK(cudaMemcpyAsync(D.z, z, sizeof(double) * 2 * N, cudaMemcpyDefault, f->stream));
    std::vector<unsigned char> a, bb, c, d;
    if (flags) {
        a.resize(N);
        bb.resize(N);
        c.resize(N);
        d.resize(N);
        for (int i = 0; i < N; i++) {
            a[i] = flags[4 * i] != 0;
            bb[i] = flags[4 * i + 1] != 0;
            c[i] = flags[4 * i + 2] != 0;
            d[i] = flags[4 * i + 3] != 0;
        }
        CK(cudaMemcpyAsync(D.has_h, a.data(), N, cudaMemcpyHostToDevice, f->stream));
        CK(cudaMemcpyAsync(D.ic, bb.data(), N, cudaMemcpyHostToDevice, f->stream));
        CK(cudaMemcpyAsync(D.li, c.data(), N, cudaMemcpyHostToDevice, f->stream));
        CK(cudaMemcpyAsync(D.hi, d.data(), N, cudaMemcpyHostToDevice, f->stream));
    }
    CK(cudaStreamSynchronize(f->stream));
    return RSLAM_OK;
}

int rslam_set_matches(rslam_filter* f, int b, const double* z, const uint8_t* ic) {
    if (!f || b < 0 || b >= f->B || !z || !ic) return fail(RSLAM_ERR_INVALID, "rslam_set_matches: bad arguments");
    CK(cudaSetDevice(f->device));
    DevFilter& D = f->hF[b];
    CK(cudaMemcpyAsync(D.z, z, sizeof(double) * 2 * D.N, cudaMemcpyDefault, f->stream));
    CK(cudaMemcpyAsync(D.ic, ic, D.N, cudaMemcpyDefault, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    return RSLAM_OK;
}

// A host image is copied into a buffer of its own: filter b's (share == 0) or the batch's shared one (share != 0).  A buffer that
// must grow is freed only while no filter outside this call's binding reads it: filter b's buffer is read by filter b alone, and the
// shared buffer only by filters that a shared binding rebinds (all of them).
static int set_images(rslam_filter* f, int b, const uint8_t* gray, int rows, int cols, int stride, int share) {
    const size_t per = (size_t)rows * stride;
    const unsigned char* img = gray;
    if (!is_device_ptr(gray)) {
        if (f->si_img.empty()) {
            f->si_img.assign(f->B, nullptr);
            f->si_cap.assign(f->B, 0);
        }
        unsigned char*& buf = share ? f->si_shared : f->si_img[b];
        size_t& cap = share ? f->si_shared_cap : f->si_cap[b];
        if (per > cap) {
            if (buf) CK(cudaFree(buf));  // synchronises with the work that still reads it
            buf = nullptr;
            cap = 0;
            CK(cudaMalloc((void**)&buf, per));
            cap = per;
        }
        CK(cudaMemcpyAsync(buf, gray, per, cudaMemcpyHostToDevice, f->stream));
        img = buf;
    }
    if (share) {
        LAUNCH(f, k_set_inputs, cdiv(f->B, 128), 128, 0, f->dF, f->B, img, 0LL, rows, cols, stride, 1, (const double*)nullptr, 0, 0);
        f->bound_iper = -1;  // bound outside rslam_frame: its cache is stale
        f->bound_nu = -1;
        for (int k = 0; k < f->B; k++) {
            f->hF[k].image = img;
            f->hF[k].img_rows = rows;
            f->hF[k].img_cols = cols;
            f->hF[k].img_stride = stride;
        }
    } else {
        DevFilter& D = f->hF[b];
        D.image = img;
        D.img_rows = rows;
        D.img_cols = cols;
        D.img_stride = stride;
        int rc = push_descr(f);
        if (rc) return rc;
    }
    f->have_image = true;
    return check_launch();
}

int rslam_set_image(rslam_filter* f, int b, const uint8_t* gray, int rows, int cols, int stride, int share) {
    if (!f || b < 0 || b >= f->B || !gray || rows <= 0 || cols <= 0 || stride < cols) return fail(RSLAM_ERR_INVALID, "rslam_set_image: bad arguments");
    CK(cudaSetDevice(f->device));
    return set_images(f, b, gray, rows, cols, stride, share);
}

int rslam_begin_frame(rslam_filter* f) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    CK(cudaSetDevice(f->device));
    if (f->hN == 0) return RSLAM_OK;
    LAUNCH(f, k_begin_frame, dim3(cdiv(f->hN, 128), f->B), 128, 0, f->dF);
    return check_launch();
}

int rslam_ekf_prediction(rslam_filter* f) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    CK(cudaSetDevice(f->device));
    LAUNCH(f, k_ekf_prediction, dim3(cdiv(f->hn > 13 ? f->hn : 13, 128), f->B), 128, 0, f->dF, f->pard, 0);
    return check_launch();
}

int rslam_predict_measurements(rslam_filter* f) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    CK(cudaSetDevice(f->device));
    if (f->hN == 0) return RSLAM_OK;
    LAUNCH(f, k_predict, dim3(cdiv(f->hN, 128), f->B), 128, 0, f->dF, f->camd, f->pard, 0, 0, 0);
    if (f->warp_patches) {
        LAUNCH(f, k_pred_patch_setup, dim3(cdiv(f->hN, 64), f->B), 64, 0, f->dF, f->camd);
        LAUNCH(f, k_pred_patch, dim3(f->hN, f->B), 192, 0, f->dF, f->camd);
    }
    return check_launch();
}

int rslam_match(rslam_filter* f) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    CK(cudaSetDevice(f->device));
    if (f->hN == 0) return RSLAM_OK;
    if (!f->have_image) return fail(RSLAM_ERR_INVALID, "rslam_match: no image is bound (rslam_set_image)");
    LAUNCH(f, k_search, dim3(f->hN, f->B), kSearchThreads, 0, f->dF, f->camd, f->pard);
    return check_launch();
}

int rslam_search_ic_matches(rslam_filter* f) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    int rc = rslam_predict_measurements(f);
    if (rc || f->hN == 0 || !f->have_image) return rc;
    return rslam_match(f);
}

static int set_u01(rslam_filter* f, const double* u01, int n_u01) {
    if (!u01 || n_u01 <= 0) return fail(RSLAM_ERR_INVALID, "u01 must hold at least one draw per filter");
    const double* base = u01;
    if (!is_device_ptr(u01)) {
        const size_t need = (size_t)n_u01 * f->B;
        if (need > f->u01_cap) {
            if (f->d_u01) CK(cudaFree(f->d_u01));
            CK(cudaMalloc((void**)&f->d_u01, need * sizeof(double)));
            f->u01_cap = need;
        }
        CK(cudaMemcpyAsync(f->d_u01, u01, need * sizeof(double), cudaMemcpyHostToDevice, f->stream));
        base = f->d_u01;
    }
    LAUNCH(f, k_set_inputs, cdiv(f->B, 128), 128, 0, f->dF, f->B, (const unsigned char*)nullptr, 0LL, 0, 0, 0, 0, base, n_u01, 1);
    f->bound_iper = -1;  // bound outside rslam_frame: its cache is stale
    f->bound_nu = -1;
    for (int b = 0; b < f->B; b++) {
        f->hF[b].u01 = base + (size_t)n_u01 * b;
        f->hF[b].n_u01 = n_u01;
    }
    return check_launch();
}

int rslam_ransac_hypotheses(rslam_filter* f, const double* u01, int n_u01) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    CK(cudaSetDevice(f->device));
    int rc = set_u01(f, u01, n_u01);
    if (rc) return rc;
    return run_ransac_core(f, true);
}

int rslam_ransac_result_get(rslam_filter* f, int b, rslam_ransac_result* out) {
    if (!f || b < 0 || b >= f->B || !out) return fail(RSLAM_ERR_INVALID, "rslam_ransac_result_get: bad arguments");
    CK(cudaSetDevice(f->device));
    int ctl[CTL_SIZE];
    CK(cudaMemcpyAsync(ctl, f->hF[b].ctl, sizeof(ctl), cudaMemcpyDeviceToHost, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    out->status = ctl[CTL_STATUS];
    out->hyp_run = ctl[CTL_HYPRUN];
    out->best_support = ctl[CTL_BEST];
    out->n_hyp = ctl[CTL_NHYP];
    out->num_ic = ctl[CTL_NIC];
    out->winner = ctl[CTL_WINNER];
    if (ctl[CTL_NCART] > 0) return fail(RSLAM_ERR_REFERENCE_UB, "cartesian features have matches: the reference's support scoring is undefined here (SURVEY A.3 Q2)");
    return RSLAM_OK;
}

int rslam_update_li(rslam_filter* f) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    CK(cudaSetDevice(f->device));
    return run_update(f, 0);
}

int rslam_rescue_hi(rslam_filter* f) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    CK(cudaSetDevice(f->device));
    if (f->hN == 0) return RSLAM_OK;
    // one CTA per filter: the hi inlier list is gathered by the same launch (consumed by the next rslam_update_hi / run_update(f, 1))
    const int fuse = cdiv(f->hN, 128) == 1 ? 1 : 0;
    if (fuse) {
        int rc = ensure_update_ws(f);  // gather_inliers writes the innovation into W
        if (rc) return rc;
    }
    LAUNCH(f, k_predict, dim3(cdiv(f->hN, 128), f->B), 128, 0, f->dF, f->camd, f->pard, 1, fuse, (fuse && f->jnorm_pending) ? 1 : 0);
    f->jnorm_pending = false;
    f->hi_gathered = fuse != 0;
    return check_launch();
}

int rslam_update_hi(rslam_filter* f) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    CK(cudaSetDevice(f->device));
    const bool gathered = f->hi_gathered;
    f->hi_gathered = false;
    return run_update(f, 1, gathered);
}

// resolve a host-or-device image batch to a device base pointer (copying host data into the handle's staging buffer)
static int resolve_images(rslam_filter* f, const uint8_t* images, int rows, int stride, int share, const unsigned char** base, long long* per_filter) {
    const size_t per = (size_t)rows * stride;
    *per_filter = share ? 0 : (long long)per;
    if (is_device_ptr(images)) {
        *base = images;
        return 0;
    }
    const size_t need = per * (share ? 1 : f->B);
    if (need > f->image_cap) {
        if (f->d_images) CK(cudaFree(f->d_images));
        CK(cudaMalloc((void**)&f->d_images, need));
        f->image_cap = need;
    }
    CK(cudaMemcpyAsync(f->d_images, images, need, cudaMemcpyHostToDevice, f->stream));
    *base = f->d_images;
    return 0;
}
static int resolve_u01(rslam_filter* f, const double* u01, int n_u01, const double** base) {
    if (is_device_ptr(u01)) {
        *base = u01;
        return 0;
    }
    const size_t need = (size_t)n_u01 * f->B;
    if (need > f->u01_cap) {
        if (f->d_u01) CK(cudaFree(f->d_u01));
        CK(cudaMalloc((void**)&f->d_u01, need * sizeof(double)));
        f->u01_cap = need;
    }
    CK(cudaMemcpyAsync(f->d_u01, u01, need * sizeof(double), cudaMemcpyHostToDevice, f->stream));
    *base = f->d_u01;
    return 0;
}

// the fixed launch sequence of one frame (src/System.cpp:111-129); inputs already bound by k_set_inputs
static int run_frame_stages(rslam_filter* f, int flags) {
    int rc;
    if (flags & 1) {  // begin_frame folded into the prediction launch (n >= N always)
        LAUNCH(f, k_ekf_prediction, dim3(cdiv(f->hn > 13 ? f->hn : 13, 128), f->B), 128, 0, f->dF, f->pard, 1);
    }
    if ((rc = rslam_search_ic_matches(f))) return rc;
    if ((rc = ensure_update_ws(f))) return rc;
    // Low-innovation update as an IF node of the frame graph, for large batches: with no low-innovation inlier in any filter (the usual
    // outcome with quirk Q1) every one of its launches exits at once, but the grids are sized for the maps, not for the inlier counts --
    // 0.27 ms per empty launch of the 4096-filter batch.  k_ransac_select arms the node when any filter has inliers.  Not for a single
    // filter: one small filter pays more for the node than for the six launches it skips, and at N = 2000 the ~90 empty launches cost
    // 0.03 ms of 25 (DESIGN.md section 8) -- and ncu cannot profile the kernel nodes of a graph that holds a conditional node.
    const bool li_cond = f->capturing && f->li_conditional && f->B > 1 && (long long)f->B * f->hN >= 4096;
    cudaGraph_t cap_graph = nullptr;
    cudaGraphConditionalHandle cond = 0;
    cudaStreamCaptureStatus cap_status;
    if (li_cond) {
        CK(cudaStreamGetCaptureInfo_v2(f->stream, &cap_status, nullptr, &cap_graph, nullptr, nullptr));
        CK(cudaGraphConditionalHandleCreate(&cond, cap_graph, 0, cudaGraphCondAssignDefault));
    }
    if ((rc = run_ransac_core(f, true, true, (unsigned long long)cond))) return rc;
    // single-CTA rescue kernel: the li update's closing quaternion normalisation rides at its head (one dependent launch less)
    const bool defer = cdiv(f->hN, 128) == 1 && f->hN > 0;
    if (li_cond) {
        const cudaGraphNode_t* deps = nullptr;
        size_t ndeps = 0;
        CK(cudaStreamGetCaptureInfo_v2(f->stream, &cap_status, nullptr, &cap_graph, &deps, &ndeps));
        cudaGraphNodeParams np = {cudaGraphNodeTypeConditional};
        np.type = cudaGraphNodeTypeConditional;
        np.conditional.handle = cond;
        np.conditional.type = cudaGraphCondTypeIf;
        np.conditional.size = 1;
        cudaGraphNode_t node = nullptr;
        CK(cudaGraphAddNode(&node, cap_graph, deps, ndeps, &np));
        cudaGraph_t body = np.conditional.phGraph_out[0];
        CK(cudaStreamUpdateCaptureDependencies(f->stream, &node, 1, cudaStreamSetCaptureDependencies));
        // the update's launches go to the body graph: capture them on the side stream, standing in for the handle's stream
        CK(cudaStreamBeginCaptureToGraph(f->side, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal));
        cudaStream_t main_stream = f->stream;
        f->stream = f->side;
        const long long before = f->launches;
        rc = run_update(f, 0, true, defer);
        f->cond_nodes = f->launches - before;
        f->stream = main_stream;
        cudaGraph_t body_out = nullptr;
        cudaError_t e = cudaStreamEndCapture(f->side, &body_out);
        if (rc) return rc;
        if (e != cudaSuccess) return fail(RSLAM_ERR_CUDA, "capture of the conditional update failed: %s", cudaGetErrorString(e));
    } else {
        f->cond_nodes = 0;
        if ((rc = run_update(f, 0, true, defer))) return rc;
    }
    f->jnorm_pending = defer;
    if ((rc = rslam_rescue_hi(f))) return rc;
    const bool gathered = f->hi_gathered;
    f->hi_gathered = false;
    if ((rc = run_update(f, 1, gathered))) return rc;
    return 0;
}

int rslam_prefetch_inputs(rslam_filter* f, const uint8_t* images, int rows, int cols, int stride, int share, const double* u01, int n_u01) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    if (!u01 || n_u01 <= 0) return fail(RSLAM_ERR_INVALID, "rslam_prefetch_inputs: u01 must hold at least one draw per filter");
    if (images && (rows <= 0 || cols <= 0 || stride < cols)) return fail(RSLAM_ERR_INVALID, "rslam_prefetch_inputs: bad image geometry");
    CK(cudaSetDevice(f->device));
    if ((images && is_device_ptr(images)) || is_device_ptr(u01))
        return fail(RSLAM_ERR_INVALID, "rslam_prefetch_inputs: inputs already on the device need no staging -- pass them to rslam_frame");
    const size_t ineed = images ? (size_t)rows * stride * (share ? 1 : f->B) : 0;
    const size_t uneed = (size_t)n_u01 * f->B;
    if (ineed > f->pf_image_cap) {
        if (f->pf_images) CK(cudaFree(f->pf_images));
        f->pf_images = nullptr;
        f->pf_image_cap = 0;
        CK(cudaMalloc((void**)&f->pf_images, ineed));
        f->pf_image_cap = ineed;
    }
    if (uneed > f->pf_u01_cap) {
        if (f->pf_u01) CK(cudaFree(f->pf_u01));
        f->pf_u01 = nullptr;
        f->pf_u01_cap = 0;
        CK(cudaMalloc((void**)&f->pf_u01, uneed * sizeof(double)));
        f->pf_u01_cap = uneed;
    }
    CK(cudaStreamWaitEvent(f->copy, f->ev_free_pf, 0));  // the last frame that read this set (no-op if there was none)
    if (images) CK(cudaMemcpyAsync(f->pf_images, images, ineed, cudaMemcpyHostToDevice, f->copy));
    CK(cudaMemcpyAsync(f->pf_u01, u01, uneed * sizeof(double), cudaMemcpyHostToDevice, f->copy));
    CK(cudaEventRecord(f->ev_staged, f->copy));
    f->staged = true;
    f->staged_img = images;
    f->staged_u01 = u01;
    f->staged_geom[0] = rows;
    f->staged_geom[1] = cols;
    f->staged_geom[2] = stride;
    f->staged_geom[3] = share;
    f->staged_geom[4] = n_u01;
    return RSLAM_OK;
}

int rslam_frame(rslam_filter* f, const uint8_t* images, int rows, int cols, int stride, int share, const double* u01, int n_u01, int flags) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    if (!u01 || n_u01 <= 0) return fail(RSLAM_ERR_INVALID, "rslam_frame: u01 must hold at least one draw per filter");
    CK(cudaSetDevice(f->device));
    int rc;
    const unsigned char* ibase = nullptr;
    long long iper = 0;
    const double* ubase = nullptr;
    if (images && (rows <= 0 || cols <= 0 || stride < cols)) return fail(RSLAM_ERR_INVALID, "rslam_frame: bad image geometry");
    const bool use_staged = f->staged && f->staged_img == (const void*)images && f->staged_u01 == (const void*)u01 && f->staged_geom[4] == n_u01 &&
                            (!images || (f->staged_geom[0] == rows && f->staged_geom[1] == cols && f->staged_geom[2] == stride && f->staged_geom[3] == share));
    f->staged = false;
    if (use_staged) {
        // the inputs were copied by rslam_prefetch_inputs: make that set the current one
        if (images) {  // (no image staged: the current one stays bound)
            std::swap(f->d_images, f->pf_images);
            std::swap(f->image_cap, f->pf_image_cap);
        }
        std::swap(f->d_u01, f->pf_u01);
        std::swap(f->u01_cap, f->pf_u01_cap);
        std::swap(f->ev_free_cur, f->ev_free_pf);
        CK(cudaStreamWaitEvent(f->stream, f->ev_staged, 0));
        if (images) {
            ibase = f->d_images;
            iper = share ? 0 : (long long)rows * stride;
        }
        ubase = f->d_u01;
    } else {
        if (images && (rc = resolve_images(f, images, rows, stride, share, &ibase, &iper))) return rc;
        if ((rc = resolve_u01(f, u01, n_u01, &ubase))) return rc;
    }
    if ((rc = ensure_update_ws(f))) return rc;
    // bind the inputs in the device descriptors -- skipped when nothing changed (host inputs always land in the same staging buffers)
    if (f->descr_dirty || f->bound_img != ibase || f->bound_iper != iper || f->bound_geom[0] != rows || f->bound_geom[1] != cols || f->bound_geom[2] != stride ||
        f->bound_u01 != ubase || f->bound_nu != n_u01 || (images != nullptr) != f->bound_has_img) {
        LAUNCH(f, k_set_inputs, cdiv(f->B, 128), 128, 0, f->dF, f->B, ibase, iper, rows, cols, stride, images ? 1 : 0, ubase, n_u01, 1);
        f->bound_img = ibase;
        f->bound_iper = iper;
        f->bound_geom[0] = rows;
        f->bound_geom[1] = cols;
        f->bound_geom[2] = stride;
        f->bound_u01 = ubase;
        f->bound_nu = n_u01;
        f->bound_has_img = images != nullptr;
    }
    for (int b = 0; b < f->B; b++) {
        if (images) {
            f->hF[b].image = ibase + iper * b;
            f->hF[b].img_rows = rows;
            f->hF[b].img_cols = cols;
            f->hF[b].img_stride = stride;
        }
        f->hF[b].u01 = ubase + (size_t)n_u01 * b;
        f->hF[b].n_u01 = n_u01;
    }
    if (images) f->have_image = true;
    if (!f->graph_enabled || f->prof) {
        if ((rc = run_frame_stages(f, flags))) return rc;
        CK(cudaEventRecord(f->ev_free_cur, f->stream));
        return check_launch();
    }
    const long long key = ((long long)f->hN << 40) ^ ((long long)f->hn << 16) ^ ((long long)f->B << 4) ^ ((flags & 1) << 1) ^ (f->have_image ? 1 : 0) ^ (f->warp_patches ? 4 : 0);
    if (!f->graph_exec || key != f->graph_key) {
        if (f->graph_exec) {
            cudaGraphExecDestroy(f->graph_exec);
            f->graph_exec = nullptr;
        }
        cudaGraph_t graph = nullptr;
        const long long before = f->launches;
        CK(cudaStreamBeginCapture(f->stream, cudaStreamCaptureModeThreadLocal));
        f->capturing = true;
        rc = run_frame_stages(f, flags);
        f->capturing = false;
        cudaError_t e = cudaStreamEndCapture(f->stream, &graph);
        if (rc) {
            if (graph) cudaGraphDestroy(graph);
            return rc;
        }
        if (e != cudaSuccess) return fail(RSLAM_ERR_CUDA, "stream capture failed: %s", cudaGetErrorString(e));
        f->graph_nodes = f->launches - before - f->cond_nodes;
        f->launches = before;
        CK(cudaGraphInstantiate(&f->graph_exec, graph, 0));
        cudaGraphDestroy(graph);
        f->graph_key = key;
    }
    CK(cudaGraphLaunch(f->graph_exec, f->stream));
    CK(cudaEventRecord(f->ev_free_cur, f->stream));
    f->launches += f->graph_nodes;
    return RSLAM_OK;
}

#ifdef RSLAM_SUP_CLOCKS
extern "C" int rslam_debug_sup_clocks(unsigned long long* out8) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out8, rslam::g_sup_clk, sizeof(unsigned long long) * 8);
    unsigned long long z[8] = {0};
    cudaMemcpyToSymbol(rslam::g_sup_clk, z, sizeof(z));
    return 0;
}
#endif
#ifdef RSLAM_PHASE_CLOCKS
// per-CTA timeline of k_gemm_dmma (record 0: the last syrk_P launch, 1: the first trsm_outer launch; filter 0): up to max_ctas
// rows of 8 values, zeroed after the read
extern "C" int rslam_debug_gemm_stamps(int record, unsigned long long* out, int max_ctas) {
    if (record < 0 || record > 1 || !out || max_ctas <= 0) return -1;
    const int n = std::min(max_ctas, rslam::kGemmStampCtas);
    const size_t row = sizeof(unsigned long long) * rslam::kGemmStampFields, off = (size_t)record * rslam::kGemmStampCtas * row;
    cudaDeviceSynchronize();
    if (cudaMemcpyFromSymbol(out, rslam::g_gemm_stamps, n * row, off) != cudaSuccess) return -1;
    void* p = nullptr;
    if (cudaGetSymbolAddress(&p, rslam::g_gemm_stamps) != cudaSuccess || cudaMemset((char*)p + off, 0, rslam::kGemmStampCtas * row) != cudaSuccess) return -1;
    cudaDeviceSynchronize();
    return n;
}
#endif
// diagnostics: the 32-double scratch block of filter b (phase clocks when built with -DRSLAM_PHASE_CLOCKS)
int rslam_debug_scratch(rslam_filter* f, int b, double* out32) {
    if (!f || b < 0 || b >= f->B || !out32) return fail(RSLAM_ERR_INVALID, "rslam_debug_scratch: bad arguments");
    CK(cudaSetDevice(f->device));
    CK(cudaStreamSynchronize(f->stream));
    CK(cudaMemcpy(out32, f->hF[b].Jn, 32 * sizeof(double), cudaMemcpyDeviceToHost));
    return RSLAM_OK;
}

int rslam_set_graph(rslam_filter* f, int enable) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    f->graph_enabled = enable != 0;
    return RSLAM_OK;
}

int rslam_profile_enable(rslam_filter* f, int enable) {
    if (!f) return fail(RSLAM_ERR_INVALID, "null handle");
    f->prof = enable != 0;
    return RSLAM_OK;
}

// text report "kernel count total_ms\n" per kernel name since the last read; waits for the stream
int rslam_profile_read(rslam_filter* f, char* buf, size_t buflen) {
    if (!f || !buf || buflen == 0) return fail(RSLAM_ERR_INVALID, "rslam_profile_read: bad arguments");
    CK(cudaSetDevice(f->device));
    CK(cudaStreamSynchronize(f->stream));
    std::vector<const char*> names;
    std::vector<double> ms;
    std::vector<long long> cnt;
    for (auto& r : f->prof_recs) {
        float t = 0.f;
        cudaEventElapsedTime(&t, r.e0, r.e1);
        size_t k = 0;
        for (; k < names.size(); k++)
            if (names[k] == r.name || !strcmp(names[k], r.name)) break;
        if (k == names.size()) {
            names.push_back(r.name);
            ms.push_back(0.0);
            cnt.push_back(0);
        }
        ms[k] += t;
        cnt[k] += 1;
        f->prof_pool.push_back(r.e0);
        f->prof_pool.push_back(r.e1);
    }
    f->prof_recs.clear();
    std::string out;
    char line[256];
    for (size_t k = 0; k < names.size(); k++) {
        snprintf(line, sizeof(line), "%s %lld %.6f\n", names[k], cnt[k], ms[k]);
        out += line;
    }
    snprintf(buf, buflen, "%s", out.c_str());
    return RSLAM_OK;
}

// enqueue one (shard of a) sweep on the handle's stream; the packed key lands in f->d_key[0], the pair count in f->d_key[1]
static int sweep_local(rslam_filter* f, const int* hyp_match_idx, int n_hyp, int hyp_begin, int hyp_end, int match_begin, int match_end, const int** d_idx_out) {
    const int N = f->hN;
    if (N == 0) return fail(RSLAM_ERR_INVALID, "rslam_support_sweep: no features uploaded");
    if (f->B != 1) return fail(RSLAM_ERR_INVALID, "rslam_support_sweep: the sweep acts on a single filter (batch == 1)");
    int rc;
    const int* d_idx = hyp_match_idx;
    if (!is_device_ptr(hyp_match_idx)) {
        if ((size_t)n_hyp > f->hyp_cap) {
            if (f->d_hyp_idx) CK(cudaFree(f->d_hyp_idx));
            f->d_hyp_idx = nullptr;
            f->hyp_cap = 0;
            CK(cudaMalloc((void**)&f->d_hyp_idx, sizeof(int) * (size_t)n_hyp));
            f->hyp_cap = n_hyp;
        }
        CK(cudaMemcpyAsync(f->d_hyp_idx + hyp_begin, hyp_match_idx + hyp_begin, sizeof(int) * (size_t)(hyp_end - hyp_begin), cudaMemcpyHostToDevice, f->stream));
        d_idx = f->d_hyp_idx;
    }
    if (d_idx_out) *d_idx_out = d_idx;
    const int q1 = (int)((f->par.quirks & RSLAM_Q1_ANGLES_FROM_POSITIONS) != 0);
    const int nh = hyp_end - hyp_begin;
    const bool dedupe = f->par.dedupe_hypotheses != 0;
    const int tlo = match_begin < N ? match_begin : N, thi = match_end < N ? match_end : N;
    // launch 1: ordered match lists; zeroes the dedupe marks, the key and the pair counter
    LAUNCH(f, k_sweep_compact, 1, N > 1024 ? 1024 : 256, 0, f->dF, f->d_used, f->Nmax, f->d_key);
    // launch 2: hypothesis constants of the distinct hypotheses this shard can score + the row table + the dedupe marks
    {
        const int nt = dedupe ? (thi - tlo) : N;
        int nb_hyp = cdiv(nt > 0 ? nt : 1, 128);
        const int nb_tab = cdiv(cdiv(N, kSupTile) * 6 * kSupTile, 4 * 128);  // four table entries per thread
        if (nb_hyp < (nb_tab < 148 ? nb_tab : 148)) nb_hyp = nb_tab < 148 ? nb_tab : 148;  // enough threads for the row table
        int nb_mark = 0;
        if (dedupe && nh > 0) nb_mark = cdiv(nh, 4 * 128) < 592 ? cdiv(nh, 4 * 128) : 592;
        LAUNCH(f, k_sweep_prep, nb_hyp + nb_mark, 128, 0, f->dF, q1, dedupe ? tlo : 0, dedupe ? thi : N, nb_hyp, d_idx, hyp_begin, hyp_end, match_begin, match_end,
               nb_mark ? f->d_used : (int*)nullptr);
    }
    if (nh > 0) {
        if (dedupe) {
            if (thi > tlo)
                LAUNCH(f, k_ransac_support, dim3(cdiv(N, SJT), cdiv(thi - tlo, SHB), 1), SUP_THREADS, kSupSmemBytes, f->dF, f->camd, f->pard, (const int*)nullptr, tlo, thi, tlo, thi,
                       (const int*)f->d_used, (int*)nullptr, f->d_key + 1);
            LAUNCH(f, k_sweep_reduce, cdiv(nh, 4 * 256) < 296 ? cdiv(nh, 4 * 256) : 296, 256, 0, f->dF, d_idx, hyp_begin, hyp_end, match_begin, match_end, (const int*)nullptr,
                   f->d_key);
        } else {
            if ((size_t)n_hyp > f->sup_h_cap) {
                if (f->d_sup_h) CK(cudaFree(f->d_sup_h));
                f->d_sup_h = nullptr;
                f->sup_h_cap = 0;
                CK(cudaMalloc((void**)&f->d_sup_h, sizeof(int) * (size_t)n_hyp));
                f->sup_h_cap = n_hyp;
            }
            CK(cudaMemsetAsync(f->d_sup_h + hyp_begin, 0, sizeof(int) * (size_t)nh, f->stream));
            LAUNCH(f, k_ransac_support, dim3(cdiv(N, SJT), cdiv(nh, SHB), 1), SUP_THREADS, kSupSmemBytes, f->dF, f->camd, f->pard, d_idx, hyp_begin, hyp_end, match_begin, match_end,
                   (const int*)nullptr, f->d_sup_h, f->d_key + 1);
            LAUNCH(f, k_sweep_reduce, cdiv(nh, 4 * 256) < 296 ? cdiv(nh, 4 * 256) : 296, 256, 0, f->dF, d_idx, hyp_begin, hyp_end, match_begin, match_end, (const int*)f->d_sup_h,
                   f->d_key);
        }
    }
    (void)rc;
    return check_launch();
}

int rslam_support_sweep(rslam_filter* f, const int* hyp_match_idx, int n_hyp, int hyp_begin, int hyp_end, int match_begin, int match_end,
                        uint64_t* best_key, uint8_t* best_mask, long long* n_pairs_scored) {
    if (!f || !hyp_match_idx || n_hyp <= 0 || hyp_begin < 0 || hyp_end > n_hyp || hyp_begin > hyp_end || match_begin < 0 || match_end < match_begin || !best_key)
        return fail(RSLAM_ERR_INVALID, "rslam_support_sweep: bad arguments");
    CK(cudaSetDevice(f->device));
    int rc;
    const int* d_idx = nullptr;
    if ((rc = sweep_local(f, hyp_match_idx, n_hyp, hyp_begin, hyp_end, match_begin, match_end, &d_idx))) return rc;
    CK(cudaMemcpyAsync(best_key, f->d_key, sizeof(uint64_t), cudaMemcpyDefault, f->stream));
    const bool key_on_host = !is_device_ptr(best_key);
    if (key_on_host || best_mask || n_pairs_scored) CK(cudaStreamSynchronize(f->stream));
    if (n_pairs_scored) {
        unsigned long long c = 0;
        CK(cudaMemcpy(&c, f->d_key + 1, sizeof(c), cudaMemcpyDeviceToHost));
        *n_pairs_scored = (long long)c;
    }
    if (best_mask) {
        unsigned long long key = 0;
        CK(cudaMemcpy(&key, f->d_key, sizeof(key), cudaMemcpyDeviceToHost));
        int ctl[CTL_SIZE];
        CK(cudaMemcpy(ctl, f->hF[0].ctl, sizeof(ctl), cudaMemcpyDeviceToHost));
        const int m = ctl[CTL_MID];
        memset(best_mask, 0, (size_t)(m + 7) / 8);
        if (key != 0) {
            const unsigned id = 0xFFFFFFFFu - (unsigned)(key & 0xFFFFFFFFull);
            int t = 0;
            CK(cudaMemcpy(&t, d_idx + id, sizeof(int), cudaMemcpyDeviceToHost));
            return rslam_sweep_mask(f, t, best_mask);
        }
    }
    return RSLAM_OK;
}

int rslam_sweep_mask(rslam_filter* f, int match_idx, uint8_t* mask) {
    if (!f || !mask || match_idx < 0) return fail(RSLAM_ERR_INVALID, "rslam_sweep_mask: bad arguments");
    CK(cudaSetDevice(f->device));
    CK(cudaStreamSynchronize(f->stream));
    int ctl[CTL_SIZE];
    CK(cudaMemcpy(ctl, f->hF[0].ctl, sizeof(ctl), cudaMemcpyDeviceToHost));
    const int m = ctl[CTL_MID];
    if (match_idx >= ctl[CTL_NIC]) return fail(RSLAM_ERR_INVALID, "rslam_sweep_mask: match index out of range");
    std::vector<unsigned> words(f->mwords);
    CK(cudaMemcpy(words.data(), f->hF[0].masks + (size_t)match_idx * f->mwords, sizeof(unsigned) * f->mwords, cudaMemcpyDeviceToHost));
    memset(mask, 0, (size_t)(m + 7) / 8);
    for (int j = 0; j < m; j++)
        if ((words[j >> 5] >> (j & 31)) & 1u) mask[j >> 3] |= (uint8_t)(1u << (j & 7));
    return RSLAM_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------------
// Map management on the device (src/Map.cpp): the covariance stays in HBM while features are deleted, converted and added
// ---------------------------------------------------------------------------------------------------------------------
namespace {

int ensure_map_ws(rslam_filter* f) {
    if (f->map_P) return 0;
    int rc;
    if ((rc = dev_alloc(f, &f->map_P, (size_t)f->ldp * f->nmax))) return rc;
    if ((rc = dev_alloc(f, &f->map_x, (size_t)f->nmax))) return rc;
    if ((rc = dev_alloc(f, &f->map_coef, (size_t)kMapScratch))) return rc;
    if ((rc = dev_alloc(f, &f->map_res, (size_t)4))) return rc;
    if ((rc = dev_alloc(f, &f->map_tmp, (size_t)f->Nmax * 1681))) return rc;
    return 0;
}

// recompute offsets / last inverse-depth index from the host type list and push them with the descriptor
int map_sync_layout(rslam_filter* f, int b) {
    DevFilter& D = f->hF[b];
    const std::vector<int>& types = f->htype[b];
    const int N = (int)types.size();
    std::vector<int> offs(N), lastid(N);
    int off = 13, last = -1;
    for (int i = 0; i < N; i++) {
        offs[i] = off;
        off += types[i] == 0 ? 6 : 3;
        if (types[i] == 0) last = i;
        lastid[i] = last;
    }
    D.N = N;
    if (N) {
        CK(cudaMemcpyAsync(D.ftype, types.data(), sizeof(int) * N, cudaMemcpyHostToDevice, f->stream));
        CK(cudaMemcpyAsync(D.foff, offs.data(), sizeof(int) * N, cudaMemcpyHostToDevice, f->stream));
        CK(cudaMemcpyAsync(D.last_id, lastid.data(), sizeof(int) * N, cudaMemcpyHostToDevice, f->stream));
    }
    f->hN = 0;
    f->hn = 0;
    for (int k = 0; k < f->B; k++) {
        f->hN = f->hF[k].N > f->hN ? f->hF[k].N : f->hN;
        f->hn = f->hF[k].n > f->hn ? f->hF[k].n : f->hn;
    }
    CK(cudaStreamSynchronize(f->stream));  // offs / lastid are stack vectors
    return push_descr(f);
}

// run P' = T P T^T + E, x' = T x into the spare buffers and swap them in
int map_apply(rslam_filter* f, int b, const MapXform& xf) {
    DevFilter& D = f->hF[b];
    LAUNCH(f, k_map_xform, dim3(cdiv(xf.n_new, 256), std::min(xf.n_new, 65535)), 256, 0, f->dF, b, xf, (const double*)f->map_coef, f->map_P, f->map_x);
    std::swap(D.P, f->map_P);
    std::swap(D.x_kk, f->map_x);
    D.n = xf.n_new;
    int rc = check_launch();
    if (rc) return rc;
    return push_descr(f);  // the next kernel must see the swapped buffers
}

// erase entry p of a per-feature device array (count entries of elem bytes), through the staging buffer
int erase_entry(rslam_filter* f, void* base, size_t elem, int count, int p) {
    const size_t tail = (size_t)(count - 1 - p) * elem;
    if (tail == 0) return 0;
    unsigned char* bp = (unsigned char*)base;
    CK(cudaMemcpyAsync(f->map_tmp, bp + (size_t)(p + 1) * elem, tail, cudaMemcpyDeviceToDevice, f->stream));
    CK(cudaMemcpyAsync(bp + (size_t)p * elem, f->map_tmp, tail, cudaMemcpyDeviceToDevice, f->stream));
    return 0;
}

// features_info.erase(it) (src/Map.cpp:27): drop the record, not the state
int map_erase_info(rslam_filter* f, int b, int p) {
    DevFilter& D = f->hF[b];
    const int N = D.N;
    int rc;
    if ((rc = erase_entry(f, D.times_predicted, sizeof(int), N, p))) return rc;
    if ((rc = erase_entry(f, D.times_measured, sizeof(int), N, p))) return rc;
    if ((rc = erase_entry(f, D.patch, sizeof(float) * kPatchPix, N, p))) return rc;
    if ((rc = erase_entry(f, D.patch_init, 1681, N, p))) return rc;
    if ((rc = erase_entry(f, D.init_pose, sizeof(double) * 14, N, p))) return rc;
    // the per-frame outputs are members of the same Feature record (ExtendKF.h:14-42) and move with it: the flags decide the
    // counters of the next Map::map_management step 2 (src/Map.cpp:34-47) and its `measured` count (:57-66)
    if ((rc = erase_entry(f, D.has_h, 1, N, p))) return rc;
    if ((rc = erase_entry(f, D.ic, 1, N, p))) return rc;
    if ((rc = erase_entry(f, D.li, 1, N, p))) return rc;
    if ((rc = erase_entry(f, D.hi, 1, N, p))) return rc;
    if ((rc = erase_entry(f, D.h, sizeof(double) * 2, N, p))) return rc;
    if ((rc = erase_entry(f, D.z, sizeof(double) * 2, N, p))) return rc;
    if ((rc = erase_entry(f, D.S, sizeof(double) * 4, N, p))) return rc;
    if ((rc = erase_entry(f, D.Hc, sizeof(double) * 14, N, p))) return rc;
    if ((rc = erase_entry(f, D.Hf, sizeof(double) * 12, N, p))) return rc;
    f->htype[b].erase(f->htype[b].begin() + p);
    D.N = N - 1;
    return 0;
}

// body of Map::delete_a_feature (src/Map.cpp:69-104): remove `size` rows / columns at state offset `off`
int map_remove_block(rslam_filter* f, int b, int off, int size) {
    DevFilter& D = f->hF[b];
    MapXform xf{};
    xf.mode = 0;
    xf.n_old = D.n;
    xf.n_new = D.n - size;
    xf.cut_at = off;
    xf.cut_cnt = size;
    xf.sp_at = xf.n_new;
    xf.sp_cnt = 0;
    return map_apply(f, b, xf);
}

}  // namespace

extern "C" {

int rslam_map_delete_feature(rslam_filter* f, int b, int index) {
    if (!f || b < 0 || b >= f->B || index < 0 || index >= f->hF[b].N) return fail(RSLAM_ERR_INVALID, "rslam_map_delete_feature: bad arguments");
    CK(cudaSetDevice(f->device));
    int rc = ensure_map_ws(f);
    if (rc) return rc;
    int off = 13;
    for (int i = 0; i < index; i++) off += f->htype[b][i] == 0 ? 6 : 3;
    const int size = f->htype[b][index] == 0 ? 6 : 3;
    if ((rc = map_remove_block(f, b, off, size))) return rc;
    if ((rc = map_erase_info(f, b, index))) return rc;
    return map_sync_layout(f, b);
}

int rslam_map_delete_features(rslam_filter* f, int b, int reference_indexing, int* n_deleted) {
    if (!f || b < 0 || b >= f->B) return fail(RSLAM_ERR_INVALID, "rslam_map_delete_features: bad arguments");
    CK(cudaSetDevice(f->device));
    int rc = ensure_map_ws(f);
    if (rc) return rc;
    DevFilter& D = f->hF[b];
    const int N0 = D.N;
    if (n_deleted) *n_deleted = 0;
    if (N0 == 0) return RSLAM_OK;
    std::vector<int> tp(N0), tm(N0);
    CK(cudaMemcpyAsync(tp.data(), D.times_predicted, sizeof(int) * N0, cudaMemcpyDeviceToHost, f->stream));
    CK(cudaMemcpyAsync(tm.data(), D.times_measured, sizeof(int) * N0, cudaMemcpyDeviceToHost, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    // src/Map.cpp:19-32.  `i` counts loop iterations (1-based) and is what delete_a_feature receives; after the first erase it runs
    // ahead of the iterator, so the reference removes the STATE block of a later feature than the record it erased, and reads the
    // type of the record that slid into position i-1.  reference_indexing != 0 reproduces exactly that; 0 deletes consistently.
    int pos = 0, deleted = 0;
    for (int i = 1; pos < (int)f->htype[b].size(); i++) {
        if (tm[pos] < tp[pos] * 0.5 && tp[pos] > 5) {
            const int erased_type = f->htype[b][pos];
            tp.erase(tp.begin() + pos);
            tm.erase(tm.begin() + pos);
            if ((rc = map_erase_info(f, b, pos))) return rc;
            const std::vector<int>& ty = f->htype[b];  // features_info AFTER the erase, which is what delete_a_feature reads
            int size, off = 13;
            if (reference_indexing) {
                if (i - 1 >= (int)ty.size()) {
                    map_sync_layout(f, b);
                    return fail(RSLAM_ERR_REFERENCE_UB, "map_management: delete_a_feature(%d) indexes past the end of features_info (src/Map.cpp:73)", i);
                }
                size = ty[i - 1] == 0 ? 6 : 3;
                for (int k = 0; k < i - 1; k++) off += ty[k] == 0 ? 6 : 3;
            } else {
                size = erased_type == 0 ? 6 : 3;
                for (int k = 0; k < pos; k++) off += ty[k] == 0 ? 6 : 3;
            }
            if (off + size > D.n) {
                map_sync_layout(f, b);
                return fail(RSLAM_ERR_REFERENCE_UB, "map_management: delete_a_feature(%d) removes rows past the end of the state (src/Map.cpp:88-101)", i);
            }
            if ((rc = map_remove_block(f, b, off, size))) return rc;
            deleted++;
        } else {
            pos++;
        }
    }
    if (n_deleted) *n_deleted = deleted;
    if ((rc = map_sync_layout(f, b))) return rc;
    int total = 13;
    for (int t : f->htype[b]) total += t == 0 ? 6 : 3;
    if (total != D.n) return fail(RSLAM_ERR_REFERENCE_UB, "map_management: state dimension %d no longer matches features_info (%d): the reference would assert", D.n, total);
    return RSLAM_OK;
}

int rslam_map_inversedepth_to_cartesian(rslam_filter* f, int b, int* converted_index) {
    if (!f || b < 0 || b >= f->B) return fail(RSLAM_ERR_INVALID, "rslam_map_inversedepth_to_cartesian: bad arguments");
    CK(cudaSetDevice(f->device));
    int rc = ensure_map_ws(f);
    if (rc) return rc;
    DevFilter& D = f->hF[b];
    if (converted_index) *converted_index = -1;
    if (D.N == 0) return RSLAM_OK;
    const int none = 0x7fffffff;
    CK(cudaMemcpyAsync(f->map_res, &none, sizeof(int), cudaMemcpyHostToDevice, f->stream));
    LAUNCH(f, k_map_linearity, cdiv(D.N, 128), 128, 0, f->dF, b, 0.1, f->map_res);
    int idx = none;
    CK(cudaMemcpyAsync(&idx, f->map_res, sizeof(int), cudaMemcpyDeviceToHost, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    if (idx == none) return RSLAM_OK;
    int ip = 13;
    for (int i = 0; i < idx; i++) ip += f->htype[b][i] == 0 ? 6 : 3;
    LAUNCH(f, k_map_prep_convert, 1, 32, 0, f->dF, b, ip, f->map_coef);
    MapXform xf{};
    xf.mode = 1;
    xf.n_old = D.n;
    xf.n_new = D.n - 3;
    xf.cut_at = ip;
    xf.cut_cnt = 6;
    xf.sp_at = ip;
    xf.sp_cnt = 3;
    xf.src_at = ip;
    xf.src_cnt = 6;
    if ((rc = map_apply(f, b, xf))) return rc;
    f->htype[b][idx] = 1;
    if (converted_index) *converted_index = idx;
    return map_sync_layout(f, b);
}

int rslam_map_add_feature(rslam_filter* f, int b, const double* uv, int* new_index) {
    if (!f || b < 0 || b >= f->B || !uv) return fail(RSLAM_ERR_INVALID, "rslam_map_add_feature: bad arguments");
    DevFilter& D = f->hF[b];
    if (D.N + 1 > f->Nmax || D.n + 6 > f->nmax) return fail(RSLAM_ERR_CAPACITY, "rslam_map_add_feature: the handle was created for at most %d features", f->Nmax);
    CK(cudaSetDevice(f->device));
    int rc = ensure_map_ws(f);
    if (rc) return rc;
    // initial_rho = 1, std_rho = 1, std_pxl = std_z (src/Map.cpp:216-219)
    LAUNCH(f, k_map_prep_add, 8, 256, 0, f->dF, b, f->camd, uv[0], uv[1], 1.0, f->par.std_z, 1.0, f->map_coef);
    MapXform xf{};
    xf.mode = 2;
    xf.n_old = D.n;
    xf.n_new = D.n + 6;
    xf.cut_at = D.n;
    xf.cut_cnt = 0;
    xf.sp_at = D.n;
    xf.sp_cnt = 6;
    xf.src_at = 0;
    xf.src_cnt = 13;
    if ((rc = map_apply(f, b, xf))) return rc;
    f->htype[b].push_back(0);
    if (new_index) *new_index = D.N;
    return map_sync_layout(f, b);
}

}  // extern "C"

extern "C" {
int rslam_feature_types(rslam_filter* f, int b, int* types) {
    if (!f || b < 0 || b >= f->B || !types) return fail(RSLAM_ERR_INVALID, "rslam_feature_types: bad arguments");
    for (size_t i = 0; i < f->htype[b].size(); i++) types[i] = f->htype[b][i];
    return RSLAM_OK;
}
int rslam_set_counters(rslam_filter* f, int b, const int* times_predicted, const int* times_measured) {
    if (!f || b < 0 || b >= f->B || !times_predicted || !times_measured) return fail(RSLAM_ERR_INVALID, "rslam_set_counters: bad arguments");
    CK(cudaSetDevice(f->device));
    const int N = f->hF[b].N;
    if (N) {
        CK(cudaMemcpyAsync(f->hF[b].times_predicted, times_predicted, sizeof(int) * N, cudaMemcpyDefault, f->stream));
        CK(cudaMemcpyAsync(f->hF[b].times_measured, times_measured, sizeof(int) * N, cudaMemcpyDefault, f->stream));
        CK(cudaStreamSynchronize(f->stream));
    }
    return RSLAM_OK;
}
int rslam_download_feature_init(rslam_filter* f, int b, int i, uint8_t* patch41, double* pose14) {
    if (!f || b < 0 || b >= f->B || i < 0 || i >= f->hF[b].N) return fail(RSLAM_ERR_INVALID, "rslam_download_feature_init: bad arguments");
    CK(cudaSetDevice(f->device));
    if (patch41) CK(cudaMemcpyAsync(patch41, f->hF[b].patch_init + (size_t)i * 1681, 1681, cudaMemcpyDeviceToHost, f->stream));
    if (pose14) CK(cudaMemcpyAsync(pose14, f->hF[b].init_pose + (size_t)i * 14, sizeof(double) * 14, cudaMemcpyDeviceToHost, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    return RSLAM_OK;
}
}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------------
// Feature initialisation (src/Map.cpp:198-338): FAST corners on the device, sampling-box test, full map_management
// ---------------------------------------------------------------------------------------------------------------------
namespace {
int fast_detect(rslam_filter* f, int b, int x0, int y0, int w, int h, int threshold, int max_kp, int* n_kp_dev_res /* device int[>=1] */) {
    const DevFilter& D = f->hF[b];
    if (!D.image) return fail(RSLAM_ERR_INVALID, "FAST: no image is bound to filter %d (rslam_set_image)", b);
    if (x0 < 0 || y0 < 0 || w < 1 || h < 1 || x0 + w > D.img_cols || y0 + h > D.img_rows) return fail(RSLAM_ERR_INVALID, "FAST: window outside the image");
    if ((size_t)w * h > f->fast_cap) {
        dev_release(f, f->fast_score);
        f->fast_score = nullptr;
        f->fast_cap = 0;
        int rc = dev_alloc(f, &f->fast_score, (size_t)w * h);
        if (rc) return rc;
        f->fast_cap = (size_t)w * h;
    }
    if (max_kp > f->fast_xy_cap) {
        dev_release(f, f->fast_xy);
        f->fast_xy = nullptr;
        f->fast_xy_cap = 0;
        int rc = dev_alloc(f, &f->fast_xy, (size_t)2 * max_kp);
        if (rc) return rc;
        f->fast_xy_cap = max_kp;
    }
    threshold = threshold < 0 ? 0 : (threshold > 255 ? 255 : threshold);
    LAUNCH(f, k_fast9_score, cdiv(w * h, 256), 256, 0, f->dF, b, x0, y0, w, h, threshold, f->fast_score);
    LAUNCH(f, k_fast9_nms, 1, 1024, 0, (const int*)f->fast_score, w, h, max_kp, n_kp_dev_res, f->fast_xy);
    return check_launch();
}
}  // namespace

extern "C" {

int rslam_fast_corner_detect_9(rslam_filter* f, int b, int x0, int y0, int w, int h, int threshold, int max_kp, int* n_kp, int* xy) {
    if (!f || b < 0 || b >= f->B || !n_kp || max_kp < 1) return fail(RSLAM_ERR_INVALID, "rslam_fast_corner_detect_9: bad arguments");
    CK(cudaSetDevice(f->device));
    int rc = ensure_map_ws(f);
    if (rc) return rc;
    if ((rc = fast_detect(f, b, x0, y0, w, h, threshold, max_kp, f->map_res))) return rc;
    CK(cudaMemcpyAsync(n_kp, f->map_res, sizeof(int), cudaMemcpyDeviceToHost, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    const int n = *n_kp < max_kp ? *n_kp : max_kp;
    if (xy && n > 0) {
        CK(cudaMemcpyAsync(xy, f->fast_xy, sizeof(int) * 2 * n, cudaMemcpyDeviceToHost, f->stream));
        CK(cudaStreamSynchronize(f->stream));
    }
    return RSLAM_OK;
}

int rslam_map_initialize_features(rslam_filter* f, int b, int step, int min_features_to_init, const double* u01, int n_pairs, int* n_initialized,
                                  int* attempts_out) {
    (void)step;
    if (!f || b < 0 || b >= f->B || (!u01 && n_pairs > 0)) return fail(RSLAM_ERR_INVALID, "rslam_map_initialize_features: bad arguments");
    CK(cudaSetDevice(f->device));
    int rc = ensure_map_ws(f);
    if (rc) return rc;
    const int max_attempts = 50, excluded_band = 21, sx = 30, sy = 20;  // src/Map.cpp:200, 215-216
    int attempts = 0, initialized = 0;
    if (n_initialized) *n_initialized = 0;
    while (initialized < min_features_to_init && attempts < max_attempts) {
        if (attempts >= n_pairs) {
            if (attempts_out) *attempts_out = attempts;
            if (n_initialized) *n_initialized = initialized;
            return fail(RSLAM_ERR_INVALID, "rslam_map_initialize_features: the uniform draws ran out after %d attempts", attempts);
        }
        const double cx = round(u01[2 * attempts] * (f->cam.nCols - 2 * excluded_band - 2 * sx)) + excluded_band + sx;
        const double cy = round(u01[2 * attempts + 1] * (f->cam.nRows - 2 * excluded_band - 2 * sy)) + excluded_band + sy;
        attempts++;
        CK(cudaMemsetAsync(f->map_res, 0, sizeof(int) * 4, f->stream));
        const DevFilter& D = f->hF[b];
        if (D.N) LAUNCH(f, k_map_box_count, cdiv(D.N, 128), 128, 0, f->dF, b, f->camd, cx, cy, (double)sx, (double)sy, f->map_res + 1);
        const int x0 = (int)(cx - sx), y0 = (int)(cy - sy);
        const int w = (int)(cx + sx + 1) - x0, h = (int)(cy + sy + 1) - y0;
        if ((rc = fast_detect(f, b, x0, y0, w, h, 100, 1, f->map_res))) return rc;
        int res[2] = {0, 0}, kp[2] = {0, 0};
        CK(cudaMemcpyAsync(res, f->map_res, sizeof(int) * 2, cudaMemcpyDeviceToHost, f->stream));
        CK(cudaMemcpyAsync(kp, f->fast_xy, sizeof(int) * 2, cudaMemcpyDeviceToHost, f->stream));
        CK(cudaStreamSynchronize(f->stream));
        if (res[0] > 0 && res[1] == 0) {
            // the port keeps MATLAB's "- 1" (src/Map.cpp:243-244): the corner lands one pixel up and left of where FAST found it
            const double uv[2] = {kp[0] + (-sx + cx - 1), kp[1] + (-sy + cy - 1)};
            if (f->hF[b].N + 1 > f->Nmax) {
                if (attempts_out) *attempts_out = attempts;
                if (n_initialized) *n_initialized = initialized;
                return fail(RSLAM_ERR_CAPACITY, "rslam_map_initialize_features: the handle was created for at most %d features", f->Nmax);
            }
            if ((rc = rslam_map_add_feature(f, b, uv, nullptr))) return rc;
            initialized++;
        }
    }
    if (attempts_out) *attempts_out = attempts;
    if (n_initialized) *n_initialized = initialized;
    return RSLAM_OK;
}

int rslam_map_management(rslam_filter* f, int b, int step, int min_features, int reference_indexing, const double* u01, int n_pairs, int* info4) {
    if (!f || b < 0 || b >= f->B) return fail(RSLAM_ERR_INVALID, "rslam_map_management: bad arguments");
    if (f->B != 1) return fail(RSLAM_ERR_INVALID, "rslam_map_management: step 2 resets the flags of every filter of the handle; use a batch of 1");
    CK(cudaSetDevice(f->device));
    int rc, nd = 0, conv = -1, init = 0, attempts = 0;
    if ((rc = rslam_map_delete_features(f, b, reference_indexing, &nd))) return rc;
    const int N = f->hF[b].N;
    int measured = 0;
    if (N) {
        std::vector<unsigned char> li(N), hi(N);
        CK(cudaMemcpyAsync(li.data(), f->hF[b].li, N, cudaMemcpyDeviceToHost, f->stream));
        CK(cudaMemcpyAsync(hi.data(), f->hF[b].hi, N, cudaMemcpyDeviceToHost, f->stream));
        CK(cudaStreamSynchronize(f->stream));
        for (int i = 0; i < N; i++) measured += (li[i] || hi[i]) ? 1 : 0;
    }
    if ((rc = rslam_begin_frame(f))) return rc;
    if ((rc = rslam_map_inversedepth_to_cartesian(f, b, &conv))) return rc;
    if (measured == 0)
        rc = rslam_map_initialize_features(f, b, step, min_features, u01, n_pairs, &init, &attempts);
    else if (measured < min_features)
        rc = rslam_map_initialize_features(f, b, step, min_features - measured, u01, n_pairs, &init, &attempts);
    if (info4) {
        info4[0] = nd;
        info4[1] = conv;
        info4[2] = init;
        info4[3] = attempts;
    }
    return rc;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------------
// Map::map_management for every filter of the handle in one fixed launch sequence (kernels_map.cuh, k_mmb_*)
// ---------------------------------------------------------------------------------------------------------------------
namespace {
int ensure_map_batch_ws(rslam_filter* f) {
    if (f->mb_ready) return 0;
    const int B = f->B, Nmax = f->Nmax, nmax = f->nmax;
    const int max_add = Nmax < kMbMaxAttempts ? Nmax : kMbMaxAttempts;
    MapBatchWs& w = f->mb;
    w.Nmax = Nmax;
    w.nmax = nmax;
    w.coef_stride = kMbAdd + max_add * kMbAddStride;
    int rc;
    double *P = nullptr, *x = nullptr;
    if ((rc = dev_alloc(f, &P, (size_t)f->ldp * nmax * B, false))) return rc;
    if ((rc = dev_alloc(f, &x, (size_t)nmax * B))) return rc;
    if ((rc = dev_alloc(f, &w.plan, (size_t)MB_INTS * B))) return rc;
    if ((rc = dev_alloc(f, &w.rowmap, (size_t)nmax * B))) return rc;
    if ((rc = dev_alloc(f, &w.recsrc, (size_t)Nmax * B))) return rc;
    if ((rc = dev_alloc(f, &w.rectail, (size_t)Nmax * B))) return rc;
    if ((rc = dev_alloc(f, &w.types, (size_t)Nmax * B))) return rc;
    if ((rc = dev_alloc(f, &w.vis, (size_t)Nmax * B))) return rc;
    if ((rc = dev_alloc(f, &w.pix, (size_t)2 * Nmax * B))) return rc;
    if ((rc = dev_alloc(f, &w.coef, (size_t)w.coef_stride * B))) return rc;
    CK(cudaMallocHost((void**)&f->mb_h_plan, sizeof(int) * ((size_t)MB_INTS + Nmax) * B));
    f->mb_P.resize(B);
    f->mb_x.resize(B);
    for (int b = 0; b < B; b++) {
        f->mb_P[b] = P + (size_t)f->ldp * nmax * b;
        f->mb_x[b] = x + (size_t)nmax * b;
    }
    f->mb_ready = true;
    return 0;
}
}  // namespace

extern "C" {

int rslam_map_management_batch(rslam_filter* f, int step, int min_features, int reference_indexing, const double* u01, int n_pairs, int* status,
                               int* info4) {
    (void)step;
    if (!f || !u01 || !status || n_pairs < kMbMaxAttempts) return fail(RSLAM_ERR_INVALID, "rslam_map_management_batch: bad arguments (u01 and status are required, n_pairs >= %d)", kMbMaxAttempts);
    for (int b = 0; b < f->B; b++)
        if (!f->hF[b].image) return fail(RSLAM_ERR_INVALID, "rslam_map_management_batch: no image is bound to filter %d (rslam_set_image)", b);
    CK(cudaSetDevice(f->device));
    int rc;
    if ((rc = ensure_map_batch_ws(f))) return rc;
    const int B = f->B;
    // inputs: the spare pointers and, from the host, the uniforms, in one copy from pinned staging
    const bool u_dev = is_device_ptr(u01);
    const size_t ptr_bytes = sizeof(double*) * 2 * B, u_bytes = u_dev ? 0 : sizeof(double) * 2 * n_pairs * B;
    if (ptr_bytes + u_bytes > f->mb_in_cap) {
        if (f->mb_h_in) CK(cudaFreeHost(f->mb_h_in));
        if (f->mb_d_in) CK(cudaFree(f->mb_d_in));
        f->mb_h_in = f->mb_d_in = nullptr;
        f->mb_in_cap = 0;
        CK(cudaMallocHost(&f->mb_h_in, ptr_bytes + u_bytes));
        CK(cudaMalloc(&f->mb_d_in, ptr_bytes + u_bytes));
        f->mb_in_cap = ptr_bytes + u_bytes;
    }
    double** hp = (double**)f->mb_h_in;
    for (int b = 0; b < B; b++) {
        hp[b] = f->mb_P[b];
        hp[B + b] = f->mb_x[b];
    }
    if (!u_dev) memcpy((char*)f->mb_h_in + ptr_bytes, u01, u_bytes);
    CK(cudaMemcpyAsync(f->mb_d_in, f->mb_h_in, ptr_bytes + u_bytes, cudaMemcpyHostToDevice, f->stream));
    if (f->descr_dirty && (rc = push_descr(f))) return rc;
    MapBatchWs w = f->mb;
    w.Pdst = (double* const*)f->mb_d_in;
    w.xdst = (double* const*)f->mb_d_in + B;
    w.u01 = u_dev ? u01 : (const double*)((char*)f->mb_d_in + ptr_bytes);
    w.n_pairs = n_pairs;
    const int words = cdiv(f->nmax, 32);
    const int max_add = f->Nmax < kMbMaxAttempts ? f->Nmax : kMbMaxAttempts;
    const int nb = f->hn + 6 * max_add < f->nmax ? f->hn + 6 * max_add : f->nmax;  // bound on every filter's new state dimension
    LAUNCH(f, k_mmb_plan, B, 256, sizeof(unsigned) * 2 * words, f->dF, w, min_features, reference_indexing);
    // initial_rho = 1, std_rho = 1, std_pxl = std_z (src/Map.cpp:216-219), like rslam_map_add_feature
    LAUNCH(f, k_mmb_init, B, 128, 0, f->dF, w, f->camd, 1.0, f->par.std_z, 1.0);
    LAUNCH(f, k_mmb_xform, dim3(cdiv(nb, 256), cdiv(nb, kMbCols), B), 256, 0, f->dF, w);
    if ((rc = check_launch())) return rc;
    // the one read-back: per-filter plans and feature types
    int* hplan = f->mb_h_plan;
    int* htypes = hplan + (size_t)MB_INTS * B;
    CK(cudaMemcpyAsync(hplan, w.plan, sizeof(int) * MB_INTS * B, cudaMemcpyDeviceToHost, f->stream));
    CK(cudaMemcpyAsync(htypes, f->hF[0].ftype, sizeof(int) * (size_t)f->Nmax * B, cudaMemcpyDeviceToHost, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    int first_bad_b = -1;
    for (int b = 0; b < B; b++) {
        const int* pl = hplan + (size_t)MB_INTS * b;
        DevFilter& D = f->hF[b];
        status[b] = pl[MB_STATUS];
        if (info4) {
            info4[4 * b] = pl[MB_DELETED];
            info4[4 * b + 1] = pl[MB_CONVERTED];
            info4[4 * b + 2] = pl[MB_INIT];
            info4[4 * b + 3] = pl[MB_ATTEMPTS];
        }
        if (pl[MB_STATUS] != RSLAM_OK && first_bad_b < 0) first_bad_b = b;
        if (pl[MB_STATUS] == RSLAM_ERR_REFERENCE_UB) continue;
        if (pl[MB_EDIT]) {
            std::swap(D.P, f->mb_P[b]);
            std::swap(D.x_kk, f->mb_x[b]);
        }
        D.N = pl[MB_N];
        D.n = pl[MB_NS];
        const int* t = htypes + (size_t)f->Nmax * b;
        f->htype[b].assign(t, t + D.N);
    }
    f->hN = 0;
    f->hn = 0;
    for (int k = 0; k < B; k++) {
        f->hN = f->hF[k].N > f->hN ? f->hF[k].N : f->hN;
        f->hn = f->hF[k].n > f->hn ? f->hF[k].n : f->hn;
    }
    if ((rc = push_descr(f))) return rc;
    if (first_bad_b < 0) return RSLAM_OK;
    return fail(status[first_bad_b], "rslam_map_management_batch: filter %d (the first of those that failed) returned %d", first_bad_b, status[first_bad_b]);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------------
// Checkpoint / resume of whole filters (kernels_ckpt.cuh; the snapshot format is documented in include/rslam.h)
// ---------------------------------------------------------------------------------------------------------------------
namespace {
constexpr size_t kCkHeader = 160, kCkEntry = 32, kCkStageMax = (size_t)256 << 20;
constexpr uint32_t kCkVersion = 1;
const char kCkMagic[8] = {'R', 'S', 'L', 'A', 'M', 'C', 'K', 'P'};

// camera and params at their fixed offsets (bytes 24..159 of the header; the library only builds for little-endian hosts)
void ck_put_config(const rslam_filter* f, unsigned char* h) {
    auto pd = [h](size_t o, double v) { memcpy(h + o, &v, 8); };
    auto pi = [h](size_t o, int32_t v) { memcpy(h + o, &v, 4); };
    memset(h + 24, 0, kCkHeader - 24);
    const rslam_camera& c = f->cam;
    const rslam_params& p = f->par;
    pd(24, c.k1), pd(32, c.k2), pi(40, c.nRows), pi(44, c.nCols), pd(48, c.Cx), pd(56, c.Cy), pd(64, c.f), pd(72, c.dx), pd(80, c.dy);
    pd(88, p.std_a), pd(96, p.std_alpha), pd(104, p.std_z), pd(112, p.chi2_095_2), pd(120, p.corr_threshold), pd(128, p.p_spurious_free);
    pi(136, p.n_hyp_initial), pd(144, p.max_ellipse_eig), pi(152, (int32_t)p.quirks), pi(156, p.dedupe_hypotheses);
}

// where everything of a snapshot of filters with these n / N lies
struct CkLayout {
    std::vector<int> n, N;
    std::vector<size_t> types_off, block_off;
    size_t dir_bytes = 0, total = 0;
    void build() {
        const size_t count = n.size();
        types_off.resize(count);
        block_off.resize(count);
        size_t o = kCkHeader + kCkEntry * count;
        for (size_t i = 0; i < count; i++) {
            types_off[i] = o;
            o += ck_al16(4 * (size_t)N[i]);
        }
        dir_bytes = o;
        for (size_t i = 0; i < count; i++) {
            block_off[i] = o;
            o += ck_rec_bytes(n[i], N[i]) + ck_tri_bytes(n[i]);
        }
        total = o;
    }
};

// header, filter table and feature types of filters [b, b + count) (from the host mirror)
void ck_put_directory(const rslam_filter* f, const CkLayout& L, int b, unsigned char* h) {
    memset(h, 0, L.dir_bytes);
    memcpy(h, kCkMagic, 8);
    const uint32_t ver = kCkVersion, cnt = (uint32_t)L.n.size();
    const uint64_t tot = L.total;
    memcpy(h + 8, &ver, 4);
    memcpy(h + 12, &cnt, 4);
    memcpy(h + 16, &tot, 8);
    ck_put_config(f, h);
    for (size_t i = 0; i < L.n.size(); i++) {
        unsigned char* e = h + kCkHeader + kCkEntry * i;
        const uint64_t bo = L.block_off[i], to = L.types_off[i];
        memcpy(e, &bo, 8);
        memcpy(e + 8, &to, 8);
        memcpy(e + 16, &L.n[i], 4);
        memcpy(e + 20, &L.N[i], 4);
        if (L.N[i]) memcpy(h + L.types_off[i], f->htype[b + i].data(), 4 * (size_t)L.N[i]);
    }
}

// Consecutive pieces of the stream of filter blocks, each at most `cap` bytes: a filter's records, or a range of whole 64-column
// tile columns of its triangle; with the work items of each piece (records and lower tiles, offsets relative to the piece)
struct CkChunk {
    size_t off, bytes;
    int rec0, nrec, tile0, ntile;
};
struct CkPlan {
    std::vector<CkptRec> recs;
    std::vector<CkptTile> tiles;
    std::vector<CkChunk> chunks;
    size_t max_chunk = 0;
};
int ck_plan(const CkLayout& L, int b, size_t cap, CkPlan& p) {
    CkChunk cur{L.dir_bytes, 0, 0, 0, 0, 0};
    auto close = [&](size_t start) {
        if (cur.bytes) {
            p.chunks.push_back(cur);
            p.max_chunk = cur.bytes > p.max_chunk ? cur.bytes : p.max_chunk;
        }
        cur = CkChunk{start, 0, (int)p.recs.size(), 0, (int)p.tiles.size(), 0};
    };
    for (size_t i = 0; i < L.n.size(); i++) {
        const long long n = L.n[i];
        const size_t rb = ck_rec_bytes(n, L.N[i]), pstart = L.block_off[i] + rb;
        if (rb > cap) return fail(RSLAM_ERR_CAPACITY, "checkpoint: the records of one filter (%zu bytes) exceed the %zu-byte staging buffer", rb, cap);
        if (cur.bytes && pstart - cur.off > cap) close(L.block_off[i]);
        p.recs.push_back(CkptRec{b + (int)i, (int)n, L.N[i], 0, (long long)(L.block_off[i] - cur.off)});
        cur.nrec++;
        cur.bytes = pstart - cur.off;
        const int T = cdiv((int)n, kCkTile);
        for (int J = 0; J < T; J++) {
            const long long j0 = (long long)kCkTile * J, j1 = j0 + kCkTile < n ? j0 + kCkTile : n;
            const size_t s = pstart + 8 * (size_t)ck_colstart(j0, n);
            const size_t e = J == T - 1 ? pstart + ck_tri_bytes(n) : pstart + 8 * (size_t)ck_colstart(j1, n);
            if (e - s > cap) return fail(RSLAM_ERR_CAPACITY, "checkpoint: one tile column (%zu bytes) exceeds the %zu-byte staging buffer", e - s, cap);
            if (cur.bytes && e - cur.off > cap) close(s);  // s is 16-byte aligned: the column start of a 64-column boundary is even
            const long long pbase = ((long long)pstart - (long long)cur.off) / 8;
            for (int I = J; I < T; I++) p.tiles.push_back(CkptTile{b + (int)i, (int)n, I, J, pbase});
            cur.ntile += T - J;
            cur.bytes = e - cur.off;
        }
    }
    close(0);
    return 0;
}

// 1: device memory on the handle's GPU, 0: host memory, -1: device memory of another GPU
int ck_where(const rslam_filter* f, const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) return 0;
    return at.device == f->device ? 1 : -1;
}

int ck_grow(rslam_filter* f, unsigned char** p, size_t* cap, size_t need) {
    if (need <= *cap) return 0;
    if (*p) {
        CK(cudaStreamSynchronize(f->stream));
        CK(cudaFree(*p));
    }
    *p = nullptr;
    *cap = 0;
    CK(cudaMalloc((void**)p, need));
    *cap = need;
    return 0;
}

// the work lists of a plan on the device, followed by `count` zeroed symmetry flags
int ck_push_lists(rslam_filter* f, const CkPlan& p, int count, CkptRec** drec, CkptTile** dtile, int** dbad) {
    const size_t rb = sizeof(CkptRec) * p.recs.size(), tb = sizeof(CkptTile) * p.tiles.size();
    int rc = ck_grow(f, &f->ck_list, &f->ck_list_cap, rb + tb + sizeof(int) * count + 16);
    if (rc) return rc;
    std::vector<unsigned char> h(rb + tb);
    if (rb) memcpy(h.data(), p.recs.data(), rb);
    if (tb) memcpy(h.data() + rb, p.tiles.data(), tb);
    // pageable source: staged before the call returns, so the vector may go
    CK(cudaMemcpyAsync(f->ck_list, h.data(), rb + tb, cudaMemcpyHostToDevice, f->stream));
    CK(cudaMemsetAsync(f->ck_list + rb + tb, 0, sizeof(int) * count, f->stream));
    *drec = (CkptRec*)f->ck_list;
    *dtile = (CkptTile*)(f->ck_list + rb);
    *dbad = (int*)(f->ck_list + rb + tb);
    return 0;
}

int ck_range(rslam_filter* f, int b, int count, CkLayout& L, const char* who) {
    if (!f || b < 0 || count < 1 || count > f->B - b) return fail(RSLAM_ERR_INVALID, "%s: filters [%d, %d + %d) are not in the handle", who, b, b, count);
    for (int i = 0; i < count; i++) {
        L.n.push_back(f->hF[b + i].n);
        L.N.push_back(f->hF[b + i].N);
    }
    L.build();
    return 0;
}
}  // namespace

extern "C" {

int rslam_checkpoint_bytes(rslam_filter* f, int b, int count, size_t* bytes) {
    CkLayout L;
    int rc = ck_range(f, b, count, L, "rslam_checkpoint_bytes");
    if (rc) return rc;
    if (!bytes) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_bytes: bytes is NULL");
    *bytes = L.total;
    return RSLAM_OK;
}

int rslam_checkpoint_save(rslam_filter* f, int b, int count, void* dst, size_t cap, size_t* written) {
    CkLayout L;
    int rc = ck_range(f, b, count, L, "rslam_checkpoint_save");
    if (rc) return rc;
    if (!dst) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_save: dst is NULL");
    CK(cudaSetDevice(f->device));
    const int where = ck_where(f, dst);
    if (where < 0) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_save: dst is device memory of another GPU than the handle's (%d)", f->device);
    if (where == 1 && ((uintptr_t)dst & 15)) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_save: device dst must be 16-byte aligned");
    if (cap < L.total) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_save: cap = %zu bytes, the snapshot needs %zu", cap, L.total);
    const bool dev = where == 1;
    CkPlan p;
    if ((rc = ck_plan(L, b, dev ? (size_t)-1 : kCkStageMax, p))) return rc;
    if (!dev && (rc = ck_grow(f, &f->ck_stage, &f->ck_stage_cap, p.max_chunk))) return rc;
    if (f->descr_dirty && (rc = push_descr(f))) return rc;
    CkptRec* drec;
    CkptTile* dtile;
    int* dbad;
    if ((rc = ck_push_lists(f, p, count, &drec, &dtile, &dbad))) return rc;
    std::vector<unsigned char> dir(L.dir_bytes);
    ck_put_directory(f, L, b, dir.data());
    if (dev)
        CK(cudaMemcpyAsync(dst, dir.data(), L.dir_bytes, cudaMemcpyHostToDevice, f->stream));
    else
        memcpy(dst, dir.data(), L.dir_bytes);
    for (const CkChunk& c : p.chunks) {
        unsigned char* base = dev ? (unsigned char*)dst + c.off : f->ck_stage;
        if (c.nrec) LAUNCH(f, k_ckpt_records_pack, dim3(c.nrec, kCkSegs), 256, 0, f->dF, drec + c.rec0, base);
        if (c.ntile) LAUNCH(f, k_ckpt_pack, c.ntile, 256, 0, f->dF, dtile + c.tile0, (double*)base, dbad, b);
        if ((rc = check_launch())) return rc;
        if (!dev) CK(cudaMemcpyAsync((unsigned char*)dst + c.off, f->ck_stage, c.bytes, cudaMemcpyDeviceToHost, f->stream));
    }
    std::vector<int> bad(count);
    CK(cudaMemcpyAsync(bad.data(), dbad, sizeof(int) * count, cudaMemcpyDeviceToHost, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    for (int i = 0; i < count; i++)
        if (bad[i]) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_save: P of filter %d is not exactly symmetric (bitwise)", b + i);
    if (written) *written = L.total;
    return RSLAM_OK;
}

int rslam_checkpoint_load(rslam_filter* f, int b, const void* src, size_t bytes, int* count_out) {
    if (!f || !src) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: bad arguments");
    CK(cudaSetDevice(f->device));
    const int where = ck_where(f, src);
    if (where < 0) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: src is device memory of another GPU than the handle's (%d)", f->device);
    if (where == 1 && ((uintptr_t)src & 15)) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: device src must be 16-byte aligned");
    const bool dev = where == 1;
    // everything is validated on the host before the first device write
    auto fetch = [&](void* h, size_t off, size_t len) -> int {
        if (!dev) {
            memcpy(h, (const unsigned char*)src + off, len);
            return 0;
        }
        CK(cudaMemcpyAsync(h, (const unsigned char*)src + off, len, cudaMemcpyDeviceToHost, f->stream));
        CK(cudaStreamSynchronize(f->stream));
        return 0;
    };
    int rc;
    if (bytes < kCkHeader) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: %zu bytes is shorter than the header", bytes);
    unsigned char hdr[kCkHeader], mine[kCkHeader];
    if ((rc = fetch(hdr, 0, kCkHeader))) return rc;
    if (memcmp(hdr, kCkMagic, 8)) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: not a snapshot (bad magic)");
    uint32_t ver, cnt;
    uint64_t tot;
    memcpy(&ver, hdr + 8, 4);
    memcpy(&cnt, hdr + 12, 4);
    memcpy(&tot, hdr + 16, 8);
    if (ver != kCkVersion) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: format version %u, this library reads %u", ver, kCkVersion);
    if (tot != bytes) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: the snapshot is %llu bytes, the buffer %zu", (unsigned long long)tot, bytes);
    ck_put_config(f, mine);
    if (memcmp(hdr + 24, mine + 24, kCkHeader - 24)) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: camera or params differ from the handle's");
    if (cnt < 1 || b < 0 || (long long)b + cnt > f->B) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: %u filters do not fit at slot %d of a batch of %d", cnt, b, f->B);
    const int count = (int)cnt;
    if (kCkHeader + kCkEntry * (size_t)count > bytes) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: truncated filter table");
    std::vector<unsigned char> tab(kCkEntry * (size_t)count);
    if ((rc = fetch(tab.data(), kCkHeader, tab.size()))) return rc;
    CkLayout L;
    for (int i = 0; i < count; i++) {
        int n, N;
        memcpy(&n, &tab[kCkEntry * i + 16], 4);
        memcpy(&N, &tab[kCkEntry * i + 20], 4);
        if (N < 0 || N > (1 << 24) || n < 13 + 3 * N || n > 13 + 6 * N) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: filter %d has n = %d, N = %d", i, n, N);
        L.n.push_back(n);
        L.N.push_back(N);
    }
    L.build();
    if (L.total != bytes) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: the filter table describes %zu bytes, the buffer holds %zu", L.total, bytes);
    for (int i = 0; i < count; i++) {
        uint64_t bo, to;
        memcpy(&bo, &tab[kCkEntry * i], 8);
        memcpy(&to, &tab[kCkEntry * i + 8], 8);
        if (bo != L.block_off[i] || to != L.types_off[i]) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: filter %d is not where the table says", i);
    }
    const size_t t0 = kCkHeader + kCkEntry * (size_t)count;
    std::vector<unsigned char> traw(L.dir_bytes - t0);
    if (!traw.empty() && (rc = fetch(traw.data(), t0, traw.size()))) return rc;
    std::vector<std::vector<int>> types(count);
    for (int i = 0; i < count; i++) {
        types[i].resize(L.N[i]);
        if (L.N[i]) memcpy(types[i].data(), traw.data() + (L.types_off[i] - t0), 4 * (size_t)L.N[i]);
        int n = 13;
        for (int t : types[i]) {
            if (t != 0 && t != 1) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: filter %d has a feature type %d", i, t);
            n += t == 0 ? 6 : 3;
        }
        if (n != L.n[i]) return fail(RSLAM_ERR_INVALID, "rslam_checkpoint_load: filter %d has n = %d, but 13 + sum(feature sizes) = %d", i, L.n[i], n);
    }
    for (int i = 0; i < count; i++)
        if (L.N[i] > f->Nmax) return fail(RSLAM_ERR_CAPACITY, "rslam_checkpoint_load: filter %d has %d features > max_features %d", i, L.N[i], f->Nmax);
    CkPlan p;
    if ((rc = ck_plan(L, b, dev ? (size_t)-1 : kCkStageMax, p))) return rc;
    if (!dev && (rc = ck_grow(f, &f->ck_stage, &f->ck_stage_cap, p.max_chunk))) return rc;
    // device writes from here on
    if (f->descr_dirty && (rc = push_descr(f))) return rc;
    CkptRec* drec;
    CkptTile* dtile;
    int* dbad;
    if ((rc = ck_push_lists(f, p, count, &drec, &dtile, &dbad))) return rc;
    for (const CkChunk& c : p.chunks) {
        const unsigned char* base = dev ? (const unsigned char*)src + c.off : f->ck_stage;
        if (!dev) CK(cudaMemcpyAsync(f->ck_stage, (const unsigned char*)src + c.off, c.bytes, cudaMemcpyHostToDevice, f->stream));
        if (c.nrec) LAUNCH(f, k_ckpt_records_unpack, dim3(c.nrec, kCkSegs - 1), 256, 0, f->dF, drec + c.rec0, base, f->nmax, f->Nmax);
        if (c.ntile) LAUNCH(f, k_ckpt_unpack, c.ntile, 256, 0, f->dF, dtile + c.tile0, (const double*)base);
        if ((rc = check_launch())) return rc;
    }
    // feature types, offsets and last inverse-depth index as rslam_upload_state builds them, cleared past N; the slots' arrays are
    // consecutive pieces (stride max_features) of one allocation each, as are their RANSAC control blocks, cleared here
    const size_t per = (size_t)f->Nmax;
    std::vector<int> ht(per * count * 3, 0);
    int* hty = ht.data();
    int* hof = hty + per * count;
    int* hli = hof + per * count;
    for (int i = 0; i < count; i++)
        for (int k = 0, off = 13, last = -1; k < L.N[i]; k++) {
            const int t = types[i][k];
            if (t == 0) last = k;
            hty[per * i + k] = t;
            hof[per * i + k] = off;
            hli[per * i + k] = last;
            off += t == 0 ? 6 : 3;
        }
    const DevFilter& D0 = f->hF[b];
    CK(cudaMemcpyAsync(D0.ftype, hty, sizeof(int) * per * count, cudaMemcpyHostToDevice, f->stream));
    CK(cudaMemcpyAsync(D0.foff, hof, sizeof(int) * per * count, cudaMemcpyHostToDevice, f->stream));
    CK(cudaMemcpyAsync(D0.last_id, hli, sizeof(int) * per * count, cudaMemcpyHostToDevice, f->stream));
    CK(cudaMemsetAsync(D0.ctl, 0, sizeof(int) * CTL_SIZE * count, f->stream));
    CK(cudaStreamSynchronize(f->stream));
    for (int i = 0; i < count; i++) {
        DevFilter& D = f->hF[b + i];
        D.n = L.n[i];
        D.N = L.N[i];
        f->htype[b + i] = types[i];
    }
    f->hN = 0;
    f->hn = 0;
    for (int k = 0; k < f->B; k++) {
        f->hN = f->hF[k].N > f->hN ? f->hF[k].N : f->hN;
        f->hn = f->hF[k].n > f->hn ? f->hF[k].n : f->hn;
    }
    if ((rc = push_descr(f))) return rc;
    if (count_out) *count_out = count;
    return RSLAM_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------------
// The sweep sharded over GPUs (SURVEY 8e): NCCL inside the library.  libnccl.so.2 is opened at run time (a process that already
// carries an NCCL -- e.g. torch's -- gets that same copy by soname), so the library itself has no link-time dependency on it.
// ---------------------------------------------------------------------------------------------------------------------
namespace {
typedef struct ncclComm* nccl_comm_t;
struct nccl_uid {
    char internal[128];
};
enum { kNcclUint32 = 3, kNcclUint64 = 5, kNcclMax = 2 };  // ncclDataType_t / ncclRedOp_t values of nccl.h (stable since NCCL 2.0)
struct NcclApi {
    void* so = nullptr;
    int (*GetUniqueId)(nccl_uid*) = nullptr;
    int (*CommInitRank)(nccl_comm_t*, int, nccl_uid, int) = nullptr;
    int (*CommInitAll)(nccl_comm_t*, int, const int*) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    int (*GetVersion)(int*) = nullptr;
};
NcclApi g_nccl;
int nccl_load() {
    if (g_nccl.so) return 0;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    void* so = nullptr;
    for (const char* nm : names)
        if ((so = dlopen(nm, RTLD_NOW | RTLD_GLOBAL))) break;
    if (!so) return fail(RSLAM_ERR_CUDA, "rslam_comm: cannot load libnccl.so.2 (%s)", dlerror());
#define SYM(field, name)                                                                           \
    *(void**)(&g_nccl.field) = dlsym(so, name);                                                    \
    if (!g_nccl.field) return fail(RSLAM_ERR_CUDA, "rslam_comm: libnccl has no symbol %s", name);
    SYM(GetUniqueId, "ncclGetUniqueId")
    SYM(CommInitRank, "ncclCommInitRank")
    SYM(CommInitAll, "ncclCommInitAll")
    SYM(CommDestroy, "ncclCommDestroy")
    SYM(AllReduce, "ncclAllReduce")
    SYM(GroupStart, "ncclGroupStart")
    SYM(GroupEnd, "ncclGroupEnd")
    SYM(GetErrorString, "ncclGetErrorString")
    SYM(GetVersion, "ncclGetVersion")
#undef SYM
    g_nccl.so = so;
    return 0;
}
#define NCK(call)                                                                                                                       \
    do {                                                                                                                                \
        int r__ = (call);                                                                                                               \
        if (r__ != 0) return fail(RSLAM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, g_nccl.GetErrorString(r__), __FILE__, __LINE__);      \
    } while (0)
}  // namespace

struct rslam_comm {
    int nranks = 0, rank0 = 0, nlocal = 0;
    std::vector<int> devs;
    std::vector<nccl_comm_t> comms;
    std::vector<unsigned long long*> d_key;  // all-reduced key per local GPU
    std::vector<unsigned*> d_words;          // winner's mask words per local GPU
    std::vector<int> words_cap;
};

extern "C" {

int rslam_comm_unique_id(void* id128) {
    if (!id128) return fail(RSLAM_ERR_INVALID, "rslam_comm_unique_id: null buffer");
    int rc = nccl_load();
    if (rc) return rc;
    nccl_uid id;
    NCK(g_nccl.GetUniqueId(&id));
    memcpy(id128, &id, sizeof(id));
    return RSLAM_OK;
}

static int comm_alloc_buffers(rslam_comm* c) {
    c->d_key.assign(c->nlocal, nullptr);
    c->d_words.assign(c->nlocal, nullptr);
    c->words_cap.assign(c->nlocal, 0);
    for (int i = 0; i < c->nlocal; i++) {
        CK(cudaSetDevice(c->devs[i]));
        CK(cudaMalloc((void**)&c->d_key[i], 2 * sizeof(unsigned long long)));
        CK(cudaMemset(c->d_key[i], 0, 2 * sizeof(unsigned long long)));
    }
    return 0;
}

int rslam_comm_init(int ndev, const int* devs, rslam_comm** out) {
    if (ndev < 1 || !out) return fail(RSLAM_ERR_INVALID, "rslam_comm_init: bad arguments");
    int have = 0;
    if (cudaGetDeviceCount(&have) != cudaSuccess || have < ndev) {
        cudaGetLastError();
        return fail(RSLAM_ERR_CUDA, "rslam_comm_init: %d GPUs requested, %d visible", ndev, have);
    }
    int rc = nccl_load();
    if (rc) return rc;
    rslam_comm* c = new rslam_comm();
    c->nranks = c->nlocal = ndev;
    c->rank0 = 0;
    for (int i = 0; i < ndev; i++) c->devs.push_back(devs ? devs[i] : i);
    c->comms.assign(ndev, nullptr);
    int r = g_nccl.CommInitAll(c->comms.data(), ndev, c->devs.data());
    if (r != 0) {
        delete c;
        return fail(RSLAM_ERR_CUDA, "ncclCommInitAll failed: %s", g_nccl.GetErrorString(r));
    }
    if ((rc = comm_alloc_buffers(c))) {
        rslam_comm_destroy(c);
        return rc;
    }
    *out = c;
    return RSLAM_OK;
}

int rslam_comm_init_rank(int nranks, int rank, const void* id128, int device, rslam_comm** out) {
    if (nranks < 1 || rank < 0 || rank >= nranks || !id128 || !out) return fail(RSLAM_ERR_INVALID, "rslam_comm_init_rank: bad arguments");
    int rc = nccl_load();
    if (rc) return rc;
    CK(cudaSetDevice(device));
    rslam_comm* c = new rslam_comm();
    c->nranks = nranks;
    c->rank0 = rank;
    c->nlocal = 1;
    c->devs.push_back(device);
    c->comms.assign(1, nullptr);
    nccl_uid id;
    memcpy(&id, id128, sizeof(id));
    int r = g_nccl.CommInitRank(&c->comms[0], nranks, id, rank);
    if (r != 0) {
        delete c;
        return fail(RSLAM_ERR_CUDA, "ncclCommInitRank failed: %s", g_nccl.GetErrorString(r));
    }
    if ((rc = comm_alloc_buffers(c))) {
        rslam_comm_destroy(c);
        return rc;
    }
    *out = c;
    return RSLAM_OK;
}

int rslam_comm_destroy(rslam_comm* c) {
    if (!c) return RSLAM_OK;
    for (int i = 0; i < c->nlocal; i++) {
        cudaSetDevice(c->devs[i]);
        if (i < (int)c->d_key.size() && c->d_key[i]) cudaFree(c->d_key[i]);
        if (i < (int)c->d_words.size() && c->d_words[i]) cudaFree(c->d_words[i]);
        if (c->comms[i] && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comms[i]);
    }
    delete c;
    return RSLAM_OK;
}
int rslam_comm_size(const rslam_comm* c) { return c ? c->nranks : -1; }
int rslam_comm_local_size(const rslam_comm* c) { return c ? c->nlocal : -1; }

int rslam_support_sweep_multi(rslam_comm* c, rslam_filter* const* filters, const int* hyp_match_idx, int n_hyp, int shard, uint64_t* best_key,
                              uint8_t* best_mask, long long* n_pairs_scored) {
    if (!c || !filters || !hyp_match_idx || n_hyp <= 0 || !best_key || (shard != RSLAM_SHARD_BY_HYPOTHESIS && shard != RSLAM_SHARD_BY_MATCH))
        return fail(RSLAM_ERR_INVALID, "rslam_support_sweep_multi: bad arguments");
    const int L = c->nlocal, G = c->nranks;
    const bool key_on_device = is_device_ptr(best_key);
    if (key_on_device && L != 1) return fail(RSLAM_ERR_INVALID, "rslam_support_sweep_multi: a device best_key needs exactly one local GPU");
    for (int i = 0; i < L; i++) {
        if (!filters[i] || filters[i]->device != c->devs[i] || filters[i]->B != 1)
            return fail(RSLAM_ERR_INVALID, "rslam_support_sweep_multi: filters[%d] must be a batch-1 handle on device %d", i, c->devs[i]);
        if (filters[i]->hN != filters[0]->hN) return fail(RSLAM_ERR_INVALID, "rslam_support_sweep_multi: the replicas hold different maps");
    }
    const int N = filters[0]->hN;
    int rc;
    std::vector<const int*> d_idx(L, nullptr);
    std::vector<int> h0(L), h1(L), t0(L), t1(L);
    for (int i = 0; i < L; i++) {
        rslam_filter* f = filters[i];
        CK(cudaSetDevice(f->device));
        const long long r = c->rank0 + i;
        if (shard == RSLAM_SHARD_BY_HYPOTHESIS) {
            h0[i] = (int)(r * n_hyp / G);
            h1[i] = (int)((r + 1) * n_hyp / G);
            t0[i] = 0;
            t1[i] = N;
        } else {
            h0[i] = 0;
            h1[i] = n_hyp;
            t0[i] = (int)(r * N / G);
            t1[i] = (int)((r + 1) * N / G);
        }
        if ((rc = sweep_local(f, hyp_match_idx, n_hyp, h0[i], h1[i], t0[i], t1[i], &d_idx[i]))) return rc;
    }
    NCK(g_nccl.GroupStart());
    for (int i = 0; i < L; i++) {
        int r = g_nccl.AllReduce(filters[i]->d_key, c->d_key[i], 1, kNcclUint64, kNcclMax, c->comms[i], filters[i]->stream);
        if (r != 0) {
            g_nccl.GroupEnd();
            return fail(RSLAM_ERR_CUDA, "ncclAllReduce(key) failed: %s", g_nccl.GetErrorString(r));
        }
    }
    NCK(g_nccl.GroupEnd());
    const int nwords = filters[0]->mwords;
    if (best_mask) {
        for (int i = 0; i < L; i++) {
            rslam_filter* f = filters[i];
            CK(cudaSetDevice(f->device));
            if (c->words_cap[i] < nwords) {
                if (c->d_words[i]) CK(cudaFree(c->d_words[i]));
                c->d_words[i] = nullptr;
                CK(cudaMalloc((void**)&c->d_words[i], sizeof(unsigned) * (size_t)nwords));
                c->words_cap[i] = nwords;
            }
            LAUNCH(f, k_sweep_winner_mask, cdiv(nwords, 256), 256, 0, f->dF, (const unsigned long long*)c->d_key[i], d_idx[i], h0[i], h1[i], t0[i], t1[i], c->d_words[i], nwords);
        }
        if ((rc = check_launch())) return rc;
        NCK(g_nccl.GroupStart());
        for (int i = 0; i < L; i++) {
            int r = g_nccl.AllReduce(c->d_words[i], c->d_words[i], (size_t)nwords, kNcclUint32, kNcclMax, c->comms[i], filters[i]->stream);
            if (r != 0) {
                g_nccl.GroupEnd();
                return fail(RSLAM_ERR_CUDA, "ncclAllReduce(mask) failed: %s", g_nccl.GetErrorString(r));
            }
        }
        NCK(g_nccl.GroupEnd());
    }
    CK(cudaSetDevice(filters[0]->device));
    CK(cudaMemcpyAsync(best_key, c->d_key[0], sizeof(uint64_t), cudaMemcpyDefault, filters[0]->stream));
    if (key_on_device && !best_mask && !n_pairs_scored) return RSLAM_OK;  // enqueue only
    std::vector<unsigned> words;
    if (best_mask) {
        words.resize(nwords);
        CK(cudaMemcpyAsync(words.data(), c->d_words[0], sizeof(unsigned) * (size_t)nwords, cudaMemcpyDeviceToHost, filters[0]->stream));
    }
    long long pairs = 0;
    for (int i = 0; i < L; i++) {
        CK(cudaSetDevice(filters[i]->device));
        CK(cudaStreamSynchronize(filters[i]->stream));
        if (n_pairs_scored) {
            unsigned long long cnt = 0;
            CK(cudaMemcpy(&cnt, filters[i]->d_key + 1, sizeof(cnt), cudaMemcpyDeviceToHost));
            pairs += (long long)cnt;
        }
    }
    if (n_pairs_scored) *n_pairs_scored = pairs;
    if (best_mask) {
        int ctl[CTL_SIZE];
        CK(cudaSetDevice(filters[0]->device));
        CK(cudaMemcpy(ctl, filters[0]->hF[0].ctl, sizeof(ctl), cudaMemcpyDeviceToHost));
        const int m = ctl[CTL_MID];
        memset(best_mask, 0, (size_t)(m + 7) / 8);
        for (int j = 0; j < m; j++)
            if ((words[j >> 5] >> (j & 31)) & 1u) best_mask[j >> 3] |= (uint8_t)(1u << (j & 7));
    }
    return RSLAM_OK;
}

}  // extern "C"
