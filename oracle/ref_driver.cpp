// ref_driver.cpp -- C entry points around the REFERENCE'S OWN classes.  TEST INFRASTRUCTURE (oracle/).
//
// oracle/_ref/libref.so = the reference's hot-path translation units, compiled UNMODIFIED from where they lie
// (/root/reference/src/{ExtendKF,Tracking,Converter,Map}.cpp against /root/reference/include), plus this driver.  Their third-party
// headers (Eigen, OpenCV, ROS, Boost) do not exist in this image, so the build points the compiler at oracle/ref_shim/ instead:
// stand-ins written for this repository (mini_eigen.h, mini_cv.h, empty ROS types).  What this pins: every line of the reference's
// own algorithm -- index arithmetic, stacking order, quirks, control flow -- is the reference's.  What it does not pin: the arithmetic
// INSIDE Eigen / OpenCV (LU pivot order, product summation order, remap rounding), which is the stand-ins' restatement (cv2-pinned for
// the OpenCV primitives).  The restated oracle (rslam_oracle.cpp) and the CUDA path are tested against this library.
//
// src/System.cpp (the ROS node) is not compiled; the two pieces of it that belong to the path are replayed here:
//   * System::System's camera set-up and object construction        (src/System.cpp:22-70)
//   * System::TrackRunning's seven-call frame sequence               (src/System.cpp:103-129)
// libc rand()/srand() are redirected at link time (-Wl,--wrap) to a caller-supplied queue so that tests feed the same draws to the
// reference (ExtendKF::rand, src/ExtendKF.cpp:220-235: t = rand() / RAND_MAX) and to the oracle / CUDA path (u01 = r / RAND_MAX).
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <ctime>
#include <vector>

#include "ransac_slam/System.h"

namespace {
std::vector<int> g_rand;
size_t g_rand_pos = 0;
long g_rand_underflow = 0;
}  // namespace

// A frame of configuration C3 (2000 features) costs the reference ~9000 dense hypotheses; the bench times a BOUNDED number of them by
// leaving Tracking::ransac_hypotheses through the draw that would start hypothesis number budget + 1.  libc declares rand() nothrow,
// so the exit is a longjmp (the loop's Eigen temporaries of that one call are not destructed: a few MB per sample, timing runs only).
#include <csetjmp>
namespace {
long g_rand_budget = -1;
std::jmp_buf g_rand_jmp;
}  // namespace
extern "C" int __wrap_rand(void) {
    if (g_rand_budget >= 0 && (long)g_rand_pos >= g_rand_budget) std::longjmp(g_rand_jmp, 1);
    if (g_rand_pos < g_rand.size()) return g_rand[g_rand_pos++];
    g_rand_underflow++;
    return 0;
}
extern "C" void __wrap_srand(unsigned) {}  // ExtendKF::ExtendKF seeds from time(NULL) (src/ExtendKF.cpp:25): draws come from the queue instead

namespace {
using namespace ransac_slam;
struct Ref {
    CamParam cam;
    ExtendKF* kf = nullptr;
    Map* map = nullptr;
    Tracking* trk = nullptr;
    long long steps = 0;
};
cv::Mat wrap_image(const uint8_t* img, int rows, int cols, int stride) {
    cv::Mat borrowed(rows, cols, CV_8U, (void*)img, (size_t)stride);
    return borrowed.clone();  // System::takeImage clones the grey image (src/System.cpp:140-152)
}
}  // namespace

extern "C" {
void ref_set_rand(const int* r, int n) {
    g_rand.assign(r, r + n);
    g_rand_pos = 0;
    g_rand_underflow = 0;
}
int ref_rand_consumed(void) { return (int)g_rand_pos; }
int ref_rand_underflow(void) { return (int)g_rand_underflow; }
int ref_rand_max(void) { return RAND_MAX; }

// System::System (src/System.cpp:22-70) without the ROS topic set-up
void* ref_create(const char* yaml_path) {
    cv::FileStorage fs;
    fs.open(yaml_path, cv::FileStorage::READ);
    if (!fs.isOpened()) return nullptr;
    Ref* R = new Ref();
    CamParam& cam = R->cam;
    cam.k1 = (double)fs["Camera.k1"];
    cam.k2 = (double)fs["Camera.k2"];
    cam.nRows = (double)fs["Camera.nRows"];
    cam.nCols = (double)fs["Camera.nCols"];
    double d = (double)fs["Camera.d"];
    cam.Cx = (double)fs["Camera.cx_d"] / d;
    cam.Cy = (double)fs["Camera.cy_d"] / d;
    cam.f = (double)fs["Camera.fps"];
    cam.dx = (double)fs["Camera.dx"];
    cam.dy = (double)fs["Camera.dy"];
    cam.model = (std::string)fs["Camera.model"];
    cam.K << (cam.f / d), 0, cam.Cx, 0, (cam.f / d), cam.Cy, 0, 0, 1;
    int min_features = (int)fs["min_number_of_features_in_image"];
    R->kf = new ExtendKF(yaml_path, &R->cam, "constant_velocity");
    R->kf->initialize_x_and_p();
    R->map = new Map(min_features, R->kf);
    R->trk = new Tracking(yaml_path, R->kf);
    R->steps = 0;
    return R;
}
void ref_destroy(void* h) {
    Ref* R = (Ref*)h;
    if (!R) return;
    delete R->trk;
    delete R->map;
    delete R->kf;
    delete R;
}
void ref_get_camera(void* h, double* cam9) {  // (k1, k2, nRows, nCols, Cx, Cy, f, dx, dy)
    const CamParam& c = ((Ref*)h)->cam;
    const double v[9] = {c.k1, c.k2, (double)c.nRows, (double)c.nCols, c.Cx, c.Cy, c.f, c.dx, c.dy};
    std::memcpy(cam9, v, sizeof(v));
}
void ref_get_params(void* h, double* p7) {  // std_a, std_alpha, std_z, v_0, std_v_0, w_0, std_w_0
    ExtendKF* k = ((Ref*)h)->kf;
    const double v[7] = {k->std_a, k->std_alpha, k->std_z, k->v_0, k->std_v_0, k->w_0, k->std_w_0};
    std::memcpy(p7, v, sizeof(v));
}

// ---- the frame, as System::TrackRunning calls it (src/System.cpp:103-129) --------------------------------------------------------
void ref_track_running(void* h, const uint8_t* img, int rows, int cols, int stride) {
    Ref* R = (Ref*)h;
    cv::Mat image = wrap_image(img, rows, cols, stride);
    R->steps++;
    R->map->map_management(image, R->steps);
    R->kf->ekf_prediction();
    R->trk->search_IC_matches(image);
    R->trk->ransac_hypotheses();
    R->kf->ekf_update_li_inliers();
    R->trk->rescue_hi_inliers();
    R->kf->ekf_update_hi_inliers();
}
// ---- the same calls one at a time (stage-level comparisons) ------------------------------------------------------------------------
void ref_map_management(void* h, const uint8_t* img, int rows, int cols, int stride, int step) {
    Ref* R = (Ref*)h;
    R->steps = step;
    R->map->map_management(wrap_image(img, rows, cols, stride), step);
}
void ref_ekf_prediction(void* h) { ((Ref*)h)->kf->ekf_prediction(); }
void ref_search_ic_matches(void* h, const uint8_t* img, int rows, int cols, int stride) {
    ((Ref*)h)->trk->search_IC_matches(wrap_image(img, rows, cols, stride));
}
void ref_ransac_hypotheses(void* h) { ((Ref*)h)->trk->ransac_hypotheses(); }
void ref_update_li(void* h) { ((Ref*)h)->kf->ekf_update_li_inliers(); }
void ref_rescue_hi(void* h) { ((Ref*)h)->trk->rescue_hi_inliers(); }
void ref_update_hi(void* h) { ((Ref*)h)->kf->ekf_update_hi_inliers(); }
// steps 1-2 of search_IC_matches only (src/Tracking.cpp:34-66): prediction, Jacobians, S_i, patch warp -- no matching
void ref_predict_only(void* h) {
    Ref* R = (Ref*)h;
    ExtendKF* k = R->kf;
    k->predict_camera_measurements(k->x_k_km1);
    R->trk->calculate_derivatives(k->x_k_km1);
    for (size_t i = 0; i < k->features_info.size(); i++)
        if (k->features_info[i].h.cols()) k->features_info[i].S = k->features_info[i].H * k->p_k_km1 * k->features_info[i].H.transpose() + k->features_info[i].R;
}
// Map::map_management step 2 alone (src/Map.cpp:34-55): counters + flag reset, used by synthetic replays that keep the map fixed
void ref_reset_flags(void* h) {
    ExtendKF* k = ((Ref*)h)->kf;
    for (size_t i = 0; i < k->features_info.size(); i++) {
        Feature& f = k->features_info[i];
        if (f.h.cols()) f.times_predicted += 1;
        if (f.low_innovation_inlier || f.high_innovation_inlier) f.times_measured += 1;
        f.individually_compatible = false;
        f.low_innovation_inlier = false;
        f.high_innovation_inlier = false;
        f.h.resize(0);
        f.z.resize(0);
        f.H.resize(0, 0);
        f.S.resize(0, 0);
    }
}

// ---- bounded samples of a frame that is too large to run whole (configuration C3, n = 12013; SURVEY 8d "per-stage sub-sampling") ----
// The stages of Tracking::search_IC_matches one at a time (all public members of the reference's classes):
void ref_predict_measurements(void* h) { ((Ref*)h)->kf->predict_camera_measurements(((Ref*)h)->kf->x_k_km1); }
void ref_calculate_derivatives(void* h) { ((Ref*)h)->trk->calculate_derivatives(((Ref*)h)->kf->x_k_km1); }
// the S_i statement of src/Tracking.cpp:41-43 for features [first, first + count) only; returns how many had a prediction
int ref_S_subset(void* h, int first, int count) {
    ExtendKF* k = ((Ref*)h)->kf;
    int done = 0;
    for (int i = first; i < first + count && i < (int)k->features_info.size(); i++)
        if (k->features_info[i].h.cols()) {
            k->features_info[i].S = (k->features_info[i].H) * (k->p_k_km1) * (k->features_info[i].H.transpose()) + (k->features_info[i].R);
            done++;
        }
    return done;
}
// Tracking::ransac_hypotheses, left after `max_hyp` hypotheses (see __wrap_rand); returns the hypotheses completed
int ref_ransac_limited(void* h, int max_hyp) {
    const size_t before = g_rand_pos;
    g_rand_budget = (long)before + max_hyp;
    if (setjmp(g_rand_jmp) == 0) ((Ref*)h)->trk->ransac_hypotheses();
    g_rand_budget = -1;
    return (int)(g_rand_pos - before);
}
// overwrite the inlier flags (to time ExtendKF::ekf_update_li_inliers / ekf_update_hi_inliers on a chosen number of measurements)
void ref_set_inlier_flags(void* h, const uint8_t* li, const uint8_t* hi) {
    ExtendKF* k = ((Ref*)h)->kf;
    for (size_t i = 0; i < k->features_info.size(); i++) {
        k->features_info[i].low_innovation_inlier = li[i] != 0;
        k->features_info[i].high_innovation_inlier = hi[i] != 0;
    }
}
// dense products of the stand-in Eigen: 0 = plain loops (what the parity vectors were made with), 1 = packed cache-blocked kernel
// (oracle/gemm.cpp, `threads` OpenMP threads) for products larger than 4 x 4 -- a fairer stand-in for Eigen's GEBP when timing
extern "C++" {
namespace orc {
void dgemm(bool tA, bool tB, int M, int N, int K, const double* A, int lda, const double* B, int ldb, double* C, int ldc);
void set_threads(int n);
}  // namespace orc
}
static void blocked_hook(long M, long N, long K, const double* A, const double* B, double* C) {
    orc::dgemm(false, false, (int)M, (int)N, (int)K, A, (int)M, B, (int)K, C, (int)M);
}
void ref_set_blocked_gemm(int on, int threads) {
    orc::set_threads(threads < 1 ? 1 : threads);
    Eigen::gemm_hook() = on ? blocked_hook : nullptr;
}
// seconds of one (m x k) * (k x n) product through the stand-in Eigen's operator* in the current product mode
double ref_gemm_seconds(int m, int n, int k) {
    Eigen::MatrixXd A = Eigen::MatrixXd::Zero(m, k), B = Eigen::MatrixXd::Zero(k, n);
    for (int j = 0; j < k; j++)
        for (int i = 0; i < m; i++) A(i, j) = 1.0 / (1 + i + j);
    for (int j = 0; j < n; j++)
        for (int i = 0; i < k; i++) B(i, j) = 1.0 / (2 + i + 2 * j);
    struct timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    Eigen::MatrixXd C = A * B;
    clock_gettime(CLOCK_MONOTONIC, &t1);
    volatile double sink = C(m - 1, n - 1);
    (void)sink;
    return (t1.tv_sec - t0.tv_sec) + 1e-9 * (t1.tv_nsec - t0.tv_nsec);
}

// ---- state access ---------------------------------------------------------------------------------------------------------------------
int ref_num_features(void* h) { return (int)((Ref*)h)->kf->features_info.size(); }
int ref_state_dim(void* h, int prior) {
    ExtendKF* k = ((Ref*)h)->kf;
    return (int)(prior ? k->x_k_km1.rows() : k->x_k_k.rows());
}
void ref_get_state(void* h, int prior, double* x, double* P_colmajor) {
    ExtendKF* k = ((Ref*)h)->kf;
    const Eigen::VectorXd& xs = prior ? k->x_k_km1 : k->x_k_k;
    const Eigen::MatrixXd& Ps = prior ? k->p_k_km1 : k->p_k_k;
    if (x) std::memcpy(x, xs.data(), sizeof(double) * (size_t)xs.rows());
    if (P_colmajor) std::memcpy(P_colmajor, Ps.data(), sizeof(double) * (size_t)(Ps.rows() * Ps.cols()));
}
void ref_set_state(void* h, int prior, const double* x, const double* P_colmajor, int n) {
    ExtendKF* k = ((Ref*)h)->kf;
    Eigen::VectorXd xs(n);
    Eigen::MatrixXd Ps(n, n);
    std::memcpy(xs.data(), x, sizeof(double) * (size_t)n);
    std::memcpy(Ps.data(), P_colmajor, sizeof(double) * (size_t)n * n);
    if (prior) {
        k->x_k_km1 = xs;
        k->p_k_km1 = Ps;
    } else {
        k->x_k_k = xs;
        k->p_k_k = Ps;
    }
}
// push_back of a feature record with the defaults of Map::initialize_a_features (src/Map.cpp:287-311); the caller supplies the state
// entries through ref_set_state.  type: 0 inverse depth, 1 cartesian.  patch41: 41 x 41 row-major uint8 (or null -> zeros).
void ref_add_feature(void* h, int type, const uint8_t* patch41, const double* patch_match13_rowmajor, const double* r_wc, const double* R_wc_rowmajor,
                     const double* uv, int init_frame) {
    ExtendKF* k = ((Ref*)h)->kf;
    Feature f;
    f.patch_when_initialized = Eigen::MatrixXd::Zero(41, 41);
    if (patch41)
        for (int i = 0; i < 41; i++)
            for (int j = 0; j < 41; j++) f.patch_when_initialized(i, j) = patch41[i * 41 + j];
    f.patch_when_matching = Eigen::MatrixXd::Zero(13, 13);
    if (patch_match13_rowmajor)
        for (int i = 0; i < 13; i++)
            for (int j = 0; j < 13; j++) f.patch_when_matching(i, j) = patch_match13_rowmajor[i * 13 + j];
    for (int i = 0; i < 3; i++) f.r_wc_when_initialized(i) = r_wc ? r_wc[i] : 0.0;
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) f.R_wc_when_initialized(i, j) = R_wc_rowmajor ? R_wc_rowmajor[i * 3 + j] : (i == j ? 1.0 : 0.0);
    f.uv_when_initialized(0) = uv ? uv[0] : 0.0;
    f.uv_when_initialized(1) = uv ? uv[1] : 0.0;
    f.half_patch_size_when_initialized = 20;
    f.half_patch_size_when_matching = 6;
    f.times_predicted = 0;
    f.times_measured = 0;
    f.init_frame = init_frame;
    f.init_measurement(0) = f.uv_when_initialized(0);
    f.init_measurement(1) = f.uv_when_initialized(1);
    f.type = type ? "cartesian" : "inversedepth";
    f.individually_compatible = false;
    f.low_innovation_inlier = false;
    f.high_innovation_inlier = false;
    f.z.resize(0);
    f.h.resize(0);
    f.H.resize(0, 0);
    f.S.resize(0, 0);
    f.state_size = type ? 3 : 6;
    f.measurement_size = 2;
    f.R = Eigen::MatrixXd::Identity(2, 2);
    k->features_info.push_back(f);
}
void ref_set_counters(void* h, const int* times_predicted, const int* times_measured) {
    ExtendKF* k = ((Ref*)h)->kf;
    for (size_t i = 0; i < k->features_info.size(); i++) {
        k->features_info[i].times_predicted = times_predicted[i];
        k->features_info[i].times_measured = times_measured[i];
    }
}
// overwrite the matching result (to drive ransac / updates from synthetic matches without an image)
void ref_set_matches(void* h, const double* z, const uint8_t* ic) {
    ExtendKF* k = ((Ref*)h)->kf;
    for (size_t i = 0; i < k->features_info.size(); i++) {
        Feature& f = k->features_info[i];
        f.individually_compatible = ic[i] != 0;
        if (ic[i]) {
            f.z.resize(2);
            f.z(0) = z[2 * i];
            f.z(1) = z[2 * i + 1];
        } else
            f.z.resize(0);
    }
}
// h (N x 2), S (N x 4 row-major), z (N x 2), flags (N x 4: has_h, ic, li, hi), counters (N x 2), types (N)
void ref_get_features(void* hd, double* h, double* S, double* z, uint8_t* flags, int* counters, int* types) {
    ExtendKF* k = ((Ref*)hd)->kf;
    for (size_t i = 0; i < k->features_info.size(); i++) {
        const Feature& f = k->features_info[i];
        const bool has_h = f.h.cols() > 0, has_S = f.S.cols() > 0, has_z = f.z.rows() > 0;
        for (int c = 0; c < 2; c++) {
            if (h) h[2 * i + c] = has_h ? f.h(c) : 0.0;
            if (z) z[2 * i + c] = has_z ? f.z(c) : 0.0;
        }
        if (S)
            for (int a = 0; a < 2; a++)
                for (int b = 0; b < 2; b++) S[4 * i + 2 * a + b] = has_S ? f.S(a, b) : 0.0;
        if (flags) {
            flags[4 * i + 0] = has_h;
            flags[4 * i + 1] = f.individually_compatible;
            flags[4 * i + 2] = f.low_innovation_inlier;
            flags[4 * i + 3] = f.high_innovation_inlier;
        }
        if (counters) {
            counters[2 * i + 0] = f.times_predicted;
            counters[2 * i + 1] = f.times_measured;
        }
        if (types) types[i] = std::strcmp(f.type.c_str(), "cartesian") == 0 ? 1 : 0;
    }
}
int ref_get_H(void* hd, int i, double* out_rowmajor, int ncols) {  // dense 2 x n Jacobian of feature i; returns its column count (0 if none)
    const Feature& f = ((Ref*)hd)->kf->features_info[(size_t)i];
    if (f.H.rows() == 0) return 0;
    if (out_rowmajor && ncols >= f.H.cols())
        for (int a = 0; a < 2; a++)
            for (int c = 0; c < f.H.cols(); c++) out_rowmajor[(size_t)a * ncols + c] = f.H(a, c);
    return (int)f.H.cols();
}
void ref_get_patch_matching(void* hd, int i, double* out13_rowmajor) {
    const Feature& f = ((Ref*)hd)->kf->features_info[(size_t)i];
    for (int a = 0; a < 13; a++)
        for (int b = 0; b < 13; b++) out13_rowmajor[a * 13 + b] = (f.patch_when_matching.rows() == 13) ? f.patch_when_matching(a, b) : 0.0;
}
void ref_get_feature_init(void* hd, int i, uint8_t* patch41, double* pose14) {  // patch + (r_wc 3, R_wc 9 row-major, uv 2)
    const Feature& f = ((Ref*)hd)->kf->features_info[(size_t)i];
    if (patch41)
        for (int a = 0; a < 41; a++)
            for (int b = 0; b < 41; b++) patch41[a * 41 + b] = (uint8_t)f.patch_when_initialized(a, b);
    if (pose14) {
        for (int a = 0; a < 3; a++) pose14[a] = f.r_wc_when_initialized(a);
        for (int a = 0; a < 3; a++)
            for (int b = 0; b < 3; b++) pose14[3 + a * 3 + b] = f.R_wc_when_initialized(a, b);
        pose14[12] = f.uv_when_initialized(0);
        pose14[13] = f.uv_when_initialized(1);
    }
}
// helpers of ExtendKF, for primitive-level pins
void ref_distort(void* hd, const double* uv, int m, double* out) {
    ExtendKF* k = ((Ref*)hd)->kf;
    Eigen::MatrixXd in(2, m), o;
    for (int i = 0; i < m; i++) {
        in(0, i) = uv[2 * i];
        in(1, i) = uv[2 * i + 1];
    }
    k->distort_fm(in, o);
    for (int i = 0; i < m; i++) {
        out[2 * i] = o(0, i);
        out[2 * i + 1] = o(1, i);
    }
}
void ref_undistort(void* hd, const double* uv, int m, double* out) {
    ExtendKF* k = ((Ref*)hd)->kf;
    Eigen::MatrixXd in(2, m), o;
    for (int i = 0; i < m; i++) {
        in(0, i) = uv[2 * i];
        in(1, i) = uv[2 * i + 1];
    }
    k->undistort_fm(in, o);
    for (int i = 0; i < m; i++) {
        out[2 * i] = o(0, i);
        out[2 * i + 1] = o(1, i);
    }
}

}  // extern "C"
