/* rslam.h -- C ABI of the B200-native 1-point-RANSAC EKF measurement-update path.
 *
 * This is the drop-in boundary for plumewind/ransac_slam's hot path.  The reference has no plugin/FFI layer: the
 * boundary there is the set of C++ methods that System::TrackRunning calls (src/System.cpp:111-129) plus the public
 * members of ExtendKF (include/ransac_slam/ExtendKF.h:154-169).  Each entry point below names the reference method it
 * replaces; the C++ classes in ransac_slam_b200/host/ (same names and signatures as the reference's ExtendKF / Tracking /
 * Map) are thin callers of this ABI.  Plain C types only; no Eigen / OpenCV / STL / torch types cross the boundary.
 *
 * Conventions
 *   - every function returns RSLAM_OK (0) or a negative rslam_status; rslam_last_error() gives the text.
 *   - a handle owns `batch` independent filters that are stepped together (batch == 1 for the reference's single
 *     filter; batch == 4096 for the batched-filter configuration).  Per-filter transfers take the filter index `b`.
 *   - all device work of a handle is issued on the handle's own CUDA stream and is asynchronous; rslam_sync() or any
 *     download waits for it.  Calls on one handle are not re-entrant; different handles are independent.
 *   - state layout: x = [r(3) q(4: w,x,y,z) v(3) w(3) | y_1 ... y_N], inverse-depth y = (x,y,z,theta,phi,rho) (6) or
 *     cartesian y = (X,Y,Z) (3) (src/ExtendKF.cpp:137-152).  P is column-major n x n with leading dimension ldp, i.e.
 *     exactly Eigen's MatrixXd::data() of the reference's p_k_k.
 *   - pointer arguments documented "host or device" may point to either (unified virtual addressing decides).
 *   - the library keeps ONE covariance per filter, updated in place: after rslam_ekf_prediction it is p_k_km1, after
 *     rslam_update_li / rslam_update_hi it is p_k_k (the reference keeps both as separate Eigen members).
 *   - there is no CPU fallback: every entry point fails with RSLAM_ERR_CUDA if no sm_100 device is usable.
 */
#ifndef RSLAM_H
#define RSLAM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rslam_filter rslam_filter; /* opaque */

typedef enum {
    RSLAM_OK = 0,
    RSLAM_ERR_INVALID = -1,   /* bad argument */
    RSLAM_ERR_CUDA = -2,      /* CUDA runtime error / no device */
    RSLAM_ERR_CAPACITY = -3,  /* exceeds max_features / workspace limits given at create */
    RSLAM_ERR_REFERENCE_UB = -4 /* input on which the reference itself is undefined (SURVEY A.3 Q2): cartesian matches in RANSAC */
} rslam_status;

/* include/ransac_slam/System.h:69-82 (CamParam), filled from initialize_param.yaml at src/System.cpp:34-58 */
typedef struct {
    double k1, k2;
    int nRows, nCols;
    double Cx, Cy, f, dx, dy;
} rslam_camera;

/* reference behaviours that change results (SURVEY.md A.3); set bit = behave like the reference */
#define RSLAM_Q1_ANGLES_FROM_POSITIONS 0x1u /* src/Tracking.cpp:448 */
#define RSLAM_Q4_JNORM_INT_EXPONENT 0x2u    /* src/ExtendKF.cpp:627 */
#define RSLAM_Q6_RESCUE_WITHOUT_R 0x4u      /* src/Tracking.cpp:589 */
#define RSLAM_Q_ALL 0x7u

typedef struct {
    double std_a, std_alpha, std_z; /* Sigma.a / Sigma.alpha / Sigma.noise (src/ExtendKF.cpp:16-18) */
    double chi2_095_2;              /* 5.9915 (src/Tracking.cpp:283,576) */
    double corr_threshold;          /* 0.80   (src/Tracking.cpp:281) */
    double p_spurious_free;         /* 0.99   (src/Tracking.cpp:354) */
    int n_hyp_initial;              /* 1000   (src/Tracking.cpp:357) */
    double max_ellipse_eig;         /* 100    (src/Tracking.cpp:303); rslam_create refuses a value that is not in (0, 100] (RSLAM_ERR_INVALID):
                                       the active search stages windows of half-width ceil(2 sqrt(S_ii)) <= 20, which lmax < 100 guarantees */
    unsigned quirks;                /* RSLAM_Q_* mask, default RSLAM_Q_ALL */
    int dedupe_hypotheses;          /* 1: score each distinct 1-point hypothesis once (identical results) */
} rslam_params;

typedef struct {
    int status;        /* 0 ok, 1 no individually-compatible matches (Q9), 3 uniform draws exhausted before termination */
    int hyp_run;       /* hypotheses evaluated by the reference's sequential loop */
    int best_support;  /* inlier count of the winning hypothesis */
    int n_hyp;         /* final adaptive hypothesis budget (src/Tracking.cpp:532) */
    int num_ic;        /* individually compatible matches */
    int winner;        /* index (into the uniform sequence) of the winning hypothesis, -1 if none */
} rslam_ransac_result;

void rslam_default_params(rslam_params* p);
const char* rslam_last_error(void);
const char* rslam_version(void);

/* lifecycle.  max_features bounds N per filter; device = CUDA ordinal. */
int rslam_create(const rslam_camera* cam, const rslam_params* par, int max_features, int batch, int device, rslam_filter** out);
int rslam_destroy(rslam_filter* f);
int rslam_sync(rslam_filter* f);
/* cudaStream_t of the handle (as void*), so callers can record events on the launching stream */
void* rslam_stream(rslam_filter* f);
/* number of kernel launches issued by this handle since creation (bench.py's gpu_launches) */
long long rslam_launch_count(rslam_filter* f);
int rslam_num_features(rslam_filter* f, int b);
int rslam_state_dim(rslam_filter* f, int b);

/* state transfer.  Replaces direct access to ExtendKF::x_k_k / p_k_k / features_info (ExtendKF.h:154-169).
 * feat_types[N]: 0 inverse depth, 1 cartesian.  x, P: host or device.  which: 0 -> x_k_k, 1 -> x_k_km1. */
int rslam_upload_state(rslam_filter* f, int b, int which, const double* x, const double* P, int n, int ldp, const int* feat_types, int N);
int rslam_download_state(rslam_filter* f, int b, int which, double* x, double* P, int ldp);
/* predicted appearance patch_when_matching (13x13 row-major per feature, values must be float-exact) */
int rslam_upload_patches(rslam_filter* f, int b, const double* patches, int N);
/* Tracking::pred_patch_fc on the device (src/Tracking.cpp:164-278).  Upload, per feature, what Map::initialize_a_features stores
 * (src/Map.cpp:286-294): the 41x41 8-bit patch cut at initialisation (row-major), the camera position r_wc[3] and rotation R_wc[9]
 * (row-major) at that time and the initial pixel uv[2]; then enable the warp: rslam_search_ic_matches recomputes
 * patch_when_matching for every predicted feature before the search (otherwise the patches given by rslam_upload_patches are used). */
int rslam_upload_feature_init(rslam_filter* f, int b, const uint8_t* patches41, const double* r_wc, const double* R_wc, const double* uv, int N);
int rslam_set_patch_warp(rslam_filter* f, int enable);
int rslam_download_patches(rslam_filter* f, int b, float* patches, int N);
/* per-feature outputs (any pointer may be NULL): h[2N], S[4N] row-major 2x2, z[2N], flags[4N] = {has_h, individually_compatible,
 * low_innovation_inlier, high_innovation_inlier}, counters[2N] = {times_predicted, times_measured} */
int rslam_download_features(rslam_filter* f, int b, double* h, double* S, double* z, uint8_t* flags, int* counters);
/* structurally non-zero part of H_i: Hc[14N] = d h / d (r,q) (2x7 row-major), Hf[12N] = d h / d y_i (2x6 row-major; 2x3 used for cartesian) */
int rslam_download_H(rslam_filter* f, int b, double* Hc, double* Hf);
/* inject a linearisation and inlier flags directly: h[2N], Hc[14N], Hf[12N], z[2N], flags[4N] = {has_h, individually_compatible,
 * low_innovation_inlier, high_innovation_inlier}; any pointer may be NULL (left as it is).  What ExtendKF::update needs when it is called
 * with caller-built H, z, h (src/ExtendKF.cpp:597) instead of through ekf_update_li_inliers / ekf_update_hi_inliers. */
int rslam_upload_linearisation(rslam_filter* f, int b, const double* h, const double* Hc, const double* Hf, const double* z, const uint8_t* flags);
/* inject matches directly (z[2N], ic[N]) instead of running the active search */
int rslam_set_matches(rslam_filter* f, int b, const double* z, const uint8_t* ic);
/* grayscale frame for filter b (host or device).  With share != 0 the same image is used by every filter of the batch.
 * Binding an image to one filter never changes what any other filter reads: a host image is copied into a device buffer owned by
 * filter b (share == 0) or by the batch's shared image (share != 0), whatever the geometry of earlier calls; a device image is read
 * in place and must stay valid while filters are bound to it. */
int rslam_set_image(rslam_filter* f, int b, const uint8_t* gray, int rows, int cols, int stride, int share);

/* --- the per-frame path (src/System.cpp:111-129) ------------------------------------------------------------- */
/* Map::map_management step 2 (src/Map.cpp:34-55): update times_predicted/times_measured, clear per-frame flags */
int rslam_begin_frame(rslam_filter* f);
/* ExtendKF::ekf_prediction (src/ExtendKF.cpp:333-388), constant-velocity model */
int rslam_ekf_prediction(rslam_filter* f);
/* Tracking::search_IC_matches (src/Tracking.cpp:32-70): h_i, H_i, S_i at x_k_km1, then ZNCC active search on the
 * image set by rslam_set_image (skipped when no image is set: only h/H/S are produced). */
int rslam_search_ic_matches(rslam_filter* f);
/* The two halves of rslam_search_ic_matches on their own (the reference exposes them as Tracking::calculate_derivatives / pred_patch_fc
 * and Tracking::matching, include/ransac_slam/Tracking.h:30-37): h_i, H_i, S_i (+ the patch warp when enabled) at x_k_km1, and the ZNCC
 * search on the bound image with the current predictions. */
int rslam_predict_measurements(rslam_filter* f);
int rslam_match(rslam_filter* f);
/* Tracking::ransac_hypotheses (src/Tracking.cpp:352-539).  u01: batch x n_u01 uniform draws in [0,1) (host or device),
 * replacing ExtendKF::rand (src/ExtendKF.cpp:220-235). */
int rslam_ransac_hypotheses(rslam_filter* f, const double* u01, int n_u01);
int rslam_ransac_result_get(rslam_filter* f, int b, rslam_ransac_result* out);
/* ExtendKF::ekf_update_li_inliers (src/ExtendKF.cpp:559-596) -> update (:597-639) */
int rslam_update_li(rslam_filter* f);
/* Tracking::rescue_hi_inliers (src/Tracking.cpp:574-597) */
int rslam_rescue_hi(rslam_filter* f);
/* ExtendKF::ekf_update_hi_inliers (src/ExtendKF.cpp:640-678) -> update */
int rslam_update_hi(rslam_filter* f);
/* all of the above in order for one frame.  flags: bit0 = run begin_frame + ekf_prediction first.
 * images: batch images (or one shared, see rslam_set_image) host or device, may be NULL to keep the current one. */
int rslam_frame(rslam_filter* f, const uint8_t* images, int rows, int cols, int stride, int share, const double* u01, int n_u01,
                int flags);
/* Input prefetch for streaming callers (not in the reference, whose loop reads an image file and calls TrackRunning on it, examples/Monocular/mono_slam.cpp:47-69):
 * copies the NEXT frame's HOST inputs (same arguments as rslam_frame; pinned memory for a truly asynchronous copy) into a second
 * staging set on the handle's copy stream and returns at once, so the transfer runs beside the frame that is still computing.  The
 * next rslam_frame that is handed the same host pointers and geometry uses the staged set instead of copying; any other call
 * drops it.  The host buffers must stay untouched until that rslam_frame has been issued. */
int rslam_prefetch_inputs(rslam_filter* f, const uint8_t* images, int rows, int cols, int stride, int share, const double* u01, int n_u01);
/* rslam_frame replays its fixed launch sequence as a CUDA graph (default on); 0 = plain stream launches */
int rslam_set_graph(rslam_filter* f, int enable);
/* diagnostics: per-launch CUDA-event timing of every kernel (slow path -- never enable inside a timed region).
 * rslam_profile_read writes "kernel_name launches total_ms\n" lines accumulated since the previous read. */
int rslam_profile_enable(rslam_filter* f, int enable);
int rslam_profile_read(rslam_filter* f, char* buf, size_t buflen);
int rslam_debug_scratch(rslam_filter* f, int b, double* out32);
/* camera pose of filter b after the frame: x_k_k[0..6] plus the 13-state head (13 doubles) */
int rslam_download_pose(rslam_filter* f, int b, double* x13);

/* --- support-scoring sweep (compute_hypothesis_support_fast, src/Tracking.cpp:424-503; Tracking.h:42) ---------- */
/* Scores the hypotheses i in [hyp_begin, hyp_end) of the list hyp_match_idx[n_hyp] (entry = index into the filter's list of
 * individually compatible matches; host or device) whose match index lies in [match_begin, match_end), against all matches of filter 0
 * at (x_k_km1, P).  The two ranges are the two ways to shard a sweep over GPUs: by hypothesis id (every hypothesis scored, the
 * "no-reuse" convention) or by match index (with dedupe_hypotheses each DISTINCT hypothesis is scored once, on exactly one GPU).  Writes
 *   *best_key = (support << 32) | (0xFFFFFFFF - hypothesis id)   (max over the selected hypotheses; 0 if none)
 * to best_key (host or device; device lets the caller all-reduce it with NCCL ncclMax without a host round trip), and,
 * if best_mask != NULL (host), the winner's inlier bit per matched feature (ceil(m/8) bytes, feature order).
 * n_pairs_scored (host, optional): number of (hypothesis, match) pairs actually evaluated on the device. */
int rslam_support_sweep(rslam_filter* f, const int* hyp_match_idx, int n_hyp, int hyp_begin, int hyp_end, int match_begin, int match_end,
                        uint64_t* best_key, uint8_t* best_mask, long long* n_pairs_scored);
/* inlier mask of one hypothesis id after a sweep that covered it (for the rank that owns the all-reduced winner) */
int rslam_sweep_mask(rslam_filter* f, int match_idx, uint8_t* mask);

/* --- the sweep sharded over GPUs (SURVEY 8e): NCCL inside the library, on the handles' own streams ------------------------------
 * Every GPU holds a replica of (x_k_km1, P, matches) in its own handle and scores a shard of the hypothesis list; one MAX all-reduce of
 * the packed 8-byte key gives every rank the winner (highest support, ties -> lowest hypothesis id, the reference's strict '>' at
 * src/Tracking.cpp:507), and, when the mask is wanted, the rank that scored the winner hands its inlier mask to all ranks (a second,
 * ceil(m/32)-word all-reduce whose root is resolved on the device: no host round trip between the two).  NCCL (libnccl.so.2) is loaded
 * at the first rslam_comm_* call; the rest of the library works without it. */
typedef struct rslam_comm rslam_comm; /* opaque */
/* single process driving ndev local GPUs (ncclCommInitAll): local rank i = CUDA device devs[i] (devs == NULL: 0 .. ndev-1) */
int rslam_comm_init(int ndev, const int* devs, rslam_comm** out);
/* one process per GPU: rank 0 obtains a 128-byte id (rslam_comm_unique_id), every rank receives it by any means (MPI, a file,
 * torch.distributed) and calls rslam_comm_init_rank (collective) */
int rslam_comm_unique_id(void* id128);
int rslam_comm_init_rank(int nranks, int rank, const void* id128, int device, rslam_comm** out);
int rslam_comm_destroy(rslam_comm* c);
int rslam_comm_size(const rslam_comm* c);       /* ranks in the communicator */
int rslam_comm_local_size(const rslam_comm* c); /* GPUs driven by this process */
#define RSLAM_SHARD_BY_HYPOTHESIS 0 /* contiguous hypothesis-id ranges: every hypothesis scored ("no reuse" convention) */
#define RSLAM_SHARD_BY_MATCH 1      /* contiguous match-index ranges: with dedupe_hypotheses each distinct hypothesis is scored once, on one GPU */
/* filters[rslam_comm_local_size]: one batch-1 handle per local GPU, created on that GPU, all holding the same state and matches.
 * hyp_match_idx[n_hyp]: host memory, or device memory readable by every local GPU.  best_key: host (the call returns after the result
 * has arrived) or, with one local GPU, device memory (the call only enqueues: the key is valid in stream order).  best_mask (host,
 * optional): the winner's inlier bit per matched feature, ceil(m/8) bytes.  n_pairs_scored (host, optional): pairs scored by the local
 * GPUs. */
int rslam_support_sweep_multi(rslam_comm* c, rslam_filter* const* filters, const int* hyp_match_idx, int n_hyp, int shard, uint64_t* best_key,
                              uint8_t* best_mask, long long* n_pairs_scored);

/* --- map management with the covariance resident on the device (src/Map.cpp; SURVEY 8f row 3) -------------------------- */
/* All of these act on x_k_k / p_k_k of filter b, like the reference between two frames (src/System.cpp:111).  Each rewrites the
 * covariance once, out of place, into a spare buffer owned by the handle and swaps the two (16 n^2 bytes of HBM traffic). */
/* features_info.erase + Map::delete_a_feature (src/Map.cpp:27-28, 69-104) for feature `index` (0-based), consistently. */
int rslam_map_delete_feature(rslam_filter* f, int b, int index);
/* Map::map_management step 1 (src/Map.cpp:19-32): delete every feature with times_measured < 0.5 * times_predicted and
 * times_predicted > 5.  reference_indexing != 0 reproduces the reference's loop exactly: delete_a_feature receives the loop counter,
 * which runs ahead of the iterator after the first erase, so from the second deletion of a pass on the state block of a LATER
 * feature is removed; RSLAM_ERR_REFERENCE_UB is returned where the reference would index past the end.  0 = consistent deletion. */
int rslam_map_delete_features(rslam_filter* f, int b, int reference_indexing, int* n_deleted);
/* Map::inversedepth_2_cartesian (src/Map.cpp:105-196): converts the FIRST inverse-depth feature whose linearity index is below 0.1
 * (at most one per call, like the reference); *converted_index = its index or -1. */
int rslam_map_inversedepth_to_cartesian(rslam_filter* f, int b, int* converted_index);
/* step 4 of Map::initialize_a_features (src/Map.cpp:268-311) for the corner uv[2] (distorted pixel): ExtendKF::hinv
 * (src/ExtendKF.cpp:236-265), Map::add_a_feature_covariance_inverse_depth (src/Map.cpp:339-400) and the new features_info record
 * (41x41 patch cut from the image currently bound to the filter, pose and pixel at initialisation). */
int rslam_map_add_feature(rslam_filter* f, int b, const double* uv, int* new_index);
/* feature types of filter b (0 inverse depth, 1 cartesian), types[N] */
int rslam_feature_types(rslam_filter* f, int b, int* types);
/* overwrite times_predicted / times_measured of filter b (restoring a saved map; tests) */
int rslam_set_counters(rslam_filter* f, int b, const int* times_predicted, const int* times_measured);
/* record stored at initialisation for feature i: patch41[1681] (row-major), pose14 = r_wc(3), R_wc row-major(9), uv(2) */
int rslam_download_feature_init(rslam_filter* f, int b, int i, uint8_t* patch41, double* pose14);

/* --- feature initialisation (src/Map.cpp:198-338; SURVEY 8f row 4) -------------------------------------------------------- */
/* Map::fast_corner_detect_9 (src/Map.cpp:324-338): cv::FAST(TYPE_9_16, non-maximum suppression) on the window (x0, y0, w, h) of the
 * image bound to filter b.  *n_kp = number of corners; the first min(*n_kp, max_kp) as xy[2 i] = (x, y) relative to the window, in
 * OpenCV's output order (row by row, left to right).  The reference uses threshold 100. */
int rslam_fast_corner_detect_9(rslam_filter* f, int b, int x0, int y0, int w, int h, int threshold, int max_kp, int* n_kp, int* xy);
/* Map::initialize_features (src/Map.cpp:198-211): up to 50 attempts of initialize_a_features (:212-323) until min_features_to_init
 * features were added.  u01 (host): 2 uniform draws in [0,1) per attempt, replacing ExtendKF::rand(2,1,0,1) (:231). */
int rslam_map_initialize_features(rslam_filter* f, int b, int step, int min_features_to_init, const double* u01, int n_pairs, int* n_initialized,
                                  int* attempts);
/* Map::map_management (src/Map.cpp:16-67), all four steps; batch-1 handles only.  info4 = {deleted, converted index or -1,
 * initialised, attempts}. */
int rslam_map_management(rslam_filter* f, int b, int step, int min_features, int reference_indexing, const double* u01, int n_pairs, int* info4);
/* Map::map_management (src/Map.cpp:16-67), all four steps, for EVERY filter of the handle at once, each exactly as
 * rslam_map_management does it on a batch-1 handle, in a fixed sequence of three kernel launches and one host synchronisation
 * whatever the batch size and the number of edits.  Each filter's covariance is rewritten once (16 n^2 bytes), for all its
 * deletions, its conversion and its new features together.
 * u01: batch x (2 * n_pairs) uniforms (host or device); filter b's pairs start at u01 + 2 * n_pairs * b.  n_pairs >= 50.
 * status[batch] (host): RSLAM_OK, RSLAM_ERR_REFERENCE_UB or RSLAM_ERR_CAPACITY per filter (RSLAM_ERR_INVALID: see below).
 * info4[4 * batch] (host, optional): {deleted, converted index or -1, initialised, attempts} per filter.
 * Returns RSLAM_OK, or the first non-OK per-filter status.
 * Unlike rslam_map_management: a filter whose delete pass is undefined in the reference (RSLAM_ERR_REFERENCE_UB) is left exactly
 * as it was (state, records, counters, flags) with info {deleted before the failure, -1, 0, 0}, and the other filters proceed; a
 * filter that reaches max_features keeps the features added before, like the per-filter path (RSLAM_ERR_CAPACITY); n_pairs < 50,
 * a NULL u01 or status, or a filter without a bound image return RSLAM_ERR_INVALID before any work.  One filter status can also be
 * RSLAM_ERR_INVALID after work: an initialisation window that leaves the filter's image (uniforms outside [0, 1), or an image smaller
 * than the camera) stops that filter's attempts, and like the per-filter path it keeps the edits made before (deletions, conversion,
 * features already added).
 * Memory: the first call allocates a spare covariance and state vector per filter (batch x ldp x (13 + 6 max_features) doubles
 * more, ldp = that dimension rounded up to 16) and per-filter plans; the filters' buffers and the spares swap on each edit, so
 * per-filter and batched calls can be mixed on one handle. */
int rslam_map_management_batch(rslam_filter* f, int step, int min_features, int reference_indexing, const double* u01, int n_pairs, int* status,
                               int* info4);

/* --- checkpoint / resume of whole filters (not in the reference; SURVEY.md section 5) ---------------------------------------------
 * A snapshot holds everything a filter carries from one frame to the next: n, N, the feature types, x_k_k, x_k_km1, the lower
 * triangle of P and, per feature, times_predicted / times_measured, has_h / ic / li / hi, h, S, z, Hc, Hf, the predicted patch,
 * patch_init and init_pose.  Loading it into a slot makes that slot continue exactly as the saved filter would have.  Not saved:
 * the per-frame scratch (RANSAC and update workspaces, warp geometry; rslam_ransac_result_get of a loaded slot reads zeros until its
 * next frame), the slot's image and uniform bindings (a loaded slot keeps its own), and handle-level switches (patch warp, graph).
 * Both calls return when the copy is complete.  Host snapshots go through one device staging buffer of at most 256 MB, allocated by
 * the first host-memory call and freed by rslam_destroy; device snapshots (memory on the handle's GPU, 16-byte aligned) are packed
 * into and unpacked from directly.  Each chunk of at most 256 MB (one filter's records, or whole 64-column tile columns of its
 * triangle) costs at most two kernel launches and one copy, whatever the batch size.
 *
 * Format, version 1: little-endian; every offset is from the start of the snapshot and every array starts 16-byte aligned;
 * padding bytes are zero, so two saves of the same state are byte-for-byte equal.
 *   header (160 bytes): char magic[8] = "RSLAMCKP"; u32 version = 1 (8); u32 count (12); u64 total bytes (16);
 *     rslam_camera at 24: f64 k1, f64 k2, i32 nRows (40), i32 nCols (44), f64 Cx (48), Cy, f, dx, dy (up to 88);
 *     rslam_params at 88: f64 std_a, std_alpha, std_z, chi2_095_2, corr_threshold, p_spurious_free (up to 136), i32 n_hyp_initial
 *     (136), 4 zero bytes, f64 max_ellipse_eig (144), u32 quirks (152), i32 dedupe_hypotheses (156)
 *   filter table at 160, count entries of 32 bytes: u64 block offset, u64 types offset, i32 n, i32 N, 8 zero bytes
 *   feature types: i32[N] per filter, in filter order
 *   filter blocks, in filter order: i32 n, i32 N, 8 zero bytes; then f64 x_k_k[n], f64 x_k_km1[n], i32 times_predicted[N],
 *     i32 times_measured[N], u8 has_h[N], u8 ic[N], u8 li[N], u8 hi[N], f64 h[2N], f64 S[4N] (2 x 2 row-major), f64 z[2N],
 *     f64 Hc[14N], f64 Hf[12N] (as rslam_download_H), f32 patch[169N] (13 x 13 row-major), u8 patch_init[1681N] (41 x 41 row-major),
 *     f64 init_pose[14N] (r_wc, R_wc row-major, uv); then P as f64[n (n + 1) / 2] in LAPACK lower packed storage (UPLO = 'L':
 *     column j holds rows j..n-1, so element (i, j), i >= j, is at j n - j (j - 1) / 2 + i - j). */
/* size in bytes of a snapshot of filters [b, b + count) */
int rslam_checkpoint_bytes(rslam_filter* f, int b, int count, size_t* bytes);
/* snapshot of filters [b, b + count) into dst (host, or device memory on the handle's GPU).  cap too small: RSLAM_ERR_INVALID
 * with the needed size in the message.  Every saved P must be exactly symmetric (bitwise, the library's invariant, checked on the
 * device): otherwise RSLAM_ERR_INVALID naming the first filter that is not.  *written (optional) = the snapshot's size. */
int rslam_checkpoint_save(rslam_filter* f, int b, int count, void* dst, size_t cap, size_t* written);
/* restore every filter of the snapshot src[bytes] (host or device) into slots [b, b + count); *count_out (optional) = count.
 * The handle may be another one, on this or another GPU, with any batch and any max_features >= each filter's N; its camera and
 * params must equal the snapshot's bit for bit.  feature offsets and the last inverse-depth index are rebuilt from the types as
 * rslam_upload_state builds them; each slot's x_k_k / x_k_km1 past the loaded n and its per-feature arrays past the loaded N are
 * cleared, while its P outside the loaded n x n block is left as it was (as rslam_upload_state leaves it: no kernel reads P past n).  Refusals, all before any device
 * write (the handle is unchanged): RSLAM_ERR_INVALID for a bad magic or version, a size other than the header's, an inconsistent
 * table or types, a camera or params mismatch, or slots outside the batch; RSLAM_ERR_CAPACITY for N > max_features. */
int rslam_checkpoint_load(rslam_filter* f, int b, const void* src, size_t bytes, int* count_out);

#ifdef __cplusplus
}
#endif
#endif /* RSLAM_H */
