/*
 * larvio_b200 — C ABI of the B200-native batched MSCKF-VIO hot path.
 *
 * Drop-in boundary for the reference's per-frame path (SURVEY.md §8b): every entry point
 * below is what a binding of LARVIO's `ImageProcessor` / `LarVio` classes would call for a
 * batch of S independent sequences (S = 1 reproduces the reference's call surface):
 *
 *   lvb_create / lvb_create_from_file  <-  ImageProcessor(std::string&) + initialize()
 *                                          (include/larvio/image_processor.h:39-47,
 *                                           src/image_processor.cpp:28-34,116-126) and
 *                                          LarVio(std::string&) + initialize()
 *                                          (include/larvio/larvio.h:42-56, src/larvio.cpp:42-47,314-360)
 *   lvb_process_images                 <-  ImageProcessor::processImage
 *                                          (image_processor.h:55-57, image_processor.cpp:130-219)
 *   lvb_process_features               <-  LarVio::processFeatures (larvio.h:63-64, larvio.cpp:363-461)
 *   lvb_step                           <-  the driver's back-to-back pair of calls
 *                                          (app/larvioMain.cpp:107,114) with the feature message
 *                                          kept in HBM between the two
 *   lvb_set_initial_state              <-  what FlexibleInitializer::tryIncInit leaves behind
 *                                          (larvio.cpp:375-391); the initialisers themselves are
 *                                          out of scope (SURVEY.md §2 row 6)
 *   lvb_get_state / lvb_get_window     <-  getTbw/getVel/getPpose/getPvel/getSwPoses (larvio.h:66-85)
 *   lvb_get_points                     <-  getStableMapPointPositions / getActiveeMapPointPositions (larvio.h:86-87)
 *
 * Plain pointers and sizes only; no torch / Eigen / OpenCV types.  All "host" pointers are
 * ordinary (preferably pinned) host memory; entry points ending in `_dev` take device pointers.
 * Return value: 0 = ok, <0 = LVB_E_* ; CUDA failures are reported, never papered over by a
 * CPU path (there is none).
 */
#ifndef LARVIO_B200_H
#define LARVIO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LVB_OK 0
#define LVB_E_ARG (-1)
#define LVB_E_CUDA (-2)
#define LVB_E_CONFIG (-3)
#define LVB_E_UNSUPPORTED (-4)
#define LVB_E_CAPACITY (-5)

/* Flat copy of every config key the hot path reads (SURVEY.md App. B). Mirrors
 * larvio_b200/config.py:LvbConfig field for field. */
typedef struct LvbConfig {
  int width, height;
  int distortion_model; /* 0 radtan, 1 equidistant */
  int _pad0;
  double fx, fy, cx, cy;
  double dist[4];
  double T_cam_imu[16]; /* row-major 4x4 exactly as in the yaml */
  int pyramid_levels, patch_size, max_iteration, max_features_num, min_distance, flag_equalize;
  double track_precision, pub_frequency, img_rate;
  double imu_rate;
  double rotation_threshold, translation_threshold, tracking_rate_threshold;
  double feature_translation_threshold;
  double td;
  double noise_gyro, noise_acc, noise_gyro_bias, noise_acc_bias, noise_feature;
  double cov_orientation, cov_velocity, cov_position, cov_gyro_bias, cov_acc_bias;
  double cov_extrin_rot, cov_extrin_trans;
  double zupt_max_feature_dis, zupt_noise_v, zupt_noise_p, zupt_noise_q;
  double static_duration;
  int max_track_len, sw_size, least_observation_number;
  int if_FEJ, estimate_extrin, estimate_td, calib_imu_instrinsic, if_ZUPT_valid;
  int max_features_in_one_grid, aug_grid_rows, aug_grid_cols, feature_idp_dim, use_schmidt, _pad1;
  /* hybrid filter: max_features_in_one_grid * aug_grid_rows * aug_grid_cols EKF-SLAM features (<= 64, 0 = pure MSCKF);
     feature_idp_dim 1 = inverse depth on the anchor bearing, anything else = 3-D (x/z, y/z, 1/z) like larvio.cpp:270-274;
     use_schmidt != 0 (larvio.cpp:277): anchor poses older than two states that leave the window stay behind the feature block
     as nuisance states (up to 16 per sequence; more is reported as LVB_E_CAPACITY) */
} LvbConfig;

/* include/sensors/ImuData.hpp:16-38 as a POD. */
typedef struct LvbImu {
  double t;
  double gyro[3];
  double acc[3];
} LvbImu;

/* One feature of MonoCameraMeasurement (include/larvio/feature_msg.h:15-47). */
typedef struct LvbFeature {
  uint64_t id;
  double u, v, u_init, v_init, u_vel, v_vel, u_init_vel, v_init_vel;
} LvbFeature;

typedef struct LvbHandle LvbHandle;

/* Parse the reference's OpenCV-yaml config file into *cfg (no OpenCV needed). */
int lvb_parse_config(const char* yaml_path, LvbConfig* cfg);

int lvb_create(const LvbConfig* cfg, int n_seq, int device, LvbHandle** out);
int lvb_create_from_file(const char* yaml_path, int n_seq, int device, LvbHandle** out);
void lvb_destroy(LvbHandle* h);
const char* lvb_last_error(void);
int lvb_feature_capacity(const LvbHandle* h); /* per-sequence capacity of feature outputs */
int lvb_n_seq(const LvbHandle* h);

/* ImageProcessor::processImage for S sequences.
 *   images      [S][height][width] u8, host
 *   t_img       [S] image stamps (s)
 *   imu         [S][imu_stride] the caller's IMU buffers (read only, like the reference)
 *   n_imu       [S] valid entries per buffer
 *   out_feat    [S][cap] caller-owned, cap = lvb_feature_capacity(); out_n [S]
 *   has_features[S] = the reference's bool return (true => a feature message was emitted) */
int lvb_process_images(LvbHandle* h, const uint8_t* images, const double* t_img, const LvbImu* imu,
                       const int* n_imu, int imu_stride, LvbFeature* out_feat, int* out_n,
                       uint8_t* has_features);

/* LarVio::processFeatures for S sequences. `valid[s]==0` skips sequence s (the driver only
 * calls processFeatures when processImage returned true).  imu buffers are MUTATED like the
 * reference's: consumed samples are erased in place and n_imu updated (larvio.cpp:510-512).
 * ok[s] = the reference's bool return. */
int lvb_process_features(LvbHandle* h, const uint8_t* valid, const double* t_msg, const LvbFeature* feat,
                         const int* n_feat, int feat_stride, LvbImu* imu, int* n_imu, int imu_stride,
                         uint8_t* ok);

/* Fused driver step (app/larvioMain.cpp:107-114 for every sequence): processImage then, where
 * it returned true, processFeatures; the feature message never leaves the GPU.
 *   images_on_device != 0: `images` is a device pointer (inputs already resident in HBM).
 *   published[s] = processFeatures' return.  IMU buffers are mutated as above. */
int lvb_step(LvbHandle* h, const uint8_t* images, int images_on_device, const double* t_img, LvbImu* imu,
             int* n_imu, int imu_stride, uint8_t* published);
int lvb_synchronize(LvbHandle* h);

/* State left by the initialiser: body->world Hamilton quaternion [x y z w], position, velocity, biases at time t; marks
 * gravity as set (larvio.cpp:378-386) and the bFirstFeatures gate as passed (the reference only reaches its initialiser behind that
 * gate, :365-376), so the lvb_process_features call that follows in the same frame runs the filter on the IMU samples the
 * initialiser left, as larvio.cpp:391 does. */
int lvb_set_initial_state(LvbHandle* h, int seq, double t, const double* q_xyzw, const double* p,
                          const double* v, const double* bg, const double* ba);

/* Inclinometer (static-scene) initialiser, HOST side, one object per sequence: StaticInitializer::tryIncInit +
 * assignInitialState (src/StaticInitializer.cpp:13-161) as FlexibleInitializer::tryIncInit runs them from
 * LarVio::processFeatures until gravity is set (src/larvio.cpp:375-391; the dynamic initialiser is out of scope).
 * Feed it every published feature message (lvb_process_images output) with the caller's IMU buffer.  Returns 1 once
 * static_duration*pub_frequency consecutive static messages were seen: state17 = t, q(4), p(3), v(3), bg(3), ba(3)
 * goes to lvb_set_initial_state, *n_consumed leading IMU samples are to be erased from the caller's buffer
 * (StaticInitializer.cpp:149-150) and gyro_old/acc_old are the sample the propagation will start from.
 * Returns 0 while not initialised, <0 on error.  Needs no GPU. */
typedef struct LvbStaticInit LvbStaticInit;
LvbStaticInit* lvb_static_init_create(const LvbConfig* cfg);
void lvb_static_init_destroy(LvbStaticInit* s);
int lvb_static_init_try(LvbStaticInit* s, const LvbFeature* feat, int n_feat, double t_msg, const LvbImu* imu,
                        int n_imu, double* state17, double* gyro_old3, double* acc_old3, int* n_consumed);

/* getTbw/getVel/getPpose/getPvel: q[4] p[3] v[3] bg[3] ba[3] P_pose[36] P_vel[9], plus time. */
int lvb_get_state(LvbHandle* h, int seq, double* t, double* q_xyzw, double* p, double* v, double* bg,
                  double* ba, double* P_pose36, double* P_vel9);
/* All sequences at once: out[S][17] = t, q(4), p(3), v(3), bg(3), ba(3). */
int lvb_get_states(LvbHandle* h, double* out);
/* getSwPoses: window poses (IMU frame) [n][7] = q(4) p(3); returns count in *n. */
int lvb_get_window(LvbHandle* h, int seq, double* qp, int cap, int* n);
/* getStableMapPointPositions / getActiveeMapPointPositions (larvio.h:86-87, larvio.cpp:2719-2733) for one sequence:
 * which = 0: EKF-SLAM features that left the state since the last read (lost_slam_features, larvio.cpp:3342);
 * which = 1: features that were in the state at the end of a step since the last read, with their latest position
 * (active_slam_features, larvio.cpp:455-458).  ids[cap], xyz[cap][3] (world frame) are caller-owned; *n entries are
 * written and the list is cleared, like the reference's getters clear their map.  LVB_E_CAPACITY if cap is too small
 * (nothing cleared) or if the device-side list overflowed since the last read (8 x the SLAM capacity, at least 64). */
int lvb_get_points(LvbHandle* h, int seq, int which, unsigned long long* ids, double* xyz, int cap, int* n);
/* Online-calibrated quantities of one sequence (StateServer / IMUState members the reference logs, larvio.h:99-142,
 * imu_state.h:70-77): R_imu_cam0[9] row-major, t_cam0_imu[3], td, and the IMU intrinsics Tg[9], As[9], Ma[9]
 * (identity / zero / identity unless calib_imu_instrinsic, larvio.cpp:127-155, 3803-3847). */
int lvb_get_calibration(LvbHandle* h, int seq, double* R_imu_cam9, double* t_cam_imu3, double* td,
                        double* Tg9, double* As9, double* Ma9);
/* Full covariance of one sequence, row-major dim x dim (dim returned). */
int lvb_get_covariance(LvbHandle* h, int seq, double* P, int cap_dim, int* dim);

/* ---- sharding over the GPUs of a node inside ONE process (SURVEY.md 8b: lvb_create(cfg, n_seq, gpu_ids, n_gpu)) ----
 * n_seq independent sequences are split into n_gpu contiguous blocks, block k lives on device gpu_ids[k] (ids may repeat:
 * several shards per GPU overlap their host work).  Sequences never interact, so there is no exchange step; lvbm_step runs
 * lvb_step of every shard on its own host thread and lvbm_get_states gathers the trajectories.  Array arguments are the
 * [n_seq]-sized arrays of lvb_step, images in HOST memory.  (Across processes - one rank per GPU - use one handle per rank
 * and any transport for the gather; bench.py does that with NCCL.) */
typedef struct LvbMulti LvbMulti;
int lvbm_create(const LvbConfig* cfg, int n_seq, const int* gpu_ids, int n_gpu, LvbMulti** out);
void lvbm_destroy(LvbMulti* m);
int lvbm_n_shards(const LvbMulti* m);
int lvbm_set_initial_state(LvbMulti* m, int seq, double t, const double* q_xyzw, const double* p, const double* v,
                           const double* bg, const double* ba);
int lvbm_step(LvbMulti* m, const uint8_t* images, const double* t_img, LvbImu* imu, int* n_imu, int imu_stride,
              uint8_t* published);
int lvbm_get_states(LvbMulti* m, double* out /* [n_seq][17] */);
long long lvbm_launch_count(const LvbMulti* m);

/* ---- stage-level entry points (host buffers; used by the parity tests and profilers) ---- */
/* CLAHE(3.0, 8x8) + 3-level padded LK pyramid + ORB blur for n images: outputs tightly packed
 * (no padding): clahe [n][H][W], l1 [n][H1][W1], l2 [n][H2][W2], blur [n][H][W]. Any may be NULL. */
int lvbk_pyramid(LvbHandle* h, const uint8_t* images, int n, uint8_t* clahe, uint8_t* l1, uint8_t* l2,
                 uint8_t* blur);
/* The same pyramid, one level WITH its REFLECT_101 pad (the LK kernel reads up to 24 px outside a level):
 * out [n][h + 48][w + 48] for level `level` (0 = the equalised image). */
int lvbk_pyramid_padded(LvbHandle* h, const uint8_t* images, int n, int level, uint8_t* out);
/* calcOpticalFlowPyrLK(prev->next, USE_INITIAL_FLOW) on raw (already equalised) image pairs:
 * prev/next [n][H][W]; pts [n][m][2]; status [n][m]. next_pts is in/out (initial flow). */
int lvbk_lk(LvbHandle* h, const uint8_t* prev, const uint8_t* next, int n, int m, const float* prev_pts,
            float* next_pts, uint8_t* status);
/* ORB angle (deg) + 32-byte descriptors at m points of n (equalised) images. */
int lvbk_orb(LvbHandle* h, const uint8_t* images, int n, int m, const float* pts, float* angles,
             uint8_t* desc);
/* goodFeaturesToTrack(img, want, 0.01, min_distance, mask) ; mask may be NULL. out_pts [n][cap][2]. */
int lvbk_detect(LvbHandle* h, const uint8_t* images, const uint8_t* masks, int n, const int* want,
                float* out_pts, int* out_n, float* eig_map);
/* undistortPoints (radtan / equidistant), to_pixels ? P=K : P=I. */
int lvbk_undistort(LvbHandle* h, const float* pts, int m, int to_pixels, float* out);
/* findFundamentalMat(FM_RANSAC, 1.0, 0.99) inlier masks for n independent point sets of m[i] points. */
int lvbk_ransac(LvbHandle* h, const float* p1, const float* p2, int n, const int* m, int stride,
                uint8_t* mask);

/* Per-kernel device timing: while enabled every kernel launch is bracketed by CUDA events on the
 * launching stream (bench.py's roofline figures come from here).  lvb_profile_get returns the number
 * of distinct kernels and fills names / accumulated ms / launch counts. */
int lvb_profile_enable(LvbHandle* h, int on);
int lvb_profile_reset(LvbHandle* h);
int lvb_profile_get(LvbHandle* h, const char** names, double* total_ms, long long* counts, int cap);

/* Cumulative work counters (device-side): [0] LK point-tracks, [1] ORB descriptors, [2] detector runs,
 * [3] published messages, [4] EKF updates, [5] sum r, [6] sum r*d*d, [7] sum stacked rows, [8] QR runs, [9] sum R*c*c,
 * [10] LK iterations, [11] LK iterations on the chain-replay (slow) path, [12] LK window set-ups on the slow path, [13] LK search
 * tile re-stages, [14] findFundamentalMat calls with 8..13 points (OpenCV switches to LMedS below 15 points and its winner is
 * then decided by rounding noise: the one front-end regime where the inlier mask is not reproducible, DESIGN.md 6),
 * [15] sum r*nc*d (nc = nonzero columns of the stacked Jacobian: the flops of T = H P are 2 r nc d). */
int lvb_get_stats(LvbHandle* h, unsigned long long* out16);

/* debug: the 32 per-sequence integers of the filter (dimension, window size, SLAM feature count, flags ...). */
int lvb_debug_icore(LvbHandle* h, int seq, int* out32);

/* number of kernel launches issued through this handle so far (bench.py gpu_launches). */
long long lvb_launch_count(const LvbHandle* h);

#ifdef __cplusplus
}
#endif
#endif /* LARVIO_B200_H */
