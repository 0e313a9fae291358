// Internal layout of a larvio_b200 handle: every per-sequence container of the reference
// (SURVEY.md Appendix D) as fixed-capacity SoA arrays resident in HBM for the whole run.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include "../../include/larvio_b200.h"

#define LVB_CAND_BINS 4096  // corner candidate histogram bins: value bits >> 19 (8 exponent + 4 mantissa bits)
#define LVB_PAD 24          // pyramid level padding (>= patch_size 21 + 1, see App. C-10)
#define LVB_MAX_LEVELS 4
#define LVB_DESC_BYTES 32

struct LvbLevel {
  int w, h;        // image size of this level
  int pitch;       // bytes per padded row
  int rows;        // padded rows
  size_t offset;   // byte offset of padded row 0 inside one sequence's pyramid block
};

struct LvbPyramidLayout {
  int n_levels;
  LvbLevel lv[LVB_MAX_LEVELS];
  size_t bytes_per_seq;
};

// pointer to pixel (0,0) of level l of sequence s in pyramid block `base`
// REFLECT_101 index of p in [0, n) (for -n < p < 2n - 1): the border rule of every front-end filter
__host__ __device__ inline int lvb_reflect101(int p, int n) {
  if (p < 0) p = -p;
  if (p >= n) p = 2 * n - 2 - p;
  return p;
}
__host__ __device__ inline const uint8_t* lvb_level_origin(const uint8_t* base, const LvbPyramidLayout& L,
                                                           int s, int l) {
  return base + (size_t)s * L.bytes_per_seq + L.lv[l].offset + (size_t)LVB_PAD * L.lv[l].pitch + LVB_PAD;
}
__host__ __device__ inline uint8_t* lvb_level_origin(uint8_t* base, const LvbPyramidLayout& L, int s, int l) {
  return base + (size_t)s * L.bytes_per_seq + L.lv[l].offset + (size_t)LVB_PAD * L.lv[l].pitch + LVB_PAD;
}

struct LvbCamera {
  double fx, fy, cx, cy;
  double dist[4];
  int model;
};

// ---- front-end state (image_processor.h:260-325), one slot set per sequence ----
struct LvbTracks {                 // prev_pts_, curr_pts_, pts_ids_, pts_lifetime_, init_pts_, vOrbDescriptors
  float2* prev; float2* curr; float2* init;   // [S][N]
  unsigned long long* ids; int* lifetime;     // [S][N]
  uint8_t* desc;                               // [S][N][32]
  int* n;                                      // [S]
};

struct LvbChain {                  // scratch of one LK<->LK<->ORB<->RANSAC chain (0 tracked, 1 new)
  int* perm;        // [S][N] alive slot indices, order preserving
  int* n;           // [S] alive count
  int* fail;        // [S] chain aborted / not started
  float2* out;      // [S][N] per-stage LK output, indexed by rank i
  uint8_t* status;  // [S][N] per-stage marker, indexed by rank i
  float2* slot_curr;  // [S][N] tracked position in the current image, indexed by slot
  uint8_t* desc;    // [S][N][32] descriptors computed in the previous image (chain 1), by slot
};

struct LvbFrontEnd {
  int S, W, H, N;                 // sequences, image size, per-sequence track capacity
  LvbPyramidLayout L;
  uint8_t* img_in;                // [S][H][W]  staging of the raw input image
  uint8_t* lut;                   // [S][64][256] CLAHE LUTs
  uint8_t* pyr[2];                // ping-pong padded pyramids (prev/curr)
  uint8_t* blur[2];               // ping-pong 7x7-blurred L0 planes [S][H][W]
  int cur;                        // index of the CURRENT pyramid / track set (host-side toggle)
  LvbTracks trk[2];
  float2* new_pts; int* n_new;    // [S][N], [S]
  LvbChain ch[2];
  // per-sequence scalars (device)
  int* image_state;               // 1 FIRST, 2 SECOND, 3 OTHER
  unsigned long long* next_id;
  double* last_pub_time; double* prev_img_time; double* curr_img_time;
  // per-frame host->device inputs
  float* Hmat;                    // [S][9] K R K^-1 (float, row-major)
  int* active;                    // [S] bFirstImg gate result for this frame
  double* t_img;                  // [S]
  // per-frame control flags
  int* do_first; int* do_second; int* do_other; int* do_publish; int* do_detect;
  int* want; int* mask_n;
  // detector scratch
  uint8_t* mask;                  // [S][H][W]
  int* eig_max;                   // [S] ordered-int key of the masked max
  unsigned long long* cand;       // [S][cand_cap] packed (value bits<<32 | pixel index)
  int* n_cand; int cand_cap;
  int* cand_hist;                 // [S][LVB_CAND_BINS] candidate count per value-bits bin (bits 30..19 of the positive float)
  int* overflow;                  // [1] sticky capacity-overflow flag
  unsigned long long* stats;      // [16] work counters: 0 LK point-tracks, 1 ORB descriptors, 2 detector runs, 3 published msgs,
                                  //      4 EKF updates, 5 sum r, 6 sum r*d*d, 7 sum stacked rows, 8 QR runs, 9 sum R*c*c
  float2* det_pts; int* det_n;    // [S][N], [S]
  // outputs
  LvbFeature* msg;                // [S][N]
  int* msg_n;                     // [S]
  uint8_t* has_msg;               // [S]
  double* msg_t;                  // [S]
};

struct LvbBackEnd;   // be_state.h

// optional per-kernel timing (CUDA events on the launching stream), see lvb_profile_* in the C ABI
struct LvbProfiler {
  bool on = false;
  std::vector<cudaEvent_t> ev;          // pairs (start, stop)
  std::vector<int> ev_name;             // name id per pair
  std::vector<std::string> names;
  std::vector<double> total_ms; std::vector<long long> count;
  int used = 0; int open_name = -1;
};

struct LvbHandle {
  LvbConfig cfg;
  int S;
  int device;
  cudaStream_t stream;
  LvbFrontEnd fe;
  LvbBackEnd* be;
  long long launches;
  LvbProfiler prof;
  // host-side per-sequence bookkeeping (mirrors ImageProcessor members that only the host needs)
  std::vector<uint8_t> h_first_img;      // bFirstImg
  std::vector<double> h_prev_img_time;
  std::vector<uint8_t> h_have_prev;
  // pinned staging
  uint8_t* pin_images; size_t pin_images_bytes;
  float* pin_H; int* pin_active; double* pin_t;
  LvbFeature* pin_msg; int* pin_msg_n; uint8_t* pin_has;
  std::vector<void*> allocs;
  int use_graph = 1;                               // lvb_step replays one captured CUDA graph per pyramid parity (LVB_NO_GRAPH=1 disables)
  CUtensorMap lk_maps[2][2][LVB_MAX_LEVELS];       // TMA descriptors of the two ping-pong pyramids x {source, search} box (fe_lk.cu), built on first use
  bool lk_maps_ok[2][2] = {{false, false}, {false, false}};
  cudaGraphExec_t gexec[2] = {nullptr, nullptr};   // one captured step per pyramid parity
  long long glaunches[2] = {0, 0};
};

extern thread_local std::string g_lvb_err;
int lvb_set_err(int code, const char* fmt, ...);

#define LVB_CUDA(x)                                                                        \
  do {                                                                                     \
    cudaError_t e_ = (x);                                                                  \
    if (e_ != cudaSuccess)                                                                 \
      return lvb_set_err(LVB_E_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
  } while (0)

void lvb_prof_begin(LvbHandle* h, const char* name);
void lvb_prof_end(LvbHandle* h);
#define LVB_PROF(h, name) do { if ((h)->prof.on) lvb_prof_begin((h), (name)); } while (0)

#define LVB_LAUNCH_CHECK(h)                                                                \
  do {                                                                                     \
    (h)->launches++;                                                                       \
    if ((h)->prof.on) lvb_prof_end(h);                                                     \
    cudaError_t e_ = cudaGetLastError();                                                   \
    if (e_ != cudaSuccess)                                                                 \
      return lvb_set_err(LVB_E_CUDA, "%s:%d launch -> %s", __FILE__, __LINE__, cudaGetErrorString(e_)); \
  } while (0)

// ---- stage launchers (each file owns its kernels) ----
LvbCamera lvb_camera(const LvbConfig& c);
int fe_build_pyramid(LvbHandle* h, const uint8_t* d_images /*[n][H][W]*/, int n, uint8_t* pyr, uint8_t* blur);
int fe_lk_launch(LvbHandle* h, const uint8_t* pyrA, const uint8_t* pyrB, int n_seq, int stride,
                 const float2* ptsA, const int* perm, const int* n_pts, const float2* init, int init_by_slot,
                 const float* Hmat, float2* out, uint8_t* status, int gate_mode, const float2* ref);
int fe_lk_launch2(LvbHandle* h, const uint8_t* pyrA, const uint8_t* pyrB, int n_seq, int stride,
                  const float2* const ptsA[2], int* const perm[2], int* const n_pts[2], const float2* const init[2],
                  int init_by_slot, const float* Hmat, float2* const out[2], uint8_t* const status[2], int gate_mode,
                  const float2* const ref[2]);
int fe_orb_launch(LvbHandle* h, const uint8_t* pyr, const uint8_t* blur, int n_seq, int stride,
                  const float2* pts, const int* perm, const int* n_pts, float* angles, uint8_t* desc_out,
                  int out_by_slot, const uint8_t* desc_ref, uint8_t* status, int* dist_out);
int fe_orb_gate_launch(LvbHandle* h, const uint8_t* pyr_cur, const uint8_t* blur_cur, const uint8_t* pyr_prev, const uint8_t* blur_prev,
                       int n_seq, int stride, const float2* const cur_pts[2], const float2* new_prev_pts, int* const perm[2],
                       int* const n_pts[2], const uint8_t* birth_desc, uint8_t* new_desc, uint8_t* const status[2]);
int fe_undistort_launch(LvbHandle* h, int n_seq, int stride, const float2* pts, const int* perm,
                        const int* n_pts, float2* out, int to_pixels);
int fe_detect_launch(LvbHandle* h, const uint8_t* pyr, int n_seq, const int* enable, int use_mask,
                     const uint8_t* ext_mask, const float2* mask_pts, const int* mask_n, const int* want,
                     float2* out, int* out_n, float* eig_out = nullptr /*[n_seq][H][W] response map, tests only*/);
int fe_ransac_launch(LvbHandle* h, int n_seq, int stride, const float2* p1, const float2* p2, const int* n,
                     uint8_t* mask, const int* enable, int* fail);
int fe_ransac_launch2(LvbHandle* h, int n_seq, int stride, const float2* const prev[2], const float2* const curr[2],
                      int* const perm[2], int* const n[2], uint8_t* const mask[2], int* const fail[2]);
int fe_process(LvbHandle* h, const uint8_t* images, int on_device, const double* t_img, const LvbImu* imu,
               const int* n_imu, int imu_stride);
int fe_fetch_messages(LvbHandle* h, LvbFeature* out_feat, int* out_n, uint8_t* has_features);
int fe_host_prep(LvbHandle* h, const uint8_t* images, int on_device, const double* t_img, const LvbImu* imu, const int* n_imu,
                 int imu_stride, bool stage_to_img_in, const uint8_t** d_images);
int fe_enqueue(LvbHandle* h, const uint8_t* d_images);
