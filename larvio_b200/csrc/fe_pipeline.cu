// Batched ImageProcessor::processImage (image_processor.cpp:130-219): the per-sequence state machine
// FIRST_IMAGE / SECOND_IMAGE / OTHER_IMAGES runs on the device (flags + counts stay in HBM, no host
// sync inside a frame); the host only replays integrateImuData (:222-263) to hand each sequence its
// gyro-predicted homography K R K^-1 (:279-283) and toggles the prev/curr ping-pong buffers.
#include <math.h>
#include <string.h>
#include "lvb_internal.h"
#include "fe_device.cuh"

template <typename T>
static int dalloc(LvbHandle* h, T** p, size_t count) {
  void* q = nullptr;
  size_t bytes = count * sizeof(T);
  if (bytes == 0) bytes = sizeof(T);
  LVB_CUDA(cudaMalloc(&q, bytes));
  LVB_CUDA(cudaMemsetAsync(q, 0, bytes, h->stream));
  h->allocs.push_back(q);
  *p = (T*)q;
  return LVB_OK;
}
#define DA(ptr, n) do { int rc_ = dalloc(h, &(ptr), (size_t)(n)); if (rc_ != LVB_OK) return rc_; } while (0)
#define PIN(ptr, T, n) do { void* q_ = nullptr; LVB_CUDA(cudaHostAlloc(&q_, sizeof(T) * (size_t)(n), cudaHostAllocDefault)); memset(q_, 0, sizeof(T) * (size_t)(n)); ptr = (T*)q_; } while (0)

namespace {
__global__ void init_state_kernel(int* image_state, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) image_state[i] = 1;
}
}  // namespace

int fe_alloc(LvbHandle* h) {
  LvbFrontEnd& fe = h->fe;
  const size_t S = fe.S, N = fe.N, npx = (size_t)fe.W * fe.H;
  DA(fe.img_in, S * npx);
  DA(fe.lut, S * 64 * 256);
  for (int k = 0; k < 2; ++k) {
    DA(fe.pyr[k], S * fe.L.bytes_per_seq);
    DA(fe.blur[k], S * npx);
    LvbTracks& t = fe.trk[k];
    DA(t.prev, S * N); DA(t.curr, S * N); DA(t.init, S * N); DA(t.ids, S * N); DA(t.lifetime, S * N);
    DA(t.desc, S * N * LVB_DESC_BYTES); DA(t.n, S);
    LvbChain& c = fe.ch[k];
    DA(c.perm, S * N); DA(c.n, S); DA(c.fail, S); DA(c.out, S * N); DA(c.status, S * N);
    DA(c.slot_curr, S * N); DA(c.desc, S * N * LVB_DESC_BYTES);
  }
  DA(fe.new_pts, S * N); DA(fe.n_new, S);
  DA(fe.image_state, S); DA(fe.next_id, S);
  DA(fe.last_pub_time, S); DA(fe.prev_img_time, S); DA(fe.curr_img_time, S);
  DA(fe.Hmat, S * 9); DA(fe.active, S); DA(fe.t_img, S);
  DA(fe.do_first, S); DA(fe.do_second, S); DA(fe.do_other, S); DA(fe.do_publish, S); DA(fe.do_detect, S);
  DA(fe.want, S); DA(fe.mask_n, S);
  DA(fe.mask, S * npx); DA(fe.eig_max, S);
  fe.cand_cap = 65536;                 // local maxima above 1 % of their tile's maximum (a superset of the final candidates)
  DA(fe.cand, S * (size_t)fe.cand_cap); DA(fe.n_cand, S); DA(fe.cand_hist, S * LVB_CAND_BINS); DA(fe.overflow, 1); DA(fe.stats, 16);
  DA(fe.det_pts, S * N); DA(fe.det_n, S);
  DA(fe.msg, S * N); DA(fe.msg_n, S); DA(fe.has_msg, S); DA(fe.msg_t, S);
  fe.cur = 0;
  LVB_PROF(h, "init_state_kernel");
  init_state_kernel<<<(fe.S + 127) / 128, 128, 0, h->stream>>>(fe.image_state, fe.S);
  LVB_LAUNCH_CHECK(h);
  PIN(h->pin_H, float, S * 9); PIN(h->pin_active, int, S); PIN(h->pin_t, double, S);
  PIN(h->pin_msg, LvbFeature, S * N); PIN(h->pin_msg_n, int, S); PIN(h->pin_has, uint8_t, S);
  h->pin_images_bytes = S * npx;
  { void* q = nullptr; LVB_CUDA(cudaHostAlloc(&q, h->pin_images_bytes, cudaHostAllocDefault)); h->pin_images = (uint8_t*)q; }
  return LVB_OK;
}

// ====================================================================== host: integrateImuData + K R K^-1
namespace {

// cv::Rodrigues(Vec3f) -> 3x3: computed in double, stored as float (OpenCV calib3d).
void rodrigues_f(const float rv[3], float R[9]) {
  const double rx = rv[0], ry = rv[1], rz = rv[2];
  const double theta = sqrt(rx * rx + ry * ry + rz * rz);
  double Rd[9];
  if (theta < 2.220446049250313e-16) {
    for (int i = 0; i < 9; ++i) Rd[i] = (i % 4 == 0) ? 1.0 : 0.0;
  } else {
    const double c = cos(theta), s = sin(theta), c1 = 1. - c, it = theta ? 1. / theta : 0.;
    const double x = rx * it, y = ry * it, z = rz * it;
    const double rrt[9] = {x * x, x * y, x * z, x * y, y * y, y * z, x * z, y * z, z * z};
    const double r_x[9] = {0, -z, y, z, 0, -x, -y, x, 0};
    for (int i = 0; i < 9; ++i) Rd[i] = c * ((i % 4 == 0) ? 1.0 : 0.0) + c1 * rrt[i] + s * r_x[i];
  }
  for (int i = 0; i < 9; ++i) R[i] = (float)Rd[i];
}

void mm33f(const float* A, const float* B, float* C) {
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      float s = 0.f;
      for (int k = 0; k < 3; ++k) s = s + A[i * 3 + k] * B[k * 3 + j];
      C[i * 3 + j] = s;
    }
}

void inv33f(const float* a, float* b) {   // cv::Matx33f::inv closed form
  float d = a[0] * (a[4] * a[8] - a[7] * a[5]) - a[1] * (a[3] * a[8] - a[6] * a[5]) + a[2] * (a[3] * a[7] - a[6] * a[4]);
  d = 1.f / d;
  b[0] = (a[4] * a[8] - a[5] * a[7]) * d; b[1] = (a[2] * a[7] - a[1] * a[8]) * d; b[2] = (a[1] * a[5] - a[2] * a[4]) * d;
  b[3] = (a[5] * a[6] - a[3] * a[8]) * d; b[4] = (a[0] * a[8] - a[2] * a[6]) * d; b[5] = (a[2] * a[3] - a[0] * a[5]) * d;
  b[6] = (a[3] * a[7] - a[4] * a[6]) * d; b[7] = (a[1] * a[6] - a[0] * a[7]) * d; b[8] = (a[0] * a[4] - a[1] * a[3]) * d;
}

// image_processor.cpp:222-263 + :279-283 for one sequence
void predict_homography(const LvbConfig& cfg, const LvbImu* imu, int n_imu, double t_prev, double t_curr, float* H) {
  int b = 0;
  while (b < n_imu && imu[b].t - t_prev < -0.0049) ++b;
  int e = b;
  while (e < n_imu && imu[e].t - t_curr < 0.0049) ++e;
  float mean[3] = {0.f, 0.f, 0.f};
  for (int k = b; k < e; ++k)
    for (int j = 0; j < 3; ++j) mean[j] = mean[j] + (float)imu[k].gyro[j];
  if (e - b > 0) { const float inv = 1.0f / (float)(e - b); for (int j = 0; j < 3; ++j) mean[j] = mean[j] * inv; }
  // R_cam_imu = R_file^T (image_processor.cpp:93); cam rate = R_cam_imu^T * mean = R_file * mean, in double
  float cam[3];
  for (int i = 0; i < 3; ++i) {
    double s = 0.0;
    for (int k = 0; k < 3; ++k) s += cfg.T_cam_imu[i * 4 + k] * (double)mean[k];
    cam[i] = (float)s;
  }
  const double dtime = t_curr - t_prev;
  float rv[3];
  for (int i = 0; i < 3; ++i) rv[i] = (float)((double)cam[i] * dtime);
  float R[9], Rt[9];
  rodrigues_f(rv, R);
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) Rt[i * 3 + j] = R[j * 3 + i];
  const float K[9] = {(float)cfg.fx, 0.f, (float)cfg.cx, 0.f, (float)cfg.fy, (float)cfg.cy, 0.f, 0.f, 1.f};
  float Ki[9], KR[9];
  inv33f(K, Ki);
  mm33f(K, Rt, KR);
  mm33f(KR, Ki, H);
}

// ====================================================================== device: control + compaction + finalize
struct FeView {
  LvbFrontEnd fe;     // by value: all device pointers
  int cur;
  int max_features; int pub_frequency;
};

// one thread per sequence: decide what this frame does (image_processor.cpp:159-205)
__global__ void frame_begin_kernel(FeView v) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= v.fe.S) return;
  const LvbFrontEnd& fe = v.fe;
  const int act = fe.active[s];
  const int st = fe.image_state[s];
  fe.do_first[s] = act && st == 1;
  fe.do_second[s] = act && st == 2;
  fe.do_other[s] = act && st == 3;
  fe.do_publish[s] = 0;
  fe.has_msg[s] = 0;
  fe.msg_n[s] = 0;
  if (act) fe.curr_img_time[s] = fe.t_img[s];
  const LvbTracks& tc = fe.trk[v.cur ^ 1];      // previous frame's track set
  for (int c = 0; c < 2; ++c) {
    const int n_src = (c == 0) ? tc.n[s] : fe.n_new[s];
    const bool en = (c == 0) ? (act && st == 3 && n_src > 0) : (act && (st == 2 || st == 3) && n_src > 0);
    fe.ch[c].n[s] = en ? n_src : 0;
    fe.ch[c].fail[s] = en ? 0 : 1;
  }
}

__global__ void iota_perm_kernel(FeView v) {
  const int s = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= v.fe.N) return;
  v.fe.ch[0].perm[(size_t)s * v.fe.N + i] = i;
  v.fe.ch[1].perm[(size_t)s * v.fe.N + i] = i;
}

// order-preserving compaction of perm by status (removeUnmarkedElements, image_processor.h:215-230).
// one CTA (N threads, N <= 1024) per (sequence, chain).  min_keep: chain aborts when fewer survive.
struct CompactArgs {
  LvbChain ch[2]; int N; unsigned long long* stats; int stage;
  int min_keep[2];           // survivors < min_keep (or == 0) => fail
  int store_curr;            // 1: slot_curr[slot] = out[i] for survivors (after forward LK)
  const int* second;         // do_second flags: chain 1 uses min 20 everywhere in SECOND state
  int min_keep_second;
};

__global__ void compact_kernel(CompactArgs a) {
  __shared__ int wsum[32];
  __shared__ int s_total;
  const int s = blockIdx.x, c = blockIdx.y;
  const LvbChain& ch = a.ch[c];
  if (ch.fail[s]) return;
  const int n = ch.n[s];
  const int i = threadIdx.x;
  if (i == 0 && a.stats) {                       // work counters for the roofline accounting (bench.py)
    if (a.stage <= 1) atomicAdd(&a.stats[0], (unsigned long long)n);
    else if (a.stage == 2) atomicAdd(&a.stats[1], (unsigned long long)(c == 0 ? n : 2 * n));
  }
  const size_t base = (size_t)s * a.N;
  const bool keep = i < n && ch.status[base + i] != 0;
  const int slot = i < n ? ch.perm[base + i] : 0;
  const float2 o = i < n ? ch.out[base + i] : make_float2(0.f, 0.f);
  const unsigned m = __ballot_sync(0xffffffffu, keep);
  const int lane = i & 31, w = i >> 5;
  if (lane == 0) wsum[w] = __popc(m);
  __syncthreads();
  if (i < 32) {
    int x = (i < (blockDim.x + 31) / 32) ? wsum[i] : 0;
    int inc = x;
    for (int o2 = 1; o2 < 32; o2 <<= 1) { const int y = __shfl_up_sync(0xffffffffu, inc, o2); if (i >= o2) inc += y; }
    wsum[i] = inc - x;
    if (i == 31) s_total = inc;
  }
  __syncthreads();
  if (keep) {
    const int pos = wsum[w] + __popc(m & ((1u << lane) - 1));
    ch.perm[base + pos] = slot;
    if (a.store_curr) ch.slot_curr[base + slot] = o;
  }
  if (i == 0) {
    const int total = s_total;
    ch.n[s] = total;
    int mk = a.min_keep[c];
    if (c == 1 && a.second && a.second[s]) mk = a.min_keep_second;
    if (total < mk || total <= 0) { ch.fail[s] = 1; ch.n[s] = 0; }
  }
}

// finalize: rebuild the track set, run the state machine, decide publishing / detection.
// one CTA per sequence.
__global__ void finalize_kernel(FeView v) {
  const int s = blockIdx.x;
  const LvbFrontEnd& fe = v.fe;
  const int N = fe.N;
  const size_t base = (size_t)s * N;
  const LvbTracks& tp = fe.trk[v.cur ^ 1];   // previous track set (slots of chain 0)
  const LvbTracks& tn = fe.trk[v.cur];       // track set being built
  const int tid = threadIdx.x;
  __shared__ int s_n0, s_n1, s_ok1;
  if (!fe.active[s]) {
    // sequence has not started (bFirstImg false): nothing happens, keep state as is
    if (tid == 0) { tn.n[s] = tp.n[s]; fe.do_detect[s] = 0; }
    for (int i = tid; i < tp.n[s]; i += blockDim.x) {
      tn.prev[base + i] = tp.prev[base + i]; tn.curr[base + i] = tp.curr[base + i]; tn.init[base + i] = tp.init[base + i];
      tn.ids[base + i] = tp.ids[base + i]; tn.lifetime[base + i] = tp.lifetime[base + i];
      for (int b = 0; b < 32; ++b) tn.desc[(base + i) * 32 + b] = tp.desc[(base + i) * 32 + b];
    }
    return;
  }
  const int st = fe.image_state[s];
  if (tid == 0) {
    s_n0 = (st == 3 && !fe.ch[0].fail[s]) ? fe.ch[0].n[s] : 0;
    s_ok1 = ((st == 2 || st == 3) && !fe.ch[1].fail[s]) ? 1 : 0;
    s_n1 = s_ok1 ? fe.ch[1].n[s] : 0;
    if (s_n0 + s_n1 > N) s_n1 = N - s_n0;    // cannot happen (tracked + new <= max_features_num)
  }
  __syncthreads();
  const int n0 = s_n0, n1 = s_n1;
  const unsigned long long id0 = fe.next_id[s];
  // tracked survivors (image_processor.cpp:795-808)
  for (int i = tid; i < n0; i += blockDim.x) {
    const int slot = fe.ch[0].perm[base + i];
    tn.prev[base + i] = tp.curr[base + slot];
    tn.curr[base + i] = fe.ch[0].slot_curr[base + slot];
    tn.ids[base + i] = tp.ids[base + slot];
    tn.lifetime[base + i] = tp.lifetime[base + slot] + 1;
    tn.init[base + i] = tp.init[base + slot];
  }
  for (int i = tid; i < n0 * 8; i += blockDim.x) {
    const int r = i >> 3, q = i & 7;
    const int slot = fe.ch[0].perm[base + r];
    reinterpret_cast<unsigned*>(tn.desc)[(base + r) * 8 + q] = reinterpret_cast<const unsigned*>(tp.desc)[(base + slot) * 8 + q];
  }
  // new survivors (:991-998 in OTHER state, :524-531 in SECOND state)
  for (int i = tid; i < n1; i += blockDim.x) {
    const int slot = fe.ch[1].perm[base + i];
    const float2 pp = fe.new_pts[base + slot];
    tn.prev[base + n0 + i] = pp;
    tn.curr[base + n0 + i] = fe.ch[1].slot_curr[base + slot];
    tn.ids[base + n0 + i] = id0 + (unsigned long long)i;
    tn.lifetime[base + n0 + i] = 2;
    tn.init[base + n0 + i] = (st == 2) ? make_float2(-1.f, -1.f) : pp;
  }
  for (int i = tid; i < n1 * 8; i += blockDim.x) {
    const int r = i >> 3, q = i & 7;
    const int slot = fe.ch[1].perm[base + r];
    reinterpret_cast<unsigned*>(tn.desc)[(base + n0 + r) * 8 + q] = reinterpret_cast<const unsigned*>(fe.ch[1].desc)[(base + slot) * 8 + q];
  }
  __syncthreads();
  if (tid == 0) {
    int n_tracks = n0 + n1;
    int state = st;
    int publish = 0, detect = 0, want = 0, mask_n = 0;
    const double t = fe.curr_img_time[s];
    const double period = 0.9 * (1.0 / (double)v.pub_frequency);
    if (st == 1) {
      n_tracks = 0;
      detect = 1; want = v.max_features; mask_n = 0;       // initializeFirstFrame
    } else if (st == 2) {
      if (!s_ok1) { state = 1; n_tracks = 0; }             // initializeFirstFeatures failed
      else {
        fe.next_id[s] = id0 + (unsigned long long)n1;
        fe.n_new[s] = 0;
        if (t - fe.last_pub_time[s] >= period) publish = 1;
        state = 3;
      }
    } else {
      if (s_ok1) { fe.next_id[s] = id0 + (unsigned long long)n1; fe.n_new[s] = 0; }
      if (t - fe.last_pub_time[s] >= period) publish = 1;
    }
    if (publish) {
      detect = (v.max_features - n_tracks) > 0;
      want = v.max_features - n_tracks; mask_n = n_tracks;
      if (!detect) fe.n_new[s] = 0;                          // new_pts_ is swapped empty before the test (:1033)
    }
    tn.n[s] = n_tracks;
    fe.image_state[s] = state;
    fe.do_publish[s] = publish;
    fe.do_detect[s] = detect;
    fe.want[s] = want;
    fe.mask_n[s] = mask_n;
  }
}

// after detection: adopt new corners, FIRST-state transition, build the feature message
// (getFeatureMsg, image_processor.cpp:1076-1128) and roll the clocks (:1170-1172, :208-216).
__global__ void publish_kernel(FeView v, LvbCamera cam) {
  const int s = blockIdx.x;
  const LvbFrontEnd& fe = v.fe;
  if (!fe.active[s]) return;
  const int N = fe.N;
  const size_t base = (size_t)s * N;
  const LvbTracks& tn = fe.trk[v.cur];
  const int tid = threadIdx.x;
  const int first = fe.do_first[s], publish = fe.do_publish[s];
  if (fe.do_detect[s]) {
    if (tid == 0) atomicAdd(&fe.stats[2], 1ull);
    const int nd = fe.det_n[s];
    for (int i = tid; i < nd; i += blockDim.x) fe.new_pts[base + i] = fe.det_pts[base + i];
    __syncthreads();
    if (tid == 0) fe.n_new[s] = nd;
  }
  const double t = fe.curr_img_time[s];
  if (first) {
    if (tid == 0) {
      fe.last_pub_time[s] = t;                               // :346
      if (fe.det_n[s] > 20) fe.image_state[s] = 2;           // :348, :160-161
    }
  }
  if (publish) {
    const int n = tn.n[s];
    const double t_prev = fe.prev_img_time[s], t_pub = fe.last_pub_time[s];
    const double dt_1 = t - t_prev;
    const bool prev_is_last = (t_prev == t_pub);
    const double dt_2 = prev_is_last ? dt_1 : (t_prev - t_pub);
    for (int i = tid; i < n; i += blockDim.x) {
      const float2 pc = tn.curr[base + i], pp = tn.prev[base + i], pi = tn.init[base + i];
      // undistortPoints with identity new camera: normalised coordinates as float
      LvbFeature f;
      // (inlined radtan/equidistant undistortion, see fe_orb.cu:undistort_one)
      const float2 cu = lvb_undistort_point(cam, pc, 0);
      const float2 pu = lvb_undistort_point(cam, pp, 0);
      f.id = tn.ids[base + i];
      f.u = (double)cu.x; f.v = (double)cu.y;
      f.u_vel = (double)__fsub_rn(cu.x, pu.x) / dt_1;
      f.v_vel = (double)__fsub_rn(cu.y, pu.y) / dt_1;
      f.u_init = 0; f.v_init = 0; f.u_init_vel = 0; f.v_init_vel = 0;
      if (pi.x == -1.f && pi.y == -1.f) {
        f.u_init = -1; f.v_init = -1;
      } else {
        const float2 iu = lvb_undistort_point(cam, pi, 0);
        f.u_init = (double)iu.x; f.v_init = (double)iu.y;
        tn.init[base + i] = make_float2(-1.f, -1.f);
        const float2 aa = prev_is_last ? cu : pu;
        f.u_init_vel = (double)__fsub_rn(aa.x, iu.x) / dt_2;
        f.v_init_vel = (double)__fsub_rn(aa.y, iu.y) / dt_2;
      }
      fe.msg[base + i] = f;
    }
    __syncthreads();
    if (tid == 0) { fe.msg_n[s] = n; fe.has_msg[s] = 1; fe.msg_t[s] = t; fe.last_pub_time[s] = t; atomicAdd(&fe.stats[3], 1ull); }
  }
  __syncthreads();
  if (tid == 0) fe.prev_img_time[s] = t;
}

}  // namespace

// ====================================================================== host orchestration
static FeView make_view(LvbHandle* h) {
  FeView v;
  v.fe = h->fe; v.cur = h->fe.cur;
  v.max_features = h->cfg.max_features_num;
  v.pub_frequency = (int)h->cfg.pub_frequency;
  return v;
}

static int run_compaction(LvbHandle* h, int stage) {
  LvbFrontEnd& fe = h->fe;
  CompactArgs ca;
  ca.ch[0] = fe.ch[0]; ca.ch[1] = fe.ch[1]; ca.N = fe.N; ca.stats = fe.stats; ca.stage = stage;
  ca.min_keep[0] = 1;
  ca.min_keep[1] = (stage == 2) ? 20 : 1;      // trackNewFeatures: "<20" only after the descriptor gate (:941)
  ca.store_curr = (stage == 0);
  ca.second = fe.do_second; ca.min_keep_second = 20;   // initializeFirstFeatures: "<20" after every gate
  LVB_PROF(h, "compact_kernel");
  compact_kernel<<<dim3(fe.S, 2), fe.N, 0, h->stream>>>(ca);
  LVB_LAUNCH_CHECK(h);
  return LVB_OK;
}

#define RC(x) do { int rc_ = (x); if (rc_ != LVB_OK) return rc_; } while (0)

// processImage for the whole batch in three pieces, shared by the plain path (fe_process) and the one-graph-per-step path
// (lvb_step_graph in be_pipeline.cu): host preparation, a capturable enqueue, and the ping-pong toggle.
//
// Host part of processImage: bFirstImg gate (:134-142), integrateImuData (:184, :359) and the image batch copy.  Returns in
// *d_images the device pointer the enqueue reads: the caller's own pointer for device-resident input, fe.img_in otherwise
// (or always, with stage_to_img_in, so that a captured graph sees one fixed source).
int fe_host_prep(LvbHandle* h, const uint8_t* images, int on_device, const double* t_img, const LvbImu* imu, const int* n_imu,
                 int imu_stride, bool stage_to_img_in, const uint8_t** d_images) {
  LvbFrontEnd& fe = h->fe;
  const int S = fe.S;
  cudaStream_t st = h->stream;
  const size_t npx = (size_t)fe.W * fe.H;
  // the pinned staging buffers of the previous call must have been consumed
  LVB_CUDA(cudaStreamSynchronize(st));
  for (int s = 0; s < S; ++s) {
    const LvbImu* b = imu + (size_t)s * imu_stride;
    const int nb = n_imu[s];
    if (!h->h_first_img[s]) {
      if (nb > 0 && b[0].t - t_img[s] <= 0.0) h->h_first_img[s] = 1;
    }
    const int act = h->h_first_img[s];
    h->pin_active[s] = act;
    h->pin_t[s] = t_img[s];
    float* H = h->pin_H + (size_t)s * 9;
    if (act && h->h_have_prev[s]) predict_homography(h->cfg, b, nb, h->h_prev_img_time[s], t_img[s], H);
    else { for (int i = 0; i < 9; ++i) H[i] = (i % 4 == 0) ? 1.f : 0.f; }
    if (act) { h->h_prev_img_time[s] = t_img[s]; h->h_have_prev[s] = 1; }
  }
  *d_images = images;
  if (!on_device) {
    // caller buffers that are already page-locked are copied directly; pageable ones go through pinned staging
    cudaPointerAttributes pa;
    const bool pinned = cudaPointerGetAttributes(&pa, images) == cudaSuccess && pa.type == cudaMemoryTypeHost;
    if (!pinned) { cudaGetLastError(); memcpy(h->pin_images, images, S * npx); }
    LVB_CUDA(cudaMemcpyAsync(fe.img_in, pinned ? images : h->pin_images, S * npx, cudaMemcpyHostToDevice, st));
    *d_images = fe.img_in;
  } else if (stage_to_img_in) {
    LVB_CUDA(cudaMemcpyAsync(fe.img_in, images, S * npx, cudaMemcpyDeviceToDevice, st));
    *d_images = fe.img_in;
  }
  return LVB_OK;
}

// Every launch of processImage for the batch (fixed sequence: grids follow capacities, decisions are device-side flags).
int fe_enqueue(LvbHandle* h, const uint8_t* d_images) {
  LvbFrontEnd& fe = h->fe;
  const int S = fe.S, N = fe.N;
  cudaStream_t st = h->stream;
  LVB_CUDA(cudaMemcpyAsync(fe.Hmat, h->pin_H, sizeof(float) * 9 * S, cudaMemcpyHostToDevice, st));
  LVB_CUDA(cudaMemcpyAsync(fe.active, h->pin_active, sizeof(int) * S, cudaMemcpyHostToDevice, st));
  LVB_CUDA(cudaMemcpyAsync(fe.t_img, h->pin_t, sizeof(double) * S, cudaMemcpyHostToDevice, st));
  const int cur = fe.cur, prv = cur ^ 1;
  RC(fe_build_pyramid(h, d_images, S, fe.pyr[cur], fe.blur[cur]));
  FeView v = make_view(h);
  LVB_PROF(h, "frame_begin_kernel");
  frame_begin_kernel<<<(S + 127) / 128, 128, 0, st>>>(v);
  LVB_LAUNCH_CHECK(h);
  LVB_PROF(h, "iota_perm_kernel");
  iota_perm_kernel<<<dim3((N + 127) / 128, S), 128, 0, st>>>(v);
  LVB_LAUNCH_CHECK(h);
  const float2* src[2] = {fe.trk[prv].curr, fe.new_pts};
  int* perm2[2] = {fe.ch[0].perm, fe.ch[1].perm};
  int* n2[2] = {fe.ch[0].n, fe.ch[1].n};
  float2* out2[2] = {fe.ch[0].out, fe.ch[1].out};
  uint8_t* st2[2] = {fe.ch[0].status, fe.ch[1].status};
  const float2* cur2[2] = {fe.ch[0].slot_curr, fe.ch[1].slot_curr};
  // forward LK (+ in-image gate), tracked and new chains in one launch
  RC(fe_lk_launch2(h, fe.pyr[prv], fe.pyr[cur], S, N, src, perm2, n2, nullptr, 0, fe.Hmat, out2, st2, 1, nullptr));
  RC(run_compaction(h, 0));
  // backward LK (+ in-image + 1-px consistency gate)
  RC(fe_lk_launch2(h, fe.pyr[cur], fe.pyr[prv], S, N, cur2, perm2, n2, src, 1, nullptr, out2, st2, 2, src));
  RC(run_compaction(h, 1));
  // descriptor gate: tracked features against the descriptor stored at birth, new ones prev vs curr (one launch)
  RC(fe_orb_gate_launch(h, fe.pyr[cur], fe.blur[cur], fe.pyr[prv], fe.blur[prv], S, N, cur2, fe.new_pts, perm2, n2, fe.trk[prv].desc,
                        fe.ch[1].desc, st2));
  RC(run_compaction(h, 2));
  // undistort to pixel coordinates + fundamental-matrix RANSAC: both chains in one launch, undistortion fused into its load
  {
    int* fail2[2] = {fe.ch[0].fail, fe.ch[1].fail};
    RC(fe_ransac_launch2(h, S, N, src, cur2, perm2, n2, st2, fail2));
  }
  RC(run_compaction(h, 3));
  LVB_PROF(h, "finalize_kernel");
  finalize_kernel<<<S, 256, 0, st>>>(v);
  LVB_LAUNCH_CHECK(h);
  RC(fe_detect_launch(h, fe.pyr[cur], S, fe.do_detect, 1, nullptr, fe.trk[cur].curr, fe.mask_n, fe.want, fe.det_pts, fe.det_n));
  LVB_PROF(h, "publish_kernel");
  publish_kernel<<<S, 256, 0, st>>>(v, lvb_camera(h->cfg));
  LVB_LAUNCH_CHECK(h);
  return LVB_OK;
}

int fe_process(LvbHandle* h, const uint8_t* images, int on_device, const double* t_img, const LvbImu* imu,
               const int* n_imu, int imu_stride) {
  const uint8_t* d_images = nullptr;
  RC(fe_host_prep(h, images, on_device, t_img, imu, n_imu, imu_stride, false, &d_images));
  RC(fe_enqueue(h, d_images));
  h->fe.cur ^= 1;
  return LVB_OK;
}

int fe_fetch_messages(LvbHandle* h, LvbFeature* out_feat, int* out_n, uint8_t* has_features) {
  LvbFrontEnd& fe = h->fe;
  const int S = fe.S, N = fe.N;
  cudaStream_t st = h->stream;
  LVB_CUDA(cudaMemcpyAsync(h->pin_msg, fe.msg, sizeof(LvbFeature) * (size_t)S * N, cudaMemcpyDeviceToHost, st));
  LVB_CUDA(cudaMemcpyAsync(h->pin_msg_n, fe.msg_n, sizeof(int) * S, cudaMemcpyDeviceToHost, st));
  LVB_CUDA(cudaMemcpyAsync(h->pin_has, fe.has_msg, S, cudaMemcpyDeviceToHost, st));
  int ovf = 0;
  LVB_CUDA(cudaMemcpyAsync(&ovf, fe.overflow, sizeof(int), cudaMemcpyDeviceToHost, st));
  LVB_CUDA(cudaStreamSynchronize(st));
  if (ovf) return lvb_set_err(LVB_E_CAPACITY, "corner candidate buffer overflow (cap %d per sequence)", fe.cand_cap);
  for (int s = 0; s < S; ++s) {
    has_features[s] = h->pin_has[s];
    out_n[s] = h->pin_has[s] ? h->pin_msg_n[s] : 0;
    if (out_feat && out_n[s] > 0) memcpy(out_feat + (size_t)s * N, h->pin_msg + (size_t)s * N, sizeof(LvbFeature) * out_n[s]);
  }
  return LVB_OK;
}

extern "C" int lvb_process_images(LvbHandle* h, const uint8_t* images, const double* t_img, const LvbImu* imu,
                                  const int* n_imu, int imu_stride, LvbFeature* out_feat, int* out_n,
                                  uint8_t* has_features) {
  if (!h || !images || !t_img || !imu || !n_imu || !out_n || !has_features)
    return lvb_set_err(LVB_E_ARG, "lvb_process_images: null argument");
  LVB_CUDA(cudaSetDevice(h->device));
  RC(fe_process(h, images, 0, t_img, imu, n_imu, imu_stride));
  return fe_fetch_messages(h, out_feat, out_n, has_features);
}
