// C ABI entry points (include/larvio_b200.h): handle life cycle + stage-level test entry points.
#include <stdarg.h>
#include <string.h>
#include <math.h>
#include "lvb_internal.h"
#include "be_state.h"

thread_local std::string g_lvb_err;

int lvb_set_err(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_lvb_err = buf;
  return code;
}

extern "C" const char* lvb_last_error(void) { return g_lvb_err.c_str(); }

template <typename T>
static int dalloc(LvbHandle* h, T** p, size_t count, bool zero = true) {
  void* q = nullptr;
  size_t bytes = count * sizeof(T);
  if (bytes == 0) bytes = sizeof(T);
  LVB_CUDA(cudaMalloc(&q, bytes));
  if (zero) LVB_CUDA(cudaMemsetAsync(q, 0, bytes, h->stream));
  h->allocs.push_back(q);
  *p = (T*)q;
  return LVB_OK;
}

static void build_layout(LvbPyramidLayout& L, int W, int H, int levels) {
  L.n_levels = levels + 1;
  size_t off = 0;
  int w = W, hh = H;
  for (int l = 0; l <= levels; ++l) {
    LvbLevel& lv = L.lv[l];
    lv.w = w; lv.h = hh;
    lv.pitch = ((w + 2 * LVB_PAD + 31) / 32) * 32;
    lv.rows = hh + 2 * LVB_PAD;
    lv.offset = off;
    off += (size_t)lv.pitch * lv.rows;
    off = (off + 255) & ~(size_t)255;
    w = (w + 1) / 2; hh = (hh + 1) / 2;
  }
  L.bytes_per_seq = off + 256;   // slack: App. C-10 one-past-pad reads stay inside the allocation
}

int fe_alloc(LvbHandle* h);   // fe_pipeline.cu
int be_alloc(LvbHandle* h);   // be_pipeline.cu
void be_free(LvbHandle* h);

extern "C" int lvb_create(const LvbConfig* cfg, int n_seq, int device, LvbHandle** out) {
  if (!cfg || !out || n_seq <= 0) return lvb_set_err(LVB_E_ARG, "lvb_create: bad argument");
  if (cfg->width % 8 || cfg->height % 8 || cfg->width % 4)
    return lvb_set_err(LVB_E_UNSUPPORTED, "image size %dx%d: CLAHE tiles need multiples of 8", cfg->width, cfg->height);
  if (cfg->pyramid_levels + 1 > LVB_MAX_LEVELS || cfg->pyramid_levels < 0)
    return lvb_set_err(LVB_E_UNSUPPORTED, "pyramid_levels %d", cfg->pyramid_levels);
  if ((cfg->width >> cfg->pyramid_levels) <= LVB_PAD + 1 || (cfg->height >> cfg->pyramid_levels) <= LVB_PAD + 1)
    return lvb_set_err(LVB_E_UNSUPPORTED, "image %dx%d with %d pyramid levels: the top level must exceed the %d-px pad", cfg->width, cfg->height, cfg->pyramid_levels, LVB_PAD);
  if (cfg->patch_size != 21) return lvb_set_err(LVB_E_UNSUPPORTED, "patch_size %d (LK kernel is specialised for 21)", cfg->patch_size);
  int ndev = 0;
  LVB_CUDA(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return lvb_set_err(LVB_E_ARG, "device %d of %d", device, ndev);
  LVB_CUDA(cudaSetDevice(device));
  LvbHandle* h = new LvbHandle();
  h->cfg = *cfg; h->S = n_seq; h->device = device; h->launches = 0; h->be = nullptr;
  h->pin_images = nullptr; h->pin_images_bytes = 0;
  LVB_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  LvbFrontEnd& fe = h->fe;
  memset(&fe, 0, sizeof(fe));
  fe.S = n_seq; fe.W = cfg->width; fe.H = cfg->height;
  fe.N = ((cfg->max_features_num + 31) / 32) * 32;
  build_layout(fe.L, fe.W, fe.H, cfg->pyramid_levels);
  int rc = fe_alloc(h);
  if (rc == LVB_OK) rc = be_alloc(h);
  if (rc != LVB_OK) { lvb_destroy(h); return rc; }
  h->h_first_img.assign(n_seq, 0);
  h->h_prev_img_time.assign(n_seq, 0.0);
  h->h_have_prev.assign(n_seq, 0);
  LVB_CUDA(cudaStreamSynchronize(h->stream));
  *out = h;
  return LVB_OK;
}

extern "C" int lvb_create_from_file(const char* yaml_path, int n_seq, int device, LvbHandle** out) {
  LvbConfig cfg;
  int rc = lvb_parse_config(yaml_path, &cfg);
  if (rc != LVB_OK) return rc;
  return lvb_create(&cfg, n_seq, device, out);
}

extern "C" void lvb_destroy(LvbHandle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  for (int i = 0; i < 2; ++i) if (h->gexec[i]) cudaGraphExecDestroy(h->gexec[i]);
  be_free(h);
  for (void* p : h->allocs) cudaFree(p);
  if (h->pin_images) cudaFreeHost(h->pin_images);
  if (h->pin_H) cudaFreeHost(h->pin_H);
  if (h->pin_active) cudaFreeHost(h->pin_active);
  if (h->pin_t) cudaFreeHost(h->pin_t);
  if (h->pin_msg) cudaFreeHost(h->pin_msg);
  if (h->pin_msg_n) cudaFreeHost(h->pin_msg_n);
  if (h->pin_has) cudaFreeHost(h->pin_has);
  cudaStreamDestroy(h->stream);
  delete h;
}

extern "C" int lvb_feature_capacity(const LvbHandle* h) { return h ? h->fe.N : 0; }
extern "C" int lvb_n_seq(const LvbHandle* h) { return h ? h->S : 0; }
extern "C" long long lvb_launch_count(const LvbHandle* h) { return h ? h->launches : 0; }
extern "C" int lvb_synchronize(LvbHandle* h) {
  if (!h) return LVB_E_ARG;
  LVB_CUDA(cudaStreamSynchronize(h->stream));
  return LVB_OK;
}

// ------------------------------------------------------------------ stage-level entry points
namespace {
struct TmpBuf {
  std::vector<void*> p;
  ~TmpBuf() { for (void* q : p) cudaFree(q); }
  template <typename T> T* get(size_t n) {
    void* q = nullptr;
    if (cudaMalloc(&q, n * sizeof(T) + 16) != cudaSuccess) return nullptr;
    p.push_back(q);
    return (T*)q;
  }
};

__global__ void unpad_kernel(const uint8_t* pyr, LvbPyramidLayout L, int level, uint8_t* out) {
  const int s = blockIdx.z;
  const LvbLevel lv = L.lv[level];
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= lv.w || y >= lv.h) return;
  out[(size_t)s * lv.w * lv.h + (size_t)y * lv.w + x] = lvb_level_origin(pyr, L, s, level)[(ptrdiff_t)y * lv.pitch + x];
}
}  // namespace

extern "C" int lvbk_pyramid(LvbHandle* h, const uint8_t* images, int n, uint8_t* clahe, uint8_t* l1,
                            uint8_t* l2, uint8_t* blur) {
  if (!h || !images || n <= 0) return lvb_set_err(LVB_E_ARG, "lvbk_pyramid: bad argument");
  LVB_CUDA(cudaSetDevice(h->device));
  LvbFrontEnd& fe = h->fe;
  TmpBuf tb;
  const size_t npx = (size_t)fe.W * fe.H;
  uint8_t* d_img = tb.get<uint8_t>(npx * n);
  uint8_t* d_pyr = tb.get<uint8_t>(fe.L.bytes_per_seq * n);
  uint8_t* d_blur = tb.get<uint8_t>(npx * n);
  uint8_t* d_out = tb.get<uint8_t>(npx * n);
  uint8_t* d_lut = tb.get<uint8_t>((size_t)n * 64 * 256);
  if (!d_img || !d_pyr || !d_blur || !d_out || !d_lut) return lvb_set_err(LVB_E_CUDA, "lvbk_pyramid: cudaMalloc failed");
  LVB_CUDA(cudaMemcpyAsync(d_img, images, npx * n, cudaMemcpyHostToDevice, h->stream));
  uint8_t* saved = fe.lut; fe.lut = d_lut;
  int rc = fe_build_pyramid(h, d_img, n, d_pyr, d_blur);
  fe.lut = saved;
  if (rc != LVB_OK) return rc;
  uint8_t* outs[3] = {clahe, l1, l2};
  for (int l = 0; l < 3 && l < fe.L.n_levels; ++l) {
    if (!outs[l]) continue;
    const LvbLevel& lv = fe.L.lv[l];
    dim3 blk(32, 8), grd((lv.w + 31) / 32, (lv.h + 7) / 8, n);
    LVB_PROF(h, "unpad_kernel");
    unpad_kernel<<<grd, blk, 0, h->stream>>>(d_pyr, fe.L, l, d_out);
    LVB_LAUNCH_CHECK(h);
    LVB_CUDA(cudaMemcpyAsync(outs[l], d_out, (size_t)lv.w * lv.h * n, cudaMemcpyDeviceToHost, h->stream));
    LVB_CUDA(cudaStreamSynchronize(h->stream));
  }
  if (blur) LVB_CUDA(cudaMemcpyAsync(blur, d_blur, npx * n, cudaMemcpyDeviceToHost, h->stream));
  LVB_CUDA(cudaStreamSynchronize(h->stream));
  return LVB_OK;
}

// Level `level` of the pyramid lvbk_pyramid builds, WITH its LVB_PAD-wide REFLECT_101 pad: out [n][h + 2 LVB_PAD][w + 2 LVB_PAD].
extern "C" int lvbk_pyramid_padded(LvbHandle* h, const uint8_t* images, int n, int level, uint8_t* out) {
  if (!h || !images || !out || n <= 0) return lvb_set_err(LVB_E_ARG, "lvbk_pyramid_padded: bad argument");
  LvbFrontEnd& fe = h->fe;
  if (level < 0 || level >= fe.L.n_levels) return lvb_set_err(LVB_E_ARG, "lvbk_pyramid_padded: level %d outside [0, %d)", level, fe.L.n_levels);
  LVB_CUDA(cudaSetDevice(h->device));
  TmpBuf tb;
  const size_t npx = (size_t)fe.W * fe.H;
  uint8_t* d_img = tb.get<uint8_t>(npx * n);
  uint8_t* d_pyr = tb.get<uint8_t>(fe.L.bytes_per_seq * n);
  uint8_t* d_lut = tb.get<uint8_t>((size_t)n * 64 * 256);
  if (!d_img || !d_pyr || !d_lut) return lvb_set_err(LVB_E_CUDA, "lvbk_pyramid_padded: cudaMalloc failed");
  LVB_CUDA(cudaMemcpyAsync(d_img, images, npx * n, cudaMemcpyHostToDevice, h->stream));
  uint8_t* saved = fe.lut; fe.lut = d_lut;
  int rc = fe_build_pyramid(h, d_img, n, d_pyr, nullptr);
  fe.lut = saved;
  if (rc != LVB_OK) return rc;
  const LvbLevel& lv = fe.L.lv[level];
  const size_t row = (size_t)lv.w + 2 * LVB_PAD, rows = (size_t)lv.h + 2 * LVB_PAD;
  for (int s = 0; s < n; ++s)
    LVB_CUDA(cudaMemcpy2DAsync(out + (size_t)s * rows * row, row, d_pyr + (size_t)s * fe.L.bytes_per_seq + lv.offset, lv.pitch,
                               row, rows, cudaMemcpyDeviceToHost, h->stream));
  LVB_CUDA(cudaStreamSynchronize(h->stream));
  return LVB_OK;
}

extern "C" int lvbk_lk(LvbHandle* h, const uint8_t* prev, const uint8_t* next, int n, int m,
                       const float* prev_pts, float* next_pts, uint8_t* status) {
  if (!h || !prev || !next || n <= 0 || m <= 0) return lvb_set_err(LVB_E_ARG, "lvbk_lk: bad argument");
  LVB_CUDA(cudaSetDevice(h->device));
  LvbFrontEnd& fe = h->fe;
  TmpBuf tb;
  const size_t npx = (size_t)fe.W * fe.H;
  uint8_t* d_img = tb.get<uint8_t>(npx * n);
  uint8_t* d_pa = tb.get<uint8_t>(fe.L.bytes_per_seq * n);
  uint8_t* d_pb = tb.get<uint8_t>(fe.L.bytes_per_seq * n);
  uint8_t* d_lut = tb.get<uint8_t>((size_t)n * 64 * 256);
  float2* d_p = tb.get<float2>((size_t)n * m);
  float2* d_q = tb.get<float2>((size_t)n * m);
  float2* d_o = tb.get<float2>((size_t)n * m);
  uint8_t* d_st = tb.get<uint8_t>((size_t)n * m);
  int* d_n = tb.get<int>(n);
  if (!d_img || !d_pa || !d_pb || !d_lut || !d_p || !d_q || !d_o || !d_st || !d_n)
    return lvb_set_err(LVB_E_CUDA, "lvbk_lk: cudaMalloc failed");
  std::vector<int> cnt(n, m);
  LVB_CUDA(cudaMemcpyAsync(d_n, cnt.data(), n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  uint8_t* saved = fe.lut; fe.lut = d_lut;
  const int eq = h->cfg.flag_equalize; h->cfg.flag_equalize = 0;   // inputs are already equalised
  LVB_CUDA(cudaMemcpyAsync(d_img, prev, npx * n, cudaMemcpyHostToDevice, h->stream));
  int rc = fe_build_pyramid(h, d_img, n, d_pa, nullptr);
  if (rc == LVB_OK) {
    LVB_CUDA(cudaMemcpyAsync(d_img, next, npx * n, cudaMemcpyHostToDevice, h->stream));
    rc = fe_build_pyramid(h, d_img, n, d_pb, nullptr);
  }
  h->cfg.flag_equalize = eq; fe.lut = saved;
  if (rc != LVB_OK) return rc;
  LVB_CUDA(cudaMemcpyAsync(d_p, prev_pts, (size_t)n * m * sizeof(float2), cudaMemcpyHostToDevice, h->stream));
  LVB_CUDA(cudaMemcpyAsync(d_q, next_pts, (size_t)n * m * sizeof(float2), cudaMemcpyHostToDevice, h->stream));
  rc = fe_lk_launch(h, d_pa, d_pb, n, m, d_p, nullptr, d_n, d_q, 0, nullptr, d_o, d_st, 0, nullptr);
  if (rc != LVB_OK) return rc;
  LVB_CUDA(cudaMemcpyAsync(next_pts, d_o, (size_t)n * m * sizeof(float2), cudaMemcpyDeviceToHost, h->stream));
  LVB_CUDA(cudaMemcpyAsync(status, d_st, (size_t)n * m, cudaMemcpyDeviceToHost, h->stream));
  LVB_CUDA(cudaStreamSynchronize(h->stream));
  return LVB_OK;
}

extern "C" int lvbk_orb(LvbHandle* h, const uint8_t* images, int n, int m, const float* pts, float* angles,
                        uint8_t* desc) {
  if (!h || !images || !pts || n <= 0 || m <= 0) return lvb_set_err(LVB_E_ARG, "lvbk_orb: bad argument");
  LVB_CUDA(cudaSetDevice(h->device));
  LvbFrontEnd& fe = h->fe;
  TmpBuf tb;
  const size_t npx = (size_t)fe.W * fe.H;
  uint8_t* d_img = tb.get<uint8_t>(npx * n);
  uint8_t* d_pyr = tb.get<uint8_t>(fe.L.bytes_per_seq * n);
  uint8_t* d_blur = tb.get<uint8_t>(npx * n);
  uint8_t* d_lut = tb.get<uint8_t>((size_t)n * 64 * 256);
  float2* d_p = tb.get<float2>((size_t)n * m);
  float* d_a = tb.get<float>((size_t)n * m);
  uint8_t* d_d = tb.get<uint8_t>((size_t)n * m * 32);
  int* d_n = tb.get<int>(n);
  if (!d_img || !d_pyr || !d_blur || !d_lut || !d_p || !d_a || !d_d || !d_n) return lvb_set_err(LVB_E_CUDA, "lvbk_orb: cudaMalloc failed");
  std::vector<int> cnt(n, m);
  LVB_CUDA(cudaMemcpyAsync(d_n, cnt.data(), n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  LVB_CUDA(cudaMemcpyAsync(d_img, images, npx * n, cudaMemcpyHostToDevice, h->stream));
  LVB_CUDA(cudaMemcpyAsync(d_p, pts, (size_t)n * m * sizeof(float2), cudaMemcpyHostToDevice, h->stream));
  uint8_t* saved = fe.lut; fe.lut = d_lut;
  const int eq = h->cfg.flag_equalize; h->cfg.flag_equalize = 0;
  int rc = fe_build_pyramid(h, d_img, n, d_pyr, d_blur);
  h->cfg.flag_equalize = eq; fe.lut = saved;
  if (rc != LVB_OK) return rc;
  rc = fe_orb_launch(h, d_pyr, d_blur, n, m, d_p, nullptr, d_n, d_a, d_d, 0, nullptr, nullptr, nullptr);
  if (rc != LVB_OK) return rc;
  if (angles) LVB_CUDA(cudaMemcpyAsync(angles, d_a, (size_t)n * m * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  if (desc) LVB_CUDA(cudaMemcpyAsync(desc, d_d, (size_t)n * m * 32, cudaMemcpyDeviceToHost, h->stream));
  LVB_CUDA(cudaStreamSynchronize(h->stream));
  return LVB_OK;
}

extern "C" int lvbk_detect(LvbHandle* h, const uint8_t* images, const uint8_t* masks, int n, const int* want,
                           float* out_pts, int* out_n, float* eig_map) {
  if (!h || !images || !want || !out_pts || !out_n || n <= 0) return lvb_set_err(LVB_E_ARG, "lvbk_detect: bad argument");
  if (n > h->S) return lvb_set_err(LVB_E_ARG, "lvbk_detect: n (%d) exceeds the handle's sequence count (%d)", n, h->S);
  LVB_CUDA(cudaSetDevice(h->device));
  LvbFrontEnd& fe = h->fe;
  TmpBuf tb;
  const size_t npx = (size_t)fe.W * fe.H;
  uint8_t* d_img = tb.get<uint8_t>(npx * n);
  uint8_t* d_pyr = tb.get<uint8_t>(fe.L.bytes_per_seq * n);
  uint8_t* d_lut = tb.get<uint8_t>((size_t)n * 64 * 256);
  uint8_t* d_mask = masks ? tb.get<uint8_t>(npx * n) : nullptr;
  int* d_want = tb.get<int>(n);
  float2* d_out = tb.get<float2>((size_t)n * fe.N);
  int* d_cnt = tb.get<int>(n);
  float* d_eig = eig_map ? tb.get<float>(npx * n) : nullptr;
  if (!d_img || !d_pyr || !d_lut || !d_want || !d_out || !d_cnt || (masks && !d_mask) || (eig_map && !d_eig)) return lvb_set_err(LVB_E_CUDA, "lvbk_detect: cudaMalloc failed");
  LVB_CUDA(cudaMemcpyAsync(d_img, images, npx * n, cudaMemcpyHostToDevice, h->stream));
  if (masks) LVB_CUDA(cudaMemcpyAsync(d_mask, masks, npx * n, cudaMemcpyHostToDevice, h->stream));
  LVB_CUDA(cudaMemcpyAsync(d_want, want, n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  uint8_t* saved = fe.lut; fe.lut = d_lut;
  const int eq = h->cfg.flag_equalize; h->cfg.flag_equalize = 0;
  int rc = fe_build_pyramid(h, d_img, n, d_pyr, nullptr);
  h->cfg.flag_equalize = eq; fe.lut = saved;
  if (rc != LVB_OK) return rc;
  rc = fe_detect_launch(h, d_pyr, n, nullptr, 0, d_mask, nullptr, nullptr, d_want, d_out, d_cnt, d_eig);
  if (rc != LVB_OK) return rc;
  LVB_CUDA(cudaMemcpyAsync(out_pts, d_out, (size_t)n * fe.N * sizeof(float2), cudaMemcpyDeviceToHost, h->stream));
  LVB_CUDA(cudaMemcpyAsync(out_n, d_cnt, n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  if (eig_map) LVB_CUDA(cudaMemcpyAsync(eig_map, d_eig, npx * n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  int ovf = 0;
  LVB_CUDA(cudaMemcpyAsync(&ovf, fe.overflow, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  LVB_CUDA(cudaStreamSynchronize(h->stream));
  if (ovf) return lvb_set_err(LVB_E_CAPACITY, "corner candidate buffer overflow");
  return LVB_OK;
}

extern "C" int lvbk_undistort(LvbHandle* h, const float* pts, int m, int to_pixels, float* out) {
  if (!h || !pts || !out || m <= 0) return lvb_set_err(LVB_E_ARG, "lvbk_undistort: bad argument");
  LVB_CUDA(cudaSetDevice(h->device));
  TmpBuf tb;
  float2* d_p = tb.get<float2>(m); float2* d_o = tb.get<float2>(m); int* d_n = tb.get<int>(1);
  if (!d_p || !d_o || !d_n) return lvb_set_err(LVB_E_CUDA, "lvbk_undistort: cudaMalloc failed");
  LVB_CUDA(cudaMemcpyAsync(d_p, pts, sizeof(float2) * m, cudaMemcpyHostToDevice, h->stream));
  LVB_CUDA(cudaMemcpyAsync(d_n, &m, sizeof(int), cudaMemcpyHostToDevice, h->stream));
  int rc = fe_undistort_launch(h, 1, m, d_p, nullptr, d_n, d_o, to_pixels);
  if (rc != LVB_OK) return rc;
  LVB_CUDA(cudaMemcpyAsync(out, d_o, sizeof(float2) * m, cudaMemcpyDeviceToHost, h->stream));
  LVB_CUDA(cudaStreamSynchronize(h->stream));
  return LVB_OK;
}

extern "C" int lvbk_ransac(LvbHandle* h, const float* p1, const float* p2, int n, const int* m, int stride,
                           uint8_t* mask) {
  if (!h || !p1 || !p2 || !m || !mask || n <= 0 || stride <= 0) return lvb_set_err(LVB_E_ARG, "lvbk_ransac: bad argument");
  LVB_CUDA(cudaSetDevice(h->device));
  TmpBuf tb;
  const size_t tot = (size_t)n * stride;
  float2* d1 = tb.get<float2>(tot); float2* d2 = tb.get<float2>(tot); int* dn = tb.get<int>(n);
  uint8_t* dm = tb.get<uint8_t>(tot);
  if (!d1 || !d2 || !dn || !dm) return lvb_set_err(LVB_E_CUDA, "lvbk_ransac: cudaMalloc failed");
  LVB_CUDA(cudaMemcpyAsync(d1, p1, tot * sizeof(float2), cudaMemcpyHostToDevice, h->stream));
  LVB_CUDA(cudaMemcpyAsync(d2, p2, tot * sizeof(float2), cudaMemcpyHostToDevice, h->stream));
  LVB_CUDA(cudaMemcpyAsync(dn, m, n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  LVB_CUDA(cudaMemsetAsync(dm, 0, tot, h->stream));
  int rc = fe_ransac_launch(h, n, stride, d1, d2, dn, dm, nullptr, nullptr);
  if (rc != LVB_OK) return rc;
  LVB_CUDA(cudaMemcpyAsync(mask, dm, tot, cudaMemcpyDeviceToHost, h->stream));
  LVB_CUDA(cudaStreamSynchronize(h->stream));
  return LVB_OK;
}

// ------------------------------------------------------------------ per-kernel timing
void lvb_prof_begin(LvbHandle* h, const char* name) {
  LvbProfiler& p = h->prof;
  int id = -1;
  for (size_t i = 0; i < p.names.size(); ++i) if (p.names[i] == name) { id = (int)i; break; }
  if (id < 0) { id = (int)p.names.size(); p.names.push_back(name); p.total_ms.push_back(0.0); p.count.push_back(0); }
  if ((size_t)(2 * p.used + 2) > p.ev.size()) {
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    p.ev.push_back(a); p.ev.push_back(b); p.ev_name.push_back(id);
  } else p.ev_name[p.used] = id;
  cudaEventRecord(p.ev[2 * p.used], h->stream);
  p.open_name = id;
}
void lvb_prof_end(LvbHandle* h) {
  LvbProfiler& p = h->prof;
  if (p.open_name < 0) return;
  cudaEventRecord(p.ev[2 * p.used + 1], h->stream);
  p.used++;
  p.open_name = -1;
}
static void lvb_prof_collect(LvbHandle* h) {
  LvbProfiler& p = h->prof;
  cudaStreamSynchronize(h->stream);
  for (int i = 0; i < p.used; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, p.ev[2 * i], p.ev[2 * i + 1]) == cudaSuccess) { p.total_ms[p.ev_name[i]] += ms; p.count[p.ev_name[i]]++; }
  }
  p.used = 0;
}
extern "C" int lvb_profile_enable(LvbHandle* h, int on) {
  if (!h) return LVB_E_ARG;
  cudaSetDevice(h->device);
  if (!on && h->prof.on) lvb_prof_collect(h);
  h->prof.on = on != 0;
  return LVB_OK;
}
extern "C" int lvb_profile_reset(LvbHandle* h) {
  if (!h) return LVB_E_ARG;
  lvb_prof_collect(h);
  for (auto& x : h->prof.total_ms) x = 0.0;
  for (auto& x : h->prof.count) x = 0;
  return LVB_OK;
}
// Fills up to cap entries; names[i] points into handle-owned storage. Returns the number of kernels.
extern "C" int lvb_profile_get(LvbHandle* h, const char** names, double* total_ms, long long* counts, int cap) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  lvb_prof_collect(h);
  const int n = (int)h->prof.names.size();
  for (int i = 0; i < n && i < cap; ++i) { names[i] = h->prof.names[i].c_str(); total_ms[i] = h->prof.total_ms[i]; counts[i] = h->prof.count[i]; }
  return n;
}

extern "C" int lvb_get_stats(LvbHandle* h, unsigned long long* out16) {
  if (!h || !out16) return lvb_set_err(LVB_E_ARG, "lvb_get_stats: null argument");
  LVB_CUDA(cudaSetDevice(h->device));
  LVB_CUDA(cudaMemcpyAsync(out16, h->fe.stats, sizeof(unsigned long long) * 16, cudaMemcpyDeviceToHost, h->stream));
  LVB_CUDA(cudaStreamSynchronize(h->stream));
  return LVB_OK;
}

// debug: raw per-sequence integer state of the back end (be_state.h I_* indices)
extern "C" int lvb_debug_icore(LvbHandle* h, int seq, int* out32) {
  if (!h || !out32 || seq < 0 || seq >= h->S) return lvb_set_err(LVB_E_ARG, "lvb_debug_icore: bad argument");
  LVB_CUDA(cudaSetDevice(h->device));
  LVB_CUDA(cudaMemcpyAsync(out32, h->be->icore + (size_t)seq * BE_ICORE, sizeof(int) * BE_ICORE, cudaMemcpyDeviceToHost, h->stream));
  LVB_CUDA(cudaStreamSynchronize(h->stream));
  return LVB_OK;
}
