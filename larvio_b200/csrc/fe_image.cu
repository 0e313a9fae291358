// Front-end image stage: CLAHE(3.0, 8x8) -> padded 3-level LK pyramid -> ORB 7x7 blur.
// Replaces ImageProcessor::createImagePyramids (image_processor.cpp:318-334: cv::CLAHE::apply +
// cv::buildOpticalFlowPyramid) and the per-frame work of ORBdescriptor::initializeLayerAndPyramid
// (ORBDescriptor.cpp:418-483, level 0 only).  Integer stages are bit-exact w.r.t. OpenCV 4.13
// (SURVEY.md App. A.1, A.2, A.4); Scharr derivative images are NOT materialised (the LK kernel
// recomputes them from the padded level), which removes 4x the pixel bytes from HBM.
#include <type_traits>
#include "lvb_internal.h"

namespace {

constexpr int kTiles = 8;   // CLAHE tilesX = tilesY = 8

// ---------------------------------------------------------------- CLAHE histogram -> LUT
// grid (64, n): one CTA per tile.  App. A.1.  The tile's rows are read as aligned V-byte words (the widest that W and the
// image base allow), bytes outside the tile masked off, into one sub-histogram per warp.
template <int V>
__global__ void __launch_bounds__(256) clahe_lut_kernel(const uint8_t* __restrict__ img, int W, int H,
                                                         uint8_t* __restrict__ lut, int clip_limit) {
  using Vec = typename std::conditional<V == 16, uint4, typename std::conditional<V == 8, uint2, uint32_t>::type>::type;
  __shared__ int whist[8][256];
  __shared__ int warp_sums[8];
  __shared__ int s_clipped;
  const int tile = blockIdx.x, s = blockIdx.y;
  const int tw = W / kTiles, th = H / kTiles;
  const int tx = tile % kTiles, ty = tile / kTiles;
  const int x0 = tx * tw, xa = x0 & ~(V - 1);                // first aligned word of a tile row
  const int nw = (x0 + tw - xa + V - 1) / V;                 // words per tile row
  const uint8_t* src = img + (size_t)s * W * H + (size_t)(ty * th) * W + xa;
  const int tid = threadIdx.x;
  int* wh = whist[tid >> 5];
#pragma unroll
  for (int w = 0; w < 8; ++w) whist[w][tid] = 0;
  if (tid == 0) s_clipped = 0;
  __syncthreads();
  const int total = tw * th;
  for (int i = tid; i < nw * th; i += 256) {
    const int y = i / nw, q = i - y * nw;
    const Vec v = *reinterpret_cast<const Vec*>(src + (size_t)y * W + q * V);
    const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
    const int xb = xa + q * V;
#pragma unroll
    for (int k = 0; k < V; ++k) {
      const int x = xb + k;
      if (x >= x0 && x < x0 + tw) atomicAdd(&wh[(u[k >> 2] >> (8 * (k & 3))) & 255], 1);
    }
  }
  __syncthreads();
  int hv = 0;
#pragma unroll
  for (int w = 0; w < 8; ++w) hv += whist[w][tid];
  int excess = hv > clip_limit ? hv - clip_limit : 0;
  if (hv > clip_limit) hv = clip_limit;
  // block reduce excess
  int v = excess;
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((tid & 31) == 0) warp_sums[tid >> 5] = v;
  __syncthreads();
  if (tid == 0) {
    int t = 0;
    for (int i = 0; i < 8; ++i) t += warp_sums[i];
    s_clipped = t;
  }
  __syncthreads();
  const int clipped = s_clipped;
  const int batch = clipped / 256;
  int residual = clipped - batch * 256;
  hv += batch;
  if (residual != 0) {
    int step = 256 / residual;
    if (step < 1) step = 1;
    // bins 0, step, 2*step, ... get +1 while residual lasts (and index < 256)
    if (tid % step == 0 && tid / step < residual) hv += 1;
  }
  // inclusive scan of hv over 256 bins
  int x = hv;
  for (int o = 1; o < 32; o <<= 1) {
    int y = __shfl_up_sync(0xffffffffu, x, o);
    if ((tid & 31) >= o) x += y;
  }
  __syncthreads();
  if ((tid & 31) == 31) warp_sums[tid >> 5] = x;
  __syncthreads();
  int base = 0;
  for (int i = 0; i < (tid >> 5); ++i) base += warp_sums[i];
  const int cum = x + base;
  const float lut_scale = 255.0f / (float)total;
  float f = __fmul_rn((float)cum, lut_scale);
  int r = __float2int_rn(f);
  r = r < 0 ? 0 : (r > 255 ? 255 : r);
  lut[((size_t)s * 64 + tile) * 256 + tid] = (uint8_t)r;
}

// REFLECT_101 pad written by the producer of a level: pixel (x, y) of a w x h level is also the value of its mirror images
// -x, 2(w-1)-x (and the same in y) wherever those fall inside the LVB_PAD-wide pad (w, h > LVB_PAD + 1 at every level we build).
__device__ __forceinline__ void store_pad_copies(uint8_t* org, int pitch, int w, int h, int x, int y, uint8_t v) {
  int xs[2], ys[2], nx = 0, ny = 0;
  if (x >= 1 && x <= LVB_PAD) xs[nx++] = -x;
  if (x <= w - 2 && x >= w - 1 - LVB_PAD) xs[nx++] = 2 * (w - 1) - x;
  if (y >= 1 && y <= LVB_PAD) ys[ny++] = -y;
  if (y <= h - 2 && y >= h - 1 - LVB_PAD) ys[ny++] = 2 * (h - 1) - y;
  for (int a = 0; a < nx; ++a) org[(ptrdiff_t)y * pitch + xs[a]] = v;
  for (int b = 0; b < ny; ++b) {
    org[(ptrdiff_t)ys[b] * pitch + x] = v;
    for (int a = 0; a < nx; ++a) org[(ptrdiff_t)ys[b] * pitch + xs[a]] = v;
  }
}

// ---------------------------------------------------------------- CLAHE apply + L0 -> L1 pyrDown + 7x7 blur, one pass
// A CTA owns a 64x32 tile of L0 (32x16 of L1).  It stages the raw image on [X-4, X+68) x [Y-3, Y+35) - the 5x5 pyrDown needs
// a 2-px apron, the 7x7 blur 3 - with REFLECT_101 coordinates, so the apron holds what the level's pad holds: CLAHE is pointwise,
// and CLAHE of the reflected raw pixel is the reflected L0 pixel.  The per-column and per-row tile indices and blend weights are
// computed once, the LUTs of the tiles they name are staged in shared memory, and L0 (+ its pad), L1 (+ its pad) and the blur
// plane are written from the equalised tile.  L2 and further levels come from pyrdown_kernel on L1, whose pad (the reflected L1
// values, which is what cv2.pyrDown of L1 sees) only exists once this kernel is done.
constexpr int FT_W = 64, FT_H = 32;                  // L0 output tile
constexpr int FR_W = FT_W + 8, FR_H = FT_H + 6;      // staged region: x from X - 4 (whole words), y from Y - 3

__global__ void __launch_bounds__(256) clahe_pyr_blur_kernel(const uint8_t* __restrict__ img, int W, int H,
                                                             const uint8_t* __restrict__ lut, uint8_t* __restrict__ pyr,
                                                             LvbPyramidLayout L, uint8_t* __restrict__ blur, int equalize) {
  constexpr int FR_WW = FR_W / 4;                   // words per staged row
  __shared__ uint32_t raw[FR_H][FR_WW];
  __shared__ uint32_t eqw[FR_H][FR_WW];
  __shared__ uint8_t slut[kTiles * kTiles][256];     // only the tiles named by this region are staged
  __shared__ int2 col_t[FR_W], row_t[FR_H];          // tile indices (t1, t2) of the region's columns / rows
  __shared__ float2 col_w[FR_W], row_w[FR_H];        // blend weights (1 - a, a)
  __shared__ int s_tx0, s_tx1, s_ty0, s_ty1;
  __shared__ unsigned short hs[FR_H][FT_W];          // horizontal 7-tap sums of the blur
  const uint8_t (*eq)[FR_W] = reinterpret_cast<const uint8_t (*)[FR_W]>(&eqw[0][0]);
  const int s = blockIdx.z, tid = threadIdx.x;
  const int X = blockIdx.x * FT_W, Y = blockIdx.y * FT_H;
  const uint8_t* src = img + (size_t)s * W * H;
  if (tid == 0) { s_tx0 = kTiles; s_tx1 = -1; s_ty0 = kTiles; s_ty1 = -1; }
  __syncthreads();
  if (X >= 4 && X + FR_W - 4 <= W && Y >= 3 && Y + FR_H - 3 <= H && ((uintptr_t)src & 3) == 0) {
    for (int i = tid; i < FR_H * FR_WW; i += 256) {  // interior tile: no reflection, whole words (W and X - 4 are multiples of 4)
      const int ty = i / FR_WW, q = i - ty * FR_WW;
      raw[ty][q] = __ldg(reinterpret_cast<const uint32_t*>(src + (size_t)(Y - 3 + ty) * W + X - 4) + q);
    }
  } else {
    for (int i = tid; i < FR_H * FR_WW; i += 256) {
      const int ty = i / FR_WW, q = i - ty * FR_WW;
      const uint8_t* row = src + (size_t)lvb_reflect101(Y - 3 + ty, H) * W;
      uint32_t w = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) w |= (uint32_t)__ldg(row + lvb_reflect101(X - 4 + 4 * q + k, W)) << (8 * k);
      raw[ty][q] = w;
    }
  }
  if (equalize) {
    const int tw = W / kTiles, th = H / kTiles;
    if (tid < FR_W + FR_H) {                          // same arithmetic as cv::CLAHE's interpolation body, per column / row
      const bool col = tid < FR_W;
      const int k = col ? tid : tid - FR_W;
      const int p = col ? lvb_reflect101(X - 4 + k, W) : lvb_reflect101(Y - 3 + k, H);
      const float inv = 1.0f / (float)(col ? tw : th);
      const float tf = __fsub_rn(__fmul_rn((float)p, inv), 0.5f);
      int t1 = (int)floorf(tf);
      int t2 = t1 + 1;
      const float wa = __fsub_rn(tf, (float)t1);
      const float wa1 = __fsub_rn(1.0f, wa);
      t1 = max(t1, 0);
      t2 = min(t2, kTiles - 1);
      if (col) { col_t[k] = make_int2(t1, t2); col_w[k] = make_float2(wa1, wa); atomicMin(&s_tx0, t1); atomicMax(&s_tx1, t2); }
      else     { row_t[k] = make_int2(t1 * kTiles, t2 * kTiles); row_w[k] = make_float2(wa1, wa); atomicMin(&s_ty0, t1); atomicMax(&s_ty1, t2); }
    }
    __syncthreads();
    const int tx0 = s_tx0, nx = s_tx1 - tx0 + 1, ty0 = s_ty0, ny = s_ty1 - ty0 + 1;
    const uint32_t* lutS = reinterpret_cast<const uint32_t*>(lut + (size_t)s * kTiles * kTiles * 256);
    for (int i = tid; i < nx * ny * 64; i += 256) {   // 64 words per LUT
      const int t = i >> 6, w = i & 63;
      const int tile = (ty0 + t / nx) * kTiles + tx0 + t % nx;
      reinterpret_cast<uint32_t*>(slut[tile])[w] = __ldg(lutS + tile * 64 + w);
    }
    __syncthreads();
    for (int i = tid; i < FR_H * FR_WW; i += 256) {   // 4 adjacent pixels of one row per item
      const int ty = i / FR_WW, q = i - ty * FR_WW;
      const uint32_t v4 = raw[ty][q];
      const int2 rt = row_t[ty];
      const float2 rw = row_w[ty];
      uint32_t o4 = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int tx = 4 * q + k, v = (v4 >> (8 * k)) & 255;
        const int2 ct = col_t[tx];
        const float2 cw = col_w[tx];
        const float l11 = (float)slut[rt.x + ct.x][v], l12 = (float)slut[rt.x + ct.y][v];
        const float l21 = (float)slut[rt.y + ct.x][v], l22 = (float)slut[rt.y + ct.y][v];
        const float top = __fadd_rn(__fmul_rn(l11, cw.x), __fmul_rn(l12, cw.y));
        const float bot = __fadd_rn(__fmul_rn(l21, cw.x), __fmul_rn(l22, cw.y));
        const float res = __fadd_rn(__fmul_rn(top, rw.x), __fmul_rn(bot, rw.y));
        const int r = __float2int_rn(res);
        o4 |= (uint32_t)(r < 0 ? 0 : (r > 255 ? 255 : r)) << (8 * k);
      }
      eqw[ty][q] = o4;
    }
  } else {
    __syncthreads();
    for (int i = tid; i < FR_H * FR_WW; i += 256) { const int ty = i / FR_WW, q = i - ty * FR_WW; eqw[ty][q] = raw[ty][q]; }
  }
  __syncthreads();
  // L0: 8 adjacent pixels per thread (origin + X is 8-byte aligned), pad copies in the border band
  {
    const LvbLevel l0 = L.lv[0];
    uint8_t* org = lvb_level_origin(pyr, L, s, 0);
    const int ly = tid >> 3, lx = (tid & 7) * 8;
    const int gx = X + lx, gy = Y + ly;
    if (gy < H && gx < W) {
      uint8_t o[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = eq[ly + 3][lx + 4 + k];
      uint8_t* dst = org + (ptrdiff_t)gy * l0.pitch + gx;
      if (gx + 8 <= W) {
        uint2 w;
        w.x = o[0] | (o[1] << 8) | (o[2] << 16) | ((uint32_t)o[3] << 24);
        w.y = o[4] | (o[5] << 8) | (o[6] << 16) | ((uint32_t)o[7] << 24);
        *reinterpret_cast<uint2*>(dst) = w;
      } else {
        for (int k = 0; k < 8 && gx + k < W; ++k) dst[k] = o[k];
      }
      if (gx <= LVB_PAD || gx + 7 >= W - 1 - LVB_PAD || gy <= LVB_PAD || gy >= H - 1 - LVB_PAD)
        for (int k = 0; k < 8 && gx + k < W; ++k) store_pad_copies(org, l0.pitch, W, H, gx + k, gy, o[k]);
    }
  }
  // L1: 2 pixels per thread, 5x5 binomial with (acc + 128) >> 8 (App. A.2)
  if (L.n_levels > 1) {
    const LvbLevel l1 = L.lv[1];
    uint8_t* org = lvb_level_origin(pyr, L, s, 1);
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int i = tid + 256 * r;
      const int ly = i >> 5, lx = i & 31;
      const int gx = X / 2 + lx, gy = Y / 2 + ly;
      if (gx >= l1.w || gy >= l1.h) continue;
      const int cx = 2 * lx + 4, cy = 2 * ly + 3;     // L0 pixel (2 gx, 2 gy) in the staged region
      const int wv[5] = {1, 4, 6, 4, 1};
      int acc = 0;
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        const uint8_t* e = &eq[cy - 2 + j][cx];
        acc += wv[j] * (e[-2] + 4 * e[-1] + 6 * e[0] + 4 * e[1] + e[2]);
      }
      const uint8_t o = (uint8_t)((acc + 128) >> 8);
      org[(ptrdiff_t)gy * l1.pitch + gx] = o;
      if (gx <= LVB_PAD || gx >= l1.w - 1 - LVB_PAD || gy <= LVB_PAD || gy >= l1.h - 1 - LVB_PAD)
        store_pad_copies(org, l1.pitch, l1.w, l1.h, gx, gy, o);
    }
  }
  if (!blur) return;
  // blur: kernel [18 34 48 56 48 34 18]/256 in both directions, out = (acc + 32768) >> 16 (App. A.4)
  const int k7[7] = {18, 34, 48, 56, 48, 34, 18};
  for (int i = tid; i < FR_H * (FT_W / 4); i += 256) {
    const int ty = i / (FT_W / 4), g = i - ty * (FT_W / 4);
    const uint32_t w0 = eqw[ty][g], w1 = eqw[ty][g + 1], w2 = eqw[ty][g + 2];
    int b[12];
#pragma unroll
    for (int q = 0; q < 4; ++q) { b[q] = (w0 >> (8 * q)) & 255; b[4 + q] = (w1 >> (8 * q)) & 255; b[8 + q] = (w2 >> (8 * q)) & 255; }
#pragma unroll
    for (int k = 0; k < 4; ++k) {                     // output column X + 4g + k sits at byte 4 + k; taps at 1 + k .. 7 + k
      int acc = 0;
#pragma unroll
      for (int t = 0; t < 7; ++t) acc += k7[t] * b[k + 1 + t];
      hs[ty][4 * g + k] = (unsigned short)acc;
    }
  }
  __syncthreads();
  {
    const int lx = (tid & 15) * 4, ly0 = (tid >> 4) * 2;   // 4 columns x 2 rows per thread
    const int gx = X + lx;
    if (gx >= W) return;
#pragma unroll
    for (int ry = 0; ry < 2; ++ry) {
      const int gy = Y + ly0 + ry;
      if (gy >= H) break;
      uint8_t o[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        int acc = 0;
#pragma unroll
        for (int t = 0; t < 7; ++t) acc += k7[t] * hs[ly0 + ry + t][lx + k];
        o[k] = (uint8_t)((acc + 32768) >> 16);
      }
      *reinterpret_cast<uchar4*>(blur + (size_t)s * W * H + (size_t)gy * W + gx) = make_uchar4(o[0], o[1], o[2], o[3]);
    }
  }
}

// ---------------------------------------------------------------- pyrDown (5x5 binomial, (x+128)>>8)
// source level must already have a valid REFLECT_101 pad (>= 2 px). App. A.2.
// each thread produces 4 adjacent destination pixels from 5 source rows x 16 bytes (four aligned 32-bit loads per row)
__global__ void __launch_bounds__(256) pyrdown_kernel(uint8_t* __restrict__ pyr, LvbPyramidLayout L, int src_level) {
  const int s = blockIdx.z;
  const LvbLevel ls = L.lv[src_level], ld = L.lv[src_level + 1];
  const int x4 = (blockIdx.x * 32 + threadIdx.x) * 4;              // first of 4 destination columns (block = 32 x 8)
  const int y = blockIdx.y * 8 + threadIdx.y;
  if (x4 >= ld.w || y >= ld.h) return;
  const uint8_t* so = lvb_level_origin((const uint8_t*)pyr, L, s, src_level);
  uint8_t* dorg = lvb_level_origin(pyr, L, s, src_level + 1);
  int acc[4] = {0, 0, 0, 0};
  const int wv[5] = {1, 4, 6, 4, 1};
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    // bytes [2*x4 - 4, 2*x4 + 12) of source row 2y-2+j; the level origin is 8-byte aligned and 2*x4 is a multiple of 8
    const uint32_t* row = reinterpret_cast<const uint32_t*>(so + (ptrdiff_t)(2 * y - 2 + j) * ls.pitch + (2 * x4 - 4));
    const uint32_t w0 = row[0], w1 = row[1], w2 = row[2], w3 = row[3];
    uint8_t b[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) { b[q] = (w0 >> (8 * q)) & 255; b[4 + q] = (w1 >> (8 * q)) & 255; b[8 + q] = (w2 >> (8 * q)) & 255; b[12 + q] = (w3 >> (8 * q)) & 255; }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int c = 4 + 2 * k;      // byte index of source column 2*(x4+k)
      acc[k] += wv[j] * (b[c - 2] + 4 * b[c - 1] + 6 * b[c] + 4 * b[c + 1] + b[c + 2]);
    }
  }
  uint8_t o[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) o[k] = (uint8_t)((acc[k] + 128) >> 8);
  uint8_t* dst = dorg + (ptrdiff_t)y * ld.pitch + x4;
  if (x4 + 3 < ld.w) *reinterpret_cast<uchar4*>(dst) = make_uchar4(o[0], o[1], o[2], o[3]);
  else for (int k = 0; k < 4 && x4 + k < ld.w; ++k) dst[k] = o[k];
  if (x4 <= LVB_PAD || x4 + 3 >= ld.w - 1 - LVB_PAD || y <= LVB_PAD || y >= ld.h - 1 - LVB_PAD) {   // the destination level's pad
    for (int k = 0; k < 4 && x4 + k < ld.w; ++k) store_pad_copies(dorg, ld.pitch, ld.w, ld.h, x4 + k, y, o[k]);
  }
}

}  // namespace

// Build CLAHE'd L0 + pyramid + blur for n images already in device memory.
int fe_build_pyramid(LvbHandle* h, const uint8_t* d_images, int n, uint8_t* pyr, uint8_t* blur) {
  LvbFrontEnd& fe = h->fe;
  const int W = fe.W, H = fe.H;
  cudaStream_t st = h->stream;
  if (h->cfg.flag_equalize) {
    const int tile_total = (W / kTiles) * (H / kTiles);
    int clip = (int)(3.0 * tile_total / 256);   // CLAHE clipLimit 3.0, histSize 256
    if (clip < 1) clip = 1;
    LVB_PROF(h, "clahe_lut_kernel");
    const uintptr_t al = (uintptr_t)d_images | (uintptr_t)W;
    if (al % 16 == 0) clahe_lut_kernel<16><<<dim3(64, n), 256, 0, st>>>(d_images, W, H, fe.lut, clip);
    else if (al % 8 == 0) clahe_lut_kernel<8><<<dim3(64, n), 256, 0, st>>>(d_images, W, H, fe.lut, clip);
    else clahe_lut_kernel<4><<<dim3(64, n), 256, 0, st>>>(d_images, W, H, fe.lut, clip);
    LVB_LAUNCH_CHECK(h);
  }
  {
    dim3 grd((W + FT_W - 1) / FT_W, (H + FT_H - 1) / FT_H, n);
    LVB_PROF(h, "clahe_pyr_blur_kernel");
    clahe_pyr_blur_kernel<<<grd, 256, 0, st>>>(d_images, W, H, fe.lut, pyr, fe.L, blur, h->cfg.flag_equalize);
    LVB_LAUNCH_CHECK(h);
  }
  for (int l = 1; l + 1 < fe.L.n_levels; ++l) {  // L2 and up: every producer writes the REFLECT_101 pad of the level it produces
    const LvbLevel& ld = fe.L.lv[l + 1];
    dim3 g2(((ld.w + 3) / 4 + 31) / 32, (ld.h + 7) / 8, n);
    LVB_PROF(h, "pyrdown_kernel");
    pyrdown_kernel<<<g2, dim3(32, 8), 0, st>>>(pyr, fe.L, l);
    LVB_LAUNCH_CHECK(h);
  }
  return LVB_OK;
}
