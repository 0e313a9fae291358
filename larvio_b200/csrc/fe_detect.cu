// Shi-Tomasi corner detection == cv::goodFeaturesToTrack(img, want, 0.01, min_distance, mask)
// (call sites image_processor.cpp:343 and :1035-1036, mask construction :1009-1030).
// Arithmetic restated from OpenCV 4.13 (SURVEY.md App. A.6) and pinned against cv2 in the tests:
//   Dx,Dy = Sobel3 scaled by 1/(4*3*255) (float, REFLECT_101), cov = 3x3 box of (Dx^2,DxDy,Dy^2)
//   summed in double, eig = (a/2+c/2) - sqrt((a/2-c/2)^2 + b^2); thr = (float)(0.01*max(eig|mask));
//   keep interior pixels > thr that equal their 3x3 max; order by value desc, ties by higher
//   address; greedy min-distance selection until `want` corners.
// The FMA placement below mirrors what OpenCV's AVX2/AVX-512 build does (v_muladd in the column
// filter, contracted row filter except in the last W%32 columns) so the response map is bit-equal
// to cv2's on such hosts; see DESIGN.md "Detector arithmetic".
#include <float.h>
#include "lvb_internal.h"

namespace {

constexpr int TW = 64, TH = 16;           // output tile
constexpr int RW = TW + 2, RH = TH + 2;   // response grid (non-maximum apron 1)
constexpr int PW = TW + 4, PH = TH + 4;   // product grid (box apron 1 more)
constexpr int LW = TW + 8, LH = TH + 6;   // image tile (Sobel apron 1 more), whole 32-bit words from bx - 4
constexpr int STRIP = 6;                  // response rows per thread in the column-sum stage (RH / STRIP strips per column)
static_assert(RH % STRIP == 0 && RW * (RH / STRIP) <= 256, "one column strip per thread");

__device__ __forceinline__ int float_order_key(float v) {
  int b = __float_as_int(v);
  return b >= 0 ? b : (b ^ 0x7fffffff);
}

struct CornerArgs {
  const uint8_t* pyr; LvbPyramidLayout L;
  const uint8_t* mask;     // [S][H][W] or null
  float* eig;              // [S][H][W] or null: the response map is only written for the stage-level test entry point
  int* eig_max_key;        // [S] ordered-int key of the masked maximum
  unsigned long long* cand; int* n_cand; int cap;
  int* hist;               // [S][LVB_CAND_BINS] candidates per value-bits bin
  const int* enable;       // [S] or null
};

// cornerMinEigenVal + the masked maximum + the 3x3 non-maximum test in ONE pass over the level (SURVEY F5: the image is read
// once; the f32 response map of the two-kernel version - 1.4 MB per sequence written and re-read - no longer exists).
// A tile computes the response on its 64x16 outputs plus a one-pixel apron (neighbours of the non-maximum test), from the
// covariance products on a 68x20 grid and the image on 70x22 (staged as 72x22 in aligned words).  The products are widened
// to double once, where they are made; the 3x3 box is separable - row sums, then column sums, in double like OpenCV's
// RowSum<float,double> / ColumnSum<double,float> - and a thread walks a 6-row strip of one response column, so each row sum
// of the strip is made once, in registers.
// The global threshold 0.01 * max is not known yet, so a tile keeps every local maximum above 0.01 * (its own masked
// maximum) - a lower bound of the final threshold - and select_kernel applies the exact one.  Every candidate is also counted
// in its sequence's value histogram (LVB_CAND_BINS bins of the float bits), from which select_kernel cuts its chunks.
__global__ void __launch_bounds__(256) corner_kernel(CornerArgs a) {
  __shared__ uint32_t imgw[LH][LW / 4];                   // image tile: byte (tx, ty) <-> pixel (bx - 4 + tx, by - 3 + ty)
  __shared__ double pxx[PH][PW], pxy[PH][PW], pyy[PH][PW];  // products: cell (cx, cy) <-> pixel (bx - 2 + cx, by - 2 + cy)
  __shared__ float se[RH][RW];                            // response: cell (ex, ey) <-> pixel (bx - 1 + ex, by - 1 + ey)
  __shared__ int blk_max;
  const int s = blockIdx.z;
  if (a.enable && !a.enable[s]) return;
  const LvbLevel lv = a.L.lv[0];
  const int W = lv.w, H = lv.h;
  const int bx = blockIdx.x * TW, by = blockIdx.y * TH;
  const uint8_t* org = lvb_level_origin(a.pyr, a.L, s, 0);
  const int tid = threadIdx.x;
  if (tid == 0) blk_max = INT_MIN;
  // the level origin is 8-byte aligned and bx - 4 a multiple of 4; clamped words (only read for cells that are never used)
  // stay inside the padded rows
  for (int i = tid; i < LH * (LW / 4); i += 256) {
    const int ty = i / (LW / 4), wq = i - ty * (LW / 4);
    const int gy = min(by - 3 + ty, H + LVB_PAD - 1);
    const int gx = min(bx - 4 + 4 * wq, lv.pitch - LVB_PAD - 4);
    imgw[ty][wq] = *reinterpret_cast<const uint32_t*>(org + (ptrdiff_t)gy * lv.pitch + gx);
  }
  __syncthreads();
  const uint8_t* img = reinterpret_cast<const uint8_t*>(&imgw[0][0]);
  const double scale = 1.0 / (4.0 * 3.0 * 255.0);
  const float k0 = (float)(2.0 * scale), k1 = (float)scale;
  const int tail_x = W & ~31;
  for (int i = tid; i < PH * PW; i += 256) {
    const int cy = i / PW, cx = i - cy * PW;
    if (bx - 2 + cx > W || by - 2 + cy > H) { pxx[cy][cx] = 0.0; pxy[cy][cx] = 0.0; pyy[cy][cx] = 0.0; continue; }
    const int gx = lvb_reflect101(bx - 2 + cx, W), gy = lvb_reflect101(by - 2 + cy, H);   // the box filter's REFLECT_101 is on the products
    const uint8_t* m = img + (gy - (by - 3)) * LW + (gx - (bx - 4));              // the pixel inside the tile
    // Dx: row diff then symmetric column filter with FMA
    const float d0 = (float)((int)m[-LW + 1] - (int)m[-LW - 1]);
    const float d1 = (float)((int)m[1] - (int)m[-1]);
    const float d2 = (float)((int)m[LW + 1] - (int)m[LW - 1]);
    const float Dx = __fmaf_rn(__fadd_rn(d0, d2), k1, __fmul_rn(d1, k0));
    // Dy: smoothing row filter (FMA chain; plain mul/add in the last W%32 columns), then row diff
    float r0, r2;
    {
      const float a0 = (float)m[-LW - 1], a1 = (float)m[-LW], a2 = (float)m[-LW + 1];
      const float b0 = (float)m[LW - 1], b1 = (float)m[LW], b2 = (float)m[LW + 1];
      if (gx < tail_x) {
        r0 = __fmaf_rn(a2, k1, __fmaf_rn(a1, k0, __fmul_rn(a0, k1)));
        r2 = __fmaf_rn(b2, k1, __fmaf_rn(b1, k0, __fmul_rn(b0, k1)));
      } else {
        r0 = __fadd_rn(__fadd_rn(__fmul_rn(a0, k1), __fmul_rn(a1, k0)), __fmul_rn(a2, k1));
        r2 = __fadd_rn(__fadd_rn(__fmul_rn(b0, k1), __fmul_rn(b1, k0)), __fmul_rn(b2, k1));
      }
    }
    const float Dy = __fsub_rn(r2, r0);
    pxx[cy][cx] = (double)__fmul_rn(Dx, Dx);
    pxy[cy][cx] = (double)__fmul_rn(Dx, Dy);
    pyy[cy][cx] = (double)__fmul_rn(Dy, Dy);
  }
  __syncthreads();
  // row sums h[cy][ex] = (p[cy][ex] + p[cy][ex + 1]) + p[cy][ex + 2], column sums (h[ey] + h[ey + 1]) + h[ey + 2], min eigenvalue
  if (tid < RW * (RH / STRIP)) {
    const int ex = tid % RW, ey0 = (tid / RW) * STRIP;
    double hx[3], hy[3], hz[3];
#pragma unroll
    for (int r = 0; r < STRIP + 2; ++r) {
      const int cy = ey0 + r;
      hx[r % 3] = (pxx[cy][ex] + pxx[cy][ex + 1]) + pxx[cy][ex + 2];
      hy[r % 3] = (pxy[cy][ex] + pxy[cy][ex + 1]) + pxy[cy][ex + 2];
      hz[r % 3] = (pyy[cy][ex] + pyy[cy][ex + 1]) + pyy[cy][ex + 2];
      if (r >= 2) {
        const double xx = (hx[(r - 2) % 3] + hx[(r - 1) % 3]) + hx[r % 3];
        const double xy = (hy[(r - 2) % 3] + hy[(r - 1) % 3]) + hy[r % 3];
        const double yy = (hz[(r - 2) % 3] + hz[(r - 1) % 3]) + hz[r % 3];
        const float fa = __fmul_rn((float)xx, 0.5f), fb = (float)xy, fc = __fmul_rn((float)yy, 0.5f);
        const float dif = __fsub_rn(fa, fc);
        se[ey0 + r - 2][ex] = __fsub_rn(__fadd_rn(fa, fc), __fsqrt_rn(__fadd_rn(__fmul_rn(dif, dif), __fmul_rn(fb, fb))));
      }
    }
  }
  __syncthreads();
  // masked maximum of this tile
  constexpr int PER = TW * TH / 256;
  float myv[PER]; bool mym[PER]; int my_key = INT_MIN;
#pragma unroll
  for (int r = 0; r < PER; ++r) {
    const int i = tid + 256 * r;
    const int oy = i / TW, ox = i - oy * TW;
    const int gx = bx + ox, gy = by + oy;
    myv[r] = 0.f; mym[r] = false;
    if (gx < W && gy < H) {
      const size_t gi = (size_t)s * W * H + (size_t)gy * W + gx;
      const float e = se[oy + 1][ox + 1];
      myv[r] = e;
      if (a.eig) a.eig[gi] = e;
      mym[r] = !a.mask || a.mask[gi];
      if (mym[r]) my_key = max(my_key, float_order_key(e));
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) my_key = max(my_key, __shfl_xor_sync(0xffffffffu, my_key, o));
  if ((tid & 31) == 0) atomicMax(&blk_max, my_key);
  __syncthreads();
  const int key = blk_max;
  if (key == INT_MIN) return;                             // nothing unmasked in this tile: no maximum, no candidate
  if (tid == 0) atomicMax(&a.eig_max_key[s], key);
  const float tile_max = __int_as_float(key >= 0 ? key : (key ^ 0x7fffffff));
  const float thr_lo = (float)((double)tile_max * 0.01);  // <= the final threshold (float)(0.01 * global max): same monotone rounding
#pragma unroll
  for (int r = 0; r < PER; ++r) {
    const int i = tid + 256 * r;
    const int oy = i / TW, ox = i - oy * TW;
    const int gx = bx + ox, gy = by + oy;
    bool is = false;
    const float v = myv[r];
    if (mym[r] && gx >= 1 && gx < W - 1 && gy >= 1 && gy < H - 1 && v > thr_lo && v > 0.f) {
      const int ey = oy + 1, ex = ox + 1;
      is = v >= se[ey][ex - 1] && v >= se[ey][ex + 1] && v >= se[ey - 1][ex - 1] && v >= se[ey - 1][ex] && v >= se[ey - 1][ex + 1] &&
           v >= se[ey + 1][ex - 1] && v >= se[ey + 1][ex] && v >= se[ey + 1][ex + 1];
    }
    // warp-aggregated append
    const unsigned m = __ballot_sync(0xffffffffu, is);
    if (m) {
      const int lane = tid & 31;
      int base = 0;
      if (lane == __ffs(m) - 1) base = atomicAdd(&a.n_cand[s], __popc(m));
      base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
      if (is) {
        const int pos = base + __popc(m & ((1u << lane) - 1));
        const unsigned bits = (unsigned)__float_as_int(v);
        if (pos < a.cap) a.cand[(size_t)s * a.cap + pos] = ((unsigned long long)bits << 32) | (unsigned)(gy * W + gx);
        atomicAdd(&a.hist[(size_t)s * LVB_CAND_BINS + (bits >> 19)], 1);
      }
    }
  }
}

// ---------------------------------------------------------------- per-sequence select: top-K chunks, sort, greedy
// Candidates are taken in chunks of consecutive descending keys; the greedy pass continues across chunks, so where a chunk
// ends does not change the result.  A chunk is cut at a histogram bin boundary: the bins below the previous cut are scanned
// from the top until they hold about CHUNK_TARGET candidates (never more than CHUNK).  Only a single bin that alone holds
// more than CHUNK is refined, by bisection over the value bits of that bin.
constexpr int CHUNK = 4096;
constexpr int CHUNK_TARGET = 1024;
constexpr int BIN_SHIFT = 19;                 // value bits >> BIN_SHIFT: LVB_CAND_BINS bins over the positive floats
static_assert((0x7fffffffu >> BIN_SHIFT) + 1 == LVB_CAND_BINS, "bins cover bits 30..BIN_SHIFT");
struct SelArgs {
  const unsigned long long* cand; const int* n_cand; int cap;
  const int* hist;          // [S][LVB_CAND_BINS]
  const int* want; int W; int min_dist; int stride;
  float2* out; int* out_n; int* overflow;
  const int* enable;
  const int* eig_max_key;   // [S]: candidates are a superset (tile-local thresholds); the exact test v > (float)(0.01 * max) happens here
};

__global__ void __launch_bounds__(1024) select_kernel(SelArgs a) {
  __shared__ unsigned long long keys[CHUNK];
  __shared__ int s_cnt, s_acc, s_done, s_rover, s_rtgt, s_pover;
  __shared__ unsigned s_upper;                  // value bits: the keys still to be taken are those below s_upper << 32
  __shared__ short2 accepted[512];
  __shared__ int red[32];
  const int s = blockIdx.x;
  const int tid = threadIdx.x;
  if (a.enable && !a.enable[s]) return;
  int n = a.n_cand[s];
  const int want = min(a.want[s], min(a.stride, 512));
  if (n > a.cap) { if (tid == 0) atomicExch(a.overflow, 1); n = a.cap; }
  const unsigned long long* c = a.cand + (size_t)s * a.cap;
  const int* hist = a.hist + (size_t)s * LVB_CAND_BINS;
  if (tid == 0) { s_acc = 0; s_done = 0; s_upper = 0x80000000u; s_rover = INT_MAX; s_rtgt = INT_MAX; }
  __syncthreads();
  if (want <= 0 || n <= 0) { if (tid == 0) a.out_n[s] = 0; return; }
  const int md2 = a.min_dist * a.min_dist;
  // v > thr for positive floats <=> value bits > thr bits <=> value bits >= lowb
  unsigned lowb = 0u;
  {
    const int key = a.eig_max_key[s];
    if (key == INT_MIN) { if (tid == 0) a.out_n[s] = 0; return; }
    const float maxv = __int_as_float(key >= 0 ? key : (key ^ 0x7fffffff));
    const float thr = (float)((double)maxv * 0.01);
    if (!(thr >= 0.f)) { if (tid == 0) a.out_n[s] = 0; return; }       // no positive response anywhere: no corner
    lowb = (unsigned)__float_as_int(thr) + 1u;
  }
  // exact count of the keys with value bits in [lo, upper), block-wide
  auto count_from = [&](unsigned lo, unsigned upper) -> int {
    const unsigned long long lok = (unsigned long long)lo << 32, upk = (unsigned long long)upper << 32;
    int cnt = 0;
    for (int i = tid; i < n; i += 1024) { const unsigned long long k = c[i]; cnt += (k >= lok && k < upk); }
#pragma unroll
    for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((tid & 31) == 0) red[tid >> 5] = cnt;
    __syncthreads();
    if (tid < 32) {
      int v = red[tid];
#pragma unroll
      for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (tid == 0) s_cnt = v;
    }
    __syncthreads();
    const int total = s_cnt;
    __syncthreads();
    return total;
  };
  const int bL = (int)(lowb >> BIN_SHIFT);
  while (true) {
    const unsigned upper = s_upper;
    // --- histogram scan: bins bU (holding upper - 1) down to bL, ranked from the top; thread t owns ranks 4t .. 4t+3.
    // A bin's count includes keys outside [lowb, upper) only in the two end bins, so every prefix is an upper bound.
    const int bU = (int)((upper - 1u) >> BIN_SHIFT), nr = bU - bL + 1;
    int hv[4], run = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) { const int r = 4 * tid + q; hv[q] = r < nr ? hist[bU - r] : 0; run += hv[q]; }
    int x = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if ((tid & 31) >= o) x += y; }
    if ((tid & 31) == 31) red[tid >> 5] = x;
    __syncthreads();
    int pre = x - run;
    for (int w = 0; w < (tid >> 5); ++w) pre += red[w];
    // the first rank whose prefix exceeds CHUNK (and the prefix above it), the first rank whose prefix reaches CHUNK_TARGET
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int r = 4 * tid + q, above = pre;
      pre += hv[q];
      if (r < nr && pre > CHUNK && above <= CHUNK) { s_rover = r; s_pover = above; }
      if (r < nr && pre >= CHUNK_TARGET && above < CHUNK_TARGET) s_rtgt = r;
    }
    __syncthreads();
    const int r_over = min(s_rover, nr), r_tgt = min(s_rtgt, nr - 1), p_over = s_pover;
    const int r_cut = min(r_over - 1, r_tgt);     // the chunk is ranks 0 .. r_cut
    unsigned cut;
    if (r_over < nr && r_cut == r_over - 1 && p_over == 0) {
      // rank r_over alone holds more than CHUNK, nothing above it: bisect inside that bin for the smallest cut that fits
      const unsigned b = (unsigned)(bU - r_over);
      unsigned lo = max(b << BIN_SHIFT, lowb), hi = min(upper, (b + 1u) << BIN_SHIFT);   // count(>= hi) == 0
      if (count_from(lo, upper) <= CHUNK) hi = lo;
      while (hi - lo > 1u) {
        const unsigned mid = lo + ((hi - lo) >> 1);
        if (count_from(mid, upper) <= CHUNK) hi = mid; else lo = mid;
      }
      cut = hi;
    } else {
      cut = max((unsigned)(bU - r_cut) << BIN_SHIFT, lowb);
    }
    if (cut >= upper) {                           // more than CHUNK candidates share one value: cannot be ordered in a chunk
      if (tid == 0) { atomicExch(a.overflow, 1); s_done = 1; }
      __syncthreads();
      break;
    }
    // --- gather chunk
    const unsigned long long cutk = (unsigned long long)cut << 32, upk = (unsigned long long)upper << 32;
    if (tid == 0) s_cnt = 0;
    for (int i = tid; i < CHUNK; i += 1024) keys[i] = 0ull;
    __syncthreads();
    for (int i = tid; i < n; i += 1024) {
      const unsigned long long k = c[i];
      if (k >= cutk && k < upk) { const int p = atomicAdd(&s_cnt, 1); if (p < CHUNK) keys[p] = k; }
    }
    __syncthreads();
    const int m = min(s_cnt, CHUNK);
    // --- bitonic sort, descending, of the smallest power of two >= m (the keys after m are 0)
    int P = 2;
    while (P < m) P <<= 1;
    for (int k2 = 2; k2 <= P; k2 <<= 1) {
      for (int j = k2 >> 1; j > 0; j >>= 1) {
        for (int i = tid; i < P; i += 1024) {
          const int ixj = i ^ j;
          if (ixj > i) {
            const unsigned long long A = keys[i], B = keys[ixj];
            const bool desc = ((i & k2) == 0);
            if (desc ? (A < B) : (A > B)) { keys[i] = B; keys[ixj] = A; }
          }
        }
        __syncthreads();
      }
    }
    // --- greedy min-distance selection by warp 0, 32 candidates at a time
    if (tid < 32) {
      int acc = s_acc;
      for (int b0 = 0; b0 < m && acc < want; b0 += 32) {
        const int idx = b0 + tid;
        const bool valid = idx < m;
        const unsigned pix = valid ? (unsigned)(keys[idx] & 0xffffffffu) : 0u;
        const int py = (int)(pix / (unsigned)a.W), px = (int)(pix - (unsigned)py * a.W);
        bool alive = valid;
        for (int q = 0; q < acc && alive; ++q) {
          const short2 t = accepted[q];
          const int dx = px - t.x, dy = py - t.y;
          if (dx * dx + dy * dy < md2) alive = false;
        }
        // resolve conflicts inside the batch in rank order
        for (int l = 0; l < 32; ++l) {
          const int al = __shfl_sync(0xffffffffu, (int)alive, l);
          if (!al) continue;
          if (acc >= want) { if (tid >= l) alive = false; break; }
          const int qx = __shfl_sync(0xffffffffu, px, l), qy = __shfl_sync(0xffffffffu, py, l);
          if (tid == l) { accepted[acc] = make_short2((short)px, (short)py); }
          acc++;
          if (tid > l && alive) {
            const int dx = px - qx, dy = py - qy;
            if (dx * dx + dy * dy < md2) alive = false;
          }
        }
        __syncwarp();
      }
      if (tid == 0) {
        s_acc = acc;
        s_done = (acc >= want) || cut <= lowb;    // a chunk may be empty (the end bins over-count): only the threshold ends
        s_upper = cut;
        s_rover = INT_MAX; s_rtgt = INT_MAX;
      }
    }
    __syncthreads();
    if (s_done) break;
  }
  const int acc = s_acc;
  for (int i = tid; i < acc; i += 1024)
    a.out[(size_t)s * a.stride + i] = make_float2((float)accepted[i].x, (float)accepted[i].y);
  if (tid == 0) a.out_n[s] = acc;
}

// ---------------------------------------------------------------- detection mask (image_processor.cpp:1009-1030)
__global__ void mask_kernel(uint8_t* mask, int W, int H, const float2* pts, const int* n_pts, int stride,
                            int min_dist, const int* enable) {
  const int s = blockIdx.y, i = blockIdx.x;
  if (enable && !enable[s]) return;
  if (i >= n_pts[s]) return;
  const float2 p = pts[(size_t)s * stride + i];
  const int ry = (int)roundf(p.y), rx = (int)roundf(p.x);     // C round(): half away from zero
  const int r0 = max(ry - min_dist, 0), r1 = min(ry + min_dist, H - 1);
  const int c0 = max(rx - min_dist, 0), c1 = min(rx + min_dist, W - 1);
  const int w = c1 - c0 + 1, hgt = r1 - r0 + 1;
  if (w <= 0 || hgt <= 0) return;
  uint8_t* m = mask + (size_t)s * W * H;
  for (int t = threadIdx.x; t < w * hgt; t += blockDim.x) {
    const int yy = t / w, xx = t - yy * w;
    m[(size_t)(r0 + yy) * W + c0 + xx] = 0;
  }
}

__global__ void fill_kernel(uint8_t* p, size_t per_seq, const int* enable, uint8_t v) {
  const int s = blockIdx.y;
  if (enable && !enable[s]) return;
  uint4 vv; const unsigned w = v * 0x01010101u; vv.x = vv.y = vv.z = vv.w = w;
  uint4* q = reinterpret_cast<uint4*>(p + (size_t)s * per_seq);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < per_seq / 16; i += (size_t)gridDim.x * blockDim.x) q[i] = vv;
}

// grid (LVB_CAND_BINS / 256, n)
__global__ void reset_detect_kernel(int* eig_max_key, int* n_cand, int* hist) {
  const int s = blockIdx.y;
  hist[(size_t)s * LVB_CAND_BINS + blockIdx.x * 256 + threadIdx.x] = 0;
  if (blockIdx.x == 0 && threadIdx.x == 0) { eig_max_key[s] = INT_MIN; n_cand[s] = 0; }
}

}  // namespace

// Detect up to want[s] corners per sequence on level 0 of `pyr`.
//   use_mask != 0: build the mask from (mask_pts, mask_n) first.  enable: per-sequence gate or null.
int fe_detect_launch(LvbHandle* h, const uint8_t* pyr, int n_seq, const int* enable, int use_mask,
                     const uint8_t* ext_mask, const float2* mask_pts, const int* mask_n, const int* want,
                     float2* out, int* out_n, float* eig_out) {
  LvbFrontEnd& fe = h->fe;
  cudaStream_t st = h->stream;
  const int W = fe.W, H = fe.H;
  const uint8_t* mask = nullptr;
  LVB_PROF(h, "reset_detect_kernel");
  reset_detect_kernel<<<dim3(LVB_CAND_BINS / 256, n_seq), 256, 0, st>>>(fe.eig_max, fe.n_cand, fe.cand_hist);
  LVB_LAUNCH_CHECK(h);
  if (ext_mask) mask = ext_mask;
  else if (use_mask) {
    LVB_PROF(h, "fill_kernel");
    fill_kernel<<<dim3(64, n_seq), 256, 0, st>>>(fe.mask, (size_t)W * H, enable, 255);
    LVB_LAUNCH_CHECK(h);
    LVB_PROF(h, "mask_kernel");
    mask_kernel<<<dim3(fe.N, n_seq), 128, 0, st>>>(fe.mask, W, H, mask_pts, mask_n, fe.N, h->cfg.min_distance, enable);
    LVB_LAUNCH_CHECK(h);
    mask = fe.mask;
  }
  CornerArgs ca; ca.pyr = pyr; ca.L = fe.L; ca.mask = mask; ca.eig = eig_out; ca.eig_max_key = fe.eig_max; ca.cand = fe.cand; ca.n_cand = fe.n_cand;
  ca.cap = fe.cand_cap; ca.hist = fe.cand_hist; ca.enable = enable;
  LVB_PROF(h, "corner_kernel");
  corner_kernel<<<dim3((W + TW - 1) / TW, (H + TH - 1) / TH, n_seq), 256, 0, st>>>(ca);
  LVB_LAUNCH_CHECK(h);
  SelArgs sa; sa.cand = fe.cand; sa.n_cand = fe.n_cand; sa.cap = fe.cand_cap; sa.hist = fe.cand_hist; sa.want = want; sa.W = W;
  sa.min_dist = h->cfg.min_distance; sa.stride = fe.N; sa.out = out; sa.out_n = out_n; sa.overflow = fe.overflow; sa.enable = enable; sa.eig_max_key = fe.eig_max;
  LVB_PROF(h, "select_kernel");
  select_kernel<<<n_seq, 1024, 0, st>>>(sa);
  LVB_LAUNCH_CHECK(h);
  return LVB_OK;
}
