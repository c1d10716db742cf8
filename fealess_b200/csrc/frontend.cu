// LINE-MOD modality extraction on sm_100a: colour-gradient quantisation, depth-normal quantisation, pyramids, and the
// fused spread -> response-map -> linear-memory kernel.  Integer/byte work, HBM-bound at best and launch-bound at VGA:
// every stage is one tiled kernel with a shared-memory halo so each input byte is read from HBM once.
//
// Reference semantics (paths relative to /root/reference, see SURVEY.md appendix A):
//   colour : quantizedOrientations + hysteresisGradient      linemod/linemod.cpp:230-385
//   pyramid: ColorGradientPyramid::pyrDown (cv::pyrDown)      linemod.cpp:434-453
//   depth  : quantizedNormals (+ medianBlur 5)                linemod.cpp:567-685, table linemod/normal_lut.i
//   depth pyramid / masks: resize(INTER_NEAREST), copyTo(mask) linemod.cpp:448, 455-459, 721-745
//   spread / computeResponseMaps / linearize                  linemod.cpp:950-965, 979-1048, 1060-1088
// Compiled with -fmad=false: the fp32 expressions below must round exactly like the (uncontracted) reference.
#include "fl_internal.cuh"
#include "fl_owned.cuh"
#include <math.h>
#include <new>

// ------------------------------------------------------------------------------------------------
// tables: NORMAL_LUT depends only on (v2, v1) -> 400 bytes; response table packs the 8 per-label responses of one
// spread byte into a uint2 (labels 0-3 in .x, 4-7 in .y), i.e. SIMILARITY_LUT (linemod.cpp:970) re-indexed by pixel value.
// ------------------------------------------------------------------------------------------------
// g_*: in global memory, copied to shared memory by every CTA that indexes them per thread (one coalesced load per thread); the
// constant cache would serialise a warp's 32 distinct addresses
__device__ __align__(4) uint8_t g_normal_plane[400];
__constant__ uint2 c_resp8[256];
__device__ uint2 g_resp8[256];

int fl_launch_tables_init() {
  uint8_t plane[400];
  for (int v2 = 0; v2 < 20; ++v2)
    for (int v1 = 0; v1 < 20; ++v1) {
      // one-hot 45-degree sector of atan2(v2-10, v1-10) + 22.5 deg: closed form of normal_lut.i:4 (sha256-pinned in tests)
      double a = atan2((double)(v2 - 10), (double)(v1 - 10)) * (180.0 / 3.14159265358979323846) + 22.5;
      a = fmod(a + 360.0, 360.0);
      plane[v2 * 20 + v1] = (uint8_t)(1u << (((int)floor(a / 45.0)) & 7));
    }
  uint2 resp[256];
  for (int v = 0; v < 256; ++v) {
    uint32_t w[2] = {0, 0};
    for (int i = 0; i < 8; ++i) {
      int best = 0;
      for (int j = 0; j < 8; ++j)
        if (v >> j & 1) {
          int d = i > j ? i - j : j - i;
          if (8 - d < d) d = 8 - d;
          int g = d == 0 ? 4 : (d == 1 ? 2 : (d == 2 ? 1 : 0));   // response per circular label distance
          if (g > best) best = g;
        }
      w[i >> 2] |= (uint32_t)best << (8 * (i & 3));
    }
    resp[v] = make_uint2(w[0], w[1]);
  }
  FL_CUDA(cudaMemcpyToSymbol(g_normal_plane, plane, sizeof plane));
  FL_CUDA(cudaMemcpyToSymbol(c_resp8, resp, sizeof resp));
  FL_CUDA(cudaMemcpyToSymbol(g_resp8, resp, sizeof resp));
  return FL_OK;
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return min(max(v, lo), hi); }

// ------------------------------------------------------------------------------------------------
// K1 colour quantisation: blur7 -> sobel3 -> strongest channel -> 16-bin angle -> &7 -> 3x3 majority vote, one kernel.
// Tile = CQ_TW x CQ_TH output pixels; halo 5 = 3 (blur) + 1 (sobel) + 1 (vote).
// ------------------------------------------------------------------------------------------------
#define CQ_TW 32
#define CQ_TH 16
#define CQ_THREADS 256

// OpenCV fastAtan2 (cv::phase, angleInDegrees) in fp32, then convertTo(CV_8U, 16/360) = rint-half-even, saturate.
__device__ __forceinline__ int angle_q16(float x, float y) {
  const float scale = (float)(180.0 / 3.14159265358979323846);
  const float p1 = 0.9997878412794807f * scale, p3 = -0.3258083974640975f * scale;
  const float p5 = 0.1555786518463281f * scale, p7 = -0.04432655554792128f * scale;
  const float eps = 2.220446049250313e-16f;
  // the two octant branches of fastAtan2 evaluate the same polynomial on min/max: one division instead of a divergent pair
  const float ax = fabsf(x), ay = fabsf(y);
  const float c = __fdiv_rn(fminf(ax, ay), __fadd_rn(fmaxf(ax, ay), eps));
  const float c2 = __fmul_rn(c, c);
  float a = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c);
  if (ax < ay) a = __fsub_rn(90.f, a);
  if (x < 0) a = __fsub_rn(180.f, a);
  if (y < 0) a = __fsub_rn(360.f, a);
  int r = __float2int_rn(__fmul_rn(a, (float)(16.0 / 360.0)));
  return min(max(r, 0), 255);
}

#include "frontend_v2.cuh"

// ------------------------------------------------------------------------------------------------
// K2 cv::pyrDown of the BGR image: 5x5 [1 4 6 4 1]^2, BORDER_REFLECT_101, (sum + 128) >> 8
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect101(int p, int n) {
  if (n == 1) return 0;
  while (p < 0 || p >= n) p = p < 0 ? -p : 2 * n - 2 - p;
  return p;
}

// one thread per output PIXEL (3 channels), CTA = 32 x 8 output pixels (the first version ran one thread per output byte
// and spent ~540 instructions on index arithmetic for each of them)
#define PD_TW 32
#define PD_TH 8
__device__ __forceinline__ int reflect101_near(int p, int n) {         // |overshoot| <= 2 and n >= 3: a single fold
  return p < 0 ? -p : (p >= n ? 2 * n - 2 - p : p);
}
// SRC_STATIC: the source was complete before this launch (the caller's frame), so it may go through L1 (neighbouring threads
// share every line); a level produced by an earlier job of the same launch must be read from L2.  A template argument: chosen
// per load at run time, the two load kinds of the unrolled 5 x 5 taps did not fit 32 registers and spilled.
template <bool SRC_STATIC>
__device__ __forceinline__ void dev_pyrdown_bgr(const uint8_t* __restrict__ src, int W, int H, uint8_t* __restrict__ dst, int bx) {
  const int dw = W / 2, dh = H / 2;
  const int gx = (dw + PD_TW - 1) / PD_TW;
  const int by = bx / gx; bx -= by * gx;
  const int x = bx * PD_TW + (threadIdx.x & 31), y = by * PD_TH + (threadIdx.x >> 5);
  if (x >= dw || y >= dh) return;
  int cx[5], ry[5];
  if (W >= 3 && H >= 3) {
#pragma unroll
    for (int t = 0; t < 5; ++t) { cx[t] = reflect101_near(2 * x + t - 2, W) * 3; ry[t] = reflect101_near(2 * y + t - 2, H); }
  } else {
#pragma unroll
    for (int t = 0; t < 5; ++t) { cx[t] = reflect101(2 * x + t - 2, W) * 3; ry[t] = reflect101(2 * y + t - 2, H); }
  }
  int s0 = 0, s1 = 0, s2 = 0;
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    const uint8_t* row = src + (size_t)ry[j] * W * 3;
    const int kj = j == 0 || j == 4 ? 1 : (j == 2 ? 6 : 4);
    int r0 = 0, r1 = 0, r2 = 0;
#pragma unroll
    for (int t = 0; t < 5; ++t) {
      const int kt = t == 0 || t == 4 ? 1 : (t == 2 ? 6 : 4);
      const uint8_t* p = row + cx[t];
      if (SRC_STATIC) { r0 += kt * __ldg(p); r1 += kt * __ldg(p + 1); r2 += kt * __ldg(p + 2); }
      else { r0 += kt * __ldcg(p); r1 += kt * __ldcg(p + 1); r2 += kt * __ldcg(p + 2); }
    }
    s0 += kj * r0; s1 += kj * r1; s2 += kj * r2;
  }
  uint8_t* o = dst + ((size_t)y * dw + x) * 3;
  o[0] = (uint8_t)((s0 + 128) >> 8); o[1] = (uint8_t)((s1 + 128) >> 8); o[2] = (uint8_t)((s2 + 128) >> 8);
}

static int pyrdown_ctas(int W, int H) { return ((W / 2 + PD_TW - 1) / PD_TW) * ((H / 2 + PD_TH - 1) / PD_TH); }

// ------------------------------------------------------------------------------------------------
// K3 depth normals: 8-tap bilateral least squares -> normal -> NORMAL_LUT, then 5x5 median, fused (halo 2 + 5).
// ------------------------------------------------------------------------------------------------
#define DQ_TW 32
#define DQ_TH 16
#define DQ_THREADS 256


// ------------------------------------------------------------------------------------------------
// K4 nearest-neighbour x1/2 (cv::resize INTER_NEAREST to (W/2, H/2)): depth labels and masks of levels that do not halve exactly
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void dev_resize_nn_half(const uint8_t* __restrict__ src, int W, int H, uint8_t* __restrict__ dst, int bx) {
  const int dw = W / 2, dh = H / 2;
  int i = bx * 256 + threadIdx.x;
  if (i >= dw * dh) return;
  int x = i % dw, y = i / dw;
  int sx = min((int)floor(x * ((double)W / dw)), W - 1);
  int sy = min((int)floor(y * ((double)H / dh)), H - 1);
  dst[i] = src[(size_t)sy * W + sx];
}
__global__ void __launch_bounds__(256) k_resize_nn_half(const uint8_t* __restrict__ src, int W, int H, uint8_t* __restrict__ dst) {
  dev_resize_nn_half(src, W, H, dst, blockIdx.x);
}
void fl_launch_resize_nn_half(const uint8_t* src, int W, int H, uint8_t* dst, cudaStream_t s) {
  int n = (W / 2) * (H / 2);
  k_resize_nn_half<<<(n + 255) / 256, 256, 0, s>>>(src, W, H, dst);
}

// ------------------------------------------------------------------------------------------------
// K5 spread + response maps + linearize, fused.  One CTA = one row of the decimated grid (T image rows) x SL_CW cells.
//   spread(y,x) = OR over the forward TxT window (clipped at the image end)                          :950-965
//   response_i  = table lookup of the spread byte (all 8 labels at once)                              :979-1048
//   LM_i[(y%T)*T + x%T][(y/T)*W' + x/T] = response_i(y,x)                                            :1060-1088
// HBM traffic = W*H read + 8*W*H written; each (label, grid-row) run of SL_CW output bytes is one full 32 B sector.
// ------------------------------------------------------------------------------------------------
#define SL_CW 32
#define SL_THREADS 256

// shared memory: response table (2 KB) + input tile + horizontal-OR tile (rows padded to whole 32-bit words + slack)
__host__ __device__ inline int spread_stride_in(int T) { return (SL_CW * T + T - 1 + 6) & ~3; }
__host__ __device__ inline int spread_stride_pw(int T) { return (SL_CW * T + 3) & ~3; }
__host__ __device__ inline size_t spread_smem_bytes(int T) {
  return 2048 + (size_t)(2 * T - 1) * spread_stride_in(T) + (size_t)(2 * T - 1) * spread_stride_pw(T);   // <= 35 KB at T = 16
}

// OR of the T bytes starting at every byte of a 32-bit word: words w[0..] hold the row from the word's own position on.
// TT > 0: T known at compile time (the loop unrolls to T funnel shifts); TT == 0: runtime T, words read on the fly.
template <int TT>
__device__ __forceinline__ uint32_t or_window(const uint32_t* __restrict__ w, int T) {
  uint32_t o = 0;
  if (TT > 0) {
    uint32_t v[(TT + 2) / 4 + 2];
#pragma unroll
    for (int i = 0; i < (TT + 2) / 4 + 2; ++i) v[i] = w[i];
#pragma unroll
    for (int k = 0; k < TT; ++k) o |= __funnelshift_r(v[k >> 2], v[(k >> 2) + 1], 8 * (k & 3));
  } else {
    for (int k = 0; k < T; ++k) o |= __funnelshift_r(w[k >> 2], w[(k >> 2) + 1], 8 * (k & 3));
  }
  return o;
}

template <int TT, bool COARSE>
// COARSE = false: the caller guarantees lm4 == mass == nullptr (every level but the coarsest), so neither the nibble stores nor the
// response sums are compiled in and the scatter loop fits the registers of __launch_bounds__(256, 8) without spilling.
// mass (nullable, the coarsest level only): += this CTA's sum of every (row, cell) response of label lab into mass[lab], one atomic per label
// per CTA - the per-frame weights by which the staged similarity kernel orders its phases (k_similarity_staged)
// mk (nullable): the frame's mask of this modality (copyTo(dst, mask), linemod.cpp:455-459, 741-745); label (y, x) of this level is kept
// where mk[(y << msh) * mst + (x << msh)] != 0.  msh = level with the level-0 mask when every level halves exactly (the NN pyramid
// then picks src(2y, 2x) at every step), 0 with a mask already resized to this level.
__device__ __forceinline__ void dev_spread_lm(const uint8_t* __restrict__ q, const fl_level_geom& g, uint8_t* __restrict__ lm,
                                              uint8_t* __restrict__ spread_out, uint8_t* __restrict__ lm4, uint32_t* __restrict__ mass,
                                              const uint8_t* __restrict__ mk, int mst, int msh, int bx, int by, uint8_t* smem, int cw) {
  const int T = TT > 0 ? TT : g.T;
  const int W = g.W, H = g.H, Wd = g.Wd;
  const int gy = by, cx0 = bx * cw;                     // cw <= SL_CW cells per CTA (fewer on small levels: more CTAs in flight)
  const int ncell = min(cw, Wd - cx0);
  const int pw = ncell * T;                             // pixels owned by this CTA per row
  const int tw = pw + T - 1, th = 2 * T - 1;
  const int px0 = cx0 * T, py0 = gy * T;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NWARP = SL_THREADS / 32;
  const int st_in = (tw + 6) & ~3;                      // row stride of the input tile: whole words, >= 3 bytes of zero slack
  const int nw = (pw + 3) >> 2, st_pw = nw << 2;        // words per row of the OR tiles
  uint2* s_resp = reinterpret_cast<uint2*>(smem);        // 256 x 8 B
  uint8_t* s_in = smem + 2048;                          // [th][st_in]   input labels (later reused for the final spread)
  uint8_t* s_hor = s_in + (size_t)(2 * T - 1) * spread_stride_in(T);   // [th][st_pw] horizontal OR
  __shared__ uint32_t s_mass[8];
  for (int i = tid; i < 256; i += SL_THREADS) s_resp[i] = g_resp8[i];
  if (tid < 8) s_mass[tid] = 0;
  if (((reinterpret_cast<uintptr_t>(q) | (uintptr_t)W | (uintptr_t)px0) & 3) == 0) {
    // word-aligned tile: whole 32-bit words, every load of the tile in flight at once (fixed trip count, unrolled).  A word is
    // either entirely inside the image or entirely outside (W % 4 == 0); bytes past the CTA's own window are real pixels of
    // the neighbour and are never read by the OR passes below.
    const int nwi = st_in >> 2;
    const int n_items = th * nwi;
    uint32_t* s_in32 = reinterpret_cast<uint32_t*>(s_in);
    for (int i0 = 0; i0 < n_items; i0 += 4 * SL_THREADS) {
      uint32_t v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {                     // 4 loads in flight per thread (the whole tile for T <= 8)
        const int i = i0 + tid + u * SL_THREADS;
        const int r = i / nwi, wi = i - r * nwi;
        const int y = py0 + r, x = px0 + 4 * wi;
        v[u] = (i < n_items && y < H && x < W) ? __ldcg(reinterpret_cast<const uint32_t*>(q + (size_t)y * W + x)) : 0u;   // clipped window == OR with zeros
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) { const int i = i0 + tid + u * SL_THREADS; if (i < n_items) s_in32[i] = v[u]; }
    }
  } else {
    for (int r = warp; r < th; r += NWARP) {            // rows by warp, bytes by lane: coalesced, no index arithmetic
      const int y = py0 + r;
      const uint8_t* src = q + (size_t)y * W + px0;
      for (int c = lane; c < st_in; c += 32) s_in[r * st_in + c] = (c < tw && px0 + c < W && y < H) ? __ldcg(src + c) : (uint8_t)0;   // clipped window == OR with zeros
    }
  }
  if (mk) {                                             // (uniform over the grid) masked frame: labels under a zero mask byte become 0
    __syncthreads();
    const int nwi = st_in >> 2;
    uint32_t* s_in32 = reinterpret_cast<uint32_t*>(s_in);
    for (int i = tid; i < th * nwi; i += SL_THREADS) {
      const int r = i / nwi, y = py0 + r, x = px0 + 4 * (i - r * nwi);
      if (y >= H || x >= W) continue;                   // outside the image the tile is zero already
      const uint8_t* mrow = mk + (size_t)(y << msh) * mst;
      uint32_t mw = 0;
      if (msh == 0 && x + 3 < W && ((reinterpret_cast<uintptr_t>(mrow) + x) & 3) == 0) mw = __ldg(reinterpret_cast<const uint32_t*>(mrow + x));
      else for (int k = 0; k < 4 && x + k < W; ++k) mw |= (uint32_t)__ldg(mrow + ((x + k) << msh)) << (8 * k);
      s_in32[i] &= __vcmpne4(mw, 0u);                   // SWAR: byte != 0 -> 0xFF
    }
  }
  __syncthreads();
  for (int r = warp; r < th; r += NWARP) {              // horizontal OR, four pixels per thread
    const uint32_t* row = reinterpret_cast<const uint32_t*>(s_in + r * st_in);
    uint32_t* dst = reinterpret_cast<uint32_t*>(s_hor + r * st_pw);
    for (int wi = lane; wi < nw; wi += 32) dst[wi] = or_window<TT>(row + wi, T);
  }
  __syncthreads();
  uint8_t* s_sp = s_in;                                 // [T][st_pw] final spread values (s_in is dead)
  for (int r = warp; r < T; r += NWARP) {               // vertical OR
    uint32_t* dst = reinterpret_cast<uint32_t*>(s_sp + r * st_pw);
    for (int wi = lane; wi < nw; wi += 32) {
      uint32_t v = 0;
      if (TT > 0) {
#pragma unroll
        for (int k = 0; k < TT; ++k) v |= reinterpret_cast<const uint32_t*>(s_hor + (r + k) * st_pw)[wi];
      } else {
        for (int k = 0; k < T; ++k) v |= reinterpret_cast<const uint32_t*>(s_hor + (r + k) * st_pw)[wi];
      }
      dst[wi] = v;
      if (spread_out)
        for (int k = 0; k < 4; ++k) if (4 * wi + k < pw) spread_out[(size_t)(py0 + r) * W + px0 + 4 * wi + k] = (uint8_t)(v >> (8 * k));
    }
  }
  __syncthreads();
  // scatter: item = (residue row ry, residue column rx, group of 4 cells); 8 labels -> 8 word stores per item
  const int ngrp = (ncell + 3) >> 2;
  const int items = T * T * ngrp;
  const size_t cells = (size_t)g.cells;
  const uint32_t inv_ngrp = (65536u + ngrp - 1) / ngrp, inv_T = (65536u + T - 1) / T;   // exact for the small ranges used here
  // response sums of labels {0, 2}, {1, 3}, {4, 6}, {5, 7}, two per word in 16-bit halves (a thread adds at most 16 per item, a warp
  // at most 32 x 16 x ceil(T^2 SL_CW / 4 / SL_THREADS) <= 8,192 per half for T <= 16)
  uint32_t m02 = 0, m13 = 0, m46 = 0, m57 = 0;
  const size_t lab_st = g.label_stride;
  const size_t off0 = (size_t)gy * Wd + cx0;            // this CTA's first cell in every (label, residue) run
  for (int i = tid; i < items; i += SL_THREADS) {
    const int rr = (int)(((uint32_t)i * inv_ngrp) >> 16), c4 = i - rr * ngrp;
    const int ry = (int)(((uint32_t)rr * inv_T) >> 16), rx = rr - ry * T;
    const int nvalid = min(4, ncell - c4 * 4);
    const uint8_t* sp = s_sp + ry * st_pw + c4 * 4 * T + rx;
    const uint2 r0 = s_resp[sp[0]];                     // c4 * 4 < ncell always
    const uint2 r1 = nvalid > 1 ? s_resp[sp[T]] : make_uint2(0, 0);
    const uint2 r2 = nvalid > 2 ? s_resp[sp[2 * T]] : make_uint2(0, 0);
    const uint2 r3 = nvalid > 3 ? s_resp[sp[3 * T]] : make_uint2(0, 0);
    if (COARSE) {
      m02 += (r0.x & 0x00FF00FFu) + (r1.x & 0x00FF00FFu) + (r2.x & 0x00FF00FFu) + (r3.x & 0x00FF00FFu);
      m13 += ((r0.x >> 8) & 0x00FF00FFu) + ((r1.x >> 8) & 0x00FF00FFu) + ((r2.x >> 8) & 0x00FF00FFu) + ((r3.x >> 8) & 0x00FF00FFu);
      m46 += (r0.y & 0x00FF00FFu) + (r1.y & 0x00FF00FFu) + (r2.y & 0x00FF00FFu) + (r3.y & 0x00FF00FFu);
      m57 += ((r0.y >> 8) & 0x00FF00FFu) + ((r1.y >> 8) & 0x00FF00FFu) + ((r2.y >> 8) & 0x00FF00FFu) + ((r3.y >> 8) & 0x00FF00FFu);
    }
    const size_t off = (size_t)rr * cells + off0 + c4 * 4;
    uint8_t* dst = lm + off;
    // one word = byte (lab & 3) of the four cells' response words, for label lab; the stride between labels is label_stride
    const bool wide = nvalid == 4 && ((((uintptr_t)dst) | lab_st) & 3) == 0;
#pragma unroll
    for (int lab = 0; lab < 8; ++lab, dst += lab_st) {
      const uint32_t sel = 0x0040u + (lab & 3) * 0x0011u;          // PRMT selector: {byte b of x, byte b of y}
      const uint32_t w = lab < 4 ? __byte_perm(__byte_perm(r0.x, r1.x, sel), __byte_perm(r2.x, r3.x, sel), 0x5410)
                                 : __byte_perm(__byte_perm(r0.y, r1.y, sel), __byte_perm(r2.y, r3.y, sel), 0x5410);
      if (wide) *reinterpret_cast<uint32_t*>(dst) = w;
      else for (int k = 0; k < nvalid; ++k) dst[k] = (uint8_t)(w >> (8 * k));
      if (COARSE && lm4) {
        // the same four responses (each 0, 1, 2 or 4) as nibbles, cell j of the label in nibble j: what the staged similarity
        // kernel reads (half the bytes).  Only passed for grids of even width, so `off` is even and nvalid is 2 or 4.  `off` is
        // a multiple of 4 only when Wd and cells are: a grid width of 2 mod 4 cells puts every other row at an odd byte.
        const uint32_t p2 = (w | (w >> 4)) & 0x00FF00FFu;
        const uint32_t p4 = (p2 | (p2 >> 8)) & 0xFFFFu;
        uint8_t* d4 = lm4 + (((size_t)lab * lab_st + off) >> 1);
        if (nvalid == 4 && (((uintptr_t)d4) & 1) == 0) *reinterpret_cast<uint16_t*>(d4) = (uint16_t)p4;
        else { d4[0] = (uint8_t)p4; if (nvalid == 4) d4[1] = (uint8_t)(p4 >> 8); }
      }
    }
  }
  if (COARSE && mass) {                                 // (uniform over the CTA)
    m02 = __reduce_add_sync(0xffffffffu, m02); m13 = __reduce_add_sync(0xffffffffu, m13);
    m46 = __reduce_add_sync(0xffffffffu, m46); m57 = __reduce_add_sync(0xffffffffu, m57);
    if (lane == 0 && (m02 | m13 | m46 | m57)) {
      atomicAdd(&s_mass[0], m02 & 0xFFFFu); atomicAdd(&s_mass[2], m02 >> 16); atomicAdd(&s_mass[1], m13 & 0xFFFFu); atomicAdd(&s_mass[3], m13 >> 16);
      atomicAdd(&s_mass[4], m46 & 0xFFFFu); atomicAdd(&s_mass[6], m46 >> 16); atomicAdd(&s_mass[5], m57 & 0xFFFFu); atomicAdd(&s_mass[7], m57 >> 16);
    }
    __syncthreads();
    if (tid < 8 && s_mass[tid]) atomicAdd(mass + tid, s_mass[tid]);
  }
}

// Compile-time T for the pyramid of LINE-MOD's default (T = 5 below the coarsest level, T = 8 at it); every other (T, level) takes the
// runtime-T instantiation.  Each instantiation is ~1.5 k instructions of the one front-end kernel, so fewer of them keep its code small.
__device__ __forceinline__ void dev_spread_lm_any(const fl_fe_job& jb, int bx, int by, uint8_t* smem) {
  if (jb.g.T == 5 && !jb.dst3 && !jb.mass)
    dev_spread_lm<5, false>(jb.src, jb.g, jb.dst, jb.dst2, nullptr, nullptr, jb.mask, jb.mask_stride, jb.mask_shift, bx, by, smem, jb.p0);
  else if (jb.g.T == 8)
    dev_spread_lm<8, true>(jb.src, jb.g, jb.dst, jb.dst2, jb.dst3, jb.mass, jb.mask, jb.mask_stride, jb.mask_shift, bx, by, smem, jb.p0);
  else
    dev_spread_lm<0, true>(jb.src, jb.g, jb.dst, jb.dst2, jb.dst3, jb.mass, jb.mask, jb.mask_stride, jb.mask_shift, bx, by, smem, jb.p0);
}

// ------------------------------------------------------------------------------------------------
// Wave kernel: at VGA every stage above moves a few hundred KB, i.e. ~1 us of HBM time against ~5-8 us of launch +
// dependency latency, so the front end is launch bound.  Jobs are therefore issued together: the grid is the concatenation
// of the jobs' grids (the whole frame, or one wave of it: fe_build, fe_run_single, fe_run_waves below).
// ------------------------------------------------------------------------------------------------
// bounded in-grid wait: true = stop waiting (this CTA timed out, or another one already did); see k_front_end_wave
__device__ __forceinline__ bool fe_dep_give_up(const fl_fe_wave& w, int job, long long t0) {
  if (w.dep_error && *reinterpret_cast<volatile int*>(w.dep_error) != 0) return true;
  if (clock64() - t0 <= (1ll << 31)) return false;
  if (w.dep_error) atomicCAS(w.dep_error, 0, 1 + job);
  if (w.dep_error_host) *reinterpret_cast<volatile int*>(w.dep_error_host) = 1 + job;
  __threadfence_system();
  return true;
}

__global__ void __launch_bounds__(256, 8) k_front_end_wave(fl_fe_wave w) {
  extern __shared__ __align__(16) uint8_t smem_dyn[];
  const int b = blockIdx.x;
  fl_grid_dep_wait();                                   // the previous kernel of the stream wrote this wave's inputs
  fl_grid_dep_launch();
  if (w.zero_me && b == 0 && threadIdx.x == 0) *w.zero_me = 0;
  // the job this CTA belongs to: last job whose first CTA is <= b.  Binary search over the (<= 16) jobs: every warp of the grid runs
  // this, and the linear walk it replaces was 10 % of the launch's instructions (ncu, round 2)
  int j = 0;
  {
    int hi = w.n_jobs - 1;
#pragma unroll 1
    while (j < hi) {
      const int mid = (j + hi + 1) >> 1;
      if (b >= w.job[mid].cta_begin) j = mid; else hi = mid - 1;
    }
  }
  const fl_fe_job& jb = w.job[j];
  const int local = b - jb.cta_begin;
  __shared__ unsigned long long s_trace0[2];            // this CTA's start (clock64, globaltimer): kept out of registers of the hot path
  if (w.trace && threadIdx.x == 0) {
    unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    s_trace0[0] = (unsigned long long)clock64(); s_trace0[1] = t;
    atomicMin(w.trace + 2 * j, t);
  }
  if (jb.wait_row_base >= 0) {
    // row-grained wait of a spread CTA (see fl_fe_job): the producer's tile rows that hold this grid row's label rows
    if (threadIdx.x == 0) {
      const int gy = local / jb.gx, T = jb.g.T;
      const int y0 = gy * T, y1 = min(gy * T + 2 * T - 2, jb.g.H - 1);
      const int by0 = (y0 << jb.wait_row_shift) >> 4, by1 = min((y1 << jb.wait_row_shift) >> 4, jb.wait_row_count - 1);
      const long long t0 = clock64();
      for (int by = by0; by <= by1; ++by) {
        const unsigned* c = w.counters + jb.wait_row_base + by;
        unsigned v;
        for (;;) {
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(c) : "memory");
          if ((int)(v - jb.wait_row_target) >= 0) break;
          if (fe_dep_give_up(w, j, t0)) break;
          __nanosleep(64);
        }
      }
    }
    __syncthreads();
  } else if (jb.wait_slot >= 0) {
    // In-grid dependency: a producing job always precedes its consumers in the grid and CTAs are dispatched in blockIdx order on
    // every configuration this was run on, so every producer CTA is resident (or done) before a consumer starts to wait here.
    // CUDA does not GUARANTEE that order (MPS time slicing, a debugger, compute-sanitizer, a future scheduler), so the wait is
    // bounded: after ~1 s the CTA records the job in dep_error (device word for the other waiters, mapped host word for the
    // library), every waiter of the grid gives up at once, the frame's result is discarded by the host, which re-runs the frame
    // as one launch per wave (no in-grid waits) and keeps this handle on that path (fe_dep_give_up, fl_match_wait).
    if (threadIdx.x == 0) {
      const unsigned* c = w.counters + jb.wait_slot;
      const long long t0 = clock64();
      unsigned v;
      for (;;) {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(c) : "memory");
        if ((int)(v - jb.wait_target) >= 0) break;
        if (fe_dep_give_up(w, j, t0)) break;
        __nanosleep(64);
      }
    }
    __syncthreads();
  }
  switch (jb.kind) {
    case FL_JOB_PYRDOWN:
      if (jb.p0) dev_pyrdown_bgr<true>(jb.src, jb.W, jb.H, jb.dst, local);
      else dev_pyrdown_bgr<false>(jb.src, jb.W, jb.H, jb.dst, local);
      break;
    case FL_JOB_RESIZE: dev_resize_nn_half(jb.src, jb.W, jb.H, jb.dst, local); break;
    case FL_JOB_SPREAD: dev_spread_lm_any(jb, local % jb.gx, local / jb.gx, smem_dyn); break;
    case FL_JOB_PREFETCH: {
      const size_t line = (size_t)local * 256 + threadIdx.x;
      if (line * 128 < (size_t)jb.W * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(jb.src + line * 128));
      break;
    }
    case FL_JOB_COLOR2: dev_color_quantize_v2(jb.src, jb.W, jb.H, jb.thr_sq, jb.dst, local % jb.gx, local / jb.gx, smem_dyn); break;
    case FL_JOB_DEPTH2:
      dev_depth_quantize_v2(reinterpret_cast<const uint16_t*>(jb.src), jb.W, jb.H, jb.p0, jb.p1, jb.dst, w, jb.gx < 0 ? -1 : (jb.thr_sq > 0.5f ? 1 : 0),
                            local % abs(jb.gx), local / abs(jb.gx), smem_dyn);
      break;
  }
  if (w.trace) {
    __syncthreads();
    if (threadIdx.x == 0) {                             // last end, and this CTA's span (dependency wait included) added to the job's SM time
      unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      const unsigned long long c = (unsigned long long)clock64();
      atomicMax(w.trace + 2 * j + 1, t);
      atomicAdd(w.trace + 2 * FL_FE_MAX_JOBS + 2 * j, c - s_trace0[0]);
      atomicAdd(w.trace + 2 * FL_FE_MAX_JOBS + 2 * j + 1, t - s_trace0[1]);
    }
  }
  if (jb.signal_slot >= 0) {
    __syncthreads();                                    // every thread's stores of this CTA ...
    if (threadIdx.x == 0) {                             // ... are visible before the counts
      __threadfence();
      if (jb.row_base >= 0) atomicAdd(w.counters + jb.row_base + local / abs(jb.gx), 1u);
      atomicAdd(w.counters + jb.signal_slot, 1u);
    }
  }
}

// ---- host side: a frame's front end is ONE list of jobs (fe_build), launched as one grid with in-grid dependencies (fe_run_single)
// or cut into waves, one launch each (fe_run_waves)

// One job of a frame, with what only the host needs: the launch of the per-wave schedule it belongs to (the labels, pyrDown and resize jobs
// of level l are in wave l, the spread job of level l in wave l + 1), the jobs whose output it reads (its labels, and a level of the mask
// pyramid; -1 = none), and for a spread job the level shift of its label rows in the producer's tile rows (-1: waits for the whole job).
struct fe_item { fl_fe_job j; int ctas; size_t smem; int wave, prod[2], row_shift; };
#define FE_LIST_MAX (FL_MAX_LEVELS * (1 + 3 * FL_MAX_MODALITIES))
struct fe_list { int n, n_depth, n_pyr; bool halves; fe_item it[FE_LIST_MAX]; fl_depth_pyr pyr[FL_FE_MAX_DPYR]; };
struct fl_fe_state {
  // the single launch's [FL_FE_MAX_JOBS job counters][1 error word][FL_FE_MAX_JOBS x FL_FE_MAX_TILE_ROWS tile-row counters], never reset between
  // frames: slot i reaches counter_base[i] + its job's CTAs (row_base[i] + tiles per row); the bases advance after every launch that went out
  fl_dev_buf<unsigned> counters; unsigned counter_base[FL_FE_MAX_JOBS] = {}, row_base[FL_FE_MAX_JOBS] = {};
  fl_mapped_buf<int> err; int* err_dev = nullptr;       // 1 + the job whose wait timed out, in mapped host memory (+ its device alias)
  bool force_waves = false, opt_waves = false, opt_dep_test = false;   // a wait timed out (one launch per wave from then on); FL_OPT_FE_*
  fl_dev_buf<unsigned long long> trace; int trace_jobs = 0, trace_kind[FL_FE_MAX_JOBS] = {}, trace_ctas[FL_FE_MAX_JOBS] = {};   // FL_DBG_FE_TRACE
  fe_list list;                                         // the current frame's jobs (20 KB: kept off the enqueue's stack)
};
void fl_fe_free::operator()(fl_fe_state* s) const { delete s; }
int fl_fe_create(fl_fe_owned* out) {
  fl_fe_owned fe(new (std::nothrow) fl_fe_state());
  if (!fe) return FL_ERR_ARG;
  const size_t n = (FL_FE_MAX_JOBS + 1) + FL_FE_MAX_JOBS * FL_FE_MAX_TILE_ROWS;
  int rc;
  if ((rc = fe->counters.alloc(n)) != FL_OK || (rc = fe->err.alloc(16)) != FL_OK) return rc;
  FL_CUDA(cudaMemset(fe->counters.get(), 0, n * sizeof(unsigned)));
  *fe->err.get() = 0;
  FL_CUDA(cudaHostGetDevicePointer((void**)&fe->err_dev, fe->err.get(), 0));
  *out = std::move(fe);
  return FL_OK;
}
int fl_fe_forget_rows(fl_fe_state* fe, cudaStream_t s) {
  FL_CUDA(cudaMemsetAsync(fe->counters.get() + (FL_FE_MAX_JOBS + 1), 0, (size_t)FL_FE_MAX_JOBS * FL_FE_MAX_TILE_ROWS * sizeof(unsigned), s));
  memset(fe->row_base, 0, sizeof fe->row_base);
  return FL_OK;
}
static fl_fe_job& fe_init(fe_item& it, int kind, int wave, int ctas, size_t smem, int prod0 = -1, int prod1 = -1, int row_shift = -1) {
  memset(&it, 0, sizeof it);
  it.j.kind = kind; it.j.wait_slot = it.j.signal_slot = it.j.row_base = it.j.wait_row_base = -1;
  it.ctas = ctas; it.smem = smem; it.wave = wave; it.prod[0] = prod0; it.prod[1] = prod1; it.row_shift = row_shift;
  return it.j;
}
// nearest-neighbour x1/2 of a level-(l - 1) image into level l; returns the job's index
static int fe_add_resize(fe_list& F, int l, const uint8_t* src, const fl_level_geom& g, uint8_t* dst, int prod) {
  fl_fe_job& j = fe_init(F.it[F.n++], FL_JOB_RESIZE, l, ((g.W / 2) * (g.H / 2) + 255) / 256, 0, prod);
  j.src = src; j.dst = dst; j.W = g.W; j.H = g.H; j.gx = 1;
  return F.n - 1;
}

// Every job of the frame, once, in the order of the single launch: the colour pyramid chain (short jobs, on the critical path of the
// coarsest level), the depth labels, the colour labels coarsest level first, then spread + response maps + linear memories coarsest level
// first (the similarity kernel needs only that one).  The resize jobs, which only the per-wave schedule takes, follow the depth labels.
static void fe_build(const fl_fe_frame& f, fe_list& F) {
  const int L = f.n_levels, M = f.n_modalities;
  F.n = F.n_depth = F.n_pyr = 0; F.halves = true;
  for (int l = 0; l + 1 < L; ++l) F.halves &= f.geom[l].W % 2 == 0 && f.geom[l].H % 2 == 0;
  bool color = false;
  for (int m = 0; m < M; ++m) color |= f.modality_kind[m] == FL_MODALITY_COLOR_GRADIENT;
  // the producing jobs: of colour level l, of the labels of (l, m), of mask level l of modality m
  int bgr[FL_MAX_LEVELS] = {-1}, lab[FL_MAX_LEVELS][FL_MAX_MODALITIES], msk[FL_MAX_LEVELS][FL_MAX_MODALITIES];
  if (color)                                            // one chain, shared by all colour modalities
    for (int l = 0; l + 1 < L; ++l) {
      const fl_level_geom& g = f.geom[l];
      fl_fe_job& j = fe_init(F.it[F.n++], FL_JOB_PYRDOWN, l, pyrdown_ctas(g.W, g.H), 0, bgr[l]);
      j.src = l == 0 ? f.bgr : f.bgr_pyr[l]; j.dst = f.bgr_pyr[l + 1]; j.W = g.W; j.H = g.H; j.gx = 1;
      j.p0 = l == 0; bgr[l + 1] = F.n - 1;              // p0: the source was complete before the launch (see dev_pyrdown_bgr)
    }
  // The depth job also writes the NN-downsampled pyramid of its labels when every level halves exactly (then dst_l(y, x) = src(2^l y, 2^l x))
  // and the launch has a pyramid slot left; otherwise resize jobs halve the labels level by level.
  for (int m = 0; m < M; ++m) {
    if (f.modality_kind[m] != FL_MODALITY_DEPTH_NORMAL) continue;
    const fl_level_geom& g = f.geom[0];
    const bool pyr = L > 1 && F.halves && L - 1 <= FL_FE_MAX_PYR && F.n_pyr < FL_FE_MAX_DPYR;
    const int gx = (g.W + D2_TW - 1) / D2_TW;
    fl_fe_job& j = fe_init(F.it[F.n++], FL_JOB_DEPTH2, 0, gx * ((g.H + D2_TH - 1) / D2_TH), D2_SMEM_BYTES);
    j.src = reinterpret_cast<const uint8_t*>(f.depth); j.dst = f.q[0][m]; j.W = g.W; j.H = g.H; j.p0 = f.dist_thr; j.p1 = f.diff_thr;
    j.gx = pyr ? gx : -gx;                              // gx < 0: no pyramid; thr_sq carries the pyramid slot
    if (pyr) {
      fl_depth_pyr& P = F.pyr[F.n_pyr];
      memset(&P, 0, sizeof P); P.n = L - 1;
      for (int k = 1; k < L; ++k) { P.W[k - 1] = f.geom[k].W; P.H[k - 1] = f.geom[k].H; P.dst[k - 1] = f.q[k][m]; }
      j.thr_sq = (float)F.n_pyr++;
    }
    ++F.n_depth; lab[0][m] = F.n - 1;
    for (int l = 1; l < L; ++l) lab[l][m] = pyr ? lab[0][m] : fe_add_resize(F, l, f.q[l - 1][m], f.geom[l - 1], f.q[l][m], lab[l - 1][m]);
  }
  // A masked modality's spread job reads the level-0 mask at a shift of l when every level halves exactly (NN-halving then picks
  // src(2y, 2x)); otherwise resize jobs build the mask pyramid next to the depth labels'.
  for (int m = 0; m < M; ++m)
    for (int l = 0; l < L; ++l)
      msk[l][m] = l > 0 && f.mask[m] && !F.halves ? fe_add_resize(F, l, l == 1 ? f.mask[m] : f.mask_pyr[l - 1][m], f.geom[l - 1], f.mask_pyr[l][m], msk[l - 1][m]) : -1;
  for (int l = L - 1; l >= 0; --l)
    for (int m = 0; m < M; ++m) {
      if (f.modality_kind[m] != FL_MODALITY_COLOR_GRADIENT) continue;
      const fl_level_geom& g = f.geom[l];
      const int gx = (g.W + C2_TW - 1) / C2_TW;
      fl_fe_job& j = fe_init(F.it[F.n++], FL_JOB_COLOR2, l, gx * ((g.H + C2_TH - 1) / C2_TH), C2_SMEM_BYTES, bgr[l]);
      j.src = l == 0 ? f.bgr : f.bgr_pyr[l]; j.dst = f.q[l][m]; j.W = g.W; j.H = g.H; j.thr_sq = f.thr_sq; j.gx = gx;
      lab[l][m] = F.n - 1;
    }
  for (int l = L - 1; l >= 0; --l)
    for (int m = 0; m < M; ++m) {
      const fl_level_geom& g = f.geom[l];
      int cw = SL_CW;                                   // small levels: narrower CTAs so that the job still fills the SMs
      while (cw > 8 && ((g.Wd + cw - 1) / cw) * g.Hd < 148) cw >>= 1;
      const int gx = (g.Wd + cw - 1) / cw;
      // labels that the level-0 job wrote (the depth job's own pyramid): row y of level l is its row y << l
      fl_fe_job& j = fe_init(F.it[F.n++], FL_JOB_SPREAD, l + 1, gx * g.Hd, spread_smem_bytes(g.T), lab[l][m], msk[l][m], lab[l][m] == lab[0][m] ? l : 0);
      const bool coarsest = l == L - 1, mpyr = msk[l][m] >= 0;
      j.src = f.q[l][m]; j.dst = f.lm[l] + (size_t)m * g.mod_stride; j.dst2 = f.spread[l][m];
      j.dst3 = coarsest && f.lm4 ? f.lm4 + (((size_t)m * g.mod_stride) >> 1) : nullptr; j.mass = coarsest && f.mass ? f.mass + 8 * m : nullptr;
      j.mask = mpyr ? f.mask_pyr[l][m] : f.mask[m]; j.mask_stride = mpyr ? g.W : f.geom[0].W; j.mask_shift = mpyr ? 0 : l;
      j.g = g; j.W = g.W; j.H = g.H; j.p0 = cw; j.gx = gx;
    }
}
static void fe_wave_begin(fl_fe_wave& w, const fe_list& F, int* zero_me) {
  w.n_jobs = w.n_ctas = 0; w.smem = 0; w.zero_me = zero_me; w.counters = nullptr; w.dep_error = w.dep_error_host = nullptr; w.trace = nullptr;
  w.n_pyr = F.n_pyr; memcpy(w.pyr, F.pyr, sizeof w.pyr);
}
static void fe_append(fl_fe_wave& w, const fe_item& it) {
  fl_fe_job& j = w.job[w.n_jobs++] = it.j;
  j.cta_begin = w.n_ctas; w.n_ctas += it.ctas; w.smem = w.smem > it.smem ? w.smem : it.smem;
}
static int fe_ctas(const fl_fe_wave& w, int i) { return (i + 1 < w.n_jobs ? w.job[i + 1].cta_begin : w.n_ctas) - w.job[i].cta_begin; }
static int fe_launch(const fl_fe_wave& w, cudaStream_t s, int64_t* launches) {
  ++*launches;
  if ((w.n_ctas > 0 ? fl_launch(k_front_end_wave, dim3(w.n_ctas), dim3(256), w.smem, s, w) : cudaSuccess) == cudaSuccess) return FL_OK;
  fl_set_error("front-end launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return FL_ERR_CUDA;
}

// Single launch: every job of the frame in ONE grid, producers before consumers, dependencies resolved by per-job CTA counters inside the
// kernel (k_front_end_wave).  Removes L launches and their dependency gaps, and lets the level-0 work fill the machine while the short
// critical chain pyrDown -> colour L(top) -> spread L(top) runs.
static int fe_run_single(fl_fe_state& S, const fl_fe_frame& f, const fe_list& F, cudaStream_t s, int64_t* launches) {
  fl_fe_wave w;
  fe_wave_begin(w, F, f.zero_me);                       // resets the candidate counter: no memset node between the kernels
  w.counters = S.counters.get(); w.dep_error = reinterpret_cast<int*>(w.counters + FL_FE_MAX_JOBS); w.dep_error_host = S.err_dev;
  for (int i = 0, room = FL_FE_MAX_JOBS - F.n; i < (room >= 6 ? 6 : room >= 3 ? 3 : 0); ++i) {
    const int lines = (int)((f.prefetch_bytes[i] + 127) / 128);
    if (lines <= 0) continue;
    fe_item it;
    fl_fe_job& j = fe_init(it, FL_JOB_PREFETCH, 0, (lines + 255) / 256, 0);
    j.src = static_cast<const uint8_t*>(f.prefetch[i]); j.W = lines; j.gx = 1;
    fe_append(w, it);
  }
  const int off = w.n_jobs;                             // list job i is job off + i of the grid and owns counter slot off + i
  for (int i = 0; i < F.n; ++i) fe_append(w, F.it[i]);
  // FL_OPT_FE_DEP_TIMEOUT_TEST: this frame's waits for whole jobs ask for one CTA more than the producer has, i.e. they time out
  const unsigned dep_test = S.opt_dep_test ? 1u : 0u;
  S.opt_dep_test = false;
  for (int i = 0; i < F.n; ++i) {                       // (no job of a single launch has a second producer: that is a mask pyramid level)
    const int p = off + F.it[i].prod[0];
    if (p < off) continue;
    fl_fe_job& j = w.job[off + i]; fl_fe_job& pj = w.job[p];
    pj.signal_slot = p;
    j.wait_slot = p; j.wait_target = S.counter_base[p] + (unsigned)fe_ctas(w, p) + dep_test;
    // a spread job waits only for the tile rows of the producer that hold its label rows (see fl_fe_job), if the producer has few enough
    const int rows = (pj.H + 15) / 16;
    if (F.it[i].row_shift < 0 || rows > FL_FE_MAX_TILE_ROWS) continue;
    pj.row_base = (FL_FE_MAX_JOBS + 1) + p * FL_FE_MAX_TILE_ROWS;
    j.wait_row_base = pj.row_base; j.wait_row_shift = F.it[i].row_shift; j.wait_row_count = rows; j.wait_row_target = S.row_base[p] + (unsigned)abs(pj.gx);
  }
  if (f.trace) {                                        // developer timeline: per job first start / last end, summed CTA spans
    if (int rc = S.trace.grow(4 * FL_FE_MAX_JOBS)) return rc;
    unsigned long long init[4 * FL_FE_MAX_JOBS] = {};
    for (int i = 0; i < FL_FE_MAX_JOBS; ++i) init[2 * i] = ~0ull;   // first CTA start (min), then last end (max), then the span sums
    FL_CUDA(cudaMemcpyAsync(S.trace.get(), init, sizeof init, cudaMemcpyHostToDevice, s));
    FL_CUDA(cudaStreamSynchronize(s));
    w.trace = S.trace.get(); S.trace_jobs = w.n_jobs;
    for (int i = 0; i < w.n_jobs; ++i) { S.trace_kind[i] = w.job[i].kind; S.trace_ctas[i] = fe_ctas(w, i); }
  }
  if (int rc = fe_launch(w, s, launches)) return rc;
  for (int i = 0; i < w.n_jobs; ++i) {                  // the bases advance only when the launch went out (a failed launch bumps no counter)
    if (w.job[i].signal_slot >= 0) S.counter_base[i] += (unsigned)fe_ctas(w, i);
    if (w.job[i].row_base >= 0) S.row_base[i] += (unsigned)abs(w.job[i].gx);
  }
  return FL_OK;
}

// Per wave: L + 1 launches, no in-grid waits; wave l produces the labels of level l and the linear memories of level l - 1.  Within a wave
// the longest jobs go first: the kernel ends with its slowest CTA, and CTAs are scheduled in job order.  (Measured alternative: slicing the
// level-0 colour quantisation over the waves and moving every spread to the last wave - 16.6 + 10.8 + 9.2 us instead of 17.7 + 9.4 + 6.0
// us, i.e. no gain: each wave has a latency floor of one colour-tile CTA, about 8 us.)
static int fe_run_waves(const fl_fe_frame& f, const fe_list& F, cudaStream_t s, int64_t* launches) {
  static const int order[] = {FL_JOB_COLOR2, FL_JOB_DEPTH2, FL_JOB_SPREAD, FL_JOB_PYRDOWN, FL_JOB_RESIZE};
  fl_fe_wave w;
  fe_wave_begin(w, F, f.zero_me);                       // the first launch resets the candidate counter
  auto flush = [&]() { const int rc = fe_launch(w, s, launches); fe_wave_begin(w, F, nullptr); return rc; };
  int rc = FL_OK;
  for (int wave = 0; wave <= f.n_levels && rc == FL_OK; ++wave) {
    for (int kind : order)
      for (int i = 0; i < F.n && rc == FL_OK; ++i) {
        if (F.it[i].wave != wave || F.it[i].j.kind != kind) continue;
        if (w.n_jobs == FL_FE_MAX_JOBS && (rc = flush()) != FL_OK) break;   // jobs of one wave are independent: splitting a wave is safe
        fe_append(w, F.it[i]);
        if (kind == FL_JOB_PYRDOWN) w.job[w.n_jobs - 1].p0 = 1;   // its source was written by an earlier launch
      }
    if (rc == FL_OK && w.n_jobs > 0) rc = flush();
  }
  return rc;
}
int fl_fe_run(fl_fe_state* fe, const fl_fe_frame& f, cudaStream_t s, int64_t* launches) {
  fe_list& F = fe->list;
  fe_build(f, F);
  // The in-grid waits know one producer per job and the depth pyramid's tile rows at a shift of the level.  So the single launch takes a
  // list in which every level halves exactly and every depth job writes its own pyramid (no resize job), and that fits one grid.
  const bool single = !fe->opt_waves && !fe->force_waves && F.halves && F.n_depth <= FL_FE_MAX_DPYR && F.n <= FL_FE_MAX_JOBS;
  return single ? fe_run_single(*fe, f, F, s, launches) : fe_run_waves(f, F, s, launches);
}
int fl_fe_take_timeout(fl_fe_state* fe, cudaStream_t s, int* job) {
  *job = *reinterpret_cast<volatile int*>(fe->err.get()) - 1;
  if (*job < 0) return FL_OK;
  *fe->err.get() = 0; fe->force_waves = true;
  FL_CUDA(cudaMemsetAsync(fe->counters.get() + FL_FE_MAX_JOBS, 0, sizeof(unsigned), s));
  return FL_OK;
}
int fl_fe_trace(const fl_fe_state* fe, void* host_out, size_t bytes) {
  if (!fe->trace.get() || fe->trace_jobs <= 0) return FL_ERR_STATE;
  if (bytes < (size_t)fe->trace_jobs * 6 * sizeof(unsigned long long)) return FL_ERR_CAPACITY;
  unsigned long long raw[4 * FL_FE_MAX_JOBS];
  FL_CUDA(cudaMemcpy(raw, fe->trace.get(), sizeof raw, cudaMemcpyDeviceToHost));
  unsigned long long* o = static_cast<unsigned long long*>(host_out);
  for (int i = 0; i < fe->trace_jobs; ++i) {
    o[6 * i] = (unsigned long long)fe->trace_kind[i]; o[6 * i + 1] = (unsigned long long)fe->trace_ctas[i]; o[6 * i + 2] = raw[2 * i]; o[6 * i + 3] = raw[2 * i + 1];
    o[6 * i + 4] = raw[2 * FL_FE_MAX_JOBS + 2 * i]; o[6 * i + 5] = raw[2 * FL_FE_MAX_JOBS + 2 * i + 1];
  }
  return fe->trace_jobs;
}
int fl_fe_option(fl_fe_state* fe, int option, int value) {
  switch (option) {
    case FL_OPT_FE_WAVES: fe->opt_waves = value != 0; return FL_OK;
    case FL_OPT_FE_DEP_TIMEOUT_TEST: fe->opt_dep_test = value != 0; return FL_OK;
    case FL_OPT_FE_FORCED_WAVES: return fe->force_waves ? 1 : 0;   // query: has a time-out switched this handle to wave launches?
  }
  return FL_ERR_ARG;
}
