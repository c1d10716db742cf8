// Word-parallel colour-gradient and depth-normal quantisers, the colour and depth jobs of k_front_end_wave (included by
// frontend.cu; they replaced the byte-granular first versions, which are deleted).
//
// The first versions spent ~900 (colour) and ~550 (depth) instructions per pixel on byte-granular shared-memory tiles.
// Here every stage works on 32-bit words of four pixels:
//   colour: BGR de-interleaved into planar tiles on load (PRMT); horizontal 7-tap blur = 2 IDP.4A per pixel and channel;
//           the 16-bit row sums are stored as VERTICAL pairs so that the vertical 7-tap is 4 IDP.2A; Sobel dx/dy = 5
//           IDP.4A with signed weights; the 3x3 majority vote is a bit-sliced adder network on one-hot bytes (all 8 bins
//           of 4 pixels at once).
//   depth : labels are kept as THERMOMETER codes (bit k set <=> label >= 1 << k), which turns the 5x5 median into
//           "per bit: at least 13 of 25 set" - a separable bit-sliced count (5 rows, then 5 columns).
// Reference: quantizedOrientations + hysteresisGradient linemod/linemod.cpp:230-385, quantizedNormals :567-685
// (medianBlur :684), DepthNormalPyramid::pyrDown :721-745.
#pragma once

__device__ __forceinline__ uint32_t idp4a_uu(uint32_t a, uint32_t b, uint32_t c) { uint32_t d; asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
__device__ __forceinline__ int idp4a_us(uint32_t a, uint32_t b, int c) { int d; asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
__device__ __forceinline__ uint32_t idp2a_lo(uint32_t a, uint32_t b, uint32_t c) { uint32_t d; asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
__device__ __forceinline__ uint32_t idp2a_hi(uint32_t a, uint32_t b, uint32_t c) { uint32_t d; asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
// bit-sliced full adder on 32 independent bit columns
__device__ __forceinline__ uint32_t bs_xor3(uint32_t a, uint32_t b, uint32_t c) { return a ^ b ^ c; }
__device__ __forceinline__ uint32_t bs_maj(uint32_t a, uint32_t b, uint32_t c) { return (a & b) | (a & c) | (b & c); }

// ------------------------------------------------------------------------------------------------
// colour quantisation, one 32 x 16 tile per CTA of 256 threads
//   s_src [3][26][48]  planar source, rows y0-5.., columns x0-8.. (BORDER_REPLICATE applied on load)
//   s_h   [3][13][40]  words (h[2rp][x] | h[2rp+1][x] << 16): horizontal 7-tap sums, column hx <-> x0-4+hx
//   s_b   [3][20][40]  blurred bytes, row by <-> y0-2+by, column bx <-> x0-4+bx
//   s_q   [18][36]     one-hot bin of quantized_unfiltered, (qy, qx) <-> (y0-1+qy, x0-1+qx)
//   s_f   [18][36]     0xFF where magnitude > threshold^2 and the pixel is not on the 1-px frame
// Blurred values at positions outside the image are never consumed: Sobel is only evaluated for 0 < x < W-1, 0 < y < H-1
// (the 1-px frame of quantized_unfiltered is zero, :318-325), so its taps stay inside the image.
// ------------------------------------------------------------------------------------------------
#define C2_TW 32
#define C2_TH 16
#define C2_SH (C2_TH + 10)
#define C2_SWW 12                       // words per source-tile row (48 pixels)
#define C2_HP (C2_SH / 2)               // 13 row pairs
#define C2_BW 40
#define C2_BH (C2_TH + 4)
#define C2_QH (C2_TH + 2)
#define C2_QWW 9                        // words per row of s_q / s_f (36 columns, 34 used)
#define C2_OFF_H (3 * C2_SH * C2_SWW * 4)
#define C2_OFF_B (C2_OFF_H + 3 * C2_HP * C2_BW * 4)
#define C2_OFF_Q (C2_OFF_B + 3 * C2_BH * C2_BW)
#define C2_OFF_F (C2_OFF_Q + C2_QH * C2_QWW * 4)
#define C2_SMEM_BYTES (C2_OFF_F + C2_QH * C2_QWW * 4)

__device__ __forceinline__ void dev_color_quantize_v2(const uint8_t* __restrict__ bgr, int W, int H, float thr_sq, uint8_t* __restrict__ q,
                                                      int bx, int by, uint8_t* smem) {
  uint32_t* s_src = reinterpret_cast<uint32_t*>(smem);
  uint32_t* s_h = reinterpret_cast<uint32_t*>(smem + C2_OFF_H);
  uint32_t* s_b = reinterpret_cast<uint32_t*>(smem + C2_OFF_B);
  uint32_t* s_q = reinterpret_cast<uint32_t*>(smem + C2_OFF_Q);
  uint32_t* s_f = reinterpret_cast<uint32_t*>(smem + C2_OFF_F);
  const int x0 = bx * C2_TW, y0 = by * C2_TH;
  const int tid = threadIdx.x;
  const bool aligned = ((reinterpret_cast<uintptr_t>(bgr) | (uintptr_t)W) & 3) == 0;   // then every 4-pixel group starts on a word

  // 1. load + de-interleave: item = (row, group of 4 pixels)
  // fixed trip count, fully unrolled: the loads of both passes are in flight together (one DRAM round trip, not two)
#pragma unroll
  for (int u = 0; u < (C2_SH * C2_SWW + 255) / 256; ++u) {
    const int i = tid + 256 * u;
    if (i >= C2_SH * C2_SWW) break;
    const int r = i / C2_SWW, k = i - r * C2_SWW;
    const int sy = clampi(y0 - 5 + r, 0, H - 1), sx = x0 - 8 + 4 * k;
    uint32_t w0, w1, w2;
    if (aligned && sx >= 0 && sx + 3 < W) {
      const uint32_t* p = reinterpret_cast<const uint32_t*>(bgr + ((size_t)sy * W + sx) * 3);
      w0 = __ldcg(p); w1 = __ldcg(p + 1); w2 = __ldcg(p + 2);           // L2 loads: a pyramid level may come from an earlier job of this launch
    } else {
      uint32_t b[12];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint8_t* p = bgr + ((size_t)sy * W + clampi(sx + j, 0, W - 1)) * 3;
        b[3 * j] = __ldcg(p); b[3 * j + 1] = __ldcg(p + 1); b[3 * j + 2] = __ldcg(p + 2);
      }
      w0 = b[0] | b[1] << 8 | b[2] << 16 | b[3] << 24;
      w1 = b[4] | b[5] << 8 | b[6] << 16 | b[7] << 24;
      w2 = b[8] | b[9] << 8 | b[10] << 16 | b[11] << 24;
    }
    // w0 = B0 G0 R0 B1 | w1 = G1 R1 B2 G2 | w2 = R2 B3 G3 R3
    s_src[(0 * C2_SH + r) * C2_SWW + k] = __byte_perm(__byte_perm(w0, w1, 0x0630), w2, 0x5210);
    s_src[(1 * C2_SH + r) * C2_SWW + k] = __byte_perm(__byte_perm(w0, w1, 0x0741), w2, 0x6210);
    s_src[(2 * C2_SH + r) * C2_SWW + k] = __byte_perm(__byte_perm(w0, w1, 0x0052), w2, 0x7410);
  }
  __syncthreads();

  // 2. horizontal 7-tap {8,28,56,72,56,28,8} for two rows x four columns per item; sums <= 65,280 fit 16 bits
  for (int i = tid; i < 3 * C2_HP * (C2_BW / 4); i += 256) {
    const int qd = i % (C2_BW / 4), t = i / (C2_BW / 4);      // t = ch * 13 + rp
    const int ch = t / C2_HP, rp = t - ch * C2_HP;
    const uint32_t* r0 = s_src + (ch * C2_SH + 2 * rp) * C2_SWW + qd;
    uint32_t h[2][4];
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      const uint32_t a = r0[rr * C2_SWW], b = r0[rr * C2_SWW + 1], c = r0[rr * C2_SWW + 2];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t A = j == 3 ? b : __funnelshift_r(a, b, 8 * (j + 1));
        const uint32_t B = j == 3 ? c : __funnelshift_r(b, c, 8 * (j + 1));
        h[rr][j] = idp4a_uu(A, 0x48381C08u, idp4a_uu(B, 0x00081C38u, 0u));
      }
    }
    uint4 o;
    o.x = h[0][0] | h[1][0] << 16; o.y = h[0][1] | h[1][1] << 16; o.z = h[0][2] | h[1][2] << 16; o.w = h[0][3] | h[1][3] << 16;
    *reinterpret_cast<uint4*>(s_h + t * C2_BW + 4 * qd) = o;
  }
  __syncthreads();

  // 3. vertical 7-tap on the row pairs, single rounding (sum + 2^15) >> 16: two rows x four columns per item
  for (int i = tid; i < 3 * (C2_BH / 2) * (C2_BW / 4); i += 256) {
    const int qd = i % (C2_BW / 4), t = i / (C2_BW / 4);      // t = ch * 10 + k
    const int ch = t / (C2_BH / 2), k = t - ch * (C2_BH / 2);
    const uint4* p = reinterpret_cast<const uint4*>(s_h + (ch * C2_HP + k) * C2_BW + 4 * qd);
    const uint4 e0 = p[0], e1 = p[C2_BW / 4], e2 = p[2 * (C2_BW / 4)], e3 = p[3 * (C2_BW / 4)];
    const uint32_t E[4][4] = {{e0.x, e1.x, e2.x, e3.x}, {e0.y, e1.y, e2.y, e3.y}, {e0.z, e1.z, e2.z, e3.z}, {e0.w, e1.w, e2.w, e3.w}};
    uint32_t ev[4], od[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      // even output row 2k: rows 2k..2k+6 -> weights (8,28)(56,72)(56,28)(8,0); odd row 2k+1: (0,8)(28,56)(72,56)(28,8)
      ev[c] = idp2a_hi(E[c][3], 0x00081C38u, idp2a_lo(E[c][2], 0x00081C38u, idp2a_hi(E[c][1], 0x48381C08u, idp2a_lo(E[c][0], 0x48381C08u, 32768u))));
      od[c] = idp2a_hi(E[c][3], 0x081C3848u, idp2a_lo(E[c][2], 0x081C3848u, idp2a_hi(E[c][1], 0x381C0800u, idp2a_lo(E[c][0], 0x381C0800u, 32768u))));
    }
    // byte 2 of each sum
    s_b[((ch * C2_BH + 2 * k) * C2_BW) / 4 + qd] = __byte_perm(__byte_perm(ev[0], ev[1], 0x0062), __byte_perm(ev[2], ev[3], 0x0062), 0x5410);
    s_b[((ch * C2_BH + 2 * k + 1) * C2_BW) / 4 + qd] = __byte_perm(__byte_perm(od[0], od[1], 0x0062), __byte_perm(od[2], od[3], 0x0062), 0x5410);
  }
  __syncthreads();

  // 4. Sobel 3x3 per channel (5 signed IDP.4A), strongest channel (ties: first, :275-292), angle bin -> one-hot; item = row x 4 columns
  for (int i = tid; i < C2_QH * C2_QWW; i += 256) {
    const int qy = i / C2_QWW, g = i - qy * C2_QWW;
    const int sy = y0 - 1 + qy;
    int bdx[4], bdy[4], bm[4];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const uint32_t* p = s_b + ((ch * C2_BH + qy) * C2_BW) / 4 + g;      // blurred rows qy, qy+1, qy+2 = sy-1, sy, sy+1
      uint32_t A[3][4];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const uint32_t a = p[r * (C2_BW / 4)], b = p[r * (C2_BW / 4) + 1];
        A[r][0] = __funnelshift_r(a, b, 16); A[r][1] = __funnelshift_r(a, b, 24); A[r][2] = b; A[r][3] = b >> 8;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int dx = idp4a_us(A[2][j], 0x000100FFu, idp4a_us(A[1][j], 0x000200FEu, idp4a_us(A[0][j], 0x000100FFu, 0)));
        const int dy = idp4a_us(A[2][j], 0x00010201u, idp4a_us(A[0][j], 0x00FFFEFFu, 0));
        const int m = dx * dx + dy * dy;
        if (ch == 0 || m > bm[j]) { bm[j] = m; bdx[j] = dx; bdy[j] = dy; }     // strict > keeps the earliest channel on ties
      }
    }
    uint32_t qw = 0, fw = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int sx = x0 - 1 + 4 * g + j;
      const bool inner = sx > 0 && sx < W - 1 && sy > 0 && sy < H - 1;
      const int bin = inner ? (angle_q16((float)bdx[j], (float)bdy[j]) & 7) : 0;   // frame pixels are 0 -> bin 0 (:318-335)
      qw |= (1u << bin) << (8 * j);
      if (inner && (float)bm[j] > thr_sq) fw |= 0xFFu << (8 * j);
    }
    s_q[i] = qw; s_f[i] = fw;
  }
  __syncthreads();

  // 5. 3x3 vote: a bin wins with >= 5 of 9 votes (:346-381; at most one bin can, so the tie rule never applies).  Bit-sliced:
  //    the nine one-hot bytes are summed per bit position by full adders, 4 pixels x 8 bins per word.
  const bool waligned = ((reinterpret_cast<uintptr_t>(q) | (uintptr_t)W) & 3) == 0;
  for (int i = tid; i < C2_TH * (C2_TW / 4); i += 256) {
    const int oy = i / (C2_TW / 4), ow = i - oy * (C2_TW / 4);
    const int y = y0 + oy, x = x0 + 4 * ow;
    if (y >= H || x >= W) continue;
    uint32_t a[9];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const uint32_t w0 = s_q[(oy + r) * C2_QWW + ow], w1 = s_q[(oy + r) * C2_QWW + ow + 1];
      a[3 * r] = w0; a[3 * r + 1] = __funnelshift_r(w0, w1, 8); a[3 * r + 2] = __funnelshift_r(w0, w1, 16);
    }
    const uint32_t f = __funnelshift_r(s_f[(oy + 1) * C2_QWW + ow], s_f[(oy + 1) * C2_QWW + ow + 1], 8);
    const uint32_t s1 = bs_xor3(a[0], a[1], a[2]), c1 = bs_maj(a[0], a[1], a[2]);
    const uint32_t s2 = bs_xor3(a[3], a[4], a[5]), c2 = bs_maj(a[3], a[4], a[5]);
    const uint32_t s3 = bs_xor3(a[6], a[7], a[8]), c3 = bs_maj(a[6], a[7], a[8]);
    const uint32_t b0 = bs_xor3(s1, s2, s3), c4 = bs_maj(s1, s2, s3);          // weight 1 -> bit 0, carry of weight 2
    const uint32_t s5 = bs_xor3(c1, c2, c3), c5 = bs_maj(c1, c2, c3);          // weight 2 (c1..c3) -> s5 (2), c5 (4)
    const uint32_t b1 = s5 ^ c4, c6 = s5 & c4;                                 // bit 1, carry of weight 4
    const uint32_t b2 = c5 ^ c6, b3 = c5 & c6;                                 // bits 2 and 3
    const uint32_t out = (b3 | (b2 & (b1 | b0))) & f;                          // count >= 5
    uint8_t* dst = q + (size_t)y * W + x;
    if (waligned && x + 3 < W) *reinterpret_cast<uint32_t*>(dst) = out;
    else for (int j = 0; j < 4 && x + j < W; ++j) dst[j] = (uint8_t)(out >> (8 * j));
  }
}

// ------------------------------------------------------------------------------------------------
// depth normals + 5x5 median, one 32 x 16 tile per CTA of 256 threads; optionally also writes the NN-downsampled pyramid
// levels (dst_l(y, x) = src(2^l y, 2^l x), DepthNormalPyramid::pyrDown :721-745) so that no resize pass is needed.
//   s_d [30][48] u16   depth, rows y0-7.., columns x0-8.. (0 outside the image)
//   s_t [20][40] u8    thermometer-coded raw labels, (ry, lx) <-> (y0-2+ry, x0-4+lx)
//   s_c [3][16][10]    bit-sliced vertical counts (0..5) of the five rows oy..oy+4, per bit position
//   s_p [20][20] u8    the normal-plane table (g_normal_plane): indexed per pixel, which the constant cache would serialise
// ------------------------------------------------------------------------------------------------
#define D2_TW 32
#define D2_TH 16
#define D2_SH (D2_TH + 14)
#define D2_SW 48
#define D2_LH (D2_TH + 4)
#define D2_LW 40
#define D2_OFF_T (D2_SH * D2_SW * 2)
#define D2_OFF_C (D2_OFF_T + D2_LH * D2_LW)
#define D2_OFF_P (D2_OFF_C + 3 * D2_TH * (D2_LW / 4) * 4)
#define D2_SMEM_BYTES (D2_OFF_P + 400)

__device__ __forceinline__ void dev_depth_quantize_v2(const uint16_t* __restrict__ depth, int W, int H, int dist_thr, int diff_thr,
                                                      uint8_t* __restrict__ q, const fl_fe_wave& wv, int pyr_slot, int bx, int by, uint8_t* smem) {
  uint16_t* s_d = reinterpret_cast<uint16_t*>(smem);
  uint8_t* s_t = smem + D2_OFF_T;
  uint32_t* s_c = reinterpret_cast<uint32_t*>(smem + D2_OFF_C);
  uint8_t* s_p = smem + D2_OFF_P;
  const int x0 = bx * D2_TW, y0 = by * D2_TH;
  const int tid = threadIdx.x;
  const bool aligned = ((reinterpret_cast<uintptr_t>(depth) & 7) | (uintptr_t)(W & 3)) == 0;
  if (tid < 100) reinterpret_cast<uint32_t*>(s_p)[tid] = reinterpret_cast<const uint32_t*>(g_normal_plane)[tid];
#pragma unroll
  for (int u = 0; u < (D2_SH * (D2_SW / 4) + 255) / 256; ++u) {     // unrolled: both passes' loads in flight together
    const int i = tid + 256 * u;
    if (i >= D2_SH * (D2_SW / 4)) break;
    const int r = i / (D2_SW / 4), k = i - r * (D2_SW / 4);
    const int sy = y0 - 7 + r, sx = x0 - 8 + 4 * k;
    uint2 v = make_uint2(0u, 0u);
    if (sy >= 0 && sy < H) {
      if (aligned && sx >= 0 && sx + 3 < W) v = __ldg(reinterpret_cast<const uint2*>(depth + (size_t)sy * W + sx));
      else {
        uint32_t d[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) d[j] = (sx + j >= 0 && sx + j < W) ? depth[(size_t)sy * W + sx + j] : 0u;
        v = make_uint2(d[0] | d[1] << 16, d[2] | d[3] << 16);
      }
    }
    *reinterpret_cast<uint2*>(s_d + r * D2_SW + 4 * k) = v;
  }
  __syncthreads();
  // raw labels for columns lx = 2..37 (x0-2 .. x0+33), rows ry = 0..19; positions outside [5, W-7] x [5, H-7] are 0 (:619, :624)
  for (int i = tid; i < D2_LH * 36; i += 256) {
    const int ry = i / 36, lx = i - ry * 36 + 2;
    const int px = x0 - 4 + lx, py = y0 - 2 + ry;
    uint32_t th = 0;
    if (px >= 5 && px < W - 6 && py >= 5 && py < H - 6) {
      const uint16_t* c = s_d + (ry + 5) * D2_SW + lx + 4;
      const int d = c[0];
      if (d < dist_thr) {
        // accumBilateral :567-579 over the 8 taps (i, j) in {-5, 0, 5}^2 \ (0, 0): with f = |delta| < diff_thr,
        // A0 = sum f i^2, A1 = sum f i j, A3 = sum f j^2, b0 = sum f i delta, b1 = sum f j delta (common factors 25 and 5 pulled out)
        int nx_ = 0, ny_ = 0, nd = 0, sbx = 0, sby = 0;         // counts of valid taps with i != 0, j != 0, signed diagonal count
#pragma unroll
        for (int j = -1; j <= 1; ++j)
#pragma unroll
          for (int ii = -1; ii <= 1; ++ii) {
            if (ii == 0 && j == 0) continue;
            const int delta = (int)c[j * 5 * D2_SW + ii * 5] - d;
            const bool f = abs(delta) < diff_thr;
            const int fd = f ? delta : 0;
            if (ii != 0) { nx_ += f; sbx += ii * fd; }
            if (j != 0) { ny_ += f; sby += j * fd; }
            if (ii != 0 && j != 0) nd += f ? ii * j : 0;
          }
        const int A0 = 25 * nx_, A3 = 25 * ny_, A1 = 25 * nd, b0 = 5 * sbx, b1 = 5 * sby;
        const int det = A0 * A3 - A1 * A1;                      // all fit int32 (SURVEY A.2)
        const int ddx = A3 * b0 - A1 * b1;
        const int ddy = -A1 * b0 + A0 * b1;
        float nx = (float)(617 * ddx), ny = (float)(617 * ddy);
        const float nz = (float)(-det * d);
        const float s = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(nx, nx), __fmul_rn(ny, ny)), __fmul_rn(nz, nz)));
        if (s > 0.f) {
          const float inv = __fdiv_rn(1.0f, s);
          nx = __fmul_rn(nx, inv); ny = __fmul_rn(ny, inv);
          const int v1 = (int)__fadd_rn(__fmul_rn(nx, 10.f), 10.f);   // C truncation :665-667
          const int v2 = (int)__fadd_rn(__fmul_rn(ny, 10.f), 10.f);
          const uint32_t lab = s_p[clampi(v2, 0, 19) * 20 + clampi(v1, 0, 19)];   // one-hot, table is v3-independent
          th = (lab << 1) - 1u;                                 // thermometer: bits 0..k for label 1 << k
        }
      }
    }
    s_t[ry * D2_LW + lx] = (uint8_t)th;
  }
  __syncthreads();
  // medianBlur 5x5 (:684) on values ordered 0 < 1 < 2 < ... < 128: bit k of the median's thermometer code = "at least 13 of
  // the 25 inputs have bit k".  Vertical pass: per bit position, the count (0..5) over rows oy..oy+4 as 3 bit planes.
  for (int i = tid; i < D2_TH * (D2_LW / 4); i += 256) {
    const int oy = i / (D2_LW / 4), lw = i - oy * (D2_LW / 4);
    const uint32_t* p = reinterpret_cast<const uint32_t*>(s_t) + oy * (D2_LW / 4) + lw;
    const uint32_t a = p[0], b = p[D2_LW / 4], c = p[2 * (D2_LW / 4)], d = p[3 * (D2_LW / 4)], e = p[4 * (D2_LW / 4)];
    const uint32_t s = bs_xor3(a, b, c), c1 = bs_maj(a, b, c);
    const uint32_t n0 = bs_xor3(s, d, e), c2 = bs_maj(s, d, e);
    s_c[(0 * D2_TH + oy) * (D2_LW / 4) + lw] = n0;
    s_c[(1 * D2_TH + oy) * (D2_LW / 4) + lw] = c1 ^ c2;
    s_c[(2 * D2_TH + oy) * (D2_LW / 4) + lw] = c1 & c2;
  }
  __syncthreads();
  const bool waligned = ((reinterpret_cast<uintptr_t>(q) | (uintptr_t)W) & 3) == 0;
  for (int i = tid; i < D2_TH * (D2_TW / 4); i += 256) {
    const int oy = i / (D2_TW / 4), ow = i - oy * (D2_TW / 4);
    const int y = y0 + oy, x = x0 + 4 * ow;
    if (y >= H || x >= W) continue;
    // five 3-bit column counts at byte offsets -2..+2 around the output word (label column lx = 4 ow + 4 + j)
    uint32_t n[5][3];
#pragma unroll
    for (int pl = 0; pl < 3; ++pl) {
      const uint32_t* p = s_c + (pl * D2_TH + oy) * (D2_LW / 4) + ow;
      const uint32_t w0 = p[0], w1 = p[1], w2 = p[2];
      n[0][pl] = __funnelshift_r(w0, w1, 16); n[1][pl] = __funnelshift_r(w0, w1, 24); n[2][pl] = w1;
      n[3][pl] = __funnelshift_r(w1, w2, 8); n[4][pl] = __funnelshift_r(w1, w2, 16);
    }
    // X = n0 + n1, Y = n2 + n3 (4 bits each), Z = X + Y (5 bits), T = Z + n4 (<= 25, 5 bits)
    uint32_t X[4], Y[4], Z[5], T[5], cy;
    X[0] = n[0][0] ^ n[1][0]; cy = n[0][0] & n[1][0];
    X[1] = bs_xor3(n[0][1], n[1][1], cy); cy = bs_maj(n[0][1], n[1][1], cy);
    X[2] = bs_xor3(n[0][2], n[1][2], cy); X[3] = bs_maj(n[0][2], n[1][2], cy);
    Y[0] = n[2][0] ^ n[3][0]; cy = n[2][0] & n[3][0];
    Y[1] = bs_xor3(n[2][1], n[3][1], cy); cy = bs_maj(n[2][1], n[3][1], cy);
    Y[2] = bs_xor3(n[2][2], n[3][2], cy); Y[3] = bs_maj(n[2][2], n[3][2], cy);
    Z[0] = X[0] ^ Y[0]; cy = X[0] & Y[0];
    Z[1] = bs_xor3(X[1], Y[1], cy); cy = bs_maj(X[1], Y[1], cy);
    Z[2] = bs_xor3(X[2], Y[2], cy); cy = bs_maj(X[2], Y[2], cy);
    Z[3] = bs_xor3(X[3], Y[3], cy); Z[4] = bs_maj(X[3], Y[3], cy);
    T[0] = Z[0] ^ n[4][0]; cy = Z[0] & n[4][0];
    T[1] = bs_xor3(Z[1], n[4][1], cy); cy = bs_maj(Z[1], n[4][1], cy);
    T[2] = bs_xor3(Z[2], n[4][2], cy); cy = bs_maj(Z[2], n[4][2], cy);
    T[3] = Z[3] ^ cy; cy = Z[3] & cy;
    T[4] = Z[4] ^ cy;
    const uint32_t ge13 = T[4] | (T[3] & T[2] & (T[1] | T[0]));       // 13 = 01101b
    const uint32_t out = ge13 ^ ((ge13 >> 1) & 0x7F7F7F7Fu);          // thermometer -> one-hot (0 stays 0)
    uint8_t* dst = q + (size_t)y * W + x;
    if (waligned && x + 3 < W) *reinterpret_cast<uint32_t*>(dst) = out;
    else for (int j = 0; j < 4 && x + j < W; ++j) dst[j] = (uint8_t)(out >> (8 * j));
    const int n_pyr = pyr_slot < 0 ? 0 : wv.pyr[pyr_slot].n;
    for (int l = 0; l < n_pyr; ++l) {                                  // NN pyramid: level l+1 takes (y, x) with y, x multiples of 2^(l+1)
      const int sh = l + 1, msk = (1 << sh) - 1;
      if (y & msk) break;
      const int yl = y >> sh, Wl = wv.pyr[pyr_slot].W[l];
      if (yl >= wv.pyr[pyr_slot].H[l]) continue;
      uint8_t* dl = wv.pyr[pyr_slot].dst[l] + (size_t)yl * Wl;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (((x + j) & msk) == 0 && x + j < W && ((x + j) >> sh) < Wl) dl[(x + j) >> sh] = (uint8_t)(out >> (8 * j));
    }
  }
}
