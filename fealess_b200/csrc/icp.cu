// ICP pose refinement on sm_100a: depth back-projection, paired-crop extraction, exact nearest neighbours on a uniform
// grid, and the point-to-point (Kabsch/SVD) iteration of the reference, one CTA per pose hypothesis, all iterations
// inside one kernel launch.
//
// Reference semantics (paths relative to /root/reference; SURVEY.md section 0 D2/D3 and appendix A.7):
//   cup_d2pc::depthTo3d ICP/depth_to_3d.cpp:99-137, 244-260      scale_mat_vec3f / is_vec3f_valid / matToVec ICP/common.cpp:261-266, 382-425
//   detection ICP/detection.cpp:11-254 (test_id == 2)             getMean / transformPoints / copyPoints / getL2distClouds ICP/ICP.cpp:8-111
//   PointsCorresponding (KD-tree 1-NN) ICP/ICP.cpp:193-279        icpCloudToCloud_Ex ICP/ICP.cpp:617-809       NMS ICP/NMS.cpp:6-39
//
// Numerics: the reference accumulates centroids, the (uncentred) covariance and the mean distance SEQUENTIALLY in fp32.
// Its rotation moves by up to ~2e-4 rad per iteration if those sums are reordered or widened (measured; DESIGN.md), which
// is more than the 1e-4 rad parity tolerance, so the sums are reproduced as ordered fp32 chains: one warp lane per
// accumulator walks the (order-preserving) correspondence list.  Everything that is order-free (back-projection,
// nearest-neighbour search, transforms, distances, compaction scans) runs on all threads of the CTA.
// Compiled with -fmad=false so fp32 products and sums round separately, as in the reference build.
#include "fl_internal.cuh"
#include <float.h>
#include <math.h>
#include <mutex>


__device__ __forceinline__ bool pt_valid(float z) { return z <= 900.0f; }   // is_vec3f_valid (NaN fails), common.cpp:261-266

// depth (u16 mm) -> point in mm exactly as depthTo3d (metres, fp32) followed by scale_mat_vec3f(., 1000)
__device__ __forceinline__ float3 backproject_mm(uint16_t dv, int u, int v, float inv_fx, float inv_fy, float cx, float cy) {
  float z = dv == 0 ? __int_as_float(0x7fc00000) : __fmul_rn((float)dv, (float)(1 / 1000.0));
  float xc = __fmul_rn(__fsub_rn((float)u, cx), inv_fx);
  float yc = __fmul_rn(__fsub_rn((float)v, cy), inv_fy);
  return make_float3(__fmul_rn(__fmul_rn(xc, z), 1000.0f), __fmul_rn(__fmul_rn(yc, z), 1000.0f), __fmul_rn(z, 1000.0f));
}

__global__ void __launch_bounds__(256) k_depth_to_3d(const uint16_t* __restrict__ depth, int W, int H, fl_intrinsics_t K,
                                                     float* __restrict__ out3) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= W * H) return;
  int u = i % W, v = i / W;
  const float inv_fx = __fdiv_rn(1.0f, K.fx), inv_fy = __fdiv_rn(1.0f, K.fy);
  uint16_t dv = depth[i];
  float z = dv == 0 ? __int_as_float(0x7fc00000) : __fmul_rn((float)dv, (float)(1 / 1000.0));
  out3[3 * (size_t)i + 0] = __fmul_rn(__fmul_rn(__fsub_rn((float)u, K.cx), inv_fx), z);
  out3[3 * (size_t)i + 1] = __fmul_rn(__fmul_rn(__fsub_rn((float)v, K.cy), inv_fy), z);
  out3[3 * (size_t)i + 2] = z;
}
void fl_launch_depth_to_3d(const uint16_t* depth, int W, int H, fl_intrinsics_t K, float* out3, cudaStream_t s) {
  k_depth_to_3d<<<(W * H + 255) / 256, 256, 0, s>>>(depth, W, H, K, out3);
}

// ------------------------------------------------------------------------------------------------
// K9-K11 fused: ONE persistent launch does, per hypothesis, everything detection() does after the two depth images are known:
// back-projection of the two crops + pairing (detection.cpp:28-44, 112-114), the centroid shift (:162-206) and the whole
// icpCloudToCloud_Ex loop (ICP.cpp:617-809).  One CTA of 1,024 threads works on one hypothesis at a time and takes the next one
// off a ticket counter, so a batch of any size keeps every SM busy and a small batch (Recognition: the top-5 matches) gets one
// SM per hypothesis.
//
// What bounds a hypothesis is NOT bandwidth but three serial fp32 sums per iteration that must round exactly like the
// reference's loops (file header): n dependent FADDs at 4 cycles each (~17 us for 8.4k points).  Everything else is arranged
// around them:
//   * the ordered sums run in warp 0, one lane per column of a record stream (3 + 3 centroid columns, 9 covariance columns, or
//     the single distance column); STAGER warps build the records (coalesced loads, the nine products m[a] * r[b]) into a
//     shared-memory ring one chunk ahead, handing buffers over with named barriers, so a step of the chain is one LDS + one
//     FADD and the chain runs at the FADD latency;
//   * the exact 1-NN search of iteration k + 1 (cvflann KD-tree in the reference) does not need the new dist_mean, only the
//     ACCEPT test does (ICP.cpp:266-273), so all other warps search while warp 0 sums the distances of iteration k; the
//     acceptance + order-preserving compaction happens once the sum is known;
//   * the reference cloud's 64x64 x/y grid (cell starts + points sorted by cell, 16 B each) lives in SHARED memory; a query
//     scans whole grid ROWS of its neighbourhood as contiguous runs (two cell-start reads per row instead of two per cell),
//     first the 3x3 block, then - only if the best distance or the accept radius demands it - the rows of the larger square
//     from the centre outwards, stopping as soon as the next row is farther than the best candidate.
// Squared distance is ((dx*dx + dy*dy) + dz*dz) in fp32 like L2_Simple; ties go to the lower point index; pairs beyond the
// accept radius are dropped by the reference anyway, so the accepted pairs equal the KD-tree's.
// ------------------------------------------------------------------------------------------------
#define ICP_NT 1024
#define ICP_NWARPS (ICP_NT / 32)
#define ICP_REC 15                               // floats per record: m.xyz, r.xyz, m[a] * r[b]
#define ICP_CH 256                               // records per ring buffer (record mode, 2 buffers)
#define ICP_CHS (ICP_CH + 4)                     // column stride inside a buffer (records are staged COLUMN-major; + 4: bank spread)
#define ICP_RBUF (ICP_REC * ICP_CHS)             // floats per record-mode buffer
#define ICP_STAGE_FLOATS (2 * ICP_RBUF + 32)     // 7,832 floats = 31,328 B, incl. slack for the consumer's look-ahead loads
#define ICP_DCH 1024                             // floats per ring buffer in distance mode
#define ICP_DNB 7                                // ... and buffers (7 x 1,024 <= 7,680)
#define ICP_NSTAGE 8                             // stager warps in record mode (one record per thread and chunk)

__device__ __forceinline__ void nb_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void nb_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
#define ICP_BAR_FULL(b) (1 + (b))
#define ICP_BAR_EMPTY(b) (8 + (b))

// block-wide exclusive scan of one int per thread (ICP_NT threads); returns the exclusive prefix, *total = sum
__device__ __forceinline__ int block_excl_scan(int v, int* s_warp, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = s_warp[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += t; }
    s_warp[lane] = w;
  }
  __syncthreads();
  int base = warp > 0 ? s_warp[warp - 1] : 0;
  *total = s_warp[ICP_NWARPS - 1];
  __syncthreads();
  return base + inc - v;
}

// The consumer half of an ordered chain: warp 0 sums NCOL columns of `n_steps` values; chunk c lives in ring buffer c % NB
// (BUF floats each) COLUMN-major: value i of column j at buf[j * STRIDE + i]; lane j owns column j and fetches four steps per
// LDS.128 one group of 16 steps ahead of the adds.  Measured (tools/micro/chain_bench.cu): 4.46 cycles per step = the FADD
// dependent-issue floor; record-major scalar loads ran at 5.3-7.4.  Called by the 32 lanes of warp 0.
template <int NCOL, int CHUNK, int NB, int BUF, int STRIDE>
__device__ __forceinline__ void chain_consume(int n_steps, const float* s_stage, float* s_sum, int bar_threads, unsigned long long* wait_cycles, unsigned long long* add_cycles) {
  const int lane = threadIdx.x & 31;
  const int n_chunks = (n_steps + CHUNK - 1) / CHUNK;
  float acc = 0.f;
  for (int c = 0; c < n_chunks; ++c) {
    const int b = c % NB;
    const long long tw = wait_cycles ? clock64() : 0;
    nb_sync(ICP_BAR_FULL(b), bar_threads);
    if (wait_cycles && lane == 0) *wait_cycles += (unsigned long long)(clock64() - tw);   // time the sum stood still waiting for data
    const int m = min(CHUNK, n_steps - c * CHUNK);
    const long long ta = wait_cycles ? clock64() : 0;
    if (lane < NCOL) {
      const float4* p = reinterpret_cast<const float4*>(s_stage + (size_t)b * BUF + lane * STRIDE);
      float4 v[4], w[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = p[u];                   // (reads past m stay inside the ring and are never added)
      const int full = m >> 2;
      int i = 0;
      for (; i + 4 <= full; i += 4) {
#pragma unroll
        for (int u = 0; u < 4; ++u) w[u] = p[i + 4 + u];
#pragma unroll
        for (int u = 0; u < 4; ++u) { acc = __fadd_rn(acc, v[u].x); acc = __fadd_rn(acc, v[u].y); acc = __fadd_rn(acc, v[u].z); acc = __fadd_rn(acc, v[u].w); }
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = w[u];
      }
      const int left = m - 4 * i;                                 // < 16 values, already in v[]
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (4 * u + 0 < left) acc = __fadd_rn(acc, v[u].x);
        if (4 * u + 1 < left) acc = __fadd_rn(acc, v[u].y);
        if (4 * u + 2 < left) acc = __fadd_rn(acc, v[u].z);
        if (4 * u + 3 < left) acc = __fadd_rn(acc, v[u].w);
      }
    }
    if (wait_cycles && lane == 0) *add_cycles += (unsigned long long)(clock64() - ta);
    __syncwarp();
    if (c + NB < n_chunks) nb_arrive(ICP_BAR_EMPTY(b), bar_threads);
  }
  if (lane < NCOL) s_sum[lane] = acc;
}

__device__ __forceinline__ void matvec3(const float* R, const float* v, float* o) {   // Matx33f * Vec3f: s = 0; s += a*b
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    float s = __fadd_rn(0.f, __fmul_rn(R[3 * i], v[0]));
    s = __fadd_rn(s, __fmul_rn(R[3 * i + 1], v[1]));
    s = __fadd_rn(s, __fmul_rn(R[3 * i + 2], v[2]));
    o[i] = s;
  }
}
__device__ __forceinline__ void matmul3(const float* A, const float* B, float* C) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      float s = __fadd_rn(0.f, __fmul_rn(A[3 * i], B[j]));
      s = __fadd_rn(s, __fmul_rn(A[3 * i + 1], B[3 + j]));
      s = __fadd_rn(s, __fmul_rn(A[3 * i + 2], B[6 + j]));
      C[3 * i + j] = s;
    }
}

// R = V * U^T of the SVD of a 3x3 fp32 matrix: one-sided (Hestenes) Jacobi on the transposed matrix, fp32 rotations with
// fp64 dot products - the scheme of OpenCV's JacobiSVD that cv::SVD::compute (ICP.cpp:741-742) runs for small matrices.
__device__ void svd3_rot(const float* cov, float* R) {
  float At[3][3], Vt[3][3];
  double Wd[3];
  for (int i = 0; i < 3; ++i) for (int k = 0; k < 3; ++k) { At[i][k] = cov[3 * k + i]; Vt[i][k] = (i == k) ? 1.f : 0.f; }
  for (int i = 0; i < 3; ++i) { double sd = 0; for (int k = 0; k < 3; ++k) sd += (double)At[i][k] * At[i][k]; Wd[i] = sd; }
  const float eps = FLT_EPSILON * 2;
  for (int iter = 0; iter < 30; ++iter) {
    bool changed = false;
    for (int i = 0; i < 2; ++i)
      for (int j = i + 1; j < 3; ++j) {
        double a = Wd[i], p = 0, b = Wd[j];
        for (int k = 0; k < 3; ++k) p += (double)At[i][k] * At[j][k];
        if (fabs(p) <= eps * sqrt(a * b)) continue;
        p *= 2;
        double beta = a - b, gamma = sqrt(p * p + beta * beta);
        float c, s;
        if (beta < 0) { double delta = (gamma - beta) * 0.5; s = (float)sqrt(delta / gamma); c = (float)(p / (gamma * s * 2)); }
        else { c = (float)sqrt((gamma + beta) / (gamma * 2)); s = (float)(p / (gamma * c * 2)); }
        a = b = 0;
        for (int k = 0; k < 3; ++k) {
          float t0 = __fadd_rn(__fmul_rn(c, At[i][k]), __fmul_rn(s, At[j][k]));
          float t1 = __fadd_rn(__fmul_rn(-s, At[i][k]), __fmul_rn(c, At[j][k]));
          At[i][k] = t0; At[j][k] = t1;
          a += (double)t0 * t0; b += (double)t1 * t1;
        }
        Wd[i] = a; Wd[j] = b;
        changed = true;
        for (int k = 0; k < 3; ++k) {
          float t0 = __fadd_rn(__fmul_rn(c, Vt[i][k]), __fmul_rn(s, Vt[j][k]));
          float t1 = __fadd_rn(__fmul_rn(-s, Vt[i][k]), __fmul_rn(c, Vt[j][k]));
          Vt[i][k] = t0; Vt[j][k] = t1;
        }
      }
    if (!changed) break;
  }
  float U[3][3];
  for (int i = 0; i < 3; ++i) {
    double sd = 0; for (int k = 0; k < 3; ++k) sd += (double)At[i][k] * At[i][k];
    sd = sqrt(sd);
    float s = (float)(sd > DBL_MIN ? 1 / sd : 0.);
    for (int k = 0; k < 3; ++k) U[i][k] = __fmul_rn(At[i][k], s);
  }
  // Mat(vt.t() * u.t()) (ICP.cpp:744) is a cv::gemm; for CV_32F its kernel accumulates the products in double and rounds once
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) {
    double s = 0.;
    for (int i = 0; i < 3; ++i) s += (double)Vt[i][r] * (double)U[i][c];   // fp32 x fp32 is exact in fp64, so contraction cannot change it
    R[3 * r + c] = (float)s;
  }
}


struct grid_info { float minx, miny, inv_cell, cell, z0, zstep; };   // z0 / zstep: quantisation of the per-cell z ranges

__device__ __forceinline__ int cell_of(float v, float mn, float inv_cell) {
  int c = (int)floorf(__fmul_rn(__fsub_rn(v, mn), inv_cell));
  return min(max(c, 0), FL_ICP_GRID - 1);
}

// exact nearest neighbour of q among the grid points, as far as it can matter: a neighbour whose squared distance exceeds
// bound2 may be missed (the caller drops such pairs).  Returns the SLOT in gp (or -1) and the squared distance.
__device__ __forceinline__ void nn_query(const float4* __restrict__ gp, const int* __restrict__ cs, const unsigned* __restrict__ zr, const grid_info gi,
                                         const float qx, const float qy, const float qz, const float bound2, float* best_out, int* slot_out) {
  float best = FLT_MAX; int bslot = -1, bidx = 0x7fffffff;
  const int cx = cell_of(qx, gi.minx, gi.inv_cell), cy = cell_of(qy, gi.miny, gi.inv_cell);
  auto scan_run = [&](int p0, int p1) {
    for (int p = p0; p < p1; ++p) {
      const float4 r = gp[p];
      const float d0 = __fsub_rn(qx, r.x), d1 = __fsub_rn(qy, r.y), d2 = __fsub_rn(qz, r.z);
      const float dd = __fadd_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)), __fmul_rn(d2, d2));
      if (dd <= best) {                                            // rare after the first few points
        const int id = __float_as_int(r.w);
        if (dd < best || id < bidx) { bidx = id; bslot = p; }
        best = dd;
      }
    }
  };
  {   // the 3 x 3 block around the query's cell: three contiguous runs
    const int x0 = max(cx - 1, 0), x1 = min(cx + 1, FL_ICP_GRID - 1);
    for (int yy = max(cy - 1, 0); yy <= min(cy + 1, FL_ICP_GRID - 1); ++yy) scan_run(cs[yy * FL_ICP_GRID + x0], cs[yy * FL_ICP_GRID + x1 + 1]);
  }
  // every point outside the 3 x 3 block is farther than one cell in x or y (0.9999 absorbs the rounding of cell_of)
  const float c1 = gi.cell * 0.9999f;
  float r2 = fminf(best, bound2);
  if (!(c1 * c1 >= r2)) {
    // The disc of radius sqrt(r2) around q, row by row from the query's row outwards, per row only the cells the disc reaches
    // (the chord), re-evaluated with the best distance found so far.  The clouds are surfaces, so while they are still apart the
    // nearest neighbour is as far as the GAP between them and the disc covers many cells whose points are all about that far
    // away: every cell therefore carries its z range, and a cell is opened only if its box can hold a closer point at all.
    // eps / the one-step slack of the z ranges cover the rounding of cell_of and of the quantisation.
    const float eps = gi.cell * 1e-3f;
    const float r = sqrtf(r2);
    const int y_lo = cell_of(qy - r - eps, gi.miny, gi.inv_cell), y_hi = cell_of(qy + r + eps, gi.miny, gi.inv_cell);
    for (int j = 0; j < FL_ICP_GRID; ++j) {
      bool any = false;
      for (int sgn = 0; sgn < (j ? 2 : 1); ++sgn) {
        const int yy = sgn ? cy - j : cy + j;
        if (yy < y_lo || yy > y_hi) continue;
        any = true;
        const float lo = gi.miny + (float)yy * gi.cell, hi = lo + gi.cell;
        const float dy = fmaxf(fmaxf(lo - qy, qy - hi) - eps, 0.f);      // distance from q to the row's band
        r2 = fminf(best, bound2);
        const float h2 = r2 - dy * dy;
        if (!(h2 > 0.f)) continue;
        const float hx = sqrtf(h2) + eps;
        const int x0 = cell_of(qx - hx, gi.minx, gi.inv_cell), x1 = cell_of(qx + hx, gi.minx, gi.inv_cell);
        for (int xx = x0; xx <= x1; ++xx) {
          if (j <= 1 && xx >= cx - 1 && xx <= cx + 1) continue;          // inside the 3 x 3 block scanned above
          const int c = yy * FL_ICP_GRID + xx;
          const int p0 = cs[c], p1 = cs[c + 1];
          if (p0 == p1) continue;
          const float lox = gi.minx + (float)xx * gi.cell;
          const float dx = fmaxf(fmaxf(lox - qx, qx - (lox + gi.cell)) - eps, 0.f);
          const unsigned zq = zr[c];
          const float zlo = gi.z0 + (float)(zq & 0xFFFFu) * gi.zstep, zhi = gi.z0 + (float)(zq >> 16) * gi.zstep;
          const float dz = fmaxf(fmaxf(zlo - qz, qz - zhi), 0.f);
          if (dx * dx + dy * dy + dz * dz >= fminf(best, bound2)) continue;   // (a lower bound with slack: a skipped cell holds nothing <= best)
          scan_run(p0, p1);
        }
      }
      if (!any && j > 0) break;
    }
  }
  *best_out = best; *slot_out = bslot;
}

// four consecutive points per thread as three 16-byte accesses: a warp moves 1.5 KB of contiguous memory per step instead of
// three stride-12 word accesses (the per-hypothesis arrays start 16-byte aligned: max_pts is a multiple of 4)
struct pts4 { float x[4], y[4], z[4]; };
__device__ __forceinline__ pts4 load_pts4(const float* p) {
  const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1], c = reinterpret_cast<const float4*>(p)[2];
  pts4 r;
  r.x[0] = a.x; r.y[0] = a.y; r.z[0] = a.z; r.x[1] = a.w; r.y[1] = b.x; r.z[1] = b.y;
  r.x[2] = b.z; r.y[2] = b.w; r.z[2] = c.x; r.x[3] = c.y; r.y[3] = c.z; r.z[3] = c.w;
  return r;
}
__device__ __forceinline__ void store_pts4(float* p, const pts4& r) {
  reinterpret_cast<float4*>(p)[0] = make_float4(r.x[0], r.y[0], r.z[0], r.x[1]);
  reinterpret_cast<float4*>(p)[1] = make_float4(r.y[1], r.z[1], r.x[2], r.y[2]);
  reinterpret_cast<float4*>(p)[2] = make_float4(r.z[2], r.x[3], r.y[3], r.z[3]);
}

struct fl_icp_args {
  fl_icp_ws ws;
  fl_icp_params_t prm;
  const fl_icp_hyp* hyps;            // NULL: cloud mode (points and counts already in the workspace)
  const uint16_t* ref_depth; int W, H; fl_intrinsics_t Kr;
  fl_icp_result_t* results;
  int* ticket;                       // zero before the launch
  int smem_pts;                      // grid points that fit the shared-memory copy (0: the grid stays in global memory)
  unsigned long long* trace;         // NULL, or FL_ICP_TRACE_WORDS words per hypothesis: SM cycles per phase (fl_profile)
};

__global__ void __launch_bounds__(ICP_NT, 1) k_icp_fused(const __grid_constant__ fl_icp_args A) {
  extern __shared__ __align__(16) uint8_t s_dyn[];              // [smem_pts float4][4097 int cell starts][4096 z ranges][ICP_STAGE_FLOATS float]
  __shared__ int s_warp[ICP_NWARPS];
  __shared__ float s_red[ICP_NWARPS * 4];
  __shared__ float s_sum[16];
  __shared__ int s_cnt2[2];
  __shared__ float s_apx;                    // unordered sum of the inlier distances: only sizes the speculative neighbour search
  __shared__ float s_Ropt[9], s_Topt[3], s_R[9], s_T[3], s_tinit[3], s_tt[3];
  __shared__ float s_dist_mean, s_dist_diff, s_ratio;
  __shared__ int s_iter, s_go, s_finite, s_h;
  __shared__ grid_info s_gi;
  const fl_icp_ws& ws = A.ws;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float4* s_gp = reinterpret_cast<float4*>(s_dyn);
  int* s_cs = reinterpret_cast<int*>(s_dyn + (size_t)A.smem_pts * 16);
  unsigned* s_zr = reinterpret_cast<unsigned*>(s_cs + FL_ICP_CELLS + 4);   // per cell: quantised {z min (low half), z max (high half)}
  float* s_stage = reinterpret_cast<float*>(s_zr + FL_ICP_CELLS);
  int* s_cur = reinterpret_cast<int*>(s_stage);                 // scatter cursors of the grid build (the ring is idle then)

  for (;;) {
    if (tid == 0) s_h = atomicAdd(A.ticket, 1);
    __syncthreads();
    const int h = s_h;
    if (h >= ws.n_hyp) break;
    float* pref = ws.pts_ref + (size_t)h * ws.max_pts * 3;
    float* tmp = ws.pts_mod + (size_t)h * ws.max_pts * 3;         // pts_mod, then pts_model_tmp
    float* cor_m = ws.cor_m + (size_t)h * ws.max_pts * 3;
    float* cor_r = ws.cor_r + (size_t)h * ws.max_pts * 3;
    float* dist = ws.dist + (size_t)h * ws.max_pts;
    float* nn_d2 = ws.nn_d2 + (size_t)h * ws.max_pts;
    int* nn_slot = ws.nn_slot + (size_t)h * ws.max_pts;
    fl_icp_result_t* res = A.results + h;
    const int status = A.hyps ? A.hyps[h].status : FL_OK;
    int n_ref = 0, n_mod = 0;
    // phase clock (developer timeline, fl_profile): thread 0 charges the cycles since the last stamp to phase p
    unsigned long long* trc = A.trace ? A.trace + (size_t)h * FL_ICP_TRACE_WORDS : nullptr;
    long long t_last = trc ? clock64() : 0;
    const long long t_begin = t_last;
    auto TR = [&](int p) { if (trc && tid == 0) { const long long t = clock64(); trc[p] += (unsigned long long)(t - t_last); t_last = t; } };
    if (trc && tid < FL_ICP_TRACE_WORDS) trc[tid] = 0;

    // ---- record-mode chain (centroids, covariance): warp 0 consumes, warps 1..ICP_NSTAGE stage, the rest wait at the barrier ----
    auto chain_records = [&](const float* pm, int n_m, const float* pr, int n_r, int n_cov) {
      const int n_steps = max(max(n_m, n_r), n_cov);
      const int bar_threads = 32 * (1 + ICP_NSTAGE);
      if (warp == 0) {
        if (n_cov > 0) chain_consume<ICP_REC, ICP_CH, 2, ICP_RBUF, ICP_CHS>(n_steps, s_stage, s_sum, bar_threads, trc ? trc + 12 : nullptr, trc ? trc + 15 : nullptr);
        else chain_consume<6, ICP_CH, 2, ICP_RBUF, ICP_CHS>(n_steps, s_stage, s_sum, bar_threads, trc ? trc + 12 : nullptr, trc ? trc + 15 : nullptr);
      } else if (warp <= ICP_NSTAGE) {
        const int k = tid - 32;                                     // record of the chunk this thread builds
        const int n_chunks = (n_steps + ICP_CH - 1) / ICP_CH;
        for (int c = 0; c < n_chunks; ++c) {
          const int b = c & 1, i = c * ICP_CH + k;
          float m0 = 0.f, m1 = 0.f, m2 = 0.f, r0 = 0.f, r1 = 0.f, r2 = 0.f;
          if (i < n_m || i < n_cov) { m0 = pm[3 * (size_t)i]; m1 = pm[3 * (size_t)i + 1]; m2 = pm[3 * (size_t)i + 2]; }
          if (i < n_r || i < n_cov) { r0 = pr[3 * (size_t)i]; r1 = pr[3 * (size_t)i + 1]; r2 = pr[3 * (size_t)i + 2]; }
          if (c >= 2) nb_sync(ICP_BAR_EMPTY(b), bar_threads);       // (the loads above are already in flight)
          float* o = s_stage + (size_t)b * ICP_RBUF + k;            // column-major: column j of this record at o[j * ICP_CHS]
          const bool im = i < n_m, ir = i < n_r, ic = i < n_cov;
          o[0 * ICP_CHS] = im ? m0 : 0.f; o[1 * ICP_CHS] = im ? m1 : 0.f; o[2 * ICP_CHS] = im ? m2 : 0.f;
          o[3 * ICP_CHS] = ir ? r0 : 0.f; o[4 * ICP_CHS] = ir ? r1 : 0.f; o[5 * ICP_CHS] = ir ? r2 : 0.f;
          if (n_cov > 0) {                                          // covariance += m * r^T (ICP.cpp:731-735): Matx product, s = 0 + a * b
            const float mm[3] = {m0, m1, m2}, rr[3] = {r0, r1, r2};
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
              for (int bb = 0; bb < 3; ++bb) o[(6 + 3 * a + bb) * ICP_CHS] = ic ? __fmul_rn(mm[a], rr[bb]) : 0.f;
          }
          nb_arrive(ICP_BAR_FULL(b), bar_threads);
        }
      }
      __syncthreads();
    };

    // ---- distance pass (getL2distClouds, ICP.cpp:68-111), first half: every index pair valid in both clouds, its distance
    // (cv::norm(Vec3f): squares accumulate in double), inlier = dist <= thr.  The inlier distances go to dist[] (0 for everything
    // else: adding +0 leaves the running sum unchanged), the two integer counters are order free.  All threads. ----
    auto distance_fill = [&](float thr, bool xf) {                // xf: first move the model points by (s_Ropt, s_Topt): transformPoints in place (:756)
      if (tid < 2) s_cnt2[tid] = 0;
      if (tid == 2) s_apx = 0.f;
      __syncthreads();
      int cnt = 0, nin = 0;
      float part = 0.f;
      auto one = [&](float rx, float ry, float rz, float mx, float my, float mz) {
        float d_eff = 0.f;
        if (pt_valid(rz) && pt_valid(mz)) {
          const float dx = __fsub_rn(mx, rx), dy = __fsub_rn(my, ry), dz = __fsub_rn(mz, rz);
          const float d = (float)sqrt((double)dx * dx + (double)dy * dy + (double)dz * dz);
          ++cnt;
          if (d <= thr) { ++nin; d_eff = d; part += d; }
        }
        return d_eff;
      };
      float Ro[9], To[3];
#pragma unroll
      for (int k = 0; k < 9; ++k) Ro[k] = xf ? s_Ropt[k] : 0.f;
#pragma unroll
      for (int k = 0; k < 3; ++k) To[k] = xf ? s_Topt[k] : 0.f;
      auto xform = [&](float& x, float& y, float& z) {
        if (!pt_valid(z)) return;
        const float p[3] = {x, y, z};
        float o[3]; matvec3(Ro, p, o);
        x = __fadd_rn(o[0], To[0]); y = __fadd_rn(o[1], To[1]); z = __fadd_rn(o[2], To[2]);
      };
      for (int i4 = 4 * tid; i4 + 4 <= n_mod; i4 += 4 * ICP_NT) {
        const pts4 r = load_pts4(pref + 3 * (size_t)i4);
        pts4 m = load_pts4(tmp + 3 * (size_t)i4);
        if (xf) {
#pragma unroll
          for (int k = 0; k < 4; ++k) xform(m.x[k], m.y[k], m.z[k]);
          store_pts4(tmp + 3 * (size_t)i4, m);
        }
        float4 d;
        d.x = one(r.x[0], r.y[0], r.z[0], m.x[0], m.y[0], m.z[0]); d.y = one(r.x[1], r.y[1], r.z[1], m.x[1], m.y[1], m.z[1]);
        d.z = one(r.x[2], r.y[2], r.z[2], m.x[2], m.y[2], m.z[2]); d.w = one(r.x[3], r.y[3], r.z[3], m.x[3], m.y[3], m.z[3]);
        *reinterpret_cast<float4*>(dist + i4) = d;
      }
      for (int i = (n_mod & ~3) + tid; i < n_mod; i += ICP_NT) {
        if (xf) xform(tmp[3 * (size_t)i], tmp[3 * (size_t)i + 1], tmp[3 * (size_t)i + 2]);
        dist[i] = one(pref[3 * (size_t)i], pref[3 * (size_t)i + 1], pref[3 * (size_t)i + 2], tmp[3 * (size_t)i], tmp[3 * (size_t)i + 1], tmp[3 * (size_t)i + 2]);
      }
      cnt = __reduce_add_sync(0xffffffffu, cnt); nin = __reduce_add_sync(0xffffffffu, nin);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
      if (lane == 0 && (cnt | nin)) { atomicAdd(&s_cnt2[0], cnt); atomicAdd(&s_cnt2[1], nin); atomicAdd(&s_apx, part); }
      __syncthreads();
    };
    // second half: warp 0 sums dist[] in order, warp 1 stages it through the ring; with `search`, the warps 2.. look up the
    // nearest reference point of every model point meanwhile (PointsCorresponding of the NEXT iteration, ICP.cpp:193-279)
    auto distance_chain = [&](bool search, float bound2, const float4* gp, const grid_info gi) {
      const int bar_threads = 64;
      if (warp == 0) {
        const long long tc = trc ? clock64() : 0;
        chain_consume<1, ICP_DCH, ICP_DNB, ICP_DCH, 0>(n_mod, s_stage, s_sum, bar_threads, trc ? trc + 13 : nullptr, trc ? trc + 16 : nullptr);
        if (trc && tid == 0) trc[14] += (unsigned long long)(clock64() - tc);
      } else if (warp == 1) {
        const int n_chunks = (n_mod + ICP_DCH - 1) / ICP_DCH;
        for (int c = 0; c < n_chunks; ++c) {
          const int b = c % ICP_DNB;
          float4 v[ICP_DCH / 128];
#pragma unroll
          for (int j = 0; j < ICP_DCH / 128; ++j) {
            const int i = c * ICP_DCH + 4 * (lane + 32 * j);
            v[j] = i < n_mod ? *reinterpret_cast<const float4*>(dist + i) : make_float4(0.f, 0.f, 0.f, 0.f);   // max_pts is a multiple of 4
          }
          if (c >= ICP_DNB) nb_sync(ICP_BAR_EMPTY(b), bar_threads);
#pragma unroll
          for (int j = 0; j < ICP_DCH / 128; ++j) *reinterpret_cast<float4*>(s_stage + (size_t)b * ICP_DCH + 4 * (lane + 32 * j)) = v[j];
          nb_arrive(ICP_BAR_FULL(b), bar_threads);
        }
      } else if (search) {
        for (int i = tid - 64; i < n_mod; i += ICP_NT - 64) {
          float best; int slot;
          nn_query(gp, s_cs, s_zr, gi, tmp[3 * (size_t)i], tmp[3 * (size_t)i + 1], tmp[3 * (size_t)i + 2], bound2, &best, &slot);
          nn_d2[i] = best; nn_slot[i] = slot;
        }
      }
      __syncthreads();
      if (tid == 0) {
        const int counter = s_cnt2[0], nin = s_cnt2[1];
        if (counter > 0) { s_dist_mean = __fdiv_rn(s_sum[0], (float)nin); s_ratio = __fdiv_rn((float)nin, (float)counter); }
        else { s_dist_mean = FLT_MAX; s_ratio = 0.f; }
      }
      __syncthreads();
    };

    float mnx = FLT_MAX, mny = FLT_MAX, mxx = -FLT_MAX, mxy = -FLT_MAX;   // x/y bounding box of the reference cloud (this thread's share)
    // ---- prepare: back-project the two crops, keep pixel pairs valid in both (order preserved), centroid shift ----
    if (A.hyps) {
      if (status == FL_OK) {
        const fl_icp_hyp& hy = A.hyps[h];
        const fl_rect_t rr = hy.rect_ref, rm = hy.rect_model;
        const uint16_t* __restrict__ mdepth = hy.model_depth;
        const int total = min(min(rr.width * rr.height, rm.width * rm.height), ws.max_pts);
        const float inv_fxr = __fdiv_rn(1.0f, A.Kr.fx), inv_fyr = __fdiv_rn(1.0f, A.Kr.fy);
        const float inv_fm = __fdiv_rn(1.0f, 608.0f);                // initInternalMat: fx = fy = 608, c = (320, 240) (common.cpp:358)
        // Order-preserving compaction with ONE block scan per 32k pixels: every WARP owns a block of consecutive pixels and walks it
        // 32 at a time (lane = pixel, so the depth loads and the point stores of a step are contiguous); pass 1 keeps one ballot per
        // step (lane j holds the ballot of step j), the warp totals are scanned across the CTA, pass 2 back-projects the kept pairs
        // and writes each at (warp base + kept pairs of the earlier steps + kept lanes below).  Validity depends on z alone.
        auto z_valid = [](uint16_t dv) { return dv != 0 && pt_valid(__fmul_rn(__fmul_rn((float)dv, (float)(1 / 1000.0)), 1000.0f)); };
        int n = 0;
        for (int base = 0; base < total; base += ICP_NT * 32) {
          const int rem = min(total - base, ICP_NT * 32);
          const int steps = ((rem + ICP_NWARPS - 1) / ICP_NWARPS + 31) >> 5;   // steps of 32 pixels per warp (<= 32)
          const int w0 = base + warp * steps * 32, w1 = min(w0 + steps * 32, base + rem);
          unsigned myb = 0;
          int wcount = 0;
          {
            int i = w0 + lane, ur = i % rr.width, vr = i / rr.width;
            for (int j0 = 0; j0 < steps; j0 += 8) {                   // eight steps at a time: their 16 loads are in flight together
              uint16_t dr[8], dm[8];
#pragma unroll
              for (int u = 0; u < 8; ++u) {
                const bool in = j0 + u < steps && i < w1;
                dr[u] = in ? A.ref_depth[(size_t)(rr.y + vr) * A.W + rr.x + ur] : (uint16_t)0;
                dm[u] = in ? mdepth[i] : (uint16_t)0;
                i += 32; ur += 32;
                while (ur >= rr.width) { ur -= rr.width; ++vr; }
              }
#pragma unroll
              for (int u = 0; u < 8; ++u) {
                const unsigned bal = __ballot_sync(0xffffffffu, z_valid(dr[u]) && z_valid(dm[u]));
                if (lane == j0 + u) myb = bal;
                wcount += __popc(bal);
              }
            }
          }
          int tot;
          int run = n + block_excl_scan(lane == 0 ? wcount : 0, s_warp, &tot);   // lane 0 of each warp carries the warp's total
          run = __shfl_sync(0xffffffffu, run, 0);
          {
            int i = w0 + lane, ur = i % rr.width, vr = i / rr.width, um = i % rm.width, vm = i / rm.width;
            for (int j = 0; j < steps; ++j) {
              const unsigned bal = __shfl_sync(0xffffffffu, myb, j);
              if ((bal >> lane) & 1u) {
                const int pos = run + __popc(bal & ((1u << lane) - 1u));
                const float3 a = backproject_mm(A.ref_depth[(size_t)(rr.y + vr) * A.W + rr.x + ur], rr.x + ur, rr.y + vr, inv_fxr, inv_fyr, A.Kr.cx, A.Kr.cy);
                const float3 b = backproject_mm(mdepth[i], rm.x + um, rm.y + vm, inv_fm, inv_fm, 320.0f, 240.0f);   // paired matToVec, common.cpp:382-405
                pref[3 * (size_t)pos] = a.x; pref[3 * (size_t)pos + 1] = a.y; pref[3 * (size_t)pos + 2] = a.z;
                tmp[3 * (size_t)pos] = b.x; tmp[3 * (size_t)pos + 1] = b.y; tmp[3 * (size_t)pos + 2] = b.z;
                mnx = fminf(mnx, a.x); mxx = fmaxf(mxx, a.x); mny = fminf(mny, a.y); mxy = fmaxf(mxy, a.y);
              }
              run += __popc(bal);
              i += 32; ur += 32; um += 32;
              while (ur >= rr.width) { ur -= rr.width; ++vr; }
              while (um >= rm.width) { um -= rm.width; ++vm; }
            }
          }
          n += tot;
        }
        n_ref = n_mod = n;
        __syncthreads();
        TR(0);
        chain_records(tmp, n, pref, n, 0);                          // getMean x2 (detection.cpp:165-166)
        TR(1);
        if (tid < 3) {
          const float mc = n > 0 ? __fdiv_rn(s_sum[tid], (float)n) : 0.f, rc = n > 0 ? __fdiv_rn(s_sum[3 + tid], (float)n) : 0.f;
          const float tt = __fsub_rn(rc, mc);                        // t_match_tmp = r_centroid - m_centroid (:177)
          s_tt[tid] = tt;
          s_tinit[tid] = __fadd_rn(tt, hy.t_match[tid]);             // t_init (:199)
        }
        __syncthreads();
        const float t0 = s_tt[0], t1 = s_tt[1], t2 = s_tt[2];
        auto shift = [&](float& x, float& y, float& z) {             // transformPoints(pts_mod, I, t_tmp) (:206), then copyPoints (ICP.cpp:667)
          if (pt_valid(z)) { x = __fadd_rn(x, t0); y = __fadd_rn(y, t1); z = __fadd_rn(z, t2); }
          if (!pt_valid(z)) { x = 0.f; y = 0.f; z = 0.f; }            // a point pushed beyond the validity range is dropped by the copy
        };
        for (int i4 = 4 * tid; i4 + 4 <= n; i4 += 4 * ICP_NT) {
          pts4 q = load_pts4(tmp + 3 * (size_t)i4);
#pragma unroll
          for (int k = 0; k < 4; ++k) shift(q.x[k], q.y[k], q.z[k]);
          store_pts4(tmp + 3 * (size_t)i4, q);
        }
        for (int i = (n & ~3) + tid; i < n; i += ICP_NT) shift(tmp[3 * (size_t)i], tmp[3 * (size_t)i + 1], tmp[3 * (size_t)i + 2]);
      }
    } else {
      n_ref = ws.n_ref[h]; n_mod = ws.n_mod[h];
    }
    __syncthreads();

    if (status != FL_OK || n_mod < 3 || n_ref < 3) {               // ICP.cpp:633-638: returns -1, R and T stay zero-initialised
      if (tid == 0) {
        fl_icp_result_t r;
        for (int k = 0; k < 9; ++k) r.R[k] = 0.f;
        for (int k = 0; k < 3; ++k) r.T[k] = 0.f;
        r.dist_mean = -1.f; r.inlier_ratio = 0.f; r.iterations = 0; r.n_points = n_mod; r.status = status;
        *res = r;
      }
      continue;
    }

    // ---- grid over the reference cloud (replaces the KD-tree build, ICP.cpp:650-659) ----
    const bool grid_in_smem = n_ref <= A.smem_pts;
    float4* gp = grid_in_smem ? s_gp : ws.grid_pts + (size_t)h * ws.max_pts;
    if (!A.hyps) {                                                  // cloud mode: the bounding box was not collected while pairing
      for (int i = tid; i < n_ref; i += ICP_NT) {
        const float x = pref[3 * (size_t)i], y = pref[3 * (size_t)i + 1], z = pref[3 * (size_t)i + 2];
        if (isfinite(x) && isfinite(y) && isfinite(z)) { mnx = fminf(mnx, x); mxx = fmaxf(mxx, x); mny = fminf(mny, y); mxy = fmaxf(mxy, y); }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o)); mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o));
      mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o)); mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
    }
    if (lane == 0) { s_red[warp * 4] = mnx; s_red[warp * 4 + 1] = mny; s_red[warp * 4 + 2] = mxx; s_red[warp * 4 + 3] = mxy; }
    for (int i = tid; i < FL_ICP_CELLS; i += ICP_NT) s_cur[i] = 0;
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < ICP_NWARPS; ++w) {
        mnx = fminf(mnx, s_red[w * 4]); mny = fminf(mny, s_red[w * 4 + 1]); mxx = fmaxf(mxx, s_red[w * 4 + 2]); mxy = fmaxf(mxy, s_red[w * 4 + 3]);
      }
      const float ext = fmaxf(fmaxf(mxx - mnx, mxy - mny), 1e-3f);
      grid_info gi; gi.minx = mnx; gi.miny = mny; gi.cell = ext / (float)FL_ICP_GRID * 1.0001f; gi.inv_cell = 1.0f / gi.cell;
      s_gi = gi;
      for (int k = 0; k < 9; ++k) s_R[k] = (k % 4 == 0) ? 1.f : 0.f;   // R = I, T = 0 (ICP.cpp:644-645)
      for (int k = 0; k < 3; ++k) s_T[k] = 0.f;
    }
    __syncthreads();
    grid_info gi = s_gi;
    for (int i = tid; i < n_ref; i += ICP_NT) {
      const float x = pref[3 * (size_t)i], y = pref[3 * (size_t)i + 1], z = pref[3 * (size_t)i + 2];
      if (isfinite(x) && isfinite(y) && isfinite(z)) atomicAdd(&s_cur[cell_of(y, gi.miny, gi.inv_cell) * FL_ICP_GRID + cell_of(x, gi.minx, gi.inv_cell)], 1);
    }
    __syncthreads();
    {   // exclusive scan of the 4,096 counters: 4 per thread
      constexpr int PER = FL_ICP_CELLS / ICP_NT;
      int loc[PER], sum = 0;
#pragma unroll
      for (int k = 0; k < PER; ++k) { loc[k] = s_cur[tid * PER + k]; sum += loc[k]; }
      int tot;
      int base = block_excl_scan(sum, s_warp, &tot);
#pragma unroll
      for (int k = 0; k < PER; ++k) { s_cs[tid * PER + k] = base; s_cur[tid * PER + k] = base; base += loc[k]; }
      if (tid == 0) s_cs[FL_ICP_CELLS] = tot;
    }
    __syncthreads();
    for (int i = tid; i < n_ref; i += ICP_NT) {
      const float x = pref[3 * (size_t)i], y = pref[3 * (size_t)i + 1], z = pref[3 * (size_t)i + 2];
      if (isfinite(x) && isfinite(y) && isfinite(z)) {
        const int slot = atomicAdd(&s_cur[cell_of(y, gi.miny, gi.inv_cell) * FL_ICP_GRID + cell_of(x, gi.minx, gi.inv_cell)], 1);
        gp[slot] = make_float4(x, y, z, __int_as_float(i));
      }
    }
    // ---- copyPoints(pts_model, pts_model_tmp) (ICP.cpp:667): invalid points become (0,0,0) (detection mode: done with the shift) ----
    if (!A.hyps)
      for (int i = tid; i < n_mod; i += ICP_NT)
        if (!pt_valid(tmp[3 * (size_t)i + 2])) { tmp[3 * (size_t)i] = 0.f; tmp[3 * (size_t)i + 1] = 0.f; tmp[3 * (size_t)i + 2] = 0.f; }
    __syncthreads();
    {   // per-cell z range, quantised to 16 bits over the cloud's z extent with one step of slack on either side (4 cells per thread)
      constexpr int PER = FL_ICP_CELLS / ICP_NT;
      float zl[PER], zh[PER], gl = FLT_MAX, gh = -FLT_MAX;
#pragma unroll
      for (int k = 0; k < PER; ++k) {
        zl[k] = FLT_MAX; zh[k] = -FLT_MAX;
        for (int p = s_cs[tid * PER + k]; p < s_cs[tid * PER + k + 1]; ++p) { const float z = gp[p].z; zl[k] = fminf(zl[k], z); zh[k] = fmaxf(zh[k], z); }
        gl = fminf(gl, zl[k]); gh = fmaxf(gh, zh[k]);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) { gl = fminf(gl, __shfl_xor_sync(0xffffffffu, gl, o)); gh = fmaxf(gh, __shfl_xor_sync(0xffffffffu, gh, o)); }
      if (lane == 0) { s_red[warp * 4] = gl; s_red[warp * 4 + 1] = gh; }
      __syncthreads();
      gl = s_red[0]; gh = s_red[1];
      for (int w = 1; w < ICP_NWARPS; ++w) { gl = fminf(gl, s_red[w * 4]); gh = fmaxf(gh, s_red[w * 4 + 1]); }
      const float zstep = fmaxf((gh - gl) / 65000.f, 1e-6f), inv_step = 1.0f / zstep;
      if (tid == 0) { s_gi.z0 = gl; s_gi.zstep = zstep; }
#pragma unroll
      for (int k = 0; k < PER; ++k) {
        unsigned q = 0xFFFFu;                                          // empty cell (never opened: its run is empty)
        if (zl[k] <= zh[k]) {
          const int lo = max((int)floorf((zl[k] - gl) * inv_step) - 1, 0), hi = min((int)ceilf((zh[k] - gl) * inv_step) + 1, 65535);
          q = (unsigned)lo | ((unsigned)hi << 16);
        }
        s_zr[tid * PER + k] = q;
      }
    }
    __syncthreads();
    gi = s_gi;                                                      // now with the z quantisation
    TR(2);

    distance_fill(FLT_MAX, false);                                  // ICP.cpp:670
    TR(3);
    distance_chain(false, 0.f, gp, gi);
    TR(4);
    if (tid == 0) { s_dist_diff = FLT_MAX; s_iter = 0; }
    __syncthreads();
    bool have_nn = false;                                           // nn_slot / nn_d2 hold the neighbours of the current tmp[]

    while (true) {
      if (tid == 0) s_go = (s_dist_mean > A.prm.dist_mean_thr && s_dist_diff > A.prm.dist_diff_thr && s_iter < A.prm.icp_it_thr) ? 1 : 0;   // :684
      __syncthreads();
      if (!s_go) break;
      if (tid == 0) ++s_iter;
      __syncthreads();
      const int iter = s_iter;
      int n_cm, n_cr;
      const float* cm = cor_m; const float* cr = cor_r;
      if (iter == 1) {                                              // :700-704: copies with invalid -> 0
        // pts_model_tmp holds no invalid point any more (copyPoints zeroed them), so its copy IS tmp[]; the reference cloud of a
        // detection() call holds only valid points too; a caller-supplied cloud may not, so cloud mode makes the copy
        cm = tmp; cr = pref;
        if (!A.hyps) {
          for (int i = tid; i < n_ref; i += ICP_NT) {
            const bool v = pt_valid(pref[3 * (size_t)i + 2]);
            cor_r[3 * (size_t)i] = v ? pref[3 * (size_t)i] : 0.f; cor_r[3 * (size_t)i + 1] = v ? pref[3 * (size_t)i + 1] : 0.f; cor_r[3 * (size_t)i + 2] = v ? pref[3 * (size_t)i + 2] : 0.f;
          }
          cr = cor_r;
        }
        n_cm = n_mod; n_cr = n_ref;
      } else {                                                      // :708 -> PointsCorresponding :193-279
        const float thr = __fmul_rn(3.f, s_dist_mean);
        if (!have_nn) {                                             // (only when the overlapped search could not be used)
          if (trc && tid == 0) trc[17] += 1;
          for (int i = tid; i < n_mod; i += ICP_NT) {
            float best; int slot;
            nn_query(gp, s_cs, s_zr, gi, tmp[3 * (size_t)i], tmp[3 * (size_t)i + 1], tmp[3 * (size_t)i + 2], thr, &best, &slot);
            nn_d2[i] = best; nn_slot[i] = slot;
          }
          __syncthreads();
        }
        // order-preserving compaction of the accepted pairs, warp-aggregated like the pairing above (coalesced loads and stores)
        int n = 0;
        for (int base = 0; base < n_mod; base += ICP_NT * 32) {
          const int rem = min(n_mod - base, ICP_NT * 32);
          const int steps = ((rem + ICP_NWARPS - 1) / ICP_NWARPS + 31) >> 5;
          const int w0 = base + warp * steps * 32, w1 = min(w0 + steps * 32, base + rem);
          unsigned myb = 0;
          int wcount = 0;
          for (int j0 = 0; j0 < steps; j0 += 8) {
            int sl[8]; float dd[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const int i = w0 + (j0 + u) * 32 + lane;
              const bool in = j0 + u < steps && i < w1;
              sl[u] = in ? nn_slot[i] : -1; dd[u] = in ? nn_d2[i] : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const unsigned bal = __ballot_sync(0xffffffffu, sl[u] >= 0 && dd[u] <= thr);   // squared distance against un-squared 3*dist_mean (:268)
              if (lane == j0 + u) myb = bal;
              wcount += __popc(bal);
            }
          }
          int tot;
          int run = n + block_excl_scan(lane == 0 ? wcount : 0, s_warp, &tot);
          run = __shfl_sync(0xffffffffu, run, 0);
          for (int j = 0; j < steps; ++j) {
            const unsigned bal = __shfl_sync(0xffffffffu, myb, j);
            const int i = w0 + j * 32 + lane;
            if ((bal >> lane) & 1u) {
              const int pos = run + __popc(bal & ((1u << lane) - 1u));
              const float4 r = gp[nn_slot[i]];
              cor_m[3 * (size_t)pos] = tmp[3 * (size_t)i]; cor_m[3 * (size_t)pos + 1] = tmp[3 * (size_t)i + 1]; cor_m[3 * (size_t)pos + 2] = tmp[3 * (size_t)i + 2];
              cor_r[3 * (size_t)pos] = r.x; cor_r[3 * (size_t)pos + 1] = r.y; cor_r[3 * (size_t)pos + 2] = r.z;
            }
            run += __popc(bal);
          }
          n += tot;
        }
        n_cm = n_cr = n;
      }
      __syncthreads();
      TR(5);
      if (n_cr < 3 || n_cm < 3) {                                   // :711-715
        if (tid == 0) s_iter = A.prm.icp_it_thr;
        __syncthreads();
        continue;
      }
      chain_records(cm, n_cm, cr, n_cr, n_cm);                      // centroids + covariance chains (:722-735)
      TR(6);
      if (tid == 0) {
        float mc[3], rc[3], cov[9], rm[3];
        for (int k = 0; k < 3; ++k) { mc[k] = __fdiv_rn(s_sum[k], (float)n_cm); rc[k] = __fdiv_rn(s_sum[3 + k], (float)n_cr); }
        for (int k = 0; k < 9; ++k) cov[k] = s_sum[6 + k];
        svd3_rot(cov, s_Ropt);                                      // :741-744
        matvec3(s_Ropt, mc, rm);
        int fin = 1;
        for (int k = 0; k < 3; ++k) { s_Topt[k] = __fsub_rn(rc[k], rm[k]); if (!isfinite(s_Topt[k])) fin = 0; }   // :747
        for (int k = 0; k < 9; ++k) if (!isfinite(s_Ropt[k])) fin = 0;
        s_finite = fin;                                             // :748-749
      }
      __syncthreads();
      TR(7);
      if (!s_finite) continue;                                      // (tmp[] unchanged: the neighbours found for it stay valid)
      TR(8);
      const float old_mean = s_dist_mean;
      distance_fill(__fmul_rn(3.f, old_mean), true);                // transformPoints (:756) fused with the distances (:778-780): one pass over the clouds
      // The neighbour search of the next iteration runs under the distance sum, so its radius cannot use the exact new
      // dist_mean yet: it uses an unordered (parallel) sum of the same distances, padded by 0.1 %; if the exact accept radius
      // 3 * dist_mean turns out larger after all (it cannot, short of pathological rounding), the search is simply redone.
      // The same estimate predicts whether the loop will go on at all (:684); a hypothesis that is about to stop is not searched
      // for (if the exact sums disagree with the prediction, the search is done afterwards instead).
      const float apx_mean = __fdiv_rn(s_apx, (float)max(s_cnt2[1], 1));
      const bool more = iter < A.prm.icp_it_thr && apx_mean > A.prm.dist_mean_thr * 0.999f &&
                        (old_mean - apx_mean) > A.prm.dist_diff_thr - 1e-3f * fabsf(old_mean);
      const float bound2 = __fmul_rn(__fmul_rn(3.f, apx_mean), 1.001f);
      TR(3);
      distance_chain(more, bound2, gp, gi);
      TR(4);
      have_nn = more && (__fmul_rn(3.f, s_dist_mean) <= bound2);
      if (tid == 0) {
        s_dist_diff = __fsub_rn(old_mean, s_dist_mean);
        float nT[3], nR[9];
        matvec3(s_Ropt, s_T, nT);                                   // :793-797
        for (int k = 0; k < 3; ++k) s_T[k] = __fadd_rn(nT[k], s_Topt[k]);
        matmul3(s_Ropt, s_R, nR);
        for (int k = 0; k < 9; ++k) s_R[k] = nR[k];
      }
      __syncthreads();
    }

    if (tid == 0) {
      fl_icp_result_t r;
      if (A.hyps) {                                                 // detection.cpp:232-234
        float ti[3] = {s_tinit[0], s_tinit[1], s_tinit[2]}, rt[3];
        matvec3(s_R, ti, rt);
        for (int k = 0; k < 3; ++k) r.T[k] = __fadd_rn(rt[k], s_T[k]);
        matmul3(s_R, A.hyps[h].r_match, r.R);
      } else {
        for (int k = 0; k < 9; ++k) r.R[k] = s_R[k];
        for (int k = 0; k < 3; ++k) r.T[k] = s_T[k];
      }
      r.dist_mean = s_dist_mean; r.inlier_ratio = s_ratio; r.iterations = s_iter; r.n_points = n_mod; r.status = FL_OK;
      *res = r;
      if (trc) { trc[9] = (unsigned long long)(clock64() - t_begin); trc[10] = (unsigned long long)s_iter; trc[11] = (unsigned long long)n_mod; }
    }
    __syncthreads();
  }
}

// dynamic shared memory of k_icp_fused for a batch whose largest cloud has max_pts points (0 grid points if they do not fit)
static int icp_smem_plan(int max_pts, int* smem_pts) {
  const int fixed = (FL_ICP_CELLS + 4) * 4 + FL_ICP_CELLS * 4 + ICP_STAGE_FLOATS * 4;
  const int avail = 227 * 1024 - 2048 - fixed;                      // 2 KB: the kernel's static shared memory
  *smem_pts = (max_pts * 16 <= avail) ? ((max_pts + 3) & ~3) : 0;
  return fixed + *smem_pts * 16;
}

// the shared-memory opt-in of k_icp_fused on the current device, for a launch with `smem` dynamic bytes
static cudaError_t icp_opt_in(int smem) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= FL_MAX_DEVICES) return cudaErrorInvalidDevice;
  static std::mutex mu;                                             // the opt-in belongs to the (device, function) pair
  static int configured[FL_MAX_DEVICES];
  std::lock_guard<std::mutex> lk(mu);
  if (smem > configured[dev]) {
    if ((e = cudaFuncSetAttribute(k_icp_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) != cudaSuccess) return e;
    configured[dev] = smem;
  }
  return cudaSuccess;
}

int fl_icp_preload(int max_pts) {
  int smem_pts = 0;
  cudaFuncAttributes a;
  FL_CUDA(cudaFuncGetAttributes(&a, k_icp_fused));
  FL_CUDA(icp_opt_in(icp_smem_plan(max_pts, &smem_pts)));
  return FL_OK;
}

int fl_launch_icp(fl_icp_ws ws, fl_icp_params_t p, const fl_icp_hyp* hyps_or_null, const uint16_t* ref_depth, int W, int H, fl_intrinsics_t K_ref,
                  fl_icp_result_t* results, int* ticket, unsigned long long* trace, int n_sm, cudaStream_t s) {
  if (ws.n_hyp <= 0) return 0;
  fl_icp_args A;
  A.ws = ws; A.prm = p; A.hyps = hyps_or_null; A.ref_depth = ref_depth; A.W = W; A.H = H; A.Kr = K_ref; A.results = results; A.ticket = ticket; A.trace = trace;
  const int smem = icp_smem_plan(ws.max_pts, &A.smem_pts);
  if (icp_opt_in(smem) != cudaSuccess) return -1;
  if (cudaMemsetAsync(ticket, 0, sizeof(int), s) != cudaSuccess) return -1;
  k_icp_fused<<<min(ws.n_hyp, n_sm), ICP_NT, smem, s>>>(A);
  return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

// ------------------------------------------------------------------------------------------------
// K12 greedy NMS (order dependent, n is small): one thread walks the list exactly like NMS.cpp:6-39
// ------------------------------------------------------------------------------------------------
__global__ void k_nms(const float* __restrict__ t3, const int32_t* __restrict__ n_model, const float* __restrict__ icp_dist, int n, float th,
                      int32_t* __restrict__ out_idx, int32_t* __restrict__ out_count, uint8_t* __restrict__ done) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  *out_count = fl_nms_greedy(t3, n_model, icp_dist, n, th, out_idx, done);
}

void fl_launch_nms(const float* t3, const int32_t* n_model, const float* icp_dist, int n, float th, int32_t* out_idx, int32_t* out_count,
                   cudaStream_t s) {
  // scratch "done" flags live after out_idx (caller allocates n ints + n bytes)
  k_nms<<<1, 32, 0, s>>>(t3, n_model, icp_dist, n, th, out_idx, out_count, reinterpret_cast<uint8_t*>(out_idx + n));
}
