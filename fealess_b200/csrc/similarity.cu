// LINE-MOD template matching on sm_100a: global similarity at the coarsest pyramid level with fused threshold ->
// candidate emission, local 16x16 refinement up the pyramid, and the final sort + duplicate pruning.
//
// Reference semantics (paths relative to /root/reference; SURVEY.md appendix A.3-A.5):
//   accessLinearMemory linemod/linemod.cpp:1094-1117   similarity :1130-1214   similarityLocal :1226-1300
//   addSimilarities :1322-1338   matchClass :1451-1577   Match ordering linemod/linemod.hpp:262-274, sort/unique :1437-1439
//
// Byte-lane arithmetic: a template has <= 63 features per modality (CV_Assert :1137) and a response is <= 4, so four
// packed u8 sums in one 32-bit register never carry across lanes (63*4 = 252): one IADD adds four cells.
#include "fl_internal.cuh"
#include <mutex>

// ------------------------------------------------------------------------------------------------
// per-geometry feature packing (runs once per frame size, not per frame)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pack_features(fl_tdb db, const fl_level_geom* __restrict__ geom, int n_entries) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;       // one thread per (template, level, modality) entry
  if (e >= n_entries) return;
  const fl_template_hdr_t h = db.hdr[e];
  const int level = (e / db.M) % db.L;
  const fl_level_geom g = geom[level];
  for (int k = 0; k < h.feature_count; ++k) {
    const fl_feature_t f = db.feat[h.feature_begin + k];
    fl_pfeat p;
    p.x = (int16_t)max(min(f.x, 32767), -32768);
    p.y = (int16_t)max(min(f.y, 32767), -32768);
    if (f.x < 0 || f.y < 0 || f.x >= g.W || f.y >= g.H) p.lm_off = FL_SKIP;          // :1179
    else p.lm_off = (uint32_t)((size_t)f.label * g.label_stride + (size_t)((f.y % g.T) * g.T + (f.x % g.T)) * g.cells +
                               (size_t)(f.y / g.T) * g.Wd + f.x / g.T);
    db.pfeat[h.feature_begin + k] = p;
  }
}

void fl_launch_pack_features(fl_tdb db, const fl_level_geom* d_geom, int n_features_total, cudaStream_t s) {
  (void)n_features_total;
  int n = db.n_templates * db.L * db.M;
  if (n > 0) k_pack_features<<<(n + 255) / 256, 256, 0, s>>>(db, d_geom, n);
}

// refinement records (fl_tdb::rrec): one thread per (template, level < L-1, modality slot)
__global__ void __launch_bounds__(256) k_pack_refine_records(fl_tdb db, const fl_level_geom* __restrict__ geom) {
  const int rec = blockIdx.x;                            // (t, level)
  const int t = rec / (db.L - 1), level = rec - t * (db.L - 1);
  const fl_level_geom g = geom[level];
  const fl_template_hdr_t* hdr = db.hdr + ((size_t)t * db.L + level) * db.M;
  uint8_t* out = db.rrec + (size_t)rec * db.rrec_bytes;
  const int gt = threadIdx.x, m = gt >> 6, k = gt & 63;
  if (gt == 0) {
    int nf = 0;
    int fc[4] = {0, 0, 0, 0};
    for (int mm = 0; mm < db.M; ++mm) { fc[mm] = hdr[mm].feature_count; nf += fc[mm]; }
    int* o = reinterpret_cast<int*>(out);
    o[0] = hdr[0].width; o[1] = hdr[0].height; o[2] = nf; o[3] = 0; o[4] = fc[0]; o[5] = fc[1]; o[6] = fc[2]; o[7] = fc[3];
  }
  if (m < db.M) {
    fl_pfeat p;
    p.lm_off = 0xFFFFFFFFu; p.x = -32768; p.y = -32768;  // empty slot: never inside the image
    if (k < hdr[m].feature_count) {
      const fl_feature_t f = db.feat[hdr[m].feature_begin + k];
      p.x = (int16_t)max(min(f.x, 32767), -32768);
      p.y = (int16_t)max(min(f.y, 32767), -32768);
      if (f.x < 0 || f.y < 0 || f.x >= g.W || f.y >= g.H) p.lm_off = FL_RSKIP | (uint32_t)f.label;
      else p.lm_off = (uint32_t)((size_t)f.label * g.label_stride + (size_t)((f.y % g.T) * g.T + (f.x % g.T)) * g.cells +
                                 (size_t)(f.y / g.T) * g.Wd + f.x / g.T);
    }
    reinterpret_cast<fl_pfeat*>(out + 32)[gt] = p;
  }
}
void fl_launch_pack_refine_records(fl_tdb db, const fl_level_geom* d_geom, cudaStream_t s) {
  const int n = db.n_templates * (db.L - 1);
  if (n > 0 && db.rrec) k_pack_refine_records<<<n, 256, 0, s>>>(db, d_geom);
}

// unaligned 4-byte window at byte offset a of a 4-byte-aligned buffer
__device__ __forceinline__ uint32_t load_u8x4(const uint8_t* __restrict__ base, uint32_t a) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(base) + (a >> 2);
  uint32_t lo = __ldg(w), hi = __ldg(w + 1);
  return __funnelshift_r(lo, hi, (a & 3) * 8);
}

__device__ __forceinline__ int raw_threshold_of(int nf, float threshold) {
  // int(2*nf + (threshold/100)*(2*nf) + 0.5f) in fp32, truncation (:1487)
  return (int)__fadd_rn(__fadd_rn((float)(2 * nf), __fmul_rn(__fdiv_rn(threshold, 100.f), (float)(2 * nf))), 0.5f);
}

// ------------------------------------------------------------------------------------------------
// K6 (baseline variant): one CTA per template, one thread per group of 4 cells, responses read through L1/L2.
// ------------------------------------------------------------------------------------------------
#define SG_THREADS 128

template <bool kDebug>
__global__ void __launch_bounds__(SG_THREADS) k_similarity_global(fl_tdb db, fl_level_geom g, const uint8_t* __restrict__ lm_level,
                                                                  float threshold, fl_match_t* __restrict__ cand, int cap,
                                                                  int* __restrict__ d_count, int t_debug, uint16_t* __restrict__ dbg) {
  fl_grid_dep_wait();
  fl_grid_dep_launch();
  const int t = kDebug ? t_debug : blockIdx.x;
  const int cls = db.class_of[t];
  if (!kDebug && !db.class_enabled[cls]) return;
  const int level = db.L - 1;
  const fl_template_hdr_t* hdr = db.hdr + ((size_t)t * db.L + level) * db.M;
  const int cells = g.cells;
  int nf = 0;
  for (int m = 0; m < db.M; ++m) nf += hdr[m].feature_count;
  const int raw_thr = raw_threshold_of(nf, threshold);
  const int off = g.T / 2 + (g.T % 2 - 1);
  const int ngroups = (cells + 3) / 4;
  for (int grp = threadIdx.x; grp < ngroups; grp += SG_THREADS) {
    uint32_t tot_lo = 0, tot_hi = 0;   // u16 x 2 each: cells (0,1) and (2,3)
    for (int m = 0; m < db.M; ++m) {
      const fl_template_hdr_t h = hdr[m];
      const int wf = (h.width - 1) / g.T + 1, hf = (h.height - 1) / g.T + 1;          // :1145-1146
      int tp = (g.Hd - hf) * g.Wd + (g.Wd - wf) + 1;                                  // template_positions :1155
      tp = min(tp, cells);
      const int j0 = grp * 4;
      if (j0 >= tp) continue;                                                          // cells beyond stay 0
      const uint8_t* lm_mod = lm_level + (size_t)m * g.mod_stride;
      const fl_pfeat* pf = db.pfeat + h.feature_begin;
      uint32_t acc = 0;
      for (int k = 0; k < h.feature_count; ++k) {
        uint32_t o = __ldg(&pf[k].lm_off);
        if (o == FL_SKIP) continue;
        acc += load_u8x4(lm_mod, o + j0);                                              // four wrapping u8 adds (:1195)
      }
      if (j0 + 4 > tp) acc &= 0xFFFFFFFFu >> (8 * (j0 + 4 - tp));                      // mask lanes >= tp
      tot_lo += (acc & 0xFF) | ((acc & 0xFF00) << 8);                                  // widen to u16 lanes (:1322-1338)
      tot_hi += ((acc >> 16) & 0xFF) | ((acc >> 24) << 16);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      int j = grp * 4 + k;
      if (j >= cells) break;
      int raw = (k < 2 ? tot_lo >> (16 * k) : tot_hi >> (16 * (k - 2))) & 0xFFFF;
      if (kDebug) { dbg[j] = (uint16_t)raw; continue; }
      if (raw > raw_thr) {                                                             // :1497-1504
        int r = j / g.Wd, c = j - r * g.Wd;
        int slot = atomicAdd(d_count, 1);
        if (slot < cap) {
          fl_match_t mt;
          mt.x = c * g.T + off; mt.y = r * g.T + off;
          mt.similarity = __fadd_rn(__fdiv_rn(__fmul_rn((float)raw, 100.f), (float)(4 * nf)), 0.5f);
          // candidates carry the handle-local template index until the last stage rewrites it to the per-class
          // template_id (which may be a global id when this handle holds only a shard of the templates)
          mt.class_idx = cls; mt.template_id = db.L == 1 ? db.tid_of[t] : t;
          cand[slot] = mt;
        }
      }
    }
  }
}

void fl_launch_similarity_global(fl_tdb db, fl_level_geom g, const uint8_t* lm_level, float threshold, fl_match_t* cand, int cap,
                                 int* d_count, cudaStream_t s) {
  if (db.n_templates > 0)
    fl_launch(k_similarity_global<false>, dim3(db.n_templates), dim3(SG_THREADS), 0, s, db, g, lm_level, threshold, cand, cap, d_count, 0, (uint16_t*)nullptr);
}
void fl_launch_similarity_debug(fl_tdb db, fl_level_geom g, const uint8_t* lm_level, int t, uint16_t* out, cudaStream_t s) {
  k_similarity_global<true><<<1, SG_THREADS, 0, s>>>(db, g, lm_level, 0.f, nullptr, 0, nullptr, t, out);
}

// ------------------------------------------------------------------------------------------------
// K7 local refinement of every candidate at one finer level: 16x16 patch of total similarity, first maximum wins.
// One CTA of 64 threads per candidate: thread = (patch row, 4-cell column group).
// ------------------------------------------------------------------------------------------------
#define RF_THREADS 256       // 4 feature groups x 64 (16 patch rows x 4 column groups of 4 cells)
#define RF_MAXF (FL_MAX_MODALITIES * 63)

struct fl_refine_smem {                        // per group of RF_THREADS threads
  uint32_t off[FL_MAX_MODALITIES * 64];        // byte offset of every feature slot's window origin inside the level's linear memories, or FL_SKIP
  int mbeg[FL_MAX_MODALITIES + 1], cnt[FL_MAX_MODALITIES];
  uint32_t part[3][64][2];
  uint32_t best[2];
  fl_match_t mt;
};

__device__ __forceinline__ void group_sync(int bar_id) { asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(RF_THREADS) : "memory"); }

// One level of local refinement of one candidate by a group of RF_THREADS threads (gt = thread index inside the group,
// bar_id = the group's named barrier).  mt is the candidate at level + 1 on entry (template_id = handle-local template index) and
// at `level` on return; template_id = -1 marks it dropped (:1570-1572).  Group-uniform control flow.
__device__ __forceinline__ void refine_level_group(const fl_tdb& db, const fl_level_geom& g, int level, const uint8_t* __restrict__ lm_level,
                                                   float threshold, fl_match_t& mt, fl_refine_smem& sm, int gt, int bar_id) {
  const int fgrp = gt >> 6, cell = gt & 63;
  const int row = cell >> 2, cg = cell & 3;
  const int T = g.T, border = 8 * T;
  const int t = mt.template_id;                                    // handle-local template index (see k_similarity_global)
  // the candidate's refinement record: header and this thread's feature slot are independent loads (one round trip)
  const uint8_t* rec = db.rrec + ((size_t)t * (db.L - 1) + level) * db.rrec_bytes;
  const int4 h0 = __ldg(reinterpret_cast<const int4*>(rec));       // width, height, n_features
  const int4 h1 = __ldg(reinterpret_cast<const int4*>(rec) + 1);   // features per modality
  fl_pfeat p; p.lm_off = 0xFFFFFFFFu; p.x = -32768; p.y = -32768;
  if (gt < db.M * 64) p = reinterpret_cast<const fl_pfeat*>(rec + 32)[gt];
  int x = mt.x * 2 + 1, y = mt.y * 2 + 1;                          // :1525-1534
  x = max(x, border); y = max(y, border);
  x = min(x, g.W - h0.x - border);
  y = min(y, g.H - h0.y - border);
  const int ox = (x / T - 8) * T, oy = (y / T - 8) * T;            // :1240-1241 (C division truncates towards zero)
  const int delta = (oy / T) * g.Wd + ox / T;
  // stage 1: one thread per feature slot resolves the feature's window origin, so that stage 2 issues nothing but
  // independent linear-memory loads
  const int nf = h0.z;
  {
    const int m = gt >> 6;
    const int fx = p.x + ox, fy = p.y + oy;
    uint32_t o = FL_SKIP;
    if (fx >= 0 && fy >= 0 && fx < g.W && fy < g.H) {              // :1257
      // the packed offset was computed for (x, y); shifting by a multiple of T moves only the cell index
      if ((p.lm_off & FL_RSKIP) == FL_RSKIP)                       // outside the image unshifted, inside when shifted
        o = (uint32_t)((size_t)(p.lm_off & 15u) * g.label_stride +
                       (size_t)((p.y % T + T) % T * T + (p.x % T + T) % T) * g.cells + (size_t)(fy / T) * g.Wd + fx / T);
      else
        o = (uint32_t)((int)p.lm_off + delta);
      o += (uint32_t)((size_t)m * g.mod_stride);
    }
    sm.off[gt] = o;
    if (gt <= db.M) sm.mbeg[gt] = gt * 64;                         // fixed 64 slots per modality
    if (gt < 4) sm.cnt[gt] = gt == 0 ? h1.x : (gt == 1 ? h1.y : (gt == 2 ? h1.z : h1.w));
  }
  group_sync(bar_id);
  // stage 2: 16x16 patch, thread = (feature group, patch row, 4-cell column group); u8 lanes per modality (<= 63 x 4)
  const uint32_t cell_off = (uint32_t)(row * g.Wd + cg * 4);
  uint32_t tot_lo = 0, tot_hi = 0;
  for (int m = 0; m < db.M; ++m) {
    uint32_t acc = 0;
    const int k1 = sm.mbeg[m] + sm.cnt[m];
    // <= 63 features per modality (:1231) = <= 16 per feature group: all loads of a modality are issued before the first
    // add (one L2 round trip instead of one per unroll step)
    for (int k0 = sm.mbeg[m] + fgrp; k0 < k1; k0 += 64) {
      uint32_t lo[16], hi[16], sh[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const int k = k0 + 4 * u;
        const uint32_t o = k < k1 ? sm.off[k] : FL_SKIP;
        const uint32_t a = o + cell_off;
        sh[u] = (a & 3) * 8;
        lo[u] = hi[u] = 0;
        if (o != FL_SKIP) {
          const uint32_t* w = reinterpret_cast<const uint32_t*>(lm_level) + (a >> 2);
          lo[u] = __ldg(w); hi[u] = __ldg(w + 1);
        }
      }
#pragma unroll
      for (int u = 0; u < 16; ++u) acc += __funnelshift_r(lo[u], hi[u], sh[u]);
    }
    tot_lo += (acc & 0xFF) | ((acc & 0xFF00) << 8);
    tot_hi += ((acc >> 16) & 0xFF) | ((acc >> 24) << 16);
  }
  if (fgrp > 0) { sm.part[fgrp - 1][cell][0] = tot_lo; sm.part[fgrp - 1][cell][1] = tot_hi; }
  group_sync(bar_id);
  if (fgrp == 0) {
#pragma unroll
    for (int gq = 0; gq < 3; ++gq) { tot_lo += sm.part[gq][cell][0]; tot_hi += sm.part[gq][cell][1]; }   // u16 lanes
    // first maximum in row-major order: key = score << 8 | (255 - index); all-zero patch -> best 0 at (-1,-1) (:1547-1562)
    uint32_t key = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      uint32_t sc = (k < 2 ? tot_lo >> (16 * k) : tot_hi >> (16 * (k - 2))) & 0xFFFF;
      uint32_t idx = row * 16 + cg * 4 + k;
      uint32_t kk = (sc << 8) | (255 - idx);
      if (sc > 0 && kk > key) key = kk;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) key = max(key, __shfl_xor_sync(0xffffffffu, key, o));
    if ((gt & 31) == 0) sm.best[gt >> 5] = key;
  }
  group_sync(bar_id);
  if (gt == 0) {
    uint32_t kb = max(sm.best[0], sm.best[1]);
    int best = (int)(kb >> 8), br = -1, bc = -1;
    if (best > 0) { int idx = 255 - (int)(kb & 255); br = idx >> 4; bc = idx & 15; }
    const int off = T / 2 + (T % 2 - 1);
    fl_match_t r = mt;
    r.x = (x / T - 8 + bc) * T + off;                              // :1564-1566
    r.y = (y / T - 8 + br) * T + off;
    r.similarity = __fdiv_rn(__fmul_rn((float)best, 100.f), (float)(4 * nf));
    if (r.similarity < threshold) r.template_id = -1;              // mark dropped (remove_if :1570)
    sm.mt = r;
  }
  group_sync(bar_id);
  mt = sm.mt;
  group_sync(bar_id);                                              // sm is free for the next level / candidate
}

__global__ void __launch_bounds__(RF_THREADS) k_refine_level(fl_tdb db, fl_level_geom g, int level, const uint8_t* __restrict__ lm_level,
                                                             float threshold, fl_match_t* __restrict__ cand, int cap,
                                                             const int* __restrict__ d_count) {
  fl_grid_dep_wait();
  fl_grid_dep_launch();
  __shared__ fl_refine_smem sm;
  const int n = min(*d_count, cap);
  for (int ci = blockIdx.x; ci < n; ci += gridDim.x) {
    fl_match_t mt = cand[ci];
    if (mt.template_id < 0) continue;                              // dropped at a coarser level (:1570-1572)
    const int t = mt.template_id;
    const int final_id = (threadIdx.x == 0 && level == 0) ? db.tid_of[t] : 0;   // issued now, needed after the refinement
    refine_level_group(db, g, level, lm_level, threshold, mt, sm, threadIdx.x, 0);
    if (threadIdx.x == 0) {
      if (mt.template_id >= 0 && level == 0) mt.template_id = final_id;       // final per-class template_id
      cand[ci] = mt;
    }
  }
}

void fl_launch_refine_level(fl_tdb db, fl_level_geom g, int level, const uint8_t* lm_level, float threshold, fl_match_t* cand,
                            int cap, const int* d_count, cudaStream_t s) {
  int grid = min(cap, 148 * 4);
  if (grid > 0) fl_launch(k_refine_level, dim3(grid), dim3(RF_THREADS), 0, s, db, g, level, lm_level, threshold, cand, cap, d_count);
}

// ------------------------------------------------------------------------------------------------
// K8 sort + unique under the canonical total order (similarity desc, template_id asc, class asc, y asc, x asc), then
// adjacent-unique on (x, y, similarity, class) (linemod.hpp:262-274).  The whole record fits a 128-bit key, so the
// sort moves keys only and the records are rebuilt from them.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ fl_sort_key make_key(const fl_match_t& m) {
  fl_sort_key k;
  k.hi = ((unsigned long long)(~__float_as_uint(m.similarity)) << 32) | (uint32_t)m.template_id;
  k.lo = ((unsigned long long)(uint32_t)m.class_idx << 32) | ((unsigned long long)((uint32_t)(m.y + 32768) & 0xFFFF) << 16) |
         ((uint32_t)(m.x + 32768) & 0xFFFF);
  return k;
}
__device__ __forceinline__ fl_match_t key_to_match(const fl_sort_key& k) {
  fl_match_t m;
  m.similarity = __uint_as_float(~(uint32_t)(k.hi >> 32));
  m.template_id = (int)(uint32_t)k.hi;
  m.class_idx = (int)(uint32_t)(k.lo >> 32);
  m.y = (int)((k.lo >> 16) & 0xFFFF) - 32768;
  m.x = (int)(k.lo & 0xFFFF) - 32768;
  return m;
}
// branch-free on purpose (| and &, not || and &&): in the sorting networks every lane compares different keys, and
// short-circuit branches would diverge on every comparison
__device__ __forceinline__ bool key_less(const fl_sort_key& a, const fl_sort_key& b) { return (a.hi < b.hi) | ((a.hi == b.hi) & (a.lo < b.lo)); }
__device__ __forceinline__ bool key_dup(const fl_sort_key& a, const fl_sort_key& b) {
  // equal x, y, similarity, class; template_id ignored (linemod.hpp:271-274)
  return (a.hi >> 32) == (b.hi >> 32) && a.lo == b.lo;
}
#define KEY_SENTINEL_HI 0xFFFFFFFFFFFFFFFFull

// gather live candidates of all lists into the key array [0, n_pad), sentinel-padded; *d_n_live = number of live keys
__global__ void __launch_bounds__(256) k_build_keys(fl_lists L, fl_sort_key* __restrict__ keys, int key_cap, int* __restrict__ d_n_live) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L.n_lists * L.list_cap) return;
  int l = i / L.list_cap, k = i - l * L.list_cap;
  int n = min(L.n_in[(size_t)l * L.n_in_stride], L.list_cap);
  if (k >= n) return;
  fl_match_t m = L.in[(size_t)l * L.list_stride + k];
  if (m.template_id < 0) return;
  int slot = atomicAdd(d_n_live, 1);
  if (slot < key_cap) keys[slot] = make_key(m);
}

#define SORT_SMEM_LARGE 8192     // keys the one-CTA sort holds in shared memory (128 KB); a power of two: the bitonic network pads to one
// Common case, ONE launch of one CTA: gather the live candidates of all lists, sort, prune duplicates.  When the lists hold
// more records than fit its shared memory it only sets *d_flag_big = 1 and the host runs the multi-kernel path (k_build_keys + global
// bitonic steps + k_unique_big).  d_scratch = {n_live, flag_big}.

// loads that must see what other CTAs of the SAME launch wrote (fused refine + sort): L2, not this SM's L1
__device__ __forceinline__ int ld_count(const fl_lists& L, int l) { return __ldcg(L.n_in + (size_t)l * L.n_in_stride); }
__device__ __forceinline__ fl_match_t ld_match(const fl_match_t* p) {
  const int* q = reinterpret_cast<const int*>(p);
  fl_match_t m;
  m.x = __ldcg(q); m.y = __ldcg(q + 1); m.similarity = __int_as_float(__ldcg(q + 2)); m.class_idx = __ldcg(q + 3); m.template_id = __ldcg(q + 4);
  return m;
}

__device__ __forceinline__ void sort_unique_body(fl_lists L, fl_xchg X, int key_cap, int smem_keys, fl_sort_key* s_k, fl_match_t* __restrict__ out,
                                                 int out_cap, int* __restrict__ d_out_count, int* __restrict__ d_hdr,
                                                 int* __restrict__ h_hdr, fl_match_t* __restrict__ h_first, int h_first_cap,
                                                 int dbg_a = 0, int dbg_b = 0, int dbg_n = 0) {   // dbg_*: caller's timeline (ns) for h_hdr[8], [9], [11]
  // d_hdr (16 ints, handle-owned) = {unique count, n_live, flag_big, raw n_in[0..10], fused-tail overflow flag, exchange time-out}.  h_hdr / h_first (nullable) are the
  // same summary and the first matches in MAPPED PINNED HOST memory: the kernel posts them over PCIe itself, so the host
  // needs no device-to-host copy (and none of its ~8 us of copy-engine hand-over) before it can read the result.
  // Stores to mapped host memory cost ~0.7 us EACH when one thread issues them one after the other (measured: 6 us for the dozen
  // header words), so the summary is staged in shared memory and leaves as ONE coalesced 64-byte store, the records as
  // contiguous 128-byte warp stores.
  __shared__ int s_warp[32];
  __shared__ int s_n;
  __shared__ int s_hdr[16];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned long long t_body0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_body0));
  if (tid < 16 && tid != 14) s_hdr[tid] = 0;                    // [15]: exchange time-out flag (1 + rank that never arrived)
  if (tid == 32) s_hdr[14] = __ldcg(d_hdr + 14);                 // overflow flag of the fused refinement tail (set by the staged kernel): posted below, then cleared
  __syncthreads();
  // one warp posts the staged summary: device copy (flag word cleared) and mapped host copy
  auto post_header = [&]() {
    if (tid < 16) { const int v = s_hdr[tid]; d_hdr[tid] = tid == 14 ? 0 : v; if (h_hdr) h_hdr[tid] = v; }
    if (tid == 16 && d_out_count != d_hdr) *d_out_count = s_hdr[0];
  };
  unsigned long long t_dbg[4] = {0, 0, 0, 0};
  if (X.world > 0) {
    // ---- peer exchange (see fl_xchg): push, publish, wait ----
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_dbg[0]));
    const size_t block_recs = (size_t)X.cap + 1;
    const size_t parity_off = FL_XCHG_SIGNALS * sizeof(unsigned) + (size_t)(X.epoch & 1u) * X.world * block_recs * sizeof(fl_match_t);
    const int* src = reinterpret_cast<const int*>(X.local_block);
    const int n_raw = __ldcg(src);                              // L2 loads: in the fused launch other CTAs have just refined these records
    const int n_local = min(max(n_raw, 0), X.cap);              // records that exist; the header keeps the RAW count so that every
    const int n_ints = 5 * (1 + n_local);                       // rank (and the host) sees an overflow; readers clamp it to the capacity
    for (int p = 0; p < X.world; ++p) {
      int* dst = reinterpret_cast<int*>(X.peer[p] + parity_off + (size_t)X.rank * block_recs * sizeof(fl_match_t));
      for (int i = tid; i < n_ints; i += blockDim.x) dst[i] = (i == 0) ? n_raw : __ldcg(src + i);
    }
    __threadfence_system();
    __syncthreads();
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_dbg[1]));
    if (tid < X.world) st_release_sys(reinterpret_cast<unsigned*>(X.peer[tid]) + X.rank, X.epoch);
    if (tid < X.world) {
      const unsigned* sig = reinterpret_cast<const unsigned*>(X.peer[X.rank]) + tid;
      const long long t0 = clock64();
      while ((int)(ld_acquire_sys(sig) - X.epoch) < 0) {
        if (clock64() - t0 > (1ll << 32)) { s_hdr[15] = 1 + tid; break; }   // ~2 s: a peer never arrived; report instead of hanging
        __nanosleep(64);
      }
    }
    __syncthreads();
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_dbg[2]));
    L.in = reinterpret_cast<const fl_match_t*>(X.peer[X.rank] + parity_off) + 1;
    L.n_in = reinterpret_cast<const int*>(X.peer[X.rank] + parity_off);
    L.n_lists = X.world; L.list_cap = X.cap; L.list_stride = X.cap + 1; L.n_in_stride = 5 * (X.cap + 1);
  }
  const int n_lists = L.n_lists, list_cap = L.list_cap;
  int total = 0;
  for (int l = 0; l < n_lists; ++l) total += min(max(ld_count(L, l), 0), list_cap);
  if (tid < 11) s_hdr[3 + tid] = tid < n_lists ? ld_count(L, tid) : 0;
  if (total > smem_keys || total > key_cap) {
    if (tid == 0) { s_hdr[0] = 0; s_hdr[1] = total; s_hdr[2] = 1; }
    __syncthreads();
    post_header();
    return;
  }
  __syncthreads();                                               // s_hdr[3..13] complete before threads retire
  // The launch always has 1,024 threads and room for SORT_SMEM_LARGE keys; frames with <= 1,024 records (the common case)
  // retire all but 256 threads here, so that the barriers stay cheap.
  const int nt = total > 1024 ? (int)blockDim.x : min(256, (int)blockDim.x);
  if (tid >= nt) return;
  auto sync_active = [&]() { asm volatile("bar.sync 1, %0;" ::"r"(nt) : "memory"); };
  auto load_key = [&](int e) {                                     // record e of the concatenated lists -> key (sentinel if dropped / past the end)
    fl_sort_key key; key.hi = KEY_SENTINEL_HI; key.lo = KEY_SENTINEL_HI;
    if (e < total) {
      int l = 0, k = e;
      for (;;) { const int c = min(max(ld_count(L, l), 0), list_cap); if (k < c) break; k -= c; ++l; }
      const fl_match_t m = ld_match(L.in + (size_t)l * L.list_stride + k);
      if (m.template_id >= 0) key = make_key(m);                   // dropped candidates carry template_id -1
    }
    return key;
  };
  unsigned long long ts[5] = {0, 0, 0, 0, 0};
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ts[0]));
  int n = 0, n_pad = 2;                                            // live keys, sorted slots (after this block s_k[0, n) is sorted)
  if (total <= 256 && nt == 256) {
    // rank sort: the rank of a record among the live ones is the number of keys that precede it (ties - fully identical
    // records - broken by index): one pass over shared memory and three barriers
    const fl_sort_key key = load_key(tid);
    const bool live = !(key.hi == KEY_SENTINEL_HI && key.lo == KEY_SENTINEL_HI);
    fl_sort_key* s_in = s_k + 256;
    s_in[tid] = key;
    const unsigned live_mask = __ballot_sync(0xffffffffu, live);
    if (lane == 0) s_warp[warp] = __popc(live_mask);
    sync_active();
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ts[1]));
    if (live) {
      int rank = 0;
      for (int j0 = 0; j0 < total; j0 += 8) {                      // 8 broadcast loads in flight per pass
        fl_sort_key o[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) o[u] = s_in[j0 + u];
#pragma unroll
        for (int u = 0; u < 8; ++u)
          rank += (int)((j0 + u < total) & (key_less(o[u], key) | ((o[u].hi == key.hi) & (o[u].lo == key.lo) & (j0 + u < tid))));
      }
      s_k[rank] = key;
    }
#pragma unroll
    for (int w = 0; w < 8; ++w) n += s_warp[w];
    n_pad = 256;
    sync_active();
  } else if (total <= 1024 && nt == 256) {
    // bitonic network on keys held in REGISTERS, four consecutive slots per thread: strides 1 and 2 stay inside a thread,
    // strides 4..64 are warp shuffles, only strides >= 128 go through shared memory (3 exchanges for 512 slots, 6 for 1,024,
    // instead of 45 / 55 barrier-separated passes), and the 4 independent keys per thread hide the compare latency.
    const int N2 = total <= 512 ? 512 : 1024;
    const bool active = tid < N2 / 4;
    fl_sort_key key[4];
    int nlive = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      key[r].hi = KEY_SENTINEL_HI; key[r].lo = KEY_SENTINEL_HI;
      if (active) key[r] = load_key(4 * tid + r);
      nlive += !(key[r].hi == KEY_SENTINEL_HI && key[r].lo == KEY_SENTINEL_HI);
    }
    nlive = __reduce_add_sync(0xffffffffu, nlive);
    if (lane == 0) s_warp[warp] = nlive;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ts[1]));
    for (int k = 2; k <= N2; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        fl_sort_key o[4];
        if (j >= 128) {
          if (active) {
#pragma unroll
            for (int r = 0; r < 4; ++r) s_k[4 * tid + r] = key[r];
          }
          sync_active();
          if (active) {
#pragma unroll
            for (int r = 0; r < 4; ++r) o[r] = s_k[(4 * tid + r) ^ j];
          }
          sync_active();
        } else if (j >= 4) {
#pragma unroll
          for (int r = 0; r < 4; ++r) { o[r].hi = __shfl_xor_sync(0xffffffffu, key[r].hi, j >> 2); o[r].lo = __shfl_xor_sync(0xffffffffu, key[r].lo, j >> 2); }
        } else {
          if (j == 1) { o[0] = key[1]; o[1] = key[0]; o[2] = key[3]; o[3] = key[2]; }
          else { o[0] = key[2]; o[1] = key[3]; o[2] = key[0]; o[3] = key[1]; }
        }
        if (active) {
#pragma unroll
          for (int r = 0; r < 4; ++r) {
            const int e = 4 * tid + r;
            const bool take_min = ((e & k) == 0) == ((e & j) == 0);
            const bool lt = key_less(o[r], key[r]), gt = key_less(key[r], o[r]);
            const bool take = take_min ? lt : gt;                  // selects, no branches
            key[r].hi = take ? o[r].hi : key[r].hi;
            key[r].lo = take ? o[r].lo : key[r].lo;
          }
        }
      }
    if (active) {
#pragma unroll
      for (int r = 0; r < 4; ++r) s_k[4 * tid + r] = key[r];
    }
    sync_active();
#pragma unroll
    for (int w = 0; w < 8; ++w) n += s_warp[w];
    n_pad = N2;
  } else {
    if (tid == 0) s_n = 0;
    sync_active();
    for (int i = tid; i < total; i += nt) {
      const fl_sort_key key = load_key(i);
      if (!(key.hi == KEY_SENTINEL_HI && key.lo == KEY_SENTINEL_HI)) s_k[atomicAdd(&s_n, 1)] = key;
    }
    sync_active();
    n = s_n;
    while (n_pad < n) n_pad <<= 1;
    for (int i = n + tid; i < n_pad; i += nt) { s_k[i].hi = KEY_SENTINEL_HI; s_k[i].lo = KEY_SENTINEL_HI; }
    sync_active();
    for (int k = 2; k <= n_pad; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = tid; i < n_pad; i += nt) {
          const int p = i ^ j;
          if (p > i) {
            const bool up = (i & k) == 0;
            const fl_sort_key a = s_k[i], b = s_k[p];
            if (key_less(b, a) == up) { s_k[i] = b; s_k[p] = a; }
          }
        }
        sync_active();
      }
  }
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ts[2]));
  // adjacent unique + ordered compaction: each thread owns a contiguous run of slots; block-wide exclusive scan of the kept counts
  const int per = (n_pad + nt - 1) / nt;
  const int b0 = tid * per;
  int cnt = 0;
  for (int i = b0; i < min(b0 + per, n); ++i) cnt += (i == 0 || !key_dup(s_k[i - 1], s_k[i])) ? 1 : 0;
  int inc = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
  sync_active();                                                   // every thread has read the live counts in s_warp
  if (lane == 31) s_warp[warp] = inc;
  sync_active();
  if (warp == 0) {
    int w = lane < (nt >> 5) ? s_warp[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += t; }
    s_warp[lane] = w;
  }
  sync_active();
  int pos = (warp > 0 ? s_warp[warp - 1] : 0) + inc - cnt;
  const int n_unique = s_warp[31];
  // records leave through a staging area in shared memory when they fit (<= 1,024 sorted slots: the keys use at most 1,024 of
  // the 8,192 slots), so that device and mapped-host copies are contiguous 128-byte warp stores
  const bool staged = n_pad <= 1024;
  int* s_out = reinterpret_cast<int*>(s_k + 1024);
  for (int i = b0; i < min(b0 + per, n); ++i)
    if (i == 0 || !key_dup(s_k[i - 1], s_k[i])) {
      const fl_match_t m = key_to_match(s_k[i]);
      if (staged) { int* o = s_out + 5 * pos; o[0] = m.x; o[1] = m.y; o[2] = __float_as_int(m.similarity); o[3] = m.class_idx; o[4] = m.template_id; }
      else {
        if (pos < out_cap) out[pos] = m;
        if (h_first && pos < h_first_cap) h_first[pos] = m;
      }
      ++pos;
    }
  if (tid == 0) {
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ts[3]));
    s_hdr[0] = n_unique; s_hdr[1] = n; s_hdr[2] = 0;
    if (n_lists == 1) { s_hdr[4] = (int)(ts[0] - t_body0); s_hdr[5] = (int)(ts[1] - ts[0]); s_hdr[6] = (int)(ts[2] - ts[1]); s_hdr[7] = (int)(ts[3] - ts[2]); }   // developer timeline (ns)
    // (words 3 .. 3 + n_lists - 1 are the per-list raw counts the host checks for overflow: developer values only go where no list lives)
    if (X.world == 0 && n_lists <= 4) { s_hdr[8] = dbg_a; s_hdr[9] = dbg_b; s_hdr[10] = (int)(ts[3] - t_body0); s_hdr[11] = dbg_n; }
    if (X.world > 0 && X.world <= 4) {                           // developer timing of the exchange (ns): push, wait, sort
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_dbg[3]));
      s_hdr[8] = (int)(t_dbg[1] - t_dbg[0]); s_hdr[9] = (int)(t_dbg[2] - t_dbg[1]); s_hdr[10] = (int)(t_dbg[3] - t_dbg[2]);
    }
  }
  sync_active();
  if (staged) {
    int* out_i = reinterpret_cast<int*>(out);
    int* hf_i = reinterpret_cast<int*>(h_first);
    const int n_out = 5 * min(n_unique, out_cap), n_hf = h_first ? 5 * min(n_unique, h_first_cap) : 0;
    for (int q = tid; q < 5 * n_unique; q += nt) {
      const int v = s_out[q];
      if (q < n_out) out_i[q] = v;
      if (q < n_hf) hf_i[q] = v;
    }
  }
  post_header();
}

__global__ void __launch_bounds__(1024) k_sort_unique_small(fl_lists L, fl_xchg X, int key_cap, int smem_keys, fl_match_t* __restrict__ out,
                                                            int out_cap, int* __restrict__ d_out_count, int* __restrict__ d_hdr,
                                                            int* __restrict__ h_hdr, fl_match_t* __restrict__ h_first, int h_first_cap) {
  extern __shared__ __align__(16) fl_sort_key s_k[];            // smem_keys keys
  fl_grid_dep_wait();
  fl_grid_dep_launch();
  sort_unique_body(L, X, key_cap, smem_keys, s_k, out, out_cap, d_out_count, d_hdr, h_hdr, h_first, h_first_cap);
}

// Refinement up the whole pyramid + sort + unique in ONE launch (the single-handle match path): RS_GROUPS groups of RF_THREADS
// threads per CTA refine candidates (a candidate stays with its group for all levels, so no grid-wide step is needed between
// levels); the CTA that finishes last (ticket on *done_ctr) then sorts the list, prunes duplicates and posts the result to
// the host.  Saves the launch + dependency gap of every refinement level and of the sort kernel.
template <int RS_GROUPS>
__global__ void __launch_bounds__(RS_GROUPS * RF_THREADS) k_refine_sort(const __grid_constant__ fl_tdb db, const __grid_constant__ fl_refine_args ra,
                                                                          float threshold, fl_match_t* cand, int cap, const int* __restrict__ d_count,
                                                                          int* done_ctr, fl_lists L, fl_xchg X, int key_cap, int smem_keys, fl_match_t* __restrict__ out,
                                                                          int out_cap, int* __restrict__ d_out_count, int* __restrict__ d_hdr,
                                                                          int* __restrict__ h_hdr, fl_match_t* __restrict__ h_first, int h_first_cap) {
  extern __shared__ __align__(16) fl_sort_key s_k[];
  __shared__ fl_refine_smem sm[RS_GROUPS];
  __shared__ int s_last;
  unsigned long long tq[4] = {0, 0, 0, 0};                          // developer timeline (ns), posted in h_hdr[8..11] when no exchange runs
  fl_grid_dep_wait();
  fl_grid_dep_launch();
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tq[0]));
  const int grp = threadIdx.x / RF_THREADS, gt = threadIdx.x - grp * RF_THREADS;
  const int n = min(*d_count, cap);
  if (ra.n_levels > 1) {
    for (int ci = blockIdx.x * RS_GROUPS + grp; ci < n; ci += gridDim.x * RS_GROUPS) {
      fl_match_t mt = cand[ci];
      if (mt.template_id < 0) continue;
      const int t = mt.template_id;
      for (int l = ra.n_levels - 2; l >= 0 && mt.template_id >= 0; --l) refine_level_group(db, ra.g[l], l, ra.lm[l], threshold, mt, sm[grp], gt, 1 + grp);
      if (gt == 0) {
        if (mt.template_id >= 0) mt.template_id = db.tid_of[t];    // final per-class template_id
        cand[ci] = mt;
      }
    }
  }
  __syncthreads();
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tq[1]));
  if (threadIdx.x == 0) {
    __threadfence();                                               // this CTA's records before its ticket
    const int ticket = atomicAdd(done_ctr, 1);
    s_last = ticket == (int)gridDim.x - 1;
    if (s_last) *done_ctr = 0;                                     // ready for the next launch
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tq[2]));
  sort_unique_body(L, X, key_cap, smem_keys, s_k, out, out_cap, d_out_count, d_hdr, h_hdr, h_first, h_first_cap, (int)(tq[1] - tq[0]), (int)(tq[2] - tq[1]), n);
}

// large path: global bitonic steps + serial-chunk unique
__global__ void __launch_bounds__(256) k_pad_keys(fl_sort_key* keys, const int* d_n_live, int key_cap, int n_pad) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int n = min(*d_n_live, key_cap);
  if (i >= n && i < n_pad) { keys[i].hi = KEY_SENTINEL_HI; keys[i].lo = KEY_SENTINEL_HI; }
}
__global__ void __launch_bounds__(256) k_bitonic_step(fl_sort_key* keys, int n_pad, int k, int j) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pad) return;
  int p = i ^ j;
  if (p > i) {
    bool up = (i & k) == 0;
    fl_sort_key a = keys[i], b = keys[p];
    if (key_less(b, a) == up) { keys[i] = b; keys[p] = a; }
  }
}
__global__ void __launch_bounds__(1024) k_unique_big(const fl_sort_key* __restrict__ keys, const int* __restrict__ d_n_live, int key_cap,
                                                     fl_match_t* __restrict__ out, int out_cap, int* __restrict__ d_out_count) {
  __shared__ int s_warp[32];
  __shared__ int s_base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = min(*d_n_live, key_cap);
  if (tid == 0) s_base = 0;
  __syncthreads();
  for (int c0 = 0; c0 < n; c0 += 1024) {
    const int i = c0 + tid;
    const int keep = (i < n && (i == 0 || !key_dup(keys[i - 1], keys[i]))) ? 1 : 0;
    int inc = keep;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      int w = s_warp[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += t; }
      s_warp[lane] = w;
    }
    __syncthreads();
    const int pos = s_base + (warp > 0 ? s_warp[warp - 1] : 0) + inc - keep;
    if (keep && pos < out_cap) out[pos] = key_to_match(keys[i]);
    __syncthreads();
    if (tid == 0) s_base += s_warp[31];
    __syncthreads();
  }
  if (tid == 0) *d_out_count = s_base;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the (device, function) pair: it is set once per device this process
// launches on (a process-wide flag would leave every device but the first without the opt-in), under a lock because handles
// on different devices may be driven by different host threads.
static bool fl_once_per_device(int which) {
  static std::mutex mu;
  static bool done[1][FL_MAX_DEVICES];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= FL_MAX_DEVICES) return false;
  std::lock_guard<std::mutex> lk(mu);
  if (done[which][dev]) return true;
  const int bytes = SORT_SMEM_LARGE * (int)sizeof(fl_sort_key);
  const cudaError_t e = cudaFuncSetAttribute(k_sort_unique_small, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return false;
  done[which][dev] = true;
  return true;
}

// Host orchestration.  Scratch int (n_live of the big path) lives right after the key array.  Return: launches made, -1 = launch error.
int fl_launch_sort_unique(fl_lists L, fl_xchg X, int key_cap, fl_match_t* d_out, int out_cap, int* d_out_count, int* d_hdr,
                          int* h_hdr, fl_match_t* h_first, int h_first_cap, cudaStream_t s) {
  if (!fl_once_per_device(0)) return -1;
  return fl_launch(k_sort_unique_small, dim3(1), dim3(1024), (size_t)SORT_SMEM_LARGE * sizeof(fl_sort_key), s, L, X, key_cap, (int)SORT_SMEM_LARGE, d_out,
                       out_cap, d_out_count, d_hdr, h_hdr, h_first, h_first_cap) == cudaSuccess ? 1 : -1;
}

// One 256-thread group per CTA, 4 CTAs per SM, shared memory for 1,024 keys + staging (no opt-in needed): as cheap to launch as
// k_refine_level; lists with more than 1,024 records come back flagged and the host runs the stand-alone sort.  (A variant with four
// groups per CTA and the full 8,192-key sort inside was measured slower to launch than the launch it saved, and removed; launching
// this kernel programmatically behind the similarity kernel was slower too - 80.4 vs 76.3 us per frame: its 592 pre-launched CTAs
// take SM slots the similarity CTAs' tails still need.)
int fl_launch_refine_sort(fl_tdb db, const fl_refine_args& ra, float threshold, fl_match_t* cand, int cap, const int* d_count, int* done_ctr, int n_sm,
                          fl_lists L, fl_xchg X, int key_cap, fl_match_t* d_out, int out_cap, int* d_out_count, int* d_hdr,
                          int* h_hdr, fl_match_t* h_first, int h_first_cap, cudaStream_t s) {
  const int keys = 1024;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = dim3(4 * (n_sm > 0 ? n_sm : 148)); cfg.blockDim = dim3(RF_THREADS); cfg.dynamicSmemBytes = (size_t)(keys + 1280) * sizeof(fl_sort_key); cfg.stream = s;
  return cudaLaunchKernelEx(&cfg, k_refine_sort<1>, db, ra, threshold, cand, cap, d_count, done_ctr, L, X, key_cap, keys, d_out, out_cap, d_out_count, d_hdr, h_hdr,
                            h_first, h_first_cap) == cudaSuccess ? 1 : -1;
}

// second stage, only when the one-CTA kernel reported more records than its shared memory holds (the host has read the flag and the
// record count n_upper)
int fl_launch_sort_unique_big(fl_lists L, fl_sort_key* keys, int key_cap, int n_upper, fl_match_t* d_out, int out_cap, int* d_out_count, cudaStream_t s) {
  int launches = 0;
  int* d_scratch = reinterpret_cast<int*>(keys + key_cap);
  cudaMemsetAsync(d_scratch, 0, sizeof(int), s);
  const int total = L.n_lists * L.list_cap;
  k_build_keys<<<(total + 255) / 256, 256, 0, s>>>(L, keys, key_cap, d_scratch); ++launches;
  int n_pad = 2;
  while (n_pad < n_upper) n_pad <<= 1;
  if (n_pad > key_cap) return -1;
  k_pad_keys<<<(n_pad + 255) / 256, 256, 0, s>>>(keys, d_scratch, key_cap, n_pad); ++launches;
  for (int k = 2; k <= n_pad; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) { k_bitonic_step<<<(n_pad + 255) / 256, 256, 0, s>>>(keys, n_pad, k, j); ++launches; }
  k_unique_big<<<1, 1024, 0, s>>>(keys, d_scratch, key_cap, d_out, out_cap, d_out_count); ++launches;
  return launches;
}

