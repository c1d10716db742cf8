// fealess_b200 internal declarations shared by the .cu translation units (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <memory>
#include "../../include/fealess_b200.h"

#define FL_MAX_DEVICES 64        // devices of one process (per-device kernel attribute tables)
#define FL_LM_PAD 4096          // zero bytes after each label's linear memory (flat-addressing over-read, see DESIGN.md)
#define FL_MAX_T 16
#define FL_SKIP 0xFFFFFFFFu     // packed-feature offset of a feature that falls outside the image

// packed feature for one pyramid level and one frame geometry: lm_off is the byte offset of the feature's first
// response inside the (level, modality) linear-memory block = label*label_stride + row*cells + (y/T)*W' + x/T
// (accessLinearMemory, reference linemod/linemod.cpp:1094-1117); x,y kept for the in-image test of similarityLocal.
struct __align__(8) fl_pfeat { uint32_t lm_off; int16_t x, y; };

struct fl_level_geom {
  int W, H, T, Wd, Hd, cells;      // image size at the level, sampling step, decimated size
  size_t label_stride;             // bytes per label (T*T*cells + pad, 32-aligned: the 4-bit copy of a label starts 16-byte aligned)
  size_t mod_stride;               // bytes per modality = 8 * label_stride
};

struct fl_sort_key { unsigned long long hi, lo; };

void fl_set_error(const char* fmt, ...);
int fl_entries_per_template(const fl_handle* h);   // n_levels * n_modalities of the handle (api.cu)

// The frame in flight on a handle (api.cu), from its enqueue to its wait.  match: fl_match_device_async and the host entry points
// that stage into it; shard: the fused local match + peer exchange (fl_match_shard_exchange_*); sort: the stand-alone exchange + sort
// (fl_exchange_sort_unique_device_async); reco: a frame with the recognition tail behind its sort, whose results are still to be collected.
enum class fl_frame_kind { none, match, shard, sort, reco };
fl_frame_kind fl_frame_in_flight(const fl_handle* h);
// What fl_frame_wait did besides waiting for the frame in flight.  After an in-grid dependency time-out of the single-launch front end
// the handle launches one kernel per wave from then on, and the frame's result is not trustworthy: a frame matched on this handle alone
// has been run again (rerun); one that exchanged with peers needs every rank, so it must be submitted again (resubmit, FL_ERR_STATE).
enum class fl_wait_note { done, rerun, resubmit };
int fl_frame_wait(fl_handle* h, fl_wait_note* note);

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------------------
// A kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may have its CTAs resident while the previous kernel
// of the stream drains: they run their prologue and block in fl_grid_dep_wait() until that kernel has completed and its writes
// are visible; fl_grid_dep_launch() tells the scheduler that the NEXT kernel may start being placed.  Rule: a kernel touches no
// mutable global buffer before fl_grid_dep_wait().  Launched without the attribute both calls are no-ops.  Only the staged
// similarity kernel is launched this way (behind the front end); for every other kernel of the frame the attribute was measured
// to give nothing or to cost (DESIGN.md), so they use the plain fl_launch below.
#ifdef __CUDACC__
__device__ __forceinline__ void fl_grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void fl_grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif
template <typename... KArgs, typename... Args>
inline cudaError_t fl_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

#define FL_CUDA(call)                                                                  \
  do {                                                                                 \
    cudaError_t e__ = (call);                                                          \
    if (e__ != cudaSuccess) {                                                          \
      fl_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return FL_ERR_CUDA;                                                              \
    }                                                                                  \
  } while (0)

// ---- front end (frontend.cu) -------------------------------------------------------------------
int fl_launch_tables_init();   // uploads the two LUTs to __constant__ memory of the current device
void fl_launch_resize_nn_half(const uint8_t* src, int W, int H, uint8_t* dst, cudaStream_t s);   // training's mask pyramid
// Per-handle response mass of the coarsest level, u32 words: the spread jobs of that level add the sum of every linear-memory
// response of (modality m, label l) into word 8 m + l; k_similarity_staged orders its phases by these sums and its last CTA to
// read them clears them again (ticket), so every frame starts from zero without a memset.  Behind them: what the last staged
// launch used (the sums, and CTA 0's phase of every visit step as bytes), for fl_debug_get(FL_DBG_STAGED_ORDER).
#define FL_MASS_TICKET 32
#define FL_MASS_USED 64
#define FL_MASS_ORDER 96
#define FL_MASS_WORDS (FL_MASS_ORDER + 64)

// one launch = several independent front-end jobs (see k_front_end_wave)
enum { FL_JOB_PYRDOWN = 2, FL_JOB_RESIZE = 3, FL_JOB_SPREAD = 4, FL_JOB_COLOR2 = 5, FL_JOB_DEPTH2 = 6, FL_JOB_PREFETCH = 7 };
struct fl_fe_job {
  int kind, cta_begin, gx, W, H, p0, p1;
  float thr_sq;
  const uint8_t* src; uint8_t* dst; uint8_t* dst2; uint8_t* dst3;   // spread job: dst = linear memories, dst2 = spread image (or NULL), dst3 = 4-bit linear memories (or NULL)
  uint32_t* mass;                                                     // spread job: response sums of the modality's 8 labels (or NULL), see FL_MASS_*
  const uint8_t* mask; int mask_stride, mask_shift;                   // spread job: the frame's mask of the modality (or NULL), see dev_spread_lm
  fl_level_geom g;
  // in-grid dependencies (single-launch front end): a CTA of this job first waits until counters[wait_slot] has reached
  // wait_target (all CTAs of the producing job have finished), and bumps counters[signal_slot] when it is done; -1 = none
  int wait_slot, signal_slot;
  unsigned wait_target;
  // finer grain for the spread jobs: a producing tile job also counts its finished tiles PER TILE ROW (counters[row_base + by]);
  // a spread CTA that owns grid row gy waits only for the tile rows that hold its label rows [gy T, gy T + 2T - 2] (row y of
  // its level lives in producer row (y << wait_row_shift) / 16), so it starts while later rows are still being quantised
  int row_base, wait_row_base, wait_row_shift, wait_row_count;
  unsigned wait_row_target;
};
#define FL_FE_MAX_TILE_ROWS 128
// NN-downsampled copies of the level-0 depth labels written by the depth job itself: entry i = pyramid level i + 1
#define FL_FE_MAX_PYR 7
struct fl_depth_pyr { int n; int W[FL_FE_MAX_PYR], H[FL_FE_MAX_PYR]; uint8_t* dst[FL_FE_MAX_PYR]; };
#define FL_FE_MAX_JOBS 16
#define FL_FE_MAX_DPYR 2
// the argument of one k_front_end_wave launch.  zero_me: int reset by CTA 0 (the candidate counter), or NULL.  pyr: the NN pyramids the
// depth jobs write (a depth job's thr_sq holds its slot).  counters (single launch only, else NULL): FL_FE_MAX_JOBS monotonic CTA
// counters, one error word (dep_error), FL_FE_MAX_JOBS x FL_FE_MAX_TILE_ROWS tile-row counters; dep_error_host: the same flag in mapped
// host memory, written only on a time-out.  trace (FL_OPT_TRACE, or NULL): per job {first CTA start, last CTA end} in globaltimer ns,
// then per job the sums of its CTAs' spans {SM cycles, ns}.
struct fl_fe_wave { int n_jobs, n_ctas; size_t smem; int* zero_me; fl_fe_job job[FL_FE_MAX_JOBS]; int n_pyr; fl_depth_pyr pyr[FL_FE_MAX_DPYR];
                    unsigned* counters; int* dep_error; int* dep_error_host;
                    unsigned long long* trace; };

// What one frame's front end reads and writes: the frame's level-0 images and masks, and the handle's buffers for its geometry.
struct fl_fe_frame {
  int n_levels, n_modalities; const int32_t* modality_kind; const fl_level_geom* geom;
  const uint8_t* bgr; const uint16_t* depth;                 // level 0 (NULL when no modality reads it)
  uint8_t* bgr_pyr[FL_MAX_LEVELS];                           // colour pyramid, levels >= 1
  uint8_t* q[FL_MAX_LEVELS][FL_MAX_MODALITIES];              // labels
  uint8_t* lm[FL_MAX_LEVELS];                                // linear memories of a level, modality m at m * mod_stride
  uint8_t* lm4; uint32_t* mass;                              // coarsest level: 4-bit linear memories, response sums (FL_MASS_*); NULL = not written
  uint8_t* spread[FL_MAX_LEVELS][FL_MAX_MODALITIES];         // spread images (NULL = not kept)
  const uint8_t* mask[FL_MAX_MODALITIES];                    // level-0 masks (NULL = unmasked)
  uint8_t* mask_pyr[FL_MAX_LEVELS][FL_MAX_MODALITIES];       // levels >= 1 of the NN mask pyramid of a geometry that does not halve exactly
  float thr_sq; int dist_thr, diff_thr;                      // colour magnitude threshold squared, depth distance / difference thresholds
  // pulled towards L2 in the single launch (one 128-byte line per thread): the staged similarity kernel's per-template feature lists, and
  // then its prologue's lookups (template -> class -> enabled), so that it does not start with DRAM round trips.  The first three
  // ranges go in when the launch has room for three more jobs, all six when it has room for six; empty ranges are skipped.
  const void* prefetch[6]; size_t prefetch_bytes[6];
  int* zero_me;                                              // reset by the first launch (the candidate counter)
  bool trace;                                                // FL_OPT_TRACE: record the single launch's job timeline
};
// Per-handle state of the front end (frontend.cu): the in-grid dependency counters and their bases, the time-out flag, the job timeline
// and the front end's switches.  Owned by the handle through fl_fe_owned.
struct fl_fe_state;
struct fl_fe_free { void operator()(fl_fe_state* s) const; };
typedef std::unique_ptr<fl_fe_state, fl_fe_free> fl_fe_owned;
int fl_fe_create(fl_fe_owned* out);                          // on the current device
// a new geometry or template set can change the job layout: the tile-row counters restart from zero (stream-ordered)
int fl_fe_forget_rows(fl_fe_state* fe, cudaStream_t s);
// enqueue the whole front end of one frame: one launch, or one per wave (FL_OPT_FE_WAVES, after a time-out, and for geometries the
// single launch does not take); *launches grows by the number of launches
int fl_fe_run(fl_fe_state* fe, const fl_fe_frame& f, cudaStream_t s, int64_t* launches);
// after the frame's wait: *job = the job whose in-grid dependency timed out, or -1.  On a time-out the flag and the error word are
// cleared and the handle launches one kernel per wave from then on.
int fl_fe_take_timeout(fl_fe_state* fe, cudaStream_t s, int* job);
int fl_fe_trace(const fl_fe_state* fe, void* host_out, size_t bytes);     // FL_DBG_FE_TRACE
int fl_fe_option(fl_fe_state* fe, int option, int value);                  // FL_OPT_FE_WAVES, FL_OPT_FE_DEP_TIMEOUT_TEST, FL_OPT_FE_FORCED_WAVES

// ---- template training, per-pixel half (train.cu) -----------------------------------------------
void fl_launch_train_magnitude(const uint8_t* bgr, int W, int H, float* mag, cudaStream_t s);
void fl_launch_train_erode3(const uint8_t* src, int W, int H, uint8_t* dst, cudaStream_t s);
void fl_launch_train_color_score(const uint8_t* angle, const float* mag, const uint8_t* mask, const uint8_t* eroded, int W, int H, float threshold_sq,
                                 float* score, cudaStream_t s);
void fl_launch_train_depth_score(const uint8_t* normal, const uint8_t* local_mask, uint16_t* hd, int* any_zero8, int W, int H, int extract_threshold,
                                 float* score, int* label_counts8, cudaStream_t s);

// ---- similarity / refinement / sort (similarity.cu) ---------------------------------------------
struct fl_tdb {                     // device template database
  int n_templates, L, M, n_classes;
  const fl_template_hdr_t* hdr;     // [n_templates*L*M]
  const fl_feature_t* feat;         // [n_features]
  const int32_t* class_of;          // [n_templates]
  const int32_t* class_first;       // [n_classes]
  const int32_t* tid_of;            // [n_templates] per-class template_id reported in matches (global id for shards)
  const uint8_t* class_enabled;     // [n_classes] (class filter of the current call)
  fl_pfeat* pfeat;                  // [n_features] packed for the current geometry
  // refinement records (levels 0 .. L-2), one fixed-size block per (template, level): {width, height, n_features, 0, fc[0..3]}
  // (32 B) + M x 64 feature slots of 8 B.  A candidate's template index alone gives the address of everything its refinement
  // reads, so header and features load concurrently (no dependent pointer chase) and can be prefetched into L2 by the kernel
  // that emits the candidate.  Slot = fl_pfeat; a feature outside the image at offset 0 carries lm_off = FL_RSKIP | label.
  uint8_t* rrec; int rrec_bytes;
};
#define FL_RSKIP 0xFFFFFFF0u
__host__ __device__ inline int fl_rrec_bytes(int M) { return (32 + M * 64 * 8 + 127) & ~127; }
void fl_launch_pack_refine_records(fl_tdb db, const fl_level_geom* d_geom, cudaStream_t s);
// plan of the shared-memory-staged global similarity kernel (similarity_staged.cu) for one frame geometry
struct fl_staged_plan {
  int phase_rows, n_rowblocks, n_phases;   // a phase = phase_rows linear-memory rows of one (modality, label) ...
  int labels_per_phase;                    // ... or, when whole labels fit, this many consecutive labels of one modality (1, 2 or 4)
  int halo_bytes, buf_bytes, n_buf;        // bytes staged past the last row; size and number of the smem ring buffers
  int n_words, nw_template, tpw;           // 32-bit words per similarity map; template parameters of the instantiation used
  int tpc, n_cta, block_threads;           // templates per CTA, grid, block
  int smem_bytes, pre_stride;              // dynamic shared memory; bytes per gpre row
  int stage_off;                           // emission staging area (one similarity map, nw_template x 32 words)
  int prune;                               // 1: drop a template once no position can reach the threshold (off: FL_OPT_SIM_NO_PRUNE)
  int rotate;                              // 1: visit the phases in the rotated order of CTA b (FL_OPT_SIM_ROTATE) instead of by response mass
  uint32_t* mass;                          // the handle's response mass (FL_MASS_WORDS words, see FL_MASS_*)
  uint32_t* gfeat;                         // [n_templates][64] feature words sorted by phase: word offset in the phase buffer << 5 | 8 * byte misalignment
  uint8_t* gpre;                           // [n_templates][pre_stride] prefix counts per phase
  int4* gmeta;                             // [n_templates] {template_positions, n_features, class, 0}
  unsigned long long* trace;               // developer timeline (FL_OPT_TRACE): 8 words per CTA, or NULL
};
bool fl_plan_staged(const fl_level_geom& g, int M, int n_templates, int max_positions, int n_sm, fl_staged_plan* plan);
void fl_launch_pack_staged(fl_tdb db, fl_level_geom g, fl_staged_plan plan, cudaStream_t s);
// every level's geometry and linear memories, for the refinement that shares a launch with the sort (k_refine_sort)
struct fl_refine_args {
  int n_levels;
  fl_level_geom g[FL_MAX_LEVELS];
  const uint8_t* lm[FL_MAX_LEVELS];
};
int fl_launch_similarity_staged(fl_tdb db, fl_level_geom g, const uint8_t* lm4_level, float threshold, fl_match_t* cand, int cap,
                                int* d_count, fl_staged_plan plan, cudaStream_t s);
void fl_launch_pack_features(fl_tdb db, const fl_level_geom* d_geom, int n_features_total, cudaStream_t s);
void fl_launch_similarity_global(fl_tdb db, fl_level_geom g, const uint8_t* lm_level, float threshold,
                                 fl_match_t* cand, int cap, int* d_count, cudaStream_t s);
void fl_launch_similarity_debug(fl_tdb db, fl_level_geom g, const uint8_t* lm_level, int t, uint16_t* out, cudaStream_t s);
void fl_launch_refine_level(fl_tdb db, fl_level_geom g, int level, const uint8_t* lm_level, float threshold,
                            fl_match_t* cand, int cap, const int* d_count, cudaStream_t s);
// candidate lists handed to sort + unique: list l holds min(n_in[l * n_in_stride], list_cap) records starting at
// in + l * list_stride.  (list_stride = list_cap, n_in_stride = 1 for plain arrays; the all-gather block layout
// [header record with the count in .x | list_cap records] has list_stride = list_cap + 1, n_in_stride = 5 * (list_cap + 1).)
struct fl_lists { const fl_match_t* in; int n_lists, list_cap, list_stride; const int* n_in; int n_in_stride; };
// Direct peer exchange fused into the head of the sort kernel (template-sharded matching, one process per GPU): every rank's
// exchange buffer = [FL_XCHG_SIGNALS u32 signal words][2 parities x world blocks of (cap + 1) records] is mapped into every
// process (peer[p] = base of rank p's buffer as seen from THIS process).  The kernel pushes this rank's block
// [count | live records] into slot `rank` of every peer's buffer over NVLink, publishes `epoch` in the peer's signal word
// `rank` (release, system scope), waits until all of its own signal words show `epoch` (acquire), and then sorts the
// union straight out of its own buffer.  world == 0: no exchange.  The parity (epoch & 1) double-buffers the blocks: a rank
// can be at most one frame ahead of a peer, because it cannot pass frame k + 1's wait before the peer has published
// epoch k + 1, which the peer's stream does only after its frame-k sort kernel has finished.
#define FL_XCHG_MAX_WORLD 8
#define FL_XCHG_SIGNALS 64
struct fl_xchg { int world, rank, cap; unsigned epoch; const fl_match_t* local_block; uint8_t* peer[FL_XCHG_MAX_WORLD]; };
#ifdef __CUDACC__
__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) { unsigned v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
#endif

// sort + unique: result in d_out/d_out_count, summary in d_hdr[16] = {unique count, live records, flag_big, raw counts...}.
// One launch; when flag_big comes back set the host runs fl_launch_sort_unique_big (key workspace: next_pow2(n_upper) keys
// + 1 int).  Both return the number of launches.  h_hdr / h_first: mapped pinned host copies of the summary and of the
// first h_first_cap matches (nullable).
int fl_launch_sort_unique(fl_lists L, fl_xchg X, int key_cap, fl_match_t* d_out, int out_cap, int* d_out_count, int* d_hdr,
                          int* h_hdr, fl_match_t* h_first, int h_first_cap, cudaStream_t s);
// refinement of every level + sort + unique in one launch (the last CTA to finish sorts); done_ctr: zero-initialised device int
int fl_launch_refine_sort(fl_tdb db, const fl_refine_args& ra, float threshold, fl_match_t* cand, int cap, const int* d_count, int* done_ctr, int n_sm,
                          fl_lists L, fl_xchg X, int key_cap, fl_match_t* d_out, int out_cap, int* d_out_count, int* d_hdr,
                          int* h_hdr, fl_match_t* h_first, int h_first_cap, cudaStream_t s);
int fl_launch_sort_unique_big(fl_lists L, fl_sort_key* keys, int key_cap, int n_upper, fl_match_t* d_out, int out_cap, int* d_out_count, cudaStream_t s);

// ---- ICP (icp.cu) --------------------------------------------------------------------------------
struct fl_icp_hyp {                 // one hypothesis of a batch, device-visible
  const uint16_t* model_depth;      // device, dense crop rows of rect_model.width (NULL for cloud mode)
  fl_rect_t rect_model, rect_ref;
  float r_match[9], t_match[3];
  int status;
};
struct fl_icp_ws {                  // per-batch workspace, all device pointers; max_pts is a multiple of 4
  int n_hyp, max_pts;
  float* pts_ref;                   // [n_hyp][max_pts][3]
  float* pts_mod;                   // [n_hyp][max_pts][3]  (pts_model_tmp)
  float* cor_m; float* cor_r;       // [n_hyp][max_pts][3]  ordered correspondences
  float* dist;                      // [n_hyp][max_pts]     inlier distances of the index pairs (0 for the others)
  float* nn_d2; int* nn_slot;       // [n_hyp][max_pts]     nearest reference point of every model point: squared distance, slot in the grid
  float4* grid_pts;                 // [n_hyp][max_pts]     ref points sorted by cell (x,y,z,index) - only for clouds that do not fit shared memory
  int* n_ref; int* n_mod;           // [n_hyp]              cloud mode only
};
#define FL_ICP_TRACE_WORDS 20      // developer timeline of the fused ICP launch: words per hypothesis (fl_debug_icp_trace)
#define FL_ICP_GRID 64
#define FL_ICP_CELLS (FL_ICP_GRID * FL_ICP_GRID)
// cv::resize INTER_LINEAR (resize.cu): device tables built by the host for one (source size -> destination size) pair
struct fl_resize_tables {
  int* xofs; int* yofs;             // [dW], [dH] source index of the left / upper tap (rows unclipped: the kernel clips)
  short2* ialpha; short2* ibeta;    // 8U: 11-bit fixed-point weight pairs
  float2* alpha; float2* beta;      // 16U: float weight pairs
};
void fl_launch_resize_linear(const void* src, int sW, int sH, int type, void* dst, int dW, int dH, const fl_resize_tables& t, cudaStream_t s);
void fl_launch_depth_to_3d(const uint16_t* depth, int W, int H, fl_intrinsics_t K, float* out3, cudaStream_t s);
// the whole of detection() / icpCloudToCloud_Ex for a batch in ONE persistent launch (icp.cu); hyps == NULL: cloud mode.
// ticket: device int (reset by the call); trace: NULL or FL_ICP_TRACE_WORDS words per hypothesis (SM cycles per phase).  Returns the number of launches, -1 on a launch error.
int fl_launch_icp(fl_icp_ws ws, fl_icp_params_t p, const fl_icp_hyp* hyps_or_null, const uint16_t* ref_depth, int W, int H, fl_intrinsics_t K_ref,
                  fl_icp_result_t* results, int* ticket, unsigned long long* trace, int n_sm, cudaStream_t s);
void fl_launch_nms(const float* t3, const int32_t* n_model, const float* icp_dist, int n, float th, int32_t* out_idx,
                   int32_t* out_count, cudaStream_t s);
#ifdef __CUDACC__
// greedy nonMaximumSuppression (order dependent, n is small): ONE thread walks the list exactly like NMS.cpp:6-39.  out_idx[k] = the
// object emitted k-th, done[i] = 1 for every object the reference marks check_done (:27).  Shared by k_nms and k_reco_finish.
__device__ inline int fl_nms_greedy(const float* __restrict__ t3, const int32_t* __restrict__ n_model, const float* __restrict__ icp_dist, int n,
                                    float th, int32_t* __restrict__ out_idx, uint8_t* __restrict__ done) {
  int cnt = 0;
  for (int i = 0; i < n; ++i) done[i] = 0;
  for (int i = 0; i < n; ++i) {
    if (done[i]) continue;
    int win = i;
    const int size_th = (int)((double)(float)n_model[i] * 0.85);   // static_cast<int>((float)size * 0.85) (:17)
    for (int j = i + 1; j < n; ++j) {
      if (done[j]) continue;
      double s = 0;
      for (int k = 0; k < 3; ++k) { double d = (double)__fsub_rn(t3[3 * win + k], t3[3 * j + k]); s += d * d; }   // cv::norm(Mat, Mat): fp32 difference, fp64 squares
      if (sqrt(s) < (double)th) {
        done[j] = 1;
        if (n_model[j] > size_th && icp_dist[j] < icp_dist[win]) win = j;
      }
    }
    out_idx[cnt++] = win;
  }
  return cnt;
}
#endif

// ---- Recognition on the device (reco.cu) -----------------------------------------------------------
// per-template record of fl_set_recognition: the template's depth crop (NULL = none) with the rect it was uploaded with (= the
// template's level-0 modality-0 box) and the pose the mirrors look up for it, rows of (R | t)
struct fl_reco_tmpl { const uint16_t* crop; fl_rect_t rect; float pose[12]; };
// per-frame selection state written by k_reco_select: {n_matches, n_hyp, deferred, 0, match index of hypothesis 0 .. max_hyp - 1}
#define FL_RECO_SEL_HDR 4
// summary words at the head of the mapped host block: {n_matches, n_hyp, n_roi, n_results, flags, ...}, records behind them
#define FL_RECO_SUMMARY_WORDS 16
#define FL_RECO_DEFERRED 1        // flags: the list was not sorted yet when the selection ran (more records than the fused sort holds)
// hypothesis selection after the sort: hyps[0, max_hyp) (padding: status FL_ERR_STATE), sel as above.  check_big: honour the sort's
// "list not sorted" flag (d_hdr[2]); 0 when the host has just sorted the list itself.
int fl_launch_reco_select(const fl_match_t* matches, const int* d_hdr, int out_cap, int check_big, const int32_t* class_first, int n_classes,
                          int n_templates, const fl_reco_tmpl* tmpl, int top_k, int per_class, int max_hyp, int W, int H,
                          fl_icp_hyp* hyps, int* sel, cudaStream_t s);
// summary word a rank that does not own a frame of a template-sharded pipe sets to 1 + owner when the owner's results never arrived
#define FL_RECO_MISSING_OWNER 5
// Result mailbox of a template-sharded pipe (fl_pipe_set_recognition_sharded): FL_RECO_MAILBOX_WORDS words at the end of every exchange
// buffer (behind the candidate blocks, fl_exchange_buffer_bytes), and its signal, one of the signal words the candidate exchange leaves
// unused (it takes words 0 .. world - 1).  A frame's owner writes [summary | records] into the mailbox of every other rank, fences, and
// publishes the slot's exchange epoch in the signal (system-scope release); k_reco_receive acquire-waits for that epoch.
// One mailbox per slot is enough: a rank's receive of epoch e runs on the slot's stream before its exchange launch of e + 1, and the
// owner of e + 1 pushes only after its own exchange has seen every rank publish e + 1 - so no push overwrites a mailbox not yet read.
#define FL_RECO_MAILBOX_WORDS (FL_RECO_SUMMARY_WORDS + FL_RECO_MAX_HYP * (int)(sizeof(fl_reco_result_t) / 4))
#define FL_XCHG_RECO_SIGNAL (FL_XCHG_SIGNALS - 1)
inline size_t fl_reco_mailbox_offset(int world, int capacity) {
  return FL_XCHG_SIGNALS * sizeof(unsigned) + (size_t)2 * world * ((size_t)capacity + 1) * sizeof(fl_match_t);
}
// the owner's push: exchange buffers (as mapped into this process) of the n ranks that do not own the frame, and the frame's epoch
struct fl_reco_push { int n; unsigned epoch; size_t mailbox_off; uint8_t* peer[FL_XCHG_MAX_WORLD]; };
// objects that came out of ICP -> [NMS] -> fl_reco_result_t records + summary posted to mapped host memory (host_block), and with
// push != NULL (push->n > 0) into the mailbox of every rank listed there
int fl_launch_reco_finish(const fl_match_t* matches, const int* sel, const fl_icp_result_t* results, int max_hyp, float th_obj_dist,
                          int* host_block, const fl_reco_push* push, cudaStream_t s);
// a rank that does not own the frame: wait (bounded, ~2 s) for `epoch` in its own buffer's mailbox signal, then copy the mailbox into
// host_block; on time-out host_block gets an empty summary with word FL_RECO_MISSING_OWNER = 1 + owner
int fl_launch_reco_receive(const uint8_t* own_buffer, size_t mailbox_off, unsigned epoch, int owner, int* host_block, cudaStream_t s);
// load the kernels of the recognition tail and of the receive on the current device now (fl_icp_preload: k_icp_fused, with its
// shared-memory opt-in for max_pts points): a first launch under lazy module loading may wait for the device, where an exchange kernel
// can be spinning until this rank's peers arrive
int fl_reco_preload();
int fl_icp_preload(int max_pts);
// the template set a recognition set-up covers, in upload order: class, level-0 modality-0 box and pose13 (nullable) of every template.
// fl_set_recognition passes the handle's own upload, fl_group_set_recognition the whole set of a template-sharded group (api.cu).
struct fl_reco_set { int n_templates; const int32_t* class_of; const fl_rect_t* box0; const float* pose13; };
int fl_reco_setup(fl_handle* h, const fl_reco_params_t* prm, const fl_reco_set& set, const int32_t* crop_of_template, const float* pose12);
// one member's part of a group frame (api.cu): stage the frame (rescaled when src != W x H); match the staged frame over the member's shard
// + exchange + sort; on the frame's owner, the recognition tail.  The group runs each step on every member before the next one (no
// member's enqueue may wait for the device while a peer's exchange kernel spins).  Finish with fl_match_wait on every member, then
// fl_reco_shard_results on the owner.
int fl_reco_shard_stage(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int src_W, int src_H, int W, int H,
                        fl_intrinsics_t K_ref);
int fl_reco_shard_match(fl_handle* h, int rank, int world, void* const* peers, int capacity, fl_match_t* block, uint32_t epoch);
int fl_reco_shard_tail(fl_handle* h, const fl_reco_push* push = nullptr);
int fl_reco_shard_results(fl_handle* h, fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary);
// a template-sharded pipe's rank that does not own the frame: k_reco_receive in place of the tail (own_buffer: this rank's exchange
// buffer of the slot); fl_reco_shard_results then reads what the owner posted, or runs the tail itself on a deferred list
int fl_reco_shard_receive(fl_handle* h, const uint8_t* own_buffer, size_t mailbox_off, uint32_t epoch, int owner);
// after fl_reco_setup on a handle of a template-sharded pipe: every kernel the handle's recognition frames launch is loaded
int fl_reco_shard_preload(fl_handle* h);
