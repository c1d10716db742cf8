// C ABI of fealess_b200 (include/fealess_b200.h): handle lifecycle, device workspaces, and the orchestration of the
// kernels in frontend.cu / similarity.cu / icp.cu on the handle's stream.  CUDA only - there is no CPU path here.
#include "fl_internal.cuh"
#include "fl_owned.cuh"
#include "resize_tables.h"
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <climits>
#include <cmath>
#include <memory>
#include <new>
#include <vector>


static thread_local char g_err[512] = "";
void fl_set_error(const char* fmt, ...) {
  va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof g_err, fmt, ap); va_end(ap);
}
extern "C" const char* fl_last_error(void) { return g_err; }
// Programmatic dependent launch for every kernel of the pipeline was measured neutral (126.7 vs 125.8 us per frame: the boundaries
// cost ~1.5 us each and griddepcontrol.wait still has to see the previous grid drain); only the similarity kernel, whose prologue is
// long enough to matter, is launched that way (similarity_staged.cu).
extern "C" const char* fl_version(void) { return "fealess_b200 0.1 (sm_100a)"; }

#define FETCH_FIRST 1024   // matches copied back together with the count in the common case

// ICP workspace, replaced as a whole when it grows (icp_reserve): what fl_handle::icp points into, the batch buffers and their host staging
struct fl_icp_bufs {
  fl_dev_buf<float> pts_ref, pts_mod, cor_m, cor_r, dist, nn_d2; fl_dev_buf<float4> grid_pts; fl_dev_buf<int> nn_slot, n_ref, n_mod, d_ticket;
  fl_dev_buf<fl_icp_hyp> d_hyps; fl_dev_buf<fl_icp_result_t> d_results; fl_dev_buf<uint16_t> d_model_crops; fl_dev_buf<unsigned long long> d_trace;
  fl_pinned_buf<uint16_t> h_model_crops; fl_pinned_buf<fl_icp_hyp> h_hyps; fl_pinned_buf<fl_icp_result_t> h_results;
};

// What d_in_bgr / d_in_depth hold: the last host frame staged on the handle (stage_host).  Its depth counts as "the matched frame" - the
// reference depth of fl_detection_batch_resident(_device) with ref_depth == NULL - only once an enqueue that used it has succeeded.
struct fl_staged_frame { int W = 0, H = 0; bool bgr = false, depth = false, matched = false; };

// The frame in flight (fl_frame_kind), from the enqueue that starts it (frame_begin) to fl_frame_wait.  The fields stay valid after the
// wait: a recognition frame's tail may run again on them, and a group re-runs its members' staged frames.
struct fl_frame {
  fl_frame_kind kind = fl_frame_kind::none;
  // the sort half (sort_launch -> sort_finish): own = the first matches go to this handle's mapped block too; fused = the launch also
  // refined the candidates (k_refine_sort, whose last CTA sorts at most 1,024 records)
  fl_lists lists = {}; fl_match_t* out = nullptr; int out_cap = 0; int* out_count = nullptr; bool own = false, fused = false;
  // what a front-end time-out re-runs; rerun = the frame was matched on this handle alone (one that exchanged with peers needs every rank)
  bool rerun = false; const void* bgr = nullptr; const void* depth = nullptr; int W = 0, H = 0; const void* masks[FL_MAX_MODALITIES] = {};
  float threshold = 0.f; std::vector<int32_t> filter;
  fl_intrinsics_t K = {};                                  // recognition frames: the intrinsics of the staged frame
};

// Every resource has one owner (fl_owned.cuh); plan, icp, rz, d_out(_count), h_small, h_first, d_reco_host point into them.
struct fl_handle {
  fl_owned_stream stream;                                  // declared first: destroyed last, after everything used on it
  fl_params_t p = {};
  int64_t launches = 0;
  // template database
  int n_templates = 0, n_features = 0, n_classes = 0;
  fl_dev_buf<fl_template_hdr_t> d_hdr; fl_dev_buf<fl_feature_t> d_feat; fl_dev_buf<int32_t> d_class_of, d_class_first; fl_dev_buf<uint8_t> d_class_enabled;
  fl_dev_buf<fl_pfeat> d_pfeat; fl_dev_buf<int32_t> d_tid_of; fl_dev_buf<uint8_t> d_rrec;
  std::vector<int32_t> tid_of_h;
  std::vector<int32_t> coarse_wh;                          // (width, height) of every template at the coarsest level
  bool staged_eligible = false, use_staged = false; int n_sm = 0; int force_baseline = 0;   // staged global-similarity kernel (similarity_staged.cu)
  fl_staged_plan plan = {};
  fl_dev_buf<uint32_t> plan_gfeat; fl_dev_buf<uint8_t> plan_gpre; fl_dev_buf<int4> plan_gmeta; fl_dev_buf<unsigned long long> plan_trace;
  std::vector<int32_t> class_first_h, class_of_h;
  std::vector<float> pose13_h;
  std::vector<uint8_t> class_enabled_h; bool class_enabled_valid = false;   // host mirror of d_class_enabled
  // geometry of the last frame
  int gW = 0, gH = 0; bool packed = false;
  fl_level_geom geom[FL_MAX_LEVELS] = {}; fl_dev_buf<fl_level_geom> d_geom;
  // frame-sized buffers
  fl_dev_buf<uint8_t> d_in_bgr; fl_dev_buf<uint16_t> d_in_depth;   // staging for host-input calls
  fl_dev_buf<uint8_t> d_bgr[FL_MAX_LEVELS];                        // colour pyramid, levels >= 1
  fl_dev_buf<uint8_t> d_q[FL_MAX_LEVELS][FL_MAX_MODALITIES];       // quantised images (unmasked: a frame's masks apply in the spread jobs and at read-back)
  // masks, sized at fl_create: level 0 = the staged masks of host-input frames, levels >= 1 = the NN mask pyramid of a geometry that
  // does not halve exactly (the resize jobs of the front end, frontend.cu)
  fl_dev_buf<uint8_t> d_mask[FL_MAX_LEVELS][FL_MAX_MODALITIES];
  fl_dev_buf<uint8_t> d_spread[FL_MAX_LEVELS][FL_MAX_MODALITIES];  // debug only
  fl_dev_buf<uint8_t> d_lm[FL_MAX_LEVELS]; fl_dev_buf<uint8_t> d_lm4;   // d_lm4: 4-bit copy of the coarsest level's linear memories
  fl_dev_buf<uint32_t> d_mass;                                         // response mass of the coarsest level (FL_MASS_*): the staged kernel's phase order
  const uint8_t* frame_mask[FL_MAX_MODALITIES] = {};               // level-0 mask (device memory) of the last frame's modality m, or NULL
  bool keep_spread = false;
  fl_frame frame; fl_staged_frame staged;
  fl_fe_owned fe;                                           // the front end's dependency counters, time-out flag, timeline and switches
  bool opt_split_refine = false, opt_trace = false, opt_no_prune = false, opt_rotate = false;   // fl_debug_option
  // candidates / matches
  fl_dev_buf<fl_match_t> d_cand; fl_dev_buf<int> d_count; fl_dev_buf<fl_sort_key> d_keys; int key_cap = 0; fl_dev_buf<uint8_t> d_outblk; fl_match_t* d_out = nullptr; int* d_out_count = nullptr;   // d_outblk = [16-int summary][matches]
  // pinned host staging
  fl_pinned_buf<uint8_t> h_bgr; fl_pinned_buf<uint16_t> h_depth; fl_pinned_buf<uint8_t> h_mask, h_outblk, h_class_enabled; int* h_small = nullptr; fl_match_t* h_first = nullptr;   // h_small/h_first point into h_outblk
  bool have_result = false, overflow = false;              // the last completed frame: its list can be fetched; it overflowed a buffer
  // profiling
  bool profile = false; fl_owned_event ev[5]; float stage_ms[4] = {}; float icp_ms = 0.f;
  // ICP workspace (grown on demand)
  int icp_hyp_cap = 0, icp_pts_cap = 0;
  fl_icp_ws icp = {}; fl_icp_bufs icpw; int icp_trace_n = 0; fl_dev_buf<uint16_t> d_ref_depth;
  // rendered template depth crops kept on the device (fl_upload_model_depths)
  fl_dev_buf<uint16_t> d_resident; std::vector<size_t> res_off; std::vector<fl_rect_t> res_rect; int res_W = 0, res_H = 0;
  fl_dev_buf<int32_t> d_nms; int nms_cap = 0;   // fl_nms workspace (hypotheses)
  bool blocking_wait = false; fl_owned_event ev_block;   // fl_set_blocking_wait
  fl_dev_buf<uint8_t> d_train;                           // fl_add_template workspace (allocated at the first call)
  // input rescale: device tables of the current (source -> destination) geometry, source-frame staging
  fl_resize_tables rz = {}; int rz_sW = 0, rz_sH = 0, rz_dW = 0, rz_dH = 0;
  fl_dev_buf<int> rz_xofs, rz_yofs; fl_dev_buf<short2> rz_ialpha, rz_ibeta; fl_dev_buf<float2> rz_alpha, rz_beta;
  fl_dev_buf<uint8_t> d_src_bgr; fl_dev_buf<uint16_t> d_src_depth;
  // Recognition on the device (fl_set_recognition, fl_recognize_*): per-template table, per-frame selection state, mapped host block
  // [summary | records] (+ its device alias)
  bool custom_tids = false, reco_set = false, reco_any_crop = false; fl_reco_params_t reco = {}; int reco_max_hyp = 0;
  fl_dev_buf<fl_reco_tmpl> d_reco_tmpl; fl_dev_buf<int> d_reco_sel; fl_mapped_buf<int> h_reco; int* d_reco_host = nullptr;
  // the template set the selection table covers: the handle's own upload, or the whole set of a template-sharded group, whose merged
  // list this handle selects from (fl_group_set_recognition)
  int reco_n_templates = 0, reco_n_classes = 0; fl_dev_buf<int32_t> d_reco_class_first;
};

// The host waits for the handle's stream.  Default: cudaStreamSynchronize (the runtime spins - lowest latency, one busy core per
// waiting thread).  fl_set_blocking_wait(h, 1): an event created with cudaEventBlockingSync, so the thread sleeps until the GPU's
// interrupt - for hosts that keep more frames in flight (threads) than they have cores to spin on.
static cudaError_t wait_stream(fl_handle* h);
#define TRY(x) do { int rc__ = (x); if (rc__ != FL_OK) return rc__; } while (0)
// (re)allocates the owner of a buffer that a kernel argument struct points to, and points `field` at it (NULL on failure)
template <typename O, typename T> static int alloc_into(O& o, size_t n, T** field, const char* file = __builtin_FILE(), int line = __builtin_LINE()) { *field = nullptr; TRY(o.alloc(n, file, line)); *field = o.get(); return FL_OK; }

extern "C" void fl_default_params(fl_params_t* p) {
  memset(p, 0, sizeof *p);
  p->n_levels = 2; p->T[0] = 5; p->T[1] = 8;                                   // T_DEFAULTS, linemod.cpp:1820
  p->n_modalities = 2; p->modality_kind[0] = FL_MODALITY_COLOR_GRADIENT; p->modality_kind[1] = FL_MODALITY_DEPTH_NORMAL;
  p->weak_threshold = 10.0f; p->distance_threshold = 2000; p->difference_threshold = 50;
  p->max_width = 640; p->max_height = 480; p->max_candidates = 1 << 16; p->device = 0;
}

static size_t level_lm_bytes(const fl_params_t& p, int l, int W, int H, fl_level_geom* g) {
  fl_level_geom gg;
  gg.W = W >> l; gg.H = H >> l; gg.T = p.T[l];
  gg.Wd = gg.W / gg.T; gg.Hd = gg.H / gg.T; gg.cells = gg.Wd * gg.Hd;
  size_t ls = (size_t)gg.T * gg.T * gg.cells + FL_LM_PAD;
  gg.label_stride = (ls + 31) & ~(size_t)31;
  gg.mod_stride = gg.label_stride * 8;
  if (g) *g = gg;
  return gg.mod_stride * p.n_modalities;
}

extern "C" int fl_create(const fl_params_t* params, fl_handle** out) {
  if (!params || !out) return FL_ERR_ARG;
  *out = nullptr;
  const fl_params_t& p = *params;
  if (p.n_levels < 1 || p.n_levels > FL_MAX_LEVELS || p.n_modalities < 1 || p.n_modalities > FL_MAX_MODALITIES) return FL_ERR_ARG;
  for (int l = 0; l < p.n_levels; ++l) if (p.T[l] < 1 || p.T[l] > FL_MAX_T) return FL_ERR_ARG;
  for (int m = 0; m < p.n_modalities; ++m) if (p.modality_kind[m] != FL_MODALITY_COLOR_GRADIENT && p.modality_kind[m] != FL_MODALITY_DEPTH_NORMAL) return FL_ERR_ARG;
  if (p.max_width < 16 || p.max_height < 16 || p.max_candidates < 1) return FL_ERR_ARG;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0 || p.device < 0 || p.device >= ndev) {
    fl_set_error("no usable CUDA device (count=%d, requested %d): %s", ndev, p.device, cudaGetErrorString(e));
    return FL_ERR_CUDA;
  }
  FL_CUDA(cudaSetDevice(p.device));
  std::unique_ptr<fl_handle> h(new (std::nothrow) fl_handle());   // a failure below deletes what was built
  if (!h) return FL_ERR_ARG;
  h->p = p; fl_default_reco_params(&h->reco);
  { cudaDeviceProp prop; FL_CUDA(cudaGetDeviceProperties(&prop, p.device)); h->n_sm = prop.multiProcessorCount; }
  TRY(h->stream.create(cudaStreamNonBlocking));
  for (fl_owned_event& e : h->ev) TRY(e.create(cudaEventDefault));
  TRY(fl_launch_tables_init());
  const size_t npx = (size_t)p.max_width * p.max_height;
  TRY(h->d_in_bgr.alloc(npx * 3)); TRY(h->d_in_depth.alloc(npx));
  TRY(h->d_geom.alloc(FL_MAX_LEVELS));
  for (int l = 0; l < p.n_levels; ++l) {
    size_t n = (size_t)(p.max_width >> l) * (p.max_height >> l);
    if (l > 0) TRY(h->d_bgr[l].alloc(n * 3));
    for (int m = 0; m < p.n_modalities; ++m) { TRY(h->d_q[l][m].alloc(n)); TRY(h->d_mask[l][m].alloc(n)); }
    // linear memories: T need not divide the maximum size, so bound the cell count from above
    int T = p.T[l];
    size_t cells = (size_t)(((p.max_width >> l) + T - 1) / T) * (((p.max_height >> l) + T - 1) / T);
    size_t ls = (((size_t)T * T * cells + FL_LM_PAD) + 31) & ~(size_t)31;
    TRY(h->d_lm[l].alloc(ls * 8 * p.n_modalities + cells + 256));   // slack: windowed reads may run one map past the last label
    if (l == p.n_levels - 1) {
      // 4-bit copy of the coarsest level's linear memories (two cells per byte), read by the staged similarity kernel
      TRY(h->d_lm4.alloc(h->d_lm[l].capacity() / 2 + 256));
      FL_CUDA(cudaMemset(h->d_lm4.get(), 0, h->d_lm4.capacity()));
    }
  }
  TRY(h->d_mass.alloc(FL_MASS_WORDS));
  FL_CUDA(cudaMemset(h->d_mass.get(), 0, FL_MASS_WORDS * sizeof(uint32_t)));
  TRY(h->d_cand.alloc((size_t)p.max_candidates)); TRY(h->d_count.alloc(4));   // [0] candidate count, [1] CTA ticket counter of k_refine_sort
  FL_CUDA(cudaMemset(h->d_count.get(), 0, 4 * sizeof(int)));
  TRY(fl_fe_create(&h->fe));
  int kc = 2; while (kc < p.max_candidates) kc <<= 1;
  h->key_cap = kc;
  TRY(h->d_keys.alloc((size_t)kc + 1));      // + room for the two scratch ints behind the keys
  TRY(h->d_outblk.alloc(64 + (size_t)p.max_candidates * sizeof(fl_match_t)));
  FL_CUDA(cudaMemset(h->d_outblk.get(), 0, 64));                                   // summary words, incl. the fused-tail overflow flag
  h->d_out_count = reinterpret_cast<int*>(h->d_outblk.get()); h->d_out = reinterpret_cast<fl_match_t*>(h->d_outblk.get() + 64);
  TRY(h->h_bgr.alloc(npx * 3)); TRY(h->h_depth.alloc(npx)); TRY(h->h_mask.alloc(npx * p.n_modalities));
  TRY(h->h_outblk.alloc(64 + FETCH_FIRST * sizeof(fl_match_t))); TRY(h->h_class_enabled.alloc(4096));
  h->h_small = reinterpret_cast<int*>(h->h_outblk.get()); h->h_first = reinterpret_cast<fl_match_t*>(h->h_outblk.get() + 64);
  *out = h.release();
  return FL_OK;
}

extern "C" int fl_destroy(fl_handle* h) {
  if (!h) return FL_OK;
  cudaSetDevice(h->p.device);
  cudaStreamSynchronize(h->stream.get());
  delete h;
  return FL_OK;
}

static cudaError_t wait_stream(fl_handle* h) {
  if (!h->blocking_wait) return cudaStreamSynchronize(h->stream.get());
  cudaError_t e = cudaEventRecord(h->ev_block.get(), h->stream.get());
  return e == cudaSuccess ? cudaEventSynchronize(h->ev_block.get()) : e;
}
extern "C" int fl_set_blocking_wait(fl_handle* h, int enable) {
  if (!h) return FL_ERR_ARG;
  FL_CUDA(cudaSetDevice(h->p.device));
  if (enable && !h->ev_block.get()) TRY(h->ev_block.create(cudaEventBlockingSync | cudaEventDisableTiming));
  h->blocking_wait = enable != 0;
  return FL_OK;
}
extern "C" int fl_sync(fl_handle* h) { if (!h) return FL_ERR_ARG; FL_CUDA(cudaStreamSynchronize(h->stream.get())); return FL_OK; }
extern "C" void* fl_stream(fl_handle* h) { return h ? (void*)h->stream.get() : nullptr; }
extern "C" int64_t fl_launch_count(fl_handle* h) { return h ? h->launches : 0; }
int fl_entries_per_template(const fl_handle* h) { return h ? h->p.n_levels * h->p.n_modalities : 0; }
fl_frame_kind fl_frame_in_flight(const fl_handle* h) { return h ? h->frame.kind : fl_frame_kind::none; }
// One frame in flight per handle: its wait reads the frame record, and a host frame would overwrite staging buffers it may still read.
static int frame_idle(const fl_handle* h) {
  if (h->frame.kind == fl_frame_kind::none) return FL_OK;
  fl_set_error("a frame is in flight on this handle: wait for it first (fl_match_wait or fl_recognize_wait)");
  return FL_ERR_STATE;
}
// the start of every entry point that enqueues frame work: nothing in flight, the handle's device, and the last frame's result is gone
static int frame_begin(fl_handle* h) {
  TRY(frame_idle(h));
  FL_CUDA(cudaSetDevice(h->p.device));
  h->have_result = h->overflow = false;
  return FL_OK;
}
extern "C" int fl_profile(fl_handle* h, int enable) { if (!h) return FL_ERR_ARG; h->profile = enable != 0; return FL_OK; }
extern "C" int fl_last_icp_ms(fl_handle* h, float* ms) { if (!h || !ms) return FL_ERR_ARG; *ms = h->icp_ms; return FL_OK; }
extern "C" int fl_debug_icp_trace(fl_handle* h, uint64_t* out, int32_t n_hyp) {
  if (!h || !out || n_hyp < 0) return FL_ERR_ARG;
  if (!h->icpw.d_trace.get() || n_hyp > h->icp_trace_n) { fl_set_error("no ICP phase clock: call fl_profile(h, 1) before the batch"); return FL_ERR_STATE; }
  FL_CUDA(cudaSetDevice(h->p.device));
  FL_CUDA(cudaMemcpy(out, h->icpw.d_trace.get(), (size_t)n_hyp * FL_ICP_TRACE_WORDS * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  return FL_OK;
}
extern "C" int fl_last_stage_ms(fl_handle* h, float out4[4]) { if (!h || !out4) return FL_ERR_ARG; memcpy(out4, h->stage_ms, sizeof h->stage_ms); return FL_OK; }
// 1 = always use the baseline (L1/L2-fed) global similarity kernel; 0 = use the shared-memory-staged kernel when eligible
extern "C" int fl_debug_force_baseline(fl_handle* h, int enable) { if (!h) return FL_ERR_ARG; h->force_baseline = enable != 0; h->packed = false; return FL_OK; }
extern "C" int fl_debug_uses_staged(fl_handle* h) { return h ? (h->use_staged ? 1 : 0) : FL_ERR_ARG; }
extern "C" int fl_debug_plan_staged(int W, int H, int T, int n_modalities, int n_templates, int max_positions, int n_sm, int32_t out[16]) {
  if (!out || T < 1 || T > FL_MAX_T || W < T || H < T || W % T || H % T || (int64_t)W * H > INT32_MAX || n_modalities < 1 ||
      n_modalities > FL_MAX_MODALITIES || n_sm < 1)
    return FL_ERR_ARG;
  memset(out, 0, 16 * sizeof(int32_t));
  fl_params_t p;
  fl_default_params(&p);
  p.n_levels = 1; p.T[0] = T; p.n_modalities = n_modalities;
  fl_level_geom g;
  level_lm_bytes(p, 0, W, H, &g);                              // the geometry ensure_geometry builds for the coarsest level
  fl_staged_plan pl;
  if (!fl_plan_staged(g, n_modalities, n_templates, max_positions, n_sm, &pl)) return 0;
  const int32_t v[] = {pl.nw_template, pl.tpw, pl.tpc, pl.n_cta, pl.block_threads, pl.phase_rows, pl.n_rowblocks, pl.labels_per_phase,
                       pl.n_phases, pl.n_buf, pl.buf_bytes, pl.halo_bytes, pl.smem_bytes};
  memcpy(out, v, sizeof v);
  return 1;
}
// developer options of one handle (all off by default; each one is exercised by tests/test_gpu_match.py::test_debug_options)
extern "C" int fl_debug_option(fl_handle* h, int option, int value) {
  if (!h) return FL_ERR_ARG;
  switch (option) {
    case FL_OPT_FE_WAVES: case FL_OPT_FE_DEP_TIMEOUT_TEST: case FL_OPT_FE_FORCED_WAVES: return fl_fe_option(h->fe.get(), option, value);
    case FL_OPT_SPLIT_REFINE: h->opt_split_refine = value != 0; return FL_OK;
    case FL_OPT_TRACE: h->opt_trace = value != 0; h->packed = false; return FL_OK;     // (the staged plan allocates its timeline at planning time)
    case FL_OPT_SIM_NO_PRUNE: h->opt_no_prune = value != 0; return FL_OK;
    case FL_OPT_SIM_ROTATE: h->opt_rotate = value != 0; return FL_OK;
  }
  return FL_ERR_ARG;
}
extern "C" int fl_debug_keep_spread(fl_handle* h, int enable) { if (!h) return FL_ERR_ARG; h->keep_spread = enable != 0; return FL_OK; }
extern "C" int fl_num_templates(fl_handle* h) { return h ? h->n_templates : FL_ERR_ARG; }

// ---------------------------------------------------------------------------------------------------
extern "C" int fl_upload_templates(fl_handle* h, int32_t n_templates, const fl_template_hdr_t* headers, const fl_feature_t* features,
                                   int32_t n_features, const int32_t* class_of, const float* pose13) {
  if (!h || n_templates < 0 || n_features < 0 || (n_templates > 0 && (!headers || !class_of)) || (n_features > 0 && !features)) return FL_ERR_ARG;
  FL_CUDA(cudaSetDevice(h->p.device));
  const int L = h->p.n_levels, M = h->p.n_modalities;
  const size_t ne = (size_t)n_templates * L * M;
  int nc = 0;
  for (int t = 0; t < n_templates; ++t) { if (class_of[t] < 0) return FL_ERR_ARG; nc = std::max(nc, class_of[t] + 1); }
  if (nc > 4096) return FL_ERR_ARG;
  std::vector<int32_t> first(nc, -1);
  for (int t = 0; t < n_templates; ++t) {
    int c = class_of[t];
    if (first[c] < 0) first[c] = t; else if (class_of[t - 1] != c) { fl_set_error("templates of class %d are not contiguous", c); return FL_ERR_ARG; }
  }
  for (size_t e = 0; e < ne; ++e) {
    const fl_template_hdr_t& hd = headers[e];
    if (hd.feature_begin < 0 || hd.feature_count < 0 || (int64_t)hd.feature_begin + hd.feature_count > n_features) return FL_ERR_ARG;
    if (hd.feature_count > 63) return FL_ERR_FEATURES;                          // CV_Assert(features.size() <= 63)
    for (int k = 0; k < hd.feature_count; ++k) { int lab = features[hd.feature_begin + k].label; if (lab < 0 || lab > 7) return FL_ERR_ARG; }
  }
  // eligibility for the shared-memory-staged global similarity kernel: u8 totals cannot overflow, one template_positions
  // per template, and every coarsest-level feature inside its template's box (keeps flat over-reads within the staged halo)
  bool eligible = n_templates > 0;
  for (int t = 0; t < n_templates && eligible; ++t) {
    const fl_template_hdr_t* hd = headers + ((size_t)t * L + (L - 1)) * M;
    int nf = 0;
    for (int m = 0; m < M; ++m) {
      nf += hd[m].feature_count;
      if (hd[m].width != hd[0].width || hd[m].height != hd[0].height || hd[m].width < 1 || hd[m].height < 1) eligible = false;
      for (int k = 0; k < hd[m].feature_count; ++k) {
        const fl_feature_t& f = features[hd[m].feature_begin + k];
        if (f.x < 0 || f.y < 0 || f.x > hd[m].width || f.y > hd[m].height) eligible = false;
      }
    }
    if (nf > 63) eligible = false;
  }
  FL_CUDA(cudaStreamSynchronize(h->stream.get()));
  h->n_templates = h->n_features = h->n_classes = 0; h->packed = h->use_staged = h->staged_eligible = h->reco_set = false;
  memset(&h->plan, 0, sizeof h->plan);
  h->d_hdr.reset(); h->d_feat.reset(); h->d_class_of.reset(); h->d_class_first.reset(); h->d_class_enabled.reset(); h->d_pfeat.reset(); h->d_rrec.reset();
  h->d_tid_of.reset(); h->plan_gfeat.reset(); h->plan_gpre.reset(); h->plan_gmeta.reset(); h->plan_trace.reset();
  h->staged_eligible = eligible;
  h->coarse_wh.resize((size_t)n_templates * 2);
  for (int t = 0; t < n_templates; ++t) {
    const fl_template_hdr_t& hd = headers[((size_t)t * L + (L - 1)) * M];
    h->coarse_wh[2 * t] = hd.width; h->coarse_wh[2 * t + 1] = hd.height;
  }
  TRY(h->d_hdr.alloc(ne)); TRY(h->d_feat.alloc((size_t)n_features)); TRY(h->d_class_of.alloc((size_t)n_templates));
  TRY(h->d_class_first.alloc((size_t)nc)); TRY(h->d_class_enabled.alloc((size_t)std::max(nc, 1))); TRY(h->d_pfeat.alloc((size_t)n_features));
  if (ne) FL_CUDA(cudaMemcpy(h->d_hdr.get(), headers, ne * sizeof(fl_template_hdr_t), cudaMemcpyHostToDevice));
  if (n_features) FL_CUDA(cudaMemcpy(h->d_feat.get(), features, (size_t)n_features * sizeof(fl_feature_t), cudaMemcpyHostToDevice));
  if (n_templates) FL_CUDA(cudaMemcpy(h->d_class_of.get(), class_of, (size_t)n_templates * sizeof(int32_t), cudaMemcpyHostToDevice));
  if (nc) FL_CUDA(cudaMemcpy(h->d_class_first.get(), first.data(), (size_t)nc * sizeof(int32_t), cudaMemcpyHostToDevice));
  h->tid_of_h.resize((size_t)n_templates);
  for (int t = 0; t < n_templates; ++t) h->tid_of_h[t] = t - first[class_of[t]];                // matchClass numbering (:1458)
  TRY(h->d_tid_of.alloc((size_t)n_templates));
  if (n_templates) FL_CUDA(cudaMemcpy(h->d_tid_of.get(), h->tid_of_h.data(), (size_t)n_templates * sizeof(int32_t), cudaMemcpyHostToDevice));
  h->n_templates = n_templates; h->n_features = n_features; h->n_classes = nc;
  h->class_first_h = first; h->class_of_h.assign(class_of, class_of + n_templates);
  h->pose13_h.clear();
  if (pose13) h->pose13_h.assign(pose13, pose13 + (size_t)n_templates * 13);
  h->class_enabled_h.assign((size_t)std::max(nc, 1), 1); h->class_enabled_valid = false;
  h->custom_tids = false;
  return FL_OK;
}

extern "C" int fl_set_template_ids(fl_handle* h, const int32_t* template_ids) {
  if (!h || !template_ids) return FL_ERR_ARG;
  if (h->n_templates == 0) return FL_OK;
  FL_CUDA(cudaSetDevice(h->p.device));
  FL_CUDA(cudaStreamSynchronize(h->stream.get()));
  for (int t = 0; t < h->n_templates; ++t) if (template_ids[t] < 0) return FL_ERR_ARG;
  h->tid_of_h.assign(template_ids, template_ids + h->n_templates);
  h->custom_tids = true; h->reco_set = false;
  FL_CUDA(cudaMemcpy(h->d_tid_of.get(), template_ids, (size_t)h->n_templates * sizeof(int32_t), cudaMemcpyHostToDevice));
  return FL_OK;
}

extern "C" int fl_get_pose_info(fl_handle* h, int32_t class_idx, int32_t template_id, float out13[13]) {
  if (!h || !out13 || class_idx < 0 || class_idx >= h->n_classes || h->pose13_h.empty()) return FL_ERR_ARG;
  // the reference keeps ONE flat TemplatePoseInfo indexed by the per-class template_id (linemod.cpp:1624-1634), which is
  // wrong for more than one class (SURVEY A.6 iv); this ABI keys the pose by (class, template_id).
  int t = -1;
  for (int k = h->class_first_h[class_idx]; k >= 0 && k < h->n_templates && h->class_of_h[k] == class_idx; ++k)
    if (h->tid_of_h[k] == template_id) { t = k; break; }
  if (t < 0) return FL_ERR_ARG;
  memcpy(out13, &h->pose13_h[(size_t)t * 13], 13 * sizeof(float));
  return FL_OK;
}

static fl_tdb make_tdb(fl_handle* h) {
  fl_tdb db;
  db.n_templates = h->n_templates; db.L = h->p.n_levels; db.M = h->p.n_modalities; db.n_classes = h->n_classes;
  db.hdr = h->d_hdr.get(); db.feat = h->d_feat.get(); db.class_of = h->d_class_of.get(); db.class_first = h->d_class_first.get();
  db.class_enabled = h->d_class_enabled.get(); db.pfeat = h->d_pfeat.get(); db.tid_of = h->d_tid_of.get();
  db.rrec = h->d_rrec.get(); db.rrec_bytes = fl_rrec_bytes(h->p.n_modalities);
  return db;
}

// largest template_positions (linemod.cpp:1155) of the uploaded templates at the coarsest level of the current geometry
static int max_positions(const fl_handle* h) {
  const fl_level_geom& g = h->geom[h->p.n_levels - 1];
  int best = 0;
  for (size_t t = 0; t + 1 < h->coarse_wh.size(); t += 2) {
    const int wf = (h->coarse_wh[t] - 1) / g.T + 1, hf = (h->coarse_wh[t + 1] - 1) / g.T + 1;
    best = std::max(best, std::min((g.Hd - hf) * g.Wd + (g.Wd - wf) + 1, g.cells));
  }
  return best;
}

static int ensure_geometry(fl_handle* h, int W, int H) {
  const fl_params_t& p = h->p;
  if (W <= 0 || H <= 0 || W > p.max_width || H > p.max_height) { fl_set_error("frame %dx%d exceeds handle capacity %dx%d", W, H, p.max_width, p.max_height); return FL_ERR_SIZE; }
  for (int l = 0; l < p.n_levels; ++l) {                                        // CV_Asserts :981, :1062-1063
    int w = W >> l, hh = H >> l, T = p.T[l];
    if (w < 1 || hh < 1 || w % T || hh % T || (w * hh) % 16) return FL_ERR_GEOMETRY;
  }
  if (W != h->gW || H != h->gH) {
    for (int l = 0; l < p.n_levels; ++l) {
      size_t need = level_lm_bytes(p, l, W, H, &h->geom[l]);
      if (need > h->d_lm[l].capacity()) { fl_set_error("internal: LM capacity"); return FL_ERR_CAPACITY; }
      FL_CUDA(cudaMemsetAsync(h->d_lm[l].get(), 0, h->d_lm[l].capacity(), h->stream.get()));       // pads must read as zero
      if (l == p.n_levels - 1) FL_CUDA(cudaMemsetAsync(h->d_lm4.get(), 0, h->d_lm4.capacity(), h->stream.get()));
    }
    FL_CUDA(cudaMemcpyAsync(h->d_geom.get(), h->geom, sizeof(fl_level_geom) * p.n_levels, cudaMemcpyHostToDevice, h->stream.get()));
    FL_CUDA(cudaStreamSynchronize(h->stream.get()));                                  // h->geom is pageable
    h->gW = W; h->gH = H; h->packed = false;
  }
  if (!h->packed) {
    TRY(fl_fe_forget_rows(h->fe.get(), h->stream.get()));
    if (h->n_templates == 0) h->packed = true;
  }
  if (!h->packed && h->n_templates > 0) {
    fl_launch_pack_features(make_tdb(h), h->d_geom.get(), h->n_features, h->stream.get()); ++h->launches;
    if (p.n_levels > 1) {
      TRY(h->d_rrec.grow((size_t)h->n_templates * (p.n_levels - 1) * fl_rrec_bytes(p.n_modalities)));
      fl_launch_pack_refine_records(make_tdb(h), h->d_geom.get(), h->stream.get()); ++h->launches;
    }
    h->use_staged = false;
    fl_staged_plan plan;
    if (h->staged_eligible && !h->force_baseline && h->n_templates >= 256 &&
        fl_plan_staged(h->geom[p.n_levels - 1], p.n_modalities, h->n_templates, max_positions(h), h->n_sm, &plan)) {
      h->plan = plan; h->plan_trace.reset();
      TRY(alloc_into(h->plan_gfeat, (size_t)h->n_templates * 64, &h->plan.gfeat));
      TRY(alloc_into(h->plan_gpre, (size_t)h->n_templates * plan.pre_stride, &h->plan.gpre));
      TRY(alloc_into(h->plan_gmeta, (size_t)h->n_templates, &h->plan.gmeta));
      if (h->opt_trace) {                                                        // developer timeline of the staged kernel (FL_DBG_STAGED_TRACE)
        TRY(alloc_into(h->plan_trace, (size_t)plan.n_cta * 136 + 8, &h->plan.trace));   // + stamps of a 1-thread kernel before / after the launch
        FL_CUDA(cudaMemsetAsync(h->plan.trace, 0, ((size_t)plan.n_cta * 136 + 8) * sizeof(unsigned long long), h->stream.get()));
      }
      fl_launch_pack_staged(make_tdb(h), h->geom[p.n_levels - 1], h->plan, h->stream.get()); ++h->launches;
      h->use_staged = true;
    }
    h->packed = true;
  }
  return FL_OK;
}

// front end + matchClass on the handle's templates; candidates land in (cand, count)
// defer_refine: leave the candidates at the coarsest level; the caller refines them in the same launch that sorts (k_refine_sort)
static int run_match_stages(fl_handle* h, const uint8_t* d_bgr, const uint16_t* d_depth, int W, int H, const void* const* d_masks,
                            float threshold, const int32_t* class_filter, int n_filter, fl_match_t* cand, int cap, int* d_count,
                            bool defer_refine = false) {
  const fl_params_t& p = h->p;
  FL_CUDA(cudaSetDevice(p.device));
  TRY(ensure_geometry(h, W, H));
  cudaStream_t s = h->stream.get();
  for (int m = 0; m < p.n_modalities; ++m) {
    if (p.modality_kind[m] == FL_MODALITY_COLOR_GRADIENT && !d_bgr) return FL_ERR_SIZE;
    if (p.modality_kind[m] == FL_MODALITY_DEPTH_NORMAL && !d_depth) return FL_ERR_SIZE;
  }
  // class filter (Detector::match :1418-1434): unknown ids are ignored, empty = all.  Uploaded only when it changes.
  if (h->n_classes > 0) {
    bool changed = false;
    for (int c = 0; c < h->n_classes; ++c) {
      uint8_t on = (n_filter > 0 && class_filter) ? 0 : 1;
      if (n_filter > 0 && class_filter) for (int k = 0; k < n_filter; ++k) if (class_filter[k] == c) on = 1;
      if (h->class_enabled_h[c] != on) { h->class_enabled_h[c] = on; changed = true; }
    }
    if (changed || !h->class_enabled_valid) {
      FL_CUDA(cudaStreamSynchronize(s));                                          // the pinned staging copy may still be in flight
      memcpy(h->h_class_enabled.get(), h->class_enabled_h.data(), (size_t)h->n_classes);
      FL_CUDA(cudaMemcpyAsync(h->d_class_enabled.get(), h->h_class_enabled.get(), (size_t)h->n_classes, cudaMemcpyHostToDevice, s));
      h->class_enabled_valid = true;
    }
  }
  if (h->profile) cudaEventRecord(h->ev[0].get(), s);
  fl_fe_frame fe = {};
  fe.n_levels = p.n_levels; fe.n_modalities = p.n_modalities; fe.modality_kind = p.modality_kind; fe.geom = h->geom; fe.bgr = d_bgr; fe.depth = d_depth;
  for (int l = 0; l < p.n_levels; ++l) {
    fe.bgr_pyr[l] = h->d_bgr[l].get(); fe.lm[l] = h->d_lm[l].get();
    for (int m = 0; m < p.n_modalities; ++m) {
      fe.q[l][m] = h->d_q[l][m].get(); fe.mask_pyr[l][m] = h->d_mask[l][m].get();
      if (h->keep_spread) { TRY(h->d_spread[l][m].grow((size_t)(p.max_width >> l) * (p.max_height >> l))); fe.spread[l][m] = h->d_spread[l][m].get(); }
    }
  }
  // the frame's masks (level 0, device memory): applied where the spread jobs read the labels, so a masked frame takes the same launches
  for (int m = 0; m < p.n_modalities; ++m) fe.mask[m] = h->frame_mask[m] = d_masks ? static_cast<const uint8_t*>(d_masks[m]) : nullptr;
  fe.lm4 = (h->geom[p.n_levels - 1].Wd & 1) == 0 ? h->d_lm4.get() : nullptr;            // two cells per byte: grids of even width only
  if (h->use_staged && h->n_templates > 0) {                                   // the response sums order the staged kernel's phases; it clears them
    fe.mass = h->d_mass.get();
    const void* pf[6] = {h->plan.gfeat, h->plan.gpre, h->plan.gmeta, h->d_class_of.get(), h->d_class_enabled.get(), h->d_tid_of.get()};
    const size_t nt = (size_t)h->n_templates;
    const size_t pb[6] = {nt * 64 * sizeof(uint32_t), nt * h->plan.pre_stride, nt * sizeof(int4), nt * sizeof(int32_t), (size_t)std::max(h->n_classes, 1), nt * sizeof(int32_t)};
    memcpy(fe.prefetch, pf, sizeof pf); memcpy(fe.prefetch_bytes, pb, sizeof pb);
  }
  fe.thr_sq = p.weak_threshold * p.weak_threshold; fe.dist_thr = p.distance_threshold; fe.diff_thr = p.difference_threshold;
  fe.zero_me = d_count; fe.trace = h->opt_trace;
  TRY(fl_fe_run(h->fe.get(), fe, s, &h->launches));
  if (h->profile) cudaEventRecord(h->ev[1].get(), s);
  if (h->n_templates > 0) {
    fl_tdb db = make_tdb(h);
    const int lowest = p.n_levels - 1;
    if (h->use_staged) {
      h->plan.prune = h->opt_no_prune ? 0 : 1;
      h->plan.rotate = h->opt_rotate ? 1 : 0;
      h->plan.mass = h->d_mass.get();
      if (fl_launch_similarity_staged(db, h->geom[lowest], h->d_lm4.get(), threshold, cand, cap, d_count, h->plan, s) != 0) {
        fl_set_error("staged similarity kernel could not be configured"); return FL_ERR_CUDA;
      }
    } else {
      fl_launch_similarity_global(db, h->geom[lowest], h->d_lm[lowest].get(), threshold, cand, cap, d_count, s);
    }
    ++h->launches;
    if (h->profile) cudaEventRecord(h->ev[2].get(), s);
    if (!defer_refine)
      for (int l = p.n_levels - 2; l >= 0; --l) { fl_launch_refine_level(db, h->geom[l], l, h->d_lm[l].get(), threshold, cand, cap, d_count, s); ++h->launches; }
  } else if (h->profile) cudaEventRecord(h->ev[2].get(), s);
  if (h->profile) cudaEventRecord(h->ev[3].get(), s);
  FL_CUDA(cudaGetLastError());
  return FL_OK;
}

// sort + unique of candidate lists into (d_out, d_out_count); handles the rare > 8,192-record path; leaves
// h_small = {count, n_live, flag, raw list counts...} and, for the handle's own output block, the first matches in h_first
struct fl_refine_req { float threshold; fl_match_t* cand; int cap; const int* d_count; };   // refine these candidates in the sort launch (k_refine_sort)
// first half of sort + unique (optionally with the refinement in the same launch): enqueue only
static int sort_launch(fl_handle* h, fl_lists L, fl_match_t* d_out, int out_cap, int* d_out_count, bool fetch_first, const fl_xchg* xchg = nullptr,
                       const fl_refine_req* refine = nullptr) {
  cudaStream_t s = h->stream.get();
  const int n_lists = L.n_lists, list_cap = L.list_cap;
  if ((int64_t)n_lists * list_cap > h->key_cap) { fl_set_error("sort capacity %d < %lld", h->key_cap, (long long)n_lists * list_cap); return FL_ERR_CAPACITY; }
  int* d_hdr = reinterpret_cast<int*>(h->d_outblk.get());
  const bool own = fetch_first && d_out == h->d_out;
  // the kernel itself posts the summary and (own output block) the first matches into the mapped pinned block h_outblk
  fl_xchg X;
  memset(&X, 0, sizeof X);
  if (xchg) X = *xchg;
  if (refine) {
    fl_refine_args ra;
    memset(&ra, 0, sizeof ra);
    ra.n_levels = h->p.n_levels;
    for (int l = 0; l < h->p.n_levels; ++l) { ra.g[l] = h->geom[l]; ra.lm[l] = h->d_lm[l].get(); }
    const int nl = fl_launch_refine_sort(make_tdb(h), ra, refine->threshold, refine->cand, refine->cap, refine->d_count, h->d_count.get() + 1, h->n_sm, L, X, h->key_cap,
                                         d_out, out_cap, d_out_count, d_hdr, h->h_small, own ? h->h_first : nullptr, std::min(FETCH_FIRST, out_cap), s);
    if (nl < 0) { fl_set_error("refinement + sort launch failed: %s", cudaGetErrorString(cudaGetLastError())); return FL_ERR_CUDA; }
    h->launches += nl;
  } else {
    const int nl = fl_launch_sort_unique(L, X, h->key_cap, d_out, out_cap, d_out_count, d_hdr, h->h_small, own ? h->h_first : nullptr,
                                         std::min(FETCH_FIRST, out_cap), s);
    if (nl < 0) { fl_set_error("sort launch failed: %s", cudaGetErrorString(cudaGetLastError())); return FL_ERR_CUDA; }
    h->launches += nl;
  }
  if (h->profile) cudaEventRecord(h->ev[4].get(), s);
  // what the second half (sort_finish) needs: it runs after the host has waited for the stream
  fl_frame& f = h->frame;
  f.lists = L; f.out = d_out; f.out_cap = out_cap; f.out_count = d_out_count; f.own = own; f.fused = refine != nullptr;
  return FL_OK;
}

// second half of sort + unique: wait for the stream, read the posted summary, run the multi-kernel path if the one-CTA sort
// reported more records than it holds
static int sort_finish(fl_handle* h) {
  cudaStream_t s = h->stream.get();
  const fl_frame& f = h->frame;
  const int n_lists = f.lists.n_lists, list_cap = f.lists.list_cap;
  FL_CUDA(wait_stream(h));
  h->overflow = false;
  int n_upper = 0;
  for (int i = 0; i < std::min(n_lists, 11); ++i) { if (h->h_small[3 + i] > list_cap) h->overflow = true; n_upper += std::min(std::max(h->h_small[3 + i], 0), list_cap); }
  if (n_lists > 11) n_upper = n_lists * list_cap;
  if (h->h_small[2] && f.fused && n_upper <= 8192) {
    // the fused refinement + sort launch sorts up to 1,024 records in its last CTA; this frame has more (already refined in
    // place): run the stand-alone one-CTA sort (8,192 keys) on them.  What the first launch reported about the exchange
    // (a peer that never arrived) survives the second launch, which knows nothing about it.
    const int keep15 = h->h_small[15];
    const bool keep_overflow = h->overflow;
    TRY(sort_launch(h, f.lists, f.out, f.out_cap, f.out_count, f.own));
    const int rc = sort_finish(h);
    if (keep15) h->h_small[15] = keep15;
    h->overflow |= keep_overflow;
    return rc;
  }
  if (h->h_small[2]) {                                                          // more records than the one-CTA sort holds: multi-kernel sort
    int rc = fl_launch_sort_unique_big(f.lists, h->d_keys.get(), h->key_cap, n_upper, f.out, f.out_cap, f.out_count, s);
    if (rc < 0) return FL_ERR_CAPACITY;
    h->launches += rc;
    FL_CUDA(cudaMemcpyAsync(h->h_small, f.out_count, sizeof(int), cudaMemcpyDeviceToHost, s));
    if (f.own) FL_CUDA(cudaMemcpyAsync(h->h_first, f.out, sizeof(fl_match_t) * (size_t)std::min(FETCH_FIRST, f.out_cap), cudaMemcpyDeviceToHost, s));
    if (h->profile) cudaEventRecord(h->ev[4].get(), s);
    FL_CUDA(wait_stream(h));
  }
  if (h->profile) for (int i = 0; i < 4; ++i) cudaEventElapsedTime(&h->stage_ms[i], h->ev[i].get(), h->ev[i + 1].get());
  FL_CUDA(cudaGetLastError());
  return FL_OK;
}

static int run_sort_unique(fl_handle* h, fl_lists L, fl_match_t* d_out, int out_cap, int* d_out_count, bool fetch_first, const fl_xchg* xchg = nullptr,
                           const fl_refine_req* refine = nullptr) {
  TRY(sort_launch(h, L, d_out, out_cap, d_out_count, fetch_first, xchg, refine));
  return sort_finish(h);
}

// A device frame on this handle: front end + matchClass into (cand, cap, d_count), then one launch that refines those candidates and sorts
// `lists` into the handle's output block - with the peer exchange X of a template-sharded frame in its last CTA, or X == NULL.
// Refinement and sort + unique share that launch (k_refine_sort: 256-thread CTAs, the last one to finish sorts up to 1,024 records);
// FL_OPT_SPLIT_REFINE keeps them as separate launches (what fl_match_shard_device needs anyway: its candidates must be refined before an
// NCCL gather).  A variant with 1,024-thread CTAs and the 8,192-key sort inside was measured slower (those CTAs cost more to launch than
// the launch they save) and removed.
static int match_launch(fl_handle* h, const void* d_bgr, const void* d_depth, int W, int H, const void* const* d_masks, float threshold,
                        const int32_t* class_filter, int n_filter, fl_match_t* cand, int cap, int* d_count, const fl_lists& lists, const fl_xchg* X) {
  const bool defer = !h->opt_split_refine && h->n_templates > 0 && h->p.n_levels > 1;
  TRY(run_match_stages(h, (const uint8_t*)d_bgr, (const uint16_t*)d_depth, W, H, d_masks, threshold, class_filter, n_filter, cand, cap, d_count, defer));
  const fl_refine_req req = {threshold, cand, cap, d_count};
  TRY(sort_launch(h, lists, h->d_out, h->p.max_candidates, h->d_out_count, true, X, defer ? &req : nullptr));
  fl_frame& f = h->frame;
  f.kind = X ? fl_frame_kind::shard : fl_frame_kind::match;
  f.rerun = !X; f.bgr = d_bgr; f.depth = d_depth; f.W = W; f.H = H; f.threshold = threshold;
  for (int m = 0; m < FL_MAX_MODALITIES; ++m) f.masks[m] = d_masks ? d_masks[m] : nullptr;
  f.filter.assign(class_filter && n_filter > 0 ? class_filter : nullptr, class_filter && n_filter > 0 ? class_filter + n_filter : nullptr);
  if (d_depth && d_depth == h->d_in_depth.get()) h->staged.matched = true;
  return FL_OK;
}

extern "C" int fl_match_device_async(fl_handle* h, const void* d_bgr, const void* d_depth, int32_t W, int32_t H, const void* const* d_masks,
                                     float threshold, const int32_t* class_filter, int32_t n_filter) {
  if (!h) return FL_ERR_ARG;
  TRY(frame_begin(h));
  const fl_lists lists = {h->d_cand.get(), 1, h->p.max_candidates, h->p.max_candidates, h->d_count.get(), 1};
  return match_launch(h, d_bgr, d_depth, W, H, d_masks, threshold, class_filter, n_filter, h->d_cand.get(), h->p.max_candidates, h->d_count.get(), lists,
                      nullptr);
}

int fl_frame_wait(fl_handle* h, fl_wait_note* note) {
  *note = fl_wait_note::done;
  fl_frame& f = h->frame;
  if (f.kind == fl_frame_kind::none) { fl_set_error("no frame in flight on this handle"); return FL_ERR_STATE; }
  f.kind = fl_frame_kind::none;
  TRY(sort_finish(h));
  int job;
  TRY(fl_fe_take_timeout(h->fe.get(), h->stream.get(), &job));
  if (job >= 0) {
    // an in-grid dependency of the single-launch front end timed out (the producer CTAs were not dispatched before their consumers:
    // see k_front_end_wave): the frame's result is not trustworthy.  From now on this handle launches one kernel per wave.
    if (!f.rerun) {
      *note = fl_wait_note::resubmit;
      fl_set_error("front end: in-grid dependency of job %d timed out; the handle now uses per-wave launches - resubmit the frame", job);
      return FL_ERR_STATE;
    }
    *note = fl_wait_note::rerun;
    const fl_lists lists = {h->d_cand.get(), 1, h->p.max_candidates, h->p.max_candidates, h->d_count.get(), 1};
    int rc = run_match_stages(h, (const uint8_t*)f.bgr, (const uint16_t*)f.depth, f.W, f.H, f.masks, f.threshold, f.filter.empty() ? nullptr : f.filter.data(),
                              (int)f.filter.size(), h->d_cand.get(), h->p.max_candidates, h->d_count.get());
    if (rc == FL_OK) rc = run_sort_unique(h, lists, h->d_out, h->p.max_candidates, h->d_out_count, true);
    if (rc != FL_OK) return rc;
  }
  if (h->h_small[15]) { fl_set_error("peer exchange timed out waiting for rank %d", h->h_small[15] - 1); return FL_ERR_STATE; }
  h->have_result = true;
  return FL_OK;
}
extern "C" int fl_match_wait(fl_handle* h) {
  if (!h) return FL_ERR_ARG;
  fl_wait_note note;
  return fl_frame_wait(h, &note);
}

extern "C" int fl_match_device(fl_handle* h, const void* d_bgr, const void* d_depth, int32_t W, int32_t H, const void* const* d_masks,
                               float threshold, const int32_t* class_filter, int32_t n_filter) {
  int rc = fl_match_device_async(h, d_bgr, d_depth, W, H, d_masks, threshold, class_filter, n_filter);
  if (rc != FL_OK) return rc;
  return fl_match_wait(h);
}

extern "C" int fl_match_fetch(fl_handle* h, fl_match_t* out, int32_t capacity, int32_t* count) {
  if (!h || !count || capacity < 0 || (capacity > 0 && !out)) return FL_ERR_ARG;
  if (!h->have_result) return FL_ERR_STATE;
  const int n = h->h_small[0];
  *count = n;
  const int ncopy = std::min(std::min(n, (int)capacity), h->p.max_candidates);
  const int nfirst = std::min(ncopy, FETCH_FIRST);
  if (nfirst > 0) memcpy(out, h->h_first, sizeof(fl_match_t) * nfirst);
  if (ncopy > nfirst) {
    FL_CUDA(cudaMemcpyAsync(out + nfirst, h->d_out + nfirst, sizeof(fl_match_t) * (size_t)(ncopy - nfirst), cudaMemcpyDeviceToHost, h->stream.get()));
    FL_CUDA(wait_stream(h));
  }
  // overflow: matchClass produced more candidates than the device buffer holds (the list is then incomplete)
  return (n > capacity || n > h->p.max_candidates || h->overflow) ? FL_ERR_CAPACITY : FL_OK;
}

static int resize_tables(fl_handle* h, int sW, int sH, int dW, int dH);
static int resize_staging(fl_handle* h, size_t npx);
// the device side of a staged host frame: d_in_bgr / d_in_depth (NULL when the frame has no such image) and the level-0 masks
struct fl_dev_frame { const uint8_t* bgr; const uint16_t* depth; const void* masks[FL_MAX_MODALITIES]; };

// The one upload of the host-buffer entry points: a src_W x src_H frame (bgr and depth, either may be NULL) into d_in_bgr / d_in_depth
// as a W x H frame, rescaled on the device (cv::resize INTER_LINEAR) when the sizes differ, and the masks (NULL or n_modalities
// pointers of W x H bytes, each NULL or not) into d_mask[0].  Same size: a caller buffer that is already page-locked (cudaHostAlloc /
// cudaHostRegister / torch pin_memory) is DMA'd directly, strided rows included, and has to stay valid until the frame has been waited
// for; pageable memory goes through the handle's pinned staging buffer first (copied before this returns).
static int stage_host(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int sW, int sH, int W, int H,
                      const uint8_t* const* masks, fl_dev_frame* d) {
  const fl_params_t& p = h->p;
  cudaStream_t s = h->stream.get();
  memset(d, 0, sizeof *d);
  h->staged = fl_staged_frame();
  if (W <= 0 || H <= 0 || W > p.max_width || H > p.max_height) return FL_ERR_SIZE;
  if ((bgr && bgr_stride < (size_t)sW * 3) || (depth && depth_stride < (size_t)sW * 2)) return FL_ERR_SIZE;
  auto is_pinned = [](const void* q) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, q) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
  };
  const bool rescale = sW != W || sH != H;
  if (rescale) {
    TRY(resize_tables(h, sW, sH, W, H));
    TRY(resize_staging(h, (size_t)sW * sH));
  }
  if (depth && rescale) {                                                          // depth first: it is the smaller image
    FL_CUDA(cudaMemcpy2DAsync(h->d_src_depth.get(), (size_t)sW * 2, depth, depth_stride, (size_t)sW * 2, sH, cudaMemcpyHostToDevice, s));
    fl_launch_resize_linear(h->d_src_depth.get(), sW, sH, FL_IMG_16UC1, h->d_in_depth.get(), W, H, h->rz, s); ++h->launches;
  } else if (depth) {
    if (is_pinned(depth)) {
      // dense rows go as ONE linear DMA (a 2-D copy of the same bytes is split into row descriptors and runs at about half the rate)
      if (depth_stride == (size_t)W * 2) FL_CUDA(cudaMemcpyAsync(h->d_in_depth.get(), depth, (size_t)W * H * 2, cudaMemcpyHostToDevice, s));
      else FL_CUDA(cudaMemcpy2DAsync(h->d_in_depth.get(), (size_t)W * 2, depth, depth_stride, (size_t)W * 2, H, cudaMemcpyHostToDevice, s));
    } else {
      for (int y = 0; y < H; ++y) memcpy(h->h_depth.get() + (size_t)y * W, (const uint8_t*)depth + (size_t)y * depth_stride, (size_t)W * 2);
      FL_CUDA(cudaMemcpyAsync(h->d_in_depth.get(), h->h_depth.get(), (size_t)W * H * 2, cudaMemcpyHostToDevice, s));
    }
  }
  if (bgr && rescale) {
    FL_CUDA(cudaMemcpy2DAsync(h->d_src_bgr.get(), (size_t)sW * 3, bgr, bgr_stride, (size_t)sW * 3, sH, cudaMemcpyHostToDevice, s));
    fl_launch_resize_linear(h->d_src_bgr.get(), sW, sH, FL_IMG_8UC3, h->d_in_bgr.get(), W, H, h->rz, s); ++h->launches;
  } else if (bgr) {
    if (is_pinned(bgr)) {
      if (bgr_stride == (size_t)W * 3) FL_CUDA(cudaMemcpyAsync(h->d_in_bgr.get(), bgr, (size_t)W * H * 3, cudaMemcpyHostToDevice, s));
      else FL_CUDA(cudaMemcpy2DAsync(h->d_in_bgr.get(), (size_t)W * 3, bgr, bgr_stride, (size_t)W * 3, H, cudaMemcpyHostToDevice, s));
    } else {
      // pageable source: stage in two halves so the second half's host copy overlaps the first half's DMA
      const int h0 = H / 2;
      for (int part = 0; part < 2; ++part) {
        const int y0 = part ? h0 : 0, y1 = part ? H : h0;
        for (int y = y0; y < y1; ++y) memcpy(h->h_bgr.get() + (size_t)y * W * 3, bgr + (size_t)y * bgr_stride, (size_t)W * 3);
        if (y1 > y0) FL_CUDA(cudaMemcpyAsync(h->d_in_bgr.get() + (size_t)y0 * W * 3, h->h_bgr.get() + (size_t)y0 * W * 3, (size_t)(y1 - y0) * W * 3, cudaMemcpyHostToDevice, s));
      }
    }
  }
  if (masks) for (int m = 0; m < p.n_modalities; ++m) if (masks[m]) {
    memcpy(h->h_mask.get() + (size_t)m * W * H, masks[m], (size_t)W * H);
    FL_CUDA(cudaMemcpyAsync(h->d_mask[0][m].get(), h->h_mask.get() + (size_t)m * W * H, (size_t)W * H, cudaMemcpyHostToDevice, s));
    d->masks[m] = h->d_mask[0][m].get();
  }
  d->bgr = bgr ? h->d_in_bgr.get() : nullptr; d->depth = depth ? h->d_in_depth.get() : nullptr;
  h->staged.W = W; h->staged.H = H; h->staged.bgr = bgr != nullptr; h->staged.depth = depth != nullptr;
  return FL_OK;
}

// The quantised image of (level l, modality m) of the last frame into host memory, as the reference's quantize() leaves it: a masked
// modality reads 0 where the level's mask - the level-0 mask NN-halved l times (linemod.cpp:448, 736) - is 0.  The mask is applied here,
// outside the frame, so that the frame's kernels only AND it into the labels they read (dev_spread_lm).  An unmasked image is only
// enqueued (the caller synchronises); a masked one is finished before this returns.
static int read_quantized(fl_handle* h, int l, int m, uint8_t* dst) {
  cudaStream_t s = h->stream.get();
  const fl_level_geom* g = h->geom;
  FL_CUDA(cudaMemcpyAsync(dst, h->d_q[l][m].get(), (size_t)g[l].W * g[l].H, cudaMemcpyDeviceToHost, s));
  if (!h->frame_mask[m]) return FL_OK;
  std::vector<uint8_t> mk((size_t)g[0].W * g[0].H), half;
  FL_CUDA(cudaMemcpyAsync(mk.data(), h->frame_mask[m], mk.size(), cudaMemcpyDeviceToHost, s));
  FL_CUDA(cudaStreamSynchronize(s));
  for (int k = 1; k <= l; ++k) {                        // cv::resize INTER_NEAREST to (W/2, H/2): the index arithmetic of dev_resize_nn_half
    const int sw = g[k - 1].W, sh = g[k - 1].H, dw = g[k].W, dh = g[k].H;
    half.resize((size_t)dw * dh);
    for (int y = 0; y < dh; ++y) {
      const int sy = std::min((int)floor(y * ((double)sh / dh)), sh - 1);
      for (int x = 0; x < dw; ++x) half[(size_t)y * dw + x] = mk[(size_t)sy * sw + std::min((int)floor(x * ((double)sw / dw)), sw - 1)];
    }
    mk.swap(half);
  }
  for (size_t i = 0; i < mk.size(); ++i) if (!mk[i]) dst[i] = 0;
  return FL_OK;
}

// enqueue-only half of fl_match: upload + every kernel of the frame on the handle's stream; fl_match_wait / fl_match_fetch finish it
extern "C" int fl_match_async(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int32_t W, int32_t H,
                              const uint8_t* const* masks, float threshold, const int32_t* class_filter, int32_t n_filter) {
  if (!h) return FL_ERR_ARG;
  fl_dev_frame d;
  TRY(frame_begin(h));
  TRY(stage_host(h, bgr, bgr_stride, depth, depth_stride, W, H, W, H, masks, &d));
  return fl_match_device_async(h, d.bgr, d.depth, W, H, d.masks, threshold, class_filter, n_filter);
}

// the end of the synchronous host-frame calls.  A frame whose wait fails leaves no matched depth frame behind.
static int wait_fetch(fl_handle* h, fl_match_t* out, int32_t capacity, int32_t* count) {
  const int rc = fl_match_wait(h);
  if (rc != FL_OK) { h->staged.matched = false; return rc; }
  return fl_match_fetch(h, out, capacity, count);
}

extern "C" int fl_match(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int32_t W, int32_t H,
                        const uint8_t* const* masks, float threshold, const int32_t* class_filter, int32_t n_filter, fl_match_t* out,
                        int32_t capacity, int32_t* count, uint8_t* const* quantized_out) {
  if (!h || !count) return FL_ERR_ARG;
  *count = 0;
  const fl_params_t& p = h->p;
  TRY(fl_match_async(h, bgr, bgr_stride, depth, depth_stride, W, H, masks, threshold, class_filter, n_filter));
  const int rc = wait_fetch(h, out, capacity, count);
  if (quantized_out && h->have_result) {
    for (int l = 0; l < p.n_levels; ++l) for (int m = 0; m < p.n_modalities; ++m)
      if (quantized_out[l * p.n_modalities + m]) TRY(read_quantized(h, l, m, quantized_out[l * p.n_modalities + m]));
    FL_CUDA(cudaStreamSynchronize(h->stream.get()));
  }
  return rc;
}

// ---------------------------------------------------------------------------------------------------
// Detector::addTemplate (linemod.cpp:1579-1615)
// ---------------------------------------------------------------------------------------------------
extern "C" void fl_default_train_params(fl_train_params_t* p) {
  if (!p) return;
  for (int m = 0; m < FL_MAX_MODALITIES; ++m) p->num_features[m] = 63;
  p->strong_threshold = 55.0f; p->extract_threshold = 2;
}

namespace {
struct train_cand { int x, y, label; float score; };
// QuantizedPyramid::selectScatteredFeatures (linemod.cpp:134-163), candidates already sorted
void select_scattered(const std::vector<train_cand>& cands, std::vector<fl_feature_t>& out, size_t num_features, float distance) {
  out.clear();
  float distance_sq = distance * distance;
  int i = 0;
  while (out.size() < num_features) {
    const train_cand& c = cands[i];
    bool keep = true;
    for (int j = 0; j < (int)out.size() && keep; ++j)
      keep = (float)((c.x - out[j].x) * (c.x - out[j].x) + (c.y - out[j].y) * (c.y - out[j].y)) >= distance_sq;
    if (keep) { fl_feature_t f = {c.x, c.y, c.label}; out.push_back(f); }
    if (++i == (int)cands.size()) { i = 0; distance -= 1.0f; distance_sq = distance * distance; }   // start over with a relaxed distance
  }
}
}  // namespace

extern "C" int fl_add_template(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, const uint8_t* mask,
                               size_t mask_stride, int32_t W, int32_t H, const fl_train_params_t* params_or_null, fl_template_hdr_t* headers,
                               fl_feature_t* features, int32_t feature_capacity, int32_t* n_features, fl_rect_t* bounding_box) {
  if (!h || !headers || !n_features || feature_capacity < 0 || (feature_capacity > 0 && !features)) return FL_ERR_ARG;
  *n_features = 0;
  fl_train_params_t tp;
  if (params_or_null) tp = *params_or_null; else fl_default_train_params(&tp);
  const fl_params_t& p = h->p;
  const int L = p.n_levels, M = p.n_modalities;
  if (mask && mask_stride < (size_t)W) return FL_ERR_SIZE;
  // 1. the front end: quantised images of every level and modality (unmasked, as the pyramids' `angle` / `normal` members), the colour
  //    pyramid.  A threshold above 100 % keeps matchClass from emitting anything if templates are loaded.
  TRY(fl_match_async(h, bgr, bgr_stride, depth, depth_stride, W, H, nullptr, 200.f, nullptr, 0));
  TRY(fl_match_wait(h));
  cudaStream_t s = h->stream.get();
  const size_t npx = (size_t)W * H;
  // training workspace of the handle: one block sized for the largest frame, allocated at the first call (a database generator calls
  // this thousands of times; a malloc / free round per view cost more than the kernels)
  const size_t cap_px = (size_t)p.max_width * p.max_height;
  TRY(h->d_train.grow(cap_px * (4 + 4 + 1 + 1 + 16 + 2) + 256));
  uint8_t* base = h->d_train.get();
  float* d_mag = reinterpret_cast<float*>(base); base += cap_px * 4;
  float* d_score = reinterpret_cast<float*>(base); base += cap_px * 4;
  uint16_t* d_hd = reinterpret_cast<uint16_t*>(base); base += cap_px * 16;
  int* d_cnt = reinterpret_cast<int*>(base); base += 256;
  uint8_t* d_er1 = base; base += cap_px;
  uint8_t* d_er2 = base; base += cap_px;
  uint8_t* d_maskpyr = base;
  std::vector<const uint8_t*> d_mask(L, nullptr);
  if (mask) {
    FL_CUDA(cudaMemcpy2DAsync(d_maskpyr, W, mask, mask_stride, W, H, cudaMemcpyHostToDevice, s));
    d_mask[0] = d_maskpyr;
    size_t off = npx;
    for (int l = 1; l < L; ++l) {                           // resize(mask, next_mask, size / 2, INTER_NEAREST) (:447-450, :734-738)
      uint8_t* dst = d_maskpyr + off;
      fl_launch_resize_nn_half(d_mask[l - 1], W >> (l - 1), H >> (l - 1), dst, s); ++h->launches;
      d_mask[l] = dst; off += (size_t)(W >> l) * (H >> l);
    }
  }
  std::vector<std::vector<fl_feature_t> > feats((size_t)L * M);
  std::vector<float> h_score(npx);
  std::vector<uint8_t> h_q(npx), h_lmask(npx);
  for (int m = 0; m < M; ++m) {
    const bool is_color = p.modality_kind[m] == FL_MODALITY_COLOR_GRADIENT;
    for (int l = 0; l < L; ++l) {
      const int w = W >> l, hh = H >> l;
      const size_t n = (size_t)w * hh;
      const size_t num_features = (size_t)tp.num_features[m] >> l;              // num_features /= 2 per pyrDown (:429, :724)
      const uint8_t* d_q = h->d_q[l][m].get();
      std::vector<train_cand> cands;
      float distance;
      int counts[16] = {0};
      if (is_color) {
        const uint8_t* d_bgr_l = l == 0 ? h->d_in_bgr.get() : h->d_bgr[l].get();
        fl_launch_train_magnitude(d_bgr_l, w, hh, d_mag, s); ++h->launches;
        if (d_mask[l]) { fl_launch_train_erode3(d_mask[l], w, hh, d_er1, s); ++h->launches; }
        fl_launch_train_color_score(d_q, d_mag, d_mask[l], d_mask[l] ? d_er1 : nullptr, w, hh, tp.strong_threshold * tp.strong_threshold, d_score, s); ++h->launches;
      } else {
        const uint8_t* d_local = nullptr;
        if (d_mask[l]) {                                     // erode(mask, local_mask, Mat(), Point(-1,-1), 2, BORDER_REPLICATE) (:753)
          fl_launch_train_erode3(d_mask[l], w, hh, d_er1, s); fl_launch_train_erode3(d_er1, w, hh, d_er2, s); h->launches += 2;
          d_local = d_er2;
          FL_CUDA(cudaMemcpyAsync(h_lmask.data(), d_er2, n, cudaMemcpyDeviceToHost, s));
        }
        fl_launch_train_depth_score(d_q, d_local, d_hd, d_cnt, w, hh, tp.extract_threshold >> l, d_score, d_cnt + 8, s); h->launches += 2;   // extract_threshold /= 2 per level (:725)
        FL_CUDA(cudaMemcpyAsync(counts, d_cnt, sizeof counts, cudaMemcpyDeviceToHost, s));
      }
      FL_CUDA(cudaMemcpyAsync(h_score.data(), d_score, n * sizeof(float), cudaMemcpyDeviceToHost, s));
      FL_CUDA(cudaMemcpyAsync(h_q.data(), d_q, n, cudaMemcpyDeviceToHost, s));
      FL_CUDA(wait_stream(h));
      for (int y = 0; y < hh; ++y)                            // candidates in row-major order: the order std::stable_sort keeps among ties
        for (int x = 0; x < w; ++x) {
          const float sc = h_score[(size_t)y * w + x];
          if (sc < 0.f) continue;
          const int q = h_q[(size_t)y * w + x];
          int label = 0; while (label < 7 && !(q & (1 << label))) ++label;      // getLabel: the set bit
          train_cand c = {x, y, label, sc};
          cands.push_back(c);
        }
      if (cands.size() < num_features) return FL_ERR_TRAIN;                       // (:500-501, :803-804)
      if (is_color) {
        distance = num_features ? static_cast<float>(cands.size() / num_features + 1) : 0.f;                         // (:506)
      } else {
        for (train_cand& c : cands) c.score /= (float)counts[8 + c.label];         // penalise labels with many candidates (:808-812)
        size_t area = n;
        if (d_mask[l]) { area = 0; for (size_t i = 0; i < n; ++i) area += h_lmask[i] != 0; }
        distance = num_features ? sqrtf((float)area) / sqrtf((float)num_features) + 1.5f : 0.f;                       // (:816-817)
      }
      std::stable_sort(cands.begin(), cands.end(), [](const train_cand& a, const train_cand& b) { return a.score > b.score; });   // Candidate::operator< (linemod.hpp:124-128)
      select_scattered(cands, feats[(size_t)l * M + m], num_features, distance);
    }
  }
  // cropTemplates (linemod.cpp:52-96)
  int min_x = INT_MAX, min_y = INT_MAX, max_x = INT_MIN, max_y = INT_MIN;
  for (int l = 0; l < L; ++l) for (int m = 0; m < M; ++m) for (const fl_feature_t& f : feats[(size_t)l * M + m]) {
    const int x = f.x << l, y = f.y << l;
    min_x = std::min(min_x, x); min_y = std::min(min_y, y); max_x = std::max(max_x, x); max_y = std::max(max_y, y);
  }
  if (min_x % 2 == 1) --min_x;
  if (min_y % 2 == 1) --min_y;
  int nf = 0;
  for (int l = 0; l < L; ++l) for (int m = 0; m < M; ++m) {
    fl_template_hdr_t& hd = headers[(size_t)l * M + m];
    hd.width = (max_x - min_x) >> l; hd.height = (max_y - min_y) >> l; hd.offset_x = min_x >> l; hd.offset_y = min_y >> l; hd.pyramid_level = l;
    hd.feature_begin = nf; hd.feature_count = (int)feats[(size_t)l * M + m].size();
    for (const fl_feature_t& f : feats[(size_t)l * M + m]) {
      if (nf >= feature_capacity) return FL_ERR_CAPACITY;
      fl_feature_t g = {f.x - hd.offset_x, f.y - hd.offset_y, f.label};
      features[nf++] = g;
    }
  }
  *n_features = nf;
  if (bounding_box) { bounding_box->x = min_x; bounding_box->y = min_y; bounding_box->width = max_x - min_x; bounding_box->height = max_y - min_y; }
  return FL_OK;
}

extern "C" int fl_match_shard_device(fl_handle* h, const void* d_bgr, const void* d_depth, int32_t W, int32_t H, const void* const* d_masks,
                                     float threshold, const int32_t* class_filter, int32_t n_filter, fl_match_t* d_candidates,
                                     int32_t capacity, int32_t* d_count) {
  if (!h || !d_candidates || !d_count || capacity < 1) return FL_ERR_ARG;
  TRY(frame_begin(h));           // (its front end shares the time-out flag that the wait of a frame in flight reads; it starts no frame itself)
  return run_match_stages(h, (const uint8_t*)d_bgr, (const uint16_t*)d_depth, W, H, d_masks, threshold, class_filter, n_filter, d_candidates,
                          capacity, d_count);
}

extern "C" int fl_sort_unique_device(fl_handle* h, const fl_match_t* d_in, int32_t n_lists, int32_t list_capacity, const int32_t* d_n_in,
                                     fl_match_t* d_out, int32_t out_capacity, int32_t* d_out_count) {
  if (!h || !d_in || !d_n_in || !d_out || !d_out_count || n_lists < 1 || list_capacity < 1 || out_capacity < 1) return FL_ERR_ARG;
  TRY(frame_begin(h));
  const fl_lists lists = {d_in, n_lists, list_capacity, list_capacity, d_n_in, 1};
  return run_sort_unique(h, lists, d_out, out_capacity, d_out_count, false);
}

extern "C" size_t fl_exchange_buffer_bytes(int32_t world, int32_t capacity) {
  if (world < 1 || capacity < 1) return 0;
  return fl_reco_mailbox_offset(world, capacity) + FL_RECO_MAILBOX_WORDS * sizeof(int);   // blocks, then the result mailbox (fl_internal.cuh)
}

// The peer exchange of a template-sharded frame: rank `rank` of `world` pushes `block` into every peer's buffer (peers: as mapped into
// this process), and `lists` is what the multi-kernel fallback sorts - this rank's own buffer at the epoch's parity, filled by the
// kernel's exchange.
static int exchange_setup(int rank, int world, void* const* peers, int capacity, const fl_match_t* block, uint32_t epoch, fl_xchg* X, fl_lists* lists) {
  if (!peers || !block || world < 1 || world > FL_XCHG_MAX_WORLD || rank < 0 || rank >= world || capacity < 1 || epoch == 0) return FL_ERR_ARG;
  memset(X, 0, sizeof *X);
  X->world = world; X->rank = rank; X->cap = capacity; X->epoch = epoch; X->local_block = block;
  for (int p = 0; p < world; ++p) { if (!peers[p]) return FL_ERR_ARG; X->peer[p] = static_cast<uint8_t*>(peers[p]); }
  const uint8_t* own = X->peer[rank] + FL_XCHG_SIGNALS * sizeof(unsigned) + (size_t)(epoch & 1u) * world * ((size_t)capacity + 1) * sizeof(fl_match_t);
  *lists = {reinterpret_cast<const fl_match_t*>(own) + 1, world, capacity, capacity + 1, reinterpret_cast<const int*>(own), 5 * (capacity + 1)};
  return FL_OK;
}

extern "C" int fl_exchange_sort_unique_device_async(fl_handle* h, int32_t rank, int32_t world, void* const* peer_buffers, int32_t capacity,
                                                    const fl_match_t* d_local_block, uint32_t epoch) {
  if (!h) return FL_ERR_ARG;
  fl_xchg X; fl_lists lists;
  TRY(exchange_setup(rank, world, peer_buffers, capacity, d_local_block, epoch, &X, &lists));
  TRY(frame_begin(h));
  if (h->profile) for (int i = 0; i < 4; ++i) cudaEventRecord(h->ev[i].get(), h->stream.get());
  TRY(sort_launch(h, lists, h->d_out, h->p.max_candidates, h->d_out_count, true, &X));
  h->frame.kind = fl_frame_kind::sort; h->frame.rerun = false;
  return FL_OK;
}

// Template-sharded frame in one go (enqueue only): front end + matchClass on this handle's shard with the candidates written
// straight into the caller's block [count | records], then ONE launch that refines them, pushes the block to every peer,
// waits for the peers' blocks and sorts the union (k_refine_sort<1> with the exchange in its last CTA).
extern "C" int fl_match_shard_exchange_device_masked_async(fl_handle* h, const void* d_bgr, const void* d_depth, int32_t W, int32_t H,
                                                           const void* const* d_masks, float threshold, const int32_t* class_filter, int32_t n_filter,
                                                           int32_t rank, int32_t world, void* const* peer_buffers, int32_t capacity,
                                                           fl_match_t* d_local_block, uint32_t epoch) {
  if (!h) return FL_ERR_ARG;
  fl_xchg X; fl_lists lists;
  TRY(exchange_setup(rank, world, peer_buffers, capacity, d_local_block, epoch, &X, &lists));
  TRY(frame_begin(h));
  return match_launch(h, d_bgr, d_depth, W, H, d_masks, threshold, class_filter, n_filter, d_local_block + 1, capacity, reinterpret_cast<int*>(d_local_block),
                      lists, &X);
}
extern "C" int fl_match_shard_exchange_device_async(fl_handle* h, const void* d_bgr, const void* d_depth, int32_t W, int32_t H, float threshold,
                                                    const int32_t* class_filter, int32_t n_filter, int32_t rank, int32_t world,
                                                    void* const* peer_buffers, int32_t capacity, fl_match_t* d_local_block, uint32_t epoch) {
  return fl_match_shard_exchange_device_masked_async(h, d_bgr, d_depth, W, H, nullptr, threshold, class_filter, n_filter, rank, world, peer_buffers, capacity,
                                                     d_local_block, epoch);
}

extern "C" int fl_match_shard_exchange_masked_async(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                                                    int32_t W, int32_t H, const uint8_t* const* masks, float threshold, const int32_t* class_filter,
                                                    int32_t n_filter, int32_t rank, int32_t world, void* const* peer_buffers, int32_t capacity,
                                                    fl_match_t* d_local_block, uint32_t epoch) {
  if (!h) return FL_ERR_ARG;
  fl_dev_frame d;
  TRY(frame_begin(h));
  TRY(stage_host(h, bgr, bgr_stride, depth, depth_stride, W, H, W, H, masks, &d));
  return fl_match_shard_exchange_device_masked_async(h, d.bgr, d.depth, W, H, d.masks, threshold, class_filter, n_filter, rank, world, peer_buffers, capacity,
                                                     d_local_block, epoch);
}
extern "C" int fl_match_shard_exchange_async(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int32_t W, int32_t H,
                                             float threshold, const int32_t* class_filter, int32_t n_filter, int32_t rank, int32_t world,
                                             void* const* peer_buffers, int32_t capacity, fl_match_t* d_local_block, uint32_t epoch) {
  return fl_match_shard_exchange_masked_async(h, bgr, bgr_stride, depth, depth_stride, W, H, nullptr, threshold, class_filter, n_filter, rank, world,
                                              peer_buffers, capacity, d_local_block, epoch);
}

extern "C" int fl_exchange_sort_unique_device(fl_handle* h, int32_t rank, int32_t world, void* const* peer_buffers, int32_t capacity,
                                              const fl_match_t* d_local_block, uint32_t epoch) {
  int rc = fl_exchange_sort_unique_device_async(h, rank, world, peer_buffers, capacity, d_local_block, epoch);
  if (rc != FL_OK) return rc;
  return fl_match_wait(h);
}

extern "C" int fl_sort_unique_blocks_device(fl_handle* h, const fl_match_t* d_blocks, int32_t n_blocks, int32_t capacity) {
  if (!h || !d_blocks || n_blocks < 1 || capacity < 1) return FL_ERR_ARG;
  TRY(frame_begin(h));
  if (h->profile) for (int i = 0; i < 4; ++i) cudaEventRecord(h->ev[i].get(), h->stream.get());   // stage times are not defined for this entry point
  const fl_lists lists = {d_blocks + 1, n_blocks, capacity, capacity + 1, reinterpret_cast<const int*>(d_blocks), 5 * (capacity + 1)};
  TRY(run_sort_unique(h, lists, h->d_out, h->p.max_candidates, h->d_out_count, true));
  h->have_result = true;
  return FL_OK;
}

// ---------------------------------------------------------------------------------------------------
extern "C" int fl_debug_get(fl_handle* h, int what, int32_t a, int32_t b, int32_t c, void* host_out, size_t bytes) {
  if (!h || !host_out) return FL_ERR_ARG;
  if (h->gW == 0) return FL_ERR_STATE;
  const fl_params_t& p = h->p;
  FL_CUDA(cudaSetDevice(p.device));
  FL_CUDA(cudaStreamSynchronize(h->stream.get()));
  if (what == FL_DBG_QUANTIZED || what == FL_DBG_SPREAD) {
    if (a < 0 || a >= p.n_levels || b < 0 || b >= p.n_modalities) return FL_ERR_ARG;
    size_t n = (size_t)h->geom[a].W * h->geom[a].H;
    if (bytes < n) return FL_ERR_CAPACITY;
    if (what == FL_DBG_QUANTIZED) {
      TRY(read_quantized(h, a, b, static_cast<uint8_t*>(host_out)));
      FL_CUDA(cudaStreamSynchronize(h->stream.get()));
      return FL_OK;
    }
    if (!h->d_spread[a][b].get()) return FL_ERR_STATE;
    FL_CUDA(cudaMemcpy(host_out, h->d_spread[a][b].get(), n, cudaMemcpyDeviceToHost));
    return FL_OK;
  }
  if (what == FL_DBG_LINEAR_MEMORY) {
    if (a < 0 || a >= p.n_levels || b < 0 || b >= p.n_modalities || c < 0 || c > 7) return FL_ERR_ARG;
    const fl_level_geom& g = h->geom[a];
    size_t n = (size_t)g.T * g.T * g.cells;
    if (bytes < n) return FL_ERR_CAPACITY;
    FL_CUDA(cudaMemcpy(host_out, h->d_lm[a].get() + (size_t)b * g.mod_stride + (size_t)c * g.label_stride, n, cudaMemcpyDeviceToHost));
    return FL_OK;
  }
  if (what == FL_DBG_SIMILARITY) {
    if (a < 0 || a >= h->n_templates) return FL_ERR_ARG;
    const fl_level_geom& g = h->geom[p.n_levels - 1];
    if (bytes < (size_t)g.cells * 2) return FL_ERR_CAPACITY;
    uint16_t* d_tmp = reinterpret_cast<uint16_t*>(h->d_keys.get());                   // scratch
    if ((size_t)g.cells * 2 > (size_t)h->key_cap * sizeof(fl_sort_key)) return FL_ERR_CAPACITY;
    fl_launch_similarity_debug(make_tdb(h), g, h->d_lm[p.n_levels - 1].get(), a, d_tmp, h->stream.get()); ++h->launches;
    FL_CUDA(cudaStreamSynchronize(h->stream.get()));
    FL_CUDA(cudaMemcpy(host_out, d_tmp, (size_t)g.cells * 2, cudaMemcpyDeviceToHost));
    return FL_OK;
  }
  if (what == FL_DBG_LAST_COUNTS) {
    if (bytes < 16 * sizeof(int)) return FL_ERR_CAPACITY;
    memcpy(host_out, h->h_small, 16 * sizeof(int));
    return FL_OK;
  }
  if (what == FL_DBG_FE_TRACE) return fl_fe_trace(h->fe.get(), host_out, bytes);   // developer: front-end job timeline (FL_OPT_TRACE)
  if (what == FL_DBG_STAGED_ORDER) {                                                           // the phase order of the last staged launch
    if (!h->use_staged) return FL_ERR_STATE;
    if (bytes < 32 * sizeof(uint32_t) + (size_t)h->plan.n_phases) return FL_ERR_CAPACITY;
    uint32_t raw[FL_MASS_WORDS];
    FL_CUDA(cudaMemcpy(raw, h->d_mass.get(), sizeof raw, cudaMemcpyDeviceToHost));
    memcpy(host_out, raw + FL_MASS_USED, 32 * sizeof(uint32_t));
    memcpy(static_cast<uint8_t*>(host_out) + 32 * sizeof(uint32_t), raw + FL_MASS_ORDER, (size_t)h->plan.n_phases);
    return h->plan.n_phases;
  }
  if (what == FL_DBG_STAGED_TRACE) {
    if (!h->use_staged || !h->plan.trace) return FL_ERR_STATE;
    size_t n = ((size_t)h->plan.n_cta * 136 + 8) * sizeof(unsigned long long);
    if (bytes < n) return FL_ERR_CAPACITY;
    FL_CUDA(cudaMemcpy(host_out, h->plan.trace, n, cudaMemcpyDeviceToHost));
    return h->plan.n_cta;
  }
  return FL_ERR_ARG;
}

// ---------------------------------------------------------------------------------------------------
// input rescale: cv::resize INTER_LINEAR tables (OpenCV imgproc/src/resize.cpp, the loops that fill xofs / alpha / yofs / beta)
// ---------------------------------------------------------------------------------------------------
static int resize_tables(fl_handle* h, int sW, int sH, int dW, int dH) {
  if (h->rz.xofs && h->rz_sW == sW && h->rz_sH == sH && h->rz_dW == dW && h->rz_dH == dH) return FL_OK;
  FL_CUDA(cudaStreamSynchronize(h->stream.get()));
  h->rz_sW = h->rz_sH = h->rz_dW = h->rz_dH = 0;                                 // no tables until all six hold the new geometry
  std::vector<int> xo, yo; std::vector<float> xa, yb;
  std::vector<short> ia, ib;
  fl_resize_axis(sW, dW, true, xo, xa, ia); fl_resize_axis(sH, dH, false, yo, yb, ib);
  TRY(alloc_into(h->rz_xofs, (size_t)dW, &h->rz.xofs)); TRY(alloc_into(h->rz_yofs, (size_t)dH, &h->rz.yofs));
  TRY(alloc_into(h->rz_ialpha, (size_t)dW, &h->rz.ialpha)); TRY(alloc_into(h->rz_ibeta, (size_t)dH, &h->rz.ibeta));
  TRY(alloc_into(h->rz_alpha, (size_t)dW, &h->rz.alpha)); TRY(alloc_into(h->rz_beta, (size_t)dH, &h->rz.beta));
  FL_CUDA(cudaMemcpy(h->rz.xofs, xo.data(), (size_t)dW * 4, cudaMemcpyHostToDevice)); FL_CUDA(cudaMemcpy(h->rz.yofs, yo.data(), (size_t)dH * 4, cudaMemcpyHostToDevice));
  FL_CUDA(cudaMemcpy(h->rz.ialpha, ia.data(), (size_t)dW * 4, cudaMemcpyHostToDevice)); FL_CUDA(cudaMemcpy(h->rz.ibeta, ib.data(), (size_t)dH * 4, cudaMemcpyHostToDevice));
  FL_CUDA(cudaMemcpy(h->rz.alpha, xa.data(), (size_t)dW * 8, cudaMemcpyHostToDevice)); FL_CUDA(cudaMemcpy(h->rz.beta, yb.data(), (size_t)dH * 8, cudaMemcpyHostToDevice));
  h->rz_sW = sW; h->rz_sH = sH; h->rz_dW = dW; h->rz_dH = dH;
  return FL_OK;
}
static int resize_staging(fl_handle* h, size_t npx) {
  if (npx * 3 <= h->d_src_bgr.capacity() && npx <= h->d_src_depth.capacity()) return FL_OK;
  FL_CUDA(cudaStreamSynchronize(h->stream.get()));
  TRY(h->d_src_bgr.alloc(npx * 3)); TRY(h->d_src_depth.alloc(npx));
  return FL_OK;
}

extern "C" int fl_resize_linear(fl_handle* h, const void* src, size_t src_stride, int32_t sW, int32_t sH, int32_t type, void* dst, int32_t W, int32_t H) {
  if (!h || !src || !dst || sW <= 0 || sH <= 0 || W <= 0 || H <= 0 || (type != FL_IMG_8UC3 && type != FL_IMG_16UC1)) return FL_ERR_ARG;
  const size_t px = type == FL_IMG_8UC3 ? 3 : 2;
  if (src_stride < (size_t)sW * px) return FL_ERR_ARG;
  FL_CUDA(cudaSetDevice(h->p.device));
  cudaStream_t s = h->stream.get();
  TRY(resize_tables(h, sW, sH, W, H));
  TRY(resize_staging(h, (size_t)sW * sH));
  void* d_src = type == FL_IMG_8UC3 ? (void*)h->d_src_bgr.get() : (void*)h->d_src_depth.get();
  fl_dev_buf<uint8_t> d_dst;                                                    // freed on every exit path
  TRY(d_dst.alloc((size_t)W * H * px));
  FL_CUDA(cudaMemcpy2DAsync(d_src, (size_t)sW * px, src, src_stride, (size_t)sW * px, sH, cudaMemcpyHostToDevice, s));
  fl_launch_resize_linear(d_src, sW, sH, type, d_dst.get(), W, H, h->rz, s); ++h->launches;
  FL_CUDA(cudaMemcpyAsync(dst, d_dst.get(), (size_t)W * H * px, cudaMemcpyDeviceToHost, s));
  FL_CUDA(cudaStreamSynchronize(s));
  FL_CUDA(cudaGetLastError());
  return FL_OK;
}

extern "C" int fl_match_rescaled(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int32_t sW, int32_t sH,
                                 int32_t W, int32_t H, float threshold, const int32_t* class_filter, int32_t n_filter, fl_match_t* out, int32_t capacity,
                                 int32_t* count, uint16_t* rescaled_depth_out) {
  if (!h || !count || sW <= 0 || sH <= 0) return FL_ERR_ARG;
  *count = 0;
  fl_dev_frame d;
  TRY(frame_begin(h));
  TRY(stage_host(h, bgr, bgr_stride, depth, depth_stride, sW, sH, W, H, nullptr, &d));
  if (rescaled_depth_out && depth) {
    if (sW == W && sH == H)                                                      // TImage2Mat resizes only when the size differs (:42)
      for (int y = 0; y < H; ++y) memcpy(rescaled_depth_out + (size_t)y * W, (const uint8_t*)depth + (size_t)y * depth_stride, (size_t)W * 2);
    else
      FL_CUDA(cudaMemcpyAsync(rescaled_depth_out, h->d_in_depth.get(), (size_t)W * H * 2, cudaMemcpyDeviceToHost, h->stream.get()));
  }
  TRY(fl_match_device_async(h, d.bgr, d.depth, W, H, nullptr, threshold, class_filter, n_filter));
  return wait_fetch(h, out, capacity, count);
}

// ---------------------------------------------------------------------------------------------------
// ICP
// ---------------------------------------------------------------------------------------------------
static int icp_reserve(fl_handle* h, int n_hyp, int max_pts) {
  if (n_hyp <= h->icp_hyp_cap && max_pts <= h->icp_pts_cap) { h->icp.n_hyp = n_hyp; return FL_OK; }
  int nh = std::max(n_hyp, h->icp_hyp_cap), np = (std::max(max_pts, h->icp_pts_cap) + 3) & ~3;
  FL_CUDA(cudaStreamSynchronize(h->stream.get()));
  // the whole workspace is released before the larger one is allocated (the peak is the new workspace alone).  What points into it is
  // invalid until the new one is complete; a recognition set up before stays valid then, because the workspace only ever grows.
  const bool reco_set = h->reco_set; h->reco_set = false;
  h->icp_hyp_cap = h->icp_pts_cap = h->icp_trace_n = 0; memset(&h->icp, 0, sizeof h->icp); h->icpw = fl_icp_bufs();
  size_t tot = (size_t)nh * np;
  TRY(alloc_into(h->icpw.pts_ref, tot * 3, &h->icp.pts_ref)); TRY(alloc_into(h->icpw.pts_mod, tot * 3, &h->icp.pts_mod));
  TRY(alloc_into(h->icpw.cor_m, tot * 3, &h->icp.cor_m)); TRY(alloc_into(h->icpw.cor_r, tot * 3, &h->icp.cor_r)); TRY(alloc_into(h->icpw.dist, tot, &h->icp.dist));
  TRY(alloc_into(h->icpw.grid_pts, tot, &h->icp.grid_pts)); TRY(alloc_into(h->icpw.nn_d2, tot, &h->icp.nn_d2)); TRY(alloc_into(h->icpw.nn_slot, tot, &h->icp.nn_slot));
  TRY(h->icpw.d_ticket.alloc(1)); TRY(alloc_into(h->icpw.n_ref, (size_t)nh, &h->icp.n_ref)); TRY(alloc_into(h->icpw.n_mod, (size_t)nh, &h->icp.n_mod));
  TRY(h->icpw.d_hyps.alloc((size_t)nh)); TRY(h->icpw.d_results.alloc((size_t)nh)); TRY(h->icpw.d_model_crops.alloc(tot));
  TRY(h->icpw.h_model_crops.alloc(tot)); TRY(h->icpw.h_hyps.alloc((size_t)nh)); TRY(h->icpw.h_results.alloc((size_t)nh));
  h->icp_hyp_cap = nh; h->icp_pts_cap = np; h->icp.max_pts = np; h->icp.n_hyp = n_hyp; h->reco_set = reco_set;
  return FL_OK;
}

extern "C" int fl_depth_to_3d(fl_handle* h, const uint16_t* depth, size_t depth_stride, int32_t W, int32_t H, fl_intrinsics_t K, float* out3) {
  if (!h || !depth || !out3 || W <= 0 || H <= 0 || depth_stride < (size_t)W * 2) return FL_ERR_ARG;
  FL_CUDA(cudaSetDevice(h->p.device));
  size_t n = (size_t)W * H;
  fl_dev_buf<uint16_t> d_d; fl_dev_buf<float> d_o;                              // freed on every exit path
  TRY(d_d.alloc(n)); TRY(d_o.alloc(n * 3));
  FL_CUDA(cudaMemcpy2DAsync(d_d.get(), (size_t)W * 2, depth, depth_stride, (size_t)W * 2, H, cudaMemcpyHostToDevice, h->stream.get()));
  fl_launch_depth_to_3d(d_d.get(), W, H, K, d_o.get(), h->stream.get()); ++h->launches;
  FL_CUDA(cudaMemcpyAsync(out3, d_o.get(), n * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream.get()));
  FL_CUDA(cudaStreamSynchronize(h->stream.get()));
  return FL_OK;
}

extern "C" int fl_icp_cloud_to_cloud_ex(fl_handle* h, const float* pts_ref, int32_t n_ref, const float* pts_model, int32_t n_model,
                                        fl_icp_params_t prm, fl_icp_result_t* out) {
  if (!h || !out || n_ref < 0 || n_model < 0 || (n_ref > 0 && !pts_ref) || (n_model > 0 && !pts_model)) return FL_ERR_ARG;
  if (n_ref >= 3 && n_model >= 3 && n_ref < n_model) { fl_set_error("icpCloudToCloud_Ex walks both clouds in lock step: n_ref (%d) must be >= n_model (%d)", n_ref, n_model); return FL_ERR_SIZE; }
  FL_CUDA(cudaSetDevice(h->p.device));
  cudaStream_t s = h->stream.get();
  TRY(icp_reserve(h, 1, std::max(std::max(n_ref, n_model), 16)));
  if (n_ref) FL_CUDA(cudaMemcpyAsync(h->icp.pts_ref, pts_ref, (size_t)n_ref * 12, cudaMemcpyHostToDevice, s));
  if (n_model) FL_CUDA(cudaMemcpyAsync(h->icp.pts_mod, pts_model, (size_t)n_model * 12, cudaMemcpyHostToDevice, s));
  FL_CUDA(cudaMemcpyAsync(h->icp.n_ref, &n_ref, 4, cudaMemcpyHostToDevice, s));
  FL_CUDA(cudaMemcpyAsync(h->icp.n_mod, &n_model, 4, cudaMemcpyHostToDevice, s));
  FL_CUDA(cudaStreamSynchronize(s));                                            // &n_ref / &n_model are stack addresses
  { const fl_intrinsics_t none = {0.f, 0.f, 0.f, 0.f};
    const int nl = fl_launch_icp(h->icp, prm, nullptr, nullptr, 0, 0, none, h->icpw.d_results.get(), h->icpw.d_ticket.get(), nullptr, h->n_sm, s);
    if (nl < 0) { fl_set_error("ICP kernel launch failed: %s", cudaGetErrorString(cudaGetLastError())); return FL_ERR_CUDA; }
    h->launches += nl; }
  FL_CUDA(cudaMemcpyAsync(h->icpw.h_results.get(), h->icpw.d_results.get(), sizeof(fl_icp_result_t), cudaMemcpyDeviceToHost, s));
  FL_CUDA(cudaStreamSynchronize(s));
  FL_CUDA(cudaGetLastError());
  *out = h->icpw.h_results.get()[0];
  return FL_OK;
}

// rects inside the W x H frame?  (cv::Mat ROI throw, detection.cpp:43-44)
static bool rect_inside(const fl_rect_t& a, int W, int H) {
  return a.x >= 0 && a.y >= 0 && a.width >= 0 && a.height >= 0 && a.x + a.width <= W && a.y + a.height <= H;
}
// the reference depth frame on the device: a host frame is uploaded into d_ref_depth; NULL selects the frame the last
// host-input fl_match left in d_in_depth (Recognition hands the same image to match and to detection, obj_reco_lmicp.cpp:101, 188)
static int icp_ref_frame(fl_handle* h, const uint16_t* ref_depth, size_t ref_stride, int W, int H, const uint16_t** d_ref) {
  if (!ref_depth) {
    const fl_staged_frame& st = h->staged;
    if (!st.matched || st.W != W || st.H != H) {
      fl_set_error("ref_depth == NULL needs a preceding fl_match of a %d x %d depth frame on this handle (have %d x %d)", W, H, st.matched ? st.W : 0, st.matched ? st.H : 0);
      return FL_ERR_STATE;
    }
    *d_ref = h->d_in_depth.get();
    return FL_OK;
  }
  if (ref_stride < (size_t)W * 2) return FL_ERR_ARG;
  TRY(h->d_ref_depth.grow((size_t)W * H));
  FL_CUDA(cudaMemcpy2DAsync(h->d_ref_depth.get(), (size_t)W * 2, ref_depth, ref_stride, (size_t)W * 2, H, cudaMemcpyHostToDevice, h->stream.get()));
  *d_ref = h->d_ref_depth.get();
  return FL_OK;
}
// h_hyps[0..n) are filled: upload them, run prepare + the ICP loop, fetch the results
static int icp_run_batch(fl_handle* h, const uint16_t* d_ref, int W, int H, fl_intrinsics_t K_ref, int n, fl_icp_params_t prm, fl_icp_result_t* out) {
  cudaStream_t s = h->stream.get();
  FL_CUDA(cudaMemcpyAsync(h->icpw.d_hyps.get(), h->icpw.h_hyps.get(), sizeof(fl_icp_hyp) * (size_t)n, cudaMemcpyHostToDevice, s));
  if (h->profile) cudaEventRecord(h->ev[0].get(), s);
  unsigned long long* trace = nullptr;
  if (h->profile) {                                                             // per-hypothesis phase clock of the fused kernel (fl_debug_icp_trace)
    TRY(h->icpw.d_trace.grow((size_t)n * FL_ICP_TRACE_WORDS));
    trace = h->icpw.d_trace.get(); h->icp_trace_n = n;
  }
  { const int nl = fl_launch_icp(h->icp, prm, h->icpw.d_hyps.get(), d_ref, W, H, K_ref, h->icpw.d_results.get(), h->icpw.d_ticket.get(), trace, h->n_sm, s);
    if (nl < 0) { fl_set_error("ICP kernel launch failed: %s", cudaGetErrorString(cudaGetLastError())); return FL_ERR_CUDA; }
    h->launches += nl; }
  if (h->profile) cudaEventRecord(h->ev[1].get(), s);
  FL_CUDA(cudaMemcpyAsync(h->icpw.h_results.get(), h->icpw.d_results.get(), sizeof(fl_icp_result_t) * (size_t)n, cudaMemcpyDeviceToHost, s));
  FL_CUDA(wait_stream(h));
  if (h->profile) cudaEventElapsedTime(&h->icp_ms, h->ev[0].get(), h->ev[1].get());
  FL_CUDA(cudaGetLastError());
  memcpy(out, h->icpw.h_results.get(), sizeof(fl_icp_result_t) * (size_t)n);
  return FL_OK;
}
static void icp_fill_pose(fl_icp_hyp& hy, const float* r_match9, const float* t_match3, int i) {
  for (int k = 0; k < 9; ++k) hy.r_match[k] = r_match9 ? r_match9[9 * i + k] : (k % 4 == 0 ? 1.f : 0.f);
  for (int k = 0; k < 3; ++k) hy.t_match[k] = t_match3 ? t_match3[3 * i + k] : 0.f;
}

extern "C" int fl_detection_batch(fl_handle* h, const uint16_t* ref_depth, size_t ref_stride, int32_t W, int32_t H, fl_intrinsics_t K_ref,
                                  const uint16_t* const* model_depth, const size_t* model_stride, const fl_rect_t* rect_model,
                                  const fl_rect_t* rect_ref, const float* r_match9, const float* t_match3, const float* d_match, int32_t n,
                                  fl_icp_params_t prm, fl_icp_result_t* out) {
  (void)d_match;   // detection() receives d_match but its live branch (test_id == 2) never reads it (detection.cpp:147, 175-178)
  if (!h || !ref_depth || !model_depth || !model_stride || !rect_model || !rect_ref || !out || n < 0 || W <= 0 || H <= 0 || ref_stride < (size_t)W * 2) return FL_ERR_ARG;
  if (n == 0) return FL_OK;
  FL_CUDA(cudaSetDevice(h->p.device));
  cudaStream_t s = h->stream.get();
  int max_pts = 16;
  std::vector<int> st(n, FL_OK);
  for (int i = 0; i < n; ++i) {
    const fl_rect_t& a = rect_model[i]; const fl_rect_t& b = rect_ref[i];
    if (!(rect_inside(a, W, H) && rect_inside(b, W, H) && model_depth[i])) { st[i] = FL_ERR_ROI; continue; }
    max_pts = std::max(max_pts, std::max(a.width * a.height, b.width * b.height));
  }
  TRY(icp_reserve(h, n, max_pts));
  const int mp = h->icp.max_pts;
  const uint16_t* d_ref = nullptr;
  TRY(icp_ref_frame(h, ref_depth, ref_stride, W, H, &d_ref));
  for (int i = 0; i < n; ++i) {
    fl_icp_hyp& hy = h->icpw.h_hyps.get()[i];
    hy.model_depth = h->icpw.d_model_crops.get() + (size_t)i * mp;
    hy.rect_model = rect_model[i]; hy.rect_ref = rect_ref[i]; hy.status = st[i];
    icp_fill_pose(hy, r_match9, t_match3, i);
    if (st[i] != FL_OK) continue;
    const fl_rect_t& a = rect_model[i];
    uint16_t* dst = h->icpw.h_model_crops.get() + (size_t)i * mp;
    for (int y = 0; y < a.height; ++y)
      memcpy(dst + (size_t)y * a.width, (const uint8_t*)model_depth[i] + (size_t)(a.y + y) * model_stride[i] + (size_t)a.x * 2, (size_t)a.width * 2);
  }
  // one copy for all crops (the staging block is contiguous): 256 separate copies cost more than the ICP itself
  FL_CUDA(cudaMemcpyAsync(h->icpw.d_model_crops.get(), h->icpw.h_model_crops.get(), (size_t)n * mp * 2, cudaMemcpyHostToDevice, s));
  return icp_run_batch(h, d_ref, W, H, K_ref, n, prm, out);
}

// The rendered template depth crops of the detector's templates, uploaded ONCE (AddObj time) and packed back to back.
extern "C" int fl_upload_model_depths(fl_handle* h, int32_t n_models, const uint16_t* const* model_depth, const size_t* model_stride,
                                      const fl_rect_t* rect_model, int32_t W, int32_t H) {
  if (!h || n_models < 0 || W <= 0 || H <= 0 || (n_models > 0 && (!model_depth || !model_stride || !rect_model))) return FL_ERR_ARG;
  FL_CUDA(cudaSetDevice(h->p.device));
  std::vector<size_t> off((size_t)n_models + 1, 0);
  for (int i = 0; i < n_models; ++i) {
    if (!model_depth[i] || model_stride[i] < (size_t)W * 2) return FL_ERR_ARG;
    if (!rect_inside(rect_model[i], W, H)) { fl_set_error("model rect %d lies outside the %d x %d image", i, W, H); return FL_ERR_ROI; }
    off[i + 1] = off[i] + (size_t)rect_model[i].width * rect_model[i].height;
  }
  std::vector<uint16_t> packed(std::max<size_t>(off[n_models], 1));
  for (int i = 0; i < n_models; ++i) {
    const fl_rect_t& a = rect_model[i];
    for (int y = 0; y < a.height; ++y)
      memcpy(&packed[off[i] + (size_t)y * a.width], (const uint8_t*)model_depth[i] + (size_t)(a.y + y) * model_stride[i] + (size_t)a.x * 2, (size_t)a.width * 2);
  }
  FL_CUDA(cudaStreamSynchronize(h->stream.get()));                                    // an ICP batch that still reads the old set
  h->reco_set = false; h->res_off.clear(); h->res_rect.clear(); h->res_W = h->res_H = 0;   // d_reco_tmpl and these describe the old set
  TRY(h->d_resident.alloc(packed.size()));
  FL_CUDA(cudaMemcpy(h->d_resident.get(), packed.data(), packed.size() * 2, cudaMemcpyHostToDevice));
  h->res_off.assign(off.begin(), off.end() - 1);
  h->res_rect.assign(rect_model, rect_model + n_models);
  h->res_W = W; h->res_H = H;
  // size the ICP workspace for the largest crop now (8 hypotheses; more grow it again): growing it later means cudaFree / cudaMalloc,
  // which synchronise the whole device - harmless for one handle, a stall for the other frames in flight on this GPU, and with a
  // peer-memory exchange in flight on another handle a cross-rank stall until that exchange times out
  int max_pts = 16;
  for (int i = 0; i < n_models; ++i) max_pts = std::max(max_pts, rect_model[i].width * rect_model[i].height);
  TRY(icp_reserve(h, std::max(h->icp_hyp_cap, 8), max_pts));
  return FL_OK;
}

static int detection_batch_resident(fl_handle* h, const uint16_t* ref_depth, size_t ref_stride, const uint16_t* d_ref_given, int32_t W, int32_t H,
                                    fl_intrinsics_t K_ref, const int32_t* model_index, const fl_rect_t* rect_ref, const float* r_match9,
                                    const float* t_match3, int32_t n, fl_icp_params_t prm, fl_icp_result_t* out) {
  if (!h || !model_index || !rect_ref || !out || n < 0 || W <= 0 || H <= 0) return FL_ERR_ARG;
  if (n == 0) return FL_OK;
  if (!h->d_resident.get() || h->res_W != W || h->res_H != H) { fl_set_error("no model depth crops uploaded for %d x %d frames (fl_upload_model_depths)", W, H); return FL_ERR_STATE; }
  FL_CUDA(cudaSetDevice(h->p.device));
  int max_pts = 16;
  std::vector<int> st(n, FL_OK);
  for (int i = 0; i < n; ++i) {
    if (model_index[i] < 0 || (size_t)model_index[i] >= h->res_rect.size()) return FL_ERR_ARG;
    const fl_rect_t& a = h->res_rect[model_index[i]]; const fl_rect_t& b = rect_ref[i];
    if (!rect_inside(b, W, H)) { st[i] = FL_ERR_ROI; continue; }
    max_pts = std::max(max_pts, std::max(a.width * a.height, b.width * b.height));
  }
  TRY(icp_reserve(h, n, max_pts));
  const uint16_t* d_ref = d_ref_given;
  if (!d_ref) TRY(icp_ref_frame(h, ref_depth, ref_stride, W, H, &d_ref));
  for (int i = 0; i < n; ++i) {
    fl_icp_hyp& hy = h->icpw.h_hyps.get()[i];
    hy.model_depth = h->d_resident.get() + h->res_off[model_index[i]];
    hy.rect_model = h->res_rect[model_index[i]]; hy.rect_ref = rect_ref[i]; hy.status = st[i];
    icp_fill_pose(hy, r_match9, t_match3, i);
  }
  return icp_run_batch(h, d_ref, W, H, K_ref, n, prm, out);
}

extern "C" int fl_detection_batch_resident(fl_handle* h, const uint16_t* ref_depth, size_t ref_stride, int32_t W, int32_t H, fl_intrinsics_t K_ref,
                                           const int32_t* model_index, const fl_rect_t* rect_ref, const float* r_match9, const float* t_match3,
                                           int32_t n, fl_icp_params_t prm, fl_icp_result_t* out) {
  return detection_batch_resident(h, ref_depth, ref_stride, nullptr, W, H, K_ref, model_index, rect_ref, r_match9, t_match3, n, prm, out);
}
// the same with the reference depth frame ALREADY ON THE DEVICE (dense rows of W u16), e.g. the frame fl_match_device* was given
extern "C" int fl_detection_batch_resident_device(fl_handle* h, const void* d_ref_depth, int32_t W, int32_t H, fl_intrinsics_t K_ref,
                                                  const int32_t* model_index, const fl_rect_t* rect_ref, const float* r_match9,
                                                  const float* t_match3, int32_t n, fl_icp_params_t prm, fl_icp_result_t* out) {
  if (!d_ref_depth) return FL_ERR_ARG;
  return detection_batch_resident(h, nullptr, 0, static_cast<const uint16_t*>(d_ref_depth), W, H, K_ref, model_index, rect_ref, r_match9, t_match3, n, prm, out);
}

extern "C" int fl_detection(fl_handle* h, const uint16_t* model_depth, size_t model_stride, const uint16_t* ref_depth, size_t ref_stride,
                            int32_t W, int32_t H, fl_intrinsics_t K_ref, fl_rect_t rect_model, fl_rect_t rect_ref, int32_t icp_it_thr,
                            float dist_mean_thr, float dist_diff_thr, const float r_match[9], const float t_match[3], float d_match,
                            float T_final[3], float R_final[9]) {
  if (!T_final || !R_final) return FL_ERR_ARG;
  fl_icp_params_t prm = {icp_it_thr, dist_mean_thr, dist_diff_thr};
  fl_icp_result_t r;
  int rc = fl_detection_batch(h, ref_depth, ref_stride, W, H, K_ref, &model_depth, &model_stride, &rect_model, &rect_ref, r_match, t_match,
                              &d_match, 1, prm, &r);
  if (rc != FL_OK) return rc;
  if (r.status != FL_OK) return r.status;
  memcpy(T_final, r.T, 12); memcpy(R_final, r.R, 36);
  return FL_OK;
}

extern "C" int fl_nms_ex(fl_handle* h, const float* t3, const int32_t* n_model_pts, const float* icp_dist, int32_t n, float th, int32_t* out_idx,
                         uint8_t* absorbed) {
  if (!h || n < 0 || (n > 0 && (!t3 || !n_model_pts || !icp_dist || !out_idx))) return FL_ERR_ARG;
  if (n == 0) return 0;
  FL_CUDA(cudaSetDevice(h->p.device));
  cudaStream_t s = h->stream.get();
  // handle-owned workspace, grown on demand: a cudaMalloc / cudaFree pair per call would synchronise the whole device - with other
  // handles' frames in flight on the same GPU that serialises them, and a kernel of theirs that is waiting for a peer rank's
  // block turns it into a cross-rank stall until the exchange times out
  if (h->nms_cap < n) {
    h->nms_cap = 0;
    const int cap = std::max(64, 2 * n);
    TRY(h->d_nms.alloc((size_t)cap * 7 + 2));
    h->nms_cap = cap;
  }
  float* d_t = reinterpret_cast<float*>(h->d_nms.get());
  int32_t* d_n = h->d_nms.get() + (size_t)h->nms_cap * 3;
  float* d_d = reinterpret_cast<float*>(h->d_nms.get() + (size_t)h->nms_cap * 4);
  int32_t* d_o = h->d_nms.get() + (size_t)h->nms_cap * 5;                        // [n out_idx][n absorbed bytes (n words reserved)][count]
  FL_CUDA(cudaMemcpyAsync(d_t, t3, (size_t)n * 12, cudaMemcpyHostToDevice, s));
  FL_CUDA(cudaMemcpyAsync(d_n, n_model_pts, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  FL_CUDA(cudaMemcpyAsync(d_d, icp_dist, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  int32_t* d_cnt = d_o + 2 * n + 1;
  fl_launch_nms(d_t, d_n, d_d, n, th, d_o, d_cnt, s); ++h->launches;       // the absorbed flags live right after out_idx (n bytes)
  int32_t cnt = 0;
  FL_CUDA(cudaMemcpyAsync(out_idx, d_o, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  if (absorbed) FL_CUDA(cudaMemcpyAsync(absorbed, d_o + n, (size_t)n, cudaMemcpyDeviceToHost, s));
  FL_CUDA(cudaMemcpyAsync(&cnt, d_cnt, 4, cudaMemcpyDeviceToHost, s));
  FL_CUDA(wait_stream(h));
  return cnt;
}

extern "C" int fl_nms(fl_handle* h, const float* t3, const int32_t* n_model_pts, const float* icp_dist, int32_t n, float th, int32_t* out_idx) {
  return fl_nms_ex(h, t3, n_model_pts, icp_dist, n, th, out_idx, nullptr);
}

// ---------------------------------------------------------------------------------------------------
// Recognition on the device (CObjRecoLmICP::Recognition, CadReco/obj_reco_lmicp.cpp:86-204)
// ---------------------------------------------------------------------------------------------------
extern "C" void fl_default_reco_params(fl_reco_params_t* p) {
  if (!p) return;
  p->threshold = 75.0f;                                                           // :52-55
  p->icp.icp_it_thr = 10; p->icp.dist_mean_thr = 0.5f; p->icp.dist_diff_thr = 0.01f;
  p->top_k = 1; p->per_class = 0; p->th_obj_dist = 0.f;                           // matches[0] only (:111)
}

// The one builder of a recognition set-up: the selection table of `set` (crop and pose of every template, in the order of the set) and
// the set's class_first, installed on the handle together with an ICP workspace sized for the frame's hypotheses.  fl_set_recognition
// passes the handle's own upload; fl_group_set_recognition passes the whole set of a template-sharded group, whose merged list every
// member's handle selects from.
int fl_reco_setup(fl_handle* h, const fl_reco_params_t* prm, const fl_reco_set& set, const int32_t* crop_of_template, const float* pose12) {
  if (!h || !prm || !crop_of_template || prm->top_k < 1 || set.n_templates < 0 || (set.n_templates > 0 && (!set.class_of || !set.box0))) return FL_ERR_ARG;
  TRY(frame_idle(h));
  if (set.n_templates == 0) { fl_set_error("fl_set_recognition: no templates uploaded"); return FL_ERR_STATE; }
  if (!pose12 && !set.pose13) { fl_set_error("fl_set_recognition: no pose table (pose12 NULL and no pose13 uploaded)"); return FL_ERR_ARG; }
  int nc = 0;
  for (int t = 0; t < set.n_templates; ++t) { if (set.class_of[t] < 0) return FL_ERR_ARG; nc = std::max(nc, set.class_of[t] + 1); }
  std::vector<int32_t> first((size_t)nc, -1);                                      // as fl_upload_templates numbers them (matchClass, :1458)
  for (int t = 0; t < set.n_templates; ++t) if (first[set.class_of[t]] < 0) first[set.class_of[t]] = t;
  const int64_t max_hyp = (int64_t)prm->top_k * (prm->per_class ? nc : 1);
  if (max_hyp > FL_RECO_MAX_HYP) { fl_set_error("fl_set_recognition: %lld hypotheses per frame > FL_RECO_MAX_HYP", (long long)max_hyp); return FL_ERR_CAPACITY; }
  FL_CUDA(cudaSetDevice(h->p.device));
  std::vector<fl_reco_tmpl> tab((size_t)set.n_templates);
  int max_pts = 16;
  bool any_crop = false;
  for (int t = 0; t < set.n_templates; ++t) {
    fl_reco_tmpl& e = tab[t];
    memset(&e, 0, sizeof e);
    const int c = crop_of_template[t];
    if (c < -1 || c >= (int)h->res_rect.size()) { fl_set_error("fl_set_recognition: crop %d of template %d is not in the uploaded set", c, t); return FL_ERR_ARG; }
    if (c >= 0) {
      const fl_rect_t& b = set.box0[t];                                             // current_template[0] (:111, :127-132)
      const fl_rect_t& r = h->res_rect[c];
      if (r.x != b.x || r.y != b.y || r.width != b.width || r.height != b.height) {
        fl_set_error("fl_set_recognition: crop %d was uploaded with a rect other than template %d's level-0 box", c, t); return FL_ERR_ARG;
      }
      e.crop = h->d_resident.get() + h->res_off[c]; e.rect = r;
      max_pts = std::max(max_pts, r.width * r.height);
      any_crop = true;
    }
    memcpy(e.pose, pose12 ? pose12 + (size_t)t * 12 : set.pose13 + (size_t)t * 13, 12 * sizeof(float));
  }
  h->reco_set = false;
  TRY(icp_reserve(h, (int)max_hyp, max_pts));                                     // now, so that no frame allocates
  TRY(h->d_reco_tmpl.alloc(tab.size()));
  FL_CUDA(cudaMemcpy(h->d_reco_tmpl.get(), tab.data(), tab.size() * sizeof(fl_reco_tmpl), cudaMemcpyHostToDevice));
  TRY(h->d_reco_class_first.alloc((size_t)nc));
  FL_CUDA(cudaMemcpy(h->d_reco_class_first.get(), first.data(), first.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  TRY(h->d_reco_sel.grow(FL_RECO_SEL_HDR + FL_RECO_MAX_HYP));
  TRY(h->h_reco.grow(FL_RECO_SUMMARY_WORDS + FL_RECO_MAX_HYP * sizeof(fl_reco_result_t) / sizeof(int)));
  FL_CUDA(cudaHostGetDevicePointer((void**)&h->d_reco_host, h->h_reco.get(), 0));
  h->reco = *prm; h->reco_max_hyp = (int)max_hyp; h->reco_any_crop = any_crop;
  h->reco_n_templates = set.n_templates; h->reco_n_classes = nc; h->reco_set = true;
  return FL_OK;
}

extern "C" int fl_set_recognition(fl_handle* h, const fl_reco_params_t* prm, const int32_t* crop_of_template, const float* pose12) {
  if (!h || !prm || !crop_of_template || prm->top_k < 1) return FL_ERR_ARG;
  TRY(frame_idle(h));
  if (h->n_templates == 0) { fl_set_error("fl_set_recognition: no templates uploaded"); return FL_ERR_STATE; }
  // matches carry the ids of fl_set_template_ids (a shard's global ids): the template behind a match is not class_first + template_id
  if (h->custom_tids) { fl_set_error("fl_set_recognition: not available on a handle with fl_set_template_ids (template shards)"); return FL_ERR_STATE; }
  FL_CUDA(cudaSetDevice(h->p.device));
  const size_t per = (size_t)h->p.n_levels * h->p.n_modalities;
  std::vector<fl_template_hdr_t> hdr((size_t)h->n_templates * per);
  FL_CUDA(cudaMemcpy(hdr.data(), h->d_hdr.get(), hdr.size() * sizeof(fl_template_hdr_t), cudaMemcpyDeviceToHost));
  std::vector<fl_rect_t> box0((size_t)h->n_templates);
  for (int t = 0; t < h->n_templates; ++t) { const fl_template_hdr_t& b = hdr[(size_t)t * per]; box0[t] = {b.offset_x, b.offset_y, b.width, b.height}; }
  const fl_reco_set set = {h->n_templates, h->class_of_h.data(), box0.data(), h->pose13_h.empty() ? nullptr : h->pose13_h.data()};
  return fl_reco_setup(h, prm, set, crop_of_template, pose12);
}

// selection -> ICP -> finish on the sorted list in d_out.  check_big: the list came from the fused refinement + sort, which leaves
// lists of more than 1,024 records unsorted and flagged (k_reco_select then selects nothing and reports the frame deferred).  push: the
// other ranks' mailboxes of a template-sharded pipe's frame that this handle owns, or NULL
static int reco_enqueue(fl_handle* h, bool check_big, const fl_reco_push* push = nullptr) {
  cudaStream_t s = h->stream.get();
  const int max_hyp = h->reco_max_hyp;
  int nl = fl_launch_reco_select(h->d_out, reinterpret_cast<const int*>(h->d_outblk.get()), h->p.max_candidates, check_big ? 1 : 0, h->d_reco_class_first.get(),
                                 h->reco_n_classes, h->reco_n_templates, h->d_reco_tmpl.get(), h->reco.top_k, h->reco.per_class, max_hyp, h->staged.W, h->staged.H,
                                 h->icpw.d_hyps.get(), h->d_reco_sel.get(), s);
  if (nl < 0) { fl_set_error("hypothesis selection launch failed: %s", cudaGetErrorString(cudaGetLastError())); return FL_ERR_CUDA; }
  h->launches += nl;
  fl_icp_ws ws = h->icp;
  ws.n_hyp = max_hyp;                                                              // padding hypotheses are skipped by the kernel
  nl = fl_launch_icp(ws, h->reco.icp, h->icpw.d_hyps.get(), h->d_in_depth.get(), h->staged.W, h->staged.H, h->frame.K, h->icpw.d_results.get(), h->icpw.d_ticket.get(), nullptr, h->n_sm, s);
  if (nl < 0) { fl_set_error("ICP kernel launch failed: %s", cudaGetErrorString(cudaGetLastError())); return FL_ERR_CUDA; }
  h->launches += nl;
  nl = fl_launch_reco_finish(h->d_out, h->d_reco_sel.get(), h->icpw.d_results.get(), max_hyp, h->reco.th_obj_dist, h->d_reco_host, push, s);
  if (nl < 0) { fl_set_error("recognition finish launch failed: %s", cudaGetErrorString(cudaGetLastError())); return FL_ERR_CUDA; }
  h->launches += nl;
  return FL_OK;
}

// the upload of a recognition frame (rescaled on the device when src_W x src_H differs from W x H, TImage2Mat :42) and its intrinsics
static int reco_stage(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int sW, int sH, int W, int H,
                      fl_intrinsics_t K_ref, fl_dev_frame* d) {
  if (!h || !depth || sW <= 0 || sH <= 0) return FL_ERR_ARG;
  TRY(frame_begin(h));
  if (!h->reco_set) { fl_set_error("fl_recognize: call fl_set_recognition after the template and crop uploads"); return FL_ERR_STATE; }
  TRY(stage_host(h, bgr, bgr_stride, depth, depth_stride, sW, sH, W, H, nullptr, d));
  if (h->reco_any_crop && (W != h->res_W || H != h->res_H)) { fl_set_error("model depth crops were uploaded for %d x %d frames, not %d x %d", h->res_W, h->res_H, W, H); return FL_ERR_STATE; }
  h->frame.K = K_ref;
  return FL_OK;
}

extern "C" int fl_recognize_async(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                                  int32_t sW, int32_t sH, int32_t W, int32_t H, fl_intrinsics_t K_ref) {
  fl_dev_frame d;
  TRY(reco_stage(h, bgr, bgr_stride, depth, depth_stride, sW, sH, W, H, K_ref, &d));
  TRY(fl_match_device_async(h, d.bgr, d.depth, W, H, nullptr, h->reco.threshold, nullptr, 0));
  TRY(reco_enqueue(h, true));
  h->frame.kind = fl_frame_kind::reco;
  return FL_OK;
}

// One member's part of a frame of a template-sharded group (fl_group_submit_recognition), in three steps that the group runs over all
// members in turn: fl_reco_shard_stage (upload [+ rescale] of the frame), fl_reco_shard_match (local match over the member's shard + the
// fused refinement / peer-memory exchange / sort of the staged frame, after which every member holds the merged list) and, on the
// frame's owner only, fl_reco_shard_tail (selection, ICP, finish on that list).  Nothing that may wait for the device - an allocation,
// the first launch of a kernel under lazy module loading - may run between one member's exchange launch and the last member's: the
// exchange kernel spins until every peer has published the frame.  The re-run after a front-end time-out calls the last two steps
// again on the frames already staged.
int fl_reco_shard_stage(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int sW, int sH, int W, int H,
                        fl_intrinsics_t K_ref) {
  fl_dev_frame d;
  return reco_stage(h, bgr, bgr_stride, depth, depth_stride, sW, sH, W, H, K_ref, &d);
}

int fl_reco_shard_match(fl_handle* h, int rank, int world, void* const* peers, int capacity, fl_match_t* block, uint32_t epoch) {
  if (!h) return FL_ERR_ARG;
  if (!h->reco_set || !h->staged.depth) { fl_set_error("no staged recognition frame on this handle"); return FL_ERR_STATE; }
  return fl_match_shard_exchange_device_async(h, h->staged.bgr ? h->d_in_bgr.get() : nullptr, h->d_in_depth.get(), h->staged.W, h->staged.H, h->reco.threshold,
                                              nullptr, 0, rank, world, peers, capacity, block, epoch);
}

int fl_reco_shard_tail(fl_handle* h, const fl_reco_push* push) {
  if (!h) return FL_ERR_ARG;
  if (h->frame.kind != fl_frame_kind::shard || !h->reco_set) { fl_set_error("no matched recognition frame on this handle"); return FL_ERR_STATE; }
  FL_CUDA(cudaSetDevice(h->p.device));
  TRY(reco_enqueue(h, true, push));
  h->frame.kind = fl_frame_kind::reco;
  return FL_OK;
}

int fl_reco_shard_receive(fl_handle* h, const uint8_t* own_buffer, size_t mailbox_off, uint32_t epoch, int owner) {
  if (!h || !own_buffer) return FL_ERR_ARG;
  if (h->frame.kind != fl_frame_kind::shard || !h->reco_set) { fl_set_error("no matched recognition frame on this handle"); return FL_ERR_STATE; }
  FL_CUDA(cudaSetDevice(h->p.device));
  if (fl_launch_reco_receive(own_buffer, mailbox_off, epoch, owner, h->d_reco_host, h->stream.get()) < 0) {
    fl_set_error("recognition receive launch failed: %s", cudaGetErrorString(cudaGetLastError())); return FL_ERR_CUDA;
  }
  ++h->launches;
  h->frame.kind = fl_frame_kind::reco;
  return FL_OK;
}

int fl_reco_shard_preload(fl_handle* h) {
  if (!h || !h->reco_set) return FL_ERR_STATE;
  FL_CUDA(cudaSetDevice(h->p.device));
  TRY(fl_reco_preload());
  return fl_icp_preload(h->icp.max_pts);
}

// after the frame's match wait: the tail once more on the final list when the selection ran on a list that was not sorted yet (or on a
// frame that has been re-run since), then the results and the summary
static int reco_results(fl_handle* h, bool rerun, fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary) {
  const volatile int* blk = h->h_reco.get();
  if (blk[FL_RECO_MISSING_OWNER]) { fl_set_error("owner rank %d did not post its results", blk[FL_RECO_MISSING_OWNER] - 1); return FL_ERR_STATE; }
  if ((blk[4] & FL_RECO_DEFERRED) || rerun) {
    TRY(reco_enqueue(h, false));
    FL_CUDA(wait_stream(h));
  }
  FL_CUDA(cudaGetLastError());
  if (h->overflow) {                                                             // matchClass produced more candidates than the buffers hold
    if (summary) summary->n_matches = h->h_small[0];
    fl_set_error("fl_recognize: more candidates than the handle's buffers hold (max_candidates, or the exchange capacity of a group)");
    return FL_ERR_CAPACITY;
  }
  const int n = blk[3];
  if (summary) { summary->n_matches = blk[0]; summary->n_hypotheses = blk[1]; summary->n_roi = blk[2]; summary->n_results = n; }
  if (std::min(n, (int)capacity) > 0) memcpy(out, h->h_reco.get() + FL_RECO_SUMMARY_WORDS, sizeof(fl_reco_result_t) * (size_t)std::min(n, (int)capacity));
  return n > capacity ? FL_ERR_CAPACITY : FL_OK;
}

// the owner's results of a group frame whose members have all been waited for (fl_match_wait)
int fl_reco_shard_results(fl_handle* h, fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary) {
  if (!h || capacity < 0 || (capacity > 0 && !out)) return FL_ERR_ARG;
  if (summary) memset(summary, 0, sizeof *summary);
  FL_CUDA(cudaSetDevice(h->p.device));
  return reco_results(h, false, out, capacity, summary);
}

extern "C" int fl_recognize_wait(fl_handle* h, fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary) {
  if (!h || capacity < 0 || (capacity > 0 && !out)) return FL_ERR_ARG;
  if (summary) memset(summary, 0, sizeof *summary);
  if (h->frame.kind != fl_frame_kind::reco) { fl_set_error("fl_recognize_wait: no recognition frame in flight on this handle"); return FL_ERR_STATE; }
  // the frame's one wait; the rare > 1,024-record sorts and the re-run after a front-end dependency time-out are fl_frame_wait's
  fl_wait_note note;
  TRY(fl_frame_wait(h, &note));
  return reco_results(h, note == fl_wait_note::rerun, out, capacity, summary);
}

extern "C" int fl_recognize(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                            int32_t sW, int32_t sH, int32_t W, int32_t H, fl_intrinsics_t K_ref,
                            fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary) {
  if (summary) memset(summary, 0, sizeof *summary);
  TRY(fl_recognize_async(h, bgr, bgr_stride, depth, depth_stride, sW, sH, W, H, K_ref));
  return fl_recognize_wait(h, out, capacity, summary);
}
