// fl_group: template-sharded matching over N handles of ONE process (one handle per GPU, or several on one GPU), for hosts that
// have no torch / NCCL / Python around - the reference's caller is a C++ class (CadReco/obj_reco_lmicp.cpp:86-204).
//
// The group has N members (one per entry of `devices`) and `depth` slots (fl_group_create_pipe; fl_group_create is depth 1).  Every
// (member, slot) pair owns a handle, an exchange buffer and a candidate block on the member's device; handle i = slot * N + member.
// Peer access is enabled between every pair of devices, so under unified addressing every handle's exchange buffer is reachable from
// every device with the pointer cudaMalloc returned: the kernel-side exchange (push into every peer's buffer, publish the epoch, wait
// for the peers' epochs, sort the union - the last CTA of k_refine_sort<1>) is the same one the one-process-per-GPU path uses with
// torch symmetric memory.  The members of one slot exchange with each other only, and every slot has its own epoch sequence.
// Templates are dealt round-robin by global index (gid % N) and carry their global per-class ids, so the merged list equals a single
// handle's (SURVEY.md 8e).  One fl_group_match = the frame copied to every device from the caller's buffers
// (fl_match_shard_exchange_async) on slot 0, ONE enqueue per handle, one wait per handle, the merged list read from handle 0.
//
// Recognition over the group (fl_group_submit_recognition / fl_group_collect_recognition): frame f goes to slot f % depth of every
// member.  Each member stages the frame, matches its shard and takes part in the exchange; after that launch every member of the slot
// holds the same merged list, and only the frame's owner, member f % N, enqueues the recognition tail (k_reco_select -> k_icp_fused ->
// k_reco_finish) on it.  ICP load is spread over the members frame by frame and nothing crosses devices after the exchange.  Every
// handle carries the selection table of the WHOLE set (built from the global class, box and pose tables the group keeps) and all crops,
// because any member can own a frame.
#include "fl_internal.cuh"
#include "fl_owned.cuh"
#include <algorithm>
#include <functional>
#include <vector>

struct fl_group {
  int n = 0, depth = 1, cap = 0;
  std::vector<int> device;                    // of member m
  std::vector<fl_handle*> h;                  // [slot * n + member]
  std::vector<fl_dev_buf<uint8_t>> xbuf;      // exchange buffer of handle i (on its member's device)
  std::vector<fl_dev_buf<fl_match_t>> block;  // candidate block [count | cap records] of handle i
  std::vector<void*> peers;                   // [slot * n + member] = xbuf as void* (the same array for every member: unified addressing)
  std::vector<uint32_t> epoch;                // last epoch of every slot
  int max_w = 0, max_h = 0;
  long long submitted = 0, collected = 0;     // recognition frames
  // the whole set as fl_group_upload_templates received it: the selection tables of fl_group_set_recognition are built from these
  std::vector<int32_t> class_of; std::vector<fl_rect_t> box0; std::vector<float> pose13;
  bool reco_set = false;
};

#define GCUDA(call)                                                                    \
  do {                                                                                 \
    cudaError_t e__ = (call);                                                          \
    if (e__ != cudaSuccess) {                                                          \
      fl_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return FL_ERR_CUDA;                                                              \
    }                                                                                  \
  } while (0)

static int in_flight(const fl_group* g) { return (int)(g->submitted - g->collected); }

// Waits for the frames of the first n members of a slot (hs): each one, whatever the others return; the first error counts.  A member
// whose single-launch front end timed out on an in-grid dependency has switched itself to per-wave launches and asks for the frame again
// (fl_frame_wait); every member has to take part in that, so `again`, when given, enqueues the frame once more on all of them.
static int wait_members(const fl_group* g, fl_handle* const* hs, int n, const char* what = nullptr, const std::function<int()>& again = nullptr) {
  for (int attempt = 0;; ++attempt) {
    int first_err = FL_OK;
    bool resubmit = false;
    for (int m = 0; m < n; ++m) {
      GCUDA(cudaSetDevice(g->device[m]));
      fl_wait_note note;
      const int rc = fl_frame_wait(hs[m], &note);
      if (note == fl_wait_note::resubmit) resubmit = true;
      else if (rc != FL_OK && first_err == FL_OK) first_err = rc;   // (incl. a peer that never arrived)
    }
    if (first_err != FL_OK || !resubmit || !again) return first_err;
    if (attempt == 1) { fl_set_error("%s: the front end timed out twice", what); return FL_ERR_STATE; }
    if ((first_err = again()) != FL_OK) return first_err;
  }
}

extern "C" int fl_group_destroy(fl_group* g) {
  if (!g) return FL_ERR_ARG;
  for (size_t i = 0; i < g->h.size(); ++i)                      // nothing may still read a buffer that is freed below
    if (g->h[i]) { cudaSetDevice(g->device[i % g->n]); fl_sync(g->h[i]); }
  for (size_t i = 0; i < g->h.size(); ++i) {
    cudaSetDevice(g->device[i % g->n]);
    if (i < g->xbuf.size()) g->xbuf[i].reset();
    if (i < g->block.size()) g->block[i].reset();
    if (g->h[i]) fl_destroy(g->h[i]);
  }
  delete g;
  return FL_OK;
}

extern "C" int fl_group_create_pipe(const fl_params_t* params, const int32_t* devices, int32_t n, int32_t exchange_capacity, int32_t depth, fl_group** out) {
  if (out) *out = nullptr;
  if (!params || !devices || !out || n < 1 || n > FL_XCHG_MAX_WORLD || exchange_capacity < 1 || depth < 1 || depth > FL_PIPE_MAX_DEPTH) return FL_ERR_ARG;
  fl_group* g = new fl_group;
  g->n = n; g->depth = depth; g->cap = exchange_capacity; g->max_w = params->max_width; g->max_h = params->max_height;
  const int nh = n * depth;
  g->device.assign(devices, devices + n); g->h.assign(nh, nullptr); g->xbuf.resize(nh); g->block.resize(nh);
  g->peers.assign(nh, nullptr); g->epoch.assign(depth, 0u);
  auto fail = [&](int rc) { fl_group_destroy(g); return rc; };
  // peer access between every pair of distinct devices (already enabled is fine)
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) {
      if (devices[i] == devices[j]) continue;
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, devices[i], devices[j]) != cudaSuccess || !can) {
        fl_set_error("device %d cannot access device %d directly (no NVLink / PCIe peer path)", devices[i], devices[j]);
        return fail(FL_ERR_CUDA);
      }
      if (cudaSetDevice(devices[i]) != cudaSuccess) return fail(FL_ERR_CUDA);
      const cudaError_t e = cudaDeviceEnablePeerAccess(devices[j], 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { fl_set_error("cudaDeviceEnablePeerAccess(%d -> %d): %s", devices[i], devices[j], cudaGetErrorString(e)); return fail(FL_ERR_CUDA); }
      cudaGetLastError();
    }
  const size_t xbytes = fl_exchange_buffer_bytes(n, exchange_capacity);
  const size_t bbytes = sizeof(fl_match_t) * ((size_t)exchange_capacity + 1);
  for (int i = 0; i < nh; ++i) {
    const int dev = devices[i % n];
    fl_params_t p = *params;
    p.device = dev;
    p.max_candidates = std::max(p.max_candidates, n * (exchange_capacity + 1) + 16);
    int rc = fl_create(&p, &g->h[i]);
    if (rc != FL_OK) return fail(rc);
    if (cudaSetDevice(dev) != cudaSuccess) return fail(FL_ERR_CUDA);
    if ((rc = g->xbuf[i].alloc(xbytes)) != FL_OK || (rc = g->block[i].alloc((size_t)exchange_capacity + 1)) != FL_OK) return fail(rc);
    if (cudaMemset(g->xbuf[i].get(), 0, xbytes) != cudaSuccess || cudaMemset(g->block[i].get(), 0, bbytes) != cudaSuccess) {
      fl_set_error("fl_group_create: cudaMemset failed on device %d: %s", dev, cudaGetErrorString(cudaGetLastError()));
      return fail(FL_ERR_CUDA);
    }
    g->peers[i] = g->xbuf[i].get();
  }
  for (int i = 0; i < n; ++i) { cudaSetDevice(devices[i]); cudaDeviceSynchronize(); }
  *out = g;
  return FL_OK;
}

extern "C" int fl_group_create(const fl_params_t* params, const int32_t* devices, int32_t n, int32_t exchange_capacity, fl_group** out) {
  return fl_group_create_pipe(params, devices, n, exchange_capacity, 1, out);
}

extern "C" fl_handle* fl_group_handle(fl_group* g, int32_t i) { return (g && i >= 0 && i < (int)g->h.size()) ? g->h[i] : nullptr; }
extern "C" int32_t fl_group_size(const fl_group* g) { return g ? g->n : 0; }
extern "C" int32_t fl_group_depth(const fl_group* g) { return g ? g->depth : 0; }
extern "C" int32_t fl_group_in_flight(const fl_group* g) { return g ? in_flight(g) : 0; }

// the whole set (layout of fl_upload_templates): template gid goes to member gid % n with its global per-class id, on every slot
extern "C" int fl_group_upload_templates(fl_group* g, int32_t n_templates, const fl_template_hdr_t* headers, const fl_feature_t* features, int32_t n_features,
                                         const int32_t* class_of, const float* pose13) {
  if (!g || n_templates < 0 || (n_templates > 0 && (!headers || !features || !class_of))) return FL_ERR_ARG;
  if (in_flight(g)) { fl_set_error("fl_group_upload_templates: %d frame(s) still in flight", in_flight(g)); return FL_ERR_STATE; }
  const int LM = fl_entries_per_template(g->h[0]);               // n_levels * n_modalities headers per template
  if (LM <= 0) return FL_ERR_STATE;
  std::vector<int32_t> first;                                   // first global index of every class
  for (int t = 0; t < n_templates; ++t) {
    const int c = class_of[t];
    if (c < 0) return FL_ERR_ARG;
    if ((int)first.size() <= c) first.resize((size_t)c + 1, -1);
    if (first[c] < 0) first[c] = t;
  }
  g->reco_set = false;
  g->class_of.clear(); g->box0.clear(); g->pose13.clear();
  for (int r = 0; r < g->n; ++r) {
    std::vector<fl_template_hdr_t> hs;
    std::vector<fl_feature_t> fs;
    std::vector<int32_t> co, ids;
    std::vector<float> pose;
    for (int t = r; t < n_templates; t += g->n) {
      for (int e = 0; e < LM; ++e) {
        fl_template_hdr_t hd = headers[(size_t)t * LM + e];
        if (hd.feature_begin < 0 || hd.feature_count < 0 || hd.feature_begin + hd.feature_count > n_features) return FL_ERR_ARG;
        const int32_t b = (int32_t)fs.size();
        fs.insert(fs.end(), features + hd.feature_begin, features + hd.feature_begin + hd.feature_count);
        hd.feature_begin = b;
        hs.push_back(hd);
      }
      co.push_back(class_of[t]);
      ids.push_back(t - first[class_of[t]]);
      if (pose13) pose.insert(pose.end(), pose13 + (size_t)t * 13, pose13 + (size_t)t * 13 + 13);
    }
    const int nt = (int)co.size();
    fl_feature_t dummy = {0, 0, 0};
    for (int s = 0; s < g->depth; ++s) {
      fl_handle* h = g->h[(size_t)s * g->n + r];
      int rc = fl_upload_templates(h, nt, nt ? hs.data() : nullptr, fs.empty() ? &dummy : fs.data(), (int32_t)fs.size(), nt ? co.data() : nullptr,
                                   pose13 && nt ? pose.data() : nullptr);
      if (rc != FL_OK) return rc;
      if (nt) { rc = fl_set_template_ids(h, ids.data()); if (rc != FL_OK) return rc; }
    }
  }
  g->class_of.assign(class_of, class_of + n_templates);
  g->box0.resize((size_t)n_templates);
  for (int t = 0; t < n_templates; ++t) {                         // level-0 modality-0 box (current_template[0], :111, :127-132)
    const fl_template_hdr_t& b = headers[(size_t)t * LM];
    g->box0[t] = {b.offset_x, b.offset_y, b.width, b.height};
  }
  if (pose13) g->pose13.assign(pose13, pose13 + (size_t)n_templates * 13);
  return FL_OK;
}

// Detector::match over the whole (sharded) set, on slot 0.  Host buffers in, merged host list out; every handle of the slot ends up
// with the same list.
// masks (NULL or n_modalities host pointers, layout of fl_match) are staged into every member's own mask buffers (allocated at fl_create):
// no member allocates between its peers' exchange launches.
extern "C" int fl_group_match_masked(fl_group* g, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int32_t W, int32_t H,
                                     const uint8_t* const* masks, float threshold, const int32_t* class_filter, int32_t n_filter, fl_match_t* out,
                                     int32_t capacity, int32_t* count) {
  if (!g || !count || (!bgr && !depth)) return FL_ERR_ARG;
  *count = 0;
  if (in_flight(g)) { fl_set_error("fl_group_match: %d recognition frame(s) in flight - collect them first", in_flight(g)); return FL_ERR_STATE; }
  if (W <= 0 || H <= 0 || W > g->max_w || H > g->max_h) return FL_ERR_SIZE;
  if ((bgr && bgr_stride < (size_t)W * 3) || (depth && depth_stride < (size_t)W * 2)) return FL_ERR_SIZE;
  auto enqueue = [&]() -> int {                                 // on every handle; nothing waits until all are under way
    const uint32_t e = ++g->epoch[0];
    for (int i = 0; i < g->n; ++i) {
      GCUDA(cudaSetDevice(g->device[i]));
      const int rc = fl_match_shard_exchange_masked_async(g->h[i], bgr, bgr_stride, depth, depth_stride, W, H, masks, threshold, class_filter, n_filter,
                                                          i, g->n, g->peers.data(), g->cap, g->block[i].get(), e);
      if (rc != FL_OK) { wait_members(g, g->h.data(), i); return rc; }   // (the ranks already launched report the missing peer instead of hanging)
    }
    return FL_OK;
  };
  int rc = enqueue();
  if (rc == FL_OK) rc = wait_members(g, g->h.data(), g->n, "fl_group_match", enqueue);
  if (rc != FL_OK) return rc;
  GCUDA(cudaSetDevice(g->device[0]));
  return fl_match_fetch(g->h[0], out, capacity, count);
}
extern "C" int fl_group_match(fl_group* g, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int32_t W, int32_t H,
                              float threshold, const int32_t* class_filter, int32_t n_filter, fl_match_t* out, int32_t capacity, int32_t* count) {
  return fl_group_match_masked(g, bgr, bgr_stride, depth, depth_stride, W, H, nullptr, threshold, class_filter, n_filter, out, capacity, count);
}

// ---- Recognition over the group -----------------------------------------------------------------------------------------------
// the crops go to every slot of every member: any member can own a frame
extern "C" int fl_group_upload_model_depths(fl_group* g, int32_t n_models, const uint16_t* const* model_depth, const size_t* model_stride,
                                            const fl_rect_t* rect_model, int32_t W, int32_t H) {
  if (!g) return FL_ERR_ARG;
  if (in_flight(g)) { fl_set_error("fl_group_upload_model_depths: %d frame(s) still in flight", in_flight(g)); return FL_ERR_STATE; }
  g->reco_set = false;
  for (fl_handle* h : g->h) {
    const int rc = fl_upload_model_depths(h, n_models, model_depth, model_stride, rect_model, W, H);
    if (rc != FL_OK) return rc;
  }
  return FL_OK;
}

// crop_of_template / pose12 cover the whole set in the order of fl_group_upload_templates; every handle gets the selection table of
// that set (fl_reco_setup), so that whichever member owns a frame selects from the merged list as a single handle would
extern "C" int fl_group_set_recognition(fl_group* g, const fl_reco_params_t* params, const int32_t* crop_of_template, const float* pose12) {
  if (!g || !params || !crop_of_template) return FL_ERR_ARG;
  if (in_flight(g)) { fl_set_error("fl_group_set_recognition: %d frame(s) still in flight", in_flight(g)); return FL_ERR_STATE; }
  g->reco_set = false;
  const fl_reco_set set = {(int)g->class_of.size(), g->class_of.data(), g->box0.data(), g->pose13.empty() ? nullptr : g->pose13.data()};
  for (fl_handle* h : g->h) {
    const int rc = fl_reco_setup(h, params, set, crop_of_template, pose12);
    if (rc != FL_OK) return rc;
  }
  g->reco_set = true;
  return FL_OK;
}

// every member of slot `s` runs its part of frame f; `restage` = false runs the frames already staged on the members again.  Each step
// runs on every member before the next one starts: the uploads, rescales and their allocations before any exchange kernel is under
// way, and the owner's tail only once every member's exchange has been launched - a member that waited for the device in between
// (an allocation, the first launch of a tail kernel under lazy module loading) would wait for an exchange kernel that waits for it.
static int enqueue_frame(fl_group* g, int s, long long f, bool restage, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                         int32_t sW, int32_t sH, int32_t W, int32_t H, fl_intrinsics_t K_ref) {
  const int owner = (int)(f % g->n);
  fl_handle* const* hs = g->h.data() + (size_t)s * g->n;
  if (restage)
    for (int m = 0; m < g->n; ++m) {
      GCUDA(cudaSetDevice(g->device[m]));
      const int rc = fl_reco_shard_stage(hs[m], bgr, bgr_stride, depth, depth_stride, sW, sH, W, H, K_ref);
      if (rc != FL_OK) { for (int k = 0; k <= m; ++k) { cudaSetDevice(g->device[k]); fl_sync(hs[k]); } return rc; }   // nothing launched yet
    }
  const uint32_t e = ++g->epoch[s];
  for (int m = 0; m < g->n; ++m) {
    int rc = cudaSetDevice(g->device[m]) == cudaSuccess ? FL_OK : FL_ERR_CUDA;
    if (rc == FL_OK) rc = fl_reco_shard_match(hs[m], m, g->n, g->peers.data() + (size_t)s * g->n, g->cap, g->block[(size_t)s * g->n + m].get(), e);
    // the members already under way report the missing peer instead of hanging: wait for them, so that the slot is free again
    if (rc != FL_OK) { wait_members(g, hs, m); return rc; }
  }
  int rc = cudaSetDevice(g->device[owner]) == cudaSuccess ? FL_OK : FL_ERR_CUDA;
  if (rc == FL_OK) rc = fl_reco_shard_tail(hs[owner]);
  if (rc != FL_OK) { wait_members(g, hs, g->n); return rc; }
  return FL_OK;
}

extern "C" int fl_group_submit_recognition(fl_group* g, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                                           int32_t src_W, int32_t src_H, int32_t W, int32_t H, fl_intrinsics_t K_ref) {
  if (!g || !depth || src_W <= 0 || src_H <= 0) return FL_ERR_ARG;
  if (in_flight(g) >= g->depth) { fl_set_error("fl_group_submit_recognition: %d frames in flight already - collect one first", g->depth); return FL_ERR_STATE; }
  if (!g->reco_set) { fl_set_error("fl_group_submit_recognition: call fl_group_set_recognition after the template and crop uploads"); return FL_ERR_STATE; }
  const long long f = g->submitted;
  const int rc = enqueue_frame(g, (int)(f % g->depth), f, true, bgr, bgr_stride, depth, depth_stride, src_W, src_H, W, H, K_ref);
  if (rc != FL_OK) return rc;
  ++g->submitted;
  return FL_OK;
}

// The oldest frame: every member of its slot is waited for (a missing peer or an overflowing exchange block is this frame's status).
// A member whose front end timed out has switched itself to per-wave launches: the frame then runs again on every member of the slot
// from the frames they staged, with the slot's next epoch, the owner's tail included.  The owner posts the results.
extern "C" int fl_group_collect_recognition(fl_group* g, fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary) {
  if (!g || capacity < 0 || (capacity > 0 && !out)) return FL_ERR_ARG;
  if (summary) memset(summary, 0, sizeof *summary);
  if (!in_flight(g)) { fl_set_error("fl_group_collect_recognition: no frame in flight"); return FL_ERR_STATE; }
  const long long f = g->collected++;                           // the slot is free again whatever the frame's status
  const int s = (int)(f % g->depth), owner = (int)(f % g->n);
  fl_handle* const* hs = g->h.data() + (size_t)s * g->n;
  const int rc = wait_members(g, hs, g->n, "fl_group_collect_recognition", [&]() {
    const fl_intrinsics_t none = {0.f, 0.f, 0.f, 0.f};           // (restage = false: each handle keeps the frame's geometry and intrinsics)
    return enqueue_frame(g, s, f, false, nullptr, 0, nullptr, 0, 0, 0, 0, 0, none);
  });
  if (rc != FL_OK) return rc;
  GCUDA(cudaSetDevice(g->device[owner]));
  return fl_reco_shard_results(hs[owner], out, capacity, summary);
}

extern "C" int fl_group_recognize(fl_group* g, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                                  int32_t src_W, int32_t src_H, int32_t W, int32_t H, fl_intrinsics_t K_ref,
                                  fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary) {
  if (summary) memset(summary, 0, sizeof *summary);
  if (g && in_flight(g)) { fl_set_error("fl_group_recognize: %d frame(s) in flight - collect them first", in_flight(g)); return FL_ERR_STATE; }
  const int rc = fl_group_submit_recognition(g, bgr, bgr_stride, depth, depth_stride, src_W, src_H, W, H, K_ref);
  if (rc != FL_OK) return rc;
  return fl_group_collect_recognition(g, out, capacity, summary);
}
