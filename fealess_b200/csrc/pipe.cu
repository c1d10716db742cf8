// fl_pipe: Detector::match over a STREAM of frames with several frames in flight on one GPU.
//
// One frame through a handle is three dependent launches (front end -> similarity -> refinement + sort) whose first and last have
// far fewer CTAs than the GPU has SM slots, followed by a host wait: a single handle leaves ~40 % of the SM time idle (DESIGN.md).
// The reference's caller loops over camera frames (CadReco/obj_reco_lmicp.cpp:86-204, test/linemod_acq.cpp:120-190) - the frames are
// independent, so the pipe owns `depth` handles on one device (each with the whole template set, its own stream, linear memories,
// candidate and result blocks), deals the submitted frames round-robin and hands the match lists back in submission order.  The GPU
// runs the front end of frame i+1 in the SM slots the similarity kernel of frame i leaves free and under its tail; the upload of
// frame i+1 and the result copy of frame i-1 ride on the copy engines meanwhile.  Nothing here synchronises more than one stream.
// fl_pipe_set_exchange turns the pipe into ONE RANK of a template-sharded detector: every slot then runs the fused local match +
// peer-memory exchange (fl_match_shard_exchange_*) with its own exchange buffers and epoch sequence, so a rank's whole per-frame host
// loop - upload, enqueue, wait, fetch - lives in fl_pipe_match_batch.  Recognition on such a pipe (fl_pipe_set_recognition_sharded):
// every rank matches its shard and takes part in the exchange, only the frame's owner (rank f % world) runs selection, ICP and
// suppression, and its k_reco_finish pushes the results into the other ranks' mailboxes, where their k_reco_receive picks them up.
#include "fl_internal.cuh"
#include <vector>

struct fl_pipe {
  int depth, device;
  std::vector<fl_handle*> h;
  long long submitted, collected;
  // template-sharded mode (fl_pipe_set_exchange): this pipe is rank `rank` of `world`; slot i owns exchange buffers peers[i * world ..]
  // and the candidate block blocks[i]; its frames carry the epochs 1, 2, 3 ... of that slot
  int rank, world, xcap;
  std::vector<void*> peers;
  std::vector<fl_match_t*> blocks;
  std::vector<uint32_t> epoch;
  bool reco_sharded = false;        // fl_pipe_set_recognition_sharded has set up every slot
};

extern "C" int fl_pipe_destroy(fl_pipe* p) {
  if (!p) return FL_ERR_ARG;
  for (fl_handle* h : p->h) if (h) { fl_sync(h); fl_destroy(h); }
  delete p;
  return FL_OK;
}

extern "C" int fl_pipe_create(const fl_params_t* params, int32_t depth, fl_pipe** out) {
  if (!params || !out || depth < 1 || depth > FL_PIPE_MAX_DEPTH) return FL_ERR_ARG;
  *out = nullptr;
  fl_pipe* p = new fl_pipe;
  p->depth = depth; p->device = params->device; p->submitted = p->collected = 0; p->rank = 0; p->world = 1; p->xcap = 0;
  p->h.assign(depth, nullptr);
  for (int i = 0; i < depth; ++i) {
    const int rc = fl_create(params, &p->h[i]);
    if (rc != FL_OK) { fl_pipe_destroy(p); return rc; }
  }
  *out = p;
  return FL_OK;
}

extern "C" int32_t fl_pipe_depth(const fl_pipe* p) { return p ? p->depth : 0; }
extern "C" int32_t fl_pipe_in_flight(const fl_pipe* p) { return p ? (int32_t)(p->submitted - p->collected) : 0; }
extern "C" fl_handle* fl_pipe_handle(fl_pipe* p, int32_t i) { return (p && i >= 0 && i < p->depth) ? p->h[i] : nullptr; }

extern "C" int fl_pipe_upload_templates(fl_pipe* p, int32_t n_templates, const fl_template_hdr_t* headers, const fl_feature_t* features, int32_t n_features,
                                        const int32_t* class_of, const float* pose13) {
  if (!p) return FL_ERR_ARG;
  if (p->submitted != p->collected) { fl_set_error("fl_pipe_upload_templates: %lld frame(s) still in flight", p->submitted - p->collected); return FL_ERR_STATE; }
  p->reco_sharded = false;
  for (fl_handle* h : p->h) {
    const int rc = fl_upload_templates(h, n_templates, headers, features, n_features, class_of, pose13);
    if (rc != FL_OK) return rc;
  }
  return FL_OK;
}

// Template-sharded pipe: every rank (process or fl_pipe) of a `world`-way sharded detector calls this once, after uploading its shard
// (fl_pipe_upload_templates) and its global template ids (fl_set_template_ids on fl_pipe_handle(p, i)).  peer_buffers: depth x world
// pointers - entry [i * world + r] is rank r's exchange buffer OF SLOT i as mapped into this process (fl_exchange_buffer_bytes each,
// zeroed once); local_blocks: depth device blocks of exchange_capacity + 1 records.  From then on fl_pipe_submit runs
// fl_match_shard_exchange_(device_)async: all ranks have to submit the same sequence of frames.
extern "C" int fl_pipe_set_exchange(fl_pipe* p, int32_t rank, int32_t world, int32_t exchange_capacity, void* const* peer_buffers, fl_match_t* const* local_blocks) {
  if (!p || world < 1 || rank < 0 || rank >= world || exchange_capacity < 1 || !peer_buffers || !local_blocks) return FL_ERR_ARG;
  if (p->submitted != p->collected) { fl_set_error("fl_pipe_set_exchange: %lld frame(s) still in flight", p->submitted - p->collected); return FL_ERR_STATE; }
  for (int i = 0; i < p->depth; ++i) {
    if (!local_blocks[i]) return FL_ERR_ARG;
    for (int r = 0; r < world; ++r) if (!peer_buffers[(size_t)i * world + r]) return FL_ERR_ARG;
  }
  p->rank = rank; p->world = world; p->xcap = exchange_capacity; p->reco_sharded = false;
  p->peers.assign(peer_buffers, peer_buffers + (size_t)p->depth * world);
  p->blocks.assign(local_blocks, local_blocks + p->depth);
  p->epoch.assign(p->depth, 0u);
  return FL_OK;
}

extern "C" int fl_pipe_submit_masked(fl_pipe* p, const void* bgr, size_t bgr_stride, const void* depth, size_t depth_stride, int32_t W, int32_t H,
                                     const void* const* masks, float threshold, const int32_t* class_filter, int32_t n_filter, int32_t on_device) {
  if (!p || (!bgr && !depth)) return FL_ERR_ARG;
  if (p->submitted - p->collected >= p->depth) { fl_set_error("fl_pipe_submit: %d frames in flight already - collect one first", p->depth); return FL_ERR_STATE; }
  const int slot = (int)(p->submitted % p->depth);
  fl_handle* h = p->h[slot];
  if (on_device && ((bgr && bgr_stride != (size_t)W * 3) || (depth && depth_stride != (size_t)W * 2))) { fl_set_error("fl_pipe_submit: device frames must have dense rows"); return FL_ERR_SIZE; }
  int rc;
  if (p->world > 1) {                                           // template-sharded: local match + peer-memory exchange + merge, one enqueue
    void* const* peers = p->peers.data() + (size_t)slot * p->world;
    const uint32_t e = p->epoch[slot] + 1;
    rc = on_device ? fl_match_shard_exchange_device_masked_async(h, bgr, depth, W, H, masks, threshold, class_filter, n_filter, p->rank, p->world, peers, p->xcap,
                                                                 p->blocks[slot], e)
                   : fl_match_shard_exchange_masked_async(h, static_cast<const uint8_t*>(bgr), bgr_stride, static_cast<const uint16_t*>(depth), depth_stride, W, H,
                                                          reinterpret_cast<const uint8_t* const*>(masks), threshold, class_filter, n_filter, p->rank, p->world,
                                                          peers, p->xcap, p->blocks[slot], e);
    if (rc == FL_OK) p->epoch[slot] = e;
  } else if (on_device) {
    rc = fl_match_device_async(h, bgr, depth, W, H, masks, threshold, class_filter, n_filter);
  } else {
    rc = fl_match_async(h, static_cast<const uint8_t*>(bgr), bgr_stride, static_cast<const uint16_t*>(depth), depth_stride, W, H,
                        reinterpret_cast<const uint8_t* const*>(masks), threshold, class_filter, n_filter);
  }
  if (rc != FL_OK) return rc;
  ++p->submitted;
  return FL_OK;
}
extern "C" int fl_pipe_submit(fl_pipe* p, const void* bgr, size_t bgr_stride, const void* depth, size_t depth_stride, int32_t W, int32_t H, float threshold,
                              const int32_t* class_filter, int32_t n_filter, int32_t on_device) {
  return fl_pipe_submit_masked(p, bgr, bgr_stride, depth, depth_stride, W, H, nullptr, threshold, class_filter, n_filter, on_device);
}

extern "C" int fl_pipe_collect(fl_pipe* p, fl_match_t* out, int32_t capacity, int32_t* count) {
  if (!p || !count) return FL_ERR_ARG;
  *count = 0;
  if (p->submitted == p->collected) { fl_set_error("fl_pipe_collect: no frame in flight"); return FL_ERR_STATE; }
  fl_handle* h = p->h[p->collected % p->depth];
  ++p->collected;                                               // the slot is free again whatever the frame's status
  const int rc = fl_match_wait(h);
  if (rc != FL_OK) return rc;
  return fl_match_fetch(h, out, capacity, count);
}

// n frames of one geometry through the pipe: frame f's list goes to out + f * capacity_per_frame, its length (before truncation)
// to counts[f].  Returns the first error; FL_ERR_CAPACITY if some list did not fit (the others are complete).
extern "C" int fl_pipe_match_batch(fl_pipe* p, int32_t n_frames, const void* const* bgr, size_t bgr_stride, const void* const* depth, size_t depth_stride,
                                   int32_t W, int32_t H, float threshold, const int32_t* class_filter, int32_t n_filter, int32_t on_device,
                                   fl_match_t* out, int32_t capacity_per_frame, int32_t* counts) {
  if (!p || n_frames < 0 || (!bgr && !depth) || !counts || capacity_per_frame < 0 || (capacity_per_frame > 0 && !out)) return FL_ERR_ARG;
  if (p->submitted != p->collected) { fl_set_error("fl_pipe_match_batch: %lld frame(s) still in flight", p->submitted - p->collected); return FL_ERR_STATE; }
  int status = FL_OK, next_out = 0;
  auto collect = [&]() -> int {
    const int rc = fl_pipe_collect(p, out + (size_t)next_out * capacity_per_frame, capacity_per_frame, counts + next_out);
    ++next_out;
    if (rc == FL_ERR_CAPACITY) { if (status == FL_OK) status = rc; return FL_OK; }
    return rc;
  };
  for (int f = 0; f < n_frames; ++f) {
    if (fl_pipe_in_flight(p) == p->depth) { const int rc = collect(); if (rc != FL_OK) { while (fl_pipe_in_flight(p)) { int32_t c; fl_pipe_collect(p, nullptr, 0, &c); } return rc; } }
    const int rc = fl_pipe_submit(p, bgr ? bgr[f] : nullptr, bgr_stride, depth ? depth[f] : nullptr, depth_stride, W, H, threshold, class_filter, n_filter, on_device);
    if (rc != FL_OK) { while (fl_pipe_in_flight(p)) { int32_t c; fl_pipe_collect(p, nullptr, 0, &c); } return rc; }
  }
  while (fl_pipe_in_flight(p)) { const int rc = collect(); if (rc != FL_OK) { while (fl_pipe_in_flight(p)) { int32_t c; fl_pipe_collect(p, nullptr, 0, &c); } return rc; } }
  return status;
}

// Recognition over the pipe (fl_recognize_async / fl_recognize_wait per slot): one host thread keeps `depth` whole frames - match, ICP,
// suppression - in flight, and takes their results back in submission order.  The crops and the recognition setup go to every slot.
extern "C" int fl_pipe_upload_model_depths(fl_pipe* p, int32_t n_models, const uint16_t* const* model_depth, const size_t* model_stride,
                                           const fl_rect_t* rect_model, int32_t W, int32_t H) {
  if (!p) return FL_ERR_ARG;
  if (p->submitted != p->collected) { fl_set_error("fl_pipe_upload_model_depths: %lld frame(s) still in flight", p->submitted - p->collected); return FL_ERR_STATE; }
  p->reco_sharded = false;
  for (fl_handle* h : p->h) {
    const int rc = fl_upload_model_depths(h, n_models, model_depth, model_stride, rect_model, W, H);
    if (rc != FL_OK) return rc;
  }
  return FL_OK;
}

extern "C" int fl_pipe_set_recognition(fl_pipe* p, const fl_reco_params_t* params, const int32_t* crop_of_template, const float* pose12) {
  if (!p) return FL_ERR_ARG;
  if (p->world > 1) { fl_set_error("fl_pipe_set_recognition: a template-sharded pipe takes fl_pipe_set_recognition_sharded"); return FL_ERR_STATE; }
  if (p->submitted != p->collected) { fl_set_error("fl_pipe_set_recognition: %lld frame(s) still in flight", p->submitted - p->collected); return FL_ERR_STATE; }
  for (fl_handle* h : p->h) {
    const int rc = fl_set_recognition(h, params, crop_of_template, pose12);
    if (rc != FL_OK) return rc;
  }
  return FL_OK;
}

// Recognition on a template-sharded pipe.  Every slot's handle gets the selection table of the WHOLE set (the ranks hold only their
// shards), and every kernel its frames launch is loaded here: after a rank's exchange launch nothing may wait for the device, since
// the exchange kernel spins until the peers arrive (group.cu explains the same hazard for a group).
extern "C" int fl_pipe_set_recognition_sharded(fl_pipe* p, const fl_reco_params_t* params, int32_t n_templates, const fl_template_hdr_t* headers,
                                               const int32_t* class_of, const int32_t* crop_of_template, const float* pose12) {
  if (!p || !params || n_templates < 0 || (n_templates > 0 && (!headers || !class_of)) || !crop_of_template || !pose12) return FL_ERR_ARG;
  if (p->world <= 1) { fl_set_error("fl_pipe_set_recognition_sharded: not a template-sharded pipe (fl_pipe_set_exchange, world > 1)"); return FL_ERR_STATE; }
  if (p->submitted != p->collected) { fl_set_error("fl_pipe_set_recognition_sharded: %lld frame(s) still in flight", p->submitted - p->collected); return FL_ERR_STATE; }
  p->reco_sharded = false;
  const int LM = fl_entries_per_template(p->h[0]);                 // level-0 modality-0 box of every template (current_template[0], :111)
  std::vector<fl_rect_t> box0((size_t)n_templates);
  for (int t = 0; t < n_templates; ++t) { const fl_template_hdr_t& b = headers[(size_t)t * LM]; box0[t] = {b.offset_x, b.offset_y, b.width, b.height}; }
  const fl_reco_set set = {n_templates, class_of, box0.data(), nullptr};
  for (fl_handle* h : p->h) {
    int rc = fl_reco_setup(h, params, set, crop_of_template, pose12);
    if (rc == FL_OK) rc = fl_reco_shard_preload(h);
    if (rc != FL_OK) return rc;
  }
  p->reco_sharded = true;
  return FL_OK;
}

// frame f of a template-sharded pipe on slot f % depth: stage, match the shard + exchange, then the tail with the push to the other
// ranks on the frame's owner (rank f % world), the receive of the owner's results everywhere else
static int submit_recognition_sharded(fl_pipe* p, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                                      int32_t src_W, int32_t src_H, int32_t W, int32_t H, fl_intrinsics_t K_ref) {
  if (!p->reco_sharded) { fl_set_error("fl_pipe_submit_recognition: call fl_pipe_set_recognition_sharded after the template and crop uploads"); return FL_ERR_STATE; }
  const long long f = p->submitted;
  const int slot = (int)(f % p->depth), owner = (int)(f % p->world);
  fl_handle* h = p->h[slot];
  void* const* peers = p->peers.data() + (size_t)slot * p->world;
  const size_t mbox = fl_reco_mailbox_offset(p->world, p->xcap);
  int rc = fl_reco_shard_stage(h, bgr, bgr_stride, depth, depth_stride, src_W, src_H, W, H, K_ref);
  if (rc != FL_OK) return rc;                                   // nothing launched that a peer waits for
  const uint32_t e = p->epoch[slot] + 1;
  rc = fl_reco_shard_match(h, p->rank, p->world, peers, p->xcap, p->blocks[slot], e);
  if (rc != FL_OK) return rc;
  p->epoch[slot] = e;
  if (owner == p->rank) {
    fl_reco_push push;
    memset(&push, 0, sizeof push);
    push.epoch = e; push.mailbox_off = mbox;
    for (int r = 0; r < p->world; ++r) if (r != p->rank) push.peer[push.n++] = static_cast<uint8_t*>(peers[r]);
    rc = fl_reco_shard_tail(h, &push);
  } else {
    rc = fl_reco_shard_receive(h, static_cast<const uint8_t*>(peers[p->rank]), mbox, e, owner);
  }
  if (rc != FL_OK) { fl_match_wait(h); return rc; }              // the exchange is under way: wait for it, so that the slot is free again
  return FL_OK;
}

extern "C" int fl_pipe_submit_recognition(fl_pipe* p, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                                          int32_t src_W, int32_t src_H, int32_t W, int32_t H, fl_intrinsics_t K_ref) {
  if (!p) return FL_ERR_ARG;
  if (p->submitted - p->collected >= p->depth) { fl_set_error("fl_pipe_submit_recognition: %d frames in flight already - collect one first", p->depth); return FL_ERR_STATE; }
  const int rc = p->world > 1 ? submit_recognition_sharded(p, bgr, bgr_stride, depth, depth_stride, src_W, src_H, W, H, K_ref)
                              : fl_recognize_async(p->h[p->submitted % p->depth], bgr, bgr_stride, depth, depth_stride, src_W, src_H, W, H, K_ref);
  if (rc != FL_OK) return rc;
  ++p->submitted;
  return FL_OK;
}

extern "C" int fl_pipe_collect_recognition(fl_pipe* p, fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary) {
  if (!p) return FL_ERR_ARG;
  if (summary) memset(summary, 0, sizeof *summary);
  if (p->submitted == p->collected) { fl_set_error("fl_pipe_collect_recognition: no frame in flight"); return FL_ERR_STATE; }
  fl_handle* h = p->h[p->collected % p->depth];
  // the oldest frame came from fl_pipe_submit: it stays in flight for fl_pipe_collect (waiting for it here would leave nothing to fetch)
  if (fl_frame_in_flight(h) != fl_frame_kind::reco) { fl_set_error("fl_pipe_collect_recognition: the oldest frame in flight is a match frame - fl_pipe_collect it"); return FL_ERR_STATE; }
  ++p->collected;                                               // the slot is free again whatever the frame's status
  if (p->world > 1) {
    // a missing peer or owner, an overflowing exchange block: this frame's status only.  A deferred list (more than the 1,024 records
    // the fused sort holds) was sorted by the wait; every rank then runs the tail itself on its copy of it (fl_reco_shard_results)
    const int rc = fl_match_wait(h);
    if (rc != FL_OK) return rc;
    return fl_reco_shard_results(h, out, capacity, summary);
  }
  return fl_recognize_wait(h, out, capacity, summary);
}
