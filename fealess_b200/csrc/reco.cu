// Recognition on the device (CObjRecoLmICP::Recognition, CadReco/obj_reco_lmicp.cpp:86-204): the two small kernels that join the match
// list to the ICP launch and the ICP results to the caller, so that a frame needs no host round trip between its stages.
//   k_reco_select  after k_refine_sort: hypothesis selection of the mirrors (fealess_b200/reco.py, include/fealess_b200/obj_reco.hpp)
//   k_reco_finish  after k_icp_fused: the objects that came out of ICP, nonMaximumSuppression (ICP/NMS.cpp:6-39), Convert (:20-30),
//                  posted to mapped pinned host memory (on a template-sharded pipe also pushed to the other ranks' mailboxes)
//   k_reco_receive on a template-sharded pipe's ranks that do not own the frame: the owner's results, from the mailbox to mapped host memory
#include "fl_internal.cuh"

// One warp walks the sorted list 32 matches at a time.  A match is taken while its key (its class with per_class, else one key for
// the whole list) has fewer than top_k taken: lanes with the same key are ranked by __match_any_sync, so a step equals the sequential
// walk of select_hypotheses over its 32 matches.  The walk stops once every key is full.
__global__ void __launch_bounds__(32) k_reco_select(const fl_match_t* __restrict__ matches, const int* __restrict__ hdr, int out_cap, int check_big,
                                                   const int32_t* __restrict__ class_first, int n_classes, int n_templates,
                                                   const fl_reco_tmpl* __restrict__ tmpl, int top_k, int per_class, int max_hyp, int W, int H,
                                                   fl_icp_hyp* __restrict__ hyps, int* __restrict__ sel) {
  extern __shared__ int s_count[];                               // matches seen per key
  const int lane = threadIdx.x;
  const unsigned lt = (1u << lane) - 1u;
  const int n_keys = per_class ? n_classes : 1;
  for (int c = lane; c < n_keys; c += 32) s_count[c] = 0;
  __syncwarp();
  const bool deferred = check_big && hdr[2] != 0;                // the fused sort holds 1,024 records: this list is not sorted yet
  const int n = deferred ? 0 : min(hdr[0], out_cap);
  int n_hyp = 0, n_full = 0;
  for (int base = 0; base < n && n_full < n_keys; base += 32) {
    const int i = base + lane;
    fl_match_t m;
    m.x = m.y = 0; m.similarity = 0.f; m.class_idx = -1; m.template_id = -1;
    if (i < n) m = matches[i];
    const int key = per_class ? m.class_idx : 0;
    const bool live = i < n && key >= 0 && key < n_keys;
    const unsigned peers = __match_any_sync(0xffffffffu, live ? key : -1) & __ballot_sync(0xffffffffu, live);
    const int before = live ? s_count[key] : top_k;
    const bool taken = live && before + __popc(peers & lt) < top_k;
    __syncwarp();
    bool filled = false;
    if (live && (peers >> lane) == 1u) {                         // the last lane of its key's group updates the key's count
      const int after = before + __popc(peers);
      s_count[key] = after;
      filled = before < top_k && after >= top_k;
    }
    n_full += __popc(__ballot_sync(0xffffffffu, filled));
    const fl_reco_tmpl* tp = nullptr;
    if (taken && m.class_idx >= 0 && m.class_idx < n_classes) {
      const int t = class_first[m.class_idx] + m.template_id;   // matchClass numbering (linemod.cpp:1458)
      if (t >= 0 && t < n_templates && tmpl[t].crop) tp = tmpl + t;
    }
    const unsigned emit = __ballot_sync(0xffffffffu, tp != nullptr);   // a selected match without a crop is dropped, as the mirrors `continue`
    const int k = n_hyp + __popc(emit & lt);
    if (tp && k < max_hyp) {
      fl_icp_hyp hy;
      hy.model_depth = tp->crop;
      hy.rect_model = tp->rect;
      hy.rect_ref.x = m.x; hy.rect_ref.y = m.y; hy.rect_ref.width = tp->rect.width; hy.rect_ref.height = tp->rect.height;   // (:127-132)
      for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) hy.r_match[3 * r + c] = tp->pose[4 * r + c];
        hy.t_match[r] = tp->pose[4 * r + 3];
      }
      const fl_rect_t& b = hy.rect_ref;                          // rect_inside: the cv::Mat ROI throw of detection.cpp:43-44
      hy.status = (b.x >= 0 && b.y >= 0 && b.width >= 0 && b.height >= 0 && b.x + b.width <= W && b.y + b.height <= H) ? FL_OK : FL_ERR_ROI;
      hyps[k] = hy;
      sel[FL_RECO_SEL_HDR + k] = i;
    }
    n_hyp = min(n_hyp + __popc(emit), max_hyp);
    __syncwarp();                                                // this step's count updates before the next step reads them
  }
  for (int k = n_hyp + lane; k < max_hyp; k += 32) {             // padding: the ICP launch is sized for max_hyp and skips these
    fl_icp_hyp hy;
    memset(&hy, 0, sizeof hy);
    hy.status = FL_ERR_STATE;
    hyps[k] = hy;
  }
  if (lane == 0) { sel[0] = n; sel[1] = n_hyp; sel[2] = deferred ? 1 : 0; sel[3] = 0; }
}

#define RECO_REC_WORDS ((int)(sizeof(fl_reco_result_t) / 4))
static_assert(sizeof(fl_reco_result_t) % 4 == 0, "fl_reco_result_t is a sequence of 32-bit words");

// One thread per hypothesis (FL_RECO_MAX_HYP threads).  The summary and the records are staged in shared memory and leave as ONE
// run of coalesced word stores: single stores to mapped host memory cost ~0.7 us each when one thread issues them in sequence.
// With push.n > 0 (the owner of a template-sharded pipe's frame) the same words go to the mailbox of every listed rank, and the frame's
// epoch is published in each mailbox signal after a system-scope fence, as the candidate exchange publishes its blocks.
__global__ void __launch_bounds__(FL_RECO_MAX_HYP) k_reco_finish(const fl_match_t* __restrict__ matches, const int* __restrict__ sel,
                                                                const fl_icp_result_t* __restrict__ results, int max_hyp, float th,
                                                                int* __restrict__ host_block, const __grid_constant__ fl_reco_push push) {
  extern __shared__ int s_out[];                                 // [FL_RECO_SUMMARY_WORDS][records]
  __shared__ float s_t3[3 * FL_RECO_MAX_HYP], s_dist[FL_RECO_MAX_HYP];
  __shared__ int32_t s_npts[FL_RECO_MAX_HYP], s_ok[FL_RECO_MAX_HYP], s_keep[FL_RECO_MAX_HYP];
  __shared__ uint8_t s_done[FL_RECO_MAX_HYP];
  __shared__ int s_wok[FL_RECO_MAX_HYP / 32], s_wroi[FL_RECO_MAX_HYP / 32], s_n_keep;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_hyp = min(sel[1], max_hyp);
  // the hypotheses whose ICP ran, in hypothesis order (the mirrors skip the others: status != 0)
  const int st = tid < n_hyp ? results[tid].status : FL_ERR_STATE;
  const unsigned ok = __ballot_sync(0xffffffffu, st == FL_OK), roi = __ballot_sync(0xffffffffu, st == FL_ERR_ROI);
  if (lane == 0) { s_wok[warp] = __popc(ok); s_wroi[warp] = __popc(roi); }
  __syncthreads();
  int pos = __popc(ok & ((1u << lane) - 1u)), n_ok = 0, n_roi = 0;
  for (int w = 0; w < FL_RECO_MAX_HYP / 32; ++w) { if (w < warp) pos += s_wok[w]; n_ok += s_wok[w]; n_roi += s_wroi[w]; }
  if (st == FL_OK) {
    const fl_icp_result_t& r = results[tid];
    s_ok[pos] = tid; s_t3[3 * pos] = r.T[0]; s_t3[3 * pos + 1] = r.T[1]; s_t3[3 * pos + 2] = r.T[2];
    s_npts[pos] = r.n_points; s_dist[pos] = r.dist_mean;
    s_keep[pos] = pos;
  }
  __syncthreads();
  if (tid == 0) s_n_keep = (th > 0.f && n_ok > 1) ? fl_nms_greedy(s_t3, s_npts, s_dist, n_ok, th, s_keep, s_done) : n_ok;
  __syncthreads();
  const int n_keep = s_n_keep;
  if (tid < n_keep) {
    const int k = s_ok[s_keep[tid]];
    const fl_match_t m = matches[sel[FL_RECO_SEL_HDR + k]];
    const fl_icp_result_t r = results[k];
    fl_reco_result_t o;
    o.class_idx = m.class_idx; o.template_id = m.template_id; o.x = m.x; o.y = m.y; o.similarity = m.similarity; o.hypothesis = k;
    for (int i = 0; i < 3; ++i) {                                // Convert (:20-30)
      for (int j = 0; j < 3; ++j) o.world2cam[4 * i + j] = r.R[3 * i + j];
      o.world2cam[4 * i + 3] = r.T[i];
      o.world2cam[12 + i] = 0.f;
    }
    o.world2cam[15] = 1.f;
    o.icp = r;
    memcpy(s_out + FL_RECO_SUMMARY_WORDS + tid * RECO_REC_WORDS, &o, sizeof o);
  }
  if (tid < FL_RECO_SUMMARY_WORDS) {
    const int v[5] = {sel[0], n_hyp, n_roi, n_keep, sel[2] ? FL_RECO_DEFERRED : 0};
    s_out[tid] = tid < 5 ? v[tid] : 0;
  }
  __syncthreads();
  const int n_words = FL_RECO_SUMMARY_WORDS + n_keep * RECO_REC_WORDS;
  for (int i = tid; i < n_words; i += blockDim.x) host_block[i] = s_out[i];
  if (push.n > 0) {
    for (int p = 0; p < push.n; ++p) {
      int* mbox = reinterpret_cast<int*>(push.peer[p] + push.mailbox_off);
      for (int i = tid; i < n_words; i += blockDim.x) mbox[i] = s_out[i];
    }
    __threadfence_system();
    __syncthreads();
    if (tid < push.n) st_release_sys(reinterpret_cast<unsigned*>(push.peer[tid]) + FL_XCHG_RECO_SIGNAL, push.epoch);
  }
}

// One CTA on a rank that does not own the frame: thread 0 acquire-waits for the frame's epoch in this rank's mailbox signal (bounded as
// the candidate exchange's wait: ~2 s of SM cycles), then the mailbox leaves for the mapped host block as one run of coalesced word stores.
__global__ void __launch_bounds__(FL_RECO_MAX_HYP) k_reco_receive(const uint8_t* __restrict__ own, size_t mailbox_off, unsigned epoch, int owner,
                                                                 int* __restrict__ host_block) {
  __shared__ int s_arrived;
  const int tid = threadIdx.x;
  if (tid == 0) {
    const unsigned* sig = reinterpret_cast<const unsigned*>(own) + FL_XCHG_RECO_SIGNAL;
    const long long t0 = clock64();
    int arrived = 1;
    while ((int)(ld_acquire_sys(sig) - epoch) < 0) {
      if (clock64() - t0 > (1ll << 32)) { arrived = 0; break; }
      __nanosleep(64);
    }
    s_arrived = arrived;
  }
  __syncthreads();
  if (!s_arrived) {                                              // an empty summary that names the owner; the host reports FL_ERR_STATE
    if (tid < FL_RECO_SUMMARY_WORDS) host_block[tid] = tid == FL_RECO_MISSING_OWNER ? 1 + owner : 0;
    return;
  }
  const int* mbox = reinterpret_cast<const int*>(own + mailbox_off);
  const int n_keep = min(max(__ldcg(mbox + 3), 0), FL_RECO_MAX_HYP);   // L2 loads: the owner wrote these over the peer link
  for (int i = tid; i < FL_RECO_SUMMARY_WORDS + n_keep * RECO_REC_WORDS; i += blockDim.x) host_block[i] = __ldcg(mbox + i);
}

int fl_launch_reco_select(const fl_match_t* matches, const int* d_hdr, int out_cap, int check_big, const int32_t* class_first, int n_classes,
                          int n_templates, const fl_reco_tmpl* tmpl, int top_k, int per_class, int max_hyp, int W, int H,
                          fl_icp_hyp* hyps, int* sel, cudaStream_t s) {
  const size_t smem = (size_t)(per_class ? n_classes : 1) * sizeof(int);
  return fl_launch(k_reco_select, dim3(1), dim3(32), smem, s, matches, d_hdr, out_cap, check_big, class_first, n_classes, n_templates, tmpl, top_k,
                   per_class, max_hyp, W, H, hyps, sel) == cudaSuccess ? 1 : -1;
}

int fl_launch_reco_finish(const fl_match_t* matches, const int* sel, const fl_icp_result_t* results, int max_hyp, float th_obj_dist,
                          int* host_block, const fl_reco_push* push, cudaStream_t s) {
  const size_t smem = (size_t)(FL_RECO_SUMMARY_WORDS + max_hyp * RECO_REC_WORDS) * sizeof(int);
  fl_reco_push P;
  memset(&P, 0, sizeof P);
  if (push) P = *push;
  return fl_launch(k_reco_finish, dim3(1), dim3(FL_RECO_MAX_HYP), smem, s, matches, sel, results, max_hyp, th_obj_dist, host_block, P) == cudaSuccess ? 1 : -1;
}

int fl_launch_reco_receive(const uint8_t* own_buffer, size_t mailbox_off, unsigned epoch, int owner, int* host_block, cudaStream_t s) {
  return fl_launch(k_reco_receive, dim3(1), dim3(FL_RECO_MAX_HYP), 0, s, own_buffer, mailbox_off, epoch, owner, host_block) == cudaSuccess ? 1 : -1;
}

int fl_reco_preload() {
  cudaFuncAttributes a;
  FL_CUDA(cudaFuncGetAttributes(&a, k_reco_select));
  FL_CUDA(cudaFuncGetAttributes(&a, k_reco_finish));
  FL_CUDA(cudaFuncGetAttributes(&a, k_reco_receive));
  return FL_OK;
}
