/* fealess_b200 - C ABI of the B200-native LINE-MOD + ICP hot path (drop-in boundary for rlvc/FEALESS).
 *
 * Every entry point is plain C: raw pointers, sizes, POD structs, an int status; nothing throws across
 * it and no OpenCV / torch type appears.  It is what a maintainer of the reference binds instead of the
 * CPU bodies of (paths relative to /root/reference):
 *
 *   fl_create / fl_upload_templates ...... cup_linemod::Detector(modalities, T_pyramid) linemod/linemod.cpp:1348-1354,
 *                                          addSyntheticTemplate :1636-1642, readClass :1700-1762 (readLinemod
 *                                          linemod/linemod_if.cpp:36-47 fills the same structures)
 *   fl_match ............................. cup_linemod::Detector::match linemod/linemod.hpp:324-327, linemod.cpp:1356-1441
 *   fl_match_shard_device /
 *   fl_sort_unique_device ................ the two halves of match() (matchClass :1451-1577 | sort+unique :1437-1439)
 *                                          exposed separately so template shards on several GPUs can exchange
 *                                          candidate lists in between (SURVEY.md 8e)
 *   fl_depth_to_3d ....................... cup_d2pc::depthTo3d ICP/depth_to_3d.h:12-13, depth_to_3d.cpp:190-221
 *   fl_icp_cloud_to_cloud_ex ............. icpCloudToCloud_Ex ICP/ICP.h:165-172, ICP/ICP.cpp:617-809
 *   fl_detection / fl_detection_batch .... detection() ICP/detection.h:9-11, ICP/detection.cpp:11-254
 *   fl_nms ............................... nonMaximumSuppression ICP/NMS.h:14-16, ICP/NMS.cpp:6-39
 *   fl_group_* ........................... the same Detector::match, and Recognition with several frames in flight, over N GPUs
 *                                          of one process (templates sharded)
 *   fl_debug_get ......................... stage-level exports for bit-exact parity checks (no reference equivalent)
 *
 * The library is CUDA-only (sm_100a): there is no CPU fallback; every call fails with FL_ERR_CUDA if no
 * usable device is present.  One handle = one GPU + one stream; calls on a handle are serialised by the
 * caller, independent handles may be used concurrently.  All functions are synchronous unless their
 * name ends in _device (those enqueue on the handle's stream and return; fl_sync waits).
 */
#ifndef FEALESS_B200_H
#define FEALESS_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FL_MAX_LEVELS 8
#define FL_MAX_MODALITIES 4

/* status codes */
enum {
  FL_OK = 0,
  FL_ERR_SIZE = -1,        /* sources/masks count or size mismatch: Detector::match returns -1 (linemod.cpp:1364-1378) */
  FL_ERR_GEOMETRY = -2,    /* W % T, H % T or (W*H) % 16 violated: CV_Assert in linearize / computeResponseMaps (:1062-1063, :981) */
  FL_ERR_ROI = -3,         /* rect leaves the image: cv::Mat ROI throw in detection() (ICP/detection.cpp:43-44) */
  FL_ERR_FEATURES = -4,    /* more than 63 features in a template: CV_Assert (:1137, :1231) */
  FL_ERR_ARG = -5,         /* null / out-of-range argument */
  FL_ERR_CAPACITY = -6,    /* an internal or caller buffer was too small; *count still reports the needed size */
  FL_ERR_CUDA = -7,        /* CUDA runtime error or no device; fl_last_error() has the text */
  FL_ERR_STATE = -8,       /* call order violated (e.g. match before upload) */
  FL_ERR_TRAIN = -9        /* fl_add_template: a pyramid level has fewer candidate features than requested (addTemplate returns -1, linemod.cpp:1600-1602) */
};

enum { FL_MODALITY_COLOR_GRADIENT = 0, FL_MODALITY_DEPTH_NORMAL = 1 };

/* cup_linemod::Match (linemod.hpp:253-286) with class_id as an index into the uploaded class list */
typedef struct { int32_t x, y; float similarity; int32_t class_idx; int32_t template_id; } fl_match_t;

/* cup_linemod::Feature (linemod.hpp:32-43) */
typedef struct { int32_t x, y, label; } fl_feature_t;

/* cup_linemod::Template (linemod.hpp:47-58); features are [feature_begin, feature_begin+feature_count) of the feature array */
typedef struct { int32_t width, height, offset_x, offset_y, pyramid_level, feature_begin, feature_count; } fl_template_hdr_t;

typedef struct {
  int32_t n_levels;                         /* T_at_level.size() */
  int32_t T[FL_MAX_LEVELS];                 /* default {5, 8} (linemod.cpp:1820) */
  int32_t n_modalities;
  int32_t modality_kind[FL_MAX_MODALITIES]; /* default {COLOR_GRADIENT, DEPTH_NORMAL} (getDefaultLINEMOD :1829-1835) */
  float   weak_threshold;                   /* ColorGradient: 10 (:515-520) */
  int32_t distance_threshold;               /* DepthNormal: 2000 (:827-833) */
  int32_t difference_threshold;             /* DepthNormal: 50 */
  int32_t max_width, max_height;            /* largest frame the handle must accept (workspace is sized once) */
  int32_t max_candidates;                   /* capacity of the candidate / match buffers on the device */
  int32_t device;                           /* CUDA device ordinal */
} fl_params_t;

typedef struct { float fx, fy, cx, cy; } fl_intrinsics_t;      /* TCamIntrinsicParam (CadReco/lotus_common.h:41-50), the 4 used fields */
typedef struct { int32_t x, y, width, height; } fl_rect_t;     /* cv::Rect_<int> */
typedef struct { int32_t icp_it_thr; float dist_mean_thr, dist_diff_thr; } fl_icp_params_t;  /* 10, 0.5, 0.01 (CadReco/obj_reco_lmicp.cpp:52-55) */

typedef struct {
  float R[9];            /* R_final row-major (detection) or R (icpCloudToCloud_Ex) */
  float T[3];            /* T_final / T, millimetres */
  float dist_mean;       /* return value of icpCloudToCloud_Ex (-1 if fewer than 3 points) */
  float inlier_ratio;    /* px_inliers_ratio */
  int32_t iterations;
  int32_t n_points;      /* paired valid points that entered ICP */
  int32_t status;        /* FL_OK or FL_ERR_ROI for this hypothesis */
} fl_icp_result_t;

typedef struct fl_handle fl_handle;

/* ---- lifecycle ---------------------------------------------------------------------------------- */
void fl_default_params(fl_params_t* p);
/* on failure nothing is kept: *out is NULL and every resource allocated so far has been released */
int  fl_create(const fl_params_t* params, fl_handle** out);
int  fl_destroy(fl_handle* h);
const char* fl_last_error(void);
const char* fl_version(void);
int  fl_sync(fl_handle* h);
/* the CUDA stream (cudaStream_t) every _device call of this handle is enqueued on */
void* fl_stream(fl_handle* h);

/* ---- template database ---------------------------------------------------------------------------
 * headers: n_templates * n_levels * n_modalities entries, template-major then level*n_modalities + modality
 * (the TemplatePyramid order of linemod.hpp:370-375); class_of[t] = class index of template t, templates of one
 * class contiguous, template_id = rank inside its class (matchClass, linemod.cpp:1458); pose13 (nullable) =
 * 13 floats per template (TemplatePoseInfo, :1617-1634) kept host-side for fl_get_pose_info. */
int fl_upload_templates(fl_handle* h, int32_t n_templates, const fl_template_hdr_t* headers,
                        const fl_feature_t* features, int32_t n_features, const int32_t* class_of,
                        const float* pose13);
/* Optional: the per-class template_id each uploaded template reports in its matches.  Default = rank inside its class
 * in upload order.  A handle that holds only a shard of a class (template-sharded multi-GPU matching) sets the GLOBAL
 * ids here so that gathered candidate lists are shard-invariant. */
int fl_set_template_ids(fl_handle* h, const int32_t* template_ids);
int fl_num_templates(fl_handle* h);
int fl_get_pose_info(fl_handle* h, int32_t class_idx, int32_t template_id, float out13[13]);

/* ---- Detector::addTemplate (template training) ------------------------------------------------------
 * One view of an object -> one template pyramid (linemod.cpp:1579-1615 with ColorGradientPyramid / DepthNormalPyramid::extractTemplate
 * :461-513, :747-825, selectScatteredFeatures :134-163, cropTemplates :52-96).  The per-pixel work runs on the device: the front end's
 * quantised images, the gradient magnitude, the mask erosions, eight chessboard distance transforms, the candidate tests; the stable
 * sort and the greedy scattered selection are sequential and run on the host.  bgr / depth / mask: host images of the handle's
 * modalities (mask nullable; 8UC1, nonzero = object).  headers: n_levels * n_modalities entries (index level * n_modalities + modality),
 * feature_begin pointing into `features` (at most feature_capacity; 63 per entry by default).  The result is what the reference's
 * addTemplate stores (bit-exact; tests/test_gpu_train.py) and can be handed to fl_upload_templates as it is.
 * FL_ERR_TRAIN: too few candidates on some level (the reference returns -1 and adds nothing).  The view goes through the handle's front
 * end, so its size has to satisfy the matching geometry (W, H divisible by T at every level: FL_ERR_GEOMETRY otherwise). */
typedef struct {
  int32_t num_features[FL_MAX_MODALITIES];  /* per modality at level 0, halved per level; default 63 (:518, :830) */
  float   strong_threshold;                 /* ColorGradient: 55 (:519) */
  int32_t extract_threshold;                /* DepthNormal: 2, halved per level (:725, :831) */
} fl_train_params_t;
void fl_default_train_params(fl_train_params_t* p);
int fl_add_template(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                    const uint8_t* mask, size_t mask_stride, int32_t W, int32_t H, const fl_train_params_t* params_or_null,
                    fl_template_hdr_t* headers, fl_feature_t* features, int32_t feature_capacity, int32_t* n_features,
                    fl_rect_t* bounding_box);

/* ---- Detector::match -------------------------------------------------------------------------------
 * Host buffers in, host matches out (sorted by the canonical total order, duplicates pruned).
 * bgr: 8UC3 rows of bgr_stride bytes; depth: 16UC1 rows of depth_stride bytes (mm); either may be NULL if no
 * modality of that kind is configured.  masks: NULL or n_modalities pointers (each NULL or W*H dense u8, nonzero =
 * keep; a masked frame runs the same launches as an unmasked one, and the handle allocates nothing for it: the level-0 masks are
 * staged in buffers sized at fl_create, (max_width * max_height * 4 / 3) * n_modalities bytes).  class_filter: NULL/0 = all classes.  quantized_out: NULL or n_levels*n_modalities host pointers
 * (index level*n_modalities + modality) receiving the quantised images, each (W>>l)*(H>>l) bytes.
 * *count = number of matches found (may exceed capacity -> FL_ERR_CAPACITY, first `capacity` are written). */
int fl_match(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
             int32_t W, int32_t H, const uint8_t* const* masks, float threshold,
             const int32_t* class_filter, int32_t n_filter,
             fl_match_t* out, int32_t capacity, int32_t* count, uint8_t* const* quantized_out);

/* Same computation with the frame already resident in device memory (dense rows).  d_masks as above but device
 * pointers (valid until fl_match_wait; fl_debug_get(FL_DBG_QUANTIZED) of such a frame reads them again).  Results stay on the device; fl_match_fetch copies them out (and synchronises). */
int fl_match_device(fl_handle* h, const void* d_bgr, const void* d_depth, int32_t W, int32_t H,
                    const void* const* d_masks, float threshold, const int32_t* class_filter, int32_t n_filter);
int fl_match_fetch(fl_handle* h, fl_match_t* out, int32_t capacity, int32_t* count);
/* The two halves of fl_match_device: ..._async only enqueues the frame's kernels on the handle's stream (fl_stream) and
 * returns; fl_match_wait waits for them and finishes the call (status as fl_match_device).  A caller can overlap its own host
 * work with the device, or bracket exactly the device work with CUDA events recorded on fl_stream (what bench.py does).
 * One frame in flight per handle: fl_match_wait must be called before the next ..._async call. */
int fl_match_device_async(fl_handle* h, const void* d_bgr, const void* d_depth, int32_t W, int32_t H,
                          const void* const* d_masks, float threshold, const int32_t* class_filter, int32_t n_filter);
int fl_match_wait(fl_handle* h);
/* How the host waits for this handle's frames (fl_match_wait, fl_match_fetch, fl_detection_batch*, fl_nms): by default the CUDA
 * runtime spins (lowest latency, one busy core per waiting thread); enable = 1 makes the calling thread sleep until the GPU's
 * interrupt (cudaEventBlockingSync) - for hosts that keep more frames in flight, one thread each, than they have cores. */
int fl_set_blocking_wait(fl_handle* h, int enable);
/* enqueue-only half of fl_match (host buffers): the upload and the frame's kernels go on the handle's stream; finish with
 * fl_match_wait + fl_match_fetch.  Page-locked caller buffers are read by DMA and must stay valid until fl_match_wait returns;
 * pageable ones are copied before this returns. */
int fl_match_async(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int32_t W, int32_t H,
                   const uint8_t* const* masks, float threshold, const int32_t* class_filter, int32_t n_filter);

/* ---- several frames in flight on one GPU -----------------------------------------------------------
 * The reference's callers run Detector::match once per camera frame in a loop (CadReco/obj_reco_lmicp.cpp:86-204,
 * test/linemod_acq.cpp:120-190); the frames are independent.  A pipe owns `depth` handles on params->device (each holds the whole
 * template set) and deals submitted frames round-robin, so that the front end of frame i+1, the upload of frame i+2 and the result
 * copy of frame i-1 overlap the similarity kernel of frame i.  Lists come back in submission order and equal fl_match's.
 * fl_pipe_submit: FL_ERR_STATE when `depth` frames are in flight already.  on_device != 0: bgr / depth are device pointers with
 * dense rows (the strides must say so); otherwise host pointers as in fl_match_async (page-locked buffers must stay valid until the
 * frame has been collected).  fl_pipe_submit_masked: the same with masks (layout of fl_match: NULL or n_modalities pointers, each NULL
 * or a dense W*H u8 image, nonzero = keep), in device memory when on_device != 0, else host memory (copied before the call returns);
 * a masked frame takes the same launches as an unmasked one, on plain and on template-sharded pipes.  fl_pipe_submit = masks NULL.
 * fl_pipe_collect: waits for the OLDEST frame in flight and writes its list (status as fl_match_fetch).
 * fl_pipe_match_batch: n_frames frames of one geometry (arrays of n_frames pointers), frame f's list at out + f *
 * capacity_per_frame and its length in counts[f]; FL_ERR_CAPACITY if some list was truncated. */
typedef struct fl_pipe fl_pipe;
#define FL_PIPE_MAX_DEPTH 8
int fl_pipe_create(const fl_params_t* params, int32_t depth, fl_pipe** out);
int fl_pipe_destroy(fl_pipe* p);
int32_t fl_pipe_depth(const fl_pipe* p);
int32_t fl_pipe_in_flight(const fl_pipe* p);
fl_handle* fl_pipe_handle(fl_pipe* p, int32_t i);
int fl_pipe_upload_templates(fl_pipe* p, int32_t n_templates, const fl_template_hdr_t* headers, const fl_feature_t* features,
                             int32_t n_features, const int32_t* class_of, const float* pose13);   /* layout of fl_upload_templates */
/* Template-sharded pipe (rank `rank` of `world`): after the shard has been uploaded (fl_pipe_upload_templates + fl_set_template_ids on
 * every fl_pipe_handle), hand over the exchange buffers - peer_buffers[i * world + r] = rank r's buffer of slot i as mapped into this
 * process (fl_exchange_buffer_bytes(world, capacity) each, zeroed once), local_blocks[i] = slot i's candidate block (capacity + 1
 * records, device memory).  fl_pipe_submit / fl_pipe_match_batch then run the fused match + exchange per frame; every rank has to
 * submit the same sequence of frames.  With this a rank's per-frame host work is inside the library (no Python / caller loop). */
int fl_pipe_set_exchange(fl_pipe* p, int32_t rank, int32_t world, int32_t exchange_capacity, void* const* peer_buffers,
                         fl_match_t* const* local_blocks);
int fl_pipe_submit(fl_pipe* p, const void* bgr, size_t bgr_stride, const void* depth, size_t depth_stride, int32_t W, int32_t H,
                   float threshold, const int32_t* class_filter, int32_t n_filter, int32_t on_device);
int fl_pipe_submit_masked(fl_pipe* p, const void* bgr, size_t bgr_stride, const void* depth, size_t depth_stride, int32_t W, int32_t H,
                          const void* const* masks, float threshold, const int32_t* class_filter, int32_t n_filter, int32_t on_device);
int fl_pipe_collect(fl_pipe* p, fl_match_t* out, int32_t capacity, int32_t* count);
int fl_pipe_match_batch(fl_pipe* p, int32_t n_frames, const void* const* bgr, size_t bgr_stride, const void* const* depth, size_t depth_stride,
                        int32_t W, int32_t H, float threshold, const int32_t* class_filter, int32_t n_filter, int32_t on_device,
                        fl_match_t* out, int32_t capacity_per_frame, int32_t* counts);

/* Template-sharded matching (one handle per GPU holds a shard of the templates):
 * fl_match_shard_device runs the front end + matchClass over this handle's templates and writes the UNSORTED
 * candidates into d_candidates[capacity] and their number into d_count[1] (both device memory, caller owned,
 * e.g. torch tensors that are then all-gathered).  fl_sort_unique_device sorts + prunes n_in records of d_in
 * (device) into d_out / d_out_count (device; d_out may alias d_in).  n_in is read from d_n_in[0..n_lists) when
 * d_n_in is not NULL: d_in then holds n_lists lists of `list_capacity` records each (the all-gather layout). */
int fl_match_shard_device(fl_handle* h, const void* d_bgr, const void* d_depth, int32_t W, int32_t H,
                          const void* const* d_masks, float threshold, const int32_t* class_filter, int32_t n_filter,
                          fl_match_t* d_candidates, int32_t capacity, int32_t* d_count);
int fl_sort_unique_device(fl_handle* h, const fl_match_t* d_in, int32_t n_lists, int32_t list_capacity,
                          const int32_t* d_n_in, fl_match_t* d_out, int32_t out_capacity, int32_t* d_out_count);

/* The all-gather layout of template-sharded matching: n_blocks blocks of (capacity + 1) records each, block b =
 * [header record whose .x is the number of candidates of rank b | capacity candidate records] (what
 * fl_match_shard_device produces when d_count points at the header of the caller's block and d_candidates at the record
 * behind it).  Sorts + prunes the union into the handle's own result buffer and synchronises; read the matches with
 * fl_match_fetch.  No intermediate copies or count extraction are needed between the collective and this call. */
int fl_sort_unique_blocks_device(fl_handle* h, const fl_match_t* d_blocks, int32_t n_blocks, int32_t capacity);

/* The same merge with the exchange done by the library itself over peer memory (NVLink / NVSwitch), fused into the head
 * of the sort kernel - no collective-library call on the data path.  Every rank owns an exchange buffer of
 * fl_exchange_buffer_bytes(world, capacity) bytes (zero-initialised once) that is mapped into every process of the
 * job (CUDA IPC, fabric handles, torch symmetric memory ...); peer_buffers[p] is the address of rank p's buffer in THIS
 * process.  The kernel pushes this rank's block [count | records] into every peer's buffer, publishes `epoch` (> 0,
 * incremented by all ranks for every frame) in the peer's signal word, waits for the epoch of all peers (bounded: a
 * missing peer yields FL_ERR_STATE after ~2 s instead of a hang), and sorts + prunes the union.  world <= 8.
 * The buffer's layout is private.  Its size includes a result mailbox of about 40 KB at the end, which only the recognition frames of
 * a template-sharded pipe use (fl_pipe_set_recognition_sharded); match-only frames never touch it. */
size_t fl_exchange_buffer_bytes(int32_t world, int32_t capacity);
int fl_exchange_sort_unique_device(fl_handle* h, int32_t rank, int32_t world, void* const* peer_buffers, int32_t capacity,
                                   const fl_match_t* d_local_block, uint32_t epoch);
/* fl_match_shard_device + the exchange in one call (enqueue only; finish with fl_match_wait): the candidates go straight into the
 * caller's block d_local_block = [count | capacity records] (device memory), and ONE launch refines them, pushes the block to
 * every peer, waits for the peers and sorts the union. */
int fl_match_shard_exchange_device_async(fl_handle* h, const void* d_bgr, const void* d_depth, int32_t W, int32_t H, float threshold,
                                         const int32_t* class_filter, int32_t n_filter, int32_t rank, int32_t world,
                                         void* const* peer_buffers, int32_t capacity, fl_match_t* d_local_block, uint32_t epoch);
/* the same with masks in device memory (d_masks as in fl_match_device; the call above = d_masks NULL) */
int fl_match_shard_exchange_device_masked_async(fl_handle* h, const void* d_bgr, const void* d_depth, int32_t W, int32_t H,
                                                const void* const* d_masks, float threshold, const int32_t* class_filter, int32_t n_filter,
                                                int32_t rank, int32_t world, void* const* peer_buffers, int32_t capacity,
                                                fl_match_t* d_local_block, uint32_t epoch);
/* the same with the frame in HOST memory (buffers as in fl_match_async): upload + local match + exchange in one call, so that a
 * rank's per-frame host work is this call, fl_match_wait and fl_match_fetch */
int fl_match_shard_exchange_async(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int32_t W, int32_t H,
                                  float threshold, const int32_t* class_filter, int32_t n_filter, int32_t rank, int32_t world,
                                  void* const* peer_buffers, int32_t capacity, fl_match_t* d_local_block, uint32_t epoch);
/* the same with host masks (masks as in fl_match; the call above = masks NULL) */
int fl_match_shard_exchange_masked_async(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                                         int32_t W, int32_t H, const uint8_t* const* masks, float threshold, const int32_t* class_filter,
                                         int32_t n_filter, int32_t rank, int32_t world, void* const* peer_buffers, int32_t capacity,
                                         fl_match_t* d_local_block, uint32_t epoch);
/* enqueue-only half; finish with fl_match_wait */
int fl_exchange_sort_unique_device_async(fl_handle* h, int32_t rank, int32_t world, void* const* peer_buffers, int32_t capacity,
                                         const fl_match_t* d_local_block, uint32_t epoch);

/* ---- template-sharded matching over N handles of ONE process (no torch, no NCCL, no Python) ---------
 * For a C++ host such as CObjRecoLmICP (CadReco/obj_reco_lmicp.cpp:86-204) that wants Detector::match spread over several GPUs:
 * the group creates one handle per entry of `devices` (the same device may appear more than once), enables peer access between
 * the devices, allocates every handle's exchange buffer and candidate block, deals the templates gid % n with their global
 * per-class ids, and runs fl_match_shard_exchange_device_async on every handle per frame.  The merged list equals a single
 * handle's list.  exchange_capacity = candidate records one handle may emit per frame (more -> FL_ERR_CAPACITY). */
typedef struct fl_group fl_group;
int fl_group_create(const fl_params_t* params, const int32_t* devices, int32_t n, int32_t exchange_capacity, fl_group** out);
/* the same with `depth` slots (1 .. FL_PIPE_MAX_DEPTH; fl_group_create = depth 1): every (member, slot) pair has its own handle,
 * exchange buffer, candidate block and epoch sequence, so that up to `depth` recognition frames are in flight (fl_group_submit_recognition).
 * FL_ERR_ARG for depth or n out of range (n <= 8) and NULL pointers; on failure *out is NULL. */
int fl_group_create_pipe(const fl_params_t* params, const int32_t* devices, int32_t n, int32_t exchange_capacity, int32_t depth, fl_group** out);
int fl_group_destroy(fl_group* g);
int32_t fl_group_size(const fl_group* g);                     /* members (n) */
int32_t fl_group_depth(const fl_group* g);
int32_t fl_group_in_flight(const fl_group* g);                /* recognition frames submitted and not collected */
/* handle i = slot * n + member, i in [0, n * depth) (e.g. for fl_get_pose_info, fl_detection_batch*, fl_launch_count); fl_group_match
 * runs on slot 0 */
fl_handle* fl_group_handle(fl_group* g, int32_t i);
int fl_group_upload_templates(fl_group* g, int32_t n_templates, const fl_template_hdr_t* headers, const fl_feature_t* features,
                              int32_t n_features, const int32_t* class_of, const float* pose13);   /* layout of fl_upload_templates, every slot */
/* FL_ERR_STATE while recognition frames are in flight */
int fl_group_match(fl_group* g, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int32_t W, int32_t H,
                   float threshold, const int32_t* class_filter, int32_t n_filter, fl_match_t* out, int32_t capacity, int32_t* count);
/* the same with host masks (masks as in fl_match; fl_group_match = masks NULL); the merged list equals a single handle's fl_match */
int fl_group_match_masked(fl_group* g, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride, int32_t W, int32_t H,
                          const uint8_t* const* masks, float threshold, const int32_t* class_filter, int32_t n_filter, fl_match_t* out,
                          int32_t capacity, int32_t* count);

/* ---- input rescale (the caller's PrepareInputData) ------------------------------------------------- */
enum { FL_IMG_8UC3 = 0, FL_IMG_16UC1 = 1 };
/* cv::resize(src, dst, Size(W, H), 0, 0, INTER_LINEAR) on the device for the two image formats of
 * CObjRecoLmICP::PrepareInputData (CadReco/obj_reco_lmicp.cpp:38-45, 255-256: TImage2Mat(..., INTER_LINEAR)); host in,
 * host out (dst dense, W*H pixels).  OpenCV's own arithmetic (imgproc/src/resize.cpp; 8U fixed point, 16U float, 2x = area). */
int fl_resize_linear(fl_handle* h, const void* src, size_t src_stride, int32_t src_W, int32_t src_H, int32_t type,
                     void* dst, int32_t W, int32_t H);
/* PrepareInputData + Detector::match in one call: the src_W x src_H frame is uploaded, rescaled ON THE DEVICE to W x H
 * (W, H within fl_params_t.max_*) and matched; the rescaled depth frame stays on the device for
 * fl_detection_batch_resident(ref_depth = NULL).  Equal sizes: plain fl_match.  rescaled_depth_out (nullable): W*H u16, the
 * frame detection() would receive (m_depth).  No masks: the caller never sets one (SetROI is a stub, obj_reco_lmicp.cpp:81-84);
 * a masked frame goes through fl_resize_linear + fl_match. */
int fl_match_rescaled(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                      int32_t src_W, int32_t src_H, int32_t W, int32_t H, float threshold, const int32_t* class_filter, int32_t n_filter,
                      fl_match_t* out, int32_t capacity, int32_t* count, uint16_t* rescaled_depth_out);

/* ---- ICP ------------------------------------------------------------------------------------------ */
/* cup_d2pc::depthTo3d for 16UC1 input: out3 = H*W*3 floats in METRES, 0 depth -> NaN (depth_to_3d.cpp:99-137, 244-260) */
int fl_depth_to_3d(fl_handle* h, const uint16_t* depth, size_t depth_stride, int32_t W, int32_t H,
                   fl_intrinsics_t K, float* out3);
/* icpCloudToCloud_Ex on host clouds (n*3 floats each, mm).  Requires n_ref >= n_model (the reference's lock-step loops). */
int fl_icp_cloud_to_cloud_ex(fl_handle* h, const float* pts_ref, int32_t n_ref, const float* pts_model, int32_t n_model,
                             fl_icp_params_t p, fl_icp_result_t* out);
/* detection() for n hypotheses against one reference depth frame.  model_depth[i] points at pixel (0,0) of the i-th
 * rendered template depth image (u16 mm, rows of model_stride[i] bytes, same W x H as the frame); only rect_model[i] is read. */
int fl_detection_batch(fl_handle* h, const uint16_t* ref_depth, size_t ref_stride, int32_t W, int32_t H, fl_intrinsics_t K_ref,
                       const uint16_t* const* model_depth, const size_t* model_stride,
                       const fl_rect_t* rect_model, const fl_rect_t* rect_ref,
                       const float* r_match9, const float* t_match3, const float* d_match, int32_t n,
                       fl_icp_params_t p, fl_icp_result_t* out);
/* The rendered template depth images of the detector's templates, cropped to their template boxes and kept on the device.
 * The reference decodes <path>/depth/<template_id>.png from disk inside EVERY Recognition call and converts it to mm
 * (CadReco/obj_reco_lmicp.cpp:156-157, 187); a caller of this library decodes them once (AddObj) and hands them over here.
 * model_depth[i] points at pixel (0,0) of the i-th W x H image (u16 mm, rows of model_stride[i] bytes); only rect_model[i]
 * is read and stored.  Replaces any set uploaded before. */
int fl_upload_model_depths(fl_handle* h, int32_t n_models, const uint16_t* const* model_depth, const size_t* model_stride,
                           const fl_rect_t* rect_model, int32_t W, int32_t H);
/* fl_detection_batch over uploaded crops: hypothesis i uses crop model_index[i] and the rect_model it was uploaded with.
 * ref_depth == NULL takes the depth frame that the last fl_match call on this handle copied to the device (Recognition
 * passes the same image to match and to detection, obj_reco_lmicp.cpp:101, 188): only the hypothesis records (100 B each)
 * cross PCIe.  FL_ERR_STATE without uploaded crops / without such a frame of the same W x H. */
int fl_detection_batch_resident(fl_handle* h, const uint16_t* ref_depth, size_t ref_stride, int32_t W, int32_t H, fl_intrinsics_t K_ref,
                                const int32_t* model_index, const fl_rect_t* rect_ref, const float* r_match9, const float* t_match3,
                                int32_t n, fl_icp_params_t p, fl_icp_result_t* out);
/* the same with the reference depth frame already on the device (dense rows of W u16; e.g. the frame given to fl_match_device*):
 * nothing but the hypothesis records crosses PCIe (detection() of CadReco/obj_reco_lmicp.cpp:187-199 in a device-resident pipeline) */
int fl_detection_batch_resident_device(fl_handle* h, const void* d_ref_depth, int32_t W, int32_t H, fl_intrinsics_t K_ref,
                                       const int32_t* model_index, const fl_rect_t* rect_ref, const float* r_match9, const float* t_match3,
                                       int32_t n, fl_icp_params_t p, fl_icp_result_t* out);
/* single-hypothesis convenience with the reference's argument order (ICP/detection.h:9-11) */
int fl_detection(fl_handle* h, const uint16_t* model_depth, size_t model_stride, const uint16_t* ref_depth, size_t ref_stride,
                 int32_t W, int32_t H, fl_intrinsics_t K_ref, fl_rect_t rect_model, fl_rect_t rect_ref,
                 int32_t icp_it_thr, float dist_mean_thr, float dist_diff_thr,
                 const float r_match[9], const float t_match[3], float d_match, float T_final[3], float R_final[9]);
/* nonMaximumSuppression over n refined objects given in the caller's order: t3 (n*3), number of model points, icp_dist.
 * out_idx receives, per emitted PoseResult, the index of the object it was taken from; returns the count (>= 0) or < 0. */
int fl_nms(fl_handle* h, const float* t3, const int32_t* n_model_pts, const float* icp_dist, int32_t n,
           float th_obj_dist, int32_t* out_idx);
/* same, and absorbed[i] (n bytes, nullable) = 1 for every object the reference would have marked check_done (NMS.cpp:27) */
int fl_nms_ex(fl_handle* h, const float* t3, const int32_t* n_model_pts, const float* icp_dist, int32_t n,
              float th_obj_dist, int32_t* out_idx, uint8_t* absorbed);

/* ---- Recognition on the device (CObjRecoLmICP::Recognition, CadReco/obj_reco_lmicp.cpp:86-204) ----------------------------------
 * The whole frame as ONE enqueue: [INTER_LINEAR rescale] + front end + similarity + refinement / sort + hypothesis selection + ICP +
 * nonMaximumSuppression + pose packing, with the results posted to mapped pinned host memory, so that fl_recognize_wait is the
 * frame's only host wait (a frame whose unique list exceeds 1,024 records, or whose front end timed out, takes the recovery of
 * fl_match_wait and one more wait).  Selection, hypotheses and results are those of the mirrors (fealess_b200/reco.py,
 * include/fealess_b200/obj_reco.hpp): the first top_k matches, or the first top_k of every class (per_class), in list order;
 * model rect = the template's level-0 modality-0 box, reference rect = that box moved to the match position; a selected match
 * whose template has no depth crop is dropped (it still counts toward top_k); a reference rect outside the W x H frame gives
 * FL_ERR_ROI for that hypothesis and no result; nonMaximumSuppression over the refined objects when th_obj_dist > 0. */
#define FL_RECO_MAX_HYP 256
typedef struct {
  float threshold;            /* matching threshold, default 75 (:52-55) */
  fl_icp_params_t icp;        /* default {10, 0.5, 0.01} (:52-55) */
  int32_t top_k, per_class;   /* default 1, 0: ICP of matches[0] (:111) */
  float th_obj_dist;          /* mm; <= 0 (default): no suppression */
} fl_reco_params_t;
void fl_default_reco_params(fl_reco_params_t* p);
/* After fl_upload_templates and fl_upload_model_depths: crop_of_template[n_templates] = index of template t's crop in the uploaded
 * set (-1 = no crop; the crop's rect must be the template's level-0 modality-0 box), pose12 (nullable: the first 12 floats of the
 * uploaded pose13) = 12 floats per template, rows of (R | t).  Sizes the ICP workspace for top_k * (per_class ? n_classes : 1)
 * hypotheses now, so that no frame allocates.  FL_ERR_CAPACITY above FL_RECO_MAX_HYP; FL_ERR_STATE on a handle with
 * fl_set_template_ids, with a frame in flight, or without templates.  A later fl_upload_templates / fl_upload_model_depths /
 * fl_set_template_ids clears the setup. */
int fl_set_recognition(fl_handle* h, const fl_reco_params_t* p, const int32_t* crop_of_template, const float* pose12);
typedef struct {
  int32_t class_idx, template_id, x, y;   /* the match the object came from */
  float similarity;
  int32_t hypothesis;                     /* its index among the frame's hypotheses */
  float world2cam[16];                    /* [R | T; 0 0 0 1] row-major (Convert, :20-30) */
  fl_icp_result_t icp;
} fl_reco_result_t;
typedef struct { int32_t n_matches, n_hypotheses, n_roi, n_results; } fl_reco_summary_t;
/* enqueue-only half: the src_W x src_H frame is uploaded, rescaled on the device to W x H when the sizes differ (as
 * fl_match_rescaled), and recognised.  depth is required (ICP reads it), bgr as in fl_match.  K_ref = the CALLER's intrinsics,
 * which the mirrors pass to detection() (:188).  Page-locked caller buffers must stay valid until fl_recognize_wait; pageable
 * ones are copied before this returns.  One frame in flight per handle. */
int fl_recognize_async(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                       int32_t src_W, int32_t src_H, int32_t W, int32_t H, fl_intrinsics_t K_ref);
/* waits for the frame, writes min(n_results, capacity) results and the summary (nullable).  FL_ERR_CAPACITY: more results than
 * capacity, or more candidates than the handle's buffers hold (then no results, as fl_match_fetch). */
int fl_recognize_wait(fl_handle* h, fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary);
int fl_recognize(fl_handle* h, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                 int32_t src_W, int32_t src_H, int32_t W, int32_t H, fl_intrinsics_t K_ref,
                 fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary);
/* The same over a pipe: one host thread keeps up to `depth` frames in flight; results come back in submission order.  Setup on
 * every slot (FL_ERR_STATE while frames are in flight).  fl_pipe_set_recognition: FL_ERR_STATE on a template-sharded pipe
 * (fl_pipe_set_exchange with world > 1), which takes fl_pipe_set_recognition_sharded instead. */
int fl_pipe_upload_model_depths(fl_pipe* p, int32_t n_models, const uint16_t* const* model_depth, const size_t* model_stride,
                                const fl_rect_t* rect_model, int32_t W, int32_t H);
int fl_pipe_set_recognition(fl_pipe* p, const fl_reco_params_t* params, const int32_t* crop_of_template, const float* pose12);
/* Recognition on a template-sharded pipe (one process, or one pipe, per rank).  The rank holds only its shard, so the set-up takes the
 * tables of the WHOLE set: headers and class_of in the layout of fl_upload_templates over the whole set (only the level-0
 * modality-0 box of each template is read), crop_of_template as in fl_set_recognition (crops uploaded with
 * fl_pipe_upload_model_depths), pose12 (required) = 12 floats per template.  Every rank passes the same set.  FL_ERR_STATE on a pipe
 * that is not template-sharded or with frames in flight; otherwise the checks and statuses of fl_set_recognition.  Cleared by a later
 * template or crop upload or fl_pipe_set_exchange.
 * fl_pipe_submit_recognition then runs frame f on slot f % depth of every rank: each rank uploads [and rescales] the frame, matches
 * its shard and takes part in the exchange; only the frame's owner, rank f % world, runs selection, ICP and suppression, and pushes
 * the results over peer memory into every other rank's exchange buffer, where a one-CTA receive kernel waits for them (bounded: an
 * owner that never posts gives FL_ERR_STATE after ~2 s).  One enqueue per frame; fl_pipe_collect_recognition is its only host wait
 * and returns on EVERY rank the results of a single handle's fl_recognize over the whole set.  A list of more than 1,024 unique
 * matches is finished by every rank on its own copy.  Collecting frees the slot whatever the frame's status (a missing peer or
 * owner, an overflowing exchange block, FL_ERR_CAPACITY).  Match frames (fl_pipe_submit) and recognition frames may be mixed; all
 * ranks submit the same sequence.  The first frame of a new source geometry allocates its rescale tables before its exchange. */
int fl_pipe_set_recognition_sharded(fl_pipe* p, const fl_reco_params_t* params, int32_t n_templates, const fl_template_hdr_t* headers,
                                    const int32_t* class_of, const int32_t* crop_of_template, const float* pose12);
int fl_pipe_submit_recognition(fl_pipe* p, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                               int32_t src_W, int32_t src_H, int32_t W, int32_t H, fl_intrinsics_t K_ref);
int fl_pipe_collect_recognition(fl_pipe* p, fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary);
/* The same over a template-sharded group (fl_group_create_pipe): frame f goes to slot f % depth of every member; each member uploads
 * [and rescales] the frame, matches its shard and takes part in the peer-memory exchange, after which every member holds the merged
 * list; only the frame's owner, member f % n, runs the selection, ICP and suppression on it.  One host thread, results in submission
 * order, equal to a single handle's fl_recognize over the whole set.
 * fl_group_upload_model_depths: layout of fl_upload_model_depths; the crops go to every slot of every member (any member can own a
 * frame).  fl_group_set_recognition: crop_of_template and pose12 (nullable: the uploaded pose13) cover the whole set in the order of
 * fl_group_upload_templates; checks and statuses of fl_set_recognition; cleared by a later template or crop upload.  Memory: every
 * slot of every member holds all crops and a 72-byte selection record per template of the set.
 * Submit / collect / recognize: arguments and statuses of their fl_pipe_* / fl_recognize counterparts; FL_ERR_STATE with `depth`
 * frames in flight, before the set-up, or on collect with nothing in flight.  Collecting frees the slot whatever the frame's status:
 * a missing peer (FL_ERR_STATE) or an overflowing exchange block (FL_ERR_CAPACITY) is that frame's status only.  A front-end time-out
 * on a member re-runs the frame on every member of its slot from the frames already staged there. */
int fl_group_upload_model_depths(fl_group* g, int32_t n_models, const uint16_t* const* model_depth, const size_t* model_stride,
                                 const fl_rect_t* rect_model, int32_t W, int32_t H);
int fl_group_set_recognition(fl_group* g, const fl_reco_params_t* params, const int32_t* crop_of_template, const float* pose12);
int fl_group_submit_recognition(fl_group* g, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                                int32_t src_W, int32_t src_H, int32_t W, int32_t H, fl_intrinsics_t K_ref);
int fl_group_collect_recognition(fl_group* g, fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary);
int fl_group_recognize(fl_group* g, const uint8_t* bgr, size_t bgr_stride, const uint16_t* depth, size_t depth_stride,
                       int32_t src_W, int32_t src_H, int32_t W, int32_t H, fl_intrinsics_t K_ref,
                       fl_reco_result_t* out, int32_t capacity, fl_reco_summary_t* summary);

/* ---- stage-level debug exports (host copies of device intermediates of the LAST match call) -------- */
enum {
  FL_DBG_QUANTIZED = 0,     /* (level, modality)         -> (W>>l)*(H>>l) u8 */
  FL_DBG_SPREAD = 1,        /* (level, modality)         -> same size u8 (only kept when fl_debug_keep_spread(h,1)) */
  FL_DBG_LINEAR_MEMORY = 2, /* (level, modality, label)  -> T*T*(W/T)*(H/T) u8 */
  FL_DBG_SIMILARITY = 3,    /* (template index)          -> (W/T)*(H/T) u16 total similarity at the coarsest level */
  FL_DBG_LAST_COUNTS = 5,   /* ()                        -> 16 ints of the last sort+unique: {matches, live candidates after refinement,
                               multi-kernel-sort flag, raw candidates emitted by the global stage per list (up to 12)} */
  FL_DBG_STAGED_TRACE = 4,  /* ()                        -> 8 u64 per CTA of the staged similarity kernel {t_start, t_ready, t_first_data,
                               t_loop_end, t_end (globaltimer ns), smid, 0, 0}; only after fl_debug_option(h, FL_OPT_TRACE, 1);
                               returns the number of CTAs */
  FL_DBG_FE_TRACE = 6,      /* ()                        -> 6 u64 per front-end job {kind, CTAs, first CTA start, last CTA end (globaltimer ns),
                               sum over the job's CTAs of the CTA's span in SM clock cycles (clock64) and in globaltimer ns}: the job's SM
                               time, dependency waits included; only after fl_debug_option(h, FL_OPT_TRACE, 1); returns the number of jobs */
  FL_DBG_STAGED_ORDER = 7   /* ()                        -> the phase order of the last staged similarity launch: 32 u32 response sums of the
                               coarsest level it ordered by (word 8 m + l = modality m, label l), then one u8 per visit step: the phase
                               CTA 0 visited at that step; returns the number of phases */
};
/* developer options of one handle; every one is off by default and covered by a test */
enum {
  FL_OPT_FE_WAVES = 0,            /* front end as one launch per pyramid wave instead of ONE launch with in-grid dependencies */
  FL_OPT_SPLIT_REFINE = 1,        /* refinement and sort + unique as separate launches instead of one */
  FL_OPT_TRACE = 2,               /* record the in-kernel timelines (FL_DBG_STAGED_TRACE, front-end job timeline); slows the frame down */
  FL_OPT_FE_DEP_TIMEOUT_TEST = 3, /* the next frame's first in-grid dependency can never be satisfied: exercises the time-out fallback (takes ~1 s) */
  FL_OPT_FE_FORCED_WAVES = 4,     /* query (value ignored): 1 if a dependency time-out has switched this handle to per-wave launches */
  FL_OPT_SIM_NO_PRUNE = 5,        /* the staged similarity kernel accumulates every template in full instead of dropping one once no
                                     position can reach the threshold (same results; for A/B measurements and tests) */
  FL_OPT_SIM_ROTATE = 6           /* the staged similarity kernel visits the phases in the order rotated by CTA instead of by the frame's
                                     response mass (same results; for A/B measurements and tests) */
};
int fl_debug_option(fl_handle* h, int option, int value);
int fl_debug_keep_spread(fl_handle* h, int enable);
/* kernel selection of the global similarity stage: the shared-memory-staged kernel is used when the template set is
 * eligible (DESIGN.md); force_baseline(1) pins the L1/L2-fed kernel (parity tests run both); uses_staged reports the
 * choice made for the last frame geometry (1 / 0). */
int fl_debug_force_baseline(fl_handle* h, int enable);
int fl_debug_uses_staged(fl_handle* h);
/* the plan of the staged kernel for one coarsest level: W x H pixels (multiples of T), step T, n_modalities, n_templates,
 * max_positions = the largest template_positions of the set at that level, n_sm multiprocessors.  Host code, no device
 * needed.  Returns 1 and fills out[0..12] = {NW (accumulator words per lane), templates per warp, templates per CTA, CTAs,
 * threads per CTA, linear-memory rows per phase, row blocks per label, labels per phase, phases, ring buffers,
 * bytes per buffer, halo bytes, dynamic shared memory bytes} (out[13..15] = 0) when the staged kernel would run; 0 when
 * the planner refuses the geometry (a handle then runs the baseline kernel); FL_ERR_ARG for a bad argument.  A handle also
 * needs 256 or more eligible templates before it plans. */
int fl_debug_plan_staged(int W, int H, int T, int n_modalities, int n_templates, int max_positions, int n_sm, int32_t out[16]);
int fl_debug_get(fl_handle* h, int what, int32_t a, int32_t b, int32_t c, void* host_out, size_t bytes);
/* number of kernels launched by this handle since creation (bench.py reports the per-step delta) */
int64_t fl_launch_count(fl_handle* h);
/* per-stage device timing of the last fl_match*(): ms for front end, global similarity, refinement, sort (needs fl_profile(h,1)) */
int fl_profile(fl_handle* h, int enable);
int fl_last_stage_ms(fl_handle* h, float out4[4]);
/* device time (ms) of the ICP launch of the last fl_detection_batch / fl_detection (needs fl_profile(h,1)) */
int fl_last_icp_ms(fl_handle* h, float* ms);
/* developer timeline of that launch (needs fl_profile(h,1)): 20 words per hypothesis, SM clock cycles spent in
 * {0 pairing, 1 centroid sums, 2 shift + grid build, 3 distances, 4 distance sum (+ neighbour search), 5 correspondences,
 *  6 centroid + covariance sums, 7 SVD, 8 transform, 9 whole hypothesis}, then {10 iterations, 11 points}, then cycles the ordered
 *  sums waited for their stagers {12 record sums, 13 distance sums}, {14 distance sums without the overlapped search} and the cycles
 *  inside the additions proper {15 record sums, 16 distance sums} */
int fl_debug_icp_trace(fl_handle* h, uint64_t* out, int32_t n_hyp);

#ifdef __cplusplus
}
#endif
#endif /* FEALESS_B200_H */
