// fealess_b200/obj_reco.hpp - C++ mirror of the reference's product API for this path: CObjRecoCAD (CadReco/obj_reco_temp.h:6-30)
// and its LINE-MOD + ICP implementation CObjRecoLmICP (CadReco/obj_reco_lmicp.h:12-58, obj_reco_lmicp.cpp:47-259), with the POD
// types of CadReco/lotus_common.h that appear in those signatures.  Same entry points, argument meaning, defaults (75 %, <= 10 ICP
// iterations, 0.5 / 0.01 mm) and status codes; everything that computes runs on the GPU through the C ABI:
//
//   AddObj(path) ........ :67-74   readLinemod(path + "/linemod_templates.yml") (linemod_io.hpp); numClasses() == 0 ->
//                                   ERROR_OPEN_FILE_FAILED.  Unlike the reference, which decodes <path>/depth/<template_id>.png from disk
//                                   inside EVERY Recognition (:156-157), the depth images are decoded here, once, converted to mm
//                                   (convertTo(CV_16UC1, 0.1), :187) and - on the first Recognition - cropped to their template boxes
//                                   and kept on the device (fl_upload_model_depths).
//   Recognition(...) .... :86-204  PrepareInputData (:216-259: argument checks, target size 640 x H*640/W, zoomed intrinsics), the
//                                   INTER_LINEAR rescale + Detector::match as ONE device pass (Detector::matchRescaled ->
//                                   fl_match_rescaled), then detection() on matches[0] (:111-189) against the depth frame that is
//                                   already on the device (fl_detection_batch_resident), pose packed by Convert (:20-30).
//   Train / ClearObj / SetROI / Set-/GetAdvancedParam: return 0 without doing anything, exactly like the reference (:62-84, 206-214).
//   SetFramesInFlight / SubmitRecognition / CollectRecognition (not in the reference): the same Recognition as a stream - every frame
//                                   is ONE enqueue on the device (fl_pipe_submit_recognition: rescale, match, hypothesis selection, ICP,
//                                   suppression), up to k frames are in flight from one thread, results come back in submission order.
//   SetDevices (not in the reference): the detector's templates are sharded over several GPUs of this process (Detector::useDevices);
//                                   Recognition and the stream then run over a template-sharded group (fl_group_*_recognition), with the
//                                   single-GPU class's results.
//
// Kept from the reference on purpose: detection() receives the CALLER's intrinsics, not the zoomed ones (:188, SURVEY.md A.6 v);
// only matches[0] is refined (:111).  A rect that leaves the frame raises cv::Exception (the reference's cv::Mat ROI assert,
// ICP/detection.cpp:43-44).  A template without a readable depth image yields no result (the reference would fail inside detection()).
#ifndef FEALESS_B200_OBJ_RECO_HPP
#define FEALESS_B200_OBJ_RECO_HPP

#include <cmath>
#include <cstring>
#include <map>
#include <sstream>
#include <string>
#include <vector>

#include "linemod_io.hpp"
#ifdef FEALESS_B200_WITH_OPENCV
#include <opencv2/imgcodecs.hpp>
#else
#include "png16.hpp"
#endif

// ---- CadReco/lotus_common.h: status codes and the POD types of the call surface (skipped when the reference's header came first) ----
#ifndef __COMMON_H__
#define __COMMON_H__
#define SUCCESS 0
#define ERROR_INVALID_PARAM 0x80000001
#define ERROR_OPEN_FILE_FAILED 0x80000002
#define ERROR_VERSION_MISMATCH 0x80000003
#define ERROR_NEW_FAILED 0x80000004
#define ERROR_UNKNOW 0x80000005
using std::string;
using std::vector;
template <typename T> struct TImage { double dTimestamp; T* pData; int nWidth; int nHeight; };   // timestamp in ms; interleaved rows, no padding
typedef TImage<unsigned char> TImageU;
typedef TImage<unsigned short int> TImageU16;
typedef TImage<float> TImageF;
struct TCamIntrinsicParam { int nWidth; int nHeight; double dFx; double dFy; double dCx; double dCy; vector<double> vdDistCoeff; };
typedef float Mat4x4F[16];
struct TScanFrame { TImageU tGrayImg; TImageU tMask; Mat4x4F tWorld2Cam; TImageF tDepthImg; };
struct TScanPackage { string strObjTag; Mat4x4F tGLPrjMatrix; vector<float> bounding_box; vector<TScanFrame> vtScanFrame; };
struct TObjRecoResult { string strObjTag; Mat4x4F tWorld2Cam; };
struct AdvancedParam { bool bEnablePoseBinFrameMatching; bool bEnablePreprocessing; };
struct TTrainParam { int nType; int nMethod; bool bPreprocessing; float img_physical_width; };
#endif

#ifndef __OBJ_RECO_TEMP__
#define __OBJ_RECO_TEMP__
class CObjRecoCAD {
 public:
  enum EObjRecoType { EObjReco_FEATURE, EObjReco_LmICP, EObjReco_BB8, EObjReco_PoseNet };
  virtual ~CObjRecoCAD() {}
  static string GetVersion() { return string("fealess_b200 CAD-based 3D object recognition (LINE-MOD + ICP on sm_100a), library ") + fl_version(); }
  static inline CObjRecoCAD* Create(EObjRecoType eType = EObjReco_LmICP);   // nullptr for the types the reference leaves unimplemented
  static void Destroy(CObjRecoCAD* pHandle) { delete pHandle; }
  virtual int Train(const string& strDataBase, const TScanPackage& tScanPackage, const TTrainParam& tObjTrainParam) = 0;
  virtual int AddObj(const string pObjModel) = 0;
  virtual int ClearObj() = 0;
  virtual int SetROI(const TImageU& tROI) = 0;
  virtual int Recognition(const TImageU& tRGB, const TImageU16& tDepth, const TCamIntrinsicParam& tCamIntrinsic, vector<TObjRecoResult>& vtResult) = 0;
  virtual int SetAdvancedParam(const AdvancedParam& advancedParam) = 0;
  virtual int GetAdvancedParam(const string& strKey, void* pvValue) = 0;
};
#endif

class CObjRecoLmICP : public CObjRecoCAD {
 public:
  CObjRecoLmICP() : m_matching_threshold(75.0f), m_icp_it_thr(10), m_dist_mean_thr(0.5f), m_dist_diff_thr(0.01f), m_proc_w(0), m_proc_h(0), m_crops_w(0), m_crops_h(0) {}   // :47-56
  virtual ~CObjRecoLmICP() { close_stream(m_stream); close_stream(m_sync); }
  virtual int Train(const string&, const TScanPackage&, const TTrainParam&) { return 0; }
  virtual int ClearObj() { return 0; }
  virtual int SetROI(const TImageU&) { return 0; }
  virtual int SetAdvancedParam(const AdvancedParam&) { return 0; }
  virtual int GetAdvancedParam(const string&, void*) { return 0; }

  virtual int AddObj(const string str_feature_path) {
    m_str_lm_feature_path = str_feature_path;
    m_lm_detector = readLinemod(m_str_lm_feature_path + string("/linemod_templates.yml"));
    m_model_depth.clear(); m_crop_index.clear(); m_crops_w = m_crops_h = 0;
    close_stream(m_stream); close_stream(m_sync);
    if (!m_devices.empty()) m_lm_detector->useDevices(m_devices, m_xcap);   // SetDevices outlives the detector it was first applied to
    if (0 == m_lm_detector->numClasses()) return (int)ERROR_OPEN_FILE_FAILED;
    // the reference names the file by template_id alone (:156), so one image serves that id in every class
    int max_templates = 0;
    const vector<cv::String> ids = m_lm_detector->classIds();
    for (size_t c = 0; c < ids.size(); ++c) max_templates = std::max(max_templates, m_lm_detector->numTemplates(ids[c]));
    for (int tid = 0; tid < max_templates; ++tid) {
      std::ostringstream name;
      name << m_str_lm_feature_path << "/depth/" << tid << ".png";
      ModelDepth md;
      if (load_depth_mm(name.str(), md)) m_model_depth[tid].swap(md);
    }
    return 0;
  }

  virtual int Recognition(const TImageU& tRGB, const TImageU16& tDepth, const TCamIntrinsicParam& tCamIntrinsic, vector<TObjRecoResult>& vtResult) {
    vtResult.clear();
    if (!m_lm_detector || 0 != PrepareInputData(tRGB, tDepth, tCamIntrinsic)) return (int)ERROR_INVALID_PARAM;
    if (m_lm_detector->getModalities().size() != 2) return (int)ERROR_INVALID_PARAM;   // match() == -1: two sources are passed (:94-96, linemod.cpp:1364)
    if (multi_device()) return recognition_on_group(tRGB, tDepth, tCamIntrinsic, vtResult);
    std::vector<cup_linemod::Match> matches;
    if (0 != m_lm_detector->matchRescaled(tRGB.pData, (size_t)tRGB.nWidth * 3, tDepth.pData, (size_t)tDepth.nWidth * 2, tRGB.nWidth, tRGB.nHeight,
                                          m_proc_w, m_proc_h, m_matching_threshold, matches))
      return (int)ERROR_INVALID_PARAM;
    if (matches.empty()) return 0;
    // Hypothesis selection.  The reference refines matches[0] only (:111); its demo walks the sorted list and takes the best match of
    // every class (test/linemod_acq.cpp:165-184).  m_top_k / m_per_class generalise both: the first m_top_k matches, or the first
    // m_top_k matches of EVERY class, in list order.  The default (1, false) is the reference's behaviour.
    std::vector<size_t> chosen;
    if (!m_per_class) {
      for (size_t i = 0; i < matches.size() && (int)chosen.size() < m_top_k; ++i) chosen.push_back(i);
    } else {
      std::map<cv::String, int> taken;
      for (size_t i = 0; i < matches.size(); ++i)
        if (taken[matches[i].class_id]++ < m_top_k) chosen.push_back(i);
    }
    upload_crops();
    std::vector<int32_t> index; std::vector<fl_rect_t> rect_ref; std::vector<float> r_match, t_match; std::vector<size_t> which;
    for (size_t k = 0; k < chosen.size(); ++k) {
      const cup_linemod::Match& cur_match = matches[chosen[k]];
      const std::vector<cup_linemod::Template>& current_template = m_lm_detector->getTemplates(cur_match.class_id, cur_match.template_id);
      std::map<std::pair<cv::String, int>, int>::const_iterator crop = m_crop_index.find(std::make_pair(cur_match.class_id, cur_match.template_id));
      if (crop == m_crop_index.end()) continue;                                       // no depth image for this template
      const fl_rect_t rr = {current_template[0].offset_x + (cur_match.x - current_template[0].offset_x),   // :127-132
                            current_template[0].offset_y + (cur_match.y - current_template[0].offset_y), current_template[0].width, current_template[0].height};
      // :140-150: rows of (R | t), then d_match.  The reference's single-hypothesis path looks the pose up by template_id alone (:140);
      // the multi-hypothesis modes, which it does not have, key it by class as well
      const std::vector<float> pose = (m_top_k == 1 && !m_per_class) ? m_lm_detector->getPoseInfo(cur_match.template_id)
                                                                     : m_lm_detector->getPoseInfo(cur_match.class_id, cur_match.template_id);
      for (int i = 0; i < 3; ++i) { for (int j = 0; j < 3; ++j) r_match.push_back(pose[4 * i + j]); }
      for (int i = 0; i < 3; ++i) t_match.push_back(pose[4 * i + 3]);
      index.push_back(crop->second); rect_ref.push_back(rr); which.push_back(chosen[k]);
    }
    if (index.empty()) return 0;
    const fl_intrinsics_t K = {(float)tCamIntrinsic.dFx, (float)tCamIntrinsic.dFy, (float)tCamIntrinsic.dCx, (float)tCamIntrinsic.dCy};   // the caller's (:188)
    const fl_icp_params_t prm = {m_icp_it_thr, m_dist_mean_thr, m_dist_diff_thr};
    std::vector<fl_icp_result_t> res(index.size());
    fealess_b200::check_status(fl_detection_batch_resident(m_lm_detector->handle(), nullptr, 0, m_proc_w, m_proc_h, K, index.data(), rect_ref.data(), r_match.data(),
                                                           t_match.data(), (int32_t)index.size(), prm, res.data()), "detection");
    if (index.size() == 1) fealess_b200::check_status(res[0].status, "detection");   // the reference's single call throws on a box outside the frame (detection.cpp:43-44)
    // objects that came out of ICP, in hypothesis order; nonMaximumSuppression (ICP/NMS.cpp:6-39) over them when a distance is set
    std::vector<size_t> ok;
    for (size_t k = 0; k < res.size(); ++k) if (res[k].status == FL_OK) ok.push_back(k);
    std::vector<size_t> keep = ok;
    if (m_th_obj_dist > 0.f && ok.size() > 1) {
      std::vector<float> t3, dist; std::vector<int32_t> npts, out_idx(ok.size());
      for (size_t k = 0; k < ok.size(); ++k) { for (int i = 0; i < 3; ++i) t3.push_back(res[ok[k]].T[i]); npts.push_back(res[ok[k]].n_points); dist.push_back(res[ok[k]].dist_mean); }
      const int n_keep = fl_nms(m_lm_detector->handle(), t3.data(), npts.data(), dist.data(), (int32_t)ok.size(), m_th_obj_dist, out_idx.data());
      if (n_keep < 0) fealess_b200::check_status(n_keep, "nonMaximumSuppression");
      keep.clear();
      for (int k = 0; k < n_keep; ++k) keep.push_back(ok[(size_t)out_idx[k]]);
    }
    for (size_t k = 0; k < keep.size(); ++k) {
      const fl_icp_result_t& r = res[keep[k]];
      TObjRecoResult cur_result;
      cur_result.strObjTag = matches[which[keep[k]]].class_id;
      for (int i = 0; i < 3; ++i) { for (int j = 0; j < 3; ++j) cur_result.tWorld2Cam[4 * i + j] = r.R[3 * i + j]; cur_result.tWorld2Cam[4 * i + 3] = r.T[i]; }   // Convert :20-30
      cur_result.tWorld2Cam[12] = cur_result.tWorld2Cam[13] = cur_result.tWorld2Cam[14] = 0.f; cur_result.tWorld2Cam[15] = 1.f;
      vtResult.push_back(cur_result);
    }
    return 0;
  }

  // NOT in the reference (its Recognition refines matches[0] only): how many hypotheses go to ICP - the first top_k matches, or the
  // first top_k of every class (per_class; top_k = 1 is the "best match per class" walk of test/linemod_acq.cpp:165-184) - and the
  // distance (mm) under which nonMaximumSuppression merges refined objects (0 = no suppression).
  void SetHypotheses(int top_k, bool per_class = false, float th_obj_dist = 0.f) { m_top_k = top_k < 1 ? 1 : top_k; m_per_class = per_class; m_th_obj_dist = th_obj_dist; }

  // NOT in the reference: Recognition as a stream.  SubmitRecognition queues what Recognition computes for the frame (same checks and
  // statuses before matching; the images must stay unchanged until the frame has been collected); CollectRecognition returns the
  // results of the oldest queued frame, equal to Recognition's, and throws where Recognition throws.  Up to k frames
  // (<= FL_PIPE_MAX_DEPTH) are in flight; SetFramesInFlight, SetHypotheses and a new frame size take effect on an empty stream.
  void SetFramesInFlight(int k) {
    if (in_flight(m_stream)) throw std::runtime_error("SetFramesInFlight: frames are in flight");
    m_frames_in_flight = k < 1 ? 1 : k > FL_PIPE_MAX_DEPTH ? FL_PIPE_MAX_DEPTH : k;
    close_stream(m_stream);
  }
  int SubmitRecognition(const TImageU& tRGB, const TImageU16& tDepth, const TCamIntrinsicParam& tCamIntrinsic) {
    if (!m_lm_detector || 0 != PrepareInputData(tRGB, tDepth, tCamIntrinsic)) return (int)ERROR_INVALID_PARAM;
    if (m_lm_detector->getModalities().size() != 2) return (int)ERROR_INVALID_PARAM;   // as Recognition
    stream_setup(m_stream, m_frames_in_flight);
    const fl_intrinsics_t K = {(float)tCamIntrinsic.dFx, (float)tCamIntrinsic.dFy, (float)tCamIntrinsic.dCx, (float)tCamIntrinsic.dCy};   // the caller's (:188)
    const int rc = m_stream.group ? fl_group_submit_recognition(m_stream.group, tRGB.pData, (size_t)tRGB.nWidth * 3, tDepth.pData, (size_t)tDepth.nWidth * 2,
                                                                tRGB.nWidth, tRGB.nHeight, m_proc_w, m_proc_h, K)
                                  : fl_pipe_submit_recognition(m_stream.pipe, tRGB.pData, (size_t)tRGB.nWidth * 3, tDepth.pData, (size_t)tDepth.nWidth * 2,
                                                               tRGB.nWidth, tRGB.nHeight, m_proc_w, m_proc_h, K);
    if (rc == FL_ERR_SIZE) return (int)ERROR_INVALID_PARAM;
    fealess_b200::check_status(rc, "SubmitRecognition");
    return 0;
  }
  int CollectRecognition(vector<TObjRecoResult>& vtResult) {
    vtResult.clear();
    if (!m_stream.pipe && !m_stream.group) fealess_b200::check_status(FL_ERR_STATE, "CollectRecognition: no frame in flight");
    std::vector<fl_reco_result_t> res(FL_RECO_MAX_HYP);
    fl_reco_summary_t sum;
    fealess_b200::check_status(m_stream.group ? fl_group_collect_recognition(m_stream.group, res.data(), (int32_t)res.size(), &sum)
                                              : fl_pipe_collect_recognition(m_stream.pipe, res.data(), (int32_t)res.size(), &sum), "CollectRecognition");
    convert_results(m_stream, res, sum, vtResult);
    return 0;
  }

  // NOT in the reference: shard the detector's templates over these GPUs of this process (Detector::useDevices; exchange_capacity =
  // candidates one GPU may emit per frame).  Kept across AddObj, which replaces the detector.  With more than one device Recognition runs
  // its frame through a depth-1 template-sharded group of its own and SubmitRecognition / CollectRecognition run over a group with
  // SetFramesInFlight slots; results, exceptions and status codes are those of one GPU.  Masks are not supported there (SetROI is a stub).
  void SetDevices(const std::vector<int>& devices, int exchange_capacity = 2048) {
    if (in_flight(m_stream)) throw std::runtime_error("SetDevices: frames are in flight");
    close_stream(m_stream); close_stream(m_sync);
    m_devices = devices; m_xcap = exchange_capacity;
    m_crops_w = m_crops_h = 0;                                   // the crops of the per-call path live on the detector's (new) handle
    if (m_lm_detector) m_lm_detector->useDevices(m_devices, m_xcap);
  }

  // mirror-only accessors (tests, callers that want the zoomed intrinsics PrepareInputData stored)
  const TCamIntrinsicParam& processingIntrinsics() const { return m_tCamParam; }
  cv::Ptr<cup_linemod::Detector> detector() const { return m_lm_detector; }
  size_t numModelDepths() const { return m_model_depth.size(); }
  struct ModelDepth {
    int width, height; std::vector<uint16_t> mm;
    ModelDepth() : width(0), height(0) {}
    void swap(ModelDepth& o) { std::swap(width, o.width); std::swap(height, o.height); mm.swap(o.mm); }
  };
  const ModelDepth* modelDepth(int template_id) const { std::map<int, ModelDepth>::const_iterator i = m_model_depth.find(template_id); return i == m_model_depth.end() ? nullptr : &i->second; }

 private:
  template <typename T> static bool CheckTImage(const TImage<T>& t) { return t.dTimestamp >= 0 && t.nHeight > 0 && t.nWidth > 0 && t.pData; }   // :32-36

  // :216-259 without the rescale itself (that runs on the device inside matchRescaled)
  int PrepareInputData(const TImageU& tRGB, const TImageU16& tDepth, const TCamIntrinsicParam& tCamIntrinsic) {
    if (!CheckTImage(tRGB) || !CheckTImage(tDepth)) return (int)ERROR_INVALID_PARAM;
    if (tRGB.nHeight != tCamIntrinsic.nHeight || tRGB.nWidth != tCamIntrinsic.nWidth || tDepth.nHeight != tCamIntrinsic.nHeight || tDepth.nWidth != tCamIntrinsic.nWidth)
      return (int)ERROR_INVALID_PARAM;
    const float fZoomCoef = 640 * 1.0f / tRGB.nWidth;                                  // PROC_IMG_WIDTH
    m_proc_w = 640; m_proc_h = tRGB.nHeight * 640 / tRGB.nWidth;
    m_tCamParam = tCamIntrinsic;
    m_tCamParam.dFx *= fZoomCoef; m_tCamParam.dFy *= fZoomCoef; m_tCamParam.dCx *= fZoomCoef; m_tCamParam.dCy *= fZoomCoef;
    m_tCamParam.nWidth = m_proc_w; m_tCamParam.nHeight = m_proc_h;
    return 0;
  }

  // imread(path, -1) + convertTo(CV_16UC1, 0.1) (:156-157, 187): fp32 scale, round half to even, saturate
  static bool load_depth_mm(const std::string& path, ModelDepth& out) {
    std::vector<uint16_t> raw;
#ifdef FEALESS_B200_WITH_OPENCV
    cv::Mat img = cv::imread(path, -1);
    if (img.empty() || img.type() != CV_16UC1) return false;
    out.width = img.cols; out.height = img.rows; raw.resize((size_t)img.cols * img.rows);
    for (int y = 0; y < img.rows; ++y) std::memcpy(&raw[(size_t)y * img.cols], img.ptr<uint16_t>(y), (size_t)img.cols * 2);
#else
    if (!fealess_b200::read_png_gray16(path, raw, out.width, out.height)) return false;
#endif
    out.mm.resize(raw.size());
    for (size_t i = 0; i < raw.size(); ++i) {
      const long v = std::lrintf((float)raw[i] * 0.1f);
      out.mm[i] = (uint16_t)(v < 0 ? 0 : v > 65535 ? 65535 : v);
    }
    return true;
  }

  // crop every template's depth image to its level-0 box and keep the crops on the device; once per detector and frame size
  void upload_crops() {
    if (m_crops_w == m_proc_w && m_crops_h == m_proc_h) return;
    std::vector<const uint16_t*> ptr; std::vector<size_t> stride; std::vector<fl_rect_t> rect;
    crop_table(m_crop_index, ptr, stride, rect);
    fealess_b200::check_status(fl_upload_model_depths(m_lm_detector->handle(), (int32_t)ptr.size(), ptr.data(), stride.data(), rect.data(), m_proc_w, m_proc_h),
                               "fl_upload_model_depths");
    m_crops_w = m_proc_w; m_crops_h = m_proc_h;
  }
  // the templates whose depth image has the processing size and holds their level-0 box: (class, template_id) -> crop index, crops
  void crop_table(std::map<std::pair<cv::String, int>, int>& index, std::vector<const uint16_t*>& ptr, std::vector<size_t>& stride, std::vector<fl_rect_t>& rect) const {
    index.clear();
    const vector<cv::String> ids = m_lm_detector->classIds();
    for (size_t c = 0; c < ids.size(); ++c)
      for (int tid = 0; tid < m_lm_detector->numTemplates(ids[c]); ++tid) {
        const ModelDepth* md = modelDepth(tid);
        const cup_linemod::Template& t0 = m_lm_detector->getTemplates(ids[c], tid)[0];
        if (!md || md->width != m_proc_w || md->height != m_proc_h || t0.offset_x < 0 || t0.offset_y < 0 || t0.offset_x + t0.width > md->width ||
            t0.offset_y + t0.height > md->height)
          continue;
        index[std::make_pair(ids[c], tid)] = (int)ptr.size();
        ptr.push_back(md->mm.data()); stride.push_back((size_t)md->width * 2);
        const fl_rect_t r = {t0.offset_x, t0.offset_y, t0.width, t0.height};
        rect.push_back(r);
      }
  }

  // what a stream was built for, and the pipe (one GPU) or template-sharded group (SetDevices with more than one device) behind it
  struct Stream {
    fl_pipe* pipe = nullptr; fl_group* group = nullptr;
    int w = 0, h = 0, top_k = 0; bool per_class = false; float th = 0.f; size_t fingerprint = 0;
    std::vector<cv::String> classes;
    std::vector<int32_t> crop;
  };
  bool multi_device() const { return m_lm_detector && m_lm_detector->devices().size() > 1; }
  static int in_flight(const Stream& st) { return st.group ? fl_group_in_flight(st.group) : st.pipe ? fl_pipe_in_flight(st.pipe) : 0; }

  // the pipe (or group) behind SubmitRecognition / the multi-device Recognition for the current frame size and hypothesis settings: the
  // detector's templates and the crops on every slot, the crop index and Recognition's pose rule per template (getPoseInfo(template_id)
  // in the reference's mode top_k = 1 without per_class, the class-keyed lookup otherwise)
  void stream_setup(Stream& st, int depth) {
    // templates added to the detector since the pipe was built: the same count check Detector::match uses before it re-uploads
    const size_t fingerprint = (size_t)m_lm_detector->numTemplates() * 4099u + (size_t)m_lm_detector->numClasses();
    const bool same_size = (st.pipe || st.group) && st.w == m_proc_w && st.h == m_proc_h && st.fingerprint == fingerprint;
    if (same_size && st.top_k == m_top_k && st.per_class == m_per_class && st.th == m_th_obj_dist) return;
    if (in_flight(st)) throw std::runtime_error("SubmitRecognition: frame size, templates or hypotheses changed with frames in flight");
    if (!same_size) {
      close_stream(st);
      std::map<std::pair<cv::String, int>, int> index;
      std::vector<const uint16_t*> ptr; std::vector<size_t> stride; std::vector<fl_rect_t> rect;
      crop_table(index, ptr, stride, rect);
      if (multi_device()) {
        st.group = m_lm_detector->createGroupPipe(depth, m_proc_w, m_proc_h);
        fealess_b200::check_status(fl_group_upload_model_depths(st.group, (int32_t)ptr.size(), ptr.data(), stride.data(), rect.data(), m_proc_w, m_proc_h),
                                   "fl_group_upload_model_depths");
      } else {
        st.pipe = m_lm_detector->createPipe(depth, m_proc_w, m_proc_h);
        fealess_b200::check_status(fl_pipe_upload_model_depths(st.pipe, (int32_t)ptr.size(), ptr.data(), stride.data(), rect.data(), m_proc_w, m_proc_h),
                                   "fl_pipe_upload_model_depths");
      }
      st.classes = m_lm_detector->classIds();
      st.crop.clear();
      for (size_t c = 0; c < st.classes.size(); ++c)
        for (int tid = 0; tid < m_lm_detector->numTemplates(st.classes[c]); ++tid) {
          std::map<std::pair<cv::String, int>, int>::const_iterator it = index.find(std::make_pair(st.classes[c], tid));
          st.crop.push_back(it == index.end() ? -1 : it->second);
        }
      st.w = m_proc_w; st.h = m_proc_h; st.fingerprint = fingerprint;
    }
    std::vector<float> pose12;
    for (size_t c = 0; c < st.classes.size(); ++c)
      for (int tid = 0; tid < m_lm_detector->numTemplates(st.classes[c]); ++tid) {
        const std::vector<float> pose = (m_top_k == 1 && !m_per_class) ? m_lm_detector->getPoseInfo(tid) : m_lm_detector->getPoseInfo(st.classes[c], tid);
        pose12.insert(pose12.end(), pose.begin(), pose.begin() + 12);
      }
    fl_reco_params_t prm;
    fl_default_reco_params(&prm);
    prm.threshold = m_matching_threshold; prm.icp.icp_it_thr = m_icp_it_thr; prm.icp.dist_mean_thr = m_dist_mean_thr; prm.icp.dist_diff_thr = m_dist_diff_thr;
    prm.top_k = m_top_k; prm.per_class = m_per_class ? 1 : 0; prm.th_obj_dist = m_th_obj_dist;
    if (st.group) fealess_b200::check_status(fl_group_set_recognition(st.group, &prm, st.crop.data(), pose12.data()), "fl_group_set_recognition");
    else fealess_b200::check_status(fl_pipe_set_recognition(st.pipe, &prm, st.crop.data(), pose12.data()), "fl_pipe_set_recognition");
    st.top_k = m_top_k; st.per_class = m_per_class; st.th = m_th_obj_dist;
  }
  static void close_stream(Stream& st) {
    if (st.pipe) fl_pipe_destroy(st.pipe);
    if (st.group) fl_group_destroy(st.group);
    st.pipe = nullptr; st.group = nullptr; st.w = st.h = 0;
  }
  // device results -> TObjRecoResult; throws where Recognition's single detection() throws (detection.cpp:43-44)
  static void convert_results(const Stream& st, const std::vector<fl_reco_result_t>& res, const fl_reco_summary_t& sum, vector<TObjRecoResult>& vtResult) {
    if (sum.n_hypotheses == 1 && sum.n_roi == 1) fealess_b200::check_status(FL_ERR_ROI, "detection");
    for (int k = 0; k < sum.n_results; ++k) {
      TObjRecoResult cur_result;
      cur_result.strObjTag = st.classes[(size_t)res[k].class_idx];
      std::memcpy(cur_result.tWorld2Cam, res[k].world2cam, sizeof cur_result.tWorld2Cam);
      vtResult.push_back(cur_result);
    }
  }
  // Recognition over several GPUs: the frame through a depth-1 group of this object's own (rescale, sharded match, selection, ICP and
  // suppression on the device), rebuilt under the conditions that rebuild the stream
  int recognition_on_group(const TImageU& tRGB, const TImageU16& tDepth, const TCamIntrinsicParam& tCamIntrinsic, vector<TObjRecoResult>& vtResult) {
    stream_setup(m_sync, 1);
    const fl_intrinsics_t K = {(float)tCamIntrinsic.dFx, (float)tCamIntrinsic.dFy, (float)tCamIntrinsic.dCx, (float)tCamIntrinsic.dCy};   // the caller's (:188)
    std::vector<fl_reco_result_t> res(FL_RECO_MAX_HYP);
    fl_reco_summary_t sum;
    const int rc = fl_group_recognize(m_sync.group, tRGB.pData, (size_t)tRGB.nWidth * 3, tDepth.pData, (size_t)tDepth.nWidth * 2, tRGB.nWidth, tRGB.nHeight,
                                      m_proc_w, m_proc_h, K, res.data(), (int32_t)res.size(), &sum);
    if (rc == FL_ERR_SIZE) return (int)ERROR_INVALID_PARAM;     // matchRescaled's -1
    fealess_b200::check_status(rc, "Recognition");
    convert_results(m_sync, res, sum, vtResult);
    return 0;
  }

  string m_str_lm_feature_path;
  cv::Ptr<cup_linemod::Detector> m_lm_detector;
  TCamIntrinsicParam m_tCamParam;
  float m_matching_threshold; int m_icp_it_thr; float m_dist_mean_thr; float m_dist_diff_thr;
  int m_proc_w, m_proc_h;
  std::map<int, ModelDepth> m_model_depth;                       // template_id -> rendered depth in mm
  std::map<std::pair<cv::String, int>, int> m_crop_index;        // (class, template_id) -> crop on the device
  int m_crops_w, m_crops_h;
  int m_top_k = 1; bool m_per_class = false; float m_th_obj_dist = 0.f;   // SetHypotheses
  // SubmitRecognition / CollectRecognition (m_stream) and the multi-device Recognition (m_sync, one slot)
  int m_frames_in_flight = 1;
  Stream m_stream, m_sync;
  std::vector<int> m_devices; int m_xcap = 2048;                 // SetDevices
  CObjRecoLmICP(const CObjRecoLmICP&) = delete;
  CObjRecoLmICP& operator=(const CObjRecoLmICP&) = delete;
};

inline CObjRecoCAD* CObjRecoCAD::Create(EObjRecoType eType) { return eType == EObjReco_LmICP ? new CObjRecoLmICP() : nullptr; }   // obj_reco_temp.cpp:13-30

#endif  // FEALESS_B200_OBJ_RECO_HPP
