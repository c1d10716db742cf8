// fealess_b200/linemod.hpp - C++ host-side mirror of the reference's LINE-MOD interface for the matching path
// (reference: linemod/linemod.hpp:24-433, linemod/linemod_if.h:15-23).  Same namespace, type names, member names,
// argument meaning and error behaviour, so that CadReco/obj_reco_lmicp.cpp compiles against it unchanged; every call
// that computes goes through the C ABI of libfealess_b200.so (include/fealess_b200.h) - there is no CPU implementation
// behind these classes.  Header-only; link with -lfealess_b200.
//
//   cup_linemod::Feature / Template / Match ........ linemod.hpp:32-58, 253-286 (same fields, same operator< / ==)
//   cup_linemod::Modality / ColorGradient / DepthNormal: parameter carriers only (linemod.hpp:127-243, defaults
//                                                     linemod.cpp:515-520, 827-833); quantisation runs on the GPU
//   cup_linemod::Detector ........................... linemod.hpp:292-412: match (:324-327), addSyntheticTemplate,
//                                                     addPoseInfo / getPoseInfo, getTemplates, getT, pyramidLevels,
//                                                     numTemplates, numClasses, classIds, getModalities
//   getDefaultLINE / getDefaultLINEMOD .............. linemod.cpp:1822-1835
//   readLinemod / writeLinemod ...................... linemod_if.cpp:36-66: in linemod_io.hpp (own FileStorage-YAML reader / writer)
// addTemplate (training, SURVEY.md 8f rank 4) goes through fl_add_template.  Not provided (out of scope, SURVEY.md section 2): colormap / drawResponse.
#ifndef FEALESS_B200_LINEMOD_HPP
#define FEALESS_B200_LINEMOD_HPP

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "../fealess_b200.h"
#include "cv_min.hpp"

namespace fealess_b200 {
// CUDA device the mirrors create their handles on (default 0); set before the first call.
inline int& device_ordinal() { static int d = 0; return d; }
inline void check_status(int rc, const char* where) {
  if (rc == FL_OK) return;
  std::string msg = std::string(where) + ": " + fl_last_error();
  // the reference's CV_Assert cases (linemod.cpp:981, 1062-1063, 1137, 1231; cv::Mat ROI in detection.cpp:43-44)
  if (rc == FL_ERR_GEOMETRY || rc == FL_ERR_FEATURES || rc == FL_ERR_ROI) throw cv::Exception(msg + " (assertion failed, status " + std::to_string(rc) + ")");
  throw std::runtime_error(msg + " (status " + std::to_string(rc) + ")");   // FL_ERR_CUDA etc.: no CPU fallback exists
}
}  // namespace fealess_b200

namespace cup_linemod {

using cv::Mat;
using cv::Ptr;
using cv::String;

struct Feature {
  int x, y, label;
  Feature() : x(0), y(0), label(0) {}
  Feature(int x_, int y_, int label_) : x(x_), y(y_), label(label_) {}
};

struct Template {
  int width, height, offset_x, offset_y, pyramid_level;
  std::vector<Feature> features;
  Template() : width(0), height(0), offset_x(0), offset_y(0), pyramid_level(0) {}
};

// Parameter carrier: the modality's quantiser itself is a CUDA kernel selected by kind().
class Modality {
 public:
  virtual ~Modality() {}
  virtual String name() const = 0;
  virtual int kind() const = 0;   // FL_MODALITY_*
};

class ColorGradient : public Modality {
 public:
  ColorGradient() : weak_threshold(10.0f), num_features(63), strong_threshold(55.0f) {}   // linemod.cpp:515-520
  ColorGradient(float weak, size_t nf, float strong) : weak_threshold(weak), num_features(nf), strong_threshold(strong) {}
  String name() const { return "ColorGradient"; }
  int kind() const { return FL_MODALITY_COLOR_GRADIENT; }
  float weak_threshold; size_t num_features; float strong_threshold;
};

class DepthNormal : public Modality {
 public:
  DepthNormal() : distance_threshold(2000), difference_threshold(50), num_features(63), extract_threshold(2) {}   // :827-833
  DepthNormal(int dist, int diff, size_t nf, int extract) : distance_threshold(dist), difference_threshold(diff), num_features(nf), extract_threshold(extract) {}
  String name() const { return "DepthNormal"; }
  int kind() const { return FL_MODALITY_DEPTH_NORMAL; }
  int distance_threshold, difference_threshold; size_t num_features; int extract_threshold;
};

struct Match {
  Match() : x(0), y(0), similarity(0), template_id(0) {}
  Match(int x_, int y_, float s, const String& c, int t) : x(x_), y(y_), similarity(s), class_id(c), template_id(t) {}
  bool operator<(const Match& rhs) const {   // high similarity first, then template_id (linemod.hpp:262-269)
    if (similarity != rhs.similarity) return similarity > rhs.similarity;
    return template_id < rhs.template_id;
  }
  bool operator==(const Match& rhs) const { return x == rhs.x && y == rhs.y && similarity == rhs.similarity && class_id == rhs.class_id; }
  int x, y;
  float similarity;
  String class_id;
  int template_id;
};

class Detector {
 public:
  Detector() : pyramid_levels(0), handle_(nullptr), group_(nullptr), xcap_(2048), dirty_(true), cap_w_(0), cap_h_(0) {}
  Detector(const std::vector<Ptr<Modality> >& modalities_, const std::vector<int>& T_pyramid)
      : modalities(modalities_), pyramid_levels((int)T_pyramid.size()), T_at_level(T_pyramid), handle_(nullptr), group_(nullptr), xcap_(2048), dirty_(true), cap_w_(0), cap_h_(0) {}
  ~Detector() { release_device(); }

  // NOT in the reference: spread match() over several GPUs of this process.  The templates are dealt round-robin over one handle per
  // entry of `devices` (fl_group_*: peer-memory candidate exchange inside the sort kernel, no NCCL / Python involved); match() returns
  // the same list as on one GPU, masks and quantized_images included.  exchange_capacity = candidates one GPU may emit per frame.
  void useDevices(const std::vector<int>& devices, int exchange_capacity = 2048) {
    release_device();
    devices_ = devices; xcap_ = exchange_capacity; dirty_ = true; cap_w_ = cap_h_ = 0;
  }
  Detector(const Detector&) = delete;
  Detector& operator=(const Detector&) = delete;

  // Detector::match (linemod.hpp:324-327, linemod.cpp:1356-1441).  Returns 0, or -1 when sources / masks do not match the
  // modalities (:1364-1378).  Matches come back in the canonical total order (similarity desc, template_id asc, class,
  // y, x) with duplicates pruned - a deterministic refinement of the reference's unstable sort + unique (SURVEY.md A.5).
  int match(const std::vector<Mat>& sources, float threshold, std::vector<Match>& matches,
            const std::vector<String>& class_ids = std::vector<String>(), cv::OutputArrayOfArrays quantized_images = cv::noArray(),
            const std::vector<Mat>& masks = std::vector<Mat>()) const {
    matches.clear();
    if (sources.size() != modalities.size()) return -1;
    if (!masks.empty() && masks.size() != modalities.size()) return -1;
    const int M = (int)modalities.size();
    const uint8_t* bgr = nullptr; size_t bgr_step = 0; const uint16_t* depth = nullptr; size_t depth_step = 0;
    int W = 0, H = 0;
    for (int m = 0; m < M; ++m) {
      const Mat& s = sources[m];
      if (s.empty()) return -1;
      if (W && (s.cols != W || s.rows != H)) return -1;
      W = s.cols; H = s.rows;
      if (modalities[m]->kind() == FL_MODALITY_COLOR_GRADIENT) {
        if (s.type() != CV_8UC3) throw cv::Exception("ColorGradient source must be CV_8UC3");   // CV_Assert, linemod.cpp:394
        bgr = s.ptr<uint8_t>(0); bgr_step = s.step;
      } else {
        if (s.type() != CV_16UC1) throw cv::Exception("DepthNormal source must be CV_16UC1");   // CV_Assert, :694
        depth = s.ptr<uint16_t>(0); depth_step = s.step;
      }
    }
    // masks: dense W*H copies (the ABI takes dense rows); empty Mat = no mask for that modality
    std::vector<std::vector<uint8_t> > mask_store(M);
    std::vector<const uint8_t*> mask_ptr(M, nullptr);
    bool any_mask = false;
    for (int m = 0; m < M && !masks.empty(); ++m) {
      const Mat& k = masks[m];
      if (k.empty()) continue;
      if (k.type() != CV_8UC1 || k.cols != W || k.rows != H) return -1;     // :1374-1377 size check
      mask_store[m].resize((size_t)W * H);
      for (int y = 0; y < H; ++y) std::memcpy(&mask_store[m][(size_t)y * W], k.ptr<uint8_t>(y), (size_t)W);
      mask_ptr[m] = mask_store[m].data(); any_mask = true;
    }
    ensure_uploaded(W, H);
    // class filter: ids the detector does not know are ignored (:1425-1433)
    std::vector<int32_t> filter;
    if (!class_ids.empty()) {
      for (size_t i = 0; i < class_ids.size(); ++i) {
        std::map<String, int>::const_iterator it = class_index_.find(class_ids[i]);
        if (it != class_index_.end()) filter.push_back(it->second);
      }
      if (filter.empty()) { fill_quantized_only(bgr, bgr_step, depth, depth_step, W, H, any_mask ? mask_ptr.data() : nullptr, quantized_images); return 0; }
    }
    const int L = pyramid_levels;
    std::vector<Mat> qimgs;
    std::vector<uint8_t*> qptr;
    if (quantized_images.needed()) {
      qimgs.resize((size_t)L * M);
      for (int l = 0; l < L; ++l) for (int m = 0; m < M; ++m) { qimgs[l * M + m].create(H >> l, W >> l, CV_8UC1); qptr.push_back(qimgs[l * M + m].ptr<uint8_t>(0)); }
    }
    std::vector<fl_match_t> out(4096);
    int32_t count = 0;
    int rc;
    if (group_) {                                                            // template-sharded over the GPUs of useDevices()
      rc = fl_group_match_masked(group_, bgr, bgr_step, depth, depth_step, W, H, any_mask ? mask_ptr.data() : nullptr, threshold,
                                 filter.empty() ? nullptr : filter.data(), (int32_t)filter.size(), out.data(), (int32_t)out.size(), &count);
      if (quantized_images.needed() && (rc == FL_OK || rc == FL_ERR_CAPACITY)) {   // the front end alone, on the first GPU
        const int32_t none = -1; fl_match_t dummy; int32_t c2 = 0;
        fealess_b200::check_status(fl_match(handle_, bgr, bgr_step, depth, depth_step, W, H, any_mask ? mask_ptr.data() : nullptr, 100.0f, &none, 1, &dummy, 1,
                                            &c2, qptr.data()), "Detector::match");
      }
    } else
    rc = fl_match(handle_, bgr, bgr_step, depth, depth_step, W, H, any_mask ? mask_ptr.data() : nullptr, threshold,
                  filter.empty() ? nullptr : filter.data(), (int32_t)filter.size(), out.data(), (int32_t)out.size(), &count,
                  qptr.empty() ? nullptr : qptr.data());
    if (rc == FL_ERR_CAPACITY && count > (int32_t)out.size()) {             // more matches than the first buffer: fetch them all
      out.resize((size_t)count);
      rc = fl_match_fetch(handle_, out.data(), (int32_t)out.size(), &count);
    }
    if (rc == FL_ERR_SIZE) return -1;
    fealess_b200::check_status(rc, "Detector::match");
    matches.reserve((size_t)count);
    for (int i = 0; i < count; ++i) matches.push_back(Match(out[i].x, out[i].y, out[i].similarity, class_names_[out[i].class_idx], out[i].template_id));
    if (quantized_images.needed()) store_quantized(quantized_images, qimgs);
    return 0;
  }

  // Mirror-only: PrepareInputData's INTER_LINEAR rescale (CadReco/obj_reco_lmicp.cpp:38-45, 255-256) + match() in one device pass
  // (fl_match_rescaled): the src_W x src_H frame is uploaded as it is, rescaled to W x H on the GPU and matched; the rescaled depth
  // frame stays on the device for fl_detection_batch_resident.  Same return values as match(); colour + depth modalities only.
  int matchRescaled(const uint8_t* bgr, size_t bgr_step, const uint16_t* depth, size_t depth_step, int src_W, int src_H, int W, int H,
                    float threshold, std::vector<Match>& matches) const {
    matches.clear();
    bool has_color = false, has_depth = false;
    for (size_t m = 0; m < modalities.size(); ++m) (modalities[m]->kind() == FL_MODALITY_COLOR_GRADIENT ? has_color : has_depth) = true;
    if ((has_color && !bgr) || (has_depth && !depth)) return -1;
    if (devices_.size() > 1) throw cv::Exception("Detector::match_rescaled is not available together with useDevices()");
    ensure_uploaded(W, H);
    std::vector<fl_match_t> out(4096);
    int32_t count = 0;
    int rc = fl_match_rescaled(handle_, has_color ? bgr : nullptr, bgr_step, has_depth ? depth : nullptr, depth_step, src_W, src_H, W, H, threshold,
                               nullptr, 0, out.data(), (int32_t)out.size(), &count, nullptr);
    if (rc == FL_ERR_CAPACITY && count > (int32_t)out.size()) { out.resize((size_t)count); rc = fl_match_fetch(handle_, out.data(), (int32_t)out.size(), &count); }
    if (rc == FL_ERR_SIZE) return -1;
    fealess_b200::check_status(rc, "Detector::matchRescaled");
    matches.reserve((size_t)count);
    for (int i = 0; i < count; ++i) matches.push_back(Match(out[i].x, out[i].y, out[i].similarity, class_names_[out[i].class_idx], out[i].template_id));
    return 0;
  }

  // Detector::addTemplate (linemod.hpp:338-339, linemod.cpp:1579-1615): extract one template pyramid from a view of the object and
  // append it to class_id.  Returns the template id, or -1 when some pyramid level has too few candidate features (nothing is added).
  // The per-pixel work runs on the device (fl_add_template); the result is the reference's, feature for feature.
  int addTemplate(const std::vector<Mat>& sources, const String& class_id, const Mat& object_mask, const float* const pose_info,
                  cv::Rect* bounding_box = nullptr) {
    if (sources.size() != modalities.size()) return -1;
    const int M = (int)modalities.size(), L = pyramid_levels;
    const uint8_t* bgr = nullptr; size_t bgr_step = 0; const uint16_t* depth = nullptr; size_t depth_step = 0;
    int W = 0, H = 0;
    fl_train_params_t tp;
    fl_default_train_params(&tp);
    for (int m = 0; m < M; ++m) {
      const Mat& s = sources[m];
      if (s.empty() || (W && (s.cols != W || s.rows != H))) return -1;
      W = s.cols; H = s.rows;
      if (const ColorGradient* cg = dynamic_cast<const ColorGradient*>(modalities[m].get())) {
        if (s.type() != CV_8UC3) throw cv::Exception("ColorGradient source must be CV_8UC3");
        bgr = s.ptr<uint8_t>(0); bgr_step = s.step; tp.num_features[m] = (int32_t)cg->num_features; tp.strong_threshold = cg->strong_threshold;
      } else if (const DepthNormal* dn = dynamic_cast<const DepthNormal*>(modalities[m].get())) {
        if (s.type() != CV_16UC1) throw cv::Exception("DepthNormal source must be CV_16UC1");
        depth = s.ptr<uint16_t>(0); depth_step = s.step; tp.num_features[m] = (int32_t)dn->num_features; tp.extract_threshold = dn->extract_threshold;
      }
    }
    if (!object_mask.empty() && (object_mask.type() != CV_8UC1 || object_mask.cols != W || object_mask.rows != H)) throw cv::Exception("addTemplate: mask must be CV_8UC1 of the sources' size");
    ensure_uploaded(W, H);
    std::vector<fl_template_hdr_t> hdr((size_t)L * M);
    std::vector<fl_feature_t> feat((size_t)L * M * 64 + 64);
    int32_t nf = 0;
    fl_rect_t bb = {0, 0, 0, 0};
    const int rc = fl_add_template(handle_, bgr, bgr_step, depth, depth_step, object_mask.empty() ? nullptr : object_mask.ptr<uint8_t>(0),
                                   object_mask.empty() ? 0 : object_mask.step, W, H, &tp, hdr.data(), feat.data(), (int32_t)feat.size(), &nf, &bb);
    if (rc == FL_ERR_TRAIN) return -1;
    fealess_b200::check_status(rc, "Detector::addTemplate");
    std::vector<Template> pyr((size_t)L * M);
    for (size_t e = 0; e < pyr.size(); ++e) {
      pyr[e].width = hdr[e].width; pyr[e].height = hdr[e].height; pyr[e].offset_x = hdr[e].offset_x; pyr[e].offset_y = hdr[e].offset_y; pyr[e].pyramid_level = hdr[e].pyramid_level;
      for (int k = 0; k < hdr[e].feature_count; ++k) { const fl_feature_t& f = feat[(size_t)hdr[e].feature_begin + k]; pyr[e].features.push_back(Feature(f.x, f.y, f.label)); }
    }
    if (pose_info) addPoseInfo(pose_info);                       // (:1586; the reference appends the pose BEFORE it knows whether the
                                                                 //  extraction succeeds and so desynchronises its flat list on a -1; the mirror does not)
    if (bounding_box) *bounding_box = cv::Rect(bb.x, bb.y, bb.width, bb.height);
    return addSyntheticTemplate(pyr, class_id);
  }
  // Detector::addSyntheticTemplate (linemod.cpp:1636-1642): templates = one TemplatePyramid, (L0 M0, L0 M1, L1 M0, ...)
  int addSyntheticTemplate(const std::vector<Template>& templates, const String& class_id) {
    std::vector<TemplatePyramid>& tp = class_templates[class_id];
    const int template_id = (int)tp.size();
    tp.push_back(templates);
    dirty_ = true;
    return template_id;
  }
  // TemplatePoseInfo is ONE flat list indexed by template_id, exactly like the reference (linemod.cpp:1617-1634): correct
  // for a single class, which is how CadReco uses it (SURVEY.md A.6 iv)
  int addPoseInfo(const float* const pose_info) { TemplatePoseInfo.push_back(std::vector<float>(pose_info, pose_info + 13)); return (int)TemplatePoseInfo.size(); }
  std::vector<float> getPoseInfo(int template_id) { return TemplatePoseInfo.at((size_t)template_id); }
  int numPoseInfos() const { return (int)TemplatePoseInfo.size(); }   // mirror-only: lets writeLinemod stay inside the list
  // mirror-only: the pose of template `template_id` of class `class_id`.  The flat list holds the classes one after the other when the
  // detector came from a file (readClass appends class by class; notePoseOffset records where each class starts); without such a
  // record this is the reference's flat lookup.
  void notePoseOffset(const String& class_id) { pose_offset_[class_id] = TemplatePoseInfo.size(); }
  std::vector<float> getPoseInfo(const String& class_id, int template_id) {
    std::map<String, size_t>::const_iterator it = pose_offset_.find(class_id);
    return TemplatePoseInfo.at((it == pose_offset_.end() ? 0 : it->second) + (size_t)template_id);
  }

  const std::vector<Ptr<Modality> >& getModalities() const { return modalities; }
  int getT(int pyramid_level) const { return T_at_level[pyramid_level]; }
  int pyramidLevels() const { return pyramid_levels; }
  const std::vector<Template>& getTemplates(const String& class_id, int template_id) const {
    TemplatesMap::const_iterator i = class_templates.find(class_id);
    if (i == class_templates.end() || i->second.size() <= (size_t)template_id) throw cv::Exception("getTemplates: unknown class or template id");   // CV_Assert :1647-1648
    return i->second[template_id];
  }
  int numTemplates() const { int n = 0; for (TemplatesMap::const_iterator i = class_templates.begin(); i != class_templates.end(); ++i) n += (int)i->second.size(); return n; }
  int numTemplates(const String& class_id) const { TemplatesMap::const_iterator i = class_templates.find(class_id); return i == class_templates.end() ? 0 : (int)i->second.size(); }
  int numClasses() const { return (int)class_templates.size(); }
  std::vector<String> classIds() const { std::vector<String> ids; for (TemplatesMap::const_iterator i = class_templates.begin(); i != class_templates.end(); ++i) ids.push_back(i->first); return ids; }

  // the C-ABI handle behind this detector (created on first match), e.g. for fl_profile / fl_last_stage_ms
  fl_handle* handle() const { return handle_; }

  // mirror-only: a pipe of `depth` handles for frames up to W x H that hold this detector's templates in the order match() uploads them
  // (classes by id, templates by template_id), on the detector's device.  The caller owns it (fl_pipe_destroy).
  fl_pipe* createPipe(int depth, int W, int H) const {
    if (devices_.size() > 1) throw cv::Exception("Detector::createPipe is not available together with useDevices()");
    fl_params_t p = device_params(W, H);
    if (devices_.size() == 1) p.device = devices_[0];
    fl_pipe* pipe = nullptr;
    fealess_b200::check_status(fl_pipe_create(&p, depth, &pipe), "fl_pipe_create");
    std::vector<fl_template_hdr_t> hdr; std::vector<fl_feature_t> feat; std::vector<int32_t> class_of;
    flatten(hdr, feat, class_of);
    const int rc = fl_pipe_upload_templates(pipe, (int32_t)class_of.size(), hdr.data(), feat.data(), (int32_t)feat.size(), class_of.data(), nullptr);
    if (rc != FL_OK) fl_pipe_destroy(pipe);
    fealess_b200::check_status(rc, "fl_pipe_upload_templates");
    return pipe;
  }
  // mirror-only: the multi-device counterpart of createPipe - a group over the useDevices() list with `depth` slots (fl_group_create_pipe)
  // for frames up to W x H, holding this detector's templates in the order match() uploads them, dealt gid % n.  The caller owns it
  // (fl_group_destroy).
  fl_group* createGroupPipe(int depth, int W, int H) const {
    if (devices_.size() < 2) throw cv::Exception("Detector::createGroupPipe needs useDevices() with two or more devices");
    fl_params_t p = device_params(W, H);
    std::vector<int32_t> dv(devices_.begin(), devices_.end());
    fl_group* group = nullptr;
    fealess_b200::check_status(fl_group_create_pipe(&p, dv.data(), (int32_t)dv.size(), xcap_, depth, &group), "fl_group_create_pipe");
    std::vector<fl_template_hdr_t> hdr; std::vector<fl_feature_t> feat; std::vector<int32_t> class_of;
    flatten(hdr, feat, class_of);
    const int rc = fl_group_upload_templates(group, (int32_t)class_of.size(), hdr.data(), feat.data(), (int32_t)feat.size(), class_of.data(), nullptr);
    if (rc != FL_OK) fl_group_destroy(group);
    fealess_b200::check_status(rc, "fl_group_upload_templates");
    return group;
  }
  // mirror-only: the device list of useDevices() (empty: the default device)
  const std::vector<int>& devices() const { return devices_; }

 protected:
  std::vector<Ptr<Modality> > modalities;
  int pyramid_levels;
  std::vector<int> T_at_level;
  typedef std::vector<Template> TemplatePyramid;
  typedef std::map<String, std::vector<TemplatePyramid> > TemplatesMap;
  TemplatesMap class_templates;
  std::vector<std::vector<float> > TemplatePoseInfo;

 private:
  // create / grow the handle for this frame size and (re-)upload the flattened template database when it changed
  void ensure_uploaded(int W, int H) const {
    if (!handle_ || W > cap_w_ || H > cap_h_) {
      release_device();
      fl_params_t p = device_params(std::max(W, cap_w_), std::max(H, cap_h_));
      if (devices_.size() > 1) {
        std::vector<int32_t> dv(devices_.begin(), devices_.end());
        fealess_b200::check_status(fl_group_create(&p, dv.data(), (int32_t)dv.size(), xcap_, &group_), "fl_group_create");
        handle_ = fl_group_handle(group_, 0);                     // (owned by the group)
      } else {
        if (devices_.size() == 1) p.device = devices_[0];
        fealess_b200::check_status(fl_create(&p, &handle_), "fl_create");
      }
      cap_w_ = p.max_width; cap_h_ = p.max_height; dirty_ = true;
    }
    // host code that fills class_templates directly (the reference's readClass does) is caught by a template-count check
    const size_t fingerprint = (size_t)numTemplates() * 4099u + class_templates.size();
    if (!dirty_ && fingerprint == uploaded_fingerprint_) return;
    uploaded_fingerprint_ = fingerprint;
    std::vector<fl_template_hdr_t> hdr; std::vector<fl_feature_t> feat; std::vector<int32_t> class_of;
    flatten(hdr, feat, class_of);
    if (group_) fealess_b200::check_status(fl_group_upload_templates(group_, (int32_t)class_of.size(), hdr.data(), feat.data(), (int32_t)feat.size(), class_of.data(), nullptr), "fl_group_upload_templates");
    else fealess_b200::check_status(fl_upload_templates(handle_, (int32_t)class_of.size(), hdr.data(), feat.data(), (int32_t)feat.size(), class_of.data(), nullptr), "fl_upload_templates");
    dirty_ = false;
  }
  // handle parameters of this detector's modalities for frames up to W x H on device_ordinal()
  fl_params_t device_params(int W, int H) const {
    fl_params_t p;
    fl_default_params(&p);
    p.n_levels = pyramid_levels;
    if (pyramid_levels < 1 || pyramid_levels > FL_MAX_LEVELS || modalities.empty() || (int)modalities.size() > FL_MAX_MODALITIES) throw cv::Exception("Detector: unsupported number of pyramid levels / modalities");
    for (int l = 0; l < pyramid_levels; ++l) p.T[l] = T_at_level[l];
    p.n_modalities = (int)modalities.size();
    for (int m = 0; m < p.n_modalities; ++m) {
      p.modality_kind[m] = modalities[m]->kind();
      if (const ColorGradient* cg = dynamic_cast<const ColorGradient*>(modalities[m].get())) p.weak_threshold = cg->weak_threshold;
      if (const DepthNormal* dn = dynamic_cast<const DepthNormal*>(modalities[m].get())) { p.distance_threshold = dn->distance_threshold; p.difference_threshold = dn->difference_threshold; }
    }
    p.max_width = W; p.max_height = H;
    p.device = fealess_b200::device_ordinal();
    return p;
  }
  // the template database flattened in std::map (sorted class id) order = the order Detector::match visits the classes (:1418-1423)
  void flatten(std::vector<fl_template_hdr_t>& hdr, std::vector<fl_feature_t>& feat, std::vector<int32_t>& class_of) const {
    class_names_.clear(); class_index_.clear();
    const size_t per = (size_t)pyramid_levels * modalities.size();
    for (TemplatesMap::const_iterator it = class_templates.begin(); it != class_templates.end(); ++it) {
      const int ci = (int)class_names_.size();
      class_names_.push_back(it->first); class_index_[it->first] = ci;
      for (size_t t = 0; t < it->second.size(); ++t) {
        const TemplatePyramid& tp = it->second[t];
        if (tp.size() != per) throw cv::Exception("template pyramid size != pyramid_levels * modalities");
        for (size_t e = 0; e < per; ++e) {
          fl_template_hdr_t h;
          h.width = tp[e].width; h.height = tp[e].height; h.offset_x = tp[e].offset_x; h.offset_y = tp[e].offset_y; h.pyramid_level = tp[e].pyramid_level;
          h.feature_begin = (int32_t)feat.size(); h.feature_count = (int32_t)tp[e].features.size();
          for (size_t k = 0; k < tp[e].features.size(); ++k) { fl_feature_t f = {tp[e].features[k].x, tp[e].features[k].y, tp[e].features[k].label}; feat.push_back(f); }
          hdr.push_back(h);
        }
        class_of.push_back(ci);
      }
    }
  }
  // class filter named only unknown classes: nothing is matched, but the quantised images are still produced (:1411-1412)
  void fill_quantized_only(const uint8_t* bgr, size_t bgr_step, const uint16_t* depth, size_t depth_step, int W, int H, const uint8_t* const* masks,
                           cv::OutputArrayOfArrays quantized_images) const {
    if (!quantized_images.needed()) return;
    const int L = pyramid_levels, M = (int)modalities.size();
    std::vector<Mat> qimgs((size_t)L * M);
    std::vector<uint8_t*> qptr;
    for (int l = 0; l < L; ++l) for (int m = 0; m < M; ++m) { qimgs[l * M + m].create(H >> l, W >> l, CV_8UC1); qptr.push_back(qimgs[l * M + m].ptr<uint8_t>(0)); }
    const int32_t none = -1;                                    // a filter that enables no class
    fl_match_t dummy; int32_t count = 0;
    int rc = fl_match(handle_, bgr, bgr_step, depth, depth_step, W, H, masks, 100.0f, &none, 1, &dummy, 1, &count, qptr.data());
    fealess_b200::check_status(rc, "Detector::match");
    store_quantized(quantized_images, qimgs);
  }
  static void store_quantized(cv::OutputArrayOfArrays dst, std::vector<Mat>& qimgs) {
#ifdef FEALESS_B200_WITH_OPENCV
    dst.create(1, (int)qimgs.size(), CV_8U);                    // linemod.cpp:1361-1362
    for (size_t i = 0; i < qimgs.size(); ++i) { dst.create(qimgs[i].rows, qimgs[i].cols, CV_8U, (int)i); qimgs[i].copyTo(dst.getMatRef((int)i)); }
#else
    if (dst.vec()) *dst.vec() = qimgs;
#endif
  }

  void release_device() const {
    if (group_) { fl_group_destroy(group_); group_ = nullptr; handle_ = nullptr; }
    if (handle_) { fl_destroy(handle_); handle_ = nullptr; }
  }
  std::map<String, size_t> pose_offset_;
  mutable fl_handle* handle_;
  mutable fl_group* group_;
  std::vector<int> devices_;
  int xcap_;
  mutable bool dirty_;
  mutable int cap_w_, cap_h_;
  mutable size_t uploaded_fingerprint_ = 0;
  mutable std::vector<String> class_names_;
  mutable std::map<String, int> class_index_;
};

// linemod.cpp:1820-1835
inline Ptr<Detector> getDefaultLINE() {
  std::vector<Ptr<Modality> > modalities;
  modalities.push_back(Ptr<Modality>(new ColorGradient()));
  const int T_DEFAULTS[] = {5, 8};
  return Ptr<Detector>(new Detector(modalities, std::vector<int>(T_DEFAULTS, T_DEFAULTS + 2)));
}
inline Ptr<Detector> getDefaultLINEMOD() {
  std::vector<Ptr<Modality> > modalities;
  modalities.push_back(Ptr<Modality>(new ColorGradient()));
  modalities.push_back(Ptr<Modality>(new DepthNormal()));
  const int T_DEFAULTS[] = {5, 8};
  return Ptr<Detector>(new Detector(modalities, std::vector<int>(T_DEFAULTS, T_DEFAULTS + 2)));
}

}  // namespace cup_linemod

#endif  // FEALESS_B200_LINEMOD_HPP
