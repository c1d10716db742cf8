// Masked frames through a template-sharded cup_linemod::Detector (useDevices, fl_group_match_masked) must give what one device gives:
// the same match list and the same quantised images, for masks on the colour modality only, on the depth modality only and on both.
// usage: masked_group_test <case file> <comma separated device ordinals, e.g. 0,0 or 0,1>
// The case file is the one tests/test_gpu_masked_frames.py writes (frame, templates, threshold, one mask per modality).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "fealess_b200/linemod.hpp"

static std::vector<unsigned char> g_buf;
static size_t g_pos = 0;
template <typename T> static T rd() { T v; std::memcpy(&v, &g_buf[g_pos], sizeof(T)); g_pos += sizeof(T); return v; }
template <typename T> static std::vector<T> rdv(size_t n) { std::vector<T> v(n); if (n) std::memcpy(v.data(), &g_buf[g_pos], n * sizeof(T)); g_pos += n * sizeof(T); return v; }
static int g_fail = 0;
#define CHECK(cond, ...) do { if (!(cond)) { std::printf("FAIL %s:%d: ", __FILE__, __LINE__); std::printf(__VA_ARGS__); std::printf("\n"); ++g_fail; } } while (0)

static void add_templates(cup_linemod::Detector& det, int L, int M, int n_templates, const std::vector<int32_t>& headers,
                          const std::vector<int32_t>& features, const std::vector<int32_t>& class_of) {
  for (int t = 0; t < n_templates; ++t) {
    std::vector<cup_linemod::Template> pyr((size_t)L * M);
    for (int e = 0; e < L * M; ++e) {
      const int32_t* h = &headers[((size_t)t * L * M + e) * 7];
      pyr[e].width = h[0]; pyr[e].height = h[1]; pyr[e].offset_x = h[2]; pyr[e].offset_y = h[3]; pyr[e].pyramid_level = h[4];
      for (int k = 0; k < h[6]; ++k) pyr[e].features.push_back(cup_linemod::Feature(features[3 * (h[5] + k)], features[3 * (h[5] + k) + 1], features[3 * (h[5] + k) + 2]));
    }
    char name[32]; std::snprintf(name, sizeof name, "obj%02d", class_of[t]);
    det.addSyntheticTemplate(pyr, name);
  }
}

int main(int argc, char** argv) {
  if (argc < 3) { std::printf("usage: masked_group_test <case file> <devices>\n"); return 2; }
  FILE* f = std::fopen(argv[1], "rb");
  if (!f) { std::printf("cannot open %s\n", argv[1]); return 2; }
  std::fseek(f, 0, SEEK_END); long sz = std::ftell(f); std::fseek(f, 0, SEEK_SET);
  g_buf.resize((size_t)sz);
  if (std::fread(g_buf.data(), 1, (size_t)sz, f) != (size_t)sz) return 2;
  std::fclose(f);
  std::vector<int> devices;
  for (char* tok = std::strtok(argv[2], ","); tok; tok = std::strtok(nullptr, ",")) devices.push_back(std::atoi(tok));

  const int W = rd<int32_t>(), H = rd<int32_t>();
  std::vector<uint8_t> bgr = rdv<uint8_t>((size_t)W * H * 3);
  std::vector<uint16_t> depth = rdv<uint16_t>((size_t)W * H);
  const int L = rd<int32_t>(), M = rd<int32_t>();
  std::vector<int32_t> T = rdv<int32_t>(L);
  const int n_templates = rd<int32_t>();
  std::vector<int32_t> headers = rdv<int32_t>((size_t)n_templates * L * M * 7);
  const int n_features = rd<int32_t>();
  std::vector<int32_t> features = rdv<int32_t>((size_t)n_features * 3);
  std::vector<int32_t> class_of = rdv<int32_t>(n_templates);
  const float threshold = rd<float>();
  std::vector<uint8_t> mask0 = rdv<uint8_t>((size_t)W * H), mask1 = rdv<uint8_t>((size_t)W * H);

  try {
    cv::Ptr<cup_linemod::Detector> one = cup_linemod::getDefaultLINEMOD(), group = cup_linemod::getDefaultLINEMOD();
    group->useDevices(devices, 4096);
    add_templates(*one, L, M, n_templates, headers, features, class_of);
    add_templates(*group, L, M, n_templates, headers, features, class_of);
    std::vector<cv::Mat> sources;
    sources.push_back(cv::Mat(H, W, CV_8UC3, bgr.data()));
    sources.push_back(cv::Mat(H, W, CV_16UC1, depth.data()));
    const cv::Mat k0(H, W, CV_8UC1, mask0.data()), k1(H, W, CV_8UC1, mask1.data()), none;
    const char* names[3] = {"colour only", "depth only", "both"};
    int total = 0;
    for (int c = 0; c < 3; ++c) {
      std::vector<cv::Mat> masks;
      masks.push_back(c == 1 ? none : k0);
      masks.push_back(c == 0 ? none : k1);
      std::vector<cup_linemod::Match> want, got;
      std::vector<cv::Mat> qwant, qgot;
      CHECK(one->match(sources, threshold, want, std::vector<cv::String>(), qwant, masks) == 0, "%s: single-device match", names[c]);
      CHECK(group->match(sources, threshold, got, std::vector<cv::String>(), qgot, masks) == 0, "%s: group match", names[c]);
      CHECK(got.size() == want.size(), "%s: %d matches, one device gives %d", names[c], (int)got.size(), (int)want.size());
      for (size_t i = 0; i < want.size() && i < got.size(); ++i)
        CHECK(got[i].x == want[i].x && got[i].y == want[i].y && got[i].similarity == want[i].similarity && got[i].template_id == want[i].template_id &&
              got[i].class_id == want[i].class_id, "%s: match %d differs", names[c], (int)i);
      CHECK((int)qgot.size() == L * M && qwant.size() == qgot.size(), "%s: quantised images", names[c]);
      for (size_t i = 0; i < qwant.size() && i < qgot.size(); ++i) {
        bool same = qgot[i].rows == qwant[i].rows && qgot[i].cols == qwant[i].cols;
        for (int y = 0; same && y < qwant[i].rows; ++y) same = std::memcmp(qgot[i].ptr<uint8_t>(y), qwant[i].ptr<uint8_t>(y), (size_t)qwant[i].cols) == 0;
        CHECK(same, "%s: quantised image %d differs", names[c], (int)i);
      }
      total += (int)want.size();
    }
    CHECK(total > 0, "no case produced a match");
    // a wrong mask count is the reference's -1 (linemod.cpp:1374-1377) in group mode too
    std::vector<cup_linemod::Match> m;
    CHECK(group->match(sources, threshold, m, std::vector<cv::String>(), cv::noArray(), std::vector<cv::Mat>(1, k0)) == -1, "mask count");
  } catch (const std::exception& e) {
    std::printf("FAIL exception: %s\n", e.what()); ++g_fail;
  }
  if (g_fail == 0) std::printf("all checks passed (%d devices)\n", (int)devices.size());
  return g_fail ? 1 : 0;
}
