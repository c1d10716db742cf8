// Driver of tests/test_gpu_reco_stream.py: CObjRecoLmICP::SubmitRecognition / CollectRecognition (include/fealess_b200/obj_reco.hpp).
//   reco_stream_test <dir> <frames_in_flight> <top_k> <per_class> <th_obj_dist> <frame.bin>...
// AddObj, SetHypotheses, SetFramesInFlight, then every frame is submitted with at most frames_in_flight in flight from this one thread
// and collected in order; one line per frame as reco_test prints it.  frame.bin = int32 W, H, double fx, fy, cx, cy, BGR bytes, depth u16.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <string>
#include <vector>

#include "fealess_b200/obj_reco.hpp"

struct Frame { std::vector<unsigned char> rgb; std::vector<unsigned short> dep; TImageU tRGB; TImageU16 tDepth; TCamIntrinsicParam K; };

static bool load(const char* path, Frame& fr) {
  FILE* f = std::fopen(path, "rb");
  if (!f) return false;
  int wh[2]; double k[4];
  bool ok = std::fread(wh, 4, 2, f) == 2 && std::fread(k, 8, 4, f) == 4;
  if (ok) {
    fr.rgb.resize((size_t)wh[0] * wh[1] * 3); fr.dep.resize((size_t)wh[0] * wh[1]);
    ok = std::fread(fr.rgb.data(), 1, fr.rgb.size(), f) == fr.rgb.size() && std::fread(fr.dep.data(), 2, fr.dep.size(), f) == fr.dep.size();
  }
  std::fclose(f);
  const TImageU tRGB = {1.0, fr.rgb.data(), wh[0], wh[1]};
  const TImageU16 tDepth = {1.0, fr.dep.data(), wh[0], wh[1]};
  const TCamIntrinsicParam K = {wh[0], wh[1], k[0], k[1], k[2], k[3], std::vector<double>()};
  fr.tRGB = tRGB; fr.tDepth = tDepth; fr.K = K;
  return ok;
}

static void print(int frame, int rc, const std::vector<TObjRecoResult>& res) {
  std::printf("frame %d status %08x results %zu", frame, (unsigned)rc, res.size());
  for (size_t i = 0; i < res.size(); ++i) {
    std::printf(" %s", res[i].strObjTag.c_str());
    for (int j = 0; j < 16; ++j) { unsigned u; std::memcpy(&u, &res[i].tWorld2Cam[j], 4); std::printf(" %08x", u); }
  }
  std::printf("\n");
}

int main(int argc, char** argv) {
  if (argc < 7) {
    std::printf("usage: reco_stream_test <dir> <frames_in_flight> <top_k> <per_class> <th_obj_dist> <frame.bin>...\n");
    return 2;
  }
  try {
    CObjRecoLmICP reco;
    std::printf("addobj %08x\n", (unsigned)reco.AddObj(argv[1]));
    const int depth = std::atoi(argv[2]);
    reco.SetHypotheses(std::atoi(argv[3]), std::atoi(argv[4]) != 0, (float)std::atof(argv[5]));
    reco.SetFramesInFlight(depth);
    std::vector<Frame> frames((size_t)(argc - 6));
    for (int a = 6; a < argc; ++a)
      if (!load(argv[a], frames[(size_t)(a - 6)])) { std::printf("cannot read %s\n", argv[a]); return 2; }
    std::deque<int> queued;
    int next = 0;
    std::vector<TObjRecoResult> res;
    while (next < (int)frames.size() || !queued.empty()) {
      if (next < (int)frames.size() && (int)queued.size() < depth) {
        const Frame& f = frames[(size_t)next];
        const int rc = reco.SubmitRecognition(f.tRGB, f.tDepth, f.K);
        if (rc != 0) { res.clear(); print(next, rc, res); } else queued.push_back(next);
        ++next;
        continue;
      }
      const int rc = reco.CollectRecognition(res);
      print(queued.front(), rc, res);
      queued.pop_front();
    }
    return 0;
  } catch (const cv::Exception& e) {
    std::printf("cv::Exception: %s\n", e.what());
    return 3;
  } catch (const std::exception& e) {
    std::printf("exception: %s\n", e.what());
    return 4;
  }
}
