// Driver of tests/test_gpu_reco_group.py: CObjRecoLmICP::SetDevices (include/fealess_b200/obj_reco.hpp) against the single-GPU class.
//   reco_group_test <dir> <devices> <frames_in_flight> <top_k> <per_class> <th_obj_dist> <frame.bin>...
// devices = comma-separated ordinals ("0,0" = two members on GPU 0).  Three passes over the frames, one line per frame each:
//   "one"     CObjRecoLmICP without SetDevices, Recognition;
//   "sync"    SetDevices(devices) before AddObj, Recognition (a depth-1 group of its own);
//   "stream"  the same object, SetFramesInFlight(frames_in_flight), SubmitRecognition / CollectRecognition from this one thread.
// A frame whose call throws prints "exception" instead of its results.  frame.bin as reco_stream_test reads it.  Then the argument
// checks: Recognition with sizes that disagree returns ERROR_INVALID_PARAM on both objects.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <sstream>
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

static void print(const char* pass, int frame, int rc, const std::vector<TObjRecoResult>& res) {
  std::printf("%s frame %d status %08x results %zu", pass, frame, (unsigned)rc, res.size());
  for (size_t i = 0; i < res.size(); ++i) {
    std::printf(" %s", res[i].strObjTag.c_str());
    for (int j = 0; j < 16; ++j) { unsigned u; std::memcpy(&u, &res[i].tWorld2Cam[j], 4); std::printf(" %08x", u); }
  }
  std::printf("\n");
}

static void recognition_pass(const char* pass, CObjRecoLmICP& reco, const std::vector<Frame>& frames) {
  std::vector<TObjRecoResult> res;
  for (size_t i = 0; i < frames.size(); ++i) {
    try {
      const int rc = reco.Recognition(frames[i].tRGB, frames[i].tDepth, frames[i].K, res);
      print(pass, (int)i, rc, res);
    } catch (const cv::Exception&) {
      std::printf("%s frame %d exception\n", pass, (int)i);
    }
  }
}

int main(int argc, char** argv) {
  if (argc < 8) {
    std::printf("usage: reco_group_test <dir> <devices> <frames_in_flight> <top_k> <per_class> <th_obj_dist> <frame.bin>...\n");
    return 2;
  }
  try {
    std::vector<int> devices;
    {
      std::stringstream ss(argv[2]);
      std::string tok;
      while (std::getline(ss, tok, ',')) devices.push_back(std::atoi(tok.c_str()));
    }
    const int depth = std::atoi(argv[3]);
    const int top_k = std::atoi(argv[4]);
    const bool per_class = std::atoi(argv[5]) != 0;
    const float th = (float)std::atof(argv[6]);
    std::vector<Frame> frames((size_t)(argc - 7));
    for (int a = 7; a < argc; ++a)
      if (!load(argv[a], frames[(size_t)(a - 7)])) { std::printf("cannot read %s\n", argv[a]); return 2; }

    CObjRecoLmICP one;
    std::printf("one addobj %08x\n", (unsigned)one.AddObj(argv[1]));
    one.SetHypotheses(top_k, per_class, th);
    recognition_pass("one", one, frames);

    CObjRecoLmICP multi;
    multi.SetDevices(devices);                                    // before AddObj: kept when AddObj replaces the detector
    std::printf("multi addobj %08x\n", (unsigned)multi.AddObj(argv[1]));
    multi.SetHypotheses(top_k, per_class, th);
    recognition_pass("sync", multi, frames);

    multi.SetFramesInFlight(depth);
    std::deque<int> queued;
    int next = 0;
    std::vector<TObjRecoResult> res;
    while (next < (int)frames.size() || !queued.empty()) {
      if (next < (int)frames.size() && (int)queued.size() < depth) {
        const Frame& f = frames[(size_t)next];
        const int rc = multi.SubmitRecognition(f.tRGB, f.tDepth, f.K);
        if (rc != 0) { res.clear(); print("stream", next, rc, res); } else queued.push_back(next);
        ++next;
        continue;
      }
      try {
        const int rc = multi.CollectRecognition(res);
        print("stream", queued.front(), rc, res);
      } catch (const cv::Exception&) {
        std::printf("stream frame %d exception\n", queued.front());
      }
      queued.pop_front();
    }

    // ERROR_INVALID_PARAM cases: sizes that disagree with the intrinsics
    const Frame& f = frames[0];
    TCamIntrinsicParam bad = f.K;
    bad.nWidth += 2;
    std::vector<TObjRecoResult> r1, r2;
    std::printf("badparams %08x %08x %08x\n", (unsigned)one.Recognition(f.tRGB, f.tDepth, bad, r1), (unsigned)multi.Recognition(f.tRGB, f.tDepth, bad, r2),
                (unsigned)multi.SubmitRecognition(f.tRGB, f.tDepth, bad));
    return 0;
  } catch (const cv::Exception& e) {
    std::printf("cv::Exception: %s\n", e.what());
    return 3;
  } catch (const std::exception& e) {
    std::printf("exception: %s\n", e.what());
    return 4;
  }
}
