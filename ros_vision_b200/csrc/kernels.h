// Launch entry points of the engine's kernels (one translation unit per pipeline phase).
#ifndef B200TAG_KERNELS_H_
#define B200TAG_KERNELS_H_

#include <cuda_runtime.h>

#include <cstdlib>
#include <string>
#include <vector>

#include "dev_types.h"

namespace b200tag {

// Optional per-kernel CUDA-event timing (b200tag_profile_device); null in normal runs.
struct KernelTimer {
  struct Span {
    const char *name;
    cudaEvent_t a, b;
  };
  std::vector<Span> spans;
  size_t cursor = 0;
  bool recording = false;
  void begin(const char *name, cudaStream_t s) {
    if (cursor == spans.size()) {
      Span sp{name, nullptr, nullptr};
      cudaEventCreate(&sp.a);
      cudaEventCreate(&sp.b);
      spans.push_back(sp);
    }
    spans[cursor].name = name;
    cudaEventRecord(spans[cursor].a, s);
  }
  void end(cudaStream_t s) {
    cudaEventRecord(spans[cursor].b, s);
    cursor++;
  }
  void rewind() { cursor = 0; }
  ~KernelTimer() {
    for (auto &sp : spans) {
      cudaEventDestroy(sp.a);
      cudaEventDestroy(sp.b);
    }
  }
};

// Side streams + events that let the three independent blob-tier kernels run concurrently (fork after the
// scatter, join before the quad search).  Owned by the detector; null = everything on the main stream.
struct SideStreams {
  cudaStream_t s[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t fork = nullptr, join[3] = {nullptr, nullptr, nullptr};
};

// Measurement switches (bit mask in the environment variable B200TAG_EXP, read once): select another variant of a
// kernel so that both can be timed in one run (tools/exp_kernels.py).  Unset = the production variants.
//    1: k_scatter with one point in flight per thread (production: 4)      32: ... with 8
//    2: k_boundary with the uncapped point list and a 512-entry CTA-local table (9 CTAs per SM; production: 16)
//    4: k_boundary with the capped list and a 512-entry table (12 CTAs per SM)
//    8: k_ccl_final without the 32-register cap (6 CTAs per SM; production: 8)
//   64: k_select at 5 instead of 8 CTAs per SM, grid sized for 4 per SM
//  512: the shared-memory tile blur for filter lengths 3, 5, 7 (production: k_blur_strip)
inline int exp_flags() {
  static const int f = [] { const char *e = getenv("B200TAG_EXP"); return e ? atoi(e) : 0; }();
  return f;
}

// Each returns the number of kernels it launched.
int launch_frontend(const FrameParams &p, int frames, cudaStream_t s, KernelTimer *kt);
int launch_blobs(const FrameParams &p, int frames, cudaStream_t s, KernelTimer *kt, const SideStreams *side);
int launch_decode(const FrameParams &p, int frames, cudaStream_t s, KernelTimer *kt);
size_t ccl_tiles_per_frame(int w, int h);  // CCL tiles of one frame and the capacity of a tile's root list
size_t ccl_root_cap();
void launch_hash_clear(const FrameParams &p, int frames, cudaStream_t s);
void launch_blobs_init(cudaStream_t s);

// The pose step (kernels_pose.cu): b200tag_estimate_pose of every raw detection, poses parallel to the records.
struct PoseLaunch {
  const b200tag_detection *dets;  // frame f's records start at dets + f * stride
  b200tag_pose *out;              // the same layout
  const Counters *counters;       // per-frame record counts; null: one list of `count` records
  uint32_t stride, count;
  double tagsize, fx, fy, cx, cy;
};
int launch_pose(const PoseLaunch &L, int frames, cudaStream_t s, KernelTimer *kt);

// JPEG luminance planes of a batch (jpeg.h): the parallel kernels for streams without restart markers, the sequential
// warp-per-frame kernel for the rest.  Returns the number of kernels launched.
struct JpegBatch;
int launch_jpeg_decode(const JpegBatch &B, bool any_parallel, cudaStream_t s);

}  // namespace b200tag

#endif
