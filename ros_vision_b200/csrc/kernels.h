// Launch entry points of the engine's kernels (one translation unit per pipeline phase).
#ifndef B200TAG_KERNELS_H_
#define B200TAG_KERNELS_H_

#include <cuda_runtime.h>

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

// The main stream of a launch sequence, the optional timer, and the number of kernels launched so far
// (b200tag_kernels_per_batch).
struct Launcher {
  cudaStream_t s;
  KernelTimer *kt;
  int count = 0;
  // One kernel, timed as span `name` on s -- also when `launch` puts it on a side stream.
  template <class F>
  void timed(const char *name, F &&launch) {
    if (kt) kt->begin(name, s);
    launch();
    if (kt) kt->end(s);
    count++;
  }
  template <class F>
  void untimed(F &&launch) {
    launch();
    count++;
  }
};

void launch_frontend(const FrameParams &p, int frames, Launcher &ln);
void launch_blobs(const FrameParams &p, int frames, Launcher &ln, const SideStreams *side);
void launch_decode(const FrameParams &p, int frames, Launcher &ln);
size_t ccl_tiles_per_frame(int w, int h);  // CCL tiles of one frame and the capacity of a tile's root list
size_t ccl_root_cap();
void launch_hash_clear(const FrameParams &p, int frames, cudaStream_t s);
void launch_blobs_init(cudaStream_t s);

// The pose step (kernels_pose.cu): b200tag_estimate_pose (k_pose) or the IPPE pose (k_pose_ippe) of every raw
// detection, poses parallel to the records.
struct PoseLaunch {
  const b200tag_detection *dets;  // frame f's records start at dets + f * stride
  b200tag_pose *out;              // the same layout
  const Counters *counters;       // per-frame record counts; null: one list of `count` records
  uint32_t stride, count;
  double tagsize, fx, fy, cx, cy;
  int method;                     // B200TAG_POSE_*
};
void launch_pose(const PoseLaunch &L, int frames, Launcher &ln);

// The field pose step (kernels_pose.cu, k_field_pose): one b200tag_field_pose per frame from the frame's raw records.
namespace pose {
struct FieldKey;
struct FieldTagData;
}  // namespace pose
struct FieldLaunch {
  const b200tag_detection *dets;     // frame f's records start at dets + f * stride
  const Counters *counters;          // per-frame record counts; null: one list of `count` records
  uint32_t stride, count;
  const b200tag_field_tag *layout;   // device copies of the layout and its sorted keys
  const pose::FieldKey *keys;
  int nlayout;
  pose::FieldTagData *scratch;       // frame f's used tags start at scratch + f * scratch_stride
  uint32_t scratch_stride;           // >= min(records, nlayout) of any frame
  double tagsize, fx, fy, cx, cy;
  double rotation[9], offset[3];
  b200tag_field_pose *out;           // one per frame
};
void launch_field_pose(const FieldLaunch &L, int frames, Launcher &ln);
size_t field_tag_bytes();            // sizeof(pose::FieldTagData)

// JPEG luminance planes of a batch (jpeg.h): the parallel kernels for streams without restart markers, the sequential
// warp-per-frame kernel for the rest.
struct JpegBatch;
void launch_jpeg_decode(const JpegBatch &B, bool any_parallel, cudaStream_t s);

}  // namespace b200tag

#endif
