// The node's pose step on the GPU through the C++ class, as INTEGRATION.md shows it: the detector's handle() turns on
// the device pose step, and after Detect the poses and robot-frame records come back parallel to Detections().
//   pose_step_test <gray.raw> <width> <height> <fx> <fy> <cx> <cy> <tagsize>
// Prints one line per detection (id, pose) and one per tag position (closest first) with every digit.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "apriltags_cuda/apriltag_gpu.h"

int main(int argc, char **argv) {
  if (argc < 9) return 2;
  const int width = std::atoi(argv[2]), height = std::atoi(argv[3]);
  const double fx = std::atof(argv[4]), fy = std::atof(argv[5]), cx = std::atof(argv[6]), cy = std::atof(argv[7]);
  const double tagsize = std::atof(argv[8]);
  std::vector<uint8_t> gray(static_cast<size_t>(width) * height);
  FILE *f = std::fopen(argv[1], "rb");
  if (!f || std::fread(gray.data(), 1, gray.size(), f) != gray.size()) return 3;
  std::fclose(f);

  apriltag_family_t *tf = tag36h11_create();
  apriltag_detector_t *td = apriltag_detector_create();
  apriltag_detector_add_family(td, tf);
  td->quad_decimate = 2.0;
  td->quad_sigma = 0.0;
  td->refine_edges = true;
  frc971::apriltag::CameraMatrix cam{fx, cx, fy, cy};
  frc971::apriltag::DistCoeffs dist{0, 0, 0, 0, 0};
  const double rotation[9] = {0, 0, 1, -1, 0, 0, 0, -1, 0}, offset[3] = {0.1, -0.2, 0.5};  // the camera's extrinsics
  int rc = 0;
  {
    frc971::apriltag::GpuDetector detector(width, height, td, cam, dist, B200TAG_FMT_GRAY8);
    if (b200tag_set_pose_estimation(detector.handle(), tagsize, fx, fy, cx, cy, rotation, offset) != 0) return 4;
    detector.Detect(gray.data());
    const zarray_t *detections = detector.Detections();
    int npose = 0, npos = 0;
    const b200tag_pose *poses = b200tag_poses(detector.handle(), 0, &npose);
    const b200tag_tag_position *tags = b200tag_tag_positions(detector.handle(), 0, &npos);
    if (npose != zarray_size(detections) || npos != npose) rc = 5;
    for (int i = 0; i < zarray_size(detections) && i < npose; i++) {
      apriltag_detection_t *det;
      zarray_get(detections, i, &det);
      std::printf("pose %d %.17g %.17g %.17g %.17g\n", det->id, poses[i].t[0], poses[i].t[1], poses[i].t[2], poses[i].err);
    }
    for (int i = 0; i < npos; i++)
      std::printf("tag %d %d %.17g %.17g %.17g %.17g\n", tags[i].index, tags[i].id, tags[i].robot[0], tags[i].robot[1],
                  tags[i].robot[2], tags[i].distance);
  }
  apriltag_detector_destroy(td);
  tag36h11_destroy(tf);
  return rc;
}
