// crop_box.h -- host-side launcher interface of crop_box.cu: pcl::CropBox<pcl::PointXYZ> (setTransform only) on the
// device, applied to the clouds of a frame batch (the stage in front of VOXEL and the radius outlier stage when a box
// is enabled; the recipe is in include/d2pc_b200.h).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace d2pc {

struct CropBoxParams {
  float mn[3], mx[3];  // the box's faces (inclusive), in the box frame
  float t[12];         // row-major 3x4 [R | t]: camera frame -> box frame
};

struct CropBoxLaunch {
  // n_frames input clouds: frame f's points at in + f * in_stride bytes, in_counts[f] of them (values above n_max
  // count as n_max; in_counts null: n_max each).  16-byte points, 16-byte aligned.
  uint32_t n_frames = 0;
  uint32_t n_max = 0;
  const uint8_t *in = nullptr;
  size_t in_stride = 0;
  const uint32_t *in_counts = nullptr;
  CropBoxParams box;       // by value: a launch keeps the setting it was enqueued with
  uint8_t *out = nullptr;  // kept points, frame f at out + f * out_stride bytes; must not overlap the input
  size_t out_stride = 0;
  uint32_t *counts = nullptr;  // per frame: points kept
  void *scratch = nullptr;     // crop_box_scratch_bytes(n_frames, n_max)
};

// Device scratch of one launch (the scan's output slots and the scan's temp storage).  Sized once per geometry;
// nothing in it needs clearing.
size_t crop_box_scratch_bytes(uint32_t n_frames, uint32_t n_max);
// n_frames * n_max <= kCropBoxMaxPoints (the scan indexes n_frames * n_max + 1 positions with int)
constexpr uint64_t kCropBoxMaxPoints = 0x7ffffffeull;
cudaError_t launch_crop_box(const CropBoxLaunch &L, cudaStream_t stream, int *launches);

// The buffer of the stage in front of VOXEL / the outlier stage: its input clouds (dense, frame f at f * n * 16
// bytes), the per-frame counts of its output where the next stage has no count slot of its own (VOXEL), then the
// stage's scratch.
struct CropBoxStage {
  uint8_t *clouds;
  uint32_t *counts;
  void *scratch;
};
size_t crop_box_stage_bytes(uint32_t n_frames, uint32_t n);
CropBoxStage crop_box_stage(void *buffer, uint32_t n_frames, uint32_t n);

}  // namespace d2pc
