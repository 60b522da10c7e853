// radius_outlier.h -- host-side launcher interface of radius_outlier.cu: pcl::RadiusOutlierRemoval<pcl::PointXYZ>
// on the device, applied to the clouds of a frame batch (the stage behind every filter mode when a radius is set;
// the recipe is in include/d2pc_b200.h).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace d2pc {

struct RorLaunch {
  // n_frames input clouds: frame f's points at in + f * in_stride bytes, in_counts[f] of them (values above n_max
  // count as n_max; in_counts null: n_max each).  16-byte points, 16-byte aligned.
  uint32_t n_frames = 0;
  uint32_t n_max = 0;
  const uint8_t *in = nullptr;
  size_t in_stride = 0;
  const uint32_t *in_counts = nullptr;
  double radius = 0.0;  // finite, > 0
  uint32_t min_neighbors = 1;
  uint8_t *out = nullptr;  // kept points, frame f at out + f * out_stride bytes; must not overlap the input
  size_t out_stride = 0;
  uint32_t *counts = nullptr;  // per frame: points kept
  void *scratch = nullptr;     // ror_scratch_bytes(n_frames, n_max)
};

// Device scratch of one launch (bounds, keys, indices, the points in cell order, flags, sort / scan temp storage).
// Sized once per geometry; nothing in it needs clearing.
size_t ror_scratch_bytes(uint32_t n_frames, uint32_t n_max);
// n_frames * n_max <= kRorMaxPoints (the sort and scan index with int)
constexpr uint64_t kRorMaxPoints = 0x7ffffffeull;
cudaError_t launch_radius_outlier(const RorLaunch &L, cudaStream_t stream, int *launches);

// The buffer of the stage behind a filter mode: the mode's clouds (dense, frame f at f * n * 16 bytes), their
// per-frame counts, then the stage's own scratch.
struct RorStage {
  uint8_t *clouds;
  uint32_t *counts;
  void *scratch;
};
size_t ror_stage_bytes(uint32_t n_frames, uint32_t n);
RorStage ror_stage(void *buffer, uint32_t n_frames, uint32_t n);

}  // namespace d2pc
