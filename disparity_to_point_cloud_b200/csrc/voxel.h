// voxel.h -- host-side launcher interface of voxel.cu: pcl::VoxelGrid<pcl::PointXYZ> on the device, applied to
// the CROP clouds of a frame batch (D2PC_FILTER_VOXEL; the recipe is in include/d2pc_b200.h).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace d2pc {

struct VoxelParams {
  float inv[3];          // 1.0f / leaf, per axis (float32 division, as PCL's inverse_leaf_size_)
  uint32_t min_points;   // min_points_per_voxel
  int limit_field;       // -1 none, 0 x, 1 y, 2 z
  double limit_min, limit_max;
};

struct VoxelLaunch {
  // n_frames clouds of at most n points each, frame f at voxel_crop(scratch) + f * n (dense, written by the CROP
  // kernels or the crop box)
  uint32_t n_frames = 0;
  uint32_t n = 0;
  // per frame (may be null: n each): the points of the frame's cloud; positions at or past it are excluded
  const uint32_t *in_counts = nullptr;
  VoxelParams p;
  uint8_t *out = nullptr;  // voxel clouds, frame f at out + f * out_stride bytes
  size_t out_stride = 0;
  uint32_t *counts = nullptr;    // per frame: points written
  uint32_t *fallback = nullptr;  // per frame (may be null): 1 when the frame took the overflow fallback
  void *scratch = nullptr;       // voxel_scratch_bytes(n_frames, n)
};

// Device scratch for one launch (the CROP clouds first, then keys, indices, sort / scan temp storage, descriptors).
// Sized once per frame geometry; nothing in it needs clearing.
size_t voxel_scratch_bytes(uint32_t n_frames, uint32_t n);
// Where the CROP kernels must write the batch's clouds (the head of the scratch).
inline float *voxel_crop(void *scratch) { return static_cast<float *>(scratch); }
// n_frames * n < 2^31 (the sort and scan index with int)
cudaError_t launch_voxel(const VoxelLaunch &L, cudaStream_t stream, int *launches);

}  // namespace d2pc
