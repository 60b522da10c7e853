// voxel.h -- host-side launcher interface of voxel.cu: pcl::VoxelGrid<pcl::PointXYZ> on the device, applied to
// the clouds of a frame batch (D2PC_FILTER_VOXEL: the CROP clouds, or the crop box's; the recipe is in
// include/d2pc_b200.h).  Input, destination and batch limit are cloud_stage.cuh's.
#pragma once
#include "cloud_stage.cuh"

namespace d2pc {

struct VoxelParams {
  float inv[3];          // 1.0f / leaf, per axis (float32 division, as PCL's inverse_leaf_size_)
  uint32_t min_points;   // min_points_per_voxel
  int limit_field;       // -1 none, 0 x, 1 y, 2 z
  double limit_min, limit_max;
};

// Device scratch for one launch (keys, indices, sort / scan temp storage, bounds, descriptors).  Sized once per frame
// geometry; nothing in it needs clearing.
size_t voxel_scratch_bytes(uint32_t n_frames, uint32_t n_max);
// The voxel clouds and their per-frame counts into out; positions at or past a frame's input count are excluded.
// fallback (may be null): per frame, 1 when the frame took the overflow fallback (its output is its input cloud).
cudaError_t launch_voxel(const CloudSrc &in, const CloudDst &out, const VoxelParams &p, uint32_t *fallback,
                         void *scratch, cudaStream_t stream, int *launches);

}  // namespace d2pc
