// radius_outlier.h -- host-side launcher interface of radius_outlier.cu: pcl::RadiusOutlierRemoval<pcl::PointXYZ>
// on the device, applied to the clouds of a frame batch (the last stage behind every filter mode when a radius is
// set; the recipe is in include/d2pc_b200.h).  Input, destination and batch limit are cloud_stage.cuh's.
#pragma once
#include "cloud_stage.cuh"

namespace d2pc {

// Device scratch of one launch (bounds, keys, indices, the points in cell order, flags, sort / scan temp storage).
// Sized once per geometry; nothing in it needs clearing.
size_t ror_scratch_bytes(uint32_t n_frames, uint32_t n_max);
// Kept points, unchanged and in input order, and their per-frame counts into out.  radius finite and > 0.
cudaError_t launch_radius_outlier(const CloudSrc &in, const CloudDst &out, double radius, uint32_t min_neighbors,
                                  void *scratch, cudaStream_t stream, int *launches);

}  // namespace d2pc
