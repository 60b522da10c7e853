// cloud_transform.h -- host-side launcher interface of cloud_transform.cu: pcl::transformPointCloud<pcl::PointXYZ>
// with an affine matrix on the device, applied to the clouds of a frame batch (the first cloud stage behind the
// reproject kernels when a transform is enabled; the recipe is in include/d2pc_b200.h).  Input, destination and batch
// limit are cloud_stage.cuh's.
#pragma once
#include "cloud_stage.cuh"

namespace d2pc {

struct CloudTransformParams {
  float m[12];  // row-major 3x4 [A | t]: camera frame -> target frame
};

// Every point below frame f's count, transformed (finite x, y, z) or copied unchanged (otherwise), in input order;
// positions at or past the count are neither read nor written.  out.counts[f] = the frame's input count where
// out.counts is non-null.  out may be exactly the input (same pointer and stride): each point is read and written by
// one thread.  per_frame null: every frame uses t (taken by value, so a launch keeps the setting it was enqueued
// with); otherwise frame f uses per_frame + 12 * f (device memory).  One launch, no scratch.
cudaError_t launch_cloud_transform(const CloudSrc &in, const CloudDst &out, const CloudTransformParams &t,
                                   const float *per_frame, cudaStream_t stream, int *launches);

}  // namespace d2pc
