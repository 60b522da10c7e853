// crop_box.h -- host-side launcher interface of crop_box.cu: pcl::CropBox<pcl::PointXYZ> (setTransform only) on the
// device, applied to the clouds of a frame batch (the first stage behind the CROP kernels when a box is enabled; the
// recipe is in include/d2pc_b200.h).  Input, destination and batch limit are cloud_stage.cuh's.
#pragma once
#include "cloud_stage.cuh"

namespace d2pc {

struct CropBoxParams {
  float mn[3], mx[3];  // the box's faces (inclusive), in the box frame
  float t[12];         // row-major 3x4 [R | t]: camera frame -> box frame
};

// Device scratch of one launch (the scan's output slots and the scan's temp storage).  Sized once per geometry;
// nothing in it needs clearing.
size_t crop_box_scratch_bytes(uint32_t n_frames, uint32_t n_max);
// Kept points, unchanged and in input order, and their per-frame counts into out.  The box is taken by value: a
// launch keeps the setting it was enqueued with.
cudaError_t launch_crop_box(const CloudSrc &in, const CloudDst &out, const CropBoxParams &box, void *scratch,
                            cudaStream_t stream, int *launches);

}  // namespace d2pc
