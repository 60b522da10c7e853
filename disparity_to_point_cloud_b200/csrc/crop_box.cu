// crop_box.cu -- pcl::CropBox<pcl::PointXYZ> (setTransform only, setNegative(false), keep_organized false) on the
// device, batched over frames: the first stage behind the CROP kernels when a box is enabled, and
// d2pc_crop_box_device.  include/d2pc_b200.h states the recipe.  The stage is the predicate `inside` and
// cloud_stage.cuh's order-preserving compaction over it, in two launches: the scan reads the predicate through a
// transform iterator (no flag array), and the scatter evaluates it again and copies the kept points.
//
// The local coordinates are cloud_stage.cuh's affine_row, the transform stage's rounding recipe.  No buffer is read
// before a kernel of the same launch has written it, so the scratch needs no clearing.
#include "crop_box.h"

namespace d2pc {
namespace {

// recipe rules 1-3: finite, then min <= l <= max on every axis (a NaN l fails)
__device__ __forceinline__ bool inside(const float4 &q, const CropBoxParams &b) {
  if (!(isfinite(q.x) && isfinite(q.y) && isfinite(q.z))) return false;
  bool in = true;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float l = affine_row(b.t + 4 * a, q);
    in = in && b.mn[a] <= l && l <= b.mx[a];
  }
  return in;
}

// point i of frame f is in the input and inside the box
struct InsideBox {
  CropBoxParams box;
  __device__ uint32_t operator()(const CloudSrc &in, uint32_t f, uint32_t i, uint32_t) const {
    return i < frame_count(in, f) && inside(__ldg(frame_points(in, f) + i), box);
  }
};

}  // namespace

size_t crop_box_scratch_bytes(uint32_t n_frames, uint32_t n_max) {
  return align_up(((size_t)n_frames * n_max + 1) * 4) + align_up(compaction_temp_bytes<InsideBox>(n_frames, n_max));
}

cudaError_t launch_crop_box(const CloudSrc &in, const CloudDst &out, const CropBoxParams &box, void *scratch,
                            cudaStream_t stream, int *launches) {
  if (launches) *launches = 0;
  if (in.n_frames == 0) return cudaSuccess;
  if ((uint64_t)in.n_frames * in.n_max > kCloudMaxPoints) return cudaErrorInvalidValue;  // the caller splits the batch
  if (in.n_max == 0) return cudaMemsetAsync(out.counts, 0, in.n_frames * sizeof(uint32_t), stream);
  uint32_t *slot = static_cast<uint32_t *>(scratch);
  void *temp = static_cast<uint8_t *>(scratch) + align_up(((size_t)in.n_frames * in.n_max + 1) * 4);
  const cudaError_t e = launch_compaction(in, InsideBox{box}, slot, temp,
                                          compaction_temp_bytes<InsideBox>(in.n_frames, in.n_max), out, stream);
  if (launches && e == cudaSuccess) *launches = 2;  // the scan (one CUB call counted once) and the scatter
  return e;
}

}  // namespace d2pc
