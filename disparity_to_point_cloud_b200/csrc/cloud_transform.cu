// cloud_transform.cu -- pcl::transformPointCloud<pcl::PointXYZ> with an affine matrix on the device, batched over
// frames: the first cloud stage behind the reproject kernels when a transform is enabled, and
// d2pc_cloud_transform_device.  include/d2pc_b200.h states the recipe.
//
// A streaming map: one thread per point, one 16-byte load and one 16-byte store with the streaming cache hint (the
// cloud is read once and not again by this kernel), nine rounded multiplies and nine rounded adds per finite point
// (cloud_stage.cuh's affine_row, the crop box's rows).  The frame number is in blockIdx.x, so a launch takes any number
// of frames.  The point count and order are unchanged, so the stage needs no scan and no scratch.
#include "cloud_transform.h"

namespace d2pc {
namespace {

// A NaN the arithmetic makes (inf + -inf after an overflow) as x86's default NaN 0xFFC00000, which is what PCL
// writes on x86-64 (the GPU's own is 0x7FFFFFFF); every other value passes unchanged.
__device__ __forceinline__ float x86_nan(float v) { return v == v ? v : __int_as_float(0xffc00000); }

// grid bpf * n_frames blocks, frame f's bpf blocks consecutive
__global__ void __launch_bounds__(kStageThreads) cloud_transform_kernel(const CloudSrc in, uint32_t bpf,
                                                                        const CloudTransformParams t,
                                                                        const float *__restrict__ per_frame,
                                                                        const CloudDst out) {
  __shared__ float m[12];
  const uint32_t f = blockIdx.x / bpf, i = (blockIdx.x - f * bpf) * kStageThreads + threadIdx.x;
  if (threadIdx.x < 12) m[threadIdx.x] = per_frame ? __ldg(per_frame + 12 * (size_t)f + threadIdx.x) : t.m[threadIdx.x];
  __syncthreads();
  const uint32_t n = frame_count(in, f);
  if (i == 0 && out.counts) out.counts[f] = n;
  if (i >= n) return;
  const float4 q = __ldcs(frame_points(in, f) + i);
  float4 r = q;  // rules 2-3: a point with a non-finite coordinate, and every w, are copied as they are
  if (isfinite(q.x) && isfinite(q.y) && isfinite(q.z))
    r.x = x86_nan(affine_row(m, q)), r.y = x86_nan(affine_row(m + 4, q)), r.z = x86_nan(affine_row(m + 8, q));
  __stcs(reinterpret_cast<float4 *>(out.points + (size_t)f * out.stride) + i, r);
}

}  // namespace

cudaError_t launch_cloud_transform(const CloudSrc &in, const CloudDst &out, const CloudTransformParams &t,
                                   const float *per_frame, cudaStream_t stream, int *launches) {
  if (launches) *launches = 0;
  if (in.n_frames == 0) return cudaSuccess;
  if ((uint64_t)in.n_frames * in.n_max > kCloudMaxPoints) return cudaErrorInvalidValue;  // the caller splits the batch
  if (in.n_max == 0)
    return out.counts ? cudaMemsetAsync(out.counts, 0, in.n_frames * sizeof(uint32_t), stream) : cudaSuccess;
  const uint32_t bpf = (in.n_max + kStageThreads - 1) / kStageThreads;
  cloud_transform_kernel<<<bpf * in.n_frames, kStageThreads, 0, stream>>>(in, bpf, t, per_frame, out);
  const cudaError_t e = cudaGetLastError();
  if (launches && e == cudaSuccess) *launches = 1;
  return e;
}

}  // namespace d2pc
