// reproject.h -- host-side launcher interface of reproject.cu
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <cuda_runtime.h>

namespace d2pc {

// Q as the kernels consume it (travels in the kernel parameter bank).
struct QParams {
  double q[16];  // row-major 4x4, as given
  // rectified-form constants (valid when rectified != 0)
  double q03, q13, q32, q33;
  double zd;     // (double)(float)((+0.0) + q23)
  float qf[16];  // float32 copy of Q for FAST mode
  float zinf;    // zd / (+0): +-inf, or the x86 NaN when zd == 0
  uint32_t dhi_bits;  // float bits of 2^64 / |q32|: larger disparities leave the straight-line path
  int rectified;
  int q33_zero;
  int zd_slow;   // zd is +-0 / inf / NaN: the straight-line path must not be used
};

struct ReprojectLaunch {
  const void *in = nullptr;  // device: frames of float32 or mono8 rows
  bool in_is_f32 = true;
  size_t step = 0, frame_stride = 0;
  uint32_t n_frames = 0, width = 0, height = 0;
  int border = 40;
  float scale = 0.125f;      // mono8 only (cpp:61)
  uint8_t *out = nullptr;    // device: points, frame f at out + f*out_stride_bytes
  size_t out_stride_bytes = 0;
  uint32_t *counts = nullptr;  // device, per frame (CROP_FINITE)
  const QParams *Q = nullptr;  // host copy; travels in the kernel parameter bank
  bool arith_fast = false;
  bool compact = false;        // CROP_FINITE
  // compaction scratch (device): tile descriptors, ticket counter, launch epoch
  void *scratch = nullptr;
  void *tables = nullptr;      // reproject_table_bytes(width, height)
  uint32_t *ticket = nullptr;
  uint32_t epoch = 1;
  int sm_count = 148;
  // tuning / test knobs (0 = automatic)
  int rows_per_unit = 0;
  int ctas_per_sm = 0;
  bool force_scalar = false;   // exercise the unaligned load path
  bool force_generic = false;  // exercise the generic-Q exact path on a rectified Q
  int exact_variant = 0;       // rectified exact quotients: 0 = guarded multiply (7 FP64 ops), 1 = Markstein (15)
  int zero_numer = 0;          // zero-numerator columns straight-line: 0 = when Q has one in the image, 1 always, -1 never
  int compact_variant = 0;     // CROP_FINITE kernel: 0 = automatic (band where Q allows, else park),
                               // 1 = park-then-compact for every Q (test hook for the fallback)
  int prefetch_dist = 0;       // L2 prefetch distance: CROP kernel in work units, band kernel in tiles
                               // (0 = automatic, < 0 = off)
  int crop_load = 0;           // CROP kernel input: 0 = TMA boxes where the rows allow, 1 = per-row LDG always
  bool crop_probe = false;     // CROP kernel stores {d, d, d, 1} without arithmetic (traffic probe, f32 only)
};

void make_qparams(const double q[16], QParams *out);
size_t reproject_scratch_bytes(uint32_t n_frames, uint32_t width, uint32_t height, int border);
size_t reproject_table_bytes(uint32_t width, uint32_t height);
cudaError_t launch_reproject(const ReprojectLaunch &L, cudaStream_t stream, int *launches);
// True when this launch would run the plain CROP kernel with the rectified guarded-multiply arithmetic (with or
// without a zero-numerator column) -- the case median.cu's fused DisparityCb kernel implements.
bool reproject_fuses_with_median(const ReprojectLaunch &L, bool *zero_numer);

}  // namespace d2pc
