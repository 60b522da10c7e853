// pcl::transformPointCloud<pcl::PointXYZ, float> (common/impl/transforms.hpp, PCL 1.10 - 1.12) restated literally
// for an affine matrix and copy_all_fields true (test infrastructure, not product code; restated from memory, PCL's
// source was not at hand).  What it keeps:
//   - the output starts as a copy of the input cloud;
//   - is_dense: every point goes through the transformer; otherwise only points with finite x, y and z do, and the
//     others stay as copied;
//   - detail::Transformer<float>::se3 in two forms: the scalar template, ((m0*x + m1*y) + m2*z) + m3 per row (built
//     here with -ffp-contract=off, so without the FMAs a compiler may form), and the SSE2 specialisation, which
//     forms a row as x*c0 + (y*c1 + (z*c2 + c3)) from the matrix's columns with _mm_mul_ps / _mm_add_ps.
// The fourth word of a transformed point is written by neither form and stays as copied.
#include <cmath>
#include <cstddef>
#include <cstring>
#include <xmmintrin.h>

namespace {

struct PointXYZ {
  float x, y, z, pad;
};

void se3_scalar(const float m[12], const float *src, float *tgt) {
  tgt[0] = static_cast<float>(m[0] * src[0] + m[1] * src[1] + m[2] * src[2] + m[3]);
  tgt[1] = static_cast<float>(m[4] * src[0] + m[5] * src[1] + m[6] * src[2] + m[7]);
  tgt[2] = static_cast<float>(m[8] * src[0] + m[9] * src[1] + m[10] * src[2] + m[11]);
}

// the SSE2 Transformer keeps the matrix as four column registers c0..c3 (lane a = row a)
void se3_sse(const float m[12], const float *src, float *tgt) {
  const __m128 c0 = _mm_setr_ps(m[0], m[4], m[8], 0.0f), c1 = _mm_setr_ps(m[1], m[5], m[9], 0.0f);
  const __m128 c2 = _mm_setr_ps(m[2], m[6], m[10], 0.0f), c3 = _mm_setr_ps(m[3], m[7], m[11], 1.0f);
  __m128 p0 = _mm_mul_ps(_mm_set1_ps(src[0]), c0);
  __m128 p1 = _mm_mul_ps(_mm_set1_ps(src[1]), c1);
  __m128 p2 = _mm_mul_ps(_mm_set1_ps(src[2]), c2);
  __m128 r = _mm_add_ps(p0, _mm_add_ps(p1, _mm_add_ps(p2, c3)));
  float v[4];
  _mm_storeu_ps(v, r);
  tgt[0] = v[0], tgt[1] = v[1], tgt[2] = v[2];
}

template <void (*se3)(const float *, const float *, float *)>
void transform_point_cloud(const PointXYZ *cloud_in, size_t n, int is_dense, const float m[12], PointXYZ *cloud_out) {
  std::memcpy(cloud_out, cloud_in, n * sizeof(PointXYZ));  // cloud_out = cloud_in (copy_all_fields)
  if (is_dense) {
    for (size_t i = 0; i < n; ++i) se3(m, &cloud_in[i].x, &cloud_out[i].x);
  } else {
    for (size_t i = 0; i < n; ++i) {
      if (!std::isfinite(cloud_in[i].x) || !std::isfinite(cloud_in[i].y) || !std::isfinite(cloud_in[i].z)) continue;
      se3(m, &cloud_in[i].x, &cloud_out[i].x);
    }
  }
}

}  // namespace

extern "C" void d2pc_transform_pcl(const float *pts, size_t n, int is_dense, const float m[12], float *out) {
  transform_point_cloud<se3_scalar>(reinterpret_cast<const PointXYZ *>(pts), n, is_dense, m,
                                    reinterpret_cast<PointXYZ *>(out));
}

extern "C" void d2pc_transform_pcl_sse(const float *pts, size_t n, int is_dense, const float m[12], float *out) {
  transform_point_cloud<se3_sse>(reinterpret_cast<const PointXYZ *>(pts), n, is_dense, m,
                                 reinterpret_cast<PointXYZ *>(out));
}
