// pcl_branches.cpp -- the two branches of pcl::RadiusOutlierRemoval<PointXYZ>::applyFilterIndices (PCL 1.8 - 1.12,
// negative_ false), restated literally with exhaustive search in place of the kd-tree (test infrastructure, not
// product code; restated from memory, PCL's source was not at hand).  Distances are FLANN's L2_Simple<float>.
//
//   is_dense input: k = nearestKSearch(p, min + 1); kept when k == min + 1 and nn_dists[k - 1] <= r * r (double).
//   otherwise:      k = radiusSearch(p, r) over the finite points, FLANN testing dist < (float)(r * r); kept when
//                   k > min.  A non-finite query point finds nothing (k = 0) and is dropped.
// Both return the kept points in input order.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

namespace {

bool finite3(const float *p) { return std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]); }

float dist2(const float *a, const float *b) {
  const float dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];
  return (dx * dx + dy * dy) + dz * dz;
}

size_t emit(const float *cloud, size_t n, const std::vector<char> &keep, float *out) {
  size_t k = 0;
  for (size_t i = 0; i < n; ++i)
    if (keep[i]) std::memcpy(out + 4 * k++, cloud + 4 * i, 16);
  return k;
}

}  // namespace

extern "C" size_t d2pc_ror_pcl_knn(const float *cloud, size_t n, double radius, uint32_t min_neighbors, float *out) {
  const size_t mean_k = (size_t)min_neighbors + 1;
  const double nn_dists_max = radius * radius;
  std::vector<char> keep(n, 0);
  std::vector<float> d;
  for (size_t i = 0; i < n; ++i) {
    const float *p = cloud + 4 * i;
    if (!finite3(p)) continue;  // an is_dense cloud has none; the kd-tree never indexes one
    d.clear();
    for (size_t j = 0; j < n; ++j)
      if (finite3(cloud + 4 * j)) d.push_back(dist2(p, cloud + 4 * j));
    const size_t k = std::min(mean_k, d.size());
    std::partial_sort(d.begin(), d.begin() + k, d.end());
    keep[i] = k == mean_k && !(d[k - 1] > nn_dists_max);
  }
  return emit(cloud, n, keep, out);
}

extern "C" size_t d2pc_ror_pcl_radius(const float *cloud, size_t n, double radius, uint32_t min_neighbors,
                                      float *out) {
  const float r2 = static_cast<float>(radius * radius);
  std::vector<char> keep(n, 0);
  for (size_t i = 0; i < n; ++i) {
    const float *p = cloud + 4 * i;
    if (!finite3(p)) continue;
    uint64_t k = 0;
    for (size_t j = 0; j < n; ++j)
      if (finite3(cloud + 4 * j) && dist2(p, cloud + 4 * j) < r2) ++k;
    keep[i] = k > min_neighbors;
  }
  return emit(cloud, n, keep, out);
}
