// pcl_order.cpp -- pcl::VoxelGrid<pcl::PointXYZ>::applyFilter as PCL 1.7.2 - 1.12 writes it (no limit field
// branch: tests call it without a limit), including its std::sort of (idx, point) pairs compared on idx alone.
// Test infrastructure: it shows what the library's stable summation order changes against PCL's own order.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <vector>

namespace {
struct cloud_point_index_idx {
  unsigned int idx;
  unsigned int cloud_point_index;
  cloud_point_index_idx(unsigned int idx_, unsigned int cloud_point_index_) : idx(idx_), cloud_point_index(cloud_point_index_) {}
  bool operator<(const cloud_point_index_idx &p) const { return (idx < p.idx); }
};
}  // namespace

extern "C" size_t d2pc_voxel_pcl_order(const float *cloud, size_t n, float leaf_x, float leaf_y, float leaf_z,
                                       uint32_t min_points_per_voxel, float *out, int *is_dense) {
  const float inverse_leaf_size[3] = {1.0f / leaf_x, 1.0f / leaf_y, 1.0f / leaf_z};
  // getMinMax3D (non-dense input: non-finite points skipped)
  float min_p[3] = {std::numeric_limits<float>::max(), std::numeric_limits<float>::max(),
                    std::numeric_limits<float>::max()};
  float max_p[3] = {-std::numeric_limits<float>::max(), -std::numeric_limits<float>::max(),
                    -std::numeric_limits<float>::max()};
  for (size_t i = 0; i < n; ++i) {
    const float *p = cloud + 4 * i;
    if (!std::isfinite(p[0]) || !std::isfinite(p[1]) || !std::isfinite(p[2])) continue;
    for (int a = 0; a < 3; ++a) min_p[a] = std::min(min_p[a], p[a]), max_p[a] = std::max(max_p[a], p[a]);
  }
  *is_dense = 1;
  std::int64_t dx = static_cast<std::int64_t>((max_p[0] - min_p[0]) * inverse_leaf_size[0]) + 1;
  std::int64_t dy = static_cast<std::int64_t>((max_p[1] - min_p[1]) * inverse_leaf_size[1]) + 1;
  std::int64_t dz = static_cast<std::int64_t>((max_p[2] - min_p[2]) * inverse_leaf_size[2]) + 1;
  if ((dx * dy * dz) > static_cast<std::int64_t>(std::numeric_limits<std::int32_t>::max())) {
    std::memcpy(out, cloud, n * 16);
    *is_dense = 0;
    return n;
  }
  int min_b[3], max_b[3], div_b[3], divb_mul[3];
  for (int a = 0; a < 3; ++a) {
    min_b[a] = static_cast<int>(std::floor(min_p[a] * inverse_leaf_size[a]));
    max_b[a] = static_cast<int>(std::floor(max_p[a] * inverse_leaf_size[a]));
    div_b[a] = max_b[a] - min_b[a] + 1;
  }
  divb_mul[0] = 1, divb_mul[1] = div_b[0], divb_mul[2] = div_b[0] * div_b[1];
  std::vector<cloud_point_index_idx> index_vector;
  index_vector.reserve(n);
  for (size_t i = 0; i < n; ++i) {
    const float *p = cloud + 4 * i;
    if (!std::isfinite(p[0]) || !std::isfinite(p[1]) || !std::isfinite(p[2])) continue;
    int ijk0 = static_cast<int>(std::floor(p[0] * inverse_leaf_size[0]) - static_cast<float>(min_b[0]));
    int ijk1 = static_cast<int>(std::floor(p[1] * inverse_leaf_size[1]) - static_cast<float>(min_b[1]));
    int ijk2 = static_cast<int>(std::floor(p[2] * inverse_leaf_size[2]) - static_cast<float>(min_b[2]));
    int idx = ijk0 * divb_mul[0] + ijk1 * divb_mul[1] + ijk2 * divb_mul[2];
    index_vector.push_back(cloud_point_index_idx(static_cast<unsigned int>(idx), static_cast<unsigned int>(i)));
  }
  std::sort(index_vector.begin(), index_vector.end(), std::less<cloud_point_index_idx>());
  unsigned int total = 0, index = 0;
  std::vector<std::pair<unsigned int, unsigned int>> first_and_last_indices_vector;
  while (index < index_vector.size()) {
    unsigned int i = index + 1;
    while (i < index_vector.size() && index_vector[i].idx == index_vector[index].idx) ++i;
    if (i - index >= min_points_per_voxel) {
      ++total;
      first_and_last_indices_vector.emplace_back(index, i);
    }
    index = i;
  }
  size_t o = 0;
  for (const auto &fl : first_and_last_indices_vector) {
    float centroid[3] = {0.0f, 0.0f, 0.0f};
    for (unsigned int li = fl.first; li < fl.second; ++li)
      for (int a = 0; a < 3; ++a) centroid[a] += cloud[4 * (size_t)index_vector[li].cloud_point_index + a];
    for (int a = 0; a < 3; ++a) centroid[a] /= static_cast<float>(fl.second - fl.first);
    float *q = out + 4 * o++;
    q[0] = centroid[0], q[1] = centroid[1], q[2] = centroid[2], q[3] = 1.0f;
  }
  return o;
}
