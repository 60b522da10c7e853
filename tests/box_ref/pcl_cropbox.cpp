// pcl::CropBox<pcl::PointXYZ>::applyFilter (PCL 1.8 - 1.12) restated literally for the case the library implements:
// setTransform only (rotation_ and translation_ zero, so PCL's inverse transform is the identity and is skipped),
// setNegative(false), keep_organized false, an input that is not dense (test infrastructure, not product code;
// restated from memory, PCL's source was not at hand).  What it keeps:
//   - the is_dense check: non-finite points are skipped;
//   - the identity shortcut: transformPoint is skipped when transform_.matrix().isIdentity(), Eigen's fuzzy test
//     (diagonal entries within prec of 1, the others at most prec in magnitude, prec = 1e-5 for float);
//   - pcl::transformPoint's order, ((m(i,0)*x + m(i,1)*y) + m(i,2)*z) + m(i,3) in float;
//   - the rejection test: outside when l < min or l > max on some axis (so a NaN l is kept).
#include <cmath>
#include <cstddef>
#include <cstring>

namespace {

struct PointXYZ {
  float x, y, z, pad;
};

// Eigen's MatrixBase::isIdentity(prec) on the 4x4 affine matrix whose last row is (0, 0, 0, 1)
bool is_identity(const float m[12]) {
  const float prec = 1e-5f;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 4; ++j) {
      const float v = m[4 * i + j];
      if (i == j) {
        if (!(std::fabs(v - 1.0f) <= prec * std::fmin(std::fabs(v), 1.0f))) return false;
      } else if (!(std::fabs(v) <= prec)) {
        return false;
      }
    }
  return true;
}

PointXYZ transform_point(const PointXYZ &p, const float m[12]) {
  PointXYZ r = p;
  r.x = static_cast<float>(m[0] * p.x + m[1] * p.y + m[2] * p.z + m[3]);
  r.y = static_cast<float>(m[4] * p.x + m[5] * p.y + m[6] * p.z + m[7]);
  r.z = static_cast<float>(m[8] * p.x + m[9] * p.y + m[10] * p.z + m[11]);
  return r;
}

}  // namespace

extern "C" size_t d2pc_box_pcl(const float *pts, size_t n, const float mn[3], const float mx[3], const float t[12],
                               float *out) {
  const PointXYZ *input = reinterpret_cast<const PointXYZ *>(pts);
  const bool transform_matrix_is_identity = is_identity(t);
  size_t k = 0;
  for (size_t index = 0; index < n; ++index) {
    const PointXYZ &q = input[index];
    if (!(std::isfinite(q.x) && std::isfinite(q.y) && std::isfinite(q.z))) continue;
    PointXYZ local_pt = q;
    if (!transform_matrix_is_identity) local_pt = transform_point(local_pt, t);
    if ((local_pt.x < mn[0] || local_pt.y < mn[1] || local_pt.z < mn[2]) ||
        (local_pt.x > mx[0] || local_pt.y > mx[1] || local_pt.z > mx[2]))
      continue;
    std::memcpy(out + 4 * k++, &q, 16);
  }
  return k;
}
