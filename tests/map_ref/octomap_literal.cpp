// octomap_literal.cpp -- OctomapServer::insertScan on an octomap::OcTree, restated literally from memory (test
// infrastructure, not product code; the octomap sources were not at hand).  octomath::Vector3 (float), OcTreeKey,
// KeyRay, OcTreeBaseImpl::coordToKeyChecked / keyToCoord / computeRayKeys, OccupancyOcTreeBase::updateNode with its
// early abort, over an unordered_map of full-depth leaves (no pruning), and the leaf iterator's order for the export.
// Compiled with -ffp-contract=off; no code is shared with the library.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <limits>
#include <unordered_map>
#include <unordered_set>
#include <vector>

namespace {

struct Vector3 {
  float data[3];
  Vector3() : data{0, 0, 0} {}
  Vector3(float x, float y, float z) : data{x, y, z} {}
  float &operator()(unsigned i) { return data[i]; }
  const float &operator()(unsigned i) const { return data[i]; }
  Vector3 operator-(const Vector3 &o) const { return Vector3(data[0] - o.data[0], data[1] - o.data[1], data[2] - o.data[2]); }
  Vector3 operator+(const Vector3 &o) const { return Vector3(data[0] + o.data[0], data[1] + o.data[1], data[2] + o.data[2]); }
  Vector3 operator*(float x) const { return Vector3(data[0] * x, data[1] * x, data[2] * x); }
  Vector3 &operator/=(float x) {
    for (int i = 0; i < 3; ++i) data[i] /= x;
    return *this;
  }
  double norm_sq() const { return (data[0] * data[0] + data[1] * data[1] + data[2] * data[2]); }
  double norm() const { return sqrt(norm_sq()); }
  Vector3 &normalize() {
    double len = norm();
    if (len > 0) *this /= (float)len;
    return *this;
  }
  Vector3 normalized() const {
    Vector3 r(*this);
    r.normalize();
    return r;
  }
};
typedef Vector3 point3d;

struct OcTreeKey {
  uint16_t k[3];
  bool operator==(const OcTreeKey &o) const { return k[0] == o.k[0] && k[1] == o.k[1] && k[2] == o.k[2]; }
  uint16_t &operator[](unsigned i) { return k[i]; }
  const uint16_t &operator[](unsigned i) const { return k[i]; }
  struct KeyHash {
    size_t operator()(const OcTreeKey &key) const {
      return (size_t)key.k[0] + 1447 * (size_t)key.k[1] + 345637 * (size_t)key.k[2];
    }
  };
};
typedef std::unordered_set<OcTreeKey, OcTreeKey::KeyHash> KeySet;
typedef std::vector<OcTreeKey> KeyRay;

float logodds(double p) { return (float)log(p / (1 - p)); }

struct OcTree {
  double resolution, resolution_factor;
  const unsigned tree_max_val = 32768;
  float prob_hit_log, prob_miss_log, clamping_thres_min, clamping_thres_max, occ_prob_thres_log;
  std::unordered_map<OcTreeKey, float, OcTreeKey::KeyHash> leaves;

  explicit OcTree(double res) : resolution(res), resolution_factor(1. / res) {}

  bool coordToKeyChecked(double coordinate, uint16_t &key) const {
    int scaledCoord = ((int)floor(resolution_factor * coordinate)) + tree_max_val;
    if ((scaledCoord >= 0) && (((unsigned int)scaledCoord) < (2 * tree_max_val))) {
      key = scaledCoord;
      return true;
    }
    return false;
  }
  bool coordToKeyChecked(const point3d &coord, OcTreeKey &key) const {
    for (unsigned i = 0; i < 3; ++i)
      if (!coordToKeyChecked(coord(i), key[i])) return false;
    return true;
  }
  double keyToCoord(uint16_t key) const { return (double((int)key - (int)tree_max_val) + 0.5) * resolution; }

  bool computeRayKeys(const point3d &origin, const point3d &end, KeyRay &ray) const {
    ray.clear();
    OcTreeKey key_origin, key_end;
    if (!coordToKeyChecked(origin, key_origin) || !coordToKeyChecked(end, key_end)) return false;
    if (key_origin == key_end) return true;
    ray.push_back(key_origin);
    point3d direction = (end - origin);
    float length = (float)direction.norm();
    direction /= length;
    int step[3];
    double tMax[3];
    double tDelta[3];
    OcTreeKey current_key = key_origin;
    for (unsigned int i = 0; i < 3; ++i) {
      if (direction(i) > 0.0) step[i] = 1;
      else if (direction(i) < 0.0) step[i] = -1;
      else step[i] = 0;
      if (step[i] != 0) {
        double voxelBorder = this->keyToCoord(current_key[i]);
        voxelBorder += (float)(step[i] * this->resolution * 0.5);
        tMax[i] = (voxelBorder - origin(i)) / direction(i);
        tDelta[i] = this->resolution / std::fabs(direction(i));
      } else {
        tMax[i] = std::numeric_limits<double>::max();
        tDelta[i] = std::numeric_limits<double>::max();
      }
    }
    bool done = false;
    unsigned guard = 0;  // the library's bound (csrc/map_math.h); octomap has none
    while (!done) {
      if (++guard > 3u * 65536u) break;
      unsigned int dim;
      if (tMax[0] < tMax[1]) {
        if (tMax[0] < tMax[2]) dim = 0;
        else dim = 2;
      } else {
        if (tMax[1] < tMax[2]) dim = 1;
        else dim = 2;
      }
      current_key[dim] += step[dim];
      tMax[dim] += tDelta[dim];
      if (current_key == key_end) {
        done = true;
        break;
      } else {
        double dist_from_origin = std::min(std::min(tMax[0], tMax[1]), tMax[2]);
        if (dist_from_origin > length) {
          done = true;
          break;
        } else {
          ray.push_back(current_key);
        }
      }
    }
    return true;
  }

  void updateNode(const OcTreeKey &key, bool occupied) {
    float log_odds_update = occupied ? prob_hit_log : prob_miss_log;
    auto it = leaves.find(key);
    if (it != leaves.end() && ((log_odds_update >= 0 && it->second >= clamping_thres_max) ||
                               (log_odds_update <= 0 && it->second <= clamping_thres_min)))
      return;
    float &v = it != leaves.end() ? it->second : (leaves[key] = 0.0f);
    v += log_odds_update;
    if (v < clamping_thres_min) {
      v = clamping_thres_min;
      return;
    }
    if (v > clamping_thres_max) v = clamping_thres_max;
  }

  // OctomapServer::insertScan with filter_ground off: every point is nonground
  void insertScan(const float *pts, size_t n, const point3d &sensorOrigin, double m_maxRange) {
    KeySet free_cells, occupied_cells;
    KeyRay keyRay;
    for (size_t i = 0; i < n; ++i) {
      const float *q = pts + 4 * i;
      if (!std::isfinite(q[0]) || !std::isfinite(q[1]) || !std::isfinite(q[2])) continue;
      point3d point(q[0], q[1], q[2]);
      if ((m_maxRange < 0.0) || ((point - sensorOrigin).norm() <= m_maxRange)) {
        if (computeRayKeys(sensorOrigin, point, keyRay)) free_cells.insert(keyRay.begin(), keyRay.end());
        OcTreeKey key;
        if (coordToKeyChecked(point, key)) occupied_cells.insert(key);
      } else {
        point3d new_end = sensorOrigin + (point - sensorOrigin).normalized() * m_maxRange;
        if (computeRayKeys(sensorOrigin, new_end, keyRay)) free_cells.insert(keyRay.begin(), keyRay.end());
      }
    }
    for (auto it = free_cells.begin(); it != free_cells.end(); ++it)
      if (occupied_cells.find(*it) == occupied_cells.end()) updateNode(*it, false);
    for (auto it = occupied_cells.begin(); it != occupied_cells.end(); ++it) updateNode(*it, true);
  }

  // the leaf iterator's order: depth first, child index (x | y << 1 | z << 2) of each level from the root down
  static bool leaf_order(const OcTreeKey &a, const OcTreeKey &b) {
    for (int d = 15; d >= 0; --d) {
      const unsigned ca = ((a[0] >> d) & 1) | (((a[1] >> d) & 1) << 1) | (((a[2] >> d) & 1) << 2);
      const unsigned cb = ((b[0] >> d) & 1) | (((b[1] >> d) & 1) << 1) | (((b[2] >> d) & 1) << 2);
      if (ca != cb) return ca < cb;
    }
    return false;
  }
  std::vector<OcTreeKey> sorted_keys() const {
    std::vector<OcTreeKey> keys;
    keys.reserve(leaves.size());
    for (const auto &kv : leaves) keys.push_back(kv.first);
    std::sort(keys.begin(), keys.end(), leaf_order);
    return keys;
  }
};

struct Handle {
  OcTree tree;
  double max_range;
  explicit Handle(double res) : tree(res), max_range(-1) {}
};

}  // namespace

extern "C" {

void *oct_new(double res) { return new Handle(res); }
void oct_free(void *h) { delete static_cast<Handle *>(h); }
void oct_clear(void *h) { static_cast<Handle *>(h)->tree.leaves.clear(); }
void oct_set_params(void *h, double hit, double miss, double cmin, double cmax, double thres, double max_range) {
  OcTree &t = static_cast<Handle *>(h)->tree;
  t.prob_hit_log = logodds(hit), t.prob_miss_log = logodds(miss);
  t.clamping_thres_min = logodds(cmin), t.clamping_thres_max = logodds(cmax);
  t.occ_prob_thres_log = logodds(thres);
  static_cast<Handle *>(h)->max_range = max_range;
}
float oct_logodds(double p) { return logodds(p); }
void oct_insert(void *h, const float *pts, size_t n, float ox, float oy, float oz) {
  Handle *H = static_cast<Handle *>(h);
  H->tree.insertScan(pts, n, point3d(ox, oy, oz), H->max_range);
}
// every leaf in leaf-iterator order: keys packed kx | ky << 16 | kz << 32, and the log-odds
size_t oct_voxels(void *h, uint64_t *keys, float *lo, size_t cap) {
  const OcTree &t = static_cast<Handle *>(h)->tree;
  const std::vector<OcTreeKey> ks = t.sorted_keys();
  for (size_t i = 0; i < ks.size() && i < cap; ++i) {
    keys[i] = (uint64_t)ks[i][0] | ((uint64_t)ks[i][1] << 16) | ((uint64_t)ks[i][2] << 32);
    lo[i] = t.leaves.at(ks[i]);
  }
  return ks.size();
}
// octomap_point_cloud_centers: PointXYZ {x, y, z, 1} of the occupied leaves in leaf-iterator order
size_t oct_centers(void *h, float *out, size_t cap) {
  const OcTree &t = static_cast<Handle *>(h)->tree;
  size_t n = 0;
  for (const OcTreeKey &k : t.sorted_keys()) {
    if (!(t.leaves.at(k) >= t.occ_prob_thres_log)) continue;
    if (n < cap) {
      out[4 * n] = (float)t.keyToCoord(k[0]), out[4 * n + 1] = (float)t.keyToCoord(k[1]);
      out[4 * n + 2] = (float)t.keyToCoord(k[2]), out[4 * n + 3] = 1.0f;
    }
    ++n;
  }
  return n;
}

// the same digest as tests/map_ref/occupancy.c's d2pc_map_rays_digest, from this restatement
void oct_rays_digest(const float *pairs, size_t n, double res, double max_range, uint64_t *out) {
  OcTree t(res);
  KeyRay ray;
  for (size_t i = 0; i < n; ++i) {
    const float *o = pairs + 6 * i, *p = pairs + 6 * i + 3;
    uint64_t count = 0, h = 0xcbf29ce484222325ull, occ = ~0ull;
    if (std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2])) {
      point3d origin(o[0], o[1], o[2]), point(p[0], p[1], p[2]);
      bool in_range = (max_range < 0.0) || ((point - origin).norm() <= max_range);
      point3d end = in_range ? point : origin + (point - origin).normalized() * max_range;
      if (t.computeRayKeys(origin, end, ray))
        for (const OcTreeKey &k : ray) {
          ++count;
          for (int a = 0; a < 3; ++a)
            for (int b = 0; b < 2; ++b) h = (h ^ ((k[a] >> (8 * b)) & 0xff)) * 0x100000001b3ull;
        }
      OcTreeKey key;
      if (in_range && t.coordToKeyChecked(point, key))
        occ = (uint64_t)key[0] | ((uint64_t)key[1] << 16) | ((uint64_t)key[2] << 32);
    }
    out[3 * i] = count, out[3 * i + 1] = h, out[3 * i + 2] = occ;
  }
}

}  // extern "C"
