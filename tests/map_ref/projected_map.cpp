// projected_map.cpp -- octomap_server's /projected_map restated literally from memory (test infrastructure, not product
// code; the octomap and octomap_server sources were not at hand): the leaf iterator's keys (computeChildKey), getX /
// getY / getZ (keyToCoord(key, depth)), getSize (getNodeSize) and getIndexKey (computeIndexKey); calcMinMax; and
// OctomapServer::publishAll's early return, handlePreNodeTraversal (incremental_2D_projection false, max depth 16), its
// leaf loop's height test and update2DMap, over the pointer tree of octree_pointer.cpp, included below.  Also an entry
// that builds that tree from (key, log-odds) pairs with setNodeValueRecurs, for maps too large to grow by insertScan.
// No code is shared with the library.
#include <cfloat>

#include "octree_pointer.cpp"

namespace {

struct Leaf {
  OcTreeKey key;  // the iterator's key: the node's centre key
  unsigned depth;
  const OcTreeNode *node;
};

struct Grid {
  uint32_t width = 0, height = 0;
  float resolution = 0;
  double origin_x = 0, origin_y = 0;
  std::vector<int8_t> data;
};
Grid g_grid;  // the last projection, until the next one

struct Projection {
  const PointerTree &tree;
  const unsigned tree_depth = 16, tree_max_val = 32768;
  double resolution, resolution_factor, sizeLookupTable[17];
  // OctomapServer's state
  double m_occupancyMinZ, m_occupancyMaxZ, m_minSizeX, m_minSizeY;
  OcTreeKey m_paddedMinKey;
  unsigned m_multires2DScale = 1;
  Grid &m_gridmap;

  Projection(const PointerTree &t, double res, Grid &grid) : tree(t), resolution(res), m_gridmap(grid) {
    resolution_factor = 1. / resolution;
    for (unsigned i = 0; i <= tree_depth; ++i) sizeLookupTable[i] = resolution * double(1 << (tree_depth - i));
  }

  double getNodeSize(unsigned depth) const { return sizeLookupTable[depth]; }
  double keyToCoord(uint16_t key) const { return (double((int)key - (int)this->tree_max_val) + 0.5) * this->resolution; }
  double keyToCoord(uint16_t key, unsigned depth) const {
    if (depth == 0) return 0.0;
    else if (depth == tree_depth) return keyToCoord(key);
    else return (floor((double(key) - double(this->tree_max_val)) / double(1 << (tree_depth - depth))) + 0.5) *
                this->getNodeSize(depth);
  }
  point3d keyToCoord(const OcTreeKey &key, unsigned depth) const {
    return point3d(float(keyToCoord(key[0], depth)), float(keyToCoord(key[1], depth)), float(keyToCoord(key[2], depth)));
  }
  bool coordToKeyChecked(double coordinate, unsigned depth, uint16_t &key) const {
    int scaledCoord = ((int)floor(resolution_factor * coordinate)) + tree_max_val;
    if ((scaledCoord >= 0) && (((unsigned int)scaledCoord) < (2 * tree_max_val))) {
      key = scaledCoord;
      (void)depth;  // adjustKeyAtDepth is the identity at depth 16
      return true;
    }
    return false;
  }
  bool coordToKeyChecked(const point3d &coord, unsigned depth, OcTreeKey &key) const {
    for (unsigned int i = 0; i < 3; i++)
      if (!coordToKeyChecked(coord(i), depth, key[i])) return false;
    return true;
  }
  static OcTreeKey computeIndexKey(unsigned level, const OcTreeKey &key) {
    if (level == 0) return key;
    const uint16_t mask = (uint16_t)(65535 << level);
    OcTreeKey result = key;
    result[0] &= mask, result[1] &= mask, result[2] &= mask;
    return result;
  }

  // the leaf iterator down to depth 16: depth first, children in index order, the root's key tree_max_val
  void leavesRecurs(const OcTreeNode *node, const OcTreeKey &key, unsigned depth, std::vector<Leaf> &out) const {
    if (depth == tree_depth || !tree.nodeHasChildren(node)) {
      out.push_back({key, depth, node});
      return;
    }
    const uint16_t center_offset_key = (uint16_t)(tree_max_val >> (depth + 1));
    for (unsigned i = 0; i < 8; ++i) {
      if (!tree.nodeChildExists(node, i)) continue;
      OcTreeKey child;  // computeChildKey
      for (unsigned a = 0; a < 3; ++a)
        child.k[a] = (i & (1u << a)) ? (uint16_t)(key.k[a] + center_offset_key)
                                     : (uint16_t)(key.k[a] - center_offset_key - (center_offset_key ? 0 : 1));
      leavesRecurs(tree.getNodeChild(node, i), child, depth + 1, out);
    }
  }
  std::vector<Leaf> leaves() const {
    std::vector<Leaf> out;
    OcTreeKey k;
    k.k[0] = k.k[1] = k.k[2] = (uint16_t)tree_max_val;
    if (tree.root) leavesRecurs(tree.root, k, 0, out);
    return out;
  }

  // OcTreeBaseImpl::calcMinMax over the leaves
  void calcMinMax(const std::vector<Leaf> &ls, double min_value[3], double max_value[3]) const {
    for (unsigned i = 0; i < 3; i++) {
      max_value[i] = -std::numeric_limits<double>::max();
      min_value[i] = std::numeric_limits<double>::max();
    }
    for (const Leaf &it : ls) {
      double size = getNodeSize(it.depth);
      double halfSize = size / 2.0;
      double x = keyToCoord(it.key[0], it.depth) - halfSize;
      double y = keyToCoord(it.key[1], it.depth) - halfSize;
      double z = keyToCoord(it.key[2], it.depth) - halfSize;
      if (x < min_value[0]) min_value[0] = x;
      if (y < min_value[1]) min_value[1] = y;
      if (z < min_value[2]) min_value[2] = z;
      x += size;
      y += size;
      z += size;
      if (x > max_value[0]) max_value[0] = x;
      if (y > max_value[1]) max_value[1] = y;
      if (z > max_value[2]) max_value[2] = z;
    }
  }

  // handlePreNodeTraversal with m_publish2DMap; false where octomap_server logs "Could not create padded ... key"
  bool handlePreNodeTraversal(const std::vector<Leaf> &ls) {
    double min_value[3], max_value[3];
    calcMinMax(ls, min_value, max_value);
    double minX = min_value[0], minY = min_value[1], minZ = min_value[2];
    double maxX = max_value[0], maxY = max_value[1], maxZ = max_value[2];
    double halfPaddedX = 0.5 * m_minSizeX;
    double halfPaddedY = 0.5 * m_minSizeY;
    minX = std::min(minX, -halfPaddedX);
    maxX = std::max(maxX, halfPaddedX);
    minY = std::min(minY, -halfPaddedY);
    maxY = std::max(maxY, halfPaddedY);
    point3d minPt(minX, minY, minZ);
    point3d maxPt(maxX, maxY, maxZ);
    OcTreeKey paddedMaxKey;
    if (!coordToKeyChecked(minPt, tree_depth, m_paddedMinKey)) return false;
    if (!coordToKeyChecked(maxPt, tree_depth, paddedMaxKey)) return false;
    m_gridmap.width = (paddedMaxKey[0] - m_paddedMinKey[0]) / m_multires2DScale + 1;
    m_gridmap.height = (paddedMaxKey[1] - m_paddedMinKey[1]) / m_multires2DScale + 1;
    point3d origin = keyToCoord(m_paddedMinKey, tree_depth);
    double gridRes = getNodeSize(tree_depth);
    m_gridmap.resolution = (float)gridRes;
    m_gridmap.origin_x = origin.data[0] - gridRes * 0.5;
    m_gridmap.origin_y = origin.data[1] - gridRes * 0.5;
    m_gridmap.data.clear();
    m_gridmap.data.resize((size_t)m_gridmap.width * m_gridmap.height, -1);
    return true;
  }

  // octomap_server's index is unsigned; size_t here, so a grid of 2^32 cells indexes too
  size_t mapIdx(int i, int j) const { return (size_t)m_gridmap.width * (size_t)j + (size_t)i; }
  void update2DMap(const Leaf &it, bool occupied) {
    if (it.depth == tree_depth) {
      size_t idx = mapIdx((it.key[0] - m_paddedMinKey[0]) / m_multires2DScale,
                          (it.key[1] - m_paddedMinKey[1]) / m_multires2DScale);
      if (occupied) m_gridmap.data[idx] = 100;
      else if (m_gridmap.data[idx] == -1) m_gridmap.data[idx] = 0;
    } else {
      int intSize = 1 << (tree_depth - it.depth);
      OcTreeKey minKey = computeIndexKey(tree_depth - it.depth, it.key);
      for (int dx = 0; dx < intSize; dx++) {
        int i = (minKey[0] + dx - m_paddedMinKey[0]) / m_multires2DScale;
        for (int dy = 0; dy < intSize; dy++) {
          size_t idx = mapIdx(i, (minKey[1] + dy - m_paddedMinKey[1]) / m_multires2DScale);
          if (occupied) m_gridmap.data[idx] = 100;
          else if (m_gridmap.data[idx] == -1) m_gridmap.data[idx] = 0;
        }
      }
    }
  }

  // publishAll's 2-D part: 1 nothing published (empty tree), 0 the grid, -3 no padded key
  int publishAll() {
    if (tree.tree_size <= 1) return 1;
    const std::vector<Leaf> ls = leaves();
    if (!handlePreNodeTraversal(ls)) return -3;
    for (const Leaf &it : ls) {
      double z = keyToCoord(it.key[2], it.depth);
      double half_size = getNodeSize(it.depth) / 2.0;
      if (z + half_size > m_occupancyMinZ && z - half_size < m_occupancyMaxZ)
        update2DMap(it, tree.isNodeOccupied(it.node));  // handleOccupiedNode / handleFreeNode
    }
    return 0;
  }
};

// OccupancyOcTreeBase::setNodeValueRecurs (lazy_eval false); setNodeValue's clamp is left out, so values set under
// any clamp setting go in as they are
OcTreeNode *setNodeValueRecurs(PointerTree &t, OcTreeNode *node, bool node_just_created, const OcTreeKey &key,
                               unsigned depth, float log_odds_value) {
  bool created_node = false;
  if (depth < t.tree_depth) {
    unsigned pos = PointerTree::computeChildIdx(key, t.tree_depth - 1 - depth);
    if (!t.nodeChildExists(node, pos)) {
      if (!t.nodeHasChildren(node) && !node_just_created) {
        t.expandNode(node);
      } else {
        t.createNodeChild(node, pos);
        created_node = true;
      }
    }
    OcTreeNode *retval = setNodeValueRecurs(t, t.getNodeChild(node, pos), created_node, key, depth + 1, log_odds_value);
    if (t.pruneNode(node)) retval = node;
    else t.updateOccupancyChildren(node);
    return retval;
  }
  node->setLogOdds(log_odds_value);
  return node;
}

}  // namespace

extern "C" {

// the tree of h becomes the one setNodeValue builds from n (packed key, log-odds) pairs, in their order
void ptr_set_values(void *h, const uint64_t *keys, const float *lo, size_t n) {
  PointerTree &t = static_cast<PtrHandle *>(h)->tree;
  t.clear();
  for (size_t i = 0; i < n; ++i) {
    OcTreeKey k;
    k.k[0] = (uint16_t)keys[i], k.k[1] = (uint16_t)(keys[i] >> 16), k.k[2] = (uint16_t)(keys[i] >> 32);
    bool createdRoot = false;
    if (!t.root) {
      t.root = new OcTreeNode();
      t.tree_size++;
      createdRoot = true;
    }
    setNodeValueRecurs(t, t.root, createdRoot, k, 0, lo[i]);
  }
}

// /projected_map of h's tree: 1 nothing published, 0 a grid (its size, resolution and origin; the cells by
// ptr_projected_cells), -3 no padded key
int ptr_projected_map(void *h, double min_z, double max_z, double min_x_size, double min_y_size, uint32_t *width,
                      uint32_t *height, float *res, double origin[2]) {
  PtrHandle *H = static_cast<PtrHandle *>(h);
  g_grid = Grid();
  Projection p(H->tree, H->scratch.resolution, g_grid);
  p.m_occupancyMinZ = min_z, p.m_occupancyMaxZ = max_z, p.m_minSizeX = min_x_size, p.m_minSizeY = min_y_size;
  const int rc = p.publishAll();
  *width = g_grid.width, *height = g_grid.height, *res = g_grid.resolution;
  origin[0] = g_grid.origin_x, origin[1] = g_grid.origin_y;
  return rc;
}
void ptr_projected_cells(int8_t *out) {
  if (!g_grid.data.empty()) std::memcpy(out, g_grid.data.data(), g_grid.data.size());
}

}  // extern "C"
