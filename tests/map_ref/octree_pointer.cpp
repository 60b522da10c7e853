// octree_pointer.cpp -- octomap's pointer OcTree restated literally from memory (test infrastructure, not product
// code; the octomap sources were not at hand): OcTreeNode with a child array, OcTreeBaseImpl::search,
// OccupancyOcTreeBase::updateNode with its early abort and updateNodeRecurs (lazy_eval false: createNodeChild,
// expandNode, pruneNode / isNodeCollapsible, updateOccupancyChildren), and the serializers OcTree::writeData
// (writeNodesRecurs), writeBinaryData (writeBinaryNode) and readData (readNodesRecurs).  Each frame is driven by the
// very insertScan of octomap_literal.cpp, included below: it runs on a scratch flat map whose leaves then hold +1 for
// the frame's occupied keys and -1 for its free ones, which this tree receives as updateNode calls in insertScan's
// order (free, then occupied).  No code is shared with the library.
#include <cstring>
#include <string>

#include "octomap_literal.cpp"

namespace {

struct OcTreeNode {
  float value = 0.0f;
  OcTreeNode **children = nullptr;
  float getLogOdds() const { return value; }
  void setLogOdds(float v) { value = v; }
  void addValue(float v) { value += v; }
  void copyData(const OcTreeNode &o) { value = o.value; }
  bool operator==(const OcTreeNode &o) const { return value == o.value; }
  float getMaxChildLogOdds() const {
    float mx = -std::numeric_limits<float>::max();
    if (children)
      for (unsigned i = 0; i < 8; ++i)
        if (children[i] && children[i]->getLogOdds() > mx) mx = children[i]->getLogOdds();
    return mx;
  }
};

struct PointerTree {
  const unsigned tree_depth = 16;
  OcTreeNode *root = nullptr;
  size_t tree_size = 0;
  float prob_hit_log = 0, prob_miss_log = 0, clamping_thres_min = 0, clamping_thres_max = 0, occ_prob_thres_log = 0;

  ~PointerTree() { clear(); }
  void deleteNodeRecurs(OcTreeNode *node) {
    if (node->children) {
      for (unsigned i = 0; i < 8; ++i)
        if (node->children[i]) deleteNodeRecurs(node->children[i]);
      delete[] node->children;
    }
    delete node;
  }
  void clear() {
    if (root) deleteNodeRecurs(root);
    root = nullptr;
    tree_size = 0;
  }

  static unsigned computeChildIdx(const OcTreeKey &key, int depth) {
    unsigned pos = 0;
    if (key.k[0] & (1 << depth)) pos += 1;
    if (key.k[1] & (1 << depth)) pos += 2;
    if (key.k[2] & (1 << depth)) pos += 4;
    return pos;
  }
  bool nodeChildExists(const OcTreeNode *node, unsigned i) const { return node->children && node->children[i]; }
  bool nodeHasChildren(const OcTreeNode *node) const {
    if (!node->children) return false;
    for (unsigned i = 0; i < 8; ++i)
      if (node->children[i]) return true;
    return false;
  }
  OcTreeNode *getNodeChild(OcTreeNode *node, unsigned i) const { return node->children[i]; }
  const OcTreeNode *getNodeChild(const OcTreeNode *node, unsigned i) const { return node->children[i]; }
  void allocNodeChildren(OcTreeNode *node) {
    node->children = new OcTreeNode *[8];
    for (unsigned i = 0; i < 8; ++i) node->children[i] = nullptr;
  }
  OcTreeNode *createNodeChild(OcTreeNode *node, unsigned i) {
    if (!node->children) allocNodeChildren(node);
    node->children[i] = new OcTreeNode();
    tree_size++;
    return node->children[i];
  }
  void deleteNodeChild(OcTreeNode *node, unsigned i) {
    deleteNodeRecurs(node->children[i]);
    node->children[i] = nullptr;
    tree_size--;
  }
  void expandNode(OcTreeNode *node) {
    for (unsigned k = 0; k < 8; ++k) {
      OcTreeNode *newNode = createNodeChild(node, k);
      newNode->copyData(*node);
    }
  }
  bool isNodeCollapsible(const OcTreeNode *node) const {
    if (!nodeChildExists(node, 0)) return false;
    const OcTreeNode *firstChild = getNodeChild(node, 0);
    if (nodeHasChildren(firstChild)) return false;
    for (unsigned i = 1; i < 8; ++i)
      if (!nodeChildExists(node, i) || nodeHasChildren(getNodeChild(node, i)) || !(*getNodeChild(node, i) == *firstChild))
        return false;
    return true;
  }
  bool pruneNode(OcTreeNode *node) {
    if (!isNodeCollapsible(node)) return false;
    node->copyData(*getNodeChild(node, 0));
    for (unsigned i = 0; i < 8; ++i) deleteNodeChild(node, i);
    delete[] node->children;
    node->children = nullptr;
    return true;
  }
  void updateOccupancyChildren(OcTreeNode *node) { node->setLogOdds(node->getMaxChildLogOdds()); }

  OcTreeNode *search(const OcTreeKey &key) const {
    if (!root) return nullptr;
    OcTreeNode *curNode = root;
    for (int i = (int)tree_depth - 1; i >= 0; --i) {
      const unsigned pos = computeChildIdx(key, i);
      if (nodeChildExists(curNode, pos)) {
        curNode = getNodeChild(curNode, pos);
      } else {
        if (!nodeHasChildren(curNode)) return curNode;  // a pruned leaf holds the key
        return nullptr;
      }
    }
    return curNode;
  }

  void updateNodeLogOdds(OcTreeNode *node, const float &update) const {
    node->addValue(update);
    if (node->getLogOdds() < clamping_thres_min) {
      node->setLogOdds(clamping_thres_min);
      return;
    }
    if (node->getLogOdds() > clamping_thres_max) node->setLogOdds(clamping_thres_max);
  }

  OcTreeNode *updateNodeRecurs(OcTreeNode *node, bool node_just_created, const OcTreeKey &key, unsigned depth,
                               const float &log_odds_update) {
    bool created_node = false;
    if (depth < tree_depth) {
      const unsigned pos = computeChildIdx(key, tree_depth - 1 - depth);
      if (!nodeChildExists(node, pos)) {
        if (!nodeHasChildren(node) && !node_just_created) {
          expandNode(node);  // a pruned node
        } else {
          createNodeChild(node, pos);
          created_node = true;
        }
      }
      OcTreeNode *retval = updateNodeRecurs(getNodeChild(node, pos), created_node, key, depth + 1, log_odds_update);
      if (pruneNode(node)) {
        retval = node;
      } else {
        updateOccupancyChildren(node);
      }
      return retval;
    }
    updateNodeLogOdds(node, log_odds_update);
    return node;
  }

  OcTreeNode *updateNode(const OcTreeKey &key, float log_odds_update) {
    OcTreeNode *leaf = search(key);
    if (leaf && ((log_odds_update >= 0 && leaf->getLogOdds() >= clamping_thres_max) ||
                 (log_odds_update <= 0 && leaf->getLogOdds() <= clamping_thres_min)))
      return leaf;
    bool createdRoot = false;
    if (!root) {
      root = new OcTreeNode();
      tree_size++;
      createdRoot = true;
    }
    return updateNodeRecurs(root, createdRoot, key, 0, log_odds_update);
  }
  OcTreeNode *updateNode(const OcTreeKey &key, bool occupied) {
    return updateNode(key, occupied ? prob_hit_log : prob_miss_log);
  }

  bool isNodeOccupied(const OcTreeNode *node) const { return node->getLogOdds() >= occ_prob_thres_log; }

  // OcTree::writeData -> writeNodesRecurs
  void writeNodesRecurs(const OcTreeNode *node, std::string &s) const {
    s.append(reinterpret_cast<const char *>(&node->value), sizeof(node->value));
    unsigned char children = 0;  // std::bitset<8>
    for (unsigned i = 0; i < 8; ++i)
      if (nodeChildExists(node, i)) children |= (unsigned char)(1u << i);
    s.push_back((char)children);
    for (unsigned i = 0; i < 8; ++i)
      if (nodeChildExists(node, i)) writeNodesRecurs(getNodeChild(node, i), s);
  }
  void writeData(std::string &s) const {
    if (root) writeNodesRecurs(root, s);
  }

  // writeBinaryData -> writeBinaryNode
  void writeBinaryNode(const OcTreeNode *node, std::string &s) const {
    unsigned char child1to4 = 0, child5to8 = 0;  // std::bitset<8> each
    for (unsigned i = 0; i < 8; ++i) {
      unsigned char &b = i < 4 ? child1to4 : child5to8;
      const unsigned j = i % 4;
      if (nodeChildExists(node, i)) {
        const OcTreeNode *child = getNodeChild(node, i);
        if (nodeHasChildren(child)) {
          b |= (unsigned char)(1u << (2 * j)), b |= (unsigned char)(1u << (2 * j + 1));
        } else if (isNodeOccupied(child)) {
          b |= (unsigned char)(1u << (2 * j + 1));
        } else {
          b |= (unsigned char)(1u << (2 * j));
        }
      }
    }
    s.push_back((char)child1to4);
    s.push_back((char)child5to8);
    for (unsigned i = 0; i < 8; ++i)
      if (nodeChildExists(node, i) && nodeHasChildren(getNodeChild(node, i))) writeBinaryNode(getNodeChild(node, i), s);
  }
  void writeBinaryData(std::string &s) const {
    if (root) writeBinaryNode(root, s);
  }

  // OcTree::readData -> readNodesRecurs
  const unsigned char *readNodesRecurs(OcTreeNode *node, const unsigned char *p) {
    std::memcpy(&node->value, p, sizeof(node->value));
    p += sizeof(node->value);
    const unsigned char children = *p++;
    for (unsigned i = 0; i < 8; ++i)
      if ((children >> i) & 1u) p = readNodesRecurs(createNodeChild(node, i), p);
    return p;
  }
  size_t readData(const unsigned char *p, size_t n) {
    clear();
    if (n == 0) return 0;
    root = new OcTreeNode();
    tree_size++;
    return (size_t)(readNodesRecurs(root, p) - p);
  }

  // every full-depth voxel under the leaves, in pre-order (children in index order)
  void expandRecurs(const OcTreeNode *node, unsigned depth, const OcTreeKey &key, std::vector<uint64_t> &keys,
                    std::vector<float> &lo, unsigned *leaf_depths) const {
    if (!nodeHasChildren(node)) {
      if (leaf_depths) ++leaf_depths[depth];
      const unsigned span = 1u << (tree_depth - depth);
      for (unsigned long long i = 0; i < (unsigned long long)span * span * span; ++i) {
        OcTreeKey k = key;
        for (unsigned b = 0; b < tree_depth - depth; ++b) {
          k.k[0] |= (uint16_t)(((i >> (3 * b)) & 1) << b);
          k.k[1] |= (uint16_t)(((i >> (3 * b + 1)) & 1) << b);
          k.k[2] |= (uint16_t)(((i >> (3 * b + 2)) & 1) << b);
        }
        keys.push_back((uint64_t)k.k[0] | ((uint64_t)k.k[1] << 16) | ((uint64_t)k.k[2] << 32));
        lo.push_back(node->getLogOdds());
      }
      return;
    }
    for (unsigned i = 0; i < 8; ++i) {
      if (!nodeChildExists(node, i)) continue;
      OcTreeKey k = key;
      const unsigned bit = tree_depth - 1 - depth;
      if (i & 1) k.k[0] |= (uint16_t)(1u << bit);
      if (i & 2) k.k[1] |= (uint16_t)(1u << bit);
      if (i & 4) k.k[2] |= (uint16_t)(1u << bit);
      expandRecurs(getNodeChild(node, i), depth + 1, k, keys, lo, leaf_depths);
    }
  }
  void expand(std::vector<uint64_t> &keys, std::vector<float> &lo, unsigned *leaf_depths) const {
    keys.clear(), lo.clear();
    if (!root) return;
    OcTreeKey k;
    k.k[0] = k.k[1] = k.k[2] = 0;
    expandRecurs(root, 0, k, keys, lo, leaf_depths);
  }
};

struct PtrHandle {
  PointerTree tree;
  OcTree scratch;  // octomap_literal.cpp's map, for its insertScan
  double max_range = -1;
  std::string out;
  explicit PtrHandle(double res) : scratch(res) {
    scratch.prob_hit_log = 1.0f, scratch.prob_miss_log = -1.0f;
    scratch.clamping_thres_min = -10.0f, scratch.clamping_thres_max = 10.0f;
  }
};

size_t copy_out(const std::vector<uint64_t> &keys, const std::vector<float> &lo, uint64_t *k, float *v, size_t cap) {
  for (size_t i = 0; i < keys.size() && i < cap; ++i) k[i] = keys[i], v[i] = lo[i];
  return keys.size();
}

}  // namespace

extern "C" {

void *ptr_new(double res) { return new PtrHandle(res); }
void ptr_free(void *h) { delete static_cast<PtrHandle *>(h); }
void ptr_clear(void *h) { static_cast<PtrHandle *>(h)->tree.clear(); }
void ptr_set_params(void *h, double hit, double miss, double cmin, double cmax, double thres, double max_range) {
  PointerTree &t = static_cast<PtrHandle *>(h)->tree;
  t.prob_hit_log = logodds(hit), t.prob_miss_log = logodds(miss);
  t.clamping_thres_min = logodds(cmin), t.clamping_thres_max = logodds(cmax);
  t.occ_prob_thres_log = logodds(thres);
  static_cast<PtrHandle *>(h)->max_range = max_range;
}
void ptr_insert(void *h, const float *pts, size_t n, float ox, float oy, float oz) {
  PtrHandle *H = static_cast<PtrHandle *>(h);
  H->scratch.leaves.clear();
  H->scratch.insertScan(pts, n, point3d(ox, oy, oz), H->max_range);
  for (int pass = 0; pass < 2; ++pass)  // insertScan's order: the free cells, then the occupied ones
    for (const auto &kv : H->scratch.leaves)
      if ((kv.second > 0.0f) == (pass == 1)) H->tree.updateNode(kv.first, pass == 1);
}
// one updateNode(key, occupied) call
void ptr_update(void *h, uint16_t kx, uint16_t ky, uint16_t kz, int occupied) {
  OcTreeKey k;
  k.k[0] = kx, k.k[1] = ky, k.k[2] = kz;
  static_cast<PtrHandle *>(h)->tree.updateNode(k, occupied != 0);
}
// writeData (binary 0) or writeBinaryData (binary 1); the bytes stay valid until the next call on h
size_t ptr_write(void *h, int binary, const char **data) {
  PtrHandle *H = static_cast<PtrHandle *>(h);
  H->out.clear();
  if (binary) H->tree.writeBinaryData(H->out);
  else H->tree.writeData(H->out);
  *data = H->out.data();
  return H->out.size();
}
// the tree expanded to full-depth voxels (packed keys, log-odds) in pre-order; leaf_depths[d]: leaves at depth d
size_t ptr_voxels(void *h, uint64_t *keys, float *lo, size_t cap, unsigned *leaf_depths) {
  std::vector<uint64_t> k;
  std::vector<float> v;
  static_cast<PtrHandle *>(h)->tree.expand(k, v, leaf_depths);
  return copy_out(k, v, keys, lo, cap);
}
// readData of a full stream into h's tree (replacing it)
void ptr_load_full(void *h, const unsigned char *data, size_t n) { static_cast<PtrHandle *>(h)->tree.readData(data, n); }
size_t ptr_tree_size(void *h) { return static_cast<PtrHandle *>(h)->tree.tree_size; }
// readData of a full stream into a fresh tree, expanded like ptr_voxels; *used: the bytes read
size_t ptr_read_full(const unsigned char *data, size_t n, uint64_t *keys, float *lo, size_t cap, size_t *used) {
  PointerTree t;
  *used = t.readData(data, n);
  std::vector<uint64_t> k;
  std::vector<float> v;
  t.expand(k, v, nullptr);
  return copy_out(k, v, keys, lo, cap);
}

}  // extern "C"
