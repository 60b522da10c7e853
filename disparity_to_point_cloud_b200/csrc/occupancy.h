// occupancy.h -- host-side launcher interface of occupancy.cu: the device occupancy map (octomap_server's insertScan
// on a depth-16 OcTree, the recipe is in include/d2pc_b200.h) and its export.  Input is cloud_stage.cuh's.
#pragma once
#include "cloud_stage.cuh"

namespace d2pc {

// A hash of 8x8x8-voxel bricks, open addressing on the brick key (key >> 3 per axis, packed 16 bits per axis).  Slot s
// owns its brick's storage: 512 float log-odds, a 512-bit known mask and 512 epoch-tagged mark words, so a brick
// needs no allocator.  All of it lives in one device allocation (map_table_bytes / map_table_carve).
struct MapTable {
  unsigned long long *keys = nullptr;  // cap slots, kMapEmpty when free
  float *log_odds = nullptr;           // cap * 512
  uint32_t *known = nullptr;           // cap * 16 mask words: bit i of word w is voxel 32 w + i
  uint32_t *marks = nullptr;           // cap * 512: epoch * 4 + 3 (hit) or + 2 (miss), monotone within an epoch range
  uint32_t *slot_epoch = nullptr;      // cap: the last epoch that touched the slot
  uint32_t *touched = nullptr;         // cap: the slots touched in the current epoch
  uint32_t *ctr = nullptr;             // [0] bricks created, [1] overflow flag, [2] touched slots
  unsigned long long *frames = nullptr;  // [0] frames applied, [1] frames dropped (overflow)
  uint32_t cap = 0;         // slots: a power of two, at least 2 * max_bricks
  uint32_t max_bricks = 0;  // bricks a frame may bring the map to
};

constexpr unsigned long long kMapEmpty = ~0ull;

// One frame's update, decided on the host and carried by value into its launches.
struct MapUpdate {
  float origin[3];     // the sensor origin
  double res, rf;      // resolution and 1.0 / resolution
  double max_range;    // < 0: unlimited
  float hit, miss;     // log-odds updates
  float clamp_min, clamp_max;
  uint32_t epoch;      // 1 .. 2^30 - 1
};

// Slots of the table for max_bricks, and the bytes of its allocation (256-byte aligned parts).
uint32_t map_table_cap(uint32_t max_bricks);
size_t map_table_bytes(uint32_t max_bricks);
MapTable map_table_carve(uint8_t *base, uint32_t max_bricks);

// The empty map (keys, known masks, counters).  marks_too: also every mark and slot epoch (the epoch wrapped).
cudaError_t map_clear(const MapTable &t, bool marks_too, cudaStream_t stream);

// One frame into the map: mark (every point's ray and endpoint), apply (the touched slots; nothing on overflow) and
// finish (frame counters, flags cleared): three launches.  `in` holds exactly one frame.
cudaError_t launch_map_insert(const CloudSrc &in, const MapTable &t, const MapUpdate &u, int sm_count,
                              cudaStream_t stream, int *launches);

// Export.  map_count: the known voxels (occupied_only: those with log-odds >= occ_thres) into *d_n.  map_export:
// the same voxels sorted by Morton code into centres (float4 {x, y, z, 1}) or (packed key, log-odds); temp holds
// map_export_temp_bytes(n).
cudaError_t map_count(const MapTable &t, bool occupied_only, float occ_thres, uint32_t *d_n, cudaStream_t stream);
size_t map_export_temp_bytes(uint32_t n);
cudaError_t map_export(const MapTable &t, bool occupied_only, float occ_thres, double res, uint32_t n, void *temp,
                       uint32_t *d_pos, float4 *centres, unsigned long long *keys, float *log_odds,
                       cudaStream_t stream);
// The first step of map_export: the voxels gathered and sorted by Morton code inside temp (*morton, *vals).
cudaError_t map_sort(const MapTable &t, bool occupied_only, float occ_thres, uint32_t n, void *temp, uint32_t *d_pos,
                     const unsigned long long **morton, const uint32_t **vals, cudaStream_t stream);

// octomap_msgs/Octomap data of the n known voxels (> 0) in two steps on one temp of octomap_temp_bytes(n), both
// asynchronous on `stream`.  octomap_plan: sorts the voxels and places the tree's records (full: every written node,
// 5 bytes; binary: every written inner node, 2 bytes), their count into the host's *records.  octomap_emit, once
// *records is there: the stream into out, which holds octomap_out_bytes(records, binary), the data in its first
// records * 5 (or * 2) bytes.
size_t octomap_temp_bytes(uint32_t n);
cudaError_t octomap_plan(const MapTable &t, uint32_t n, bool binary, void *temp, uint32_t *d_pos,
                         unsigned long long *records, cudaStream_t stream);
size_t octomap_out_bytes(unsigned long long records, bool binary);
cudaError_t octomap_emit(const MapTable &t, uint32_t n, bool binary, float occ_thres, void *temp,
                         unsigned long long records, uint8_t *out, cudaStream_t stream);

// octomap_server's projected 2-D map of the n known voxels (> 0), on one temp of octomap_temp_bytes(n), in three
// steps.  projmap_extent (asynchronous on `stream`): sorts and levels the voxels as octomap_plan does and reads the
// tree's extent into the host's h_ext[6] through d_ext[6].  projmap_grid (host, once h_ext is there): the padded grid,
// false when a padded corner has no key.  projmap_fill (asynchronous): the grid's int8 cells into `cells`, which
// holds projmap_cells_bytes(g).
struct ProjGrid {
  uint16_t min_key[2];  // the padded min key on x and y: cell (0, 0)
  uint32_t width, height;
  double origin[2];     // OccupancyGrid's info.origin.position x and y
};
cudaError_t projmap_extent(const MapTable &t, uint32_t n, double res, void *temp, uint32_t *d_pos,
                           unsigned long long *d_ext, unsigned long long *h_ext, cudaStream_t stream);
bool projmap_grid(const unsigned long long ext[6], double res, double min_x_size, double min_y_size, ProjGrid *g);
size_t projmap_cells_bytes(const ProjGrid &g);
cudaError_t projmap_fill(const MapTable &t, uint32_t n, double res, double min_z, double max_z, float occ_thres,
                         void *temp, const ProjGrid &g, uint8_t *cells, cudaStream_t stream);

}  // namespace d2pc
