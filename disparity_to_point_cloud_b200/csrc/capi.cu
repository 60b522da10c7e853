// capi.cu -- the C ABI of include/d2pc_b200.h: contexts, pinned / device buffers,
// the three-stream slot pipeline (H2D | kernels | D2H) and the entry points.
//
// Host-side replacement of the body of Disparity2PCloud::DisparityCb
// (src/disparity_to_point_cloud.cpp:46-92) and of
// DepthMapFusion::publishFusedDepthMap (src/depth_map_fusion.cpp:103-136):
// what used to be six full-frame passes through OpenCV / PCL temporaries is
// H2D -> [median] -> reproject+crop+pack -> D2H.
//
// No CPU fallback exists in this file: every compute entry point either runs
// the CUDA kernels or returns an error.
#include "../../include/d2pc_b200.h"

#include <algorithm>
#include <atomic>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include <nvtx3/nvToolsExt.h>
#include <sys/mman.h>

#include "cloud_transform.h"
#include "crop_box.h"
#include "fusion.h"
#include "laser_scan.h"
#include "median.h"
#include "occupancy.h"
#include "radius_outlier.h"
#include "reproject.h"
#include "score.h"
#include "voxel.h"

using namespace d2pc;

namespace {

constexpr size_t kAlign = 256;
inline size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct DevBuf {
  uint8_t *p = nullptr;
  size_t cap = 0;
};
struct PinBuf {
  uint8_t *p = nullptr;
  size_t cap = 0;
};

// The filter stages that run on clouds already on the device (cloud_stage.cuh), in the order a plan runs them.
enum class CloudStage { transform, box, voxel, ror };

// The laser scan of a plan (d2pc_set_laser_scan), derived once per setting and carried by value into each submission.
struct ScanPlan {
  bool on = false;
  bool keep_cloud = true;  // false: only the ranges leave the device
  LaserScanParams p{};
  d2pc_laser_scan msg{};   // the message fields (ranges unset)
};

// The occupancy map update of a plan (d2pc_set_occupancy): the setting and the sensor origin in force at submission,
// carried by value (the epoch is given when the step is enqueued).
struct MapPlan {
  bool on = false;
  bool keep_cloud = true;  // false: the cloud stays on the device
  MapUpdate u{};
};

// What the filter mode, the cloud transform, the crop box and the radius outlier stage make of one frame geometry
// (plan_cloud), decided once per call.
struct CloudPlan {
  uint64_t n = 0;           // crop points per frame
  bool compact = false;     // the reproject kernels keep only finite points (CROP_FINITE without the box)
  // the cloud stages that run, in order: the transform, the crop box on the CROP cloud, VOXEL, the outlier stage
  CloudStage stages[4];
  int n_stages = 0;
  bool counted = false;     // the cloud's size is known only on the device: the kept count decides the bytes
  uint32_t count_words = 1; // count words a slot reads back (Slot::d_count)
  bool fallback_decides_dense = false;  // VOXEL alone: the overflow fallback flag clears is_dense
  ScanPlan scan;                        // the host entries' laser scan (add_scan)
  MapPlan map;                          // the host entries' occupancy map update (add_map)
};

// The device buffers between a batch's input frames and its cloud: one set per slot, one for the device batch.
struct StageBufs {
  DevBuf med;       // median-filtered frames
  DevBuf scratch;   // CROP_FINITE tile descriptors (epoch-tagged: zero when allocated, see next_epoch)
  DevBuf tables;    // CROP_FINITE tables
  DevBuf cloud[2];  // the clouds between the steps (dense, frame f at f * n * 16 bytes), then their per-frame counts
  DevBuf stage;     // the scratch of the cloud stages: they run one after another on one stream, so they share it
};

// One cloud submission on a slot.  The caller fills the first five fields; submit_front decides the rest.
struct Submission {
  uint8_t *user_dst;    // the caller's destination (d2pc_*_into); nullptr = the slot's h_out
  size_t user_cap;
  bool sync_call;       // the caller waits for this cloud right away (d2pc_process_*, d2pc_fuse_then_process)
  bool mono8;
  cudaStream_t stream;  // where the slot's kernels run: s_compute, or a fusion slot's own s_kern
  CloudPlan p;
  bool user_pinned;
  // synchronous call into a PAGEABLE caller buffer: no D2H at submit; d2pc_wait copies device -> caller directly
  // (driver-staged in chunks: 280 vs 346 us for a 752x480 cloud against D2H into pinned memory + memcpy)
  bool late_copy;
  uint8_t *d_direct;    // the device alias the kernels store the cloud into (direct output); nullptr = s.d_out
};

struct Slot {
  PinBuf h_in, h_out;
  DevBuf d_in, d_out;
  StageBufs stages;
  // fusion pipeline (d2pc_submit_fusion): the four input frames, the two preprocessed scores, merge outputs
  DevBuf d_fuse_in[4], d_pre[2], d_container, d_combined, d_fused;
  DevBuf d_ranges;  // the laser scan of the pending submission (ScanPlan), and its host copy
  PinBuf h_ranges;
  uint32_t *d_count = nullptr;  // [0] = kept points, [1] = compaction ticket, [2] = VOXEL overflow fallback taken
  uint32_t *h_count = nullptr;  // pinned
  cudaEvent_t ev_h2d = nullptr, ev_kernel = nullptr, ev_d2h = nullptr;
  cudaEvent_t ev_start = nullptr;  // recorded in front of the H2D copy when per-call timing is on (d2pc_set_timing)
  cudaEvent_t ev_map = nullptr;    // the map step of the last submission has read the slot's cloud
  bool map_pending = false;
  bool timed = false;              // the last submission on this slot recorded all four events with timing
  cudaStream_t s_kern = nullptr;  // fusion pipeline: this slot's own kernel stream (small kernels of consecutive sets overlap)
  bool pending = false;
  Submission sub{};  // the pending submission (the last one armed)
};

}  // namespace

struct d2pc_ctx {
  d2pc_config cfg;
  int device = 0;
  int sm_count = 148;
  cudaStream_t s_h2d = nullptr, s_compute = nullptr, s_d2h = nullptr;
  double q[16];
  QParams Q;
  std::vector<Slot> slots;
  uint32_t epoch = 0;
  uint64_t launches = 0;
  std::string last_cuda_error;
  StageBufs batch;  // the device-batch entries' stage buffers (their kernels run on s_compute)
  uint32_t *d_ticket = nullptr;
  d2pc_voxel_grid voxel;  // D2PC_FILTER_VOXEL parameters (d2pc_set_voxel_grid)
  bool voxel_set = false;
  d2pc_radius_outlier ror;  // the radius outlier stage behind every mode (d2pc_set_radius_outlier; radius 0: off)
  d2pc_crop_box box;        // the crop box in front of VOXEL and the outlier stage (d2pc_set_crop_box; enabled 0: off)
  d2pc_cloud_transform xform;  // the first cloud stage (d2pc_set_cloud_transform; enabled 0: off)
  d2pc_laser_scan_params scan;  // the laser scan output (d2pc_set_laser_scan; enabled 0: off)
  ScanPlan scan_plan;           // derived from `scan`
  d2pc_laser_scan last_scan{};  // d2pc_last_scan: the scan of the cloud last returned
  bool last_scan_on = false;
  d2pc_occupancy_params occ;  // the occupancy map (d2pc_set_occupancy; enabled 0: no updates)
  DevBuf map_mem;             // the map's table (allocated on first use, cleared then)
  MapTable map;               // carved from map_mem
  uint32_t map_epoch = 0;     // of the last frame inserted (marks are tagged with it)
  DevBuf map_tmp, map_out, map_n;  // export scratch, output staging and counters
  PinBuf octomap;                  // d2pc_occupancy_octomap's data, valid until the next call
  PinBuf projmap;                  // d2pc_occupancy_projected_map's cells, valid until the next call
  cudaStream_t s_map = nullptr;    // every map step and export, in submission order
  cudaEvent_t ev_map_in = nullptr; // orders d2pc_occupancy_insert_device behind the compute stream
  // fusion buffers
  DevBuf d_fuse_in[4], d_container, d_combined, d_fused;
  PinBuf h_fused, h_combined;
  DevBuf d_score_in, d_score_out[2];
  PinBuf h_score[2];
  DevBuf d_color_in, d_color_out, d_color_lut;
  PinBuf h_color;
  PinBuf h_stage;  // pinned staging of the synchronous fusion entries' pageable inputs (upload_dense)
  bool color_lut_ready = false;
  cudaEvent_t ev_fuse = nullptr;
  // tuning / test hooks
  int rows_per_unit = 0, ctas_per_sm = 0, median_strip = 0, median_variant = 0;
  bool force_scalar = false, force_generic = false;
  int compact_variant = 0, exact_variant = 0, prefetch_dist = 0, zero_numer = 0, crop_load = 0, crop_probe = 0;
  int fuse_median = 0;  // mono8 callback as one fused launch where possible: 0 yes, -1 never (two launches)
  // CROP clouds written by the kernel straight into the page-locked host buffer (no D2H copy after the kernel; the
  // transfer overlaps the kernel): 0 = the synchronous single-frame mono8 entries only (the median makes that
  // kernel long enough to hide: -6..-8 % per call; a float frame's 5 us kernel hides nothing and SM stores cross
  // PCIe ~15 % slower than the copy engine, so streams and float frames keep the copy; so do plans with a cloud
  // stage after the reproject kernel, the transform: its 1.6 us store kernel hides nothing either), 1 = every CROP
  // submission, -1 = never
  int direct_out = 0;
  bool timing = false;  // d2pc_set_timing: slot events carry timestamps
  std::vector<std::pair<uintptr_t, bool>> pin_cache;  // host pointer -> pinned (cudaHostAlloc / cudaHostRegister)?
  uint64_t pin_cache_gen = 0;                         // value of g_host_gen the cache was filled under
};

namespace {

// NVTX range for the host-side span of an entry point (SURVEY.md section 5: ranges around H2D / kernels / D2H);
// free when no profiler is attached.
struct NvtxRange {
  explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

// bumped whenever pinned host memory is released (d2pc_host_free / d2pc_host_unregister): a context's
// pointer -> "is pinned" cache is only trusted while this has not moved, so a freed and re-allocated address is
// looked up again instead of answered from memory.
std::atomic<uint64_t> g_host_gen{1};

int cuda_fail(d2pc_ctx *ctx, cudaError_t e, const char *what) {
  if (ctx) {
    ctx->last_cuda_error = std::string(what) + ": " + cudaGetErrorString(e);
  }
  if (e == cudaErrorMemoryAllocation) return D2PC_ERR_NOMEM;
  if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorInvalidDevice)
    return D2PC_ERR_NO_DEVICE;
  return D2PC_ERR_CUDA;
}

#define CU(ctx, call)                                      \
  do {                                                     \
    cudaError_t e__ = (call);                              \
    if (e__ != cudaSuccess) return cuda_fail(ctx, e__, #call); \
  } while (0)

// clear_on: a new buffer is zeroed on this stream, the one whose kernels read it, so the clear is ordered before
// them (a legacy-stream cudaMemset is not ordered with cudaStreamNonBlocking streams)
int grow_dev(d2pc_ctx *ctx, DevBuf &b, size_t bytes, cudaStream_t clear_on = nullptr) {
  if (bytes <= b.cap) return D2PC_OK;
  if (b.p) CU(ctx, cudaFree(b.p));
  b.p = nullptr;
  b.cap = 0;
  const size_t cap = round_up(bytes, 1 << 16);
  CU(ctx, cudaMalloc(&b.p, cap));
  if (clear_on) CU(ctx, cudaMemsetAsync(b.p, 0, cap, clear_on));
  b.cap = cap;
  return D2PC_OK;
}
// Page-locked host memory.  Default: cudaHostAlloc.  With D2PC_PINNED_THP=1 in the environment: an anonymous
// 2 MB-aligned mapping advised MADV_HUGEPAGE, touched, then cudaHostRegister'ed -- 512x fewer pages for the IOMMU
// and the DMA engines to walk (an experiment for the multi-GPU end-to-end path, see DESIGN.md section 5).
struct HostBlock {
  void *p;
  size_t bytes;
};
std::mutex g_thp_mutex;
std::vector<HostBlock> g_thp_blocks;

cudaError_t pinned_alloc(void **out, size_t bytes) {
  static const bool thp = [] {
    const char *v = getenv("D2PC_PINNED_THP");
    return v && atoi(v) != 0;
  }();
  if (!thp) return cudaHostAlloc(out, bytes, cudaHostAllocDefault);
  const size_t huge = (size_t)2 << 20, len = round_up(bytes, huge);
  void *p = mmap(nullptr, len + huge, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
  if (p == MAP_FAILED) return cudaErrorMemoryAllocation;
  uint8_t *a = reinterpret_cast<uint8_t *>(round_up(reinterpret_cast<uintptr_t>(p), huge));
  // give back the unaligned head and tail so that munmap(a, len) releases everything
  if (a != p) munmap(p, (size_t)(a - static_cast<uint8_t *>(p)));
  const size_t tail = (static_cast<uint8_t *>(p) + len + huge) - (a + len);
  if (tail) munmap(a + len, tail);
  madvise(a, len, MADV_HUGEPAGE);
  for (size_t i = 0; i < len; i += 4096) a[i] = 0;  // fault the pages in (as huge pages where the kernel can)
  cudaError_t e = cudaHostRegister(a, len, cudaHostRegisterDefault);
  if (e != cudaSuccess) {
    munmap(a, len);
    return e;
  }
  {
    std::lock_guard<std::mutex> lk(g_thp_mutex);
    g_thp_blocks.push_back({a, len});
  }
  *out = a;
  return cudaSuccess;
}
cudaError_t pinned_free(void *p) {
  {
    std::lock_guard<std::mutex> lk(g_thp_mutex);
    for (size_t i = 0; i < g_thp_blocks.size(); ++i)
      if (g_thp_blocks[i].p == p) {
        const size_t len = g_thp_blocks[i].bytes;
        g_thp_blocks.erase(g_thp_blocks.begin() + (long)i);
        cudaError_t e = cudaHostUnregister(p);
        munmap(p, len);
        return e;
      }
  }
  return cudaFreeHost(p);
}

int grow_pin(d2pc_ctx *ctx, PinBuf &b, size_t bytes) {
  if (bytes <= b.cap) return D2PC_OK;
  if (b.p) CU(ctx, pinned_free(b.p));
  b.p = nullptr;
  b.cap = 0;
  const size_t cap = round_up(bytes, 1 << 16);
  void *p = nullptr;
  CU(ctx, pinned_alloc(&p, cap));
  b.p = static_cast<uint8_t *>(p);
  b.cap = cap;
  return D2PC_OK;
}
void free_dev(DevBuf &b) {
  if (b.p) cudaFree(b.p);
  b = DevBuf{};
}
void free_pin(PinBuf &b) {
  if (b.p) pinned_free(b.p);
  b = PinBuf{};
}
void free_stages(StageBufs &b) {
  for (DevBuf *d : {&b.med, &b.scratch, &b.tables, &b.cloud[0], &b.cloud[1], &b.stage}) free_dev(*d);
}

uint64_t crop_points(uint32_t w, uint32_t h, int border) {
  const long cw = (long)w - 2L * border, ch = (long)h - 2L * border;
  return (cw > 0 && ch > 0) ? (uint64_t)cw * (uint64_t)ch : 0;
}

CloudPlan plan_cloud(const d2pc_ctx *ctx, uint32_t w, uint32_t h) {
  CloudPlan p;
  p.n = crop_points(w, h, ctx->cfg.border);
  const bool xform = ctx->xform.enabled != 0, box = ctx->box.enabled != 0,
             voxel = ctx->cfg.filter_mode == D2PC_FILTER_VOXEL, ror = ctx->ror.radius > 0.0;
  // the box drops non-finite points itself: CROP_FINITE + box runs the CROP kernels and lets the box compact once
  p.compact = ctx->cfg.filter_mode == D2PC_FILTER_CROP_FINITE && !box;
  if (xform) p.stages[p.n_stages++] = CloudStage::transform;
  if (box) p.stages[p.n_stages++] = CloudStage::box;
  if (voxel) p.stages[p.n_stages++] = CloudStage::voxel;
  if (ror) p.stages[p.n_stages++] = CloudStage::ror;
  // the transform keeps every point: only the stages that change the count make it decide the bytes
  p.counted = p.compact || box || voxel || ror;
  p.count_words = voxel ? 3 : 1;  // the kept count [, the ticket, the VOXEL fallback flag]
  // the box's and the outlier stage's outputs are always dense, so is a VOXEL fallback that copies the box's cloud
  p.fallback_decides_dense = voxel && !ror && !box;
  return p;
}

// The host entries' laser scan: the context's setting, when it is on.
void add_scan(const d2pc_ctx *ctx, CloudPlan &p) {
  if (ctx->scan.enabled) p.scan = ctx->scan_plan;
}
// The host entries' map update: the context's setting, when it is on, from the cloud transform's translation.
float log_odds(double p) { return (float)log(p / (1.0 - p)); }
MapUpdate map_update(const d2pc_ctx *ctx, const float origin[3]) {
  const d2pc_occupancy_params &q = ctx->occ;
  MapUpdate u{};
  for (int a = 0; a < 3; ++a) u.origin[a] = origin[a];
  u.res = q.resolution, u.rf = 1.0 / q.resolution, u.max_range = q.max_range;
  u.hit = log_odds(q.prob_hit), u.miss = log_odds(q.prob_miss);
  u.clamp_min = log_odds(q.clamp_min), u.clamp_max = log_odds(q.clamp_max);
  return u;
}
void add_map(const d2pc_ctx *ctx, CloudPlan &p) {
  if (!ctx->occ.enabled) return;
  const float *m = ctx->xform.matrix;
  const float zero[3] = {0.0f, 0.0f, 0.0f}, t[3] = {m[3], m[7], m[11]};
  p.map.on = true;
  p.map.keep_cloud = ctx->occ.keep_cloud != 0;
  p.map.u = map_update(ctx, ctx->xform.enabled ? t : zero);
}
// the cloud leaves the device unless an enabled scan or an enabled map keeps it there (keep_cloud 0)
bool cloud_out(const CloudPlan &p) {
  return (!p.scan.on || p.scan.keep_cloud) && (!p.map.on || p.map.keep_cloud);
}

// A scan setting checked (d2pc_set_laser_scan's rules) and derived.
int scan_plan_of(const d2pc_laser_scan_params *q, ScanPlan *out) {
  if (!q || q->struct_size != sizeof(*q)) return D2PC_ERR_INVALID_ARG;
  for (double v : {q->angle_min, q->angle_max, q->angle_increment, q->range_min, q->range_max})
    if (!std::isfinite(v)) return D2PC_ERR_INVALID_ARG;
  if (std::isnan(q->min_height) || std::isnan(q->max_height)) return D2PC_ERR_INVALID_ARG;
  if (!(q->range_min >= 0.0) || !(q->range_max >= q->range_min) || !(q->inf_epsilon >= 0.0) ||
      !std::isfinite(q->inf_epsilon))
    return D2PC_ERR_INVALID_ARG;
  ScanPlan s;
  d2pc_laser_scan &m = s.msg;
  m.angle_min = (float)q->angle_min, m.angle_max = (float)q->angle_max;
  m.angle_increment = (float)q->angle_increment;
  m.time_increment = 0.0f, m.scan_time = (float)q->scan_time;
  m.range_min = (float)q->range_min, m.range_max = (float)q->range_max;
  if (!(m.angle_increment > 0.0f) || !(m.angle_min <= m.angle_max)) return D2PC_ERR_INVALID_ARG;
  // the reference's size, in float arithmetic from the message's fields
  const float span = m.angle_max - m.angle_min;
  const float nf = ceilf(span / m.angle_increment);
  if (!(nf <= (float)(1u << 20))) return D2PC_ERR_INVALID_ARG;
  m.n_ranges = (uint32_t)nf;
  const float init = q->use_inf ? INFINITY : (float)((double)m.range_max + q->inf_epsilon);
  s.on = q->enabled != 0;
  s.keep_cloud = q->keep_cloud != 0;
  LaserScanParams &p = s.p;
  p.min_height = q->min_height, p.max_height = q->max_height;
  p.range_min = q->range_min, p.range_max = q->range_max;
  p.angle_min = (double)m.angle_min, p.angle_max = (double)m.angle_max, p.angle_increment = (double)m.angle_increment;
  p.n = m.n_ranges;
  memcpy(&p.init_bits, &init, 4);
  *out = s;
  return D2PC_OK;
}

// a cloud's size: all crop points, or the count the device kept (0 when only the scan leaves the device)
uint64_t kept_points(const CloudPlan &p, const uint32_t *h_count) {
  if (!cloud_out(p)) return 0;
  return p.counted && p.n ? h_count[0] : p.n;
}
// a cloud's is_dense: 0 in CROP mode (cpp:81); 1 for a counted cloud, except a VOXEL frame that took the overflow
// fallback
bool cloud_is_dense(const CloudPlan &p, const uint32_t *h_count) {
  return p.counted && !(p.fallback_decides_dense && h_count[2]);
}

uint32_t next_epoch(d2pc_ctx *ctx) {
  // 30-bit launch epoch inside the tile descriptors; 0 is "never written".  The wrap clears every descriptor buffer
  // with the device idle and waits for the clear, so it precedes the next launch on any stream.
  if (++ctx->epoch >= (1u << 30)) {
    ctx->epoch = 1;
    cudaDeviceSynchronize();
    for (auto &s : ctx->slots)
      if (s.stages.scratch.p) cudaMemsetAsync(s.stages.scratch.p, 0, s.stages.scratch.cap, ctx->s_compute);
    if (ctx->batch.scratch.p) cudaMemsetAsync(ctx->batch.scratch.p, 0, ctx->batch.scratch.cap, ctx->s_compute);
    cudaStreamSynchronize(ctx->s_compute);
  }
  return ctx->epoch;
}

void fill_cloud(const d2pc_ctx *ctx, const uint8_t *data, uint64_t n, bool is_dense, d2pc_cloud *out) {
  // src/disparity_to_point_cloud.cpp:79-85 + pcl::toROSMsg<PointXYZ> (SURVEY.md A.3)
  memset(out, 0, sizeof(*out));
  out->data = data;
  out->height = 1;
  out->width = (uint32_t)n;
  out->point_step = 16;
  out->row_step = (uint32_t)(16 * n);
  out->is_bigendian = 0;
  out->is_dense = is_dense ? 1 : 0;
  out->n_fields = 3;
  static const char *names[3] = {"x", "y", "z"};
  for (int i = 0; i < 3; ++i) {
    strncpy(out->fields[i].name, names[i], sizeof(out->fields[i].name) - 1);
    out->fields[i].offset = 4u * i;
    out->fields[i].datatype = 7;
    out->fields[i].count = 1;
  }
  (void)ctx;
}

bool is_pinned_host(const void *p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeHost;
}

// Is this host pointer page-locked (cudaHostAlloc / cudaHostRegister)?  Looked up once per distinct buffer (a
// subscriber reuses a handful of message buffers); the cache is dropped when pinned memory has been released since.
bool lookup_pinned(d2pc_ctx *ctx, const void *p) {
  const uint64_t gen = g_host_gen.load(std::memory_order_acquire);
  if (ctx->pin_cache_gen != gen) {
    ctx->pin_cache.clear();
    ctx->pin_cache_gen = gen;
  }
  const uintptr_t p0 = reinterpret_cast<uintptr_t>(p);
  for (const auto &e : ctx->pin_cache)
    if (e.first == p0) return e.second;
  const bool pinned = is_pinned_host(p);
  if (ctx->pin_cache.size() >= 64) ctx->pin_cache.clear();
  ctx->pin_cache.emplace_back(p0, pinned);
  return pinned;
}

// One caller image (w bytes x h rows, `step` apart) into a DENSE device image on `stream`, for the synchronous
// fusion entries.  Dense rows travel as ONE 1-D copy straight from the caller's memory (page-locked: DMA in place;
// pageable: the driver's own chunked staging, which beats a memcpy into pinned staging followed by a DMA -- 103 vs
// 110 us for a 1280x720 score callback).  Padded rows are packed into pinned staging at `stage_off` first (the caller
// has grown ctx->h_stage and the stream is idle).  What must be avoided is a PITCHED copy from pageable memory, which
// the driver stages row by row: with 256-byte-pitched device images the 665 x 665 colouriser input took ~250 us
// that way and a 752-wide score frame 60 us more than it does now.
int upload_dense(d2pc_ctx *ctx, size_t stage_off, uint8_t *dst, const uint8_t *src, uint32_t w, uint32_t h, size_t step,
                 cudaStream_t stream) {
  const size_t bytes = (size_t)w * h;
  if (step != w) {
    uint8_t *stage = ctx->h_stage.p + stage_off;
    for (uint32_t y = 0; y < h; ++y) memcpy(stage + (size_t)y * w, src + (size_t)y * step, w);
    src = stage;
  }
  CU(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream));
  return D2PC_OK;
}

// A batch of frames on the device: frame f at data + f * frame_stride, rows `step` bytes apart.
struct FrameBatch {
  const uint8_t *data;
  bool is_f32;
  uint32_t n_frames, w, h;
  size_t step, frame_stride;
};

size_t stage_scratch_bytes(CloudStage st, uint32_t n_frames, uint32_t n) {
  return st == CloudStage::transform ? 0
         : st == CloudStage::box   ? crop_box_scratch_bytes(n_frames, n)
         : st == CloudStage::voxel ? voxel_scratch_bytes(n_frames, n)
                                   : ror_scratch_bytes(n_frames, n);
}

// A cloud buffer of StageBufs: n_frames dense clouds of n points, then their per-frame counts.
size_t cloud_buf_bytes(uint32_t n_frames, uint32_t n) {
  return align_up((size_t)n_frames * n * 16) + (size_t)n_frames * 4;
}
CloudDst cloud_buf(const DevBuf &b, uint32_t n_frames, uint32_t n) {
  const size_t clouds = align_up((size_t)n_frames * n * 16);
  return {b.p, (size_t)n * 16, b.p ? reinterpret_cast<uint32_t *>(b.p + clouds) : nullptr};
}

// Grows a stage-buffer set for batch `in` under plan p.  `stream` is where the set's kernels run; a new CROP_FINITE
// descriptor buffer is cleared there.  in_use: work queued on `stream` may still use the set, so the stream is
// synchronised before the first buffer is replaced (and only then).
int grow_stages(d2pc_ctx *ctx, StageBufs &b, const CloudPlan &p, const FrameBatch &in, cudaStream_t stream,
                bool in_use) {
  const uint32_t n = (uint32_t)p.n;
  const bool median = !in.is_f32 && ctx->cfg.median_ksize > 1;
  const int stages = p.n_stages;
  size_t scratch = 0;
  for (int i = 0; i < stages; ++i) scratch = std::max(scratch, stage_scratch_bytes(p.stages[i], in.n_frames, n));
  const struct {
    DevBuf &buf;
    size_t bytes;
    bool zero;
  } need[] = {
      {b.med, median ? in.frame_stride * (in.n_frames - 1) + in.step * in.h : 0, false},
      {b.scratch, p.compact ? reproject_scratch_bytes(in.n_frames, in.w, in.h, ctx->cfg.border) : 0, true},
      {b.tables, p.compact ? reproject_table_bytes(in.w, in.h) : 0, false},
      {b.cloud[0], stages > 0 ? cloud_buf_bytes(in.n_frames, n) : 0, false},
      {b.cloud[1], stages > 1 ? cloud_buf_bytes(in.n_frames, n) : 0, false},
      {b.stage, scratch, false},
  };
  for (const auto &x : need) {
    if (x.bytes <= x.buf.cap) continue;
    if (in_use) CU(ctx, cudaStreamSynchronize(stream));
    in_use = false;
    const int rc = grow_dev(ctx, x.buf, x.bytes, x.zero ? stream : nullptr);
    if (rc) return rc;
  }
  return D2PC_OK;
}

// Frames per launch of the cloud stages: at most kCloudMaxPoints points (but at least one frame).
uint32_t frames_per_chunk(uint32_t n_frames, uint64_t points_per_frame) {
  const uint64_t by_points = std::max<uint64_t>(1, kCloudMaxPoints / std::max<uint64_t>(points_per_frame, 1));
  return (uint32_t)std::min<uint64_t>(n_frames, by_points);
}

// A batch of clouds on the device in frames_per_chunk chunks: fn(f0, chunk) for the chunk of frames f0, f0 + 1, ...
template <class Fn>
int for_each_chunk(const uint8_t *d_in, uint32_t n_frames, uint32_t n_max, size_t in_stride, const uint32_t *d_in_counts,
                   Fn fn) {
  const uint32_t chunk = frames_per_chunk(n_frames, n_max);
  for (uint32_t f0 = 0; f0 < n_frames; f0 += chunk) {
    const int rc = fn(f0, CloudSrc{d_in + f0 * in_stride, in_stride, d_in_counts ? d_in_counts + f0 : nullptr,
                                   std::min(chunk, n_frames - f0), n_max});
    if (rc) return rc;
  }
  return D2PC_OK;
}

CloudTransformParams transform_params(const d2pc_ctx *ctx) {
  CloudTransformParams t;
  for (int k = 0; k < 12; ++k) t.m[k] = ctx->xform.matrix[k];
  return t;
}

// One cloud stage with the context's setting on a batch of clouds, on `stream`.  The setting travels by value, so a
// later d2pc_set_* cannot reach a queued launch.  fallback: VOXEL's per-frame overflow fallback flags (may be null).
int enqueue_stage(d2pc_ctx *ctx, CloudStage st, const CloudSrc &in, const CloudDst &out, uint32_t *fallback,
                  void *scratch, cudaStream_t stream) {
  int nl = 0;
  cudaError_t e;
  if (st == CloudStage::transform) {
    e = launch_cloud_transform(in, out, transform_params(ctx), nullptr, stream, &nl);
  } else if (st == CloudStage::box) {
    const d2pc_crop_box &box = ctx->box;
    CropBoxParams b;
    for (int a = 0; a < 3; ++a) b.mn[a] = box.min_pt[a], b.mx[a] = box.max_pt[a];
    for (int k = 0; k < 12; ++k) b.t[k] = box.transform[k];
    e = launch_crop_box(in, out, b, scratch, stream, &nl);
  } else if (st == CloudStage::voxel) {
    const d2pc_voxel_grid &g = ctx->voxel;
    VoxelParams v;
    v.inv[0] = 1.0f / g.leaf_x, v.inv[1] = 1.0f / g.leaf_y, v.inv[2] = 1.0f / g.leaf_z;
    v.min_points = g.min_points_per_voxel;
    v.limit_field = g.limit_field;
    v.limit_min = g.limit_min, v.limit_max = g.limit_max;
    e = launch_voxel(in, out, v, fallback, scratch, stream, &nl);
  } else {
    e = launch_radius_outlier(in, out, ctx->ror.radius, ctx->ror.min_neighbors, scratch, stream, &nl);
  }
  CU(ctx, e);
  ctx->launches += nl;
  return D2PC_OK;
}

// [median] + reproject of a batch into dst.
int enqueue_reproject(d2pc_ctx *ctx, const CloudPlan &p, const FrameBatch &in, StageBufs &b, const CloudDst &dst,
                      uint32_t *ticket, cudaStream_t stream) {
  const d2pc_config &c = ctx->cfg;
  int nl = 0;
  ReprojectLaunch L;
  L.in = in.data;
  L.in_is_f32 = in.is_f32;
  L.step = in.step;
  L.frame_stride = in.frame_stride;
  L.n_frames = in.n_frames;
  L.width = in.w;
  L.height = in.h;
  L.border = c.border;
  L.scale = c.disparity_scale;
  L.out = dst.points;
  L.out_stride_bytes = dst.stride;
  L.counts = dst.counts;
  L.Q = &ctx->Q;
  L.arith_fast = c.arith_mode == D2PC_ARITH_FAST;
  L.compact = p.compact;
  L.scratch = b.scratch.p;
  L.tables = b.tables.p;
  L.ticket = ticket;
  L.sm_count = ctx->sm_count;
  L.rows_per_unit = ctx->rows_per_unit;
  L.ctas_per_sm = ctx->ctas_per_sm;
  L.force_scalar = ctx->force_scalar;
  L.force_generic = ctx->force_generic;
  L.compact_variant = ctx->compact_variant;
  L.exact_variant = ctx->exact_variant;
  L.zero_numer = ctx->zero_numer;
  L.prefetch_dist = ctx->prefetch_dist;
  L.crop_load = ctx->crop_load;
  L.crop_probe = ctx->crop_probe != 0;
  if (!in.is_f32 && c.median_ksize > 1) {
    // cpp:55-57: only crop pixels are consumed downstream, so only those medians are produced
    // (the replicate border is still the image edge, which matters when border < ksize/2).
    MedianLaunch M;
    M.src = in.data;
    M.dst = b.med.p;
    M.src_step = M.dst_step = in.step;
    M.src_frame_stride = M.dst_frame_stride = in.frame_stride;
    M.n_frames = in.n_frames;
    M.width = (int)in.w;
    M.height = (int)in.h;
    M.ox0 = c.border;
    M.oy0 = c.border;
    M.ow = (int)in.w - 2 * c.border;
    M.oh = (int)in.h - 2 * c.border;
    M.ksize = c.median_ksize;
    M.sm_count = ctx->sm_count;
    M.strip_rows = ctx->median_strip;
    M.variant = ctx->median_variant;
    // the whole callback in one launch where the arithmetic allows it (the default Q does): median -> x 1/8 ->
    // reproject -> PointXYZ, no intermediate image
    bool zero_numer = false;
    const bool fuse = ctx->fuse_median >= 0 && M.ow > 0 && M.oh > 0 && (c.median_ksize > 3 || M.variant != 0) &&
                      reproject_fuses_with_median(L, &zero_numer);
    if (fuse) {
      M.zero_numer = zero_numer;
      M.points = dst.points;
      M.points_stride_bytes = dst.stride;
      M.Q = &ctx->Q;
      M.scale = c.disparity_scale;
    }
    CU(ctx, launch_median_u8(M, stream, &nl));
    ctx->launches += nl;
    if (fuse) return D2PC_OK;
    L.in = b.med.p;
  }
  L.epoch = L.compact ? next_epoch(ctx) : 0;
  CU(ctx, launch_reproject(L, stream, &nl));
  ctx->launches += nl;
  return D2PC_OK;
}

// Enqueue the plan's steps for one frame batch already on the device: [median] + reproject, then each cloud stage
// in plan order.  The reproject kernels write cloud buffer 0; each stage reads one buffer and writes the other, so
// its input and output never overlap; the last step writes `out`.  fallback: VOXEL's per-frame overflow fallback
// flags (may be null).  ranges: with the plan's scan on, the scan of `out` is the last step and writes each frame's
// ranges there (frame f at f * 4 * n bytes).
int enqueue_kernels(d2pc_ctx *ctx, const CloudPlan &p, const FrameBatch &in, StageBufs &b, const CloudDst &out,
                    uint32_t *fallback, uint32_t *ticket, cudaStream_t stream, float *ranges) {
  const uint32_t n = (uint32_t)p.n;
  const int stages = p.n_stages;
  const CloudDst buf[2] = {cloud_buf(b.cloud[0], in.n_frames, n), cloud_buf(b.cloud[1], in.n_frames, n)};
  int rc = enqueue_reproject(ctx, p, in, b, stages ? buf[0] : out, ticket, stream);
  for (int i = 0; i < stages && !rc; ++i) {
    const CloudDst &src = buf[i & 1];
    // a CROP cloud straight from the reproject kernels has all n points; every other cloud's count is on the device
    const CloudSrc cloud{src.points, src.stride, i > 0 || p.compact ? src.counts : nullptr, in.n_frames, n};
    rc = enqueue_stage(ctx, p.stages[i], cloud, i + 1 < stages ? buf[(i + 1) & 1] : out, fallback, b.stage.p, stream);
  }
  if (rc || !p.scan.on || !ranges) return rc;
  // an uncounted plan's cloud has all n points in every frame
  const CloudSrc cloud{out.points, out.stride, p.counted ? out.counts : nullptr, in.n_frames, n};
  int nl = 0;
  CU(ctx, launch_laser_scan(cloud, p.scan.p, ranges, (size_t)p.scan.p.n * 4, stream, &nl));
  ctx->launches += nl;
  return D2PC_OK;
}

int check_frame(const d2pc_ctx *ctx, const void *data, uint32_t w, uint32_t h, size_t step, int esz) {
  if (!ctx || !data) return D2PC_ERR_INVALID_ARG;
  if (w == 0 || h == 0 || w > (1u << 16) || h > (1u << 16)) return D2PC_ERR_BAD_DIMS;
  if (step < (size_t)w * esz) return D2PC_ERR_BAD_DIMS;
  if (esz == 4 && (step % 4 != 0 || reinterpret_cast<uintptr_t>(data) % 4 != 0)) return D2PC_ERR_BAD_DIMS;
  return D2PC_OK;
}

int slot_wait_idle(d2pc_ctx *ctx, Slot &s) {
  if (s.pending) {
    CU(ctx, cudaEventSynchronize(s.ev_d2h));
    s.pending = false;
  }
  if (s.map_pending) {  // the map step still reads the slot's cloud
    CU(ctx, cudaEventSynchronize(s.ev_map));
    s.map_pending = false;
  }
  return D2PC_OK;
}

// The map's table, allocated and cleared on s_map on first use (and after a change of max_bricks).
int map_ready(d2pc_ctx *ctx) {
  if (ctx->map_mem.p) return D2PC_OK;
  const int rc = grow_dev(ctx, ctx->map_mem, map_table_bytes(ctx->occ.max_bricks));
  if (rc) return rc;
  ctx->map = map_table_carve(ctx->map_mem.p, ctx->occ.max_bricks);
  CU(ctx, map_clear(ctx->map, true, ctx->s_map));
  ctx->map_epoch = 0;
  return D2PC_OK;
}

// One frame into the map on s_map, after `after` (the kernels that wrote the cloud).  The epoch wraps as next_epoch's
// does: every mark and slot epoch is cleared with s_map idle.
int enqueue_map(d2pc_ctx *ctx, MapUpdate u, const CloudSrc &cloud, cudaEvent_t after) {
  int rc = map_ready(ctx);
  if (rc) return rc;
  if (++ctx->map_epoch >= (1u << 30)) {
    ctx->map_epoch = 1;
    CU(ctx, cudaStreamSynchronize(ctx->s_map));
    CU(ctx, cudaMemsetAsync(ctx->map.marks, 0, (size_t)ctx->map.cap * 512 * 4, ctx->s_map));
    CU(ctx, cudaMemsetAsync(ctx->map.slot_epoch, 0, (size_t)ctx->map.cap * 4, ctx->s_map));
  }
  u.epoch = ctx->map_epoch;
  if (after) CU(ctx, cudaStreamWaitEvent(ctx->s_map, after, 0));
  int nl = 0;
  CU(ctx, launch_map_insert(cloud, ctx->map, u, ctx->sm_count, ctx->s_map, &nl));
  ctx->launches += nl;
  return D2PC_OK;
}

// A slot's map step: its cloud `out` (all n points, or the count the device kept), behind ev_kernel.
int enqueue_slot_map(d2pc_ctx *ctx, Slot &s, const CloudPlan &p, const CloudDst &out) {
  if (!p.map.on) return D2PC_OK;
  const CloudSrc cloud{out.points, out.stride, p.counted ? out.counts : nullptr, 1, (uint32_t)p.n};
  const int rc = enqueue_map(ctx, p.map.u, cloud, s.ev_kernel);
  if (rc) return rc;
  CU(ctx, cudaEventRecord(s.ev_map, ctx->s_map));
  s.map_pending = true;
  return D2PC_OK;
}

// The device alias of page-locked host memory, for a kernel's point stores into it; null where there is none or it is
// not 16-byte aligned.
uint8_t *direct_alias(void *host) {
  void *dp = nullptr;
  if (cudaHostGetDevicePointer(&dp, host, 0) == cudaSuccess && reinterpret_cast<uintptr_t>(dp) % 16 == 0)
    return static_cast<uint8_t *>(dp);
  cudaGetLastError();
  return nullptr;
}

// A slot's D2H (stream 3), behind its kernels: the count words when the count decides the bytes (the payload copy is
// issued in d2pc_wait), else the whole cloud into dst (dst null: the cloud leaves elsewhere, or not at all); then the
// scan's ranges.
int enqueue_readback(d2pc_ctx *ctx, Slot &s, const CloudPlan &p, uint8_t *dst) {
  CU(ctx, cudaStreamWaitEvent(ctx->s_d2h, s.ev_kernel, 0));
  if (dst && cloud_out(p)) {
    if (p.counted)
      CU(ctx, cudaMemcpyAsync(s.h_count, s.d_count, p.count_words * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                              ctx->s_d2h));
    else if (p.n)
      CU(ctx, cudaMemcpyAsync(dst, s.d_out.p, p.n * 16, cudaMemcpyDeviceToHost, ctx->s_d2h));
  }
  if (p.scan.on && p.scan.p.n)
    CU(ctx, cudaMemcpyAsync(s.h_ranges.p, s.d_ranges.p, (size_t)p.scan.p.n * 4, cudaMemcpyDeviceToHost, ctx->s_d2h));
  CU(ctx, cudaEventRecord(s.ev_d2h, ctx->s_d2h));
  return D2PC_OK;
}

// What every slot submission does before its input reaches the device: the plan for a w x h frame, its checks, and
// the slot's output buffers.  Nothing is allocated or read before the checks.
int submit_front(d2pc_ctx *ctx, Slot &s, uint32_t w, uint32_t h, Submission &sub) {
  CU(ctx, cudaSetDevice(ctx->device));
  int rc = slot_wait_idle(ctx, s);
  if (rc) return rc;
  CloudPlan &p = sub.p;
  p = plan_cloud(ctx, w, h);
  add_scan(ctx, p);
  add_map(ctx, p);
  const uint64_t n = p.n;
  if (n * 16 > 0xffffffffull) return D2PC_ERR_BAD_DIMS;  // PointCloud2.row_step / width are uint32
  const bool out_cloud = cloud_out(p);
  uint8_t *const dst = sub.user_dst;
  if (dst && !p.counted && out_cloud && sub.user_cap < n * 16) return D2PC_ERR_BUFFER_TOO_SMALL;
  sub.user_pinned = dst && reinterpret_cast<uintptr_t>(dst) % 16 == 0 && lookup_pinned(ctx, dst);
  sub.late_copy = sub.sync_call && dst && !sub.user_pinned && !p.counted && n && out_cloud;
  if (!sub.user_pinned && !sub.late_copy && out_cloud && (rc = grow_pin(ctx, s.h_out, n * 16 + 16))) return rc;
  if (p.scan.on && ((rc = grow_dev(ctx, s.d_ranges, (size_t)p.scan.p.n * 4)) ||
                    (rc = grow_pin(ctx, s.h_ranges, (size_t)p.scan.p.n * 4))))
    return rc;
  // direct output: the kernel's point stores go over PCIe into the page-locked destination while it runs, so a lone
  // frame no longer pays kernel + copy back to back (CROP only: a compacted cloud's size is not known up front; not
  // with the scan or the map, which read the cloud on the device)
  sub.d_direct = nullptr;
  if (!p.counted && n && !sub.late_copy && !p.scan.on && !p.map.on &&
      (ctx->direct_out > 0 ||
       (ctx->direct_out == 0 && sub.sync_call && sub.mono8 && ctx->cfg.median_ksize > 1 && p.n_stages == 0)))
    sub.d_direct = direct_alias(sub.user_pinned ? dst : s.h_out.p);
  if (!sub.d_direct && (rc = grow_dev(ctx, s.d_out, n * 16 + 16))) return rc;
  return D2PC_OK;
}

// What every slot submission does once its input frame `in` is on the device, or queued to be, ahead of sub.stream:
// the plan's kernels, the map step, the cloud's way to the host, and the slot armed for d2pc_wait.
int submit_back(d2pc_ctx *ctx, Slot &s, const FrameBatch &in, const Submission &sub) {
  const CloudPlan &p = sub.p;
  const uint64_t n = p.n;
  int rc;
  {
    NvtxRange nvtx_k("d2pc kernels");
    if ((rc = grow_stages(ctx, s.stages, p, in, sub.stream, false)) ||
        (rc = enqueue_kernels(ctx, p, in, s.stages, {sub.d_direct ? sub.d_direct : s.d_out.p, n * 16 + 16, s.d_count},
                              s.d_count + 2, s.d_count + 1, sub.stream, reinterpret_cast<float *>(s.d_ranges.p))))
      return rc;
  }
  CU(ctx, cudaEventRecord(s.ev_kernel, sub.stream));
  // the map step runs on s_map behind ev_kernel, so every slot updates the map in submission order
  if ((rc = enqueue_slot_map(ctx, s, p, {s.d_out.p, n * 16 + 16, s.d_count}))) return rc;

  NvtxRange nvtx_d2h("d2pc D2H");
  if ((sub.d_direct || sub.late_copy) && !p.scan.on) {
    // the cloud is already in host memory when the kernel ends (direct output), or leaves the device in d2pc_wait
    // (pageable destination of a synchronous call): the slot completes on its kernel stream
    CU(ctx, cudaEventRecord(s.ev_d2h, sub.stream));
  } else {
    // a page-locked caller buffer receives the cloud by DMA directly; a pageable one is filled from h_out in wait
    // (a late copy with the scan on: only the ranges here)
    uint8_t *const dst = sub.late_copy ? nullptr : sub.user_pinned ? sub.user_dst : s.h_out.p;
    if ((rc = enqueue_readback(ctx, s, p, dst))) return rc;
  }
  s.pending = true;
  s.sub = sub;
  return D2PC_OK;
}

int submit_common(d2pc_ctx *ctx, int slot, const void *data, uint32_t w, uint32_t h, uint32_t step, bool is_f32,
                  uint8_t *user_dst, size_t user_cap, bool sync_call) {
  if (!ctx || slot < 0 || slot >= (int)ctx->slots.size()) return D2PC_ERR_INVALID_ARG;
  const int esz = is_f32 ? 4 : 1;
  int rc = check_frame(ctx, data, w, h, step, esz);
  if (rc) return rc;
  Slot &s = ctx->slots[slot];
  NvtxRange nvtx_submit(is_f32 ? "d2pc submit f32" : "d2pc submit mono8");
  Submission sub{user_dst, user_cap, sync_call, !is_f32, ctx->s_compute};
  if ((rc = submit_front(ctx, s, w, h, sub))) return rc;

  const size_t row_bytes = (size_t)w * esz;
  // rows that are already 16-byte multiples stay dense on the device: the H2D copy is then one contiguous DMA.  So do
  // mono8 rows of any width (the callback kernel reads bytes; a 665-wide fused map is then one DMA instead of a
  // pitched 2-D copy); float rows that are not 16-byte multiples keep a 256-byte pitch for the vector loads.
  const size_t d_pitch = (row_bytes % 16 == 0 || !is_f32) ? row_bytes : round_up(row_bytes, kAlign);
  if ((rc = grow_dev(ctx, s.d_in, d_pitch * h))) return rc;

  // ---- H2D (stream 1).  Pinned caller memory is DMA'd in place; pageable memory is staged.
  const void *src = data;
  size_t src_pitch = step;
  // (a dense pageable frame goes to cudaMemcpyAsync as it is: the driver stages it chunk by chunk, overlapping its
  // own copy with the DMA, and returns once the caller's buffer has been read -- measured against a memcpy into
  // pinned staging followed by one DMA: 752x480 float call 225 -> 180 us, 1280x720 float 540 -> 440 us, mono8
  // 1280x720 327 -> 313 us; only padded pageable rows are still packed into pinned staging here)
  const bool pinned = lookup_pinned(ctx, data) || (step == row_bytes && d_pitch == row_bytes);
  if (!pinned) {
    // rows are laid out in the staging buffer with the DEVICE pitch, so what follows is one 1-D DMA (a pitched 2-D
    // copy is the slow way in, even from pinned memory)
    if ((rc = grow_pin(ctx, s.h_in, d_pitch * h))) return rc;
    for (uint32_t y = 0; y < h; ++y)
      memcpy(s.h_in.p + (size_t)y * d_pitch, static_cast<const uint8_t *>(data) + (size_t)y * step, row_bytes);
    src = s.h_in.p;
    src_pitch = d_pitch;
  }
  s.timed = ctx->timing && s.ev_start;
  if (s.timed) CU(ctx, cudaEventRecord(s.ev_start, ctx->s_h2d));
  {
    NvtxRange nvtx_h2d("d2pc H2D");
    if (src_pitch == d_pitch)  // same layout on both sides (dense, or staged with the device pitch): one 1-D copy
      CU(ctx, cudaMemcpyAsync(s.d_in.p, src, d_pitch * (h - 1) + row_bytes, cudaMemcpyHostToDevice, ctx->s_h2d));
    else
      CU(ctx, cudaMemcpy2DAsync(s.d_in.p, d_pitch, src, src_pitch, row_bytes, h, cudaMemcpyHostToDevice, ctx->s_h2d));
    CU(ctx, cudaEventRecord(s.ev_h2d, ctx->s_h2d));
  }

  // ---- kernels (stream 2)
  CU(ctx, cudaStreamWaitEvent(ctx->s_compute, s.ev_h2d, 0));
  return submit_back(ctx, s, {s.d_in.p, is_f32, 1, w, h, d_pitch, d_pitch * h}, sub);
}

// A stream of n items over the slots: item i is read from base + (i % ring_len) * stride (ring_len 0: no wrap) and
// submitted with submit(item, slot) while a slot is free -- the H2D of item i+2, the kernels of i+1 and the D2H of i
// overlap on the three streams -- then the oldest is waited on and handed to the sink, in submission order.
template <class Submit>
int run_ring(d2pc_ctx *ctx, const uint8_t *base, uint64_t n, size_t stride, uint64_t ring_len, Submit submit,
             d2pc_cloud_sink sink, void *user) {
  const uint64_t ns = ctx->slots.size();
  d2pc_cloud cloud;
  uint64_t submitted = 0, retired = 0;
  while (retired < n) {
    while (submitted < n && submitted - retired < ns) {
      const int rc = submit(base + (ring_len ? submitted % ring_len : submitted) * stride, (int)(submitted % ns));
      if (rc) return rc;
      ++submitted;
    }
    const int rc = d2pc_wait(ctx, (int)(retired % ns), &cloud);
    if (rc) return rc;
    if (sink) sink(user, retired, &cloud);
    ++retired;
  }
  return D2PC_OK;
}

}  // namespace

// ---------------------------------------------------------------------------
// lifecycle
// ---------------------------------------------------------------------------
extern "C" {

void d2pc_config_default(d2pc_config *c) {
  if (!c) return;
  memset(c, 0, sizeof(*c));
  c->struct_size = sizeof(*c);
  c->fx = 714.24, c->fy = 713.5, c->cx = 376.0, c->cy = 240.0, c->baseline = 0.09;
  c->rect_width = 752, c->rect_height = 480;
  c->border = 40;
  c->median_ksize = 11;
  c->disparity_scale = 1.0f / 8.0f;
  c->filter_mode = D2PC_FILTER_CROP;
  c->arith_mode = D2PC_ARITH_EXACT;
  strncpy(c->frame_id, "/camera_optical_frame", sizeof(c->frame_id) - 1);
  c->offset_x = 0, c->offset_y = 0;  // depth_map_fusion.hpp:76-77 (the launch file sets -7 / 15)
  c->fuse_rule = D2PC_FUSE_GRAD_FILTER;
  c->fuse_median_ksize = 3;
  c->fuse_crop_left = 0, c->fuse_crop_right = 40, c->fuse_crop_top = 30, c->fuse_crop_bottom = 10;
  c->max_width = 0, c->max_height = 0, c->max_batch = 0;
  c->n_slots = 4;
}

int d2pc_abi_version(void) { return D2PC_ABI_VERSION; }

int d2pc_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) == cudaSuccess && major == 10) ++ok;
  }
  return ok;
}

int d2pc_q_from_intrinsics(double fx, double fy, double cx, double cy, double baseline, int rect_w, int rect_h,
                           double q[16]) {
  // disparity_to_point_cloud.hpp:90-104: stereoRectify(K, 0, K, 0, size, I, (-b,0,0)).  For that call OpenCV's
  // rectification is the identity, the new focal length is fy, and the new principal point comes from the four
  // image corners normalised with K (float32), re-projected with the new focal length (float32) and averaged.
  if (!q || !(fx != 0.0) || !(fy != 0.0) || !(baseline != 0.0) || rect_w <= 0 || rect_h <= 0 || !std::isfinite(fx) ||
      !std::isfinite(fy) || !std::isfinite(cx) || !std::isfinite(cy) || !std::isfinite(baseline))
    return D2PC_ERR_INVALID_ARG;
  const double f = fy, inv_fx = 1.0 / fx, inv_fy = 1.0 / fy;
  const float corner_x[2] = {0.0f, (float)(rect_w - 1)}, corner_y[2] = {0.0f, (float)(rect_h - 1)};
  double mean_x = 0.0, mean_y = 0.0;
  for (int k = 0; k < 4; ++k) {
    const float ux = (float)(((double)corner_x[k & 1] - cx) * inv_fx);
    const float uy = (float)(((double)corner_y[k >> 1] - cy) * inv_fy);
    mean_x += (double)(float)((double)ux * f + 0.0);
    mean_y += (double)(float)((double)uy * f + 0.0);
  }
  mean_x /= 4.0;
  mean_y /= 4.0;
  const double pcx = (rect_w - 1) * 0.5 - mean_x, pcy = (rect_h - 1) * 0.5 - mean_y;
  const double tx = -baseline;
  for (int i = 0; i < 16; ++i) q[i] = 0.0;
  q[0] = 1.0, q[3] = -pcx;
  q[5] = 1.0, q[7] = -pcy;
  q[11] = f;
  q[14] = -1.0 / tx;
  q[15] = (pcx - pcx) / tx;  // both cameras share K: zero numerator, sign of tx survives as -0.0
  return D2PC_OK;
}

int d2pc_create(const d2pc_config *cfg, int device, d2pc_ctx **out) {
  if (!out) return D2PC_ERR_INVALID_ARG;
  *out = nullptr;
  d2pc_config c;
  d2pc_config_default(&c);
  if (cfg) {
    if (cfg->struct_size == 0 || cfg->struct_size > sizeof(c)) return D2PC_ERR_INVALID_ARG;
    memcpy(&c, cfg, cfg->struct_size);
    c.struct_size = sizeof(c);
  }
  if (c.border < 0 || c.n_slots < 1 || c.n_slots > 64 || c.median_ksize < 1 || c.median_ksize > 15 ||
      (c.median_ksize & 1) == 0 || c.fuse_median_ksize < 1 || c.fuse_median_ksize > 15 ||
      (c.fuse_median_ksize & 1) == 0 || c.filter_mode < 0 || c.filter_mode > 1 || c.arith_mode < 0 ||
      c.arith_mode > 1 || c.fuse_rule < 0 || c.fuse_rule > 7)
    return D2PC_ERR_INVALID_ARG;
  c.frame_id[sizeof(c.frame_id) - 1] = 0;

  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    return D2PC_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= n) return D2PC_ERR_NO_DEVICE;
  int major = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
  if (major != 10) return D2PC_ERR_NO_DEVICE;  // the library carries sm_100a code only

  d2pc_ctx *ctx = new (std::nothrow) d2pc_ctx();
  if (!ctx) return D2PC_ERR_NOMEM;
  ctx->cfg = c;
  ctx->device = device;
  int rc = D2PC_OK;
  auto fail = [&](int code) {
    d2pc_destroy(ctx);
    return code;
  };
  if (cudaSetDevice(device) != cudaSuccess) return fail(D2PC_ERR_NO_DEVICE);
  cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
  if (cudaStreamCreateWithFlags(&ctx->s_h2d, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->s_compute, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->s_d2h, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_fuse, cudaEventDisableTiming) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->s_map, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_map_in, cudaEventDisableTiming) != cudaSuccess)
    return fail(D2PC_ERR_CUDA);
  if (cudaMalloc(&ctx->d_ticket, 64) != cudaSuccess) return fail(D2PC_ERR_NOMEM);
  ctx->slots.resize(c.n_slots);
  for (auto &s : ctx->slots) {
    if (cudaEventCreateWithFlags(&s.ev_h2d, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.ev_kernel, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.ev_d2h, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.ev_map, cudaEventDisableTiming) != cudaSuccess ||
        cudaStreamCreateWithFlags(&s.s_kern, cudaStreamNonBlocking) != cudaSuccess)
      return fail(D2PC_ERR_CUDA);
    if (cudaMalloc(&s.d_count, 64) != cudaSuccess) return fail(D2PC_ERR_NOMEM);
    if (cudaHostAlloc(&s.h_count, 64, cudaHostAllocDefault) != cudaSuccess) return fail(D2PC_ERR_NOMEM);
    cudaMemsetAsync(s.d_count, 0, 64, ctx->s_compute);
  }
  rc = d2pc_q_from_intrinsics(c.fx, c.fy, c.cx, c.cy, c.baseline, c.rect_width, c.rect_height, ctx->q);
  if (rc) return fail(rc);
  make_qparams(ctx->q, &ctx->Q);
  d2pc_voxel_grid_default(&ctx->voxel);
  d2pc_radius_outlier_default(&ctx->ror);
  d2pc_crop_box_default(&ctx->box);
  d2pc_cloud_transform_default(&ctx->xform);
  d2pc_laser_scan_params_default(&ctx->scan);
  scan_plan_of(&ctx->scan, &ctx->scan_plan);
  d2pc_occupancy_params_default(&ctx->occ);

  if (const char *v = getenv("D2PC_ROWS_PER_UNIT")) ctx->rows_per_unit = atoi(v);
  if (const char *v = getenv("D2PC_CTAS_PER_SM")) ctx->ctas_per_sm = atoi(v);
  if (const char *v = getenv("D2PC_CROP_LOAD")) ctx->crop_load = atoi(v);
  if (const char *v = getenv("D2PC_MEDIAN_STRIP")) ctx->median_strip = atoi(v);
  if (const char *v = getenv("D2PC_EXACT_VARIANT")) ctx->exact_variant = atoi(v);

  // pre-size the slots when the caller told us the largest frame
  if (c.max_width > 0 && c.max_height > 0) {
    for (auto &s : ctx->slots) {
      const size_t pitch = round_up((size_t)c.max_width * 4, kAlign);
      const uint64_t np = crop_points(c.max_width, c.max_height, c.border);
      if ((rc = grow_dev(ctx, s.d_in, pitch * c.max_height)) ||
          (rc = grow_dev(ctx, s.stages.med, pitch * c.max_height)) ||
          (rc = grow_dev(ctx, s.d_out, np * 16 + 16)) || (rc = grow_pin(ctx, s.h_out, np * 16 + 16)) ||
          (rc = grow_pin(ctx, s.h_in, (size_t)c.max_width * 4 * c.max_height)))
        return fail(rc);
    }
  }
  *out = ctx;
  return D2PC_OK;
}

void d2pc_destroy(d2pc_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (auto &s : ctx->slots) {
    free_pin(s.h_in), free_pin(s.h_out);
    free_dev(s.d_in), free_dev(s.d_out), free_stages(s.stages), free_dev(s.d_ranges), free_pin(s.h_ranges);
    for (auto &b : s.d_fuse_in) free_dev(b);
    free_dev(s.d_pre[0]), free_dev(s.d_pre[1]), free_dev(s.d_container), free_dev(s.d_combined), free_dev(s.d_fused);
    if (s.d_count) cudaFree(s.d_count);
    if (s.h_count) cudaFreeHost(s.h_count);
    if (s.ev_h2d) cudaEventDestroy(s.ev_h2d);
    if (s.ev_kernel) cudaEventDestroy(s.ev_kernel);
    if (s.ev_d2h) cudaEventDestroy(s.ev_d2h);
    if (s.ev_start) cudaEventDestroy(s.ev_start);
    if (s.ev_map) cudaEventDestroy(s.ev_map);
    if (s.s_kern) cudaStreamDestroy(s.s_kern);
  }
  free_stages(ctx->batch);
  for (auto &b : ctx->d_fuse_in) free_dev(b);
  free_dev(ctx->d_container), free_dev(ctx->d_combined), free_dev(ctx->d_fused);
  free_pin(ctx->h_fused), free_pin(ctx->h_combined);
  free_dev(ctx->d_score_in), free_dev(ctx->d_score_out[0]), free_dev(ctx->d_score_out[1]);
  free_pin(ctx->h_score[0]), free_pin(ctx->h_score[1]);
  free_dev(ctx->d_color_in), free_dev(ctx->d_color_out), free_dev(ctx->d_color_lut), free_pin(ctx->h_color);
  free_pin(ctx->h_stage);
  free_dev(ctx->map_mem), free_dev(ctx->map_tmp), free_dev(ctx->map_out), free_dev(ctx->map_n);
  free_pin(ctx->octomap), free_pin(ctx->projmap);
  if (ctx->ev_map_in) cudaEventDestroy(ctx->ev_map_in);
  if (ctx->s_map) cudaStreamDestroy(ctx->s_map);
  if (ctx->d_ticket) cudaFree(ctx->d_ticket);
  if (ctx->ev_fuse) cudaEventDestroy(ctx->ev_fuse);
  if (ctx->s_h2d) cudaStreamDestroy(ctx->s_h2d);
  if (ctx->s_compute) cudaStreamDestroy(ctx->s_compute);
  if (ctx->s_d2h) cudaStreamDestroy(ctx->s_d2h);
  cudaGetLastError();
  delete ctx;
}

int d2pc_set_q(d2pc_ctx *ctx, const double q[16]) {
  if (!ctx || !q) return D2PC_ERR_INVALID_ARG;
  memcpy(ctx->q, q, sizeof(ctx->q));
  make_qparams(ctx->q, &ctx->Q);
  return D2PC_OK;
}
int d2pc_get_q(const d2pc_ctx *ctx, double q[16]) {
  if (!ctx || !q) return D2PC_ERR_INVALID_ARG;
  memcpy(q, ctx->q, sizeof(ctx->q));
  return D2PC_OK;
}
int d2pc_set_filter_mode(d2pc_ctx *ctx, int m) {
  if (!ctx || m < 0 || m > 2 || (m == D2PC_FILTER_VOXEL && !ctx->voxel_set)) return D2PC_ERR_INVALID_ARG;
  ctx->cfg.filter_mode = m;
  return D2PC_OK;
}

void d2pc_voxel_grid_default(d2pc_voxel_grid *g) {
  if (!g) return;
  memset(g, 0, sizeof(*g));
  g->struct_size = sizeof(*g);
  g->limit_field = -1;
}
int d2pc_set_voxel_grid(d2pc_ctx *ctx, const d2pc_voxel_grid *g) {
  if (!ctx || !g || g->struct_size != sizeof(*g)) return D2PC_ERR_INVALID_ARG;
  for (float leaf : {g->leaf_x, g->leaf_y, g->leaf_z})
    if (!(std::isfinite(leaf) && leaf > 0.0f)) return D2PC_ERR_INVALID_ARG;
  if (g->limit_field < -1 || g->limit_field > 2) return D2PC_ERR_INVALID_ARG;
  if (!(g->limit_min <= g->limit_max)) return D2PC_ERR_INVALID_ARG;
  ctx->voxel = *g;
  ctx->voxel_set = true;
  return D2PC_OK;
}
int d2pc_get_voxel_grid(const d2pc_ctx *ctx, d2pc_voxel_grid *g) {
  if (!ctx || !g) return D2PC_ERR_INVALID_ARG;
  *g = ctx->voxel;
  return D2PC_OK;
}
void d2pc_radius_outlier_default(d2pc_radius_outlier *p) {
  if (!p) return;
  memset(p, 0, sizeof(*p));
  p->struct_size = sizeof(*p);
  p->min_neighbors = 1;
}
int d2pc_set_radius_outlier(d2pc_ctx *ctx, const d2pc_radius_outlier *p) {
  if (!ctx || !p || p->struct_size != sizeof(*p)) return D2PC_ERR_INVALID_ARG;
  if (!(std::isfinite(p->radius) && p->radius >= 0.0)) return D2PC_ERR_INVALID_ARG;
  ctx->ror = *p;
  return D2PC_OK;
}
int d2pc_get_radius_outlier(const d2pc_ctx *ctx, d2pc_radius_outlier *p) {
  if (!ctx || !p) return D2PC_ERR_INVALID_ARG;
  *p = ctx->ror;
  return D2PC_OK;
}
void d2pc_crop_box_default(d2pc_crop_box *b) {
  if (!b) return;
  memset(b, 0, sizeof(*b));
  b->struct_size = sizeof(*b);
  for (int a = 0; a < 3; ++a) b->min_pt[a] = -1.0f, b->max_pt[a] = 1.0f, b->transform[5 * a] = 1.0f;
}
int d2pc_set_crop_box(d2pc_ctx *ctx, const d2pc_crop_box *b) {
  if (!ctx || !b || b->struct_size != sizeof(*b)) return D2PC_ERR_INVALID_ARG;
  for (int a = 0; a < 3; ++a)  // NaN fails; +-inf bounds make a half-open box
    if (!(b->min_pt[a] <= b->max_pt[a])) return D2PC_ERR_INVALID_ARG;
  for (float t : b->transform)
    if (!std::isfinite(t)) return D2PC_ERR_INVALID_ARG;
  ctx->box = *b;
  return D2PC_OK;
}
int d2pc_get_crop_box(const d2pc_ctx *ctx, d2pc_crop_box *b) {
  if (!ctx || !b) return D2PC_ERR_INVALID_ARG;
  *b = ctx->box;
  return D2PC_OK;
}
void d2pc_cloud_transform_default(d2pc_cloud_transform *t) {
  if (!t) return;
  memset(t, 0, sizeof(*t));
  t->struct_size = sizeof(*t);
  for (int a = 0; a < 3; ++a) t->matrix[5 * a] = 1.0f;
}
int d2pc_set_cloud_transform(d2pc_ctx *ctx, const d2pc_cloud_transform *t) {
  if (!ctx || !t || t->struct_size != sizeof(*t)) return D2PC_ERR_INVALID_ARG;
  for (float m : t->matrix)
    if (!std::isfinite(m)) return D2PC_ERR_INVALID_ARG;
  ctx->xform = *t;
  return D2PC_OK;
}
int d2pc_get_cloud_transform(const d2pc_ctx *ctx, d2pc_cloud_transform *t) {
  if (!ctx || !t) return D2PC_ERR_INVALID_ARG;
  *t = ctx->xform;
  return D2PC_OK;
}
void d2pc_laser_scan_params_default(d2pc_laser_scan_params *p) {
  if (!p) return;
  memset(p, 0, sizeof(*p));
  p->struct_size = sizeof(*p);
  p->min_height = DBL_MIN, p->max_height = DBL_MAX;
  p->angle_min = -M_PI, p->angle_max = M_PI, p->angle_increment = M_PI / 180.0;
  p->scan_time = 1.0 / 30.0;
  p->range_min = 0.0, p->range_max = DBL_MAX;
  p->use_inf = 1, p->inf_epsilon = 1.0;
  p->keep_cloud = 1;
}
int d2pc_set_laser_scan(d2pc_ctx *ctx, const d2pc_laser_scan_params *p) {
  if (!ctx) return D2PC_ERR_INVALID_ARG;
  ScanPlan s;
  const int rc = scan_plan_of(p, &s);
  if (rc) return rc;
  ctx->scan = *p;
  ctx->scan_plan = s;
  return D2PC_OK;
}
int d2pc_get_laser_scan(const d2pc_ctx *ctx, d2pc_laser_scan_params *p) {
  if (!ctx || !p) return D2PC_ERR_INVALID_ARG;
  *p = ctx->scan;
  return D2PC_OK;
}
int d2pc_laser_scan_ranges(const d2pc_laser_scan_params *p, uint32_t *n) {
  ScanPlan s;
  const int rc = n ? scan_plan_of(p, &s) : D2PC_ERR_INVALID_ARG;
  if (rc) return rc;
  *n = s.msg.n_ranges;
  return D2PC_OK;
}
int d2pc_last_scan(const d2pc_ctx *ctx, d2pc_laser_scan *out) {
  if (!ctx || !out) return D2PC_ERR_INVALID_ARG;
  if (!ctx->last_scan_on) return D2PC_ERR_NOT_READY;
  *out = ctx->last_scan;
  return D2PC_OK;
}
void d2pc_occupancy_params_default(d2pc_occupancy_params *p) {
  if (!p) return;
  memset(p, 0, sizeof(*p));
  p->struct_size = sizeof(*p);
  p->resolution = 0.05;
  p->prob_hit = 0.7, p->prob_miss = 0.4;
  p->clamp_min = 0.12, p->clamp_max = 0.97;
  p->occupancy_thres = 0.5;
  p->max_range = -1.0;
  p->max_bricks = 1u << 18;
  p->keep_cloud = 1;
}
int d2pc_set_occupancy(d2pc_ctx *ctx, const d2pc_occupancy_params *p) {
  if (!ctx || !p || p->struct_size != sizeof(*p)) return D2PC_ERR_INVALID_ARG;
  if (!(std::isfinite(p->resolution) && p->resolution > 0.0)) return D2PC_ERR_INVALID_ARG;
  for (double v : {p->prob_hit, p->prob_miss, p->clamp_min, p->clamp_max, p->occupancy_thres})
    if (!(v > 0.0 && v < 1.0)) return D2PC_ERR_INVALID_ARG;
  if (!(p->prob_hit >= 0.5) || !(p->prob_miss <= 0.5) || !(p->clamp_min <= p->clamp_max)) return D2PC_ERR_INVALID_ARG;
  if (std::isnan(p->max_range) || p->max_bricks == 0 || p->max_bricks > (1u << 26)) return D2PC_ERR_INVALID_ARG;
  CU(ctx, cudaSetDevice(ctx->device));
  if (ctx->map_mem.p && p->max_bricks != ctx->occ.max_bricks) {
    // a new table: every frame submitted so far is done with the old one, which goes (map_ready makes the new one)
    CU(ctx, cudaStreamSynchronize(ctx->s_map));
    free_dev(ctx->map_mem);
  } else if (ctx->map_mem.p && p->resolution != ctx->occ.resolution) {
    CU(ctx, map_clear(ctx->map, false, ctx->s_map));
  }
  ctx->occ = *p;
  return D2PC_OK;
}
int d2pc_get_occupancy(const d2pc_ctx *ctx, d2pc_occupancy_params *p) {
  if (!ctx || !p) return D2PC_ERR_INVALID_ARG;
  *p = ctx->occ;
  return D2PC_OK;
}
int d2pc_occupancy_reset(d2pc_ctx *ctx) {
  if (!ctx) return D2PC_ERR_INVALID_ARG;
  CU(ctx, cudaSetDevice(ctx->device));
  if (ctx->map_mem.p) CU(ctx, map_clear(ctx->map, false, ctx->s_map));
  return D2PC_OK;
}

// The number of exported voxels (all known, or the occupied ones), read back with s_map idle.
static int map_export_count(d2pc_ctx *ctx, bool occupied_only, uint32_t *n) {
  *n = 0;
  if (!ctx->map_mem.p) return D2PC_OK;  // no frame since the table was made: nothing is known
  const int rc = grow_dev(ctx, ctx->map_n, 16);
  if (rc) return rc;
  CU(ctx, map_count(ctx->map, occupied_only, log_odds(ctx->occ.occupancy_thres), reinterpret_cast<uint32_t *>(ctx->map_n.p),
                    ctx->s_map));
  CU(ctx, cudaMemcpyAsync(n, ctx->map_n.p, 4, cudaMemcpyDeviceToHost, ctx->s_map));
  CU(ctx, cudaStreamSynchronize(ctx->s_map));
  return D2PC_OK;
}

// The exported voxels sorted into ctx->map_out: n float4 centres, or n packed keys then n log-odds.
static int map_export_run(d2pc_ctx *ctx, bool centres, uint32_t n) {
  int rc;
  const size_t out_bytes = centres ? (size_t)n * 16 : align_up((size_t)n * 8) + (size_t)n * 4;
  if ((rc = grow_dev(ctx, ctx->map_tmp, map_export_temp_bytes(n))) || (rc = grow_dev(ctx, ctx->map_out, out_bytes)))
    return rc;
  uint8_t *o = ctx->map_out.p;
  CU(ctx, map_export(ctx->map, centres, log_odds(ctx->occ.occupancy_thres), ctx->occ.resolution, n, ctx->map_tmp.p,
                     reinterpret_cast<uint32_t *>(ctx->map_n.p) + 1, centres ? reinterpret_cast<float4 *>(o) : nullptr,
                     centres ? nullptr : reinterpret_cast<unsigned long long *>(o),
                     centres ? nullptr : reinterpret_cast<float *>(o + align_up((size_t)n * 8)), ctx->s_map));
  return D2PC_OK;
}

int d2pc_occupancy_stats(d2pc_ctx *ctx, d2pc_occupancy_info *out) {
  if (!ctx || !out) return D2PC_ERR_INVALID_ARG;
  CU(ctx, cudaSetDevice(ctx->device));
  memset(out, 0, sizeof(*out));
  uint32_t known = 0, occupied = 0, ctr[4] = {0, 0, 0, 0};
  unsigned long long frames[2] = {0, 0};
  int rc;
  if ((rc = map_export_count(ctx, false, &known)) || (rc = map_export_count(ctx, true, &occupied))) return rc;
  out->bricks_capacity = ctx->occ.max_bricks;
  if (!ctx->map_mem.p) return D2PC_OK;
  CU(ctx, cudaMemcpyAsync(ctr, ctx->map.ctr, sizeof(ctr), cudaMemcpyDeviceToHost, ctx->s_map));
  CU(ctx, cudaMemcpyAsync(frames, ctx->map.frames, sizeof(frames), cudaMemcpyDeviceToHost, ctx->s_map));
  CU(ctx, cudaStreamSynchronize(ctx->s_map));
  out->frames_inserted = frames[0], out->frames_dropped = frames[1];
  out->known_voxels = known, out->occupied_voxels = occupied;
  out->bricks_used = ctr[0];
  return D2PC_OK;
}

int d2pc_occupancy_centers(d2pc_ctx *ctx, uint8_t *dst, size_t cap, d2pc_cloud *out) {
  if (!ctx || !out) return D2PC_ERR_INVALID_ARG;
  CU(ctx, cudaSetDevice(ctx->device));
  uint32_t n = 0;
  int rc = map_export_count(ctx, true, &n);
  if (rc) return rc;
  if (cap < (size_t)n * 16 || (n && !dst)) {
    fill_cloud(ctx, nullptr, n, true, out);
    return D2PC_ERR_BUFFER_TOO_SMALL;
  }
  if (n && (rc = map_export_run(ctx, true, n))) return rc;
  if (n) CU(ctx, cudaMemcpyAsync(dst, ctx->map_out.p, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->s_map));
  CU(ctx, cudaStreamSynchronize(ctx->s_map));
  fill_cloud(ctx, dst, n, true, out);
  return D2PC_OK;
}

int d2pc_occupancy_voxels(d2pc_ctx *ctx, uint64_t *keys, float *log_odds_out, uint64_t cap, uint64_t *n_out) {
  if (!ctx || !n_out) return D2PC_ERR_INVALID_ARG;
  CU(ctx, cudaSetDevice(ctx->device));
  uint32_t n = 0;
  int rc = map_export_count(ctx, false, &n);
  if (rc) return rc;
  *n_out = n;
  if (cap < n || (n && (!keys || !log_odds_out))) return D2PC_ERR_BUFFER_TOO_SMALL;
  if (n && (rc = map_export_run(ctx, false, n))) return rc;
  if (n) {
    CU(ctx, cudaMemcpyAsync(keys, ctx->map_out.p, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->s_map));
    CU(ctx, cudaMemcpyAsync(log_odds_out, ctx->map_out.p + align_up((size_t)n * 8), (size_t)n * 4,
                            cudaMemcpyDeviceToHost, ctx->s_map));
  }
  CU(ctx, cudaStreamSynchronize(ctx->s_map));
  return D2PC_OK;
}

int d2pc_occupancy_octomap(d2pc_ctx *ctx, int binary, d2pc_octomap *out) {
  if (!ctx || !out || binary < 0 || binary > 1) return D2PC_ERR_INVALID_ARG;
  CU(ctx, cudaSetDevice(ctx->device));
  uint32_t n = 0;
  int rc = map_export_count(ctx, false, &n);
  if (rc) return rc;
  unsigned long long records = 0;
  if (n) {
    if ((rc = grow_dev(ctx, ctx->map_tmp, octomap_temp_bytes(n)))) return rc;
    CU(ctx, octomap_plan(ctx->map, n, binary, ctx->map_tmp.p, reinterpret_cast<uint32_t *>(ctx->map_n.p) + 1,
                         &records, ctx->s_map));
    CU(ctx, cudaStreamSynchronize(ctx->s_map));  // the size of the stream sizes the result
  }
  const size_t bytes = records * (binary ? 2 : 5);
  if (bytes && (rc = grow_dev(ctx, ctx->map_out, octomap_out_bytes(records, binary)))) return rc;
  if (bytes > ctx->octomap.cap) {
    // a new buffer before the old one goes, so a failed allocation leaves the last result as it was
    void *p = nullptr;
    const size_t cap = round_up(bytes, 1 << 16);
    CU(ctx, pinned_alloc(&p, cap));
    free_pin(ctx->octomap);
    ctx->octomap.p = static_cast<uint8_t *>(p), ctx->octomap.cap = cap;
  }
  if (bytes) {
    CU(ctx, octomap_emit(ctx->map, n, binary, log_odds(ctx->occ.occupancy_thres), ctx->map_tmp.p, records,
                         ctx->map_out.p, ctx->s_map));
    CU(ctx, cudaMemcpyAsync(ctx->octomap.p, ctx->map_out.p, bytes, cudaMemcpyDeviceToHost, ctx->s_map));
    CU(ctx, cudaStreamSynchronize(ctx->s_map));
  }
  out->data = bytes ? ctx->octomap.p : nullptr;
  out->size = bytes;
  out->resolution = ctx->occ.resolution;
  out->binary = binary;
  return D2PC_OK;
}

void d2pc_projected_map_params_default(d2pc_projected_map_params *p) {
  if (!p) return;
  memset(p, 0, sizeof(*p));
  p->struct_size = sizeof(*p);
  p->occupancy_min_z = -DBL_MAX, p->occupancy_max_z = DBL_MAX;
}

int d2pc_occupancy_projected_map(d2pc_ctx *ctx, const d2pc_projected_map_params *p, d2pc_grid_map *out) {
  if (!ctx || !p || !out || p->struct_size != sizeof(*p)) return D2PC_ERR_INVALID_ARG;
  if (std::isnan(p->occupancy_min_z) || std::isnan(p->occupancy_max_z)) return D2PC_ERR_INVALID_ARG;
  for (double v : {p->min_x_size, p->min_y_size})
    if (!(std::isfinite(v) && v >= 0.0)) return D2PC_ERR_INVALID_ARG;
  CU(ctx, cudaSetDevice(ctx->device));
  uint32_t n = 0;
  int rc = map_export_count(ctx, false, &n);
  if (rc) return rc;
  const double res = ctx->occ.resolution;
  ProjGrid g{};
  size_t bytes = 0;
  if (n) {
    if ((rc = grow_dev(ctx, ctx->map_tmp, octomap_temp_bytes(n))) || (rc = grow_dev(ctx, ctx->map_n, 64))) return rc;
    unsigned long long ext[6];
    CU(ctx, projmap_extent(ctx->map, n, res, ctx->map_tmp.p, reinterpret_cast<uint32_t *>(ctx->map_n.p) + 1,
                           reinterpret_cast<unsigned long long *>(ctx->map_n.p + 16), ext, ctx->s_map));
    CU(ctx, cudaStreamSynchronize(ctx->s_map));  // the tree's extent sizes the grid
    if (!projmap_grid(ext, res, p->min_x_size, p->min_y_size, &g)) return D2PC_ERR_BAD_DIMS;
    bytes = (size_t)g.width * g.height;
    if ((rc = grow_dev(ctx, ctx->map_out, projmap_cells_bytes(g)))) return rc;
    if (bytes > ctx->projmap.cap) {
      // a new buffer before the old one goes, so a failed allocation leaves the last result as it was
      void *q = nullptr;
      const size_t cap = round_up(bytes, 1 << 16);
      CU(ctx, pinned_alloc(&q, cap));
      free_pin(ctx->projmap);
      ctx->projmap.p = static_cast<uint8_t *>(q), ctx->projmap.cap = cap;
    }
    CU(ctx, projmap_fill(ctx->map, n, res, p->occupancy_min_z, p->occupancy_max_z,
                         log_odds(ctx->occ.occupancy_thres), ctx->map_tmp.p, g, ctx->map_out.p, ctx->s_map));
    CU(ctx, cudaMemcpyAsync(ctx->projmap.p, ctx->map_out.p, bytes, cudaMemcpyDeviceToHost, ctx->s_map));
    CU(ctx, cudaStreamSynchronize(ctx->s_map));
  }
  out->data = bytes ? reinterpret_cast<const int8_t *>(ctx->projmap.p) : nullptr;
  out->width = g.width, out->height = g.height;
  out->resolution = (float)res;
  out->origin_x = g.origin[0], out->origin_y = g.origin[1];
  return D2PC_OK;
}

int d2pc_set_arith_mode(d2pc_ctx *ctx, int m) {
  if (!ctx || m < 0 || m > 1) return D2PC_ERR_INVALID_ARG;
  ctx->cfg.arith_mode = m;
  return D2PC_OK;
}
int d2pc_set_tuning(d2pc_ctx *ctx, const char *key, int value) {
  if (!ctx || !key) return D2PC_ERR_INVALID_ARG;
  const std::string k(key);
  if (k == "rows_per_unit") ctx->rows_per_unit = value;
  else if (k == "ctas_per_sm") ctx->ctas_per_sm = value;
  else if (k == "median_strip") ctx->median_strip = value;
  else if (k == "median_variant") ctx->median_variant = value;
  else if (k == "force_scalar") ctx->force_scalar = value != 0;
  else if (k == "force_generic") ctx->force_generic = value != 0;
  else if (k == "force_park" || k == "compact_variant") ctx->compact_variant = value;
  else if (k == "exact_variant") ctx->exact_variant = value;
  else if (k == "zero_numer") ctx->zero_numer = value;
  else if (k == "fuse_median") ctx->fuse_median = value;
  else if (k == "direct_out") ctx->direct_out = value;
  else if (k == "prefetch_dist") ctx->prefetch_dist = value;
  else if (k == "crop_load") ctx->crop_load = value;
  else if (k == "crop_probe") ctx->crop_probe = value;
  else if (k == "median_ksize") {
    if (value < 1 || value > 15 || !(value & 1)) return D2PC_ERR_INVALID_ARG;
    ctx->cfg.median_ksize = value;
  } else if (k == "border") {
    if (value < 0) return D2PC_ERR_INVALID_ARG;
    ctx->cfg.border = value;
  } else if (k == "offset_x") ctx->cfg.offset_x = value;
  else if (k == "offset_y") ctx->cfg.offset_y = value;
  else if (k == "fuse_rule") {
    if (value < 0 || value > 7) return D2PC_ERR_INVALID_ARG;
    ctx->cfg.fuse_rule = value;
  } else if (k == "fuse_median_ksize") {
    if (value < 1 || value > 15 || !(value & 1)) return D2PC_ERR_INVALID_ARG;
    ctx->cfg.fuse_median_ksize = value;
  } else if (k == "fuse_crop_left") ctx->cfg.fuse_crop_left = value;
  else if (k == "fuse_crop_right") ctx->cfg.fuse_crop_right = value;
  else if (k == "fuse_crop_top") ctx->cfg.fuse_crop_top = value;
  else if (k == "fuse_crop_bottom") ctx->cfg.fuse_crop_bottom = value;
  else return D2PC_ERR_INVALID_ARG;
  return D2PC_OK;
}

// ---------------------------------------------------------------------------
// host-buffer entry points
// ---------------------------------------------------------------------------
int d2pc_submit_mono8(d2pc_ctx *ctx, int slot, const uint8_t *data, uint32_t w, uint32_t h, uint32_t step) {
  return submit_common(ctx, slot, data, w, h, step, false, nullptr, 0, false);
}
int d2pc_submit_f32(d2pc_ctx *ctx, int slot, const float *disp, uint32_t w, uint32_t h, uint32_t step) {
  return submit_common(ctx, slot, disp, w, h, step, true, nullptr, 0, false);
}

int d2pc_wait(d2pc_ctx *ctx, int slot, d2pc_cloud *out) {
  if (!ctx || slot < 0 || slot >= (int)ctx->slots.size()) return D2PC_ERR_INVALID_ARG;
  Slot &s = ctx->slots[slot];
  if (!s.pending) return D2PC_ERR_NOT_READY;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaEventSynchronize(s.ev_d2h));
  const Submission &sub = s.sub;
  const CloudPlan &p = sub.p;
  const uint64_t n = kept_points(p, s.h_count);
  if (p.counted && sub.user_dst && sub.user_cap < n * 16) {
    s.pending = false;
    ctx->last_scan_on = false;  // no cloud is returned, so there is no last scan either
    return D2PC_ERR_BUFFER_TOO_SMALL;
  }
  // a counted cloud and a late copy leave the device here: the copy is synchronous anyway, so it goes straight to
  // the caller's buffer, page-locked or not
  const bool copy_here = p.counted || sub.late_copy;
  uint8_t *const dst = sub.user_dst ? sub.user_dst : s.h_out.p;
  if (copy_here && n) {
    CU(ctx, cudaMemcpyAsync(dst, s.d_out.p, n * 16, cudaMemcpyDeviceToHost, ctx->s_d2h));
    CU(ctx, cudaStreamSynchronize(ctx->s_d2h));
  }
  // otherwise a page-locked caller buffer already holds the cloud; a pageable one is filled from h_out
  if (sub.user_dst && !sub.user_pinned && !copy_here && n) memcpy(sub.user_dst, s.h_out.p, n * 16);
  s.pending = false;
  if (ctx->cfg.verbose) printf("Cloud size: %llu\n", (unsigned long long)n);  // cpp:82
  if (out) {
    if (cloud_out(p)) fill_cloud(ctx, dst, n, cloud_is_dense(p, s.h_count), out);
    else fill_cloud(ctx, nullptr, 0, true, out);
  }
  // d2pc_last_scan's answer from now on: the scan of the cloud just returned
  ctx->last_scan_on = p.scan.on;
  ctx->last_scan = p.scan.msg;
  ctx->last_scan.ranges = reinterpret_cast<const float *>(s.h_ranges.p);
  return D2PC_OK;
}

int d2pc_submit_mono8_into(d2pc_ctx *ctx, int slot, const uint8_t *data, uint32_t w, uint32_t h, uint32_t step,
                           uint8_t *dst, size_t cap) {
  if (!dst) return D2PC_ERR_INVALID_ARG;
  return submit_common(ctx, slot, data, w, h, step, false, dst, cap, false);
}
int d2pc_submit_f32_into(d2pc_ctx *ctx, int slot, const float *disp, uint32_t w, uint32_t h, uint32_t step,
                         uint8_t *dst, size_t cap) {
  if (!dst) return D2PC_ERR_INVALID_ARG;
  return submit_common(ctx, slot, disp, w, h, step, true, dst, cap, false);
}
int d2pc_process_mono8_into(d2pc_ctx *ctx, const uint8_t *data, uint32_t w, uint32_t h, uint32_t step, uint8_t *dst,
                            size_t cap, d2pc_cloud *out) {
  if (!dst) return D2PC_ERR_INVALID_ARG;
  int rc = submit_common(ctx, 0, data, w, h, step, false, dst, cap, true);
  return rc ? rc : d2pc_wait(ctx, 0, out);
}
int d2pc_process_f32_into(d2pc_ctx *ctx, const float *disp, uint32_t w, uint32_t h, uint32_t step, uint8_t *dst,
                          size_t cap, d2pc_cloud *out) {
  if (!dst) return D2PC_ERR_INVALID_ARG;
  int rc = submit_common(ctx, 0, disp, w, h, step, true, dst, cap, true);
  return rc ? rc : d2pc_wait(ctx, 0, out);
}

int d2pc_process_mono8(d2pc_ctx *ctx, const uint8_t *data, uint32_t w, uint32_t h, uint32_t step, d2pc_cloud *out) {
  if (!out) return D2PC_ERR_INVALID_ARG;
  int rc = submit_common(ctx, 0, data, w, h, step, false, nullptr, 0, true);
  return rc ? rc : d2pc_wait(ctx, 0, out);
}
int d2pc_process_f32(d2pc_ctx *ctx, const float *disp, uint32_t w, uint32_t h, uint32_t step, d2pc_cloud *out) {
  if (!out) return D2PC_ERR_INVALID_ARG;
  int rc = submit_common(ctx, 0, disp, w, h, step, true, nullptr, 0, true);
  return rc ? rc : d2pc_wait(ctx, 0, out);
}

// ---- per-call timing (SURVEY.md section 5: "per-call timing struct returned through the C ABI") ---------------
int d2pc_set_timing(d2pc_ctx *ctx, int enable) {
  if (!ctx) return D2PC_ERR_INVALID_ARG;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaDeviceSynchronize());  // no slot may be in flight while its events are replaced
  const unsigned flags = enable ? cudaEventDefault : cudaEventDisableTiming;
  for (auto &s : ctx->slots) {
    s.pending = false;
    s.timed = false;
    cudaEvent_t *evs[4] = {&s.ev_start, &s.ev_h2d, &s.ev_kernel, &s.ev_d2h};
    for (cudaEvent_t *e : evs) {
      if (*e) CU(ctx, cudaEventDestroy(*e));
      *e = nullptr;
      CU(ctx, cudaEventCreateWithFlags(e, flags));
    }
  }
  ctx->timing = enable != 0;
  return D2PC_OK;
}

int d2pc_slot_timing(d2pc_ctx *ctx, int slot, d2pc_timing *out) {
  if (!ctx || !out || slot < 0 || slot >= (int)ctx->slots.size()) return D2PC_ERR_INVALID_ARG;
  Slot &s = ctx->slots[slot];
  if (!ctx->timing || !s.timed || s.pending) return D2PC_ERR_NOT_READY;  // enable timing, submit, wait, then ask
  CU(ctx, cudaSetDevice(ctx->device));
  float h2d = 0.f, ker = 0.f, d2h = 0.f, tot = 0.f;
  CU(ctx, cudaEventElapsedTime(&h2d, s.ev_start, s.ev_h2d));
  CU(ctx, cudaEventElapsedTime(&ker, s.ev_h2d, s.ev_kernel));
  CU(ctx, cudaEventElapsedTime(&d2h, s.ev_kernel, s.ev_d2h));
  CU(ctx, cudaEventElapsedTime(&tot, s.ev_start, s.ev_d2h));
  out->h2d_us = h2d * 1e3f, out->kernels_us = ker * 1e3f, out->d2h_us = d2h * 1e3f, out->total_us = tot * 1e3f;
  out->points = kept_points(s.sub.p, s.h_count);
  return D2PC_OK;
}

int d2pc_host_alloc(void **ptr, size_t bytes) {
  if (!ptr) return D2PC_ERR_INVALID_ARG;
  *ptr = nullptr;
  cudaError_t e = pinned_alloc(ptr, bytes ? bytes : 1);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? D2PC_ERR_NOMEM : D2PC_ERR_CUDA;
  }
  return D2PC_OK;
}
int d2pc_host_free(void *ptr) {
  if (!ptr) return D2PC_OK;
  g_host_gen.fetch_add(1, std::memory_order_acq_rel);  // contexts forget what they knew about this address
  return pinned_free(ptr) == cudaSuccess ? D2PC_OK : D2PC_ERR_CUDA;
}
int d2pc_host_register(void *ptr, size_t bytes) {
  if (!ptr || !bytes) return D2PC_ERR_INVALID_ARG;
  g_host_gen.fetch_add(1, std::memory_order_acq_rel);  // a pageable address becomes pinned: cached answers are stale
  cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterDefault);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? D2PC_ERR_NOMEM : D2PC_ERR_CUDA;
  }
  return D2PC_OK;
}
int d2pc_host_unregister(void *ptr) {
  if (!ptr) return D2PC_OK;
  g_host_gen.fetch_add(1, std::memory_order_acq_rel);
  if (cudaHostUnregister(ptr) != cudaSuccess) {
    cudaGetLastError();
    return D2PC_ERR_CUDA;
  }
  return D2PC_OK;
}

int d2pc_process_stream(d2pc_ctx *ctx, const void *frames, uint64_t n_frames, size_t frame_stride, uint64_t ring_len,
                        int is_f32, uint32_t w, uint32_t h, uint32_t step, d2pc_cloud_sink sink, void *user) {
  if (!ctx || (!frames && n_frames)) return D2PC_ERR_INVALID_ARG;
  auto submit = [&](const uint8_t *f, int slot) {
    return submit_common(ctx, slot, f, w, h, step, is_f32 != 0, nullptr, 0, false);
  };
  return run_ring(ctx, static_cast<const uint8_t *>(frames), n_frames, frame_stride, ring_len, submit, sink, user);
}

// ---------------------------------------------------------------------------
// device-resident entry points
// ---------------------------------------------------------------------------
static int reproject_device_common(d2pc_ctx *ctx, const void *d_in, bool is_f32, uint32_t n_frames, uint32_t w,
                                   uint32_t h, size_t step, size_t frame_stride, uint8_t *d_points,
                                   size_t points_stride, uint32_t *d_counts) {
  if (!ctx || !d_in || !d_points) return D2PC_ERR_INVALID_ARG;
  const int esz = is_f32 ? 4 : 1;
  if (w == 0 || h == 0 || step < (size_t)w * esz || (n_frames > 1 && frame_stride < step * h))
    return D2PC_ERR_BAD_DIMS;
  const CloudPlan p = plan_cloud(ctx, w, h);
  const uint64_t n = p.n;
  if (n * 16 > 0xffffffffull) return D2PC_ERR_BAD_DIMS;  // per-frame counts and PointCloud2.row_step are uint32
  if (reinterpret_cast<uintptr_t>(d_points) % 16 || points_stride % 16 || (n_frames > 1 && points_stride < n * 16))
    return D2PC_ERR_BAD_DIMS;
  if (p.counted && !d_counts) return D2PC_ERR_INVALID_ARG;
  if (n_frames == 0) return D2PC_OK;  // an empty batch: nothing to launch (and no size below may wrap)
  CU(ctx, cudaSetDevice(ctx->device));
  // a batch of more than kCloudMaxPoints crop points runs the cloud stages in chunks
  const uint32_t chunk = p.n_stages ? frames_per_chunk(n_frames, n) : n_frames;
  FrameBatch in{static_cast<const uint8_t *>(d_in), is_f32, chunk, w, h, step, frame_stride};
  int rc = grow_stages(ctx, ctx->batch, p, in, ctx->s_compute, true);
  if (rc) return rc;
  for (uint32_t f0 = 0; f0 < n_frames; f0 += chunk) {
    in.data = static_cast<const uint8_t *>(d_in) + f0 * frame_stride;
    in.n_frames = std::min(chunk, n_frames - f0);
    if ((rc = enqueue_kernels(ctx, p, in, ctx->batch,
                              {d_points + f0 * points_stride, points_stride, d_counts ? d_counts + f0 : nullptr},
                              nullptr, ctx->d_ticket, ctx->s_compute, nullptr)))
      return rc;
  }
  return D2PC_OK;
}

// The argument rules of the stages that run alone on clouds already on the device: n_frames clouds of n_max points
// at d_in, in_stride bytes apart, and per frame out_bytes of output at d_out, out_stride bytes apart, both
// out_align-aligned (16 for a cloud, 4 for laser-scan ranges; no output: null, 0, 0, 1).  in_place: the output may
// also be exactly the input.
static int check_cloud_batch(const uint8_t *d_in, uint32_t n_frames, uint32_t n_max, size_t in_stride,
                             const void *d_out, size_t out_stride, uint64_t out_bytes, size_t out_align,
                             bool in_place) {
  const uint64_t bytes = (uint64_t)n_max * 16;
  if (bytes > 0xffffffffull) return D2PC_ERR_BAD_DIMS;  // per-frame counts and PointCloud2.row_step are uint32
  if (reinterpret_cast<uintptr_t>(d_in) % 16 || in_stride % 16 || reinterpret_cast<uintptr_t>(d_out) % out_align ||
      out_stride % out_align || (n_frames > 1 && (in_stride < bytes || out_stride < out_bytes)))
    return D2PC_ERR_BAD_DIMS;
  if (n_frames == 0 || out_bytes == 0 || (in_place && d_in == d_out && in_stride == out_stride)) return D2PC_OK;
  // kept points are copied from the input after every flag is known: the two must not share bytes
  const uintptr_t in0 = reinterpret_cast<uintptr_t>(d_in), out0 = reinterpret_cast<uintptr_t>(d_out);
  const uint64_t in_end = in0 + (uint64_t)(n_frames - 1) * in_stride + bytes;
  const uint64_t out_end = out0 + (uint64_t)(n_frames - 1) * out_stride + out_bytes;
  if (bytes && in0 < out_end && out0 < in_end) return D2PC_ERR_INVALID_ARG;
  return D2PC_OK;
}

// One cloud stage alone on clouds already on the device (d2pc_radius_outlier_device, d2pc_crop_box_device).
static int cloud_stage_device(d2pc_ctx *ctx, CloudStage st, bool on, const uint8_t *d_in, uint32_t n_frames,
                              uint32_t n_max, size_t in_stride, const uint32_t *d_in_counts, uint8_t *d_out,
                              size_t out_stride, uint32_t *d_out_counts) {
  if (!ctx || !d_in || !d_out || !d_out_counts || !on) return D2PC_ERR_INVALID_ARG;
  const int rc0 = check_cloud_batch(d_in, n_frames, n_max, in_stride, d_out, out_stride, (uint64_t)n_max * 16, 16, false);
  if (rc0 || n_frames == 0) return rc0;
  CU(ctx, cudaSetDevice(ctx->device));
  const size_t need = stage_scratch_bytes(st, frames_per_chunk(n_frames, n_max), n_max);
  if (need > ctx->batch.stage.cap) {
    CU(ctx, cudaStreamSynchronize(ctx->s_compute));
    const int rc = grow_dev(ctx, ctx->batch.stage, need);
    if (rc) return rc;
  }
  return for_each_chunk(d_in, n_frames, n_max, in_stride, d_in_counts, [&](uint32_t f0, const CloudSrc &in) -> int {
    return enqueue_stage(ctx, st, in, {d_out + f0 * out_stride, out_stride, d_out_counts + f0}, nullptr,
                         ctx->batch.stage.p, ctx->s_compute);
  });
}

int d2pc_radius_outlier_device(d2pc_ctx *ctx, const uint8_t *d_in, uint32_t n_frames, uint32_t n_max,
                               size_t in_stride, const uint32_t *d_in_counts, uint8_t *d_out, size_t out_stride,
                               uint32_t *d_out_counts) {
  return cloud_stage_device(ctx, CloudStage::ror, ctx && ctx->ror.radius > 0.0, d_in, n_frames, n_max, in_stride,
                            d_in_counts, d_out, out_stride, d_out_counts);
}

int d2pc_crop_box_device(d2pc_ctx *ctx, const uint8_t *d_in, uint32_t n_frames, uint32_t n_max, size_t in_stride,
                         const uint32_t *d_in_counts, uint8_t *d_out, size_t out_stride, uint32_t *d_out_counts) {
  return cloud_stage_device(ctx, CloudStage::box, ctx && ctx->box.enabled, d_in, n_frames, n_max, in_stride,
                            d_in_counts, d_out, out_stride, d_out_counts);
}

int d2pc_cloud_transform_device(d2pc_ctx *ctx, const uint8_t *d_in, uint32_t n_frames, uint32_t n_max,
                                size_t in_stride, const uint32_t *d_in_counts, uint8_t *d_out, size_t out_stride,
                                uint32_t *d_out_counts, const float *d_transforms) {
  if (!ctx || !d_in || !d_out || (!d_transforms && !ctx->xform.enabled)) return D2PC_ERR_INVALID_ARG;
  const int rc0 = check_cloud_batch(d_in, n_frames, n_max, in_stride, d_out, out_stride, (uint64_t)n_max * 16, 16, true);
  if (rc0 || n_frames == 0) return rc0;
  CU(ctx, cudaSetDevice(ctx->device));
  const CloudTransformParams t = transform_params(ctx);
  return for_each_chunk(d_in, n_frames, n_max, in_stride, d_in_counts, [&](uint32_t f0, const CloudSrc &in) -> int {
    const CloudDst out{d_out + f0 * out_stride, out_stride, d_out_counts ? d_out_counts + f0 : nullptr};
    int nl = 0;
    CU(ctx, launch_cloud_transform(in, out, t, d_transforms ? d_transforms + 12 * (size_t)f0 : nullptr, ctx->s_compute,
                                   &nl));
    ctx->launches += nl;
    return D2PC_OK;
  });
}

int d2pc_laser_scan_device(d2pc_ctx *ctx, const uint8_t *d_in, uint32_t n_frames, uint32_t n_max, size_t in_stride,
                           const uint32_t *d_in_counts, float *d_ranges, size_t ranges_stride) {
  if (!ctx || !d_in || !d_ranges || !ctx->scan.enabled) return D2PC_ERR_INVALID_ARG;
  const LaserScanParams &p = ctx->scan_plan.p;
  const uint64_t rbytes = (uint64_t)p.n * 4;
  const int rc0 = check_cloud_batch(d_in, n_frames, n_max, in_stride, d_ranges, ranges_stride, rbytes, 4, false);
  if (rc0 || n_frames == 0 || p.n == 0) return rc0;
  CU(ctx, cudaSetDevice(ctx->device));
  return for_each_chunk(d_in, n_frames, n_max, in_stride, d_in_counts, [&](uint32_t f0, const CloudSrc &in) -> int {
    int nl = 0;
    CU(ctx, launch_laser_scan(in, p, reinterpret_cast<float *>(reinterpret_cast<uint8_t *>(d_ranges) + f0 * ranges_stride),
                              ranges_stride, ctx->s_compute, &nl));
    ctx->launches += nl;
    return D2PC_OK;
  });
}

int d2pc_occupancy_insert_device(d2pc_ctx *ctx, const uint8_t *d_in, uint32_t n_frames, uint32_t n_max,
                                 size_t in_stride, const uint32_t *d_in_counts, const float *origins) {
  if (!ctx || !d_in || !origins || !ctx->occ.enabled) return D2PC_ERR_INVALID_ARG;
  const int rc0 = check_cloud_batch(d_in, n_frames, n_max, in_stride, nullptr, 0, 0, 1, false);
  if (rc0 || n_frames == 0) return rc0;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaEventRecord(ctx->ev_map_in, ctx->s_compute));
  // one frame per map step: a frame of at most 2^28 points is always within kCloudMaxPoints, so no chunk spans frames
  for (uint32_t f = 0; f < n_frames; ++f) {
    const CloudSrc in{d_in + (size_t)f * in_stride, in_stride, d_in_counts ? d_in_counts + f : nullptr, 1, n_max};
    const int rc = enqueue_map(ctx, map_update(ctx, origins + 3 * (size_t)f), in, f == 0 ? ctx->ev_map_in : nullptr);
    if (rc) return rc;
  }
  return D2PC_OK;
}

int d2pc_reproject_f32_device(d2pc_ctx *ctx, const float *d_disp, uint32_t n_frames, uint32_t w, uint32_t h,
                              size_t step, size_t frame_stride, uint8_t *d_points, size_t points_stride,
                              uint32_t *d_counts) {
  if (step % 4 || frame_stride % 4 || reinterpret_cast<uintptr_t>(d_disp) % 4) return D2PC_ERR_BAD_DIMS;
  return reproject_device_common(ctx, d_disp, true, n_frames, w, h, step, frame_stride, d_points, points_stride,
                                 d_counts);
}
int d2pc_reproject_mono8_device(d2pc_ctx *ctx, const uint8_t *d_img, uint32_t n_frames, uint32_t w, uint32_t h,
                                size_t step, size_t frame_stride, uint8_t *d_points, size_t points_stride,
                                uint32_t *d_counts) {
  return reproject_device_common(ctx, d_img, false, n_frames, w, h, step, frame_stride, d_points, points_stride,
                                 d_counts);
}

int d2pc_median_u8_device(d2pc_ctx *ctx, const uint8_t *d_src, uint32_t w, uint32_t h, size_t src_step,
                          uint8_t *d_dst, size_t dst_step, int ksize) {
  if (!ctx || !d_src || !d_dst) return D2PC_ERR_INVALID_ARG;
  if (w == 0 || h == 0 || src_step < w || dst_step < w) return D2PC_ERR_BAD_DIMS;
  if (ksize < 3 || ksize > 15 || !(ksize & 1)) return D2PC_ERR_INVALID_ARG;
  CU(ctx, cudaSetDevice(ctx->device));
  MedianLaunch M;
  M.src = d_src, M.dst = d_dst;
  M.src_step = src_step, M.dst_step = dst_step;
  M.width = (int)w, M.height = (int)h;
  M.ox0 = 0, M.oy0 = 0, M.ow = (int)w, M.oh = (int)h;
  M.ksize = ksize;
  M.sm_count = ctx->sm_count;
  M.strip_rows = ctx->median_strip;
  M.variant = ctx->median_variant;
  int nl = 0;
  CU(ctx, launch_median_u8(M, ctx->s_compute, &nl));
  ctx->launches += nl;
  return D2PC_OK;
}

void *d2pc_compute_stream(d2pc_ctx *ctx) { return ctx ? (void *)ctx->s_compute : nullptr; }
int d2pc_sync(d2pc_ctx *ctx) {
  if (!ctx) return D2PC_ERR_INVALID_ARG;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaStreamSynchronize(ctx->s_h2d));
  CU(ctx, cudaStreamSynchronize(ctx->s_compute));
  for (auto &s : ctx->slots)
    if (s.s_kern) CU(ctx, cudaStreamSynchronize(s.s_kern));
  CU(ctx, cudaStreamSynchronize(ctx->s_d2h));
  CU(ctx, cudaStreamSynchronize(ctx->s_map));
  return D2PC_OK;
}
uint64_t d2pc_launch_count(const d2pc_ctx *ctx) { return ctx ? ctx->launches : 0; }

// ---------------------------------------------------------------------------
// depth_map_fusion
// ---------------------------------------------------------------------------
int d2pc_fuse_geometry(const d2pc_ctx *ctx, uint32_t w, uint32_t h, int rect1[4], int rect2[4], int rectc[4],
                       int dims[3]) {
  if (!ctx) return D2PC_ERR_INVALID_ARG;
  FuseGeometry g;
  const d2pc_config &c = ctx->cfg;
  const bool ok = fuse_geometry((int)w, (int)h, c.offset_x, c.offset_y, c.fuse_crop_left, c.fuse_crop_right,
                                c.fuse_crop_top, c.fuse_crop_bottom, &g);
  if (rect1) memcpy(rect1, g.r1, sizeof(g.r1));
  if (rect2) memcpy(rect2, g.r2, sizeof(g.r2));
  if (rectc) memcpy(rectc, g.rc, sizeof(g.rc));
  if (dims) dims[0] = g.n, dims[1] = g.out_w, dims[2] = g.out_h;
  return ok ? D2PC_OK : D2PC_ERR_GEOMETRY;
}

static int fuse_device_impl(d2pc_ctx *ctx, const uint8_t *d1, const uint8_t *d2, const uint8_t *s1, const uint8_t *s2,
                            uint32_t w, uint32_t h, size_t step, uint8_t *d_fused, uint8_t *d_combined,
                            FuseGeometry *g_out, bool scores_cropped = false, DevBuf *container = nullptr,
                            cudaStream_t stream = nullptr) {
  if (!stream) stream = ctx->s_compute;
  const d2pc_config &c = ctx->cfg;
  FuseGeometry g;
  if (!fuse_geometry((int)w, (int)h, c.offset_x, c.offset_y, c.fuse_crop_left, c.fuse_crop_right, c.fuse_crop_top,
                     c.fuse_crop_bottom, &g))
    return D2PC_ERR_GEOMETRY;
  int rc;
  DevBuf &cont = container ? *container : ctx->d_container;
  if ((size_t)g.nc * g.nc > cont.cap) {
    CU(ctx, cudaStreamSynchronize(ctx->s_compute));
    if ((rc = grow_dev(ctx, cont, (size_t)g.nc * g.nc))) return rc;
  }
  FuseLaunch L;
  L.d1 = d1, L.d2 = d2, L.s1 = s1, L.s2 = s2;
  L.step = step;
  L.width = (int)w, L.height = (int)h;
  L.g = g;
  L.rule = c.fuse_rule;
  L.scores_cropped = scores_cropped;
  L.container = cont.p;
  L.combined = d_combined;
  int nl = 0;
  CU(ctx, launch_fuse_merge(L, stream, &nl));
  ctx->launches += nl;
  if (c.fuse_median_ksize > 1) {
    // :124 medianBlur on the container ROI (its edge is the replicate border), then :130 cropMat -- produced as
    // one kernel that only evaluates the pixels that survive the trim.
    MedianLaunch M;
    M.src = cont.p;
    M.src_step = (size_t)g.nc;
    M.width = g.nc, M.height = g.nc;
    M.ox0 = g.out_x, M.oy0 = g.out_y, M.ow = g.out_w, M.oh = g.out_h;
    M.dst_step = (size_t)g.out_w;
    // dst is addressed with container coordinates: bias the pointer so (out_y, out_x) lands on d_fused[0]
    M.dst = reinterpret_cast<uint8_t *>(reinterpret_cast<uintptr_t>(d_fused) - ((size_t)g.out_y * g.out_w + g.out_x));
    M.ksize = c.fuse_median_ksize;
    M.sm_count = ctx->sm_count;
    M.variant = ctx->median_variant;
    CU(ctx, launch_median_u8(M, stream, &nl));
    ctx->launches += nl;
  } else {
    CU(ctx, cudaMemcpy2DAsync(d_fused, g.out_w, cont.p + (size_t)g.out_y * g.nc + g.out_x, g.nc, g.out_w,
                              g.out_h, cudaMemcpyDeviceToDevice, stream));
  }
  if (g_out) *g_out = g;
  return D2PC_OK;
}

int d2pc_fuse_device(d2pc_ctx *ctx, const uint8_t *d_d1, const uint8_t *d_d2, const uint8_t *d_s1,
                     const uint8_t *d_s2, uint32_t w, uint32_t h, size_t step, uint8_t *d_fused,
                     uint8_t *d_combined) {
  if (!ctx || !d_d1 || !d_d2 || !d_s1 || !d_s2 || !d_fused) return D2PC_ERR_INVALID_ARG;
  if (w == 0 || h == 0 || step < w) return D2PC_ERR_BAD_DIMS;
  CU(ctx, cudaSetDevice(ctx->device));
  return fuse_device_impl(ctx, d_d1, d_d2, d_s1, d_s2, w, h, step, d_fused, d_combined, nullptr);
}

int d2pc_fuse_preprocessed_device(d2pc_ctx *ctx, const uint8_t *d_d1, const uint8_t *d_d2, const uint8_t *d_s1c,
                                  const uint8_t *d_s2c, uint32_t w, uint32_t h, size_t step, uint8_t *d_fused,
                                  uint8_t *d_combined) {
  if (!ctx || !d_d1 || !d_d2 || !d_s1c || !d_s2c || !d_fused) return D2PC_ERR_INVALID_ARG;
  if (w == 0 || h == 0 || step < w) return D2PC_ERR_BAD_DIMS;
  CU(ctx, cudaSetDevice(ctx->device));
  return fuse_device_impl(ctx, d_d1, d_d2, d_s1c, d_s2c, w, h, step, d_fused, d_combined, nullptr, /*scores_cropped=*/true);
}

static int fuse_upload_and_run(d2pc_ctx *ctx, const uint8_t *const in[4], uint32_t w, uint32_t h, uint32_t step,
                               FuseGeometry *g) {
  int rc;
  const size_t pitch = w, fb = (size_t)w * h;  // dense device images
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaStreamSynchronize(ctx->s_compute));
  if ((rc = grow_pin(ctx, ctx->h_stage, 4 * fb))) return rc;
  for (int i = 0; i < 4; ++i) {
    if ((rc = grow_dev(ctx, ctx->d_fuse_in[i], fb)) ||
        (rc = upload_dense(ctx, i * fb, ctx->d_fuse_in[i].p, in[i], w, h, step, ctx->s_compute)))
      return rc;
  }
  const size_t side = (size_t)(w < h ? w : h);
  if ((rc = grow_dev(ctx, ctx->d_fused, side * side)) || (rc = grow_dev(ctx, ctx->d_combined, side * side)))
    return rc;
  return fuse_device_impl(ctx, ctx->d_fuse_in[0].p, ctx->d_fuse_in[1].p, ctx->d_fuse_in[2].p, ctx->d_fuse_in[3].p, w, h,
                          pitch, ctx->d_fused.p, ctx->d_combined.p, g);
}

int d2pc_fuse(d2pc_ctx *ctx, const uint8_t *d1, const uint8_t *d2, const uint8_t *s1, const uint8_t *s2, uint32_t w,
              uint32_t h, uint32_t step, d2pc_image *fused, d2pc_image *combined) {
  if (!ctx || !d1 || !d2 || !s1 || !s2 || !fused) return D2PC_ERR_INVALID_ARG;
  if (w == 0 || h == 0 || step < w) return D2PC_ERR_BAD_DIMS;
  const uint8_t *in[4] = {d1, d2, s1, s2};
  FuseGeometry g;
  int rc = fuse_upload_and_run(ctx, in, w, h, step, &g);
  if (rc) return rc;
  if ((rc = grow_pin(ctx, ctx->h_fused, (size_t)g.out_w * g.out_h)) ||
      (rc = grow_pin(ctx, ctx->h_combined, (size_t)g.n * g.n)))
    return rc;
  CU(ctx, cudaMemcpyAsync(ctx->h_fused.p, ctx->d_fused.p, (size_t)g.out_w * g.out_h, cudaMemcpyDeviceToHost,
                          ctx->s_compute));
  CU(ctx, cudaMemcpyAsync(ctx->h_combined.p, ctx->d_combined.p, (size_t)g.n * g.n, cudaMemcpyDeviceToHost,
                          ctx->s_compute));
  CU(ctx, cudaStreamSynchronize(ctx->s_compute));
  fused->data = ctx->h_fused.p;
  fused->width = (uint32_t)g.out_w, fused->height = (uint32_t)g.out_h, fused->step = (uint32_t)g.out_w;
  if (combined) {
    combined->data = ctx->h_combined.p;
    combined->width = combined->height = combined->step = (uint32_t)g.n;
  }
  return D2PC_OK;
}

// ---- matching-score preprocessing -----------------------------------------------------------------------
static int score_device_impl(d2pc_ctx *ctx, const uint8_t *d_score, uint32_t w, uint32_t h, size_t step, int which,
                             uint8_t *d_out, int *n_out, cudaStream_t stream = nullptr) {
  if (!stream) stream = ctx->s_compute;
  const d2pc_config &c = ctx->cfg;
  FuseGeometry g;
  fuse_geometry((int)w, (int)h, c.offset_x, c.offset_y, c.fuse_crop_left, c.fuse_crop_right, c.fuse_crop_top,
                c.fuse_crop_bottom, &g);
  // MatchingScoreCb only needs its own cropToSquare rectangle to lie inside the (rotated) frame (:66 / :85); the
  // rest of the fusion geometry (container, final trim) is publishFusedDepthMap's business.
  const int *rr = which == 2 ? g.r2 : g.r1;
  const int fc = which == 2 ? (int)h : (int)w, fr = which == 2 ? (int)w : (int)h;
  if (rr[2] <= 0 || rr[3] != rr[2] || rr[0] < 0 || rr[1] < 0 || rr[0] + rr[2] > fc || rr[1] + rr[3] > fr)
    return D2PC_ERR_GEOMETRY;
  const int n = rr[2];
  ScoreLaunch L;
  L.frame = d_score;
  L.step = step;
  L.width = (int)w, L.height = (int)h;
  L.rotated = which == 2;
  const int *r = which == 2 ? g.r2 : g.r1;  // :66 cropToSquare(image, ox, oy) / :85 cropToSquare(rot, -ox, -oy)
  for (int i = 0; i < 4; ++i) L.rect[i] = r[i];
  L.out = d_out;
  int nl = 0;
  CU(ctx, launch_score_preprocess(L, stream, &nl));
  ctx->launches += nl;
  if (n_out) *n_out = n;
  return D2PC_OK;
}

int d2pc_preprocess_score_device(d2pc_ctx *ctx, const uint8_t *d_score, uint32_t w, uint32_t h, size_t step, int which,
                                 uint8_t *d_out) {
  if (!ctx || !d_score || !d_out || (which != 1 && which != 2)) return D2PC_ERR_INVALID_ARG;
  if (w == 0 || h == 0 || step < w) return D2PC_ERR_BAD_DIMS;
  CU(ctx, cudaSetDevice(ctx->device));
  return score_device_impl(ctx, d_score, w, h, step, which, d_out, nullptr);
}

int d2pc_preprocess_score(d2pc_ctx *ctx, const uint8_t *score, uint32_t w, uint32_t h, uint32_t step, int which,
                          d2pc_image *out) {
  if (!ctx || !score || !out || (which != 1 && which != 2)) return D2PC_ERR_INVALID_ARG;
  if (w == 0 || h == 0 || step < w) return D2PC_ERR_BAD_DIMS;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaStreamSynchronize(ctx->s_compute));
  int rc;
  const size_t pitch = w;  // dense device image
  const size_t side = (size_t)(w < h ? w : h);
  DevBuf &d_out = ctx->d_score_out[which - 1];
  PinBuf &h_out = ctx->h_score[which - 1];
  if ((rc = grow_dev(ctx, ctx->d_score_in, pitch * h)) || (rc = grow_dev(ctx, d_out, side * side)) ||
      (rc = grow_pin(ctx, h_out, side * side)) || (rc = grow_pin(ctx, ctx->h_stage, pitch * h)) ||
      (rc = upload_dense(ctx, 0, ctx->d_score_in.p, score, w, h, step, ctx->s_compute)))
    return rc;
  int n = 0;
  if ((rc = score_device_impl(ctx, ctx->d_score_in.p, w, h, pitch, which, d_out.p, &n))) return rc;
  CU(ctx, cudaMemcpyAsync(h_out.p, d_out.p, (size_t)n * n, cudaMemcpyDeviceToHost, ctx->s_compute));
  CU(ctx, cudaStreamSynchronize(ctx->s_compute));
  out->data = h_out.p;
  out->width = out->height = out->step = (uint32_t)n;
  return D2PC_OK;
}

int d2pc_fuse_preprocessed(d2pc_ctx *ctx, const uint8_t *d1, const uint8_t *d2, const uint8_t *s1c, const uint8_t *s2c,
                           uint32_t w, uint32_t h, uint32_t step, d2pc_image *fused, d2pc_image *combined) {
  if (!ctx || !d1 || !d2 || !s1c || !s2c || !fused) return D2PC_ERR_INVALID_ARG;
  if (w == 0 || h == 0 || step < w) return D2PC_ERR_BAD_DIMS;
  const d2pc_config &c = ctx->cfg;
  FuseGeometry g;
  if (!fuse_geometry((int)w, (int)h, c.offset_x, c.offset_y, c.fuse_crop_left, c.fuse_crop_right, c.fuse_crop_top,
                     c.fuse_crop_bottom, &g))
    return D2PC_ERR_GEOMETRY;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaStreamSynchronize(ctx->s_compute));
  int rc;
  const size_t pitch = w, nn = (size_t)g.n * g.n;  // dense device images
  const size_t side = (size_t)(w < h ? w : h);
  if ((rc = grow_pin(ctx, ctx->h_stage, 2 * pitch * h + 2 * nn))) return rc;
  for (int i = 0; i < 2; ++i)
    if ((rc = grow_dev(ctx, ctx->d_fuse_in[i], pitch * h))) return rc;
  for (int i = 2; i < 4; ++i)
    if ((rc = grow_dev(ctx, ctx->d_fuse_in[i], std::max(pitch * h, nn)))) return rc;
  if ((rc = grow_dev(ctx, ctx->d_fused, side * side)) || (rc = grow_dev(ctx, ctx->d_combined, side * side)) ||
      (rc = grow_pin(ctx, ctx->h_fused, (size_t)g.out_w * g.out_h)) || (rc = grow_pin(ctx, ctx->h_combined, nn)))
    return rc;
  if ((rc = upload_dense(ctx, 0, ctx->d_fuse_in[0].p, d1, w, h, step, ctx->s_compute)) ||
      (rc = upload_dense(ctx, pitch * h, ctx->d_fuse_in[1].p, d2, w, h, step, ctx->s_compute)) ||
      (rc = upload_dense(ctx, 2 * pitch * h, ctx->d_fuse_in[2].p, s1c, (uint32_t)g.n, (uint32_t)g.n, (size_t)g.n,
                         ctx->s_compute)) ||
      (rc = upload_dense(ctx, 2 * pitch * h + nn, ctx->d_fuse_in[3].p, s2c, (uint32_t)g.n, (uint32_t)g.n, (size_t)g.n,
                         ctx->s_compute)))
    return rc;
  rc = fuse_device_impl(ctx, ctx->d_fuse_in[0].p, ctx->d_fuse_in[1].p, ctx->d_fuse_in[2].p, ctx->d_fuse_in[3].p, w, h,
                        pitch, ctx->d_fused.p, ctx->d_combined.p, nullptr, /*scores_cropped=*/true);
  if (rc) return rc;
  CU(ctx, cudaMemcpyAsync(ctx->h_fused.p, ctx->d_fused.p, (size_t)g.out_w * g.out_h, cudaMemcpyDeviceToHost,
                          ctx->s_compute));
  CU(ctx, cudaMemcpyAsync(ctx->h_combined.p, ctx->d_combined.p, nn, cudaMemcpyDeviceToHost, ctx->s_compute));
  CU(ctx, cudaStreamSynchronize(ctx->s_compute));
  fused->data = ctx->h_fused.p;
  fused->width = (uint32_t)g.out_w, fused->height = (uint32_t)g.out_h, fused->step = (uint32_t)g.out_w;
  if (combined) {
    combined->data = ctx->h_combined.p;
    combined->width = combined->height = combined->step = (uint32_t)g.n;
  }
  return D2PC_OK;
}

int d2pc_colorize_depth(d2pc_ctx *ctx, const uint8_t *gray, uint32_t w, uint32_t h, uint32_t step, d2pc_image *out) {
  if (!ctx || !gray || !out) return D2PC_ERR_INVALID_ARG;
  if (w == 0 || h == 0 || step < w) return D2PC_ERR_BAD_DIMS;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaStreamSynchronize(ctx->s_compute));
  int rc;
  const size_t pitch = w, px = (size_t)w * h;  // dense device image
  if ((rc = grow_dev(ctx, ctx->d_color_in, pitch * h)) || (rc = grow_dev(ctx, ctx->d_color_out, px * 3)) ||
      (rc = grow_dev(ctx, ctx->d_color_lut, 1024)) || (rc = grow_pin(ctx, ctx->h_color, px * 3)) ||
      (rc = grow_pin(ctx, ctx->h_stage, px)) ||
      (rc = upload_dense(ctx, 0, ctx->d_color_in.p, gray, w, h, step, ctx->s_compute)))
    return rc;
  int nl = 0;
  CU(ctx, launch_colorize(ctx->d_color_in.p, pitch, (int)w, (int)h, ctx->d_color_lut.p, !ctx->color_lut_ready,
                          ctx->d_color_out.p, ctx->s_compute, &nl));
  ctx->color_lut_ready = true;
  ctx->launches += nl;
  CU(ctx, cudaMemcpyAsync(ctx->h_color.p, ctx->d_color_out.p, px * 3, cudaMemcpyDeviceToHost, ctx->s_compute));
  CU(ctx, cudaStreamSynchronize(ctx->s_compute));
  out->data = ctx->h_color.p;
  out->width = w, out->height = h, out->step = 3 * w;
  return D2PC_OK;
}

int d2pc_fuse_then_process(d2pc_ctx *ctx, const uint8_t *d1, const uint8_t *d2, const uint8_t *s1, const uint8_t *s2,
                           uint32_t w, uint32_t h, uint32_t step, d2pc_cloud *out) {
  if (!ctx || !d1 || !d2 || !s1 || !s2 || !out) return D2PC_ERR_INVALID_ARG;
  if (w == 0 || h == 0 || step < w) return D2PC_ERR_BAD_DIMS;
  const d2pc_config &c = ctx->cfg;
  FuseGeometry g;
  if (!fuse_geometry((int)w, (int)h, c.offset_x, c.offset_y, c.fuse_crop_left, c.fuse_crop_right, c.fuse_crop_top,
                     c.fuse_crop_bottom, &g))
    return D2PC_ERR_GEOMETRY;
  // a synchronous mono8 submission on slot 0 whose frame is the fused map: it stays on the device and enters
  // DisparityCb's mono8 path there (cpp:55-85); there is no H2D of it to time
  const uint32_t fw = (uint32_t)g.out_w, fh = (uint32_t)g.out_h;
  Slot &s = ctx->slots[0];
  s.timed = false;
  Submission sub{nullptr, 0, true, true, ctx->s_compute};
  const uint8_t *in[4] = {d1, d2, s1, s2};
  int rc;
  if ((rc = submit_front(ctx, s, fw, fh, sub)) || (rc = fuse_upload_and_run(ctx, in, w, h, step, nullptr)) ||
      (rc = submit_back(ctx, s, {ctx->d_fused.p, false, 1, fw, fh, fw, (size_t)fw * fh}, sub)))
    return rc;
  return d2pc_wait(ctx, 0, out);
}

// ---- the whole fusion node + DisparityCb per frame set, on the slot pipeline ------------------------------------
int d2pc_submit_fusion(d2pc_ctx *ctx, int slot, const uint8_t *d1, const uint8_t *d2, const uint8_t *s1,
                       const uint8_t *s2, uint32_t w, uint32_t h, uint32_t step, int preprocess_scores) {
  if (!ctx || slot < 0 || slot >= (int)ctx->slots.size() || !d1 || !d2 || !s1 || !s2) return D2PC_ERR_INVALID_ARG;
  if (w == 0 || h == 0 || w > (1u << 16) || h > (1u << 16) || step < w) return D2PC_ERR_BAD_DIMS;
  const d2pc_config &c = ctx->cfg;
  FuseGeometry g;
  if (!fuse_geometry((int)w, (int)h, c.offset_x, c.offset_y, c.fuse_crop_left, c.fuse_crop_right, c.fuse_crop_top,
                     c.fuse_crop_bottom, &g))
    return D2PC_ERR_GEOMETRY;
  Slot &s = ctx->slots[slot];
  NvtxRange nvtx_submit("d2pc submit fusion set");
  const uint32_t fw = (uint32_t)g.out_w, fh = (uint32_t)g.out_h;
  Submission sub{nullptr, 0, false, true, s.s_kern};
  int rc = submit_front(ctx, s, fw, fh, sub);
  if (rc) return rc;
  // rows that are 16-byte multiples stay dense on the device, so a frame (or a whole contiguous set) is one 1-D DMA:
  // four pitched 2-D copies per set ran at 43 GB/s and bounded the stream at 6.6 k sets/s (one 1-D copy: 9.2 k)
  // (mono8 frames of any width: the fusion kernels read bytes, and a pitched 2-D copy is the slow way in)
  const size_t pitch = w, frame_bytes = (size_t)w * h, nn = (size_t)g.n * g.n;
  // the four input frames of a set live in one allocation, so that a contiguous pinned set is one DMA
  if ((rc = grow_dev(ctx, s.d_fuse_in[0], 4 * pitch * h))) return rc;
  uint8_t *const fin[4] = {s.d_fuse_in[0].p, s.d_fuse_in[0].p + pitch * h, s.d_fuse_in[0].p + 2 * pitch * h,
                           s.d_fuse_in[0].p + 3 * pitch * h};
  if ((rc = grow_dev(ctx, s.d_pre[0], nn)) || (rc = grow_dev(ctx, s.d_pre[1], nn)) ||
      (rc = grow_dev(ctx, s.d_container, (size_t)g.nc * g.nc)) || (rc = grow_dev(ctx, s.d_combined, nn)) ||
      (rc = grow_dev(ctx, s.d_fused, (size_t)fw * fh)))
    return rc;

  s.timed = ctx->timing && s.ev_start;
  if (s.timed) CU(ctx, cudaEventRecord(s.ev_start, ctx->s_h2d));
  // ---- H2D (stream 1): pinned caller frames are DMA'd in place, pageable ones are staged
  const uint8_t *in[4] = {d1, d2, s1, s2};
  const bool one_block = step == w && pitch == w && d2 == d1 + frame_bytes && s1 == d2 + frame_bytes &&
                         s2 == s1 + frame_bytes && lookup_pinned(ctx, d1) && lookup_pinned(ctx, s2);
  if (one_block) CU(ctx, cudaMemcpyAsync(fin[0], d1, 4 * frame_bytes, cudaMemcpyHostToDevice, ctx->s_h2d));
  for (int i = 0; i < 4 && !one_block; ++i) {
    const uint8_t *src = in[i];
    size_t src_pitch = step;
    if (!lookup_pinned(ctx, in[i])) {
      if ((rc = grow_pin(ctx, s.h_in, 4 * frame_bytes))) return rc;
      uint8_t *stage = s.h_in.p + i * frame_bytes;
      if (step == w) memcpy(stage, in[i], frame_bytes);
      else
        for (uint32_t y = 0; y < h; ++y) memcpy(stage + (size_t)y * w, in[i] + (size_t)y * step, w);
      src = stage, src_pitch = w;
    }
    if (src_pitch == w && pitch == w) CU(ctx, cudaMemcpyAsync(fin[i], src, frame_bytes, cudaMemcpyHostToDevice, ctx->s_h2d));
    else CU(ctx, cudaMemcpy2DAsync(fin[i], pitch, src, src_pitch, w, h, cudaMemcpyHostToDevice, ctx->s_h2d));
  }
  CU(ctx, cudaEventRecord(s.ev_h2d, ctx->s_h2d));

  // ---- kernels: MatchingScoreCb1/2 -> merge -> median 3 + trim -> DisparityCb on the fused map.  Six small
  // kernels (~100 us together, none of which fills the chip): each slot launches them on its own stream, so the
  // sets of consecutive slots overlap on the GPU instead of queueing behind each other.
  cudaStream_t sk = s.s_kern;
  CU(ctx, cudaStreamWaitEvent(sk, s.ev_h2d, 0));
  const uint8_t *sc1 = fin[2], *sc2 = fin[3];
  if (preprocess_scores) {
    if ((rc = score_device_impl(ctx, fin[2], w, h, pitch, 1, s.d_pre[0].p, nullptr, sk)) ||
        (rc = score_device_impl(ctx, fin[3], w, h, pitch, 2, s.d_pre[1].p, nullptr, sk)))
      return rc;
    sc1 = s.d_pre[0].p, sc2 = s.d_pre[1].p;
  }
  if ((rc = fuse_device_impl(ctx, fin[0], fin[1], sc1, sc2, w, h, pitch, s.d_fused.p, s.d_combined.p,
                             nullptr, preprocess_scores != 0, &s.d_container, sk)))
    return rc;
  return submit_back(ctx, s, {s.d_fused.p, false, 1, fw, fh, fw, (size_t)fw * fh}, sub);
}

int d2pc_process_fusion_stream(d2pc_ctx *ctx, const uint8_t *sets, uint64_t n_sets, size_t set_stride, uint64_t ring_len,
                               uint32_t w, uint32_t h, uint32_t step, int preprocess_scores, d2pc_cloud_sink sink,
                               void *user) {
  if (!ctx || (!sets && n_sets)) return D2PC_ERR_INVALID_ARG;
  const size_t fb = (size_t)step * h;
  auto submit = [&](const uint8_t *f, int slot) {
    return d2pc_submit_fusion(ctx, slot, f, f + fb, f + 2 * fb, f + 3 * fb, w, h, step, preprocess_scores);
  };
  return run_ring(ctx, sets, n_sets, set_stride, ring_len, submit, sink, user);
}

// ---------------------------------------------------------------------------
// ROS1 wire image of the published PointCloud2
// ---------------------------------------------------------------------------
size_t d2pc_serialize_pointcloud2(const d2pc_ctx *ctx, const d2pc_cloud *cloud, uint32_t seq, uint32_t sec,
                                  uint32_t nsec, uint8_t *out, size_t cap) {
  if (!ctx || !cloud) return 0;
  // std_msgs/Header, then the sensor_msgs/PointCloud2 members in declaration order, little endian,
  // strings and arrays length-prefixed with uint32 (ROS1 serialisation rules).
  const char *fid = ctx->cfg.frame_id;
  const uint32_t fid_len = (uint32_t)strlen(fid);
  size_t need = 12 + 4 + fid_len + 8 + 4;
  for (uint32_t i = 0; i < cloud->n_fields; ++i) need += 4 + strlen(cloud->fields[i].name) + 4 + 1 + 4;
  const size_t data_len = (size_t)cloud->row_step * cloud->height;
  need += 1 + 4 + 4 + 4 + data_len + 1;
  if (!out || cap < need) return need;
  uint8_t *p = out;
  auto u32 = [&](uint32_t v) {
    memcpy(p, &v, 4);
    p += 4;
  };
  auto bytes = [&](const void *s, size_t n) {
    if (n) memcpy(p, s, n);
    p += n;
  };
  u32(seq), u32(sec), u32(nsec);
  u32(fid_len), bytes(fid, fid_len);
  u32(cloud->height), u32(cloud->width);
  u32(cloud->n_fields);
  for (uint32_t i = 0; i < cloud->n_fields; ++i) {
    const uint32_t nl = (uint32_t)strlen(cloud->fields[i].name);
    u32(nl), bytes(cloud->fields[i].name, nl);
    u32(cloud->fields[i].offset);
    *p++ = cloud->fields[i].datatype;
    u32(cloud->fields[i].count);
  }
  *p++ = cloud->is_bigendian;
  u32(cloud->point_step), u32(cloud->row_step);
  u32((uint32_t)data_len), bytes(cloud->data, data_len);
  *p++ = cloud->is_dense;
  return need;
}

size_t d2pc_serialize_laserscan(const d2pc_ctx *ctx, const d2pc_laser_scan *scan, uint32_t seq, uint32_t sec,
                                uint32_t nsec, uint8_t *out, size_t cap) {
  if (!ctx || !scan || (scan->n_ranges && !scan->ranges)) return 0;
  // std_msgs/Header, then the sensor_msgs/LaserScan members in declaration order: seven float32, ranges and
  // intensities as length-prefixed float32 arrays (intensities empty)
  const char *fid = ctx->cfg.frame_id;
  const uint32_t fid_len = (uint32_t)strlen(fid);
  const size_t need = 12 + 4 + fid_len + 7 * 4 + 4 + (size_t)scan->n_ranges * 4 + 4;
  if (!out || cap < need) return need;
  uint8_t *p = out;
  auto u32 = [&](uint32_t v) {
    memcpy(p, &v, 4);
    p += 4;
  };
  auto f32 = [&](float v) {
    memcpy(p, &v, 4);
    p += 4;
  };
  u32(seq), u32(sec), u32(nsec);
  u32(fid_len);
  memcpy(p, fid, fid_len);
  p += fid_len;
  f32(scan->angle_min), f32(scan->angle_max), f32(scan->angle_increment), f32(scan->time_increment);
  f32(scan->scan_time), f32(scan->range_min), f32(scan->range_max);
  u32(scan->n_ranges);
  if (scan->n_ranges) memcpy(p, scan->ranges, (size_t)scan->n_ranges * 4);
  p += (size_t)scan->n_ranges * 4;
  u32(0);
  return need;
}

const char *d2pc_strerror(int status) {
  switch (status) {
    case D2PC_OK: return "ok";
    case D2PC_ERR_INVALID_ARG: return "invalid argument";
    case D2PC_ERR_BAD_ENCODING: return "unsupported image encoding (mono8 / 8UC1 / 32FC1 only)";
    case D2PC_ERR_BAD_DIMS: return "bad image dimensions, step or alignment";
    case D2PC_ERR_CUDA: return "CUDA runtime error";
    case D2PC_ERR_NO_DEVICE: return "no usable sm_100 (B200) device";
    case D2PC_ERR_NOMEM: return "out of memory";
    case D2PC_ERR_GEOMETRY: return "fusion crop rectangle leaves the image";
    case D2PC_ERR_NOT_READY: return "nothing submitted on this slot / inputs not yet received";
    case D2PC_ERR_BUFFER_TOO_SMALL: return "output buffer too small";
    default: return "unknown status";
  }
}
const char *d2pc_last_cuda_error(const d2pc_ctx *ctx) { return ctx ? ctx->last_cuda_error.c_str() : ""; }

}  // extern "C"
