/*
 * d2pc_b200.h -- C ABI of libd2pc_b200.so: the B200 (sm_100a) implementation of
 * the per-frame hot path of PX4/disparity_to_point_cloud.
 *
 * The reference has no plugin/operator API: its boundary is the ROS1 callback
 *   void Disparity2PCloud::DisparityCb(const sensor_msgs::ImageConstPtr&)
 *       include/disparity_to_point_cloud/disparity_to_point_cloud.hpp:108
 *       src/disparity_to_point_cloud.cpp:46-92
 * and, for the fusion node, the four callbacks of
 *       include/disparity_to_point_cloud/depth_map_fusion.hpp:127-130
 *       src/depth_map_fusion.cpp:46-136.
 * Each entry point below names the reference lines it replaces.  Plain
 * pointers and sizes only; no C++ or torch types; no exception crosses this
 * boundary; every function returns a d2pc_status (0 = OK, negative = error).
 *
 * Threading (reference: one ros::spin() thread, src/disparity_to_point_cloud_node.cpp:50):
 * a context is single-caller.  Different contexts are independent and may live
 * on different GPUs / host threads.
 *
 * There is NO CPU fallback: every compute entry point fails with
 * D2PC_ERR_NO_DEVICE / D2PC_ERR_CUDA if the GPU path is unavailable.
 *
 * (file:line citations are relative to the reference repository root.)
 */
#ifndef D2PC_B200_H_
#define D2PC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define D2PC_ABI_VERSION 1

typedef enum d2pc_status {
  D2PC_OK = 0,
  D2PC_ERR_INVALID_ARG = -1,  /* NULL pointer, bad enum, bad slot ...              */
  D2PC_ERR_BAD_ENCODING = -2, /* image encoding other than mono8 / 8UC1 / 32FC1     */
  D2PC_ERR_BAD_DIMS = -3,     /* width/height/step inconsistent or over capacity    */
  D2PC_ERR_CUDA = -4,         /* a CUDA runtime call failed (see d2pc_last_cuda_error) */
  D2PC_ERR_NO_DEVICE = -5,    /* no usable sm_100 device                            */
  D2PC_ERR_NOMEM = -6,        /* host or device allocation failed                   */
  D2PC_ERR_GEOMETRY = -7,     /* fusion crop rectangle leaves the image (cv::Mat ROI would throw) */
  D2PC_ERR_NOT_READY = -8,    /* wait on a slot with nothing submitted / caches empty */
  D2PC_ERR_BUFFER_TOO_SMALL = -9
} d2pc_status;

/* src/disparity_to_point_cloud.cpp:69-76: the reference's only point filter is
 * the fixed border crop (CROP).  CROP_FINITE is an extension: crop, then drop
 * points with a non-finite x, y or z, order preserved (decoupled look-back
 * stream compaction).  VOXEL is an extension too: pcl::VoxelGrid<pcl::PointXYZ>
 * applied to the CROP cloud on the device (d2pc_voxel_grid below; selectable once
 * a grid has been set with d2pc_set_voxel_grid). */
typedef enum d2pc_filter_mode {
  D2PC_FILTER_CROP = 0,
  D2PC_FILTER_CROP_FINITE = 1,
  D2PC_FILTER_VOXEL = 2
} d2pc_filter_mode;

/* EXACT reproduces cv::reprojectImageTo3D's float64 rounding sequence bit for
 * bit (src/disparity_to_point_cloud.cpp:63-64).  FAST is float32 only
 * (<= 1e-5 relative to depth, not bit-exact). */
typedef enum d2pc_arith_mode { D2PC_ARITH_EXACT = 0, D2PC_ARITH_FAST = 1 } d2pc_arith_mode;

/* src/depth_map_fusion.cpp:150-235: the rule getFusedDistance dispatches to.
 * GRAD_FILTER is the one the reference is compiled with. */
typedef enum d2pc_fuse_rule {
  D2PC_FUSE_GRAD_FILTER = 0,
  D2PC_FUSE_MAX_DIST = 1,
  D2PC_FUSE_MAX_DIST_UNLESS_BLACK = 2,
  D2PC_FUSE_BETTER_SCORE = 3,
  D2PC_FUSE_ONLY_GOOD_1 = 4,
  D2PC_FUSE_ONLY_GOOD_AVG = 5,
  D2PC_FUSE_OVERLAP = 6,
  D2PC_FUSE_BLACK_TO_WHITE = 7
} d2pc_fuse_rule;

/* Every constant the reference hard-codes or reads from ROS params, with the
 * reference values as defaults (d2pc_config_default). */
typedef struct d2pc_config {
  uint32_t struct_size; /* sizeof(d2pc_config), for ABI growth */
  /* Disparity2PCloud */
  double fx, fy, cx, cy, baseline; /* hpp:66-71, 84-88: 714.24, 713.5, 376, 240, 0.09 */
  int32_t rect_width, rect_height; /* hpp:101-103: 752 x 480, independent of the frame size */
  int32_t border;                  /* cpp:70,72: 40 */
  int32_t median_ksize;            /* cpp:57: 11 (odd, 1 disables) */
  float disparity_scale;           /* cpp:61: 1/8 */
  int32_t filter_mode;             /* d2pc_filter_mode */
  int32_t arith_mode;              /* d2pc_arith_mode */
  char frame_id[64];               /* cpp:89: "/camera_optical_frame" */
  int32_t verbose;                 /* cpp:82: print "Cloud size: N" when non-zero */
  /* DepthMapFusion */
  int32_t offset_x, offset_y; /* depth_map_fusion.hpp:76-77, launch/depth_map_fusion.launch:8-9 */
  int32_t fuse_rule;          /* d2pc_fuse_rule */
  int32_t fuse_median_ksize;  /* depth_map_fusion.cpp:124: 3 */
  int32_t fuse_crop_left, fuse_crop_right, fuse_crop_top, fuse_crop_bottom; /* :130: 0,40,30,10 */
  /* capacity / pipeline */
  int32_t max_width, max_height; /* largest frame the context will see (buffers are sized once) */
  int32_t max_batch;             /* frames per batched call chunk */
  int32_t n_slots;               /* async pipeline depth (>= 1, default 4) */
} d2pc_config;

typedef struct d2pc_ctx d2pc_ctx;

/* sensor_msgs/PointField as pcl::toROSMsg<pcl::PointXYZ> fills it (SURVEY.md A.3). */
typedef struct d2pc_point_field {
  char name[8];
  uint32_t offset;
  uint8_t datatype; /* 7 = FLOAT32 */
  uint32_t count;
} d2pc_point_field;

/* The sensor_msgs/PointCloud2 payload DisparityCb publishes
 * (src/disparity_to_point_cloud.cpp:79-90).  `data` is library-owned pinned
 * host memory, valid until the next call that uses the same slot -- or the
 * caller's own buffer when one of the *_into entry points was used. */
typedef struct d2pc_cloud {
  const uint8_t *data; /* width * 16 bytes: {f32 x, f32 y, f32 z, f32 1.0} */
  uint32_t height;     /* 1 */
  uint32_t width;      /* number of points */
  uint32_t point_step; /* 16 */
  uint32_t row_step;   /* 16 * width */
  uint8_t is_bigendian; /* 0 */
  uint8_t is_dense;     /* 0 in CROP mode (cpp:81); 1 in CROP_FINITE; VOXEL: 1, 0 for the overflow fallback;
                           1 behind the crop box or the radius outlier stage; the cloud transform keeps it */
  uint32_t n_fields;    /* 3 */
  d2pc_point_field fields[3];
} d2pc_cloud;

/* A mono8 sensor_msgs/Image payload (fusion outputs). Library-owned pinned memory. */
typedef struct d2pc_image {
  const uint8_t *data;
  uint32_t width, height, step;
} d2pc_image;

/* ---- lifecycle ------------------------------------------------------------ */

void d2pc_config_default(d2pc_config *cfg);

/* Replaces the Disparity2PCloud / DepthMapFusion constructors
 * (disparity_to_point_cloud.hpp:75-106, depth_map_fusion.hpp:97-124) minus the
 * ROS wiring: selects the device, creates streams, sizes pinned + device
 * buffers and derives Q from the intrinsics in cfg. */
int d2pc_create(const d2pc_config *cfg, int device, d2pc_ctx **out);
void d2pc_destroy(d2pc_ctx *ctx);

/* cv::stereoRectify(K,0,K,0,Size(rect_w,rect_h),I,(-b,0,0)) -> Q, row-major 4x4
 * (disparity_to_point_cloud.hpp:90-104).  Host only. */
int d2pc_q_from_intrinsics(double fx, double fy, double cx, double cy, double baseline, int rect_w, int rect_h,
                           double q_out[16]);
int d2pc_set_q(d2pc_ctx *ctx, const double q[16]);
int d2pc_get_q(const d2pc_ctx *ctx, double q_out[16]);
int d2pc_set_filter_mode(d2pc_ctx *ctx, int filter_mode); /* VOXEL: D2PC_ERR_INVALID_ARG until a grid is set */
int d2pc_set_arith_mode(d2pc_ctx *ctx, int arith_mode);

/* ---- voxel-grid downsampling (D2PC_FILTER_VOXEL) ------------------------------
 *
 * The published cloud is pcl::VoxelGrid<pcl::PointXYZ> (PCL 1.7.2 - 1.12, downsample_all_data = true,
 * filter_limit_negative = false) applied to exactly the cloud CROP mode publishes for the same frame, +-inf and
 * NaN points included.  The recipe, float32 throughout unless stated, no FMA contraction:
 *   1. inv[a] = 1.0f / leaf[a] for a in {x, y, z}.
 *   2. A point is included when x, y and z are finite and, with a limit field set, that coordinate widened to
 *      double lies in [limit_min, limit_max] (both ends inclusive).
 *   3. min_p / max_p: per-axis float min / max over the included points.  None included: the empty cloud
 *      (width 0, is_dense 1).
 *   4. Overflow guard: d[a] = (int64)((max_p[a] - min_p[a]) * inv[a]) + 1; when dx*dy*dz > INT32_MAX the output is
 *      the input cloud unchanged (all N crop points, is_dense 0) -- PCL's `output = *input_` after its warning.
 *   5. min_b[a] = (int)floorf(min_p[a] * inv[a]), max_b[a] = (int)floorf(max_p[a] * inv[a]),
 *      div_b = max_b - min_b + 1, mul = (1, div_b.x, div_b.x * div_b.y).
 *   6. ijk[a] = (int)(floorf(p[a] * inv[a]) - (float)min_b[a]); idx = ijk.x + ijk.y * mul.y + ijk.z * mul.z in
 *      64 bits (PCL's int wherever PCL's does not overflow).  Where PCL's int arithmetic WOULD overflow -- a
 *      floorf bound outside int32, or an idx that can reach 2^31 - 1 -- PCL's result is undefined; this library
 *      then takes the step-4 fallback as well.
 *   7. Voxels are emitted in ascending idx; a voxel with fewer than min_points_per_voxel points is dropped.
 *   8. centroid = (sum x, sum y, sum z) / (float)count, each sum a float32 left fold, IEEE division; the point is
 *      {cx, cy, cz, 1.0f}, 16 bytes with the same fields and point_step as every other mode.
 *      Summation order: ascending point index (row-major crop order) within the voxel.  PCL orders a voxel's
 *      points with std::sort, which is not stable, so its order -- and the last bits of its centroids -- is
 *      unspecified; the stable order is the one a GPU and a CPU reference can both meet bit for bit.
 *   9. height 1, width = number of voxels, is_dense 1 (0 only for the fallback), row_step = 16 * width.
 * The size of a VOXEL cloud is known only when the frame has been processed, so the rules of CROP_FINITE apply:
 * BUFFER_TOO_SMALL is reported by d2pc_wait, the kernel never stores into host memory ("direct_out" does not
 * apply), d2pc_slot_timing's d2h_us covers the count, and the device batch entries need d_counts (frame f's voxels
 * at d_points + f * points_stride; every frame of a batch is its own grid). */
typedef struct d2pc_voxel_grid {
  uint32_t struct_size;          /* sizeof(d2pc_voxel_grid) */
  float leaf_x, leaf_y, leaf_z;  /* finite, > 0 */
  uint32_t min_points_per_voxel; /* PCL default 0 */
  int32_t limit_field;           /* -1 none, 0 x, 1 y, 2 z */
  double limit_min, limit_max;   /* limit_min <= limit_max */
} d2pc_voxel_grid;

/* leaf 0 (not yet valid), no limit, min_points_per_voxel 0. */
void d2pc_voxel_grid_default(d2pc_voxel_grid *grid);
/* D2PC_ERR_INVALID_ARG for a leaf that is not finite and > 0, a limit_field outside -1..2, limit_min > limit_max
 * (PCL would accept it and return nothing) or a wrong struct_size; the previous grid is kept then. */
int d2pc_set_voxel_grid(d2pc_ctx *ctx, const d2pc_voxel_grid *grid);
/* The grid last set (d2pc_voxel_grid_default's until then). */
int d2pc_get_voxel_grid(const d2pc_ctx *ctx, d2pc_voxel_grid *grid);

/* ---- radius outlier removal (a stage behind every filter mode) -------------------
 *
 * Off by default (radius 0).  With a radius set, the published cloud is pcl::RadiusOutlierRemoval<pcl::PointXYZ>
 * (setNegative(false), keep_organized false) applied on the device to exactly the cloud the current filter mode
 * would publish for that frame: CROP's N points (+-inf and NaN included), CROP_FINITE's compacted cloud, VOXEL's
 * centroids (or, for a frame that took VOXEL's overflow fallback, its CROP cloud).  So CROP + this stage and
 * CROP_FINITE + this stage publish the same bytes.  The setting is independent of d2pc_set_filter_mode.  The recipe:
 *   1. r2 = radius * radius, in double.
 *   2. A point takes part only when x, y and z are all finite.  A non-finite point is dropped and is nobody's
 *      neighbour (PCL's kd-tree does not index it).
 *   3. The squared distance of points i and j is float32 with no FMA: dx = xi - xj (likewise dy, dz),
 *      s = (dx*dx + dy*dy) + dz*dz, each operation rounded.  (FLANN's L2_Simple<float>, as PCL's KdTreeFLANN uses it.)
 *   4. neighbours(i) = the number of finite j with (double)s(i, j) <= r2; it counts i itself and any duplicate of i.
 *   5. i is kept when neighbours(i) >= min_neighbors + 1, so min_neighbors = 0 keeps every finite point.
 *   6. Kept points are copied unchanged, all 16 bytes, in input order; height 1, width = kept, is_dense 1,
 *      row_step = 16 * width.
 * Relation to PCL (RadiusOutlierRemoval::applyFilterIndices, PCL 1.8 - 1.12; restated from memory, PCL's source was
 * not at hand when this was written -- the same footing as DESIGN.md section 0.1 for the OpenCV dispatch):
 *   - is_dense input (CROP_FINITE, VOXEL): PCL runs nearestKSearch(k = min_neighbors + 1) per point and keeps it when
 *     k neighbours were found and nn_dists[k - 1] <= r2 in double.  The k-th smallest distance is <= r2 exactly when
 *     at least k distances are, which is rules 4-5.
 *   - non-dense input (CROP, the VOXEL fallback): PCL runs radiusSearch, whose FLANN result set is believed to
 *     test dist < (float)r2.  This library applies rule 4 to every input; the two differ only for a pair whose
 *     distance lies exactly on the boundary (s == (float)r2, or between r2 and (float)r2).
 *   - is_dense of the output: PCL's filter path copies the kept points into a fresh cloud; whether that copy sets
 *     is_dense is not verified here.  The library publishes 1 (every kept point is finite).
 * With a radius set every mode is a counted mode, as CROP_FINITE is: BUFFER_TOO_SMALL is reported by d2pc_wait, the
 * kernel never stores into host memory ("direct_out" does not apply), d2pc_slot_timing's d2h_us covers the count,
 * and the device batch entries need d_counts.  With radius 0 nothing of this applies. */
typedef struct d2pc_radius_outlier {
  uint32_t struct_size;   /* sizeof(d2pc_radius_outlier) */
  double radius;          /* 0: the stage is off (the default); otherwise finite and > 0 */
  uint32_t min_neighbors; /* PCL's setMinNeighborsInRadius; default 1 */
} d2pc_radius_outlier;

/* radius 0 (off), min_neighbors 1. */
void d2pc_radius_outlier_default(d2pc_radius_outlier *p);
/* D2PC_ERR_INVALID_ARG for a radius that is negative, NaN or infinite, or a wrong struct_size; the previous
 * setting is kept then. */
int d2pc_set_radius_outlier(d2pc_ctx *ctx, const d2pc_radius_outlier *p);
/* The setting last made (d2pc_radius_outlier_default's until then). */
int d2pc_get_radius_outlier(const d2pc_ctx *ctx, d2pc_radius_outlier *p);

/* ---- crop box (a stage in front of VOXEL and the radius outlier stage) -----------
 *
 * Off by default (enabled 0).  With a box enabled, the published cloud is pcl::CropBox<pcl::PointXYZ> with
 * setTransform only (no setRotation / setTranslation), setNegative(false) and keep_organized false, applied on the
 * device to the CROP cloud of that frame; VOXEL and the radius outlier stage then run on the box's cloud.  The
 * recipe, float32 throughout, no FMA contraction:
 *   1. A point takes part only when x, y and z are all finite (the CROP cloud is not dense, and PCL then skips such
 *      points).
 *   2. l = T * p with T = transform (row-major 3x4 [R | t], camera frame -> box frame), each operation rounded:
 *      lx = ((t00*x + t01*y) + t02*z) + t03, likewise ly (row 1) and lz (row 2).
 *   3. The point is kept when min_pt[a] <= l[a] <= max_pt[a] on all three axes: the faces are inside the box.
 *   4. Kept points are copied unchanged -- the original camera-frame coordinates, all 16 bytes -- in input order;
 *      height 1, width = kept, is_dense 1, row_step = 16 * width.
 * Composition with the filter mode:
 *   - CROP + box and CROP_FINITE + box publish the same bytes: the box drops non-finite points anyway, so both run
 *     the CROP kernels and the box does the one compaction.
 *   - VOXEL + box is VoxelGrid(CropBox(CROP cloud)): the grid's bounds come from the box's points.  A frame that
 *     takes VOXEL's overflow fallback publishes the box's cloud with is_dense 1 (all of its points are finite;
 *     whether PCL's copy in that fallback would set is_dense is not verified here).
 *   - The radius outlier stage runs on whatever the steps before it produced.
 *   - With a cloud transform enabled (d2pc_set_cloud_transform) the box runs on the transformed cloud: "camera frame"
 *     above then reads "target frame", and the points it keeps are target-frame points.
 * Relation to PCL (CropBox::applyFilter and pcl::transformPoint, PCL 1.8 - 1.12; restated from memory, PCL's source
 * was not at hand when this was written -- the same footing as DESIGN.md section 0.1 for the OpenCV dispatch):
 *   - transformPoint computes each row as ((m(i,0)*x + m(i,1)*y) + m(i,2)*z) + m(i,3) in float, which is rule 2.
 *   - PCL skips the transform when transform_.matrix().isIdentity(), Eigen's fuzzy test (every entry within 1e-5 of
 *     the identity's for float).  For the exact identity this changes no decision (1*x + 0*y + 0*z + 0 is x up to
 *     the sign of a zero).  A transform that is within that tolerance but not exactly the identity is applied here,
 *     and skipped by PCL: the two can then differ for points within about 1e-5 * |p| of a face.
 *   - PCL rejects a point when l[a] < min_pt[a] or l[a] > max_pt[a], so it would keep a point whose l is NaN.  Such
 *     an l needs T * p to overflow float (|p| and |T| near 1e38); this library drops that point (rule 3).
 * With a box enabled every mode is a counted mode, as CROP_FINITE is: BUFFER_TOO_SMALL is reported by d2pc_wait,
 * the kernel never stores into host memory ("direct_out" does not apply), d2pc_slot_timing's d2h_us covers the
 * count, and the device batch entries need d_counts.  With enabled 0 nothing of this applies. */
typedef struct d2pc_crop_box {
  uint32_t struct_size; /* sizeof(d2pc_crop_box) */
  int32_t enabled;      /* 0: off (the default) */
  float min_pt[3];      /* PCL setMin (x, y, z); default -1 */
  float max_pt[3];      /* PCL setMax; default 1 */
  float transform[12];  /* row-major 3x4 [R | t], PCL setTransform (camera frame -> box frame); default identity */
} d2pc_crop_box;

/* enabled 0, min_pt (-1, -1, -1), max_pt (1, 1, 1), the identity transform. */
void d2pc_crop_box_default(d2pc_crop_box *b);
/* D2PC_ERR_INVALID_ARG for a NaN bound, min_pt > max_pt on an axis, a non-finite transform entry or a wrong
 * struct_size; the previous setting is kept then.  +-inf bounds are allowed (a half-open box). */
int d2pc_set_crop_box(d2pc_ctx *ctx, const d2pc_crop_box *b);
/* The setting last made (d2pc_crop_box_default's until then). */
int d2pc_get_crop_box(const d2pc_ctx *ctx, d2pc_crop_box *b);

/* ---- cloud transform (the first stage: in front of the crop box, VOXEL and the radius outlier stage) ----------
 *
 * Off by default (enabled 0).  With a transform enabled, the published cloud is pcl::transformPointCloud<PointXYZ>
 * with an affine matrix, applied on the device to the cloud of the filter mode's reproject step (CROP's N points or
 * CROP_FINITE's compacted ones) before any other stage: reproject -> transform -> crop box -> VOXEL -> outlier stage.
 * So the crop box's transform maps the TARGET frame to the box frame, VOXEL's grid lies in the target frame, and the
 * outlier stage sees target-frame points.  The recipe, float32 throughout, no FMA contraction:
 *   1. A point whose x, y and z are all finite becomes x' = ((m00*x + m01*y) + m02*z) + m03, likewise y' (row 1)
 *      and z' (row 2), each operation rounded: the crop box's rule 2, one shared device routine.
 *   2. A point with a non-finite coordinate is copied unchanged, all 16 bytes, NaN payloads included (PCL's
 *      non-dense branch; for dense input every point is finite and both PCL branches are rule 1).
 *   3. The fourth word (1.0f) is copied; the point count and the input order are kept.
 *   4. is_dense is the input's.  A finite point whose T * p overflows is written as computed (+-inf or NaN), as PCL
 *      writes it, so CROP_FINITE with an extreme transform can publish a non-finite point with is_dense 1.  A NaN
 *      the arithmetic makes (inf + -inf) is written as 0xFFC00000, the default NaN of x86 SSE arithmetic and so what
 *      PCL writes on x86-64.
 * The identity maps every finite coordinate to itself except -0, which becomes +0 (-0 * 1 + 0 * y + ... is +0).
 * Relation to PCL (transformPointCloud in common/impl/transforms.hpp, PCL 1.8 - 1.12; restated from memory, PCL's
 * source was not at hand when this was written -- the same footing as DESIGN.md section 0.1 for the OpenCV dispatch):
 *   - transformPointCloud copies the cloud, then transforms every point if is_dense, otherwise only the points with
 *     finite x, y and z (rules 1 and 2).
 *   - PCL >= 1.10 computes a point through detail::Transformer<float>.  Its SSE2 specialisation is believed to form
 *     each row as x*c0 + (y*c1 + (z*c2 + c3)); its scalar template as ((m0*x + m1*y) + m2*z) + m3, which a compiler
 *     may contract to FMAs.  PCL 1.8 - 1.9 use Eigen's matrix product.  No single PCL rounding order exists; this
 *     library uses the scalar template's order without contraction (rule 1), the crop box's order.
 *   - Measured on three 752x480 S2 scenes (tests/test_oracle_transform.py; yaw 30, pitch 20, roll 10 degrees and a
 *     translation): the SSE2 order gives a different float on 41 % of the finite points' output coordinates, by at
 *     most 4 ulp of the row's largest term (a result that cancels towards zero can differ by more of its own ulp).
 * With a transform and no other cloud stage, CROP stays an uncounted mode (no payload copy in d2pc_wait,
 * BUFFER_TOO_SMALL at submit, and the device batch entries may pass d_counts NULL); the synchronous mono8 entries then
 * copy the cloud out of a device buffer instead of storing it into host memory from the kernel ("direct_out" 1
 * forces the latter).  The setting in force when a frame is submitted is
 * the one its slot uses: set a frame's pose, submit it, then set the next one. */
typedef struct d2pc_cloud_transform {
  uint32_t struct_size; /* sizeof(d2pc_cloud_transform) */
  int32_t enabled;      /* 0: off (the default) */
  float matrix[12];     /* row-major 3x4 [A | t], camera frame -> target frame; any finite affine map; default
                           identity */
} d2pc_cloud_transform;

/* enabled 0, the identity matrix. */
void d2pc_cloud_transform_default(d2pc_cloud_transform *t);
/* D2PC_ERR_INVALID_ARG for a non-finite matrix entry or a wrong struct_size; the previous setting is kept then. */
int d2pc_set_cloud_transform(d2pc_ctx *ctx, const d2pc_cloud_transform *t);
/* The setting last made (d2pc_cloud_transform_default's until then). */
int d2pc_get_cloud_transform(const d2pc_ctx *ctx, d2pc_cloud_transform *t);

/* ---- laser scan (an output next to the cloud: pointcloud_to_laserscan on the device) -------------------------------
 *
 * Off by default (enabled 0).  With the scan on, every host entry point that publishes a cloud (the process_* and
 * *_into calls, submit / d2pc_wait, d2pc_process_stream, the fusion entries) also produces the sensor_msgs/LaserScan
 * that pointcloud_to_laserscan would publish for exactly that cloud: after the transform, the crop box, VOXEL and the
 * outlier stage, in the cloud's frame (the target frame with the cloud transform on: the scan needs a z-up frame).
 * d2pc_last_scan returns it.  The d2pc_reproject_*_device batch entries make no scan; d2pc_laser_scan_device makes one
 * of clouds already on the device.
 * Reference: PointCloudToLaserScanNodelet::cloudCb, pointcloud_to_laserscan ROS1 1.4.x, restated from memory (its
 * source was not at hand when this was written -- the same footing as DESIGN.md section 0.1 for the OpenCV dispatch).
 * The recipe:
 *   - message fields: angle_min_f, angle_max_f, angle_increment_f, scan_time, range_min, range_max are the double
 *     params rounded to float; time_increment 0; no intensities.
 *   - n = (uint32)ceilf((angle_max_f - angle_min_f) / angle_increment_f), float arithmetic (the reference computes it
 *     from the message's float fields).
 *   - every range starts at init = +inf when use_inf, otherwise (float)((double)range_max_f + inf_epsilon).
 *   - per point, in this order:
 *       1. skip if x, y or z is NaN (only NaN: +-inf goes on, as std::isnan lets it);
 *       2. skip if (double)z > max_height or (double)z < min_height;
 *       3. r = range(x, y); skip if r < range_min or r > range_max (the double params, not the float fields);
 *       4. a = angle(y, x); skip if a < (double)angle_min_f or a > (double)angle_max_f;
 *       5. k = (int)((a - (double)angle_min_f) / (double)angle_increment_f), double arithmetic, truncated;
 *       6. skip if k >= n.  The reference writes past its vector there (a point exactly on angle_max when the span
 *          is a whole number of increments); this library drops the point.
 *   - ranges[k] = min(init, min over the bin's points of (float)r).
 *     This is the reference's sequential `if (range < ranges[k]) ranges[k] = range` in every point order: with m the
 *     current float value, r < m implies (float)r <= m and r >= m implies (float)r >= m (rounding is monotone and m
 *     is a float), so every step sets m = min(m, (float)r), and a min does not depend on the order.  Every value is
 *     >= 0 (r is a square root, init >= 0 by the checks below), so the device takes the min on the floats' bits.
 *   - range and angle are the library's own (csrc/scan_math.h, one source for the kernel and the C reference):
 *     range = sqrt((double)x*x + (double)y*y) (exact products, one rounded add, a correctly rounded sqrt) and angle a
 *     double atan2 built from IEEE add, sub, mul, div, sqrt and fma only, within 1 ulp for float inputs.  glibc's
 *     hypot and atan2 are within 1 ulp too; the two can pick a different bin or range only for a point within a few
 *     ulp of a bin edge, an angle limit or a range limit (tests/test_oracle_laser_scan.py measures it).
 *   - Defaults follow the nodelet as recalled, unverified: min_height DBL_MIN and max_height DBL_MAX (so z <= 0 is
 *     dropped), angles -pi, pi, pi/180 (n = 360), scan_time 1/30, range_min 0, range_max DBL_MAX, use_inf 1,
 *     inf_epsilon 1.
 * keep_cloud 1 (the default): both outputs; the cloud's bytes, timing spans and BUFFER_TOO_SMALL rules are what they
 * are with the scan off.  keep_cloud 0: the cloud never leaves the device -- no payload copy, no count read-back, only
 * the ranges are copied; d2pc_wait returns a cloud of width 0, data NULL, is_dense 1, and a *_into destination is
 * neither written nor checked against cap.  The ranges' copy runs on the D2H stream behind the kernels, so
 * d2pc_slot_timing's d2h_us covers it.  Plans with the scan never store the cloud from the kernel into host memory
 * ("direct_out").  The setting in force when a frame is submitted is the one its slot uses. */
typedef struct d2pc_laser_scan_params {
  uint32_t struct_size; /* sizeof(d2pc_laser_scan_params) */
  int32_t enabled;      /* 0: off (the default) */
  double min_height, max_height;                 /* DBL_MIN, DBL_MAX; not NaN (+-inf allowed) */
  double angle_min, angle_max, angle_increment;  /* -pi, pi, pi/180; finite */
  double scan_time;                              /* 1/30 */
  double range_min, range_max;                   /* 0, DBL_MAX; finite, 0 <= range_min <= range_max */
  int32_t use_inf;                               /* 1 */
  double inf_epsilon;                            /* 1; finite, >= 0 */
  int32_t keep_cloud;                            /* 1: the cloud is produced as well; 0: only the scan leaves */
} d2pc_laser_scan_params;

/* A scan: the message fields and the ranges.  `ranges` is library-owned pinned host memory, valid until the next call
 * that uses the same pipeline slot (inside a stream sink: until the sink returns). */
typedef struct d2pc_laser_scan {
  float angle_min, angle_max, angle_increment, time_increment, scan_time, range_min, range_max;
  uint32_t n_ranges;
  const float *ranges;
} d2pc_laser_scan;

/* enabled 0, keep_cloud 1, the nodelet's defaults above. */
void d2pc_laser_scan_params_default(d2pc_laser_scan_params *p);
/* D2PC_ERR_INVALID_ARG, keeping the previous setting, for: a non-finite angle or range param; angle_increment_f <= 0
 * or angle_min_f > angle_max_f; range_min < 0, range_max < range_min or inf_epsilon < 0 (NaN included); a NaN height;
 * more than 2^20 ranges; a wrong struct_size. */
int d2pc_set_laser_scan(d2pc_ctx *ctx, const d2pc_laser_scan_params *p);
/* The setting last made (d2pc_laser_scan_params_default's until then). */
int d2pc_get_laser_scan(const d2pc_ctx *ctx, d2pc_laser_scan_params *p);
/* n for these params, with the recipe's float formula (the other checks of d2pc_set_laser_scan apply as well). */
int d2pc_laser_scan_ranges(const d2pc_laser_scan_params *p, uint32_t *n);
/* The scan of the cloud this context last returned (d2pc_wait, the synchronous process_* / *_into and
 * d2pc_fuse_then_process; inside a stream sink, the cloud handed to it).  D2PC_ERR_NOT_READY when the scan was off
 * for that submission, when no cloud has been returned yet, or after a d2pc_wait that returned
 * D2PC_ERR_BUFFER_TOO_SMALL (no cloud was returned then). */
int d2pc_last_scan(const d2pc_ctx *ctx, d2pc_laser_scan *out);
/* The scan alone (the context's setting, which must be enabled) of clouds already on the device, with the argument
 * rules of d2pc_crop_box_device for the input: frame f's input is d_in + f*in_stride bytes, d_in_counts[f] points
 * (NULL: n_max each; a count above n_max counts as n_max), pointers and strides 16-byte aligned, in_stride >= 16*n_max
 * when n_frames > 1, n_max*16 < 2^32, batches of more than 2^31 - 2 points run in chunks of frames.  Frame f's n
 * ranges go to d_ranges + f*ranges_stride bytes: d_ranges and ranges_stride 4-byte aligned, ranges_stride >= 4*n when
 * n_frames > 1, no overlap with the input (D2PC_ERR_INVALID_ARG). */
int d2pc_laser_scan_device(d2pc_ctx *ctx, const uint8_t *d_in, uint32_t n_frames, uint32_t n_max, size_t in_stride,
                           const uint32_t *d_in_counts, float *d_ranges, size_t ranges_stride);

/* ---- occupancy map (octomap_server's insertScan on the device, updated by every published cloud) -------------------
 *
 * Off by default (enabled 0).  With the map on, every host entry point that publishes a cloud (the process_* and
 * *_into calls, submit / d2pc_wait, d2pc_process_stream, d2pc_submit_fusion, d2pc_process_fusion_stream and
 * d2pc_fuse_then_process) also inserts exactly that cloud -- after the transform, the crop box, VOXEL and the outlier
 * stage, in the cloud's frame -- into one occupancy map the context keeps on the device.  The d2pc_reproject_*_device
 * batches do not update it; d2pc_occupancy_insert_device inserts clouds already on the device.
 * Reference: OctomapServer::insertScan (octomap_server) with filter_ground off and compress_map off, on an
 * octomap::OcTree of depth 16, restated from memory (neither octomap's nor octomap_server's source was at hand when
 * this was written -- the footing of the laser scan above).  The recipe:
 *   - origin: o = the cloud transform's translation (m03, m13, m23) when the transform is on, else (0, 0, 0); a float
 *     point3d.
 *   - a point with a non-finite x, y or z is skipped (the pass-through filters drop NaN; coordToKey of +-inf is
 *     undefined).
 *   - keys: per axis k = (int)floor(res_factor * (double)c) + 32768 with res_factor = 1.0 / resolution (double); valid
 *     only when 0 <= k < 65536 (coordToKeyChecked).  A key's centre is ((double)(k - 32768) + 0.5) * resolution.
 *   - range test: d = (p - o).norm(): float subtracts, the sum of squares ((x*x + y*y) + z*z) in float with no FMA,
 *     widened to double, a double sqrt.
 *       - max_range < 0 or d <= max_range: the free cells of computeRayKeys(o, p) join the frame's free set, and
 *         key(p) joins its occupied set when valid;
 *       - otherwise e = o + normalized(p - o) * (float)max_range (octomath's float normalize: each component divided
 *         by (float)norm), and the free cells of computeRayKeys(o, e) join the free set; no occupied cell.
 *   - computeRayKeys(o, e), Amanatides & Woo in 3-D:
 *       1. empty when either key is invalid or the two keys are equal;
 *       2. otherwise the ray starts with the origin's key;
 *       3. length = (float)norm(e - o), dir = (e - o) / length in float;
 *       4. per axis: step = sign(dir); tMax = (centre(k_o) + (double)(float)(step * res * 0.5) - (double)o) /
 *          (double)dir and tDelta = res / fabs(dir), in double; DBL_MAX for both when dir is 0;
 *       5. loop: the axis of the least tMax with strict < in octomap's nesting (tMax0 < tMax1 ? (tMax0 < tMax2 ? 0 : 2)
 *          : (tMax1 < tMax2 ? 1 : 2)); step the key (uint16) and add tDelta; stop when the key equals the end key (not
 *          added) or when min(tMax) > length; otherwise add the key.
 *     csrc/map_math.h holds this math once for the kernels and the C reference.
 *   - update, after every point of the frame: each key of the free set that is not in the occupied set gets one miss,
 *     each key of the occupied set one hit.  A key is updated once per frame, so the order within a frame does not
 *     matter.
 *   - updateNode(key, update): a known voxel that is already >= clamp_max under an update >= 0, or <= clamp_min under
 *     an update <= 0, is left as it is (the early abort -- it matters when the clamp bounds change between frames);
 *     otherwise value = value + update in float (a new voxel starts at 0), then clamped to [clamp_min, clamp_max].
 *   - log-odds: prob_hit, prob_miss, clamp_min, clamp_max and occupancy_thres are probabilities, each converted on the
 *     host as octomap does, (float)log(p / (1 - p)).  A voxel is occupied when log_odds >= occ_thres_log.
 * What rests on recollection and is not verified against the sources: the float / double mix of the DDA (float
 * direction and length, double tMax and tDelta, the float cast of the half-voxel offset); octomath's normalize and
 * norm as float sums; the early abort; that a new voxel starts at log-odds 0; that the max-range branch adds no cell
 * for e itself (some octomap_server versions also mark key(e) free); octomap_server's param names and defaults
 * (resolution 0.05, sensor_model/hit 0.7, /miss 0.4, /min 0.12, /max 0.97, occupancy 0.5 as the OcTree default,
 * sensor_model/max_range -1).
 * Export: the known voxels in Morton order (bits interleaved z, y, x from bit 15 down), which is octomap's leaf
 * iterator order at full depth.  d2pc_occupancy_centers is then what octomap_server publishes on
 * octomap_point_cloud_centers with compress_map off, byte for byte: {(float)centre(kx), (float)centre(ky),
 * (float)centre(kz), 1.0f} per occupied voxel.  octomap merges eight equal siblings into one coarser leaf when it
 * prunes (compress_map on, and as recalled also inside updateNode); it would then publish one coarser point for a
 * uniform octant where this library publishes the eight full-depth voxels with the same value.  d2pc_occupancy_centers
 * stays per full-depth voxel; d2pc_occupancy_octomap below follows updateNode's pruning.
 * The device map: a hash of 8x8x8-voxel bricks (max_bricks of them; the table has 2 * max_bricks slots rounded up to a
 * power of two, each about 4.2 KB).  A frame that would take the map past max_bricks bricks is dropped as a whole: the
 * known map stays bit for bit what it was and d2pc_occupancy_stats counts the drop.  Bricks made by a dropped frame stay
 * unknown (invisible to the export) but count as used.
 * Ordering: updates follow submission order (fusion slots too); the map step of a slot reads its cloud before the slot
 * can be reused.  A d2pc_wait that returns D2PC_ERR_BUFFER_TOO_SMALL has still updated the map.  Plans with the map
 * never store the cloud from the kernel into host memory ("direct_out").
 * keep_cloud: the cloud leaves the device unless an enabled scan or an enabled map says keep_cloud 0; then the host
 * entries return a cloud of width 0, data NULL, is_dense 1 (the laser scan's rules above). */
typedef struct d2pc_occupancy_params {
  uint32_t struct_size; /* sizeof(d2pc_occupancy_params) */
  int32_t enabled;      /* 0: off (the default); the map stays readable */
  double resolution;    /* 0.05 (m); finite, > 0.  A change clears the map */
  double prob_hit, prob_miss;     /* 0.7, 0.4; in (0, 1), hit >= 0.5 >= miss */
  double clamp_min, clamp_max;    /* 0.12, 0.97; in (0, 1), min <= max */
  double occupancy_thres;         /* 0.5; in (0, 1): the export's occupied test */
  double max_range;               /* -1 (m): negative means unlimited; not NaN */
  uint32_t max_bricks;            /* 262144 (about 2.2 GB of device memory); >= 1, <= 2^26.  A change clears the map */
  int32_t keep_cloud;             /* 1: the cloud is produced as well; 0: it stays on the device */
} d2pc_occupancy_params;

/* Counters of the map (d2pc_occupancy_stats). */
typedef struct d2pc_occupancy_info {
  uint64_t frames_inserted; /* frames applied since the map was last cleared */
  uint64_t frames_dropped;  /* frames dropped because the map would pass max_bricks */
  uint64_t known_voxels, occupied_voxels;
  uint64_t bricks_used, bricks_capacity;
} d2pc_occupancy_info;

/* enabled 0, keep_cloud 1, octomap_server's defaults above. */
void d2pc_occupancy_params_default(d2pc_occupancy_params *p);
/* D2PC_ERR_INVALID_ARG, keeping the previous setting, for: a resolution that is not finite and > 0; a probability
 * outside (0, 1); prob_hit < 0.5 or prob_miss > 0.5; clamp_min > clamp_max; a NaN max_range; max_bricks 0 or above
 * 2^26; a wrong struct_size.  A change of resolution or max_bricks clears the map (every frame submitted before the
 * call); every other field travels by value into each submission, like the transform's pose. */
int d2pc_set_occupancy(d2pc_ctx *ctx, const d2pc_occupancy_params *p);
/* The setting last made (d2pc_occupancy_params_default's until then). */
int d2pc_get_occupancy(const d2pc_ctx *ctx, d2pc_occupancy_params *p);
/* Clears the map: every frame submitted before the call is gone, frames submitted after it are inserted. */
int d2pc_occupancy_reset(d2pc_ctx *ctx);
/* Synchronous; reflects every frame submitted before the call. */
int d2pc_occupancy_stats(d2pc_ctx *ctx, d2pc_occupancy_info *out);
/* The centres of the occupied voxels (log_odds >= the current occupancy_thres) as a PointCloud2 of 16-byte PointXYZ
 * {x, y, z, 1.0f} in Morton order, written to dst (cap bytes); *out describes it (is_dense 1, data = dst).
 * Synchronous; reflects every frame submitted before the call.  D2PC_ERR_BUFFER_TOO_SMALL when cap < 16 * n, with
 * out->width = n and out->data NULL. */
int d2pc_occupancy_centers(d2pc_ctx *ctx, uint8_t *dst, size_t cap, d2pc_cloud *out);
/* Every known voxel in Morton order: keys[i] = kx | ky << 16 | kz << 32 and its log-odds.  *n = the number of known
 * voxels; D2PC_ERR_BUFFER_TOO_SMALL when cap < *n (nothing written).  Synchronous, like d2pc_occupancy_centers. */
int d2pc_occupancy_voxels(d2pc_ctx *ctx, uint64_t *keys, float *log_odds, uint64_t cap, uint64_t *n);
/* Inserts clouds already on the device, frame f (in order) from the host origin origins[3f .. 3f+2], with the
 * context's setting, which must be enabled.  The input follows d2pc_crop_box_device's rules: frame f at d_in +
 * f*in_stride bytes, d_in_counts[f] points (NULL: n_max each; above n_max counts as n_max), pointers and strides
 * 16-byte aligned, in_stride >= 16*n_max when n_frames > 1, n_max*16 < 2^32, batches of more than 2^31 - 2 points run
 * in chunks of frames.  Asynchronous: the map step runs after the work queued on the compute stream
 * (d2pc_compute_stream) and after every earlier map update; d2pc_sync waits for it. */
int d2pc_occupancy_insert_device(d2pc_ctx *ctx, const uint8_t *d_in, uint32_t n_frames, uint32_t n_max,
                                 size_t in_stride, const uint32_t *d_in_counts, const float *origins);

/* ---- the map as octomap_msgs/Octomap (octomap_server's /octomap_full and /octomap_binary) ----------------------------
 *
 * Reference: octomap_msgs::fullMapToMsg / binaryMapToMsg of the OcTree octomap_server keeps, restated from memory like
 * the recipe above.  The recipe:
 *   1. tree shape: OccupancyOcTreeBase::updateNode with lazy_eval false (as insertScan calls it) prunes on its way
 *      back up every update path: pruneNode collapses a node when isNodeCollapsible holds (all 8 children exist, none
 *      has children, every child's value == child 0's, a float compare), otherwise updateOccupancyChildren sets the
 *      node to the max of its existing children's log-odds.  Updating a key under a pruned leaf first expands it (8
 *      children with the parent's value).
 *   2. consequence: after any sequence of updates the tree is a function of the known full-depth voxels alone.  A
 *      level-L node (L = 0 the root, 16 a voxel) exists iff some known voxel has its top L Morton digits; it is a leaf
 *      iff L = 16, or all 8^(16-L) voxels under it are known with equal log-odds; it is written iff no proper ancestor
 *      is a leaf; its value is the max log-odds of the voxels under it.  (Every ancestor on an update path is
 *      re-checked bottom-up and nodes off the path do not change, so maximal pruning is an invariant; pruning is
 *      lossless and expanding restores equal children, so each voxel's value is the flat map's.  Log-odds are never
 *      NaN and never -0.0 -- logodds(0.5) is +0 and a new voxel starts at +0 -- so == and bit equality agree.)
 *      tests/test_oracle_octomap_msg.py checks this against a pointer tree that restates updateNode literally.
 *   3. child index at level L: x_bit | y_bit << 1 | z_bit << 2 of key bit 15 - L, the Morton digit the export sorts
 *      by, so pre-order is Morton order, parent before child.
 *   4. full (fullMapToMsg -> OcTree::writeData -> writeNodesRecurs): pre-order over the written nodes; each writes its
 *      float value (4 bytes, little endian), then one byte of std::bitset<8> child-exists mask (bit i = child i; 0 for
 *      a leaf), then its children in index order.  An empty tree writes 0 bytes.
 *   5. binary (binaryMapToMsg -> the const writeBinaryData, so no toMaxLikelihood or prune -> writeBinaryNode): each
 *      written inner node writes 2 bytes in pre-order, children 0-3 then 4-7, child i in the 2 bits at 2i (of its
 *      byte): 0 unknown, 1 free leaf (octomap's "10": bit 2i set), 2 occupied leaf (log-odds >= occ_thres_log of the
 *      current occupancy_thres), 3 has children.  The recursion visits only children with children; the root is
 *      always written as an inner node.  An empty map writes 0 bytes.
 *   6. message: id "OcTree", resolution as float64, binary 0 / 1, data the bytes above without the .ot file header.
 * What rests on recollection and is not verified against the sources: all of items 1, 4, 5 and 6 -- that updateNode
 * prunes with lazy_eval false, isNodeCollapsible's three conditions and its float ==, updateOccupancyChildren's max,
 * expandNode's copies, writeNodesRecurs' value-then-mask layout, writeBinaryNode's bit pairs and its skip of leaf
 * children, that binaryMapToMsg neither converts to maximum likelihood nor prunes, and the message's id and fields.
 * On the device: the known voxels are sorted as for d2pc_occupancy_voxels, then every node's first voxel, leaf level
 * and record offset come from two scans, and one thread per voxel writes the nodes that voxel starts
 * (csrc/occupancy.cu).  The library does this work only when this call is made. */
typedef struct d2pc_octomap {
  const uint8_t *data; /* page-locked memory the library owns: valid until the next call on the context or
                          d2pc_destroy; NULL when size is 0 */
  uint64_t size;       /* bytes of data */
  double resolution;   /* the map's resolution (m) */
  int32_t binary;      /* 0: octomap_full's data, 1: octomap_binary's */
} d2pc_octomap;

/* The map serialized as octomap_msgs/Octomap data: binary 0 the full format, 1 the binary format (recipe above).
 * Synchronous; reflects every frame submitted before the call, like d2pc_occupancy_centers.  An empty map gives size 0
 * and D2PC_OK.  D2PC_ERR_INVALID_ARG for binary outside {0, 1}; D2PC_ERR_NOMEM when a host or device allocation fails,
 * leaving the map and the previous result as they were. */
int d2pc_occupancy_octomap(d2pc_ctx *ctx, int binary, d2pc_octomap *out);

/* ---- the map projected to 2-D as nav_msgs/OccupancyGrid (octomap_server's /projected_map) -----------------------------
 *
 * Reference: OctomapServer::publishAll -> handlePreNodeTraversal, then per leaf handleOccupiedNode / handleFreeNode ->
 * update2DMap, restated from memory like the recipes above, for max_depth 16 (the default), incremental_2D_projection
 * false (the complete map is projected every time), filter_speckles and filter_ground off.  The leaves are the pruned
 * tree's (d2pc_occupancy_octomap's recipe, item 2): a leaf at depth d has a key k per axis (any key inside it).
 *   1. empty map: publishAll returns early when octree.size() <= 1, so no known voxel gives no grid.
 *   2. extent (OcTreeBaseImpl::calcMinMax over the leaves, in double): size = getNodeSize(d) = res * (double)(1 << (16
 *      - d)); c = keyToCoord(k, d), which is ((double)(k - 32768) + 0.5) * res at d = 16 and otherwise
 *      (floor(((double)k - 32768.0) / (double)(1 << (16 - d))) + 0.5) * size (0 at d = 0); lo = c - size / 2.0 and hi =
 *      lo + size (two roundings, not c + size / 2).  min = the least lo, max = the greatest hi, per axis.
 *   3. padding: minX = std::min(minX, -0.5 * min_x_size), maxX = std::max(maxX, 0.5 * min_x_size), the same on y with
 *      min_y_size (so with the default 0 the grid always holds key 32768, the world origin, on x and y; -0.0 and 0.0
 *      give the same key).  The corners become float point3d (z the unpadded min / max) and coordToKeyChecked runs on
 *      all three axes; when either corner has no valid key octomap_server logs an error and this library returns
 *      D2PC_ERR_BAD_DIMS (a voxel at key 65535 can put the max face out of range).
 *   4. grid: width = paddedMax.x - paddedMin.x + 1, height likewise on y; resolution = (float)res; origin.position.x =
 *      (double)(float)keyToCoord(paddedMin.x) - res * 0.5, likewise y; z 0, the orientation left at the message's
 *      default; map_load_time 0.
 *   5. cells, row-major, index (kx - paddedMin.x) + (ky - paddedMin.y) * width, all -1 first.  A leaf passes when c_z
 *      + h > occupancy_min_z && c_z - h < occupancy_max_z (its double centre and h = size / 2.0, strict); it then
 *      covers its 2^(16-d) x 2^(16-d) square of cells: an occupied leaf (log_odds >= the current occupancy_thres) sets
 *      100, a free one sets 0 where the cell is still -1.  So a cell is 100 when a passing occupied leaf covers it,
 *      else 0 when a passing free leaf covers it, else -1, in any leaf order.
 * Per voxel: every known voxel inside a leaf has the leaf's depth and value, and the leaf is complete (all its voxels
 * are known), so the union of its voxels' columns is the leaf's square.  Items 2 and 5 are therefore each voxel doing
 * its own leaf's extent, height test and value over its own column.  A full-depth voxel's own centre and size would
 * not do: they differ from the leaf's in the height test at finite z limits and in the last bit of the extent, which
 * can move a padded key by one.  tests/test_oracle_projected_map.py checks the per-voxel recipe against a pointer tree.
 * What rests on recollection and is not verified against the sources: the early return on size() <= 1; calcMinMax's
 * lo-then-add-size arithmetic; keyToCoord(k, d)'s floor form and its 0 at the root; the padding with std::min /
 * std::max and the float point3d corners; coordToKeyChecked on z too; the origin's float round trip; the height test
 * on the leaf's extent (some older octomap_server releases test the centre alone); occupied overriding free; that the
 * orientation is all four components 0; the param names occupancy_min_z / occupancy_max_z (default -DBL_MAX /
 * DBL_MAX) and min_x_size / min_y_size (default 0).
 * On the device: the known voxels are sorted and each one's leaf level found as for d2pc_occupancy_octomap; one thread
 * per voxel reduces the extent (the host reads six values back and sizes the grid), then ORs a free or occupied code
 * into its cell, and the codes become the cell values (csrc/occupancy.cu).  The library does this work only when this
 * call is made. */
typedef struct d2pc_projected_map_params {
  uint32_t struct_size;   /* sizeof(d2pc_projected_map_params) */
  double occupancy_min_z; /* -DBL_MAX (m): a leaf must reach above it; not NaN (+-inf allowed) */
  double occupancy_max_z; /* DBL_MAX (m): a leaf must reach below it; not NaN (+-inf allowed) */
  double min_x_size;      /* 0 (m): the grid spans at least [-min_x_size / 2, min_x_size / 2]; finite, >= 0 */
  double min_y_size;      /* 0 (m): likewise on y */
} d2pc_projected_map_params;

typedef struct d2pc_grid_map {
  const int8_t *data; /* width * height cells, row-major (row y, column x), each -1, 0 or 100: page-locked memory the
                         library owns, valid until the next call on the context or d2pc_destroy; NULL when empty */
  uint32_t width, height;      /* cells; 0 for an empty map.  width * height can reach 2^32 */
  float resolution;            /* info.resolution (m), the map's resolution as float */
  double origin_x, origin_y;   /* info.origin.position x and y (m) of cell (0, 0)'s corner */
} d2pc_grid_map;

/* octomap_server's defaults above. */
void d2pc_projected_map_params_default(d2pc_projected_map_params *p);
/* The map projected to 2-D (recipe above).  Synchronous; reflects every frame submitted before the call.  An empty map
 * gives width = height = 0, data NULL and D2PC_OK.  D2PC_ERR_INVALID_ARG for a NaN z limit, a min size that is
 * negative or not finite, or a wrong struct_size; D2PC_ERR_BAD_DIMS when a padded corner has no key (item 3);
 * D2PC_ERR_NOMEM when a host or device allocation fails.  The previous result is left as it was on every error. */
int d2pc_occupancy_projected_map(d2pc_ctx *ctx, const d2pc_projected_map_params *p, d2pc_grid_map *out);

/* ---- the disparity callback, host buffers (the reference-facing calls) ------ */

/* Whole DisparityCb (src/disparity_to_point_cloud.cpp:46-92) on one mono8
 * frame in host memory: H2D, median 11, x(1/8), reproject with Q, crop 40,
 * pack {x,y,z,1}, D2H.  Synchronous: `out` is complete on return.  (In CROP mode without a cloud transform the
 * kernel of this call stores the points straight into the page-locked destination, so the transfer to the host
 * runs while the kernel does instead of as a copy behind it: tuning key "direct_out".) */
int d2pc_process_mono8(d2pc_ctx *ctx, const uint8_t *data, uint32_t width, uint32_t height, uint32_t step,
                       d2pc_cloud *out);

/* DisparityCb entered after convertTo (cpp:63 onwards) on a float disparity
 * frame in host memory; step in bytes. */
int d2pc_process_f32(d2pc_ctx *ctx, const float *disp, uint32_t width, uint32_t height, uint32_t step,
                     d2pc_cloud *out);

/* Asynchronous variants on pipeline slot `slot` (0 <= slot < n_slots): H2D,
 * kernels and D2H are enqueued on three streams chained by events, so slots
 * overlap.  The input buffer may be reused once d2pc_wait(slot) returns (it is
 * read by the DMA engine directly when it is pinned -- see d2pc_host_alloc --
 * and staged through library pinned memory otherwise, in which case it may be
 * reused as soon as submit returns). */
int d2pc_submit_mono8(d2pc_ctx *ctx, int slot, const uint8_t *data, uint32_t width, uint32_t height, uint32_t step);
int d2pc_submit_f32(d2pc_ctx *ctx, int slot, const float *disp, uint32_t width, uint32_t height, uint32_t step);
int d2pc_wait(d2pc_ctx *ctx, int slot, d2pc_cloud *out);

/* The same calls with a CALLER-SUPPLIED destination for the cloud (SURVEY.md 8(b) "Ownership"): what
 * pcl::toROSMsg's memcpy into PointCloud2.data does in the reference (src/disparity_to_point_cloud.cpp:84-85)
 * becomes the device-to-host copy itself.  `dst` must hold the whole cloud (16 bytes per point; `cap` bytes are
 * available, D2PC_ERR_BUFFER_TOO_SMALL otherwise -- in CROP mode at submit, in CROP_FINITE mode, where the count
 * is only known afterwards, at wait).  When `dst` is page-locked (d2pc_host_alloc, or any buffer passed through
 * d2pc_host_register, e.g. the storage of a message's data vector) and 16-byte aligned the DMA engine writes
 * straight into it; a pageable `dst` is filled from the library's pinned buffer when the slot is waited on.
 * `dst` must stay valid until d2pc_wait(slot) returns; the cloud returned by d2pc_wait then points at `dst`. */
int d2pc_submit_mono8_into(d2pc_ctx *ctx, int slot, const uint8_t *data, uint32_t width, uint32_t height,
                           uint32_t step, uint8_t *dst, size_t cap);
int d2pc_submit_f32_into(d2pc_ctx *ctx, int slot, const float *disp, uint32_t width, uint32_t height, uint32_t step,
                         uint8_t *dst, size_t cap);
int d2pc_process_mono8_into(d2pc_ctx *ctx, const uint8_t *data, uint32_t width, uint32_t height, uint32_t step,
                            uint8_t *dst, size_t cap, d2pc_cloud *out);
int d2pc_process_f32_into(d2pc_ctx *ctx, const float *disp, uint32_t width, uint32_t height, uint32_t step,
                          uint8_t *dst, size_t cap, d2pc_cloud *out);

/* Per-call timing (the reference's only instrumentation is nine printf lines per frame,
 * src/disparity_to_point_cloud.cpp:47-91).  d2pc_set_timing(ctx, 1) makes the slots' events carry timestamps
 * (waits for the device; call it between frames); after d2pc_wait(slot) d2pc_slot_timing reports where that
 * submission's time went on the device: the spans between the events that chain H2D copy -> kernels -> D2H copy
 * (queueing behind other slots included).  In CROP_FINITE mode d2h_us covers the 4-byte count only (the payload
 * is copied inside d2pc_wait); where the kernel stores the cloud into host memory itself ("direct_out": the
 * synchronous mono8 entries) the transfer is part of kernels_us and d2h_us is ~0; a synchronous call into a pageable
 * caller buffer moves its cloud inside d2pc_wait, outside these spans.  The host-side spans of every entry point are also NVTX ranges ("d2pc submit ...",
 * "d2pc H2D", "d2pc kernels", "d2pc D2H") for Nsight. */
typedef struct d2pc_timing {
  float h2d_us, kernels_us, d2h_us, total_us;
  uint64_t points; /* points of that cloud */
} d2pc_timing;
int d2pc_set_timing(d2pc_ctx *ctx, int enable);
int d2pc_slot_timing(d2pc_ctx *ctx, int slot, d2pc_timing *out);

/* Pinned host memory for buffers the caller wants DMA'd without staging: allocate it here, or page-lock memory
 * the caller already owns (cudaHostRegister; costs about as much as touching every page once, so register
 * long-lived buffers, not one per message). */
int d2pc_host_alloc(void **ptr, size_t bytes);
int d2pc_host_free(void *ptr);
int d2pc_host_register(void *ptr, size_t bytes);
int d2pc_host_unregister(void *ptr);

/* Streams `n_frames` same-sized frames through the slot pipeline and hands every finished cloud to `sink` in
 * frame order (sink may be NULL: the clouds are then produced and dropped).  Frame i is read from
 * frames + (i % ring_len) * frame_stride bytes (ring_len 0 means n_frames, i.e. a plain array); is_f32 selects
 * the float vs mono8 entry.  This is the loop a subscriber thread would run; it is what bench.py's end-to-end
 * figure times. */
typedef void (*d2pc_cloud_sink)(void *user, uint64_t frame_index, const d2pc_cloud *cloud);
int d2pc_process_stream(d2pc_ctx *ctx, const void *frames, uint64_t n_frames, size_t frame_stride, uint64_t ring_len,
                        int is_f32, uint32_t width, uint32_t height, uint32_t step, d2pc_cloud_sink sink,
                        void *user);

/* ---- device-resident entry points (kernel-only figures, chaining) ---------- */

/* All pointers are DEVICE pointers on the context's device; work is enqueued
 * on the context's compute stream and NOT synchronised (d2pc_sync, or CUDA
 * events recorded on d2pc_compute_stream()). */

/* cpp:63-85 for a batch of float frames: frame f at d_disp + f*frame_stride
 * bytes, rows `step` bytes apart.  Points of frame f start at
 * d_points + f*points_stride bytes.  In CROP mode every frame produces
 * (w-2b)*(h-2b) points; in CROP_FINITE mode d_counts[f] (uint32, may be NULL
 * in CROP mode) receives the number of points kept. */
int d2pc_reproject_f32_device(d2pc_ctx *ctx, const float *d_disp, uint32_t n_frames, uint32_t width,
                              uint32_t height, size_t step, size_t frame_stride, uint8_t *d_points,
                              size_t points_stride, uint32_t *d_counts);

/* cpp:55-85 for a batch of mono8 frames (median ksize from the config). */
int d2pc_reproject_mono8_device(d2pc_ctx *ctx, const uint8_t *d_img, uint32_t n_frames, uint32_t width,
                                uint32_t height, size_t step, size_t frame_stride, uint8_t *d_points,
                                size_t points_stride, uint32_t *d_counts);

/* The radius outlier stage alone (the context's d2pc_radius_outlier, which must have a radius > 0), on clouds
 * already on the device -- for chaining, and for clouds that did not come from a disparity frame.  Frame f's
 * input is d_in + f*in_stride bytes, d_in_counts[f] points of 16 bytes (d_in_counts NULL: n_max each; a count
 * above n_max counts as n_max); its kept points go to d_out + f*out_stride and their number to d_out_counts[f].
 * Pointers and strides 16-byte aligned, strides >= 16*n_max when n_frames > 1, n_max*16 < 2^32; the input and the
 * output must not overlap (D2PC_ERR_INVALID_ARG).  n_frames has no other limit: batches of more than 2^31 - 2
 * points run in chunks of frames. */
int d2pc_radius_outlier_device(d2pc_ctx *ctx, const uint8_t *d_in, uint32_t n_frames, uint32_t n_max,
                               size_t in_stride, const uint32_t *d_in_counts, uint8_t *d_out, size_t out_stride,
                               uint32_t *d_out_counts);

/* The crop box alone (the context's d2pc_crop_box, which must be enabled), on clouds already on the device, with the
 * argument rules of d2pc_radius_outlier_device: frame f's input is d_in + f*in_stride bytes, d_in_counts[f] points
 * (NULL: n_max each; a count above n_max counts as n_max), its kept points go to d_out + f*out_stride and their
 * number to d_out_counts[f]; pointers and strides 16-byte aligned, strides >= 16*n_max when n_frames > 1,
 * n_max*16 < 2^32, no overlap of input and output; batches of more than 2^31 - 2 points run in chunks of frames. */
int d2pc_crop_box_device(d2pc_ctx *ctx, const uint8_t *d_in, uint32_t n_frames, uint32_t n_max, size_t in_stride,
                         const uint32_t *d_in_counts, uint8_t *d_out, size_t out_stride, uint32_t *d_out_counts);

/* The cloud transform alone, on clouds already on the device, with the argument rules of d2pc_crop_box_device except:
 *   - d_transforms NULL applies the context's d2pc_cloud_transform, which must be enabled; otherwise frame f uses
 *     the 12 device floats at d_transforms + 12*f (row-major 3x4 [A | t], finiteness not checked), whatever the
 *     context's setting;
 *   - d_out_counts may be NULL; otherwise d_out_counts[f] = frame f's input count (clamped to n_max);
 *   - the output may be the input exactly (d_out == d_in and out_stride == in_stride, in place, as
 *     pcl::transformPointCloud(c, c, T) allows); any other overlap is D2PC_ERR_INVALID_ARG.
 * Positions at or past a frame's count are neither read nor written. */
int d2pc_cloud_transform_device(d2pc_ctx *ctx, const uint8_t *d_in, uint32_t n_frames, uint32_t n_max,
                                size_t in_stride, const uint32_t *d_in_counts, uint8_t *d_out, size_t out_stride,
                                uint32_t *d_out_counts, const float *d_transforms);

/* cv::medianBlur on CV_8UC1, replicate border (cpp:55-57 with ksize 11,
 * depth_map_fusion.cpp:124 with ksize 3).  ksize odd, 3..15. */
int d2pc_median_u8_device(d2pc_ctx *ctx, const uint8_t *d_src, uint32_t width, uint32_t height, size_t src_step,
                          uint8_t *d_dst, size_t dst_step, int ksize);

void *d2pc_compute_stream(d2pc_ctx *ctx); /* cudaStream_t */
int d2pc_sync(d2pc_ctx *ctx);
/* Number of kernels this context has launched since creation (bench.py's gpu_launches). */
uint64_t d2pc_launch_count(const d2pc_ctx *ctx);

/* ---- depth_map_fusion -------------------------------------------------------- */

/* Geometry of src/depth_map_fusion.cpp:237-265 for a w x h frame: rect1 (map /
 * score 1), rect2 (map / score 2, in the rotated frame), rectc (output
 * container), each {x, y, w, h}; dims = {n, fused_w, fused_h}. */
int d2pc_fuse_geometry(const d2pc_ctx *ctx, uint32_t width, uint32_t height, int rect1[4], int rect2[4],
                       int rectc[4], int dims[3]);

/* One DisparityCb1 + DisparityCb2 + publishFusedDepthMap pass
 * (src/depth_map_fusion.cpp:46-62, 103-136) on four same-sized mono8 frames in
 * host memory: rotate map/score 2, crop all four to the common square, merge
 * per pixel, median 3, final border trim.  s1/s2 are the preprocessed score
 * images (what the caches cropped_score_{1,2}_ hold, :77/:96).
 * fused  -> what is published on /fused_depth_map (:134-136)
 * combined -> what is published on /combined_score (:126-127); may be NULL. */
int d2pc_fuse(d2pc_ctx *ctx, const uint8_t *d1, const uint8_t *d2, const uint8_t *s1, const uint8_t *s2,
              uint32_t width, uint32_t height, uint32_t step, d2pc_image *fused, d2pc_image *combined);

/* MatchingScoreCb1 (which = 1, src/depth_map_fusion.cpp:64-80) / MatchingScoreCb2 (which = 2, :82-99) on one
 * mono8 score frame in host memory: [rotate for 2 ->] cropToSquare -> GaussianBlur 13 sigma 3 -> Sobel 2nd
 * derivative ksize 7 x0.03 -> threshold 30 -> GaussianBlur 21 sigma 10 -> score + 2*grad (saturating).
 * out is the n x n image the node caches as cropped_score_k_ (library-owned pinned memory, one buffer per
 * `which`, valid until the next call with the same `which`). */
int d2pc_preprocess_score(d2pc_ctx *ctx, const uint8_t *score, uint32_t width, uint32_t height, uint32_t step,
                          int which, d2pc_image *out);
/* Same with device pointers; d_out is n x n dense. */
int d2pc_preprocess_score_device(d2pc_ctx *ctx, const uint8_t *d_score, uint32_t width, uint32_t height, size_t step,
                                 int which, uint8_t *d_out);

/* d2pc_fuse with the two score inputs given as the n x n preprocessed caches (d2pc_preprocess_score output)
 * instead of full frames: exactly the state publishFusedDepthMap works from. */
int d2pc_fuse_preprocessed(d2pc_ctx *ctx, const uint8_t *d1, const uint8_t *d2, const uint8_t *s1_cropped,
                           const uint8_t *s2_cropped, uint32_t width, uint32_t height, uint32_t step,
                           d2pc_image *fused, d2pc_image *combined);

/* Same, device pointers, enqueued on the compute stream.  d_fused is
 * fused_w x fused_h dense; d_combined n x n dense (may be NULL). */
int d2pc_fuse_device(d2pc_ctx *ctx, const uint8_t *d_d1, const uint8_t *d_d2, const uint8_t *d_s1,
                     const uint8_t *d_s2, uint32_t width, uint32_t height, size_t step, uint8_t *d_fused,
                     uint8_t *d_combined);

/* d2pc_fuse_device with the two scores given as the n x n preprocessed caches (d2pc_preprocess_score_device
 * output, dense): the device-resident form of d2pc_fuse_preprocessed. */
int d2pc_fuse_preprocessed_device(d2pc_ctx *ctx, const uint8_t *d_d1, const uint8_t *d_d2, const uint8_t *d_s1_cropped,
                                  const uint8_t *d_s2_cropped, uint32_t width, uint32_t height, size_t step,
                                  uint8_t *d_fused, uint8_t *d_combined);

/* DepthMapFusion::colorizeDepth (src/depth_map_fusion.cpp:304-358), the RAINBOW_WITH_BLACK colouring of the
 * node's debug views: mono8 in host memory -> 3 bytes per pixel in the byte order the reference stores (and labels
 * "rgb8", :298-299).  out->width = width, out->step = 3 * width. */
int d2pc_colorize_depth(d2pc_ctx *ctx, const uint8_t *gray, uint32_t width, uint32_t height, uint32_t step,
                        d2pc_image *out);

/* BASELINE config 5: fuse four host frames, then run the whole DisparityCb on
 * the fused map without leaving the device. */
int d2pc_fuse_then_process(d2pc_ctx *ctx, const uint8_t *d1, const uint8_t *d2, const uint8_t *s1,
                           const uint8_t *s2, uint32_t width, uint32_t height, uint32_t step, d2pc_cloud *out);

/* The same frame set on the slot pipeline (asynchronous, like d2pc_submit_mono8): H2D of the four frames,
 * [MatchingScoreCb1/2 when preprocess_scores != 0: s1 / s2 are then the raw matching-score frames of
 * src/depth_map_fusion.cpp:64-99; with 0 they are full frames that already hold the preprocessed scores, as for
 * d2pc_fuse], the merge, median 3 + trim, DisparityCb on the fused map and the D2H of the cloud are enqueued on the
 * three streams; collect the cloud with d2pc_wait(ctx, slot, &cloud).  Slots overlap frame sets. */
int d2pc_submit_fusion(d2pc_ctx *ctx, int slot, const uint8_t *d1, const uint8_t *d2, const uint8_t *s1,
                       const uint8_t *s2, uint32_t width, uint32_t height, uint32_t step, int preprocess_scores);

/* Streams n_sets frame sets through d2pc_submit_fusion / d2pc_wait with every slot busy; set i is read from
 * sets + (i % ring_len) * set_stride (ring_len 0 = n_sets) as four frames of step * height bytes back to back in
 * the order d1, d2, s1, s2.  What bench.py --config 5 times end to end. */
int d2pc_process_fusion_stream(d2pc_ctx *ctx, const uint8_t *sets, uint64_t n_sets, size_t set_stride,
                               uint64_t ring_len, uint32_t width, uint32_t height, uint32_t step,
                               int preprocess_scores, d2pc_cloud_sink sink, void *user);

/* ---- ROS1 wire helpers (what Publisher::publish serialises) ------------------- */

/* sensor_msgs/PointCloud2 with header {seq, stamp, cfg.frame_id}; returns the
 * byte count (write happens only if cap suffices; pass NULL/0 to size). */
size_t d2pc_serialize_pointcloud2(const d2pc_ctx *ctx, const d2pc_cloud *cloud, uint32_t seq, uint32_t stamp_sec,
                                  uint32_t stamp_nsec, uint8_t *out, size_t cap);
/* sensor_msgs/LaserScan with header {seq, stamp, cfg.frame_id} and empty intensities; same return rule. */
size_t d2pc_serialize_laserscan(const d2pc_ctx *ctx, const d2pc_laser_scan *scan, uint32_t seq, uint32_t stamp_sec,
                                uint32_t stamp_nsec, uint8_t *out, size_t cap);

/* ---- diagnostics ---------------------------------------------------------------- */

/* Tuning / test hook: integer knobs by name.  Not needed in normal use.
 *   kernels : "rows_per_unit" (CROP: rows per work unit; band / pipeline kernels: rows per tile), "ctas_per_sm",
 *             "median_strip", "median_variant" (0 default: window histogram, 3x3 selection network; 2 window
 *             histogram for every size),
 *             "compact_variant" (0 auto: band kernel where Q allows; 1 park kernel for every Q),
 *             "prefetch_dist" (L2 prefetch distance in work units / tiles; 0 automatic, < 0 off),
 *             "crop_load" (CROP kernel input: 0 TMA box loads where the rows allow, 1 per-row vector loads),
 *             "crop_probe" (1: the CROP kernel stores {d, d, d, 1} instead of points -- a measurement hook that
 *             moves the kernel's traffic without its arithmetic; float input only),
 *             "exact_variant" (0 guarded multiply, 1 Markstein), "zero_numer" (kernel variant that keeps an
 *             exactly-zero X numerator column straight-line: 0 when Q has such a column, 1 always, -1 never),
 *             "fuse_median" (mono8 callback: 0 one fused median + reproject launch where Q allows, -1 always two),
 *             "direct_out" (CROP clouds stored by the kernel straight into the page-locked destination instead of
 *             a D2H copy behind the kernel: 0 the synchronous mono8 entries only, 1 every submission, -1 never),
 *             "force_scalar", "force_generic"
 *   config  : "median_ksize", "border", "offset_x", "offset_y", "fuse_rule", "fuse_median_ksize",
 *             "fuse_crop_left|right|top|bottom" */
int d2pc_set_tuning(d2pc_ctx *ctx, const char *key, int value);

const char *d2pc_strerror(int status);
const char *d2pc_last_cuda_error(const d2pc_ctx *ctx);
int d2pc_abi_version(void);
/* Devices with compute capability 10.x visible to the process. */
int d2pc_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* D2PC_B200_H_ */
