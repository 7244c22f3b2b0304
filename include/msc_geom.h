/*
 * msc_geom.h -- C-ABI of the B200-native geometric-evidence path (libmsc_geom.so).
 *
 * The reference (AgustinRoca/multimodal-scene-captioning) has NO native/FFI interface: its boundary for
 * this path is a set of Python callables (SURVEY.md section 8(b)).  This header is the C-ABI those
 * callables bind to in the drop-in (ctypes, see INTEGRATION.md); each entry point cites the reference
 * function(s) it replaces.  All pointers are DEVICE pointers unless the name ends in _host; sizes are
 * element counts; every call is asynchronous on `stream` (a cudaStream_t passed as void*), never
 * allocates or frees caller-visible memory, never throws, and returns 0 on success or a negative
 * msc_status.  msc_last_error() returns a thread-local message for the last failure.
 *
 * Conventions: quaternions are [w,x,y,z]; a pose7 is (tx,ty,tz,qw,qx,qy,qz) f64; box sizes are (w,l,h)
 * as in nuscenes_loader.py:184; raw sweep points are the .pcd.bin rows (x,y,z,intensity,ring) f32.
 */
#ifndef MSC_GEOM_H
#define MSC_GEOM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSC_ABI_VERSION 2
#define MSC_MAX_CAMS 8
#define MSC_MAX_BOXES_FUSED 255 /* per sample, fused kernel (cull cells hold u8 box ids; 0xff = empty) */
#define MSC_STATS_STRIDE 16
#define MSC_MAX_REPLICAS 8 /* result-table replicas written by the fused kernels themselves (the other GPUs of one box) */

typedef enum {
    MSC_OK = 0,
    MSC_ERR_BAD_ARGUMENT = -1,
    MSC_ERR_LAUNCH = -2,
    MSC_ERR_UNSUPPORTED = -3,
    MSC_ERR_NO_DEVICE = -4
} msc_status;

/* Scalar parameters; names follow the reference's attributes where one exists. */
typedef struct {
    float remove_close_radius; /* devkit remove_close (App. A.1), 1.0                                     */
    float range_min;           /* lidar_agent.py:107 `distances > 1.0`                                    */
    float range_max;           /* lidar_agent.py:107 `distances < self.bev_range`                         */
    float z_min;               /* lidar_agent.py:110 `pc[:,2] > -3.0`                                     */
    float z_max;               /* lidar_agent.py:110 `pc[:,2] < 5.0`                                      */
    float ground_z;            /* lidar_agent.py:115 ground_threshold = -1.4                              */
    float bev_range;           /* lidar_agent.py:49  self.bev_range = 50                                  */
    int32_t bev_res;           /* lidar_agent.py:48  self.bev_resolution (800) / 200 for the [EXT] grid   */
    int32_t image_w;           /* 1600 */
    int32_t image_h;           /* 900  */
    int32_t n_cams;            /* 6, <= MSC_MAX_CAMS */
    uint32_t fov_keep_mask;    /* 0: count per-camera wedge membership only; else keep points in any set camera */
    int32_t centroid_shift;    /* fraction bits of the fixed-point centroid sums, <= 17 (|c| < 64 m)       */
    int32_t intensity_shift;   /* fraction bits of the fixed-point intensity sums (8)                     */
    /* square-root-free range thresholds on s = x*x + y*y (host: msc_geom.geometry.sqrt_thresholds) */
    float s_lo;                /* smallest f32 s with sqrtf(s) > range_min */
    float s_hi;                /* largest  f32 s with sqrtf(s) < range_max */
} msc_params;

/* A batch of samples laid out for the fused kernel.  Sweeps of all samples are concatenated; each sweep's
 * first point must start at a multiple of 4 points (16-byte aligned rows for the bulk copies) and the
 * points buffer must extend 16 bytes past the last sweep. */
typedef struct {
    int32_t n_samples;
    int32_t max_boxes_per_sample;    /* max over samples of the box count (sizes the smem box tables)     */
    int32_t n_boxes;                 /* total boxes in the batch (= sample_box_off[n_samples])            */
    int32_t points_per_sample_hint;  /* typical points per sample (0 = unknown: a 10-sweep sample is assumed); only steers how a batch
                                        smaller than the SM count is split over CTAs, never the results                       */
    const float* points;             /* [n_points_padded, 5] raw sweep rows                               */
    const int32_t* sample_sweep_off; /* [n_samples + 1] index into the sweep arrays                       */
    const uint32_t* sweep_start;     /* [n_sweeps] first point of the sweep (multiple of 4)               */
    const uint32_t* sweep_count;     /* [n_sweeps] points in the sweep                                    */
    const double* sweep_pose;        /* [n_sweeps, 12] row-major 3x4 ref_from_sensor (App. A.1)           */
    const int32_t* sample_box_off;   /* [n_samples + 1] index into boxes                                  */
    const double* boxes;             /* [n_boxes, 10] global frame: center3, size(w,l,h), quat(w,x,y,z)   */
    const double* ego_pose;          /* [n_samples, 7] ego pose at the LIDAR_TOP keyframe                 */
    const double* lidar_calib;       /* [n_samples, 7] LIDAR_TOP calibrated sensor                        */
    const double* cam_ego_pose;      /* [n_samples, n_cams, 7] ego pose at each camera's timestamp        */
    const double* cam_calib;         /* [n_samples, n_cams, 7]                                            */
    const double* cam_K;             /* [n_samples, n_cams, 9] row-major intrinsics                       */
} msc_batch_in;

/* Result tables.  bev_ci interleaves (count u32, intensity sum in Q<intensity_shift> u32) per cell so a
 * cell is one 8-byte word for the out-of-window 64-bit reductions; the kernels zero-fill it themselves. */
typedef struct {
    uint32_t* box_count;   /* [n_boxes]           points inside the box (devkit points_in_box, App. A.2)  */
    float* box_nearest;    /* [n_boxes]           BEV distance of the nearest member point (+inf if none) */
    float* box_centroid;   /* [n_boxes, 3]        centroid of member points (0 if none)                   */
    uint8_t* proj_visible; /* [n_boxes, n_cams]   BoxVisibility.ANY flag (App. A.3)                       */
    float* proj_extent;    /* [n_boxes, n_cams,4] umin,vmin,umax,vmax clipped to the image (0 if hidden)  */
    uint32_t* bev_ci;      /* [n_samples, res, res, 2]                                                    */
    float* bev_height;     /* [n_samples, res, res] running max of z, 0-initialised (lidar_agent.py:543,560) */
    uint32_t* stats;       /* [n_samples, 16]: 0 n_in 1 n_after_close 2 n_kept 3 n_ground 4 n_object
                                               5..12 per-camera wedge counts, 13 flags (bit0: a cell count
                                               reached 65536, intensity sum may have wrapped)              */
} msc_batch_out;

int msc_abi_version(void);
const char* msc_last_error(void);

/* Device properties the host needs for launch configuration and reporting. */
int msc_device_info(int32_t* sm_count, int32_t* smem_optin_bytes, int32_t* cc_major, int32_t* cc_minor);

/*
 * The fused hot path: per-sweep rigid transform + remove_close + range/height filter + FOV wedges +
 * ground/object split + oriented-box membership (count / nearest / centroid) + BEV occupancy/height/
 * intensity grid + box->camera projection, one pass over the raw sweeps.
 * Replaces: LiDARAgent._preprocess_point_cloud / _segment_ground (lidar_agent.py:103-132) and the raster
 * half of _generate_multi_layer_bev (:539-560) for batches, plus the [EXT] rows e1-e5 of SURVEY.md
 * section 8(a) (devkit from_file_multisweep, points_in_box, get_sample_data/view_points/box_in_image).
 * Four launches: fused_tables_kernel (prepared boxes + box -> camera projection + camera wedges + the warp-tile prefix of the batch),
 * fused_cullids_kernel (candidate-box ids per cull cell -> workspace), stream4_straddle_kernel (zero-fill of the samples that are
 * processed in parts) and the streaming kernel stream4_kernel (csrc/stream4.cu).  The batch is partitioned statically in warp tiles:
 * CTA b of G owns tiles [b T / G, (b + 1) T / G), so every SM streams the same number of points whatever the batch size; a sample that
 * straddles CTA boundaries merges its parts with integer reductions (results do not depend on the partition).  fov_keep_mask != 0
 * takes the one-sample-per-CTA kernel of csrc/fused_stream.cu (three launches).
 * workspace: >= msc_fused_workspace_bytes() bytes, 256-byte aligned, owned by the caller, one per stream in flight.
 * Layout rules the library cannot check (the arrays are on the device; msc_geom.engine.DeviceBatch.check_layout does, on the host copy):
 * sweep_start[] multiples of 4, the points buffer 16 bytes longer than the last sweep row.
 * stats[13] bit 0 (a cell count reached 65536) covers the cells of the shared-memory window (the centre of the grid, where counts are
 * high), whatever the partition: a sample split over CTAs sets it exactly when the same sample on one CTA would; cells outside the
 * window are accumulated with 64-bit global reductions and are not scanned.  Bit 31: the sample holds more boxes than the kernel has
 * room for (max_boxes_per_sample under-declared); words 14 and 15 are 0.
 *
 * Context: options, the timing ring and the facts about the last call live in an msc_fused_ctx, created on the current
 * device.  Calls that share a context are serialised by it; contexts are independent, so host threads / streams / devices that each
 * own one never share mutable state.
 */
typedef struct msc_fused_ctx msc_fused_ctx;
int msc_fused_create(msc_fused_ctx** out);
int msc_fused_destroy(msc_fused_ctx* ctx);
size_t msc_fused_workspace_bytes(const msc_fused_ctx* ctx, const msc_params* params, int32_t n_samples, int32_t n_boxes);
int msc_fused_evidence_batch(msc_fused_ctx* ctx, const msc_params* params, const msc_batch_in* in, const msc_batch_out* out,
                             void* workspace, size_t workspace_bytes, void* stream);

/* The same call for one shard of a batch that is spread over the GPUs of one box (SURVEY.md section 8(e): samples are independent,
 * only the small result tables are gathered).  replicas[r] describes where shard-local table entry i also has to land on peer r: the
 * per-box tables, the projection tables and stats of replicas[r] must point at THIS shard's slice of peer r's gathered tables (device
 * pointers into peer-mapped memory, e.g. torch symmetric memory; bev_* members are ignored -- BEV grids stay sharded).  The kernels that
 * produce a table entry store it locally and through every replica (P2P stores over NVLink / NVSwitch), so there is no collective and no
 * copy after the call; the caller only needs a cross-GPU barrier before the gathered tables are read.  n_replicas <= MSC_MAX_REPLICAS;
 * n_replicas = 0 is msc_fused_evidence_batch.  Not available with fov_keep_mask != 0. */
int msc_fused_evidence_batch_replicated(msc_fused_ctx* ctx, const msc_params* params, const msc_batch_in* in, const msc_batch_out* out,
                                        int32_t n_replicas, const msc_batch_out* replicas_host, void* workspace, size_t workspace_bytes,
                                        void* stream);

/* Tunables of the fused kernel (for the benchmark sweep; defaults are chosen at build time).
 * set: "fov" (0/1 per-camera wedge counting), "window" (BEV smem window width in cells, 0 = auto), "fastdiv", "cull_shift" (-1 auto: cull cells of at most 2 m, coarser if the grid would exceed 64 x 64 cells),
 * "config" (0 = auto, the default: stream4.cu; 10 / 7 force stream4.cu / fused_stream.cu; fov_keep_mask != 0 always takes
 * fused_stream.cu), "ppt" (stream4.cu launch shape: 2 = 1024 threads x 2 points per lane, 4 = 512 threads x 4), "grid" (CTAs of the
 * stream4.cu launch, 0 = auto), "time_kernel".  get: also "last_window", "last_smem", "last_fastdiv", "last_grid", "last_config",
 * "tile_pts", "threads", "last_launches". */
int msc_fused_set_option(msc_fused_ctx* ctx, const char* key, int32_t value);
int msc_fused_get_option(msc_fused_ctx* ctx, const char* key, int32_t* value);

/* Measurement aid (no reference counterpart): with option "time_kernel" = 1 every msc_fused_evidence_batch call brackets its
 * streaming kernel -- not the small table kernels before it -- with CUDA events on the caller's stream (a ring of 64 pairs per context).
 * Copies the durations in ms of the most recent n timed calls, oldest first, to out_ms_host after synchronising on their end
 * events.  Returns the number written (<= n) or a negative msc_status.  get_option("last_launches") = kernels the last call launched. */
int msc_fused_kernel_times(msc_fused_ctx* ctx, float* out_ms_host, int32_t n);

/*
 * Materialised multi-sweep aggregation (devkit LidarPointCloud.from_file_multisweep, App. A.1) for one
 * sample: order-preserving, writes rows (x',y',z',intensity) and the per-point time lag.
 * n_out (device u32) receives the number of rows.  block_counts: scratch of ceil(n_sweeps_points/1024)+1 u32.
 */
int msc_aggregate_sweeps(float remove_close_radius, const float* points, int32_t n_sweeps,
                         const uint32_t* sweep_start, const uint32_t* sweep_count, const double* sweep_pose,
                         const float* sweep_time_lag, uint32_t max_points_per_sweep, float* out_xyzi, float* out_time,
                         uint32_t* n_out, uint32_t* scratch, size_t scratch_elems, void* stream);

/*
 * Keyframe path, bit-exact drop-in for LiDARAgent._preprocess_point_cloud + _segment_ground
 * (lidar_agent.py:103-132): order-preserving compaction of the kept rows into `kept` and of the ground /
 * object subsets.  pts has `pitch` floats per row (4 mock loader, 5 devkit view, nuscenes_loader.py:152-155);
 * outputs are dense (n,4).  counts (device u32[3]) = n_kept, n_ground, n_object.  split_only != 0 skips the range/height
 * gate: that is _segment_ground on its own (every row is kept; rows whose z is NaN land in `object`, like pc[~mask]).
 */
int msc_keyframe_filter_split(const msc_params* params, const float* pts, uint32_t n, int32_t pitch, int32_t split_only,
                              float* kept, float* ground, float* object, uint32_t* counts, uint32_t* scratch,
                              size_t scratch_elems, void* stream);

/*
 * Keyframe BEV raster layers, bit-exact for the pre-overlay half of LiDARAgent._generate_multi_layer_bev
 * (lidar_agent.py:539-597): count u32, height f32 (0-initialised running max), semantic BGR u8 (ground
 * colour, then object hot-colormap, last point in array order wins).  ground/object are dense (n,4).
 * winner: scratch u32[res*res]; zrange: scratch u32[2].  Arrays are not flipped.
 */
int msc_keyframe_bev(const msc_params* params, const float* ground, uint32_t n_ground, const float* object,
                     uint32_t n_object, uint32_t* count, float* height, uint8_t* semantic_bgr, uint32_t* winner,
                     uint32_t* zrange, void* stream);

/* Raw-cloud statistics (RawGPT4oBaseline._describe_point_cloud, baseline_gpt4o.py:276-285):
 * out7 (device f64[7]) = min x,y,z, max x,y,z, sum of sqrt(x^2+y^2). */
int msc_cloud_stats(const float* pts, uint32_t n, int32_t pitch, double* out7, void* stream);

/* Per-annotation table (SceneGraphAgent._parse_annotations, scenegraph_agent.py:186-225; zones :281-295;
 * RawGPT4oBaseline._describe_annotations region flags, baseline_gpt4o.py:304-317).  xy, vel: [n,2] f64.
 * direction: 0 front 1 left 2 back 3 right; zone: 0..8 in the order of scenegraph_agent.py:136-146, 255 none;
 * region_bits: bit0 x>0, bit1 y>0. */
int msc_annotation_table(int32_t n, const double* xy, const double* vel, double* distance, uint8_t* direction,
                         uint8_t* moving, uint8_t* zone, uint8_t* region_bits, void* stream);

/* Box footprints for the relation table: rect [n,6] f64 = x, y, ux, uy, half_len, half_wid in the ego frame
 * of ego_pose (NULL: stay in the loader's global frame). */
int msc_box_footprints(int32_t n, const double* boxes, const double* ego_pose, double* rect, void* stream);

/* [EXT] pairwise relation table for n annotations: dist/bearing f32 [n,n], category/overlap u8 [n,n]. */
int msc_relation_table(int32_t n, const double* rect, float* dist, float* bearing, uint8_t* category,
                       uint8_t* overlap, void* stream);

/* Batched form: sample s owns rect rows [box_off[s], box_off[s+1]) (box_off: device i32[n_samples+1]) and writes its n_s x n_s tables
 * at element offset pair_off[s] (device i64[n_samples]) of the four output arrays.  max_boxes = max n_s. */
int msc_relation_table_batch(int32_t n_samples, int32_t max_boxes, const int32_t* box_off, const int64_t* pair_off, const double* rect,
                             float* dist, float* bearing, uint8_t* category, uint8_t* overlap, void* stream);

/*
 * Camera-image decode for the on-disk step (SURVEY.md section 8(f) rank 3).  Replaces `np.array(Image.open(path))` in
 * NuScenesLoader._load_camera (nuscenes_loader.py:136-144), i.e. libjpeg(-turbo)'s default decompression (ISLOW integer IDCT, "fancy"
 * chroma upsampling, fixed-point YCbCr -> RGB), BIT-IDENTICALLY.  The entropy decode is sequential per image and runs on the host
 * (msc_jpeg_entropy_decode_host: thread-safe, call it from one thread per image); dequantisation + IDCT + upsampling + colour
 * conversion run on the device (msc_jpeg_reconstruct).  Baseline / extended-sequential Huffman, 8 bits, grayscale or JFIF YCbCr in
 * one interleaved scan, 4:4:4 / 4:2:2 / 4:2:0, restart intervals; anything else returns MSC_ERR_UNSUPPORTED.
 */
typedef struct {
    int32_t h, v;                /* sampling factors                                                  */
    int32_t blocks_x, blocks_y;  /* 8x8 blocks per row / column of the (MCU-padded) component plane   */
    int32_t ds_w, ds_h;          /* libjpeg's downsampled_width / downsampled_height                  */
    int64_t coef_off;            /* first coefficient of the component in the coefficient buffer      */
    int64_t plane_off;           /* first byte of the component in the plane scratch buffer           */
    uint16_t qt[64];             /* quantisation table, natural (row-major) order                     */
} msc_jpeg_comp;
typedef struct {
    int32_t width, height, n_comp, hmax, vmax, mcus_x, mcus_y, reserved_;
    int64_t coef_elems;          /* int16 coefficients the entropy decode produces (all components)   */
    int64_t plane_bytes;         /* device scratch for the component planes                           */
    msc_jpeg_comp comp[3];
} msc_jpeg_desc;
/* host only: parse the headers of a JPEG stream held in host memory */
int msc_jpeg_info(const uint8_t* jpeg_host, size_t nbytes, msc_jpeg_desc* desc_host);
/* host only: Huffman-decode the scan into coef_host[desc->coef_elems] (per component: [blocks_y][blocks_x][64], natural order) */
int msc_jpeg_entropy_decode_host(const uint8_t* jpeg_host, size_t nbytes, const msc_jpeg_desc* desc_host, int16_t* coef_host);
/* device: coef (device, as produced above) -> out (device): [height, width, 3] RGB u8, or [height, width] for one component.
 * planes: device scratch of desc->plane_bytes bytes. */
int msc_jpeg_reconstruct(const msc_jpeg_desc* desc_host, const int16_t* coef, uint8_t* planes, uint8_t* out, void* stream);

/* [EXT] standalone box -> camera projection (also fused into msc_fused_evidence_batch). */
int msc_project_boxes(int32_t n_boxes, const double* boxes, int32_t n_cams, const double* cam_ego_pose,
                      const double* cam_calib, const double* cam_K, int32_t image_w, int32_t image_h,
                      uint8_t* visible, float* extent, void* stream);

/* Per-cluster axis-aligned metadata (lidar_agent.py:200-204): out [n_clusters, 11] f32 =
 * min3, max3, center3, distance, num_points.  labels: i32 per row of pts (-1 = noise). */
int msc_cluster_aabb(const float* pts, uint32_t n, int32_t pitch, const int32_t* labels, int32_t n_clusters,
                     float* out11, void* stream);

/* Per-cluster 4-view raster the reference sends to its VLM (LiDARAgent._generate_cluster_visualization,
 * lidar_agent.py:241-356), points only (axes / titles / mosaic are drawn on the host afterwards).
 * pts_xyzi: dense (n,4) object points; order: point indices grouped by cluster, original order inside a cluster;
 * cluster_off: [n_clusters+1] offsets into order; center_scale: [n_clusters,4] f32 = cluster mean (:255) and scale (:264),
 * computed on the host with the reference's own arithmetic; keys: scratch u32 [n_clusters,512,512]; irange: scratch
 * u32 [n_clusters,4,2]; out_bgr: u8 [n_clusters,512,512,3]. */
int msc_cluster_views(const float* pts_xyzi, const uint32_t* order, const int32_t* cluster_off, int32_t n_clusters,
                      int32_t max_cluster_points, const float* center_scale, uint32_t* keys, uint32_t* irange, uint8_t* out_bgr,
                      void* stream);

/* DBSCAN with scikit-learn's labelling (reference call site LiDARAgent._detect_objects_3d, lidar_agent.py:148-153):
 * float64 neighbour relation, clusters numbered by their smallest core index, border points take the smallest adjacent
 * cluster number, noise = -1.  pts: rows of `pitch` floats (xyz first).  origin / cell / dims describe a host-chosen grid
 * of cubic cells (cell >= eps) covering the points.  labels: device i32[n]; n_clusters_host: host int.  SYNCHRONOUS on
 * `stream`.  workspace >= msc_dbscan_workspace_bytes(n, dims). */
size_t msc_dbscan_workspace_bytes(uint32_t n, const int32_t dims[3]);
int msc_dbscan(const float* pts, uint32_t n, int32_t pitch, double eps, int32_t min_samples, const double origin[3], double cell,
               const int32_t dims[3], int32_t* labels, int32_t* n_clusters_host, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MSC_GEOM_H */
