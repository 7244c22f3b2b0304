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

#define MSC_ABI_VERSION 3
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

/*
 * Batched camera-frame decode with every stage on the device, the Huffman decode included (DESIGN.md section 4.9).
 *
 * msc_jpeg_decode_plan (host only) parses a file's headers with the same parser as msc_jpeg_info -- so it accepts and refuses exactly
 * the same files with the same status -- and fills a fixed-size record: the descriptor, where the entropy-coded scan lies in the file
 * (scan_off: the byte after the SOS header; scan_bytes: from there to the end of the file), the restart interval, the per-component
 * Huffman table selectors and the decode tables of every table the file defines (Annex F.2.2.3, plus a 9-bit lookahead).
 *
 * msc_jpeg_decode_batch decodes n files in one stream-ordered call.  files: device bytes, file i at files[file_off_host[i]] (its
 * plans_host[i] must come from those bytes).  Image i writes
 *   coef[coef_off_host[i] .. + plans_host[i].desc.coef_elems): int16, equal to msc_jpeg_entropy_decode_host (per component
 *          [blocks_y][blocks_x][64], natural order, DC predicted); `coef` must be 16-byte aligned and coef_off_host[i] a multiple of 8;
 *   out[out_off_host[i] ..): the frame, equal to msc_jpeg_reconstruct -- [height][width][3] RGB u8, or [height][width] for one component;
 *   status[i] (device i32): 0, or MSC_ERR_BAD_ARGUMENT where msc_jpeg_entropy_decode_host fails (a corrupt code, a DC size above 15,
 *          an AC run past coefficient 63, a missing restart marker).  A failed image's coef and out regions hold unspecified values;
 *          every other image of the call is decoded exactly, and nothing outside the n regions is written.
 * The bit stream reads like the host decoder's: a stuffed FF 00 is one FF byte; at any other marker, and past the end of the file, it
 * reads as zero bits; decoding stops at the MCU count.  With a restart interval, segment k starts after the k-th FF D0..D7 of the scan.
 * Four launches whatever the data, no allocation, no host synchronisation; plans_host and the offsets are copied into the workspace
 * (one cudaMemcpyAsync), so they may be reused when the call returns.  workspace >= msc_jpeg_decode_batch_workspace_bytes(n, plans_host)
 * bytes, 256-byte aligned (0 = arguments out of range).  n < 0, a NULL pointer with n > 0, a plan that is not a supported sequential
 * file, a scan of 2^28 bytes or more, a misaligned `coef` or coef offset, a workspace that is short or not 256-byte aligned:
 * MSC_ERR_BAD_ARGUMENT before anything is launched.
 * n = 0 is a successful no-op.
 */
typedef struct {
    uint16_t look[512];  /* 9-bit lookahead: (code length << 8) | symbol, 0 = the code is longer than 9 bits */
    int32_t maxcode[18]; /* per code length the largest code, -1 when there is none                          */
    int32_t valptr[17];  /* per code length: index in vals of its first symbol minus its first code          */
    uint8_t vals[256];   /* symbols in code order                                                           */
} msc_jpeg_huff;
typedef struct {
    msc_jpeg_desc desc;
    int64_t scan_off, scan_bytes;
    int32_t restart_interval; /* MCUs per restart segment, 0 = none */
    int32_t td[3], ta[3];     /* DC / AC table of each component     */
    int32_t reserved_;
    msc_jpeg_huff dc[4], ac[4]; /* tables the file does not define are zero */
} msc_jpeg_plan;
int msc_jpeg_decode_plan(const uint8_t* jpeg_host, size_t nbytes, msc_jpeg_plan* plan_host);
size_t msc_jpeg_decode_batch_workspace_bytes(int32_t n, const msc_jpeg_plan* plans_host);
int msc_jpeg_decode_batch(int32_t n, const msc_jpeg_plan* plans_host, const uint8_t* files, const int64_t* file_off_host, int16_t* coef,
                          const int64_t* coef_off_host, uint8_t* out, const int64_t* out_off_host, int32_t* status, void* workspace,
                          size_t workspace_bytes, void* stream);

/*
 * Camera-frame encode (CameraAgent._encode_image, camera_agent.py:128-137): image i of the batch becomes, byte for byte, the file
 * `PIL.Image.fromarray(rgb[i]).save(buf, "JPEG", quality=quality)` writes -- libjpeg-turbo's default compression: JFIF 1.01, 4:2:0, the
 * Annex K tables (quantisation scaled by jpeg_set_quality, standard Huffman tables), slow-integer FDCT, no restart markers.
 * rgb: device [n_images][height][width][3] u8, contiguous.  The files go back to back into the device arena `out`; image i is
 * out[out_off[i] .. out_off[i + 1]) (out_off: device i64[n_images + 1]).  status (device i32[1]) is written by the call: 0, or 1 when
 * the files need more than out_bytes -- then nothing is written to `out`, but out_off is still exact, so out_off[n_images] is the arena
 * size a second call needs.  Stream-ordered: no host synchronisation, no allocation; the results do not depend on the other images of the
 * batch.  workspace: >= msc_jpeg_encode_workspace_bytes(...) bytes, 256-byte aligned (the size does not depend on out_bytes: each
 * image's scan is packed in a region sized for its worst case before its stuffed size is known; 0 = arguments out of range).
 * quality outside 1..100, height or width outside 1..65535, a NULL pointer with n_images > 0 or a short workspace: MSC_ERR_BAD_ARGUMENT
 * before anything is launched.  n_images = 0 is a successful no-op.
 */
size_t msc_jpeg_encode_workspace_bytes(int32_t n_images, int32_t height, int32_t width, size_t out_bytes);
int msc_jpeg_encode_batch(int32_t n_images, int32_t height, int32_t width, int32_t quality, const uint8_t* rgb, uint8_t* out, size_t out_bytes,
                          int64_t* out_off, int32_t* status, void* workspace, size_t workspace_bytes, void* stream);

/* [EXT] standalone box -> camera projection (also fused into msc_fused_evidence_batch). */
int msc_project_boxes(int32_t n_boxes, const double* boxes, int32_t n_cams, const double* cam_ego_pose,
                      const double* cam_calib, const double* cam_K, int32_t image_w, int32_t image_h,
                      uint8_t* visible, float* extent, void* stream);

/*
 * [EXT] row e7: LiDAR -> camera projection (devkit NuScenesExplorer.map_pointcloud_to_image), batched.  Per sample and camera a
 * downsampled depth map -- the minimum depth of the returns that land in each ds x ds pixel block -- and per (box, camera) how much of
 * the box's projected extent has LiDAR returns on it or in front of it.
 * Points: the multi-sweep cloud of msc_aggregate_sweeps (remove_close in the sweep's frame, then the f64 fma transform into the keyframe
 * LIDAR_TOP frame "ref"); no range or height gate.  Per (sample, camera) P = K [R | t] (3x4, f64 composed without FMA, rounded once to
 * f32) maps ref to the image; a point lands in camera c iff w > min_dist and 1 < u < W-1 and 1 < v < H-1 (all strict), where
 * (a, b, w) = P (x, y, z, 1) in f32 fmaf chains, u = a / w, v = b / w (IEEE division).  For nuScenes intrinsics (third row of K is
 * (0, 0, 1)) w is the camera-frame depth.  The pixel is ((int)u, (int)v), its block (px / ds, py / ds); NaN rows land nowhere; a point
 * may land in several cameras.  The normative definition is orc_camera_depth_sample / orc_box_depth_support of the test oracle.
 * Outputs (every element is written by the call; the caller does not pre-fill):
 *   depth       f32 [n_samples, n_cams, ceil(H/ds), ceil(W/ds)]: minimum w per block, +inf where no point lands;
 *   cam_points  u32 [n_samples, n_cams]: points that land in the camera;
 *   box_support u32 [n_boxes, n_cams, 4] (may be NULL): n_blocks, n_hit, n_front, n_on over the blocks of the box's clipped image
 *               extent (the proj_visible / proj_extent of msc_project_boxes): blocks bx in [(int)umin / ds, min((int)umax, W-1) / ds],
 *               likewise by; n_hit: finite depth; n_front: hit and (double)d < zlo - margin (something nearer hides the box);
 *               n_on: other hits with (double)d <= zhi + margin, where zlo / zhi are the min / max camera-frame Z of the 8 corners
 *               (f64).  All four are 0 for a box that is not visible.
 * From msc_params only remove_close_radius, image_w, image_h and n_cams are used.  The results are bit-reproducible and independent of
 * the launch shape (the depth minimum and the counts are order-independent integer reductions).  Stream-ordered: no host
 * synchronisation, no allocation.  n_samples = 0 is a successful no-op.
 */
typedef struct {
    float min_dist;       /* devkit map_pointcloud_to_image min_dist, 1.0; >= 0 */
    int32_t downsample;   /* ds >= 1: pixel block edge of the depth map, 8 */
    float support_margin; /* metres, >= 0, 0.5 */
} msc_depth_params;
typedef struct {
    float* depth;
    uint32_t* cam_points;
    uint32_t* box_support; /* may be NULL */
} msc_depth_out;
int msc_camera_depth_batch(const msc_params* params, const msc_depth_params* dp, const msc_batch_in* in, const msc_depth_out* out,
                           void* stream);

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
 * cluster number, noise = -1.  pts: rows of `pitch` floats (xyz first), n < 2^31 - 1.  origin / cell / dims describe a
 * host-chosen grid of cubic cells (cell >= eps, fewer than 2^31 cells) covering the points; it sets only the width of the sorted
 * cell keys, the workspace is O(n).  labels: device i32[n]; n_clusters_host: host int.  SYNCHRONOUS on `stream` (one host
 * synchronisation).  workspace >= msc_dbscan_workspace_bytes(n, dims), which is 0 for n or dims out of range. */
size_t msc_dbscan_workspace_bytes(uint32_t n, const int32_t dims[3]);
int msc_dbscan(const float* pts, uint32_t n, int32_t pitch, double eps, int32_t min_samples, const double origin[3], double cell,
               const int32_t dims[3], int32_t* labels, int32_t* n_clusters_host, void* workspace, size_t workspace_bytes, void* stream);

/*
 * The reference's own LiDAR evidence (LiDARAgent.process up to the classifier, lidar_agent.py:103-209) for every sample of a packed
 * batch in one stream-ordered call.  The keyframe of sample s is sweep sample_sweep_off[s] (raw rows, sensor frame); a sample without
 * sweeps has an empty keyframe.  Per sample, bit-identical to the single-keyframe path run on that keyframe:
 *   ground / object rows (x, y, z, intensity) in input order, as msc_keyframe_filter_split; counts [s] = kept, ground, object;
 *   labels of the object rows, as msc_dbscan(eps, min_samples) (scikit-learn's labelling; points of different samples are never
 *   neighbours), numbered per sample from 0;
 *   the cluster table, as msc_cluster_aabb: record k of sample s at row object_off[s] + k (k < n_clusters[s] <= object rows), plus
 *   cluster_first, the smallest object-row index (within the sample) labelled k, and noise_first[s], that of the first noise row
 *   (-1: none).
 * Only the keyframe's gate and split parameters of msc_params are used (range_min, range_max, z_min, z_max, ground_z); the DBSCAN grid
 * is derived from them.  Row arrays are sized by row_capacity >= the batch's total keyframe rows; ground and object rows of sample s
 * start at ground_off[s] / object_off[s].  status (device u32[1]) is written by the call: 0 on success, bit 0 if the component merge
 * left an edge unmerged, bit 1 if the keyframes hold more than row_capacity rows (every sample then reads as empty).  A set bit means
 * the results must not be used.  No host synchronisation, no allocation: workspace >= msc_lidar_batch_workspace_bytes(...), 256-byte
 * aligned.  eps <= 0, min_samples < 1, NULL outputs or a short workspace: MSC_ERR_BAD_ARGUMENT.  n_samples = 0 is a successful no-op.
 */
typedef struct {
    uint32_t row_capacity;
    uint32_t* counts;         /* [n_samples, 3] kept, ground, object            */
    uint32_t* ground_off;     /* [n_samples]                                     */
    uint32_t* object_off;     /* [n_samples]                                     */
    float* ground;            /* [row_capacity, 4]                               */
    float* object;            /* [row_capacity, 4]                               */
    int32_t* labels;          /* [row_capacity] per object row, -1 noise        */
    int32_t* n_clusters;      /* [n_samples]                                     */
    float* clusters;          /* [row_capacity, 11] min3 max3 center3 distance num_points */
    int32_t* cluster_first;   /* [row_capacity]                                  */
    int32_t* noise_first;     /* [n_samples]                                     */
    uint32_t* status;         /* [1]                                             */
} msc_lidar_batch_out;
size_t msc_lidar_batch_workspace_bytes(const msc_params* params, double eps, int32_t n_samples, uint32_t row_capacity);
int msc_lidar_batch(const msc_params* params, double eps, int32_t min_samples, const msc_batch_in* in, const msc_lidar_batch_out* out,
                    void* workspace, size_t workspace_bytes, void* stream);

/*
 * [EXT] LiDAR clusters -> annotated boxes, for every sample of an msc_lidar_batch result in one stream-ordered call.  `in` is the batch
 * given to msc_lidar_batch and `rows` its output; n_samples must equal in->n_samples.  Box b of sample s is prepared as in the fused
 * path (global -> ego_pose[s] -> lidar_calib[s] in f64, the points_in_box vectors rounded to f32) and an object row (x, y, z) of
 * sample s -- as msc_lidar_batch wrote it, in the keyframe's sensor frame -- lies in it iff the devkit points_in_box test (App. A.2,
 * f32 fmaf chains, closed intervals) holds; NaN rows lie in no box.  The normative definition is orc_cluster_match_sample of the test
 * oracle.  Outputs (only these elements are written; the caller does not pre-fill):
 *   cluster i32 [row_capacity, 3]: cluster k of sample s at row object_off[s] + k (k < n_clusters[s], the cluster table's indexing):
 *           match_box (the sample-local box holding most of the cluster's rows; ties: the smaller index; -1: no row in any box),
 *           match_points (its rows in that box), in_any_box (its rows inside at least one box);
 *   box     i32 [in->n_boxes, 5]: rows (object rows inside, noise included), cluster_rows (rows inside with a label >= 0), clusters
 *           (labels with a row inside), best_cluster (the label with most rows inside; ties: the smaller label; -1: none),
 *           best_points (its rows inside).
 * Any number of clusters and boxes per sample: work items of 128 boxes x 64 labels re-read the sample's rows.  Results are integers and do
 * not depend on the launch shape or the row order.  A set msc_lidar_batch status means the rows, and so these results, must not be used.
 * No host synchronisation, no allocation: workspace >= msc_cluster_match_batch_workspace_bytes(...) (O(row_capacity + n_boxes)),
 * 256-byte aligned.  NULL arguments or buffers, a short workspace, n_samples different from the batch's and negative counts:
 * MSC_ERR_BAD_ARGUMENT before anything is launched.  n_samples = 0 is a successful no-op.
 */
typedef struct {
    int32_t* cluster; /* [row_capacity, 3] match_box, match_points, in_any_box                    */
    int32_t* box;     /* [n_boxes, 5] rows, cluster_rows, clusters, best_cluster, best_points   */
} msc_cluster_match_out;
size_t msc_cluster_match_batch_workspace_bytes(int32_t n_samples, int32_t n_boxes, uint32_t row_capacity);
int msc_cluster_match_batch(const msc_batch_in* in, const msc_lidar_batch_out* rows, int32_t n_samples, const msc_cluster_match_out* out,
                            void* workspace, size_t workspace_bytes, void* stream);

/*
 * The finished BEV of LiDARAgent._generate_multi_layer_bev (lidar_agent.py:539-634) for samples [first, first + n) of an
 * msc_lidar_batch result of n_samples samples, in one stream-ordered call.  From `rows` only ground, object, ground_off, object_off and
 * counts are read; from msc_params only bev_res (res) and bev_range.  Image i (sample first + i), byte-identical to the host path
 * finish_bev_layers(msc_keyframe_bev(...)) on that sample's rows:
 *   semantic u8 [n, res, res, 3] BGR: the raster colours, flipped vertically, with the overlays written over them;
 *   height   f32 [n, res, res]: the largest z > 0 per cell (0 elsewhere), flipped;
 *   density  u8 [n, res, res]: (u8)(lut[c] / lut[cmax] * 255) in float32 (round to nearest per step, truncated), c the cell's rows and
 *            cmax the sample's largest c, flipped; all 0 when cmax = 0.
 * lut f32 [lut_len]: the density table, entry c = NumPy's float32 log1p(c).  A sample whose cmax >= lut_len sets bit 0 of *status
 * (device u32, OR-ed into: the caller clears it) and gets density 0; the results must then not be used.
 * stamp u32 [stamp_len, 2]: the overlays as (pixel index y * res + x, B | G << 8 | R << 16), written last; pixels >= res * res are
 * skipped.  Nothing outside the n images is written.  No host synchronisation, no allocation: workspace >=
 * msc_keyframe_bev_batch_workspace_bytes(res, n) (8 res^2 bytes per sample and 16 more), 256-byte aligned.  res outside
 * [1, 8192], a window outside [0, n_samples), n > 65535, lut_len < 1, NULL buffers or a short workspace: MSC_ERR_BAD_ARGUMENT.
 * n = 0 is a successful no-op.
 */
size_t msc_keyframe_bev_batch_workspace_bytes(int32_t bev_res, int32_t n);
int msc_keyframe_bev_batch(const msc_params* params, const msc_lidar_batch_out* rows, int32_t n_samples, int32_t first, int32_t n,
                           const float* lut, int32_t lut_len, const uint32_t* stamp, int32_t stamp_len, uint8_t* semantic, float* height,
                           uint8_t* density, uint32_t* status, void* workspace, size_t workspace_bytes, void* stream);

/*
 * The finished 4-view images of LiDARAgent._generate_cluster_visualization (lidar_agent.py:241-356) for n_views clusters in one
 * stream-ordered call.  rows: f32 [*, 4] (x, y, z, intensity) and labels i32 [*] on the device; views: HOST i32 [n_views, 3] =
 * (row_begin, row_end, label), copied into the workspace.  The points of view v are the rows r in [row_begin, row_end) with
 * labels[r] == label, in row order (for msc_lidar_batch's output: (object_off[s], object_off[s] + object count, k) is cluster k of
 * sample s).  Image v, out_bgr u8 [n_views, 512, 512, 3], is byte-identical to the host path: msc_cluster_views with the cluster mean
 * (NumPy's float32 mean: a sequential sum in row order over n) and scale (fl32(89.6 / max_range), 1 when max_range is 0), then the
 * axes and titles given as stamp u32 [stamp_len, 2] (pixel y * 512 + x, B | G << 8 | R << 16), written last.  A view of more than
 * max_view_points points sets bit 0 of *status (device u32, OR-ed into: the caller clears it); its image must not be used.
 * No host synchronisation, no allocation: workspace >= msc_cluster_views_batch_workspace_bytes(n_views, max_view_points) (1 MiB of
 * keys and 4 max_view_points bytes per view, plus a few words), 256-byte aligned.  n_views outside [0, 65535], max_view_points outside
 * [0, 2^24), an empty or inverted row range, NULL buffers or a short workspace: MSC_ERR_BAD_ARGUMENT.  n_views = 0 is a successful
 * no-op.
 */
size_t msc_cluster_views_batch_workspace_bytes(int32_t n_views, int32_t max_view_points);
int msc_cluster_views_batch(const float* rows, const int32_t* labels, const int32_t* views, int32_t n_views, int32_t max_view_points,
                            const uint32_t* stamp, int32_t stamp_len, uint8_t* out_bgr, uint32_t* status, void* workspace,
                            size_t workspace_bytes, void* stream);

/*
 * PNG files of n 8-bit images (h x w x c; c = 3: RGB, colour type 2; c = 1: grey, colour type 0) in one stream-ordered call.  Each file
 * is the signature, IHDR (width, height, depth 8, colour type, 0, 0, 0: Pillow's), one IDAT and IEND, every CRC-32 correct.  The IDAT
 * data is one zlib stream (header 78 9C, Adler-32) that inflates to exactly the payload of Pillow's Image.fromarray(img).save(buf, "PNG"):
 * per row (the row above row 0 is zeros) a filter byte and the filtered row, the filter chosen as ZipEncode.c does -- None, Up, Sub,
 * Paeth tried in that order, cost sum(v < 128 ? v : 256 - v) over the filtered bytes, a candidate taken only when strictly cheaper,
 * Average never.  The deflate data is one dynamic-Huffman block or stored blocks of up to 65,535 bytes, whichever is smaller, so a file
 * is never larger than 57 + 6 + raw + 5 ceil(raw / 65535) bytes (raw = h (1 + w c)).  swap_rb reads BGR pixels as RGB.  A file depends
 * only on its image: not on the other images of the call, nor on the launch shape.
 * Images may differ in shape; rows are row_pitch bytes apart on the device.  The descriptors are copied into the workspace.  The files
 * are back to back in `out`: file i is out[out_off[i] .. out_off[i + 1]) (out_off: device i64 [n + 1]).  *status (device i32) is 1 when
 * they need more than out_bytes; then nothing is written to `out`, but out_off is exact.  No host synchronisation, no allocation:
 * workspace >= msc_png_encode_workspace_bytes(n, images) (the filtered streams, their tokens and their worst-case deflate data; it does
 * not depend on out_bytes), 256-byte aligned.  Channels other than 1 or 3, swap_rb with one channel, h or w outside 1..65535, raw >= 2^31
 * or a stored zlib stream beyond the 2^31 - 1 bytes of one PNG chunk, a pitch below w c, NULL pointers or a short workspace:
 * MSC_ERR_BAD_ARGUMENT before anything is launched (the workspace size is then 0).  n = 0 is a successful no-op.
 */
typedef struct {
    const uint8_t* pixels;
    int64_t row_pitch;
    int32_t height, width, channels, swap_rb;
} msc_png_image;
size_t msc_png_encode_workspace_bytes(int32_t n, const msc_png_image* images_host);
int msc_png_encode_batch(int32_t n, const msc_png_image* images_host, uint8_t* out, size_t out_bytes, int64_t* out_off, int32_t* status,
                         void* workspace, size_t workspace_bytes, void* stream);

/*
 * The classifier mosaics of LiDARAgent._classify_batch_with_llm (lidar_agent.cluster_mosaic) for n groups of 512 x 512 BGR cluster views
 * already on the device, in one stream-ordered call.  groups: HOST i32 [n, 2] = (first, count), count in 1..10, first + count <= n_views;
 * mosaic j is cluster_mosaic(views[first_j .. first_j + count_j)): the view itself for a count of 1, else a sheet of min(3, count)
 * columns and ceil(count / 3) rows of views with the '#idx' labels and white empty cells.  The labels and the white come from
 * stamps u32 [*, 2] (pixel y * W + x, B | G << 8 | R << 16) of lidar_agent.mosaic_stamp, written over the copied views: the stamp of a
 * count k >= 2 is stamps[stamp_off[k] .. stamp_off[k + 1]) (stamp_off: HOST i32 [12]).  The mosaics are back to back in out_bgr, each
 * (512 rows) x (512 cols) x 3.  No host synchronisation, no allocation: workspace >= msc_cluster_mosaics_workspace_bytes(n),
 * 256-byte aligned; views and out_bgr 16-byte aligned.  A group out of range, NULL buffers, a misaligned buffer or a short workspace:
 * MSC_ERR_BAD_ARGUMENT.  n = 0 is a successful no-op.
 */
size_t msc_cluster_mosaics_workspace_bytes(int32_t n);
int msc_cluster_mosaics(const uint8_t* views, int32_t n_views, const int32_t* groups, int32_t n, const uint32_t* stamps, const int32_t* stamp_off,
                        uint8_t* out_bgr, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MSC_GEOM_H */
