/*
 * msc_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Scalar, single-threaded CPU restatement of the geometric-evidence hot path of
 * AgustinRoca/multimodal-scene-captioning.  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may load this library.  The shipped
 * path (multimodal-scene-captioning_b200/) never links, imports or calls it.
 *
 * Two families of functions live here:
 *
 *  (A) restatements of code that EXISTS in the reference (pinned by golden vectors produced
 *      by importing the reference itself, tests/golden/make_golden.py):
 *        orc_keyframe_filter_split  <- src/agents/content_transform/lidar_agent.py:103-132
 *        orc_keyframe_bev_raster    <- src/agents/content_transform/lidar_agent.py:539-597
 *        orc_cloud_stats            <- src/baseline_gpt4o.py:270-287
 *        orc_annotation_table       <- src/agents/content_transform/scenegraph_agent.py:180-247,
 *                                      :281-295 (zones :136-146); src/baseline_gpt4o.py:304-317
 *        orc_cluster_aabb           <- src/agents/content_transform/lidar_agent.py:198-218
 *
 *  (B) [EXT] features that north_star names but the reference never implements (multi-sweep
 *      aggregation, oriented-box membership, 200x200 BEV with intensity, box->camera projection,
 *      pairwise relations, FOV wedges).  They follow nuscenes-devkit semantics (un-vendored,
 *      unpinned dependency, requirements.txt:4) as restated in SURVEY.md Appendix A.
 *      PARITY UNPINNED: no reference test, call site or golden vector constrains these; this file
 *      is their normative definition, with every floating-point operation spelled out in a fixed
 *      order so the CUDA kernels can match it bit for bit.
 *
 * Arithmetic rules (compile with -O2 -ffp-contract=off, no -ffast-math, no -march flags):
 *   - plain + - * / sqrt are single IEEE-754 round-to-nearest operations;
 *   - a fused multiply-add happens ONLY where fma()/fmaf() is written explicitly;
 *   - float->int is truncation unless lrintf() (round-half-even) is written.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_MAX_CAMS 8

typedef struct {
    float remove_close_radius; /* devkit remove_close(), App. A.1; default 1.0                   */
    float range_min;           /* lidar_agent.py:107  distances > 1.0                            */
    float range_max;           /* lidar_agent.py:107  distances < self.bev_range (50)            */
    float z_min;               /* lidar_agent.py:110  z > -3.0                                   */
    float z_max;               /* lidar_agent.py:110  z <  5.0                                   */
    float ground_z;            /* lidar_agent.py:115,128  z < -1.4 => ground                     */
    float bev_range;           /* lidar_agent.py:49   50 m                                       */
    int32_t bev_res;           /* 200 for the [EXT] grid, 800 for the reference grid             */
    int32_t image_w;           /* 1600 */
    int32_t image_h;           /* 900  */
    int32_t n_cams;            /* 6    */
    uint32_t fov_keep_mask;    /* 0 = count only; else keep points inside any selected wedge      */
    int32_t centroid_shift;    /* fixed-point fraction bits of centroid sums (<= 17: the biased coordinate is a 24-bit value)       */
    int32_t intensity_shift;   /* fixed-point fraction bits of intensity sums (8)                */
} orc_params;

/* ------------------------------------------------------------------------------------------ */
/* small f64 helpers (no FMA)                                                                 */
/* ------------------------------------------------------------------------------------------ */

/* unit quaternion (w,x,y,z) -> row-major 3x3 rotation; normalises first */
static void quat_to_rot(const double q[4], double R[9]) {
    double w = q[0], x = q[1], y = q[2], z = q[3];
    double n = sqrt(((w * w + x * x) + y * y) + z * z);
    w = w / n; x = x / n; y = y / n; z = z / n;
    double xx = x * x, yy = y * y, zz = z * z;
    double xy = x * y, xz = x * z, yz = y * z;
    double wx = w * x, wy = w * y, wz = w * z;
    R[0] = 1.0 - 2.0 * (yy + zz); R[1] = 2.0 * (xy - wz);       R[2] = 2.0 * (xz + wy);
    R[3] = 2.0 * (xy + wz);       R[4] = 1.0 - 2.0 * (xx + zz); R[5] = 2.0 * (yz - wx);
    R[6] = 2.0 * (xz - wy);       R[7] = 2.0 * (yz + wx);       R[8] = 1.0 - 2.0 * (xx + yy);
}

/* out = A^T * v  (A row-major 3x3) */
static void rot_t_vec(const double A[9], const double v[3], double out[3]) {
    out[0] = (A[0] * v[0] + A[3] * v[1]) + A[6] * v[2];
    out[1] = (A[1] * v[0] + A[4] * v[1]) + A[7] * v[2];
    out[2] = (A[2] * v[0] + A[5] * v[1]) + A[8] * v[2];
}

/* out = A^T * B */
static void rot_t_mat(const double A[9], const double B[9], double out[9]) {
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c)
            out[r * 3 + c] = (A[0 * 3 + r] * B[0 * 3 + c] + A[1 * 3 + r] * B[1 * 3 + c]) + A[2 * 3 + r] * B[2 * 3 + c];
}

/* devkit Box.translate(-t); Box.rotate(q^-1)  (SURVEY App. A.3): c' = R(q)^T (c - t), R' = R(q)^T R */
static void frame_change(const double pose[7], double c[3], double R[9]) {
    double Rp[9], d[3], c2[3], R2[9];
    quat_to_rot(pose + 3, Rp);
    d[0] = c[0] - pose[0]; d[1] = c[1] - pose[1]; d[2] = c[2] - pose[2];
    rot_t_vec(Rp, d, c2);
    rot_t_mat(Rp, R, R2);
    memcpy(c, c2, sizeof(c2));
    memcpy(R, R2, sizeof(R2));
}

/* ------------------------------------------------------------------------------------------ */
/* (B) [EXT]  box preparation: global box -> reference-sensor frame -> devkit points_in_box     */
/*     vectors (SURVEY App. A.2).  box = center3, size(w,l,h), quat(w,x,y,z), all f64 global.   */
/*     out16 (f32): p1[3], i[3], j[3], k[3], ii, jj, kk, pad                                    */
/* ------------------------------------------------------------------------------------------ */
void orc_box_prepare(const double box[10], const double ego_pose[7], const double lidar_calib[7],
                     float out16[16], float corners_xy[16]) {
    double c[3] = {box[0], box[1], box[2]};
    double R[9];
    quat_to_rot(box + 6, R);
    frame_change(ego_pose, c, R);    /* global -> ego   */
    frame_change(lidar_calib, c, R); /* ego -> sensor   */
    double w = box[3], l = box[4], h = box[5];
    double hl = l / 2.0, hw = w / 2.0, hh = h / 2.0;
    /* corner0 = c + R * (+l/2, +w/2, +h/2) */
    double p1[3];
    for (int r = 0; r < 3; ++r) p1[r] = ((R[r * 3 + 0] * hl + R[r * 3 + 1] * hw) + R[r * 3 + 2] * hh) + c[r];
    float *P1 = out16, *I = out16 + 3, *J = out16 + 6, *K = out16 + 9;
    for (int r = 0; r < 3; ++r) {
        P1[r] = (float)p1[r];
        I[r] = (float)(-(l * R[r * 3 + 0])); /* corner4 - corner0 */
        J[r] = (float)(-(w * R[r * 3 + 1])); /* corner1 - corner0 */
        K[r] = (float)(-(h * R[r * 3 + 2])); /* corner3 - corner0 */
    }
    out16[12] = fmaf(I[2], I[2], fmaf(I[1], I[1], I[0] * I[0]));
    out16[13] = fmaf(J[2], J[2], fmaf(J[1], J[1], J[0] * J[0]));
    out16[14] = fmaf(K[2], K[2], fmaf(K[1], K[1], K[0] * K[0]));
    out16[15] = 0.0f;
    if (corners_xy) { /* xy of the 8 corners (f32), used only by tests of the GPU cull grid */
        static const double sx[8] = {1, 1, 1, 1, -1, -1, -1, -1};
        static const double sy[8] = {1, -1, -1, 1, 1, -1, -1, 1};
        static const double sz[8] = {1, 1, -1, -1, 1, 1, -1, -1};
        for (int k = 0; k < 8; ++k) {
            double lx = sx[k] * hl, ly = sy[k] * hw, lz = sz[k] * hh;
            corners_xy[2 * k + 0] = (float)(((R[0] * lx + R[1] * ly) + R[2] * lz) + c[0]);
            corners_xy[2 * k + 1] = (float)(((R[3] * lx + R[4] * ly) + R[5] * lz) + c[1]);
        }
    }
}

/* ------------------------------------------------------------------------------------------ */
/* (B) [EXT] camera wedges for the FOV filter.  For camera c the horizontal field of view is the  */
/*     wedge, in the reference sensor's xy-plane, between the rays through image columns u=0 and  */
/*     u=W at the principal row, with its apex at the camera centre.  wedge6 (f32): ox, oy,       */
/*     e_left(x,y), e_right(x,y).  A point q=(x-ox, y-oy) is inside iff                           */
/*        cross(e_right, q) >= 0  and  cross(q, e_left) >= 0   (cross(a,b) = fmaf(ax,by,-(ay*bx)))*/
/*     ego pose of the lidar keyframe is used for both sensors (rig geometry only).               */
/* ------------------------------------------------------------------------------------------ */
void orc_cam_wedge(const double lidar_calib[7], const double cam_calib[7], const double K[9], int image_w,
                   float wedge6[6]) {
    double Rl[9], Rc[9];
    quat_to_rot(lidar_calib + 3, Rl);
    quat_to_rot(cam_calib + 3, Rc);
    /* camera centre in the lidar frame: Rl^T (tc - tl) */
    double d[3] = {cam_calib[0] - lidar_calib[0], cam_calib[1] - lidar_calib[1], cam_calib[2] - lidar_calib[2]};
    double o[3];
    rot_t_vec(Rl, d, o);
    /* ray directions in the camera frame: ((u - cx)/fx, 0, 1) for u = 0 and u = W */
    double fx = K[0], cx = K[2];
    double dl_cam[3] = {(0.0 - cx) / fx, 0.0, 1.0};
    double dr_cam[3] = {((double)image_w - cx) / fx, 0.0, 1.0};
    double dl_ego[3], dr_ego[3], dl[3], dr[3];
    for (int r = 0; r < 3; ++r) {
        dl_ego[r] = (Rc[r * 3 + 0] * dl_cam[0] + Rc[r * 3 + 1] * dl_cam[1]) + Rc[r * 3 + 2] * dl_cam[2];
        dr_ego[r] = (Rc[r * 3 + 0] * dr_cam[0] + Rc[r * 3 + 1] * dr_cam[1]) + Rc[r * 3 + 2] * dr_cam[2];
    }
    rot_t_vec(Rl, dl_ego, dl);
    rot_t_vec(Rl, dr_ego, dr);
    wedge6[0] = (float)o[0]; wedge6[1] = (float)o[1];
    /* image column u=0 is the LEFT image edge; with x-right camera axes it is the counter-clockwise edge */
    wedge6[2] = (float)dl[0]; wedge6[3] = (float)dl[1];
    wedge6[4] = (float)dr[0]; wedge6[5] = (float)dr[1];
}

static inline int in_wedge(const float w[6], float x, float y) {
    float qx = x - w[0], qy = y - w[1];
    float c_r = fmaf(w[4], qy, -(w[5] * qx)); /* cross(e_right, q) */
    float c_l = fmaf(-w[2], qy, w[3] * qx);   /* cross(q, e_left): same shape as c_r -- product on the x term, fma on the y term */
    return (c_r >= 0.0f) && (c_l >= 0.0f);
}

/* BEV cell index, lidar_agent.py:547-552: clip(trunc((c + r) / (2 r) * res), 0, res-1), float32 */
static inline int bev_index(float c, float r, float two_r, float resf, int res) {
    float t = ((c + r) / two_r) * resf;
    int i = (int)t; /* trunc toward zero, like ndarray.astype(int) */
    if (i < 0) i = 0;
    if (i > res - 1) i = res - 1;
    return i;
}

/* ------------------------------------------------------------------------------------------ */
/* (B) [EXT] the fused evidence pass for ONE sample.                                            */
/*   points    : concatenated raw sweeps, n x 5 f32 (x,y,z,intensity,ring) as in .pcd.bin       */
/*   sweep_start/sweep_count (points), sweep_pose (3x4 f64 row-major ref_from_sensor_s)         */
/*   boxes     : n_boxes x 10 f64 global (center, wlh, quat wxyz)                               */
/*   outputs   : see DESIGN.md "result tables"                                                  */
/* ------------------------------------------------------------------------------------------ */
void orc_fused_evidence_sample(const orc_params* P, const float* points, int n_sweeps, const uint32_t* sweep_start,
                               const uint32_t* sweep_count, const double* sweep_pose, int n_boxes,
                               const double* boxes, const double* ego_pose, const double* lidar_calib,
                               const double* cam_calib /* n_cams x 7 */, const double* cam_K /* n_cams x 9 */,
                               uint32_t* box_count, float* box_nearest, float* box_centroid,
                               uint32_t* bev_count, float* bev_height, uint32_t* bev_isum_q, uint32_t* stats16) {
    const int res = P->bev_res;
    const float r = P->bev_range, two_r = 2.0f * P->bev_range, resf = (float)res;
    const size_t ncell = (size_t)res * (size_t)res;
    float* bp = (float*)malloc(sizeof(float) * 16 * (size_t)(n_boxes > 0 ? n_boxes : 1));
    int64_t* csum = (int64_t*)calloc((size_t)(n_boxes > 0 ? n_boxes : 1) * 3, sizeof(int64_t));
    float* smin = (float*)malloc(sizeof(float) * (size_t)(n_boxes > 0 ? n_boxes : 1));
    uint64_t* isum = (uint64_t*)calloc(ncell, sizeof(uint64_t));
    float wedges[ORC_MAX_CAMS][6];
    for (int b = 0; b < n_boxes; ++b) {
        orc_box_prepare(boxes + 10 * b, ego_pose, lidar_calib, bp + 16 * b, NULL);
        box_count[b] = 0;
        smin[b] = INFINITY;
    }
    for (int c = 0; c < P->n_cams; ++c) orc_cam_wedge(lidar_calib, cam_calib + 7 * c, cam_K + 9 * c, P->image_w, wedges[c]);
    memset(bev_count, 0, ncell * sizeof(uint32_t));
    for (size_t i = 0; i < ncell; ++i) bev_height[i] = 0.0f; /* lidar_agent.py:543 zero-initialised */
    memset(stats16, 0, 16 * sizeof(uint32_t));
    const float cscale = (float)(1 << P->centroid_shift);
    const float iscale = (float)(1 << P->intensity_shift);

    for (int s = 0; s < n_sweeps; ++s) {
        const double* M = sweep_pose + 12 * s;
        const float* pts = points + (size_t)sweep_start[s] * 5;
        for (uint32_t n = 0; n < sweep_count[s]; ++n) {
            float x = pts[5 * (size_t)n + 0], y = pts[5 * (size_t)n + 1], z = pts[5 * (size_t)n + 2];
            float inten = pts[5 * (size_t)n + 3];
            stats16[0] += 1;
            /* A.1 remove_close: |x| < r and |y| < r in the sweep's own sensor frame */
            if (fabsf(x) < P->remove_close_radius && fabsf(y) < P->remove_close_radius) continue;
            stats16[1] += 1;
            /* A.1 transform: f64 matrix times f32 point, stored back as f32 */
            double xd = (double)x, yd = (double)y, zd = (double)z;
            float xr = (float)fma(M[0], xd, fma(M[1], yd, fma(M[2], zd, M[3])));
            float yr = (float)fma(M[4], xd, fma(M[5], yd, fma(M[6], zd, M[7])));
            float zr = (float)fma(M[8], xd, fma(M[9], yd, fma(M[10], zd, M[11])));
            /* lidar_agent.py:106-110 range / height filter, float32, separate roundings, strict */
            float s2 = xr * xr + yr * yr;
            float dist = sqrtf(s2);
            if (!(dist > P->range_min && dist < P->range_max && zr < P->z_max && zr > P->z_min)) continue;
            /* FOV wedges: counted on range-kept points; optional filter */
            uint32_t cam_bits = 0;
            for (int c = 0; c < P->n_cams; ++c)
                if (in_wedge(wedges[c], xr, yr)) { cam_bits |= 1u << c; stats16[5 + c] += 1; }
            if (P->fov_keep_mask && !(cam_bits & P->fov_keep_mask)) continue;
            stats16[2] += 1;
            /* lidar_agent.py:128 ground split */
            if (zr < P->ground_z) stats16[3] += 1; else stats16[4] += 1;
            /* BEV layers, lidar_agent.py:547-560 with res/range from params; [y, x] indexing */
            int ix = bev_index(xr, r, two_r, resf, res), iy = bev_index(yr, r, two_r, resf, res);
            size_t cell = (size_t)iy * (size_t)res + (size_t)ix;
            bev_count[cell] += 1;
            if (zr > bev_height[cell]) bev_height[cell] = zr;
            {   /* Q<intensity_shift> fixed point, clamped to [0, 65535]; NaN -> 0 */
                float qf = inten * iscale;
                if (!(qf >= 0.0f)) qf = 0.0f;
                if (qf > 65535.0f) qf = 65535.0f;
                isum[cell] += (uint64_t)lrintf(qf);
            }
            /* A.2 points_in_box, float32 with fmaf chains, closed intervals */
            for (int b = 0; b < n_boxes; ++b) {
                const float* B = bp + 16 * b;
                float v0 = xr - B[0], v1 = yr - B[1], v2 = zr - B[2];
                float iv = fmaf(B[5], v2, fmaf(B[4], v1, B[3] * v0));
                float jv = fmaf(B[8], v2, fmaf(B[7], v1, B[6] * v0));
                float kv = fmaf(B[11], v2, fmaf(B[10], v1, B[9] * v0));
                if (iv >= 0.0f && iv <= B[12] && jv >= 0.0f && jv <= B[13] && kv >= 0.0f && kv <= B[14]) {
                    box_count[b] += 1;
                    if (s2 < smin[b]) smin[b] = s2;
                    csum[3 * b + 0] += (int64_t)lrintf(xr * cscale);
                    csum[3 * b + 1] += (int64_t)lrintf(yr * cscale);
                    csum[3 * b + 2] += (int64_t)lrintf(zr * cscale);
                }
            }
        }
    }
    for (int b = 0; b < n_boxes; ++b) {
        if (box_count[b] == 0) {
            box_nearest[b] = INFINITY;
            box_centroid[3 * b + 0] = box_centroid[3 * b + 1] = box_centroid[3 * b + 2] = 0.0f;
        } else {
            box_nearest[b] = sqrtf(smin[b]);
            double den = (double)box_count[b] * (double)cscale;
            for (int k = 0; k < 3; ++k) box_centroid[3 * b + k] = (float)((double)csum[3 * b + k] / den);
        }
    }
    for (size_t i = 0; i < ncell; ++i) bev_isum_q[i] = (uint32_t)isum[i]; /* device accumulators are u32 (mod 2^32) */
    (void)iscale;
    free(bp); free(csum); free(smin); free(isum);
}

/* ------------------------------------------------------------------------------------------ */
/* (B) [EXT] materialised multi-sweep aggregation (devkit from_file_multisweep, App. A.1):       */
/*     out rows: x', y', z', intensity ; out_time: time lag per point.  Returns rows written.    */
/* ------------------------------------------------------------------------------------------ */
uint32_t orc_aggregate_sweeps(float remove_close_radius, const float* points, int n_sweeps, const uint32_t* sweep_start,
                              const uint32_t* sweep_count, const double* sweep_pose, const float* sweep_time_lag,
                              float* out_xyzi, float* out_time) {
    uint32_t m = 0;
    for (int s = 0; s < n_sweeps; ++s) {
        const double* M = sweep_pose + 12 * s;
        const float* pts = points + (size_t)sweep_start[s] * 5;
        for (uint32_t n = 0; n < sweep_count[s]; ++n) {
            float x = pts[5 * (size_t)n], y = pts[5 * (size_t)n + 1], z = pts[5 * (size_t)n + 2];
            if (fabsf(x) < remove_close_radius && fabsf(y) < remove_close_radius) continue;
            double xd = (double)x, yd = (double)y, zd = (double)z;
            out_xyzi[4 * (size_t)m + 0] = (float)fma(M[0], xd, fma(M[1], yd, fma(M[2], zd, M[3])));
            out_xyzi[4 * (size_t)m + 1] = (float)fma(M[4], xd, fma(M[5], yd, fma(M[6], zd, M[7])));
            out_xyzi[4 * (size_t)m + 2] = (float)fma(M[8], xd, fma(M[9], yd, fma(M[10], zd, M[11])));
            out_xyzi[4 * (size_t)m + 3] = pts[5 * (size_t)n + 3];
            out_time[m] = sweep_time_lag[s];
            ++m;
        }
    }
    return m;
}

/* ------------------------------------------------------------------------------------------ */
/* (B) [EXT] box -> camera projection (devkit get_sample_data + view_points + box_in_image,      */
/*     BoxVisibility.ANY; App. A.3).  All f64, no FMA.  extent is clipped to the image.          */
/* ------------------------------------------------------------------------------------------ */
void orc_project_boxes(int n_boxes, const double* boxes, int n_cams, const double* cam_ego_pose /* n_cams x 7 */,
                       const double* cam_calib /* n_cams x 7 */, const double* cam_K /* n_cams x 9 */, int image_w,
                       int image_h, uint8_t* visible /* n_boxes x n_cams */, float* extent /* n_boxes x n_cams x 4 */) {
    static const double sx[8] = {1, 1, 1, 1, -1, -1, -1, -1};
    static const double sy[8] = {1, -1, -1, 1, 1, -1, -1, 1};
    static const double sz[8] = {1, 1, -1, -1, 1, 1, -1, -1};
    const double W = (double)image_w, H = (double)image_h;
    for (int b = 0; b < n_boxes; ++b) {
        const double* box = boxes + 10 * b;
        double hl = box[4] / 2.0, hw = box[3] / 2.0, hh = box[5] / 2.0;
        for (int c = 0; c < n_cams; ++c) {
            double ctr[3] = {box[0], box[1], box[2]};
            double R[9];
            quat_to_rot(box + 6, R);
            frame_change(cam_ego_pose + 7 * c, ctr, R);
            frame_change(cam_calib + 7 * c, ctr, R);
            const double* K = cam_K + 9 * c;
            int any_vis = 0, all_front = 1;
            double umin = INFINITY, vmin = INFINITY, umax = -INFINITY, vmax = -INFINITY;
            for (int k = 0; k < 8; ++k) {
                double lx = sx[k] * hl, ly = sy[k] * hw, lz = sz[k] * hh;
                double X = ((R[0] * lx + R[1] * ly) + R[2] * lz) + ctr[0];
                double Y = ((R[3] * lx + R[4] * ly) + R[5] * lz) + ctr[1];
                double Z = ((R[6] * lx + R[7] * ly) + R[8] * lz) + ctr[2];
                double pu = (K[0] * X + K[1] * Y) + K[2] * Z;
                double pv = (K[3] * X + K[4] * Y) + K[5] * Z;
                double pw = (K[6] * X + K[7] * Y) + K[8] * Z;
                double u = pu / pw, v = pv / pw;
                int vis = (u > 0.0) && (u < W) && (v > 0.0) && (v < H) && (Z > 1.0);
                if (vis) any_vis = 1;
                if (!(Z > 0.1)) all_front = 0;
                if (u < umin) umin = u;
                if (u > umax) umax = u;
                if (v < vmin) vmin = v;
                if (v > vmax) vmax = v;
            }
            int ok = any_vis && all_front;
            visible[b * n_cams + c] = (uint8_t)ok;
            float* e = extent + ((size_t)b * n_cams + c) * 4;
            if (ok) {
                if (umin < 0.0) umin = 0.0;
                if (vmin < 0.0) vmin = 0.0;
                if (umax > W) umax = W;
                if (vmax > H) vmax = H;
                e[0] = (float)umin; e[1] = (float)vmin; e[2] = (float)umax; e[3] = (float)vmax;
            } else {
                e[0] = e[1] = e[2] = e[3] = 0.0f;
            }
        }
    }
}

/* 4-way bearing category with the bins of scenegraph_agent.py:190-201, written as exact predicates on
 * (dx, dy): 0=front [45,135)  1=left [135,225)  2=back [225,315)  3=right otherwise (incl. NaN, (+0,+-0));
 * (-0,+-0) is left, because atan2(+-0, -0) = +-pi.
 * Equivalent to the reference's atan2 formula wherever that formula is exact (verified on the diagonals
 * and axes by tests/test_oracle_golden.py against the reference itself). */
static inline uint8_t bearing4(double dx, double dy) {
    if (dx == 0.0 && dy == 0.0) return signbit(dx) ? 1 : 3; /* atan2(+-0, -0) = +-pi: left; atan2(+-0, +0) = +-0: right */
    if (dy > 0.0 && dx <= dy && -dx < dy) return 0;
    if (dx < 0.0 && dy <= -dx && dy > dx) return 1;
    if (dy < 0.0 && dx >= dy && dx < -dy) return 2;
    return 3;
}

/* ------------------------------------------------------------------------------------------ */
/* (A) per-annotation table.  Follows scenegraph_agent.py:186-201 (distance, direction),         */
/*     :209-225 (state; NaN speed compares false => stopped), :281-295 zones (first match),      */
/*     baseline_gpt4o.py:304-317 region flags.  xy/vel are the annotation's translation[:2] and  */
/*     velocity[:2] exactly as the loader hands them over (global frame -- the reference's frame  */
/*     bug, SURVEY.md section 0.3, is preserved).                                                */
/*     zone codes: 0 front_close 1 front_medium 2 front_far 3 left_close 4 left_medium           */
/*                 5 right_close 6 right_medium 7 back_close 8 back_medium, 255 = none           */
/* ------------------------------------------------------------------------------------------ */
void orc_annotation_table(int n, const double* xy, const double* vel, double* distance, uint8_t* direction,
                          uint8_t* moving, uint8_t* zone, uint8_t* region_bits) {
    static const double zmin[9] = {0, 10, 30, 0, 10, 0, 10, 0, 10};
    static const double zmax[9] = {10, 30, 50, 10, 30, 10, 30, 10, 30};
    static const uint8_t zdir[9] = {0, 0, 0, 1, 1, 3, 3, 2, 2};
    /* The reference squares with Python's `**` (scenegraph_agent.py:189, :216), i.e. libm pow(), which is within 1 ulp
     * of -- but not always equal to -- the correctly rounded product (1326.916**2 != 1326.916*1326.916).  The oracle
     * follows the reference literally; `two` is volatile so the compiler cannot rewrite pow(x, 2.0) as x*x. */
    volatile double two = 2.0;
    for (int i = 0; i < n; ++i) {
        double x = xy[2 * i], y = xy[2 * i + 1];
        double d = sqrt(pow(x, two) + pow(y, two));
        distance[i] = d;
        uint8_t dir = bearing4(x, y);
        direction[i] = dir;
        double vx = vel[2 * i], vy = vel[2 * i + 1];
        double sp = sqrt(pow(vx, two) + pow(vy, two));
        moving[i] = (uint8_t)(sp > 0.5);
        uint8_t zc = 255;
        for (int k = 0; k < 9; ++k)
            if (dir == zdir[k] && zmin[k] <= d && d < zmax[k]) { zc = (uint8_t)k; break; }
        zone[i] = zc;
        region_bits[i] = (uint8_t)((x > 0.0 ? 1 : 0) | (y > 0.0 ? 2 : 0));
    }
}

/* ------------------------------------------------------------------------------------------ */
/* (B) [EXT] pairwise relation table.  rect: n x 6 f64 = (x, y, ux, uy, half_len, half_wid) with */
/*     (ux,uy) the unit heading in the same frame as (x,y).  For every ordered pair (i, j):      */
/*     distance f32, bearing of j seen from i in degrees [0,360) f32, category u8 (bearing4),    */
/*     overlap u8 (separating-axis test of the two oriented rectangles, closed).  Diagonal: 0,0,3,1 */
/* ------------------------------------------------------------------------------------------ */
void orc_relation_table(int n, const double* rect, float* dist, float* bearing, uint8_t* category, uint8_t* overlap) {
    const double RAD2DEG_NUM = 180.0, PI = 3.14159265358979323846;
    for (int i = 0; i < n; ++i) {
        const double* A = rect + 6 * i;
        for (int j = 0; j < n; ++j) {
            const double* B = rect + 6 * j;
            size_t o = (size_t)i * n + j;
            double dx = B[0] - A[0], dy = B[1] - A[1];
            dist[o] = (float)sqrt(dx * dx + dy * dy);
            double ang = atan2(dy, dx) * RAD2DEG_NUM / PI; /* scenegraph_agent.py:190 */
            ang = fmod(ang + 360.0, 360.0);                 /* :191 */
            bearing[o] = (float)ang;
            category[o] = bearing4(dx, dy);
            /* SAT over the 4 edge normals */
            double ax[4][2] = {{A[2], A[3]}, {-A[3], A[2]}, {B[2], B[3]}, {-B[3], B[2]}};
            int sep = 0;
            for (int k = 0; k < 4; ++k) {
                double ex = ax[k][0], ey = ax[k][1];
                double t = fabs(dx * ex + dy * ey);
                double ra = A[4] * fabs(A[2] * ex + A[3] * ey) + A[5] * fabs(-A[3] * ex + A[2] * ey);
                double rb = B[4] * fabs(B[2] * ex + B[3] * ey) + B[5] * fabs(-B[3] * ex + B[2] * ey);
                if (t > ra + rb) sep = 1;
            }
            overlap[o] = (uint8_t)(!sep);
        }
    }
}

/* (B) [EXT] footprint rectangles for the relation table from global boxes: position and heading in the
 * ego frame of `ego_pose` (pass NULL to stay in the loader's global frame).  heading = normalised xy
 * projection of the box x-axis; half extents l/2, w/2. */
void orc_box_footprints(int n, const double* boxes, const double* ego_pose, double* rect) {
    for (int b = 0; b < n; ++b) {
        const double* box = boxes + 10 * b;
        double c[3] = {box[0], box[1], box[2]};
        double R[9];
        quat_to_rot(box + 6, R);
        if (ego_pose) frame_change(ego_pose, c, R);
        double ux = R[0], uy = R[3];
        double nn = sqrt(ux * ux + uy * uy);
        if (nn > 0.0) { ux = ux / nn; uy = uy / nn; } else { ux = 1.0; uy = 0.0; }
        double* o = rect + 6 * b;
        o[0] = c[0]; o[1] = c[1]; o[2] = ux; o[3] = uy; o[4] = box[4] / 2.0; o[5] = box[3] / 2.0;
    }
}

/* ------------------------------------------------------------------------------------------ */
/* (A) keyframe filter + ground split, lidar_agent.py:103-132.  pts: n rows with `pitch` floats   */
/*     between rows (4 for the mock loader, 5 for the devkit view, nuscenes_loader.py:152-155).   */
/*     Writes order-preserving index lists; returns counts through n_ground / n_object.          */
/* ------------------------------------------------------------------------------------------ */
void orc_keyframe_filter_split(const float* pts, uint32_t n, int pitch, float range_min, float range_max, float z_min,
                               float z_max, float ground_z, uint32_t* kept_idx, uint32_t* n_kept, uint32_t* ground_idx,
                               uint32_t* n_ground, uint32_t* object_idx, uint32_t* n_object) {
    uint32_t k = 0, g = 0, o = 0;
    for (uint32_t i = 0; i < n; ++i) {
        const float* p = pts + (size_t)i * pitch;
        float d = sqrtf(p[0] * p[0] + p[1] * p[1]);                        /* :106 */
        int ok = (d > range_min) && (d < range_max) && (p[2] < z_max) && (p[2] > z_min); /* :107-110 */
        if (!ok) continue;
        kept_idx[k++] = i;
        if (p[2] < ground_z) ground_idx[g++] = i; else object_idx[o++] = i; /* :128-130 */
    }
    *n_kept = k; *n_ground = g; *n_object = o;
}

/* ------------------------------------------------------------------------------------------ */
/* (A) BEV raster layers before the cv2 overlays, lidar_agent.py:539-597.                         */
/*     count u32 [res*res], height f32 (0-initialised running max, :543,:560), semantic BGR u8     */
/*     with ground colour then object hot-colormap, last point in array order wins (:567-597).    */
/*     Arrays are NOT flipped (the flip at :612-614 and everything after stays on the host).      */
/* ------------------------------------------------------------------------------------------ */
void orc_keyframe_bev_raster(const float* pts, int pitch, const uint32_t* ground_idx, uint32_t n_ground,
                             const uint32_t* object_idx, uint32_t n_object, float bev_range, int res, uint32_t* count,
                             float* height, uint8_t* semantic_bgr) {
    const float r = bev_range, two_r = 2.0f * bev_range, resf = (float)res;
    const size_t ncell = (size_t)res * res;
    memset(count, 0, ncell * sizeof(uint32_t));
    for (size_t i = 0; i < ncell; ++i) height[i] = 0.0f;
    memset(semantic_bgr, 0, ncell * 3);
    for (int pass = 0; pass < 2; ++pass) { /* np.vstack([ground, object]) order, :555 */
        const uint32_t* idx = pass ? object_idx : ground_idx;
        uint32_t m = pass ? n_object : n_ground;
        for (uint32_t t = 0; t < m; ++t) {
            const float* p = pts + (size_t)idx[t] * pitch;
            size_t cell = (size_t)bev_index(p[1], r, two_r, resf, res) * res + bev_index(p[0], r, two_r, resf, res);
            count[cell] += 1;
            if (p[2] > height[cell]) height[cell] = p[2];
        }
    }
    for (uint32_t t = 0; t < n_ground; ++t) { /* :570-572 */
        const float* p = pts + (size_t)ground_idx[t] * pitch;
        size_t cell = (size_t)bev_index(p[1], r, two_r, resf, res) * res + bev_index(p[0], r, two_r, resf, res);
        semantic_bgr[3 * cell + 0] = 80; semantic_bgr[3 * cell + 1] = 80; semantic_bgr[3 * cell + 2] = 120;
    }
    if (n_object == 0) return;
    float hmin = INFINITY, hmax = -INFINITY; /* :579-582 */
    for (uint32_t t = 0; t < n_object; ++t) {
        float z = pts[(size_t)object_idx[t] * pitch + 2];
        if (z < hmin) hmin = z;
        if (z > hmax) hmax = z;
    }
    int degenerate = !(hmax > hmin);
    float span = hmax - hmin;
    for (uint32_t t = 0; t < n_object; ++t) { /* :584-597 */
        const float* p = pts + (size_t)object_idx[t] * pitch;
        int g;
        if (degenerate) {
            g = 255; /* norm = 0.5 (float64): int(255 * (1 - (0.5 - 0.5) * 2)) */
        } else {
            float hn = (p[2] - hmin) / span;
            if (hn < 0.5f) g = (int)(255.0f * (1.0f - hn * 2.0f));
            else g = (int)(255.0f * (1.0f - (hn - 0.5f) * 2.0f));
        }
        size_t cell = (size_t)bev_index(p[1], r, two_r, resf, res) * res + bev_index(p[0], r, two_r, resf, res);
        semantic_bgr[3 * cell + 0] = 0; semantic_bgr[3 * cell + 1] = (uint8_t)g; semantic_bgr[3 * cell + 2] = 255;
    }
}

/* (A) raw-cloud statistics, baseline_gpt4o.py:276-285: min/max per axis (exact) and the sum of
 * sqrt(x^2+y^2) accumulated in f64 (numpy's float32 pairwise mean is matched to 1e-5 relative). */
void orc_cloud_stats(const float* pts, uint32_t n, int pitch, float* minmax6, double* radial_sum) {
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    double acc = 0.0;
    for (uint32_t i = 0; i < n; ++i) {
        const float* p = pts + (size_t)i * pitch;
        for (int k = 0; k < 3; ++k) { if (p[k] < mn[k]) mn[k] = p[k]; if (p[k] > mx[k]) mx[k] = p[k]; }
        acc += (double)sqrtf(p[0] * p[0] + p[1] * p[1]);
    }
    for (int k = 0; k < 3; ++k) { minmax6[k] = mn[k]; minmax6[3 + k] = mx[k]; }
    *radial_sum = acc;
}

/* (A) per-cluster axis-aligned metadata, lidar_agent.py:200-204, float32: min, max, dimensions=max-min,
 * center=(min+max)/2, distance=sqrt(cx^2+cy^2).  labels[i] in [0,n_clusters) or -1.  out: n_clusters x 11
 * (min3, max3, center3, distance, num_points). */
void orc_cluster_aabb(const float* pts, uint32_t n, int pitch, const int32_t* labels, int n_clusters, float* out11) {
    for (int c = 0; c < n_clusters; ++c) {
        float* o = out11 + 11 * c;
        o[0] = o[1] = o[2] = INFINITY; o[3] = o[4] = o[5] = -INFINITY; o[10] = 0.0f;
    }
    for (uint32_t i = 0; i < n; ++i) {
        int c = labels[i];
        if (c < 0 || c >= n_clusters) continue;
        const float* p = pts + (size_t)i * pitch;
        float* o = out11 + 11 * c;
        for (int k = 0; k < 3; ++k) { if (p[k] < o[k]) o[k] = p[k]; if (p[k] > o[3 + k]) o[3 + k] = p[k]; }
        o[10] += 1.0f;
    }
    for (int c = 0; c < n_clusters; ++c) {
        float* o = out11 + 11 * c;
        for (int k = 0; k < 3; ++k) o[6 + k] = (o[k] + o[3 + k]) / 2.0f;
        o[9] = sqrtf(o[6] * o[6] + o[7] * o[7]);
    }
}

int orc_abi_version(void) { return 1; }
