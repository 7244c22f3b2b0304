/*
 * depth_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * (B) [EXT] row e7, LiDAR -> camera projection: the normative scalar definition of msc_camera_depth_batch
 * (csrc/camera_depth.cu).  It follows nuscenes-devkit NuScenesExplorer.map_pointcloud_to_image applied to the cloud of
 * LidarPointCloud.from_file_multisweep, with every floating-point operation spelled out in a fixed order so the kernels can match
 * it bit for bit.  This file includes oracle/c/msc_oracle.c for its f64 pose helpers (quat_to_rot, frame_change) and the box
 * projection (orc_project_boxes), and is built on its own with the same flags (-O2 -ffp-contract=off -fno-fast-math, no -march):
 * tests/depth_oracle.py compiles it.  Arithmetic rules as in msc_oracle.c: plain + - * / are single IEEE-754 round-to-nearest
 * operations, a fused multiply-add happens only where fma()/fmaf() is written, float -> int truncates.
 */
#include "../oracle/c/msc_oracle.c"

/* c <- R(q) c + t, R <- R(q) R for pose7 = (t, q): the devkit's rotate-then-translate of a sensor -> parent pose */
static void rigid_apply(const double pose[7], double c[3], double R[9]) {
    double Q[9], c2[3], R2[9];
    quat_to_rot(pose + 3, Q);
    for (int r = 0; r < 3; ++r) {
        c2[r] = ((Q[r * 3 + 0] * c[0] + Q[r * 3 + 1] * c[1]) + Q[r * 3 + 2] * c[2]) + pose[r];
        for (int k = 0; k < 3; ++k) R2[r * 3 + k] = (Q[r * 3 + 0] * R[0 * 3 + k] + Q[r * 3 + 1] * R[1 * 3 + k]) + Q[r * 3 + 2] * R[2 * 3 + k];
    }
    memcpy(c, c2, sizeof(c2));
    memcpy(R, R2, sizeof(R2));
}

/* ------------------------------------------------------------------------------------------ */
/* Projection matrix of one (sample, camera): P = K [R | t] with [R | t] = cam_from_ref, composed in f64 without FMA in this   */
/* order, starting from (t, R) = (t, R(q)) of lidar_calib (ref -> ego, c' = R c + t):                                            */
/*   ego -> global with ego_pose (c' = R c + t);                                                                                 */
/*   global -> camera ego with cam_ego_pose, camera ego -> camera with cam_calib (frame_change: c' = R^T (c - t), as project_box)*/
/* then P[r][k] = (K[r][0] R[0][k] + K[r][1] R[1][k]) + K[r][2] R[2][k] (t in column 3), rounded once to f32.  P12 row-major.    */
/* ------------------------------------------------------------------------------------------ */
void orc_camera_matrix(const double ego_pose[7], const double lidar_calib[7], const double cam_ego_pose[7], const double cam_calib[7],
                       const double K[9], float P12[12]) {
    double c[3] = {lidar_calib[0], lidar_calib[1], lidar_calib[2]};
    double R[9];
    quat_to_rot(lidar_calib + 3, R);
    rigid_apply(ego_pose, c, R);
    frame_change(cam_ego_pose, c, R);
    frame_change(cam_calib, c, R);
    for (int r = 0; r < 3; ++r) {
        for (int k = 0; k < 3; ++k) P12[r * 4 + k] = (float)((K[r * 3 + 0] * R[0 * 3 + k] + K[r * 3 + 1] * R[1 * 3 + k]) + K[r * 3 + 2] * R[2 * 3 + k]);
        P12[r * 4 + 3] = (float)((K[r * 3 + 0] * c[0] + K[r * 3 + 1] * c[1]) + K[r * 3 + 2] * c[2]);
    }
}

/* ------------------------------------------------------------------------------------------ */
/* Depth maps of ONE sample.                                                                                                    */
/*  1. Points: the multi-sweep cloud exactly as orc_aggregate_sweeps defines it -- remove_close (|x| < r and |y| < r) in the     */
/*     sweep's own frame, then (float)fma(m0,x,fma(m1,y,fma(m2,z,m3))) into the keyframe LIDAR_TOP frame ("ref").  No range or  */
/*     height gate (the devkit applies none here); intensity and ring are unused.                                               */
/*  2. Per camera P = orc_camera_matrix(...).                                                                                   */
/*  3. Per point and camera, f32: a = fmaf(P00,x,fmaf(P01,y,fmaf(P02,z,P03))), b and w likewise with rows 1 and 2.  The point    */
/*     lands in the camera iff w > min_dist, and with u = a / w, v = b / w (IEEE division): u > 1, u < W - 1, v > 1, v < H - 1 */
/*     (the devkit's map_pointcloud_to_image mask, all strict; W - 1 and H - 1 as f32).  For nuScenes intrinsics the third row  */
/*     of K is (0, 0, 1), so w is the camera-frame depth.  NaN rows fail every compare.  Pixel ((int)u, (int)v), block          */
/*     (px / ds, py / ds).  A point may land in several cameras.                                                                */
/*  4. depth [n_cams, ceil(H/ds), ceil(W/ds)] f32: minimum w over the points in each block, +inf where there are none           */
/*     (order-independent); cam_points [n_cams]: the number of points that land in each camera.                                 */
/*  pixel (may be NULL): [rows, n_cams] i32, per input row of the sweeps in order (sweep_count summed) py * W + px or -1.       */
/* ------------------------------------------------------------------------------------------ */
void orc_camera_depth_sample(float remove_close_radius, int image_w, int image_h, int n_cams, float min_dist, int ds,
                             const float* points, int n_sweeps, const uint32_t* sweep_start, const uint32_t* sweep_count,
                             const double* sweep_pose, const double* ego_pose, const double* lidar_calib,
                             const double* cam_ego_pose /* n_cams x 7 */, const double* cam_calib /* n_cams x 7 */,
                             const double* cam_K /* n_cams x 9 */, float* depth, uint32_t* cam_points, int32_t* pixel) {
    const int hb = (image_h + ds - 1) / ds, wb = (image_w + ds - 1) / ds;
    const float u_hi = (float)(image_w - 1), v_hi = (float)(image_h - 1);
    float P[ORC_MAX_CAMS][12];
    for (int c = 0; c < n_cams; ++c) {
        orc_camera_matrix(ego_pose, lidar_calib, cam_ego_pose + 7 * c, cam_calib + 7 * c, cam_K + 9 * c, P[c]);
        cam_points[c] = 0;
    }
    for (size_t i = 0; i < (size_t)n_cams * hb * wb; ++i) depth[i] = INFINITY;
    size_t row = 0;
    for (int s = 0; s < n_sweeps; ++s) {
        const double* M = sweep_pose + 12 * s;
        const float* pts = points + (size_t)sweep_start[s] * 5;
        for (uint32_t n = 0; n < sweep_count[s]; ++n, ++row) {
            if (pixel)
                for (int c = 0; c < n_cams; ++c) pixel[row * n_cams + c] = -1;
            float x = pts[5 * (size_t)n], y = pts[5 * (size_t)n + 1], z = pts[5 * (size_t)n + 2];
            if (fabsf(x) < remove_close_radius && fabsf(y) < remove_close_radius) continue;
            double xd = (double)x, yd = (double)y, zd = (double)z;
            float xr = (float)fma(M[0], xd, fma(M[1], yd, fma(M[2], zd, M[3])));
            float yr = (float)fma(M[4], xd, fma(M[5], yd, fma(M[6], zd, M[7])));
            float zr = (float)fma(M[8], xd, fma(M[9], yd, fma(M[10], zd, M[11])));
            for (int c = 0; c < n_cams; ++c) {
                const float* p = P[c];
                float a = fmaf(p[0], xr, fmaf(p[1], yr, fmaf(p[2], zr, p[3])));
                float b = fmaf(p[4], xr, fmaf(p[5], yr, fmaf(p[6], zr, p[7])));
                float w = fmaf(p[8], xr, fmaf(p[9], yr, fmaf(p[10], zr, p[11])));
                if (!(w > min_dist)) continue;
                float u = a / w, v = b / w;
                if (!(u > 1.0f && u < u_hi && v > 1.0f && v < v_hi)) continue;
                int px = (int)u, py = (int)v;
                float* d = depth + ((size_t)c * hb + (size_t)(py / ds)) * wb + (size_t)(px / ds);
                if (w < *d) *d = w;
                cam_points[c] += 1;
                if (pixel) pixel[row * n_cams + c] = py * image_w + px;
            }
        }
    }
}

/* ------------------------------------------------------------------------------------------ */
/* LiDAR support of each (box, camera) of ONE sample over that sample's depth maps (layout of orc_camera_depth_sample).         */
/* out [n_boxes, n_cams, 4] u32 = n_blocks, n_hit, n_front, n_on.                                                                */
/*  - visible and the clipped extent (umin, vmin, umax, vmax) are orc_project_boxes' (f64, devkit box_in_image ANY); zlo / zhi   */
/*    are the min / max camera-frame Z of the 8 corners with the same corner arithmetic.                                          */
/*  - a box that is not visible: all four counts 0.                                                                               */
/*  - otherwise the blocks bx in [(int)umin / ds, min((int)umax, W - 1) / ds], by in [(int)vmin / ds, min((int)vmax, H - 1) / ds]  */
/*    (umin.. are the f32 extent); n_blocks = their number; n_hit: blocks whose depth d is finite; n_front: hit blocks with       */
/*    (double)d < zlo - margin (something nearer hides the box); n_on: the other hit blocks with (double)d <= zhi + margin (the    */
/*    nearest return lies on the box).  zlo - margin and zhi + margin are f64 with margin widened from f32.                        */
/* ------------------------------------------------------------------------------------------ */
void orc_box_depth_support(int n_boxes, const double* boxes, int n_cams, const double* cam_ego_pose, const double* cam_calib,
                           const double* cam_K, int image_w, int image_h, int ds, float margin, const float* depth, uint32_t* out) {
    const int hb = (image_h + ds - 1) / ds, wb = (image_w + ds - 1) / ds;
    for (int b = 0; b < n_boxes; ++b) {
        const double* box = boxes + 10 * b;
        const double hl = box[4] / 2.0, hw = box[3] / 2.0, hh = box[5] / 2.0;
        for (int c = 0; c < n_cams; ++c) {
            uint8_t vis;
            float e[4];
            orc_project_boxes(1, box, 1, cam_ego_pose + 7 * c, cam_calib + 7 * c, cam_K + 9 * c, image_w, image_h, &vis, e);
            uint32_t* o = out + ((size_t)b * n_cams + c) * 4;
            o[0] = o[1] = o[2] = o[3] = 0;
            if (!vis) continue;
            double ctr[3] = {box[0], box[1], box[2]}, R[9];
            quat_to_rot(box + 6, R);
            frame_change(cam_ego_pose + 7 * c, ctr, R);
            frame_change(cam_calib + 7 * c, ctr, R);
            double zlo = INFINITY, zhi = -INFINITY;
            for (int k = 0; k < 8; ++k) {
                static const double sx[8] = {1, 1, 1, 1, -1, -1, -1, -1};
                static const double sy[8] = {1, -1, -1, 1, 1, -1, -1, 1};
                static const double sz[8] = {1, 1, -1, -1, 1, 1, -1, -1};
                double lx = sx[k] * hl, ly = sy[k] * hw, lz = sz[k] * hh;
                double Z = ((R[6] * lx + R[7] * ly) + R[8] * lz) + ctr[2];
                if (Z < zlo) zlo = Z;
                if (Z > zhi) zhi = Z;
            }
            int ux1 = (int)e[2], vy1 = (int)e[3];
            if (ux1 > image_w - 1) ux1 = image_w - 1;
            if (vy1 > image_h - 1) vy1 = image_h - 1;
            const int bx0 = (int)e[0] / ds, bx1 = ux1 / ds, by0 = (int)e[1] / ds, by1 = vy1 / ds;
            const double zf = zlo - (double)margin, zo = zhi + (double)margin;
            const float* img = depth + (size_t)c * hb * wb;
            o[0] = (uint32_t)((bx1 - bx0 + 1) * (by1 - by0 + 1));
            for (int by = by0; by <= by1; ++by)
                for (int bx = bx0; bx <= bx1; ++bx) {
                    float d = img[(size_t)by * wb + bx];
                    if (!(d < INFINITY)) continue;
                    o[1] += 1;
                    if ((double)d < zf) o[2] += 1;
                    else if ((double)d <= zo) o[3] += 1;
                }
        }
    }
}
