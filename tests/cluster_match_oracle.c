/*
 * cluster_match_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * (B) [EXT] LiDAR clusters -> annotated boxes: the normative scalar definition of msc_cluster_match_batch (csrc/cluster_match.cu).
 * This file includes oracle/c/msc_oracle.c for the box preparation (orc_box_prepare: global -> ego -> sensor in f64, the devkit
 * points_in_box vectors in f32) and uses the same f32 fmaf-chain membership test as orc_fused_evidence_sample (App. A.2).  It is built
 * on its own with the same flags (-O2 -ffp-contract=off -fno-fast-math, no -march): tests/cluster_match_oracle.py compiles it.
 */
#include "../oracle/c/msc_oracle.c"

/* A.2 points_in_box of one row against one prepared box B (orc_box_prepare layout), float32 with fmaf chains, closed intervals; NaN rows
 * fail every compare */
static int orc_in_box(const float* B, float x, float y, float z) {
    float v0 = x - B[0], v1 = y - B[1], v2 = z - B[2];
    float iv = fmaf(B[5], v2, fmaf(B[4], v1, B[3] * v0));
    float jv = fmaf(B[8], v2, fmaf(B[7], v1, B[6] * v0));
    float kv = fmaf(B[11], v2, fmaf(B[10], v1, B[9] * v0));
    return iv >= 0.0f && iv <= B[12] && jv >= 0.0f && jv <= B[13] && kv >= 0.0f && kv <= B[14];
}

/* ------------------------------------------------------------------------------------------ */
/* Cluster <-> box match of ONE sample.                                                                                          */
/*  rows    : n object rows (x, y, z, intensity) f32 in the keyframe's sensor frame, as msc_lidar_batch writes them               */
/*  labels  : n i32, -1 noise, else in [0, n_clusters)                                                                            */
/*  boxes   : n_boxes x 10 f64 global; ego_pose / lidar_calib: the sample's                                                      */
/*  cluster : [n_clusters, 3] i32 = match_box (box with the most rows of the cluster; ties: the smaller box; -1: no row in a box), */
/*            match_points (rows of the cluster in it), in_any_box (rows of the cluster in at least one box)                     */
/*  box     : [n_boxes, 5] i32 = rows (rows inside, noise included), cluster_rows (rows inside with label >= 0), clusters (labels  */
/*            with a row inside), best_cluster (label with the most rows inside; ties: the smaller label; -1: none), best_points */
/*  member  : (may be NULL) [n, n_boxes] u8, 1 where the row lies in the box                                                     */
/* ------------------------------------------------------------------------------------------ */
void orc_cluster_match_sample(int n, const float* rows, const int32_t* labels, int n_clusters, int n_boxes, const double* boxes,
                              const double* ego_pose, const double* lidar_calib, int32_t* cluster, int32_t* box, uint8_t* member) {
    float* bp = (float*)malloc(sizeof(float) * 16 * (size_t)(n_boxes > 0 ? n_boxes : 1));
    /* cnt[b][k]: rows of label k inside box b */
    uint32_t* cnt = (uint32_t*)calloc((size_t)(n_boxes > 0 ? n_boxes : 1) * (size_t)(n_clusters > 0 ? n_clusters : 1), sizeof(uint32_t));
    for (int b = 0; b < n_boxes; ++b) {
        orc_box_prepare(boxes + 10 * b, ego_pose, lidar_calib, bp + 16 * b, NULL);
        for (int k = 0; k < 5; ++k) box[5 * b + k] = 0;
    }
    for (int k = 0; k < n_clusters; ++k) cluster[3 * k + 2] = 0;
    for (int i = 0; i < n; ++i) {
        const float x = rows[4 * (size_t)i], y = rows[4 * (size_t)i + 1], z = rows[4 * (size_t)i + 2];
        const int lab = labels[i];
        int any = 0;
        for (int b = 0; b < n_boxes; ++b) {
            const int in = orc_in_box(bp + 16 * b, x, y, z);
            if (member) member[(size_t)i * n_boxes + b] = (uint8_t)in;
            if (!in) continue;
            any = 1;
            box[5 * b + 0] += 1;
            if (lab >= 0) {
                box[5 * b + 1] += 1;
                cnt[(size_t)b * n_clusters + lab] += 1;
            }
        }
        if (any && lab >= 0) cluster[3 * lab + 2] += 1;
    }
    for (int b = 0; b < n_boxes; ++b) {
        int best = -1;
        uint32_t best_n = 0;
        for (int k = 0; k < n_clusters; ++k) {
            const uint32_t c = cnt[(size_t)b * n_clusters + k];
            if (c > 0) box[5 * b + 2] += 1;
            if (c > best_n) { best_n = c; best = k; } /* strict: the smaller label keeps a tie */
        }
        box[5 * b + 3] = best;
        box[5 * b + 4] = (int32_t)best_n;
    }
    for (int k = 0; k < n_clusters; ++k) {
        int best = -1;
        uint32_t best_n = 0;
        for (int b = 0; b < n_boxes; ++b) {
            const uint32_t c = cnt[(size_t)b * n_clusters + k];
            if (c > best_n) { best_n = c; best = b; } /* strict: the smaller box keeps a tie */
        }
        cluster[3 * k + 0] = best;
        cluster[3 * k + 1] = (int32_t)best_n;
    }
    free(bp);
    free(cnt);
}
