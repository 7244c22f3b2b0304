// lidar_common.cuh -- what the single-keyframe path (keyframe.cu, dbscan.cu) and the batched one (keyframe_batch.cu) share: one
// copy of the gate / split rule, of the cluster-box arithmetic and of the DBSCAN pipeline, so the two paths cannot drift apart.
#pragma once
#include "msc_common.cuh"

namespace msc {

constexpr int kCompactThreads = 1024;

// monotonic float <-> uint mapping so integer atomicMin/Max order floats correctly (including negatives)
__device__ __forceinline__ uint32_t f2ord(float f) {
    uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t u) {
    uint32_t b = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
    return __uint_as_float(b);
}

// lidar_agent.py:106-110 (float32, separate roundings, strict compares) and :128
// split_only: _segment_ground alone (no gate; a NaN z compares false and lands in `object`, like pc[~mask])
__device__ __forceinline__ uint32_t keyframe_class(const float* __restrict__ p, const msc_params& P, bool split_only) {
    const float d = __fsqrt_rn(__fadd_rn(__fmul_rn(p[0], p[0]), __fmul_rn(p[1], p[1])));
    const bool ok = split_only || ((d > P.range_min) && (d < P.range_max) && (p[2] < P.z_max) && (p[2] > P.z_min));
    if (!ok) return 0u;
    return (p[2] < P.ground_z) ? 1u : 2u;  // 1 ground, 2 object
}

// exclusive scan of per-block (ground, object) counts, single block; defined in keyframe.cu
__global__ void __launch_bounds__(1024) kf_scan_kernel(uint32_t* __restrict__ block_counts, uint32_t n_blocks, uint32_t* __restrict__ counts);

// ---------------------------------------------------------------- keyframe BEV (lidar_agent.py:539-597): keyframe.cu and lidar_images.cu
// cell of a row: x and y cells of :547-552, [y, x] indexing (:559)
__device__ __forceinline__ void bev_xy(const float4& p, float bev_range, float two_r, float resf, int res, int* ix, int* iy) {
    *ix = bev_cell<false>(p.x, bev_range, two_r, 0.0f, resf, res - 1);
    *iy = bev_cell<false>(p.y, bev_range, two_r, 0.0f, resf, res - 1);
}
// semantic BGR of a cell from its winner key (0 empty, 1 ground, 2 + i object row i of `object`) and the ordered-int min / max
// of the object heights in zrange[0..1]
__device__ __forceinline__ void bev_colour(uint32_t w, const float4* __restrict__ object, const uint32_t* __restrict__ zrange, uint8_t* b,
                                           uint8_t* g, uint8_t* r) {
    *b = 0; *g = 0; *r = 0;
    if (w == 1u) { *b = 80; *g = 80; *r = 120; }  // :572
    else if (w >= 2u) {
        const float hmin = ord2f(zrange[0]), hmax = ord2f(zrange[1]);
        int gv;
        if (!(hmax > hmin)) gv = 255;  // :581-582 norm = 0.5 -> int(255 * (1 - (0.5 - 0.5) * 2))
        else {
            const float hn = __fdiv_rn(__fsub_rn(object[w - 2u].z, hmin), __fsub_rn(hmax, hmin));  // :580
            if (hn < 0.5f) gv = __float2int_rz(__fmul_rn(255.0f, __fsub_rn(1.0f, __fmul_rn(hn, 2.0f))));  // :589
            else gv = __float2int_rz(__fmul_rn(255.0f, __fsub_rn(1.0f, __fmul_rn(__fsub_rn(hn, 0.5f), 2.0f))));  // :594
        }
        *b = 0; *g = (uint8_t)gv; *r = 255;  // :597 BGR
    }
}

// ---------------------------------------------------------------- cluster 4-view raster (cluster_views.cu), also run by lidar_images.cu
constexpr int kView = 256, kGrid = 512;  // img_size and the 2x2 grid (lidar_agent.py:242, :267)
__global__ void __launch_bounds__(256) cluster_splat_kernel(const float4* __restrict__ pts, const uint32_t* __restrict__ order,
                                                           const int32_t* __restrict__ cluster_off, int n_clusters, const float* __restrict__ center_scale,
                                                           uint32_t* __restrict__ keys, uint32_t* __restrict__ irange);
__global__ void __launch_bounds__(256) cluster_colour_kernel(const float4* __restrict__ pts, const uint32_t* __restrict__ order,
                                                            const int32_t* __restrict__ cluster_off, const uint32_t* __restrict__ keys,
                                                            const uint32_t* __restrict__ irange, uint8_t* __restrict__ out);

// ---------------------------------------------------------------- DBSCAN over the rows of many samples (dbscan.cu)
constexpr uint32_t kDbUnmerged = 1u, kLbOverflow = 2u;  // bits of msc_lidar_batch's status word (include/msc_geom.h)

// cubic cells of side 1 / inv_cell from (ox, oy, oz); a row's key is sample * ncells + its cell
struct DbGrid {
    double ox, oy, oz, inv_cell;
    int nx, ny, nz;
    uint64_t ncells;
};

// the per-sample cluster table: the label kernel initialises the slot of every cluster, msc_lidar_batch fills and finishes them
struct ClusterTable {
    const uint32_t* object_off;
    const uint32_t* rank;     // exclusive scan of is_root
    uint32_t* slots;          // [cap, 11]: ordered min3, max3, -, -, -, -, count; finished in place
    uint32_t* first;          // [cap]: smallest row of the slot's cluster (the caller's cluster_first)
    int32_t* labels;
    int32_t* noise_first;
};

// byte offsets of DBSCAN's buffers in a caller's workspace, for `cap` rows whose keys lie below pad_key
struct DbWs {
    size_t keys_in, keys_out, vals_in, sidx, core, parent, is_root, rank, temp, temp_bytes, end;
    uint32_t cap;
    uint64_t pad_key;  // n_samples * ncells: the key of the rows past the last object row
    int end_bit;
};
// lays the buffers out from byte `base` (256-aligned) on; W->end is the first byte past them
cudaError_t db_layout(size_t base, uint32_t cap, int n_samples, const DbGrid& G, DbWs* W);

// Enqueues on `stream`: key -> radix sort -> core -> hook -> verify -> flatten -> exclusive scan of is_root into W.rank -> label, over
// rows [0, totals[2]) of `object`; row i belongs to sample object_sample[i], and rows of different samples are never neighbours.
// Writes t.labels (numbered per sample from 0), t.noise_first and the initial slot of every cluster of t; sets kDbUnmerged in
// *status if the merge left an edge unmerged.  is_root and rank (cap + 1 entries each; rank[cap] is the number of clusters) stay
// in the workspace.  t.rank must point at W.rank.
cudaError_t db_enqueue(const DbWs& W, unsigned char* ws, const DbGrid& G, const float4* object, const uint32_t* object_sample,
                       const uint32_t* totals, double eps, uint32_t min_samples, const ClusterTable& t, uint32_t* status,
                       cudaStream_t stream);

// per-cluster box (lidar_agent.py:200-204) from 11 words: ordered-int min3, max3, -, -, -, -, count -> f32 min3, max3, center3,
// distance, num_points, in place
__device__ __forceinline__ void cluster_finish(uint32_t* s) {
    float* o = reinterpret_cast<float*>(s);
    float mn[3], mx[3];
    const uint32_t cnt = s[10];
#pragma unroll
    for (int k = 0; k < 3; ++k) { mn[k] = cnt ? ord2f(s[k]) : INFINITY; mx[k] = cnt ? ord2f(s[3 + k]) : -INFINITY; }
#pragma unroll
    for (int k = 0; k < 3; ++k) { o[k] = mn[k]; o[3 + k] = mx[k]; o[6 + k] = __fdiv_rn(__fadd_rn(mn[k], mx[k]), 2.0f); }  // :203
    o[9] = __fsqrt_rn(__fadd_rn(__fmul_rn(o[6], o[6]), __fmul_rn(o[7], o[7])));                                             // :204
    o[10] = (float)cnt;
}

}  // namespace msc
