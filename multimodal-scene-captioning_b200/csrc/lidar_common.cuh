// lidar_common.cuh -- device helpers of the keyframe path that both the single-keyframe kernels (keyframe.cu, dbscan.cu) and
// the batched ones (keyframe_batch.cu) use: one copy of the gate / split rule, of the neighbour relation, of the union-find
// and of the cluster-box arithmetic, so the two paths cannot drift apart.
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

// DBSCAN neighbour relation: squared distance in float64, accumulated x -> y -> z (scikit-learn's KD-tree reduced distance)
__device__ __forceinline__ double db_dist2(double px, double py, double pz, const float* __restrict__ q) {
    const double dx = px - (double)q[0], dy = py - (double)q[1], dz = pz - (double)q[2];
    double d = dx * dx;
    d = d + dy * dy;
    d = d + dz * dz;
    return d;
}

__device__ __forceinline__ uint32_t db_find(const uint32_t* parent, uint32_t a) {
    uint32_t p = ((const volatile uint32_t*)parent)[a];
    while (p != a) { a = p; p = ((const volatile uint32_t*)parent)[a]; }
    return a;
}

// union of the trees of i and j: the larger root is hung under the smaller one (atomicMin), so a component's root converges to its
// smallest index.  When the atomicMin finds hi already relinked (by another thread) to old < hi, hi's subtree moves under lo and this
// thread goes on to merge old's tree with lo's, so the edge it cut is restored before it returns.  on_hook() runs on every atomic.
template <class F>
__device__ __forceinline__ void db_union(uint32_t* parent, uint32_t i, uint32_t j, F on_hook) {
    uint32_t a = db_find(parent, i), b = db_find(parent, j);
    while (a != b) {
        const uint32_t hi = max(a, b), lo = min(a, b);
        const uint32_t old = atomicMin(&parent[hi], lo);
        on_hook();
        if (old == hi) break;   // hi was a root and now hangs under lo
        a = db_find(parent, old);  // hi already had a smaller parent: merge that tree with lo
        b = db_find(parent, lo);
    }
}

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
