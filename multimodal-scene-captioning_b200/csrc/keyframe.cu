// keyframe.cu -- bit-exact device versions of the reference's single-keyframe LiDAR functions
// (lidar_agent.py:103-132 filter/split, :539-597 BEV raster, :198-204 cluster boxes, baseline_gpt4o.py:276-285
// cloud statistics) and the materialised multi-sweep aggregation (devkit from_file_multisweep, App. A.1).
//
// These are the latency path behind the drop-in LiDARAgent methods: one keyframe (35k points) at a time,
// many CTAs per cloud, global (L2) atomics into an 800x800 grid that cannot be privatised in shared memory
// (5 MB), order-preserving compaction through block counts + a scan + an ordered scatter.
#include "lidar_common.cuh"

namespace msc {

// pass 1: per-block counts of kept / ground / object rows
__global__ void __launch_bounds__(kCompactThreads) kf_count_kernel(const __grid_constant__ msc_params P, const float* __restrict__ pts,
                                                                  uint32_t n, int pitch, bool split_only, uint32_t* __restrict__ block_counts) {
    __shared__ uint32_t s_cnt[2];
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t i = blockIdx.x * kCompactThreads + threadIdx.x;
    uint32_t cls = 0;
    if (i < n) cls = keyframe_class(pts + (size_t)i * pitch, P, split_only);
    const uint32_t g = __popc(__ballot_sync(0xffffffffu, cls == 1u));
    const uint32_t o = __popc(__ballot_sync(0xffffffffu, cls == 2u));
    if ((threadIdx.x & 31) == 0) { atomicAdd(&s_cnt[0], g); atomicAdd(&s_cnt[1], o); }
    __syncthreads();
    if (threadIdx.x < 2) block_counts[blockIdx.x * 2 + threadIdx.x] = s_cnt[threadIdx.x];
}

// pass 2: exclusive scan of the per-block counts (single block), totals to counts[3] = kept, ground, object
__global__ void __launch_bounds__(1024) kf_scan_kernel(uint32_t* __restrict__ block_counts, uint32_t n_blocks, uint32_t* __restrict__ counts) {
    __shared__ uint32_t s_warp[2][32];
    __shared__ uint32_t s_carry[2];
    if (threadIdx.x < 2) s_carry[threadIdx.x] = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_blocks; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        uint32_t v[2] = {0, 0};
        if (i < n_blocks) { v[0] = block_counts[i * 2]; v[1] = block_counts[i * 2 + 1]; }
        uint32_t incl[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            uint32_t x = v[k];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
                if ((threadIdx.x & 31) >= d) x += y;
            }
            incl[k] = x;
            if ((threadIdx.x & 31) == 31) s_warp[k][threadIdx.x >> 5] = x;
        }
        __syncthreads();
        if (threadIdx.x < 32) {
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                uint32_t x = s_warp[k][threadIdx.x];
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
                    if (threadIdx.x >= d) x += y;
                }
                s_warp[k][threadIdx.x] = x;  // inclusive over warps
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const uint32_t warp_off = (threadIdx.x >> 5) ? s_warp[k][(threadIdx.x >> 5) - 1] : 0u;
            const uint32_t excl = s_carry[k] + warp_off + incl[k] - v[k];
            if (i < n_blocks) block_counts[i * 2 + k] = excl;
        }
        __syncthreads();
        if (threadIdx.x == 0) { s_carry[0] += s_warp[0][31]; s_carry[1] += s_warp[1][31]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { counts[0] = s_carry[0] + s_carry[1]; counts[1] = s_carry[0]; counts[2] = s_carry[1]; }
}

// pass 3: ordered scatter.  Within a block, ranks come from warp ballots + a warp-offset scan, so row order is
// exactly the input order (boolean-mask indexing, lidar_agent.py:112,129-130).
__global__ void __launch_bounds__(kCompactThreads) kf_scatter_kernel(const __grid_constant__ msc_params P, const float* __restrict__ pts,
                                                                    uint32_t n, int pitch, bool split_only, const uint32_t* __restrict__ block_offsets,
                                                                    float* __restrict__ kept, float* __restrict__ ground,
                                                                    float* __restrict__ object) {
    __shared__ uint32_t s_w[2][32];
    const uint32_t i = blockIdx.x * kCompactThreads + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t cls = 0;
    float4 row = make_float4(0, 0, 0, 0);
    if (i < n) {
        const float* p = pts + (size_t)i * pitch;
        cls = keyframe_class(p, P, split_only);
        row = make_float4(p[0], p[1], p[2], p[3]);
    }
    const uint32_t bg = __ballot_sync(0xffffffffu, cls == 1u), bo = __ballot_sync(0xffffffffu, cls == 2u);
    if (lane == 0) { s_w[0][warp] = __popc(bg); s_w[1][warp] = __popc(bo); }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            uint32_t v = s_w[k][lane], x = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
                if (lane >= d) x += y;
            }
            s_w[k][lane] = x - v;  // exclusive
        }
    }
    __syncthreads();
    if (cls == 0u) return;
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t g_rank = block_offsets[blockIdx.x * 2 + 0] + s_w[0][warp] + __popc(bg & lt);
    const uint32_t o_rank = block_offsets[blockIdx.x * 2 + 1] + s_w[1][warp] + __popc(bo & lt);
    // kept rank = ground-before + object-before (both lists are order-preserving subsequences of kept)
    reinterpret_cast<float4*>(kept)[g_rank + o_rank] = row;
    if (cls == 1u) reinterpret_cast<float4*>(ground)[g_rank] = row;
    else reinterpret_cast<float4*>(object)[o_rank] = row;
}

// ---------------------------------------------------------------- keyframe BEV raster (lidar_agent.py:539-597)
__global__ void __launch_bounds__(256) kf_bev_raster_kernel(const __grid_constant__ msc_params P, const float4* __restrict__ ground,
                                                           uint32_t n_ground, const float4* __restrict__ object, uint32_t n_object,
                                                           uint32_t* __restrict__ count, float* __restrict__ height,
                                                           uint32_t* __restrict__ winner, uint32_t* __restrict__ zrange) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n = n_ground + n_object;
    const int res = P.bev_res;
    const float two_r = __fmul_rn(2.0f, P.bev_range), resf = (float)res;
    uint32_t zlo = 0xffffffffu, zhi = 0u;
    if (i < n) {
        const bool is_obj = i >= n_ground;
        const float4 p = is_obj ? object[i - n_ground] : ground[i];
        int ix, iy;
        bev_xy(p, P.bev_range, two_r, resf, res, &ix, &iy);
        const size_t cell = (size_t)iy * res + ix;  // [y, x] indexing, :559
        atomicAdd(&count[cell], 1u);                                                   // :559
        if (p.z > 0.0f) atomicMax(reinterpret_cast<int*>(height) + cell, __float_as_int(p.z));  // :560, 0-initialised
        // last writer wins (:571-572, :584-597): objects are drawn after ground, later array index wins
        atomicMax(&winner[cell], is_obj ? (2u + (i - n_ground)) : 1u);
        if (is_obj) { zlo = f2ord(p.z); zhi = zlo; }
    }
    // per-warp min/max of object heights (:579-580)
    zlo = __reduce_min_sync(0xffffffffu, zlo);
    zhi = __reduce_max_sync(0xffffffffu, zhi);
    if ((threadIdx.x & 31) == 0 && zlo != 0xffffffffu) { atomicMin(&zrange[0], zlo); atomicMax(&zrange[1], zhi); }
}

__global__ void __launch_bounds__(256) kf_bev_colour_kernel(const float4* __restrict__ object, const uint32_t* __restrict__ winner,
                                                           const uint32_t* __restrict__ zrange, uint32_t ncell,
                                                           uint8_t* __restrict__ semantic_bgr) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncell) return;
    uint8_t b, g, r;
    bev_colour(winner[c], object, zrange, &b, &g, &r);
    semantic_bgr[(size_t)c * 3 + 0] = b; semantic_bgr[(size_t)c * 3 + 1] = g; semantic_bgr[(size_t)c * 3 + 2] = r;
}

// ---------------------------------------------------------------- raw-cloud statistics (baseline_gpt4o.py:276-285)
__global__ void __launch_bounds__(256) cloud_stats_kernel(const float* __restrict__ pts, uint32_t n, int pitch, uint32_t* __restrict__ mm_ord,
                                                         double* __restrict__ radial_sum) {
    uint32_t lo[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, hi[3] = {0, 0, 0};
    double acc = 0.0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float* p = pts + (size_t)i * pitch;
#pragma unroll
        for (int k = 0; k < 3; ++k) { const uint32_t o = f2ord(p[k]); lo[k] = min(lo[k], o); hi[k] = max(hi[k], o); }
        acc += (double)__fsqrt_rn(__fadd_rn(__fmul_rn(p[0], p[0]), __fmul_rn(p[1], p[1])));
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        lo[k] = __reduce_min_sync(0xffffffffu, lo[k]);
        hi[k] = __reduce_max_sync(0xffffffffu, hi[k]);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) { atomicMin(&mm_ord[k], lo[k]); atomicMax(&mm_ord[3 + k], hi[k]); }
        atomicAdd(radial_sum, acc);
    }
}
// mm_ord aliases out7[3..5]; every lane reads its word before any lane writes (single warp + __syncwarp)
__global__ void cloud_stats_finish_kernel(const uint32_t* mm_ord, double* out7) {
    float v = 0.0f;
    if (threadIdx.x < 6) v = ord2f(mm_ord[threadIdx.x]);
    __syncwarp();
    if (threadIdx.x < 6) out7[threadIdx.x] = (double)v;
}

// ---------------------------------------------------------------- per-cluster boxes (lidar_agent.py:200-204)
__global__ void __launch_bounds__(256) cluster_minmax_kernel(const float* __restrict__ pts, uint32_t n, int pitch, const int32_t* __restrict__ labels,
                                                            int n_clusters, uint32_t* __restrict__ scratch11) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int c = labels[i];
    if (c < 0 || c >= n_clusters) return;
    const float* p = pts + (size_t)i * pitch;
    uint32_t* o = scratch11 + (size_t)c * 11;
#pragma unroll
    for (int k = 0; k < 3; ++k) { const uint32_t v = f2ord(p[k]); atomicMin(&o[k], v); atomicMax(&o[3 + k], v); }
    atomicAdd(&o[10], 1u);
}
__global__ void cluster_init_kernel(uint32_t* __restrict__ scratch11, int n_clusters) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_clusters * 11) return;
    const int k = i % 11;
    scratch11[i] = (k < 3) ? 0xffffffffu : 0u;
}
__global__ void cluster_finish_kernel(uint32_t* __restrict__ scratch11, int n_clusters) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_clusters) return;
    cluster_finish(scratch11 + (size_t)c * 11);
}

// ---------------------------------------------------------------- materialised multi-sweep aggregation (App. A.1)
__device__ __forceinline__ bool sweep_locate(uint32_t gi, uint32_t max_pts, int n_sweeps, const uint32_t* __restrict__ sweep_count, int* s,
                                             uint32_t* local) {
    *s = (int)(gi / max_pts);
    *local = gi - (uint32_t)(*s) * max_pts;
    return (*s < n_sweeps) && (*local < sweep_count[*s]);
}
__global__ void __launch_bounds__(kCompactThreads) agg_count_kernel(float rc, const float* __restrict__ points, int n_sweeps,
                                                                   const uint32_t* __restrict__ sweep_start, const uint32_t* __restrict__ sweep_count,
                                                                   uint32_t max_pts, uint32_t* __restrict__ block_counts) {
    const uint32_t gi = blockIdx.x * kCompactThreads + threadIdx.x;
    int s; uint32_t local;
    bool keep = false;
    if (sweep_locate(gi, max_pts, n_sweeps, sweep_count, &s, &local)) {
        const float* p = points + ((size_t)sweep_start[s] + local) * 5;
        keep = !(fabsf(p[0]) < rc && fabsf(p[1]) < rc);
    }
    const uint32_t c = __popc(__ballot_sync(0xffffffffu, keep));
    __shared__ uint32_t s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_cnt, c);
    __syncthreads();
    if (threadIdx.x == 0) { block_counts[blockIdx.x * 2] = s_cnt; block_counts[blockIdx.x * 2 + 1] = 0; }
}
__global__ void __launch_bounds__(kCompactThreads) agg_scatter_kernel(float rc, const float* __restrict__ points, int n_sweeps,
                                                                     const uint32_t* __restrict__ sweep_start, const uint32_t* __restrict__ sweep_count,
                                                                     const double* __restrict__ sweep_pose, const float* __restrict__ sweep_time_lag,
                                                                     uint32_t max_pts, const uint32_t* __restrict__ block_offsets,
                                                                     float* __restrict__ out_xyzi, float* __restrict__ out_time) {
    __shared__ uint32_t s_w[32];
    const uint32_t gi = blockIdx.x * kCompactThreads + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int s = 0; uint32_t local = 0;
    bool keep = false;
    const float* p = nullptr;
    if (sweep_locate(gi, max_pts, n_sweeps, sweep_count, &s, &local)) {
        p = points + ((size_t)sweep_start[s] + local) * 5;
        keep = !(fabsf(p[0]) < rc && fabsf(p[1]) < rc);
    }
    const uint32_t bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s_w[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
        uint32_t v = s_w[lane], x = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += y; }
        s_w[lane] = x - v;
    }
    __syncthreads();
    if (!keep) return;
    const uint32_t rank = block_offsets[blockIdx.x * 2] + s_w[warp] + __popc(bal & ((1u << lane) - 1u));
    const double* M = sweep_pose + (size_t)s * 12;
    const double xd = (double)p[0], yd = (double)p[1], zd = (double)p[2];
    float4 o;
    o.x = (float)__fma_rn(M[0], xd, __fma_rn(M[1], yd, __fma_rn(M[2], zd, M[3])));
    o.y = (float)__fma_rn(M[4], xd, __fma_rn(M[5], yd, __fma_rn(M[6], zd, M[7])));
    o.z = (float)__fma_rn(M[8], xd, __fma_rn(M[9], yd, __fma_rn(M[10], zd, M[11])));
    o.w = p[3];
    reinterpret_cast<float4*>(out_xyzi)[rank] = o;
    out_time[rank] = sweep_time_lag[s];
}

}  // namespace msc

extern "C" {

int msc_keyframe_filter_split(const msc_params* params, const float* pts, uint32_t n, int32_t pitch, int32_t split_only, float* kept,
                              float* ground, float* object, uint32_t* counts, uint32_t* scratch, size_t scratch_elems, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(params && counts && scratch, "null argument");
    MSC_REQUIRE(pitch >= 4, "pitch must be >= 4 floats");
    cudaStream_t stream = (cudaStream_t)stream_v;
    const uint32_t n_blocks = (n + kCompactThreads - 1) / kCompactThreads;
    MSC_REQUIRE(scratch_elems >= (size_t)n_blocks * 2 + 2, "scratch too small: need %zu u32", (size_t)n_blocks * 2 + 2);
    if (n == 0) { MSC_CUDA(cudaMemsetAsync(counts, 0, 3 * sizeof(uint32_t), stream)); return MSC_OK; }
    MSC_REQUIRE(pts && kept && ground && object, "null buffer");
    kf_count_kernel<<<n_blocks, kCompactThreads, 0, stream>>>(*params, pts, n, pitch, split_only != 0, scratch);
    kf_scan_kernel<<<1, 1024, 0, stream>>>(scratch, n_blocks, counts);
    kf_scatter_kernel<<<n_blocks, kCompactThreads, 0, stream>>>(*params, pts, n, pitch, split_only != 0, scratch, kept, ground, object);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

int msc_keyframe_bev(const msc_params* params, const float* ground, uint32_t n_ground, const float* object, uint32_t n_object,
                     uint32_t* count, float* height, uint8_t* semantic_bgr, uint32_t* winner, uint32_t* zrange, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(params && count && height && semantic_bgr && winner && zrange, "null argument");
    MSC_REQUIRE(params->bev_res > 0 && params->bev_res <= 8192, "bev_res out of range");
    cudaStream_t stream = (cudaStream_t)stream_v;
    const size_t ncell = (size_t)params->bev_res * params->bev_res;
    MSC_CUDA(cudaMemsetAsync(count, 0, ncell * 4, stream));
    MSC_CUDA(cudaMemsetAsync(height, 0, ncell * 4, stream));
    MSC_CUDA(cudaMemsetAsync(winner, 0, ncell * 4, stream));
    MSC_CUDA(cudaMemsetAsync(zrange, 0xff, 4, stream));
    MSC_CUDA(cudaMemsetAsync(zrange + 1, 0, 4, stream));
    const uint32_t n = n_ground + n_object;
    if (n) {
        kf_bev_raster_kernel<<<(n + 255) / 256, 256, 0, stream>>>(*params, reinterpret_cast<const float4*>(ground), n_ground,
                                                                  reinterpret_cast<const float4*>(object), n_object, count, height, winner,
                                                                  zrange);
    }
    kf_bev_colour_kernel<<<(unsigned)((ncell + 255) / 256), 256, 0, stream>>>(reinterpret_cast<const float4*>(object), winner, zrange,
                                                                              (uint32_t)ncell, semantic_bgr);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

int msc_cloud_stats(const float* pts, uint32_t n, int32_t pitch, double* out7, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(out7, "null argument");
    MSC_REQUIRE(pitch >= 3, "pitch must be >= 3 floats");
    cudaStream_t stream = (cudaStream_t)stream_v;
    // out7[0..5] double slots double as scratch: first 6 u32 of the buffer hold ordered min/max during the pass
    uint32_t* mm = reinterpret_cast<uint32_t*>(out7 + 3);  // bytes 24..47: slots 3,4,5 (rewritten by finish)
    MSC_CUDA(cudaMemsetAsync(mm, 0xff, 12, stream));
    MSC_CUDA(cudaMemsetAsync(mm + 3, 0, 12, stream));
    MSC_CUDA(cudaMemsetAsync(out7 + 6, 0, 8, stream));
    if (n) {
        int blocks = (int)((n + 255) / 256);
        if (blocks > 1184) blocks = 1184;
        cloud_stats_kernel<<<blocks, 256, 0, stream>>>(pts, n, pitch, mm, out7 + 6);
    }
    // finish reads the 6 ordered words and writes 6 doubles; one warp, reads complete before writes (registers)
    cloud_stats_finish_kernel<<<1, 32, 0, stream>>>(mm, out7);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

int msc_cluster_aabb(const float* pts, uint32_t n, int32_t pitch, const int32_t* labels, int32_t n_clusters, float* out11, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(n_clusters >= 0, "negative n_clusters");
    if (n_clusters == 0) return MSC_OK;
    MSC_REQUIRE(out11 && (n == 0 || (pts && labels)), "null argument");
    cudaStream_t stream = (cudaStream_t)stream_v;
    uint32_t* scratch = reinterpret_cast<uint32_t*>(out11);
    cluster_init_kernel<<<(n_clusters * 11 + 255) / 256, 256, 0, stream>>>(scratch, n_clusters);
    if (n) cluster_minmax_kernel<<<(n + 255) / 256, 256, 0, stream>>>(pts, n, pitch, labels, n_clusters, scratch);
    cluster_finish_kernel<<<(n_clusters + 127) / 128, 128, 0, stream>>>(scratch, n_clusters);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

int msc_aggregate_sweeps(float remove_close_radius, const float* points, int32_t n_sweeps, const uint32_t* sweep_start,
                         const uint32_t* sweep_count, const double* sweep_pose, const float* sweep_time_lag,
                         uint32_t max_points_per_sweep, float* out_xyzi, float* out_time, uint32_t* n_out, uint32_t* scratch,
                         size_t scratch_elems, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(n_out && scratch, "null argument");
    MSC_REQUIRE(n_sweeps >= 0, "negative n_sweeps");
    cudaStream_t stream = (cudaStream_t)stream_v;
    const uint64_t span = (uint64_t)n_sweeps * max_points_per_sweep;
    MSC_REQUIRE(span < 0xffffffffull, "too many points");
    const uint32_t n_blocks = (uint32_t)((span + kCompactThreads - 1) / kCompactThreads);
    MSC_REQUIRE(scratch_elems >= (size_t)n_blocks * 2 + 8, "scratch too small: need %zu u32", (size_t)n_blocks * 2 + 8);
    if (span == 0) { MSC_CUDA(cudaMemsetAsync(n_out, 0, 4, stream)); return MSC_OK; }
    MSC_REQUIRE(points && sweep_start && sweep_count && sweep_pose && sweep_time_lag && out_xyzi && out_time, "null buffer");
    uint32_t* totals = scratch + (size_t)n_blocks * 2;  // kf_scan writes 3 totals; [0] is the kept count
    agg_count_kernel<<<n_blocks, kCompactThreads, 0, stream>>>(remove_close_radius, points, n_sweeps, sweep_start, sweep_count,
                                                                 max_points_per_sweep, scratch);
    kf_scan_kernel<<<1, 1024, 0, stream>>>(scratch, n_blocks, totals);
    agg_scatter_kernel<<<n_blocks, kCompactThreads, 0, stream>>>(remove_close_radius, points, n_sweeps, sweep_start, sweep_count, sweep_pose,
                                                                   sweep_time_lag, max_points_per_sweep, scratch, out_xyzi, out_time);
    MSC_CUDA(cudaMemcpyAsync(n_out, totals, 4, cudaMemcpyDeviceToDevice, stream));
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

}  // extern "C"
