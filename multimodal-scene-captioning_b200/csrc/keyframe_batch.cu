// keyframe_batch.cu -- the reference's LiDAR evidence (keyframe filter + ground split, DBSCAN, per-cluster boxes; lidar_agent.py:103-209)
// for every sample of a packed batch in one stream-ordered pass (DESIGN.md section 4.5).
//
// Per sample the results are those of msc_keyframe_filter_split, msc_dbscan and msc_cluster_aabb on the sample's keyframe: the gate /
// split rule and the cluster-box arithmetic are the same code (lidar_common.cuh), and DBSCAN is the same pipeline (dbscan.cu).
//   1. filter / split: 1024-row tiles of keyframe rows, never spanning two samples; per-tile counts, one exclusive scan over the tiles
//      (tile order is sample order, so the scan also gives each sample's ground / object offset), an ordered scatter.
//   2. DBSCAN over the object rows of all samples at once (db_enqueue).
//   3. cluster table: ordered-int min / max, count and first row per (sample, cluster) slot object_off[s] + k, then the finish pass.
#include "lidar_common.cuh"

#include <cub/block/block_scan.cuh>

namespace msc {

// ---------------------------------------------------------------- 1. keyframe filter / split
// one block of 256: keyframe rows per sample, tile offsets (exclusive scan of ceil(rows / 1024)), status and noise_first initialised
__global__ void __launch_bounds__(256) lb_plan_kernel(int n_samples, const int32_t* __restrict__ sample_sweep_off,
                                                       const uint32_t* __restrict__ sweep_count, uint32_t row_capacity,
                                                       uint32_t* __restrict__ kf_n, uint32_t* __restrict__ tile_off,
                                                       int32_t* __restrict__ noise_first, uint32_t* __restrict__ status) {
    using Scan = cub::BlockScan<unsigned long long, 256>;
    __shared__ typename Scan::TempStorage tmp;
    __shared__ unsigned long long s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < n_samples; base += 256) {
        const int s = base + threadIdx.x;
        uint32_t n = 0;
        if (s < n_samples) {
            const int a = sample_sweep_off[s];
            n = (sample_sweep_off[s + 1] > a) ? sweep_count[a] : 0u;
            kf_n[s] = n;
            noise_first[s] = 0x7fffffff;
        }
        // rows in the high word, tiles in the low word: one scan for both
        const unsigned long long v = ((unsigned long long)n << 32) | ((n + kCompactThreads - 1) / kCompactThreads);
        unsigned long long excl, total;
        Scan(tmp).ExclusiveSum(v, excl, total);
        excl += s_carry;
        if (s < n_samples) tile_off[s] = (uint32_t)excl;
        __syncthreads();
        if (threadIdx.x == 0) s_carry += total;
        __syncthreads();
    }
    const bool overflow = (s_carry >> 32) > row_capacity;
    if (threadIdx.x == 0) {
        tile_off[n_samples] = overflow ? 0u : (uint32_t)s_carry;
        *status = overflow ? kLbOverflow : 0u;
    }
    if (overflow)  // every sample reads as empty; the status word says why
        for (int s = threadIdx.x; s < n_samples; s += 256) { kf_n[s] = 0; tile_off[s] = 0; }
}

// sample owning tile b: the last s with tile_off[s] <= b (samples without tiles have tile_off[s] == tile_off[s + 1])
__device__ __forceinline__ int lb_tile_sample(const uint32_t* __restrict__ tile_off, int n_samples, uint32_t b) {
    int lo = 0, hi = n_samples;  // tile_off[lo] <= b < tile_off[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (tile_off[mid] <= b) lo = mid; else hi = mid;
    }
    return lo;
}

struct LbTile {
    int s;
    uint32_t cls;
    const float* p;
};
__device__ __forceinline__ LbTile lb_tile_row(const msc_params& P, const float* __restrict__ points, const int32_t* __restrict__ sample_sweep_off,
                                              const uint32_t* __restrict__ sweep_start, const uint32_t* __restrict__ kf_n,
                                              const uint32_t* __restrict__ tile_off, int n_samples) {
    LbTile t{-1, 0u, nullptr};
    const uint32_t b = blockIdx.x;
    if (b >= tile_off[n_samples]) return t;
    t.s = lb_tile_sample(tile_off, n_samples, b);
    const uint32_t local = (b - tile_off[t.s]) * kCompactThreads + threadIdx.x;
    if (local < kf_n[t.s]) {
        t.p = points + ((size_t)sweep_start[sample_sweep_off[t.s]] + local) * 5;
        t.cls = keyframe_class(t.p, P, false);
    }
    return t;
}

// per-tile ground / object counts (tiles past the batch's last one count zero)
__global__ void __launch_bounds__(kCompactThreads) lb_count_kernel(const __grid_constant__ msc_params P, const float* __restrict__ points,
                                                                  const int32_t* __restrict__ sample_sweep_off, const uint32_t* __restrict__ sweep_start,
                                                                  const uint32_t* __restrict__ kf_n, const uint32_t* __restrict__ tile_off,
                                                                  int n_samples, uint32_t* __restrict__ block_counts) {
    __shared__ uint32_t s_cnt[2];
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const LbTile t = lb_tile_row(P, points, sample_sweep_off, sweep_start, kf_n, tile_off, n_samples);
    const uint32_t g = __popc(__ballot_sync(0xffffffffu, t.cls == 1u));
    const uint32_t o = __popc(__ballot_sync(0xffffffffu, t.cls == 2u));
    if ((threadIdx.x & 31) == 0) { atomicAdd(&s_cnt[0], g); atomicAdd(&s_cnt[1], o); }
    __syncthreads();
    if (threadIdx.x < 2) block_counts[blockIdx.x * 2 + threadIdx.x] = s_cnt[threadIdx.x];
}

// per-sample counts and offsets from the scanned tile counts (n_tiles: the launch's tile count; totals[1..2]: the scan's totals)
__global__ void __launch_bounds__(256) lb_offsets_kernel(int n_samples, const uint32_t* __restrict__ tile_off, const uint32_t* __restrict__ block_counts,
                                                        uint32_t n_tiles, const uint32_t* __restrict__ totals, uint32_t* __restrict__ counts,
                                                        uint32_t* __restrict__ ground_off, uint32_t* __restrict__ object_off) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_samples) return;
    const uint32_t a = tile_off[s], b = tile_off[s + 1];
    uint32_t lo[2], hi[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        lo[k] = a < n_tiles ? block_counts[a * 2 + k] : totals[1 + k];
        hi[k] = b < n_tiles ? block_counts[b * 2 + k] : totals[1 + k];
    }
    ground_off[s] = lo[0];
    object_off[s] = lo[1];
    counts[s * 3 + 0] = (hi[0] - lo[0]) + (hi[1] - lo[1]);
    counts[s * 3 + 1] = hi[0] - lo[0];
    counts[s * 3 + 2] = hi[1] - lo[1];
}

// ordered scatter (the ranks of kf_scatter_kernel); every object row also records its sample
__global__ void __launch_bounds__(kCompactThreads) lb_scatter_kernel(const __grid_constant__ msc_params P, const float* __restrict__ points,
                                                                    const int32_t* __restrict__ sample_sweep_off, const uint32_t* __restrict__ sweep_start,
                                                                    const uint32_t* __restrict__ kf_n, const uint32_t* __restrict__ tile_off,
                                                                    int n_samples, const uint32_t* __restrict__ block_offsets,
                                                                    float4* __restrict__ ground, float4* __restrict__ object,
                                                                    uint32_t* __restrict__ object_sample) {
    __shared__ uint32_t s_w[2][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const LbTile t = lb_tile_row(P, points, sample_sweep_off, sweep_start, kf_n, tile_off, n_samples);
    const uint32_t bg = __ballot_sync(0xffffffffu, t.cls == 1u), bo = __ballot_sync(0xffffffffu, t.cls == 2u);
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
            s_w[k][lane] = x - v;
        }
    }
    __syncthreads();
    if (t.cls == 0u) return;
    const uint32_t lt = (1u << lane) - 1u;
    const float4 row = make_float4(t.p[0], t.p[1], t.p[2], t.p[3]);
    if (t.cls == 1u) {
        ground[block_offsets[blockIdx.x * 2 + 0] + s_w[0][warp] + __popc(bg & lt)] = row;
    } else {
        const uint32_t r = block_offsets[blockIdx.x * 2 + 1] + s_w[1][warp] + __popc(bo & lt);
        object[r] = row;
        object_sample[r] = (uint32_t)t.s;
    }
}

// ---------------------------------------------------------------- 3. per-sample cluster table
__global__ void __launch_bounds__(256) lb_minmax_kernel(const float4* __restrict__ object, const uint32_t* __restrict__ object_sample,
                                                       const uint32_t* __restrict__ totals, const ClusterTable t) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= totals[2]) return;
    const int c = t.labels[i];
    if (c < 0) return;
    const uint32_t off = t.object_off[object_sample[i]];
    const float4 p = object[i];
    uint32_t* o = t.slots + (size_t)(off + c) * 11;
    const float xyz[3] = {p.x, p.y, p.z};
#pragma unroll
    for (int k = 0; k < 3; ++k) { const uint32_t v = f2ord(xyz[k]); atomicMin(&o[k], v); atomicMax(&o[3 + k], v); }
    atomicAdd(&o[10], 1u);
    atomicMin(&t.first[off + c], i - off);
}

// rows: finish the slot of every root; samples: cluster count and the noise marker
__global__ void __launch_bounds__(256) lb_finish_kernel(uint32_t n_threads, int n_samples, const uint32_t* __restrict__ object_sample,
                                                       const uint32_t* __restrict__ totals, const uint32_t* __restrict__ is_root,
                                                       const uint32_t* __restrict__ counts, const ClusterTable t, int32_t* __restrict__ n_clusters) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_threads) return;
    if (i < totals[2] && is_root[i]) {
        const uint32_t off = t.object_off[object_sample[i]];
        cluster_finish(t.slots + (size_t)(off + (t.rank[i] - t.rank[off])) * 11);
    }
    if (i < (uint32_t)n_samples) {
        const uint32_t off = t.object_off[i];
        n_clusters[i] = (int32_t)(t.rank[off + counts[i * 3 + 2]] - t.rank[off]);
        if (t.noise_first[i] == 0x7fffffff) t.noise_first[i] = -1;
    }
}

// ---------------------------------------------------------------- host side
// cubic cells a hair above eps (as ops.dbscan) over the box every object row lies in: |x|, |y| < range_max (the gate's
// sqrt(x^2 + y^2) < range_max), max(ground_z, z_min) <= z < z_max; coarser cells while one sample's grid would not fit 32 bits
static DbGrid lb_grid(const msc_params& P, double eps) {
    DbGrid G;
    double cell = eps * (1.0 + 1e-6);
    const double r = (double)P.range_max, zlo = (double)fmaxf(P.ground_z, P.z_min), zhi = (double)P.z_max;
    G.ox = -r; G.oy = -r; G.oz = zlo;
    for (;;) {
        auto dim = [&](double ext) { const double d = floor(fmax(ext, 0.0) / cell) + 1.0; return d < 2e9 ? d : 2e9; };
        const double nx = dim(2.0 * r), ny = dim(2.0 * r), nz = dim(zhi - zlo);
        if (nx * ny * nz < 4294967296.0 || cell > 1e30) {
            G.nx = (int)nx; G.ny = (int)ny; G.nz = (int)nz;
            break;
        }
        cell *= 2.0;  // coarser cells stay correct (cell >= eps), only slower
    }
    G.inv_cell = 1.0 / cell;
    G.ncells = (uint64_t)G.nx * G.ny * G.nz;
    return G;
}

struct LbWs {
    size_t kf_n, tile_off, block_counts, totals, object_sample;
    uint32_t n_tiles;
    DbGrid G;
    DbWs db;  // DBSCAN's buffers follow; db.end is the total
};

static cudaError_t lb_layout(const msc_params& P, double eps, int n_samples, uint32_t cap, LbWs* W) {
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    W->G = lb_grid(P, eps);
    W->n_tiles = (uint32_t)((cap + (uint64_t)kCompactThreads - 1) / kCompactThreads + (uint64_t)n_samples);
    const size_t S = (size_t)n_samples, n = cap;
    size_t o = 0;
    W->kf_n = o; o = al(o + S * 4);
    W->tile_off = o; o = al(o + (S + 1) * 4);
    W->block_counts = o; o = al(o + (size_t)W->n_tiles * 8);
    W->totals = o; o = al(o + 16);
    W->object_sample = o; o = al(o + n * 4);
    return db_layout(o, cap, n_samples, W->G, &W->db);
}

static bool lb_args_ok(const msc_params* params, double eps, int32_t n_samples, uint32_t cap) {
    return params && eps > 0.0 && n_samples >= 0 && cap < 0x7fffffffu - kCompactThreads;
}

}  // namespace msc

extern "C" {

size_t msc_lidar_batch_workspace_bytes(const msc_params* params, double eps, int32_t n_samples, uint32_t row_capacity) {
    using namespace msc;
    if (!lb_args_ok(params, eps, n_samples, row_capacity)) return 0;
    LbWs W;
    if (lb_layout(*params, eps, n_samples, row_capacity, &W) != cudaSuccess) return 0;
    return W.db.end;
}

int msc_lidar_batch(const msc_params* params, double eps, int32_t min_samples, const msc_batch_in* in, const msc_lidar_batch_out* out,
                    void* workspace, size_t workspace_bytes, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(params && in && out, "msc_lidar_batch: null argument");
    MSC_REQUIRE(eps > 0.0 && eps < 1e30, "msc_lidar_batch: eps must be > 0 (got %g)", eps);
    MSC_REQUIRE(min_samples >= 1, "msc_lidar_batch: min_samples must be >= 1 (got %d)", (int)min_samples);
    MSC_REQUIRE(in->n_samples >= 0, "msc_lidar_batch: negative n_samples");
    if (in->n_samples == 0) return MSC_OK;
    const int S = in->n_samples;
    const uint32_t cap = out->row_capacity;
    MSC_REQUIRE(lb_args_ok(params, eps, S, cap), "msc_lidar_batch: row_capacity too large (%u)", cap);
    MSC_REQUIRE(out->counts && out->ground_off && out->object_off && out->n_clusters && out->noise_first && out->status,
                "msc_lidar_batch: null per-sample output");
    MSC_REQUIRE(cap == 0 || (out->ground && out->object && out->labels && out->clusters && out->cluster_first), "msc_lidar_batch: null row output");
    MSC_REQUIRE(in->points && in->sample_sweep_off && in->sweep_start && in->sweep_count, "msc_lidar_batch: null input array");
    MSC_REQUIRE(workspace, "msc_lidar_batch: null workspace");
    LbWs W;
    MSC_CUDA(lb_layout(*params, eps, S, cap, &W));
    MSC_REQUIRE(workspace_bytes >= W.db.end, "msc_lidar_batch: workspace too small: need %zu bytes, got %zu", W.db.end, workspace_bytes);
    cudaStream_t stream = (cudaStream_t)stream_v;
    unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
    uint32_t* kf_n = (uint32_t*)(ws + W.kf_n); uint32_t* tile_off = (uint32_t*)(ws + W.tile_off);
    uint32_t* block_counts = (uint32_t*)(ws + W.block_counts); uint32_t* totals = (uint32_t*)(ws + W.totals);
    uint32_t* object_sample = (uint32_t*)(ws + W.object_sample);
    const uint32_t* is_root = (const uint32_t*)(ws + W.db.is_root); const uint32_t* rank = (const uint32_t*)(ws + W.db.rank);
    const float4* object = reinterpret_cast<const float4*>(out->object);

    // 1. filter / split
    lb_plan_kernel<<<1, 256, 0, stream>>>(S, in->sample_sweep_off, in->sweep_count, cap, kf_n, tile_off, out->noise_first, out->status);
    lb_count_kernel<<<W.n_tiles, kCompactThreads, 0, stream>>>(*params, in->points, in->sample_sweep_off, in->sweep_start, kf_n, tile_off, S,
                                                               block_counts);
    kf_scan_kernel<<<1, 1024, 0, stream>>>(block_counts, W.n_tiles, totals);
    lb_offsets_kernel<<<(S + 255) / 256, 256, 0, stream>>>(S, tile_off, block_counts, W.n_tiles, totals, out->counts, out->ground_off,
                                                           out->object_off);
    lb_scatter_kernel<<<W.n_tiles, kCompactThreads, 0, stream>>>(*params, in->points, in->sample_sweep_off, in->sweep_start, kf_n, tile_off, S,
                                                                 block_counts, reinterpret_cast<float4*>(out->ground),
                                                                 reinterpret_cast<float4*>(out->object), object_sample);
    MSC_CUDA(cudaGetLastError());

    // 2. DBSCAN over every sample's object rows
    const ClusterTable t{out->object_off, rank, reinterpret_cast<uint32_t*>(out->clusters), reinterpret_cast<uint32_t*>(out->cluster_first), out->labels, out->noise_first};
    MSC_CUDA(db_enqueue(W.db, ws, W.G, object, object_sample, totals, eps, (uint32_t)min_samples, t, out->status, stream));

    // 3. cluster table
    const unsigned nb256 = (cap + 255) / 256 + 1;
    lb_minmax_kernel<<<nb256, 256, 0, stream>>>(object, object_sample, totals, t);
    const uint32_t n_fin = cap > (uint32_t)S ? cap : (uint32_t)S;
    lb_finish_kernel<<<(n_fin + 255) / 256, 256, 0, stream>>>(n_fin, S, object_sample, totals, is_root, out->counts, t, out->n_clusters);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

}  // extern "C"
