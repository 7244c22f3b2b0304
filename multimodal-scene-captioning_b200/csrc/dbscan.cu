// dbscan.cu -- DBSCAN with the labelling of scikit-learn's implementation, on the device
// (reference call site: LiDARAgent._detect_objects_3d, lidar_agent.py:148-153; SURVEY.md section 8(f) rank 2).
//
// scikit-learn's result is a deterministic function of the neighbour relation:
//   * neighbours: sum_k (a_k - b_k)^2 <= eps^2 in float64, accumulated x -> y -> z (KDTree reduced distance);
//   * core points have >= min_samples neighbours (the point itself included);
//   * clusters are the connected components of core points, numbered by their smallest core index (the outer loop of
//     dbscan_inner visits points in index order and fully expands one cluster before starting the next);
//   * a non-core point adjacent to core points takes the smallest of their cluster numbers (the first cluster that
//     reaches it keeps it); otherwise it is noise (-1).
// Everything is float64 with -fmad=false, so the neighbour relation -- and therefore every label -- is identical to scikit-learn's
// whenever scikit-learn uses a tree (n >= 12 points).  For n <= 11 scikit-learn brute-forces the neighbour search with a BLAS
// expansion |a|^2 - 2ab + |b|^2 that can drop a pair at exactly eps; this file keeps the rule above there too, so labels can differ
// from scikit-learn's only through such pairs.
//
// One pipeline (db_enqueue) serves msc_lidar_batch, over the object rows of all samples of a batch at once, and msc_dbscan, as a
// batch of one sample: 64-bit keys (sample, cell) over cells at least eps wide, sorted with CUB, cells found by binary search, so memory
// is O(rows) whatever the number of samples or cells; one hooking sweep, one verify sweep, flatten, an exclusive scan of the root flags
// (per-sample numbering = global rank minus the rank at the sample's first row), labelling.
#include "lidar_common.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

namespace msc {

// neighbour relation: squared distance in float64, accumulated x -> y -> z (scikit-learn's KD-tree reduced distance)
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
// thread goes on to merge old's tree with lo's, so the edge it cut is restored before it returns.
__device__ __forceinline__ void db_union(uint32_t* parent, uint32_t i, uint32_t j) {
    uint32_t a = db_find(parent, i), b = db_find(parent, j);
    while (a != b) {
        const uint32_t hi = max(a, b), lo = min(a, b);
        const uint32_t old = atomicMin(&parent[hi], lo);
        if (old == hi) break;   // hi was a root and now hangs under lo
        a = db_find(parent, old);  // hi already had a smaller parent: merge that tree with lo
        b = db_find(parent, lo);
    }
}

__device__ __forceinline__ void db_cell(const DbGrid& G, float4 p, int* cx, int* cy, int* cz) {
    *cx = min(max((int)floor(((double)p.x - G.ox) * G.inv_cell), 0), G.nx - 1);
    *cy = min(max((int)floor(((double)p.y - G.oy) * G.inv_cell), 0), G.ny - 1);
    *cz = min(max((int)floor(((double)p.z - G.oz) * G.inv_cell), 0), G.nz - 1);
}

// key of every object row (rows past the batch's object count get the largest key, so they sort last)
__global__ void __launch_bounds__(256) db_key_kernel(const float4* __restrict__ object, const uint32_t* __restrict__ object_sample,
                                                    const uint32_t* __restrict__ totals, uint32_t cap, DbGrid G, uint64_t pad_key,
                                                    uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cap) return;
    uint64_t k = pad_key;
    if (i < totals[2]) {
        int cx, cy, cz;
        db_cell(G, object[i], &cx, &cy, &cz);
        k = (uint64_t)object_sample[i] * G.ncells + ((uint64_t)cz * G.ny + cy) * G.nx + cx;
    }
    keys[i] = k;
    vals[i] = i;
}

// visit every neighbour j of object row i (same sample, squared distance <= eps2 in float64, x -> y -> z) and call f(j).  The three
// cells along x of one (z, y) row are consecutive keys: one binary search per row, nine per point.
template <class F>
__device__ __forceinline__ void db_for_each_neighbour(const float4* __restrict__ object, const DbGrid& G, double eps2, uint32_t s,
                                                      const uint64_t* __restrict__ skey, const uint32_t* __restrict__ sidx, uint32_t m,
                                                      uint32_t i, F f) {
    const float4 p = object[i];
    const double px = (double)p.x, py = (double)p.y, pz = (double)p.z;
    int cx, cy, cz;
    db_cell(G, p, &cx, &cy, &cz);
    const uint64_t base = (uint64_t)s * G.ncells;
    for (int z = max(cz - 1, 0); z <= min(cz + 1, G.nz - 1); ++z)
        for (int y = max(cy - 1, 0); y <= min(cy + 1, G.ny - 1); ++y) {
            const uint64_t row = base + ((uint64_t)z * G.ny + y) * G.nx;
            const uint64_t k0 = row + max(cx - 1, 0), k1 = row + min(cx + 1, G.nx - 1);
            uint32_t lo = 0, hi = m;
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (skey[mid] < k0) lo = mid + 1; else hi = mid;
            }
            for (uint32_t k = lo; k < m && skey[k] <= k1; ++k) {
                const uint32_t j = sidx[k];
                if (db_dist2(px, py, pz, &object[j].x) <= eps2) f(j);
            }
        }
}

// the four neighbour-search kernels are declared with a minimum of 8 blocks per SM (<= 64 registers): without it ptxas picks 32
// registers for the hook and label kernels and spills
struct DbArgs {
    const float4* object;
    const uint32_t* object_sample;
    const uint32_t* totals;  // [2] = object rows of the batch
    const uint64_t* skey;
    const uint32_t* sidx;
    DbGrid G;
    double eps2;
};

__global__ void __launch_bounds__(128, 8) db_core_kernel(const DbArgs a, uint32_t min_samples, uint8_t* __restrict__ core, uint32_t* __restrict__ parent) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t m = a.totals[2];
    if (i >= m) return;
    uint32_t cnt = 0;
    db_for_each_neighbour(a.object, a.G, a.eps2, a.object_sample[i], a.skey, a.sidx, m, i, [&](uint32_t) { ++cnt; });
    core[i] = cnt >= min_samples ? 1 : 0;
    parent[i] = i;
}

// the one hooking sweep: every thread completes the union of each of its edges before it moves on (DESIGN.md section 4.5)
__global__ void __launch_bounds__(128, 8) db_hook_kernel(const DbArgs a, const uint8_t* __restrict__ core, uint32_t* __restrict__ parent) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t m = a.totals[2];
    if (i >= m || !core[i]) return;
    db_for_each_neighbour(a.object, a.G, a.eps2, a.object_sample[i], a.skey, a.sidx, m, i, [=](uint32_t j) {
        if (j < i && core[j]) db_union(parent, i, j);
    });
}

// the verify sweep over the same edges: two endpoints with different roots set kDbUnmerged, never a silently under-merged labelling
__global__ void __launch_bounds__(128, 8) db_verify_kernel(const DbArgs a, const uint8_t* __restrict__ core, const uint32_t* __restrict__ parent,
                                                       uint32_t* __restrict__ status) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t m = a.totals[2];
    if (i >= m || !core[i]) return;
    const uint32_t ri = db_find(parent, i);
    bool bad = false;
    db_for_each_neighbour(a.object, a.G, a.eps2, a.object_sample[i], a.skey, a.sidx, m, i, [=, &bad](uint32_t j) {
        if (j < i && core[j] && db_find(parent, j) != ri) bad = true;
    });
    if (bad) atomicOr(status, kDbUnmerged);
}

// parent -> root for core rows; is_root has cap + 1 entries (zero past the object rows) so its exclusive scan also gives the totals
__global__ void __launch_bounds__(256) db_flatten_kernel(uint32_t cap, const uint32_t* __restrict__ totals, const uint8_t* __restrict__ core,
                                                        uint32_t* __restrict__ parent, uint32_t* __restrict__ is_root) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > cap) return;
    uint32_t root = 0;
    if (i < totals[2] && core[i]) {
        const uint32_t r = db_find(parent, i);
        parent[i] = r;  // roots keep pointing at themselves, so concurrent finds stay valid
        root = r == i;
    }
    is_root[i] = root;
}

// labels numbered per sample (the smallest core index of a component is its root; roots in row order give scikit-learn's numbering);
// a border row takes the smallest adjacent cluster number.  The root of cluster k initialises the k-th slot of its sample.
__global__ void __launch_bounds__(128, 8) db_label_kernel(const DbArgs a, const uint8_t* __restrict__ core, const uint32_t* __restrict__ parent,
                                                      const ClusterTable t) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t m = a.totals[2];
    if (i >= m) return;
    const uint32_t s = a.object_sample[i], off = t.object_off[s], base = t.rank[off];
    if (core[i]) {
        const uint32_t r = parent[i], k = t.rank[r] - base;
        t.labels[i] = (int32_t)k;
        if (r == i) {
            uint32_t* o = t.slots + (size_t)(off + k) * 11;
#pragma unroll
            for (int w = 0; w < 11; ++w) o[w] = (w < 3) ? 0xffffffffu : 0u;
            t.first[off + k] = 0xffffffffu;
        }
        return;
    }
    uint32_t best = 0xffffffffu;
    db_for_each_neighbour(a.object, a.G, a.eps2, s, a.skey, a.sidx, m, i, [=, &best](uint32_t j) {
        if (core[j]) best = min(best, t.rank[parent[j]]);
    });
    if (best == 0xffffffffu) {
        t.labels[i] = -1;
        atomicMin(&t.noise_first[s], (int32_t)(i - off));
    } else {
        t.labels[i] = (int32_t)(best - base);
    }
}

// ---------------------------------------------------------------- host side
static size_t al256(size_t v) { return (v + 255) & ~(size_t)255; }

static int db_bits(uint64_t v) {  // bits needed to hold v
    int b = 0;
    while (b < 64 && (v >> b) != 0) ++b;
    return b;
}

cudaError_t db_layout(size_t base, uint32_t cap, int n_samples, const DbGrid& G, DbWs* W) {
    W->cap = cap;
    W->pad_key = (uint64_t)n_samples * G.ncells;
    W->end_bit = db_bits(W->pad_key);  // the largest key, S * ncells, pads the sort
    const size_t n = cap;
    size_t o = base;
    W->keys_in = o; o = al256(o + n * 8);
    W->keys_out = o; o = al256(o + n * 8);
    W->vals_in = o; o = al256(o + n * 4);
    W->sidx = o; o = al256(o + n * 4);
    W->core = o; o = al256(o + n);
    W->parent = o; o = al256(o + n * 4);
    W->is_root = o; o = al256(o + (n + 1) * 4);
    W->rank = o; o = al256(o + (n + 1) * 4);
    size_t sort_bytes = 0, scan_bytes = 0;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const uint32_t*)nullptr,
                                                    (uint32_t*)nullptr, (int)n, 0, W->end_bit);
    if (e != cudaSuccess) return e;
    e = cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)n + 1);
    if (e != cudaSuccess) return e;
    W->temp = o;
    W->temp_bytes = al256(sort_bytes > scan_bytes ? sort_bytes : scan_bytes);
    W->end = al256(o + W->temp_bytes);
    return cudaSuccess;
}

cudaError_t db_enqueue(const DbWs& W, unsigned char* ws, const DbGrid& G, const float4* object, const uint32_t* object_sample,
                       const uint32_t* totals, double eps, uint32_t min_samples, const ClusterTable& t, uint32_t* status,
                       cudaStream_t stream) {
    uint64_t* keys_in = (uint64_t*)(ws + W.keys_in); uint64_t* keys_out = (uint64_t*)(ws + W.keys_out);
    uint32_t* vals_in = (uint32_t*)(ws + W.vals_in); uint32_t* sidx = (uint32_t*)(ws + W.sidx);
    uint8_t* core = (uint8_t*)(ws + W.core); uint32_t* parent = (uint32_t*)(ws + W.parent);
    uint32_t* is_root = (uint32_t*)(ws + W.is_root); uint32_t* rank = (uint32_t*)(ws + W.rank);
    void* temp = ws + W.temp;
    const uint32_t cap = W.cap;
    const unsigned nb256 = (cap + 255) / 256 + 1, nb128 = (cap + 127) / 128 + 1;
    db_key_kernel<<<nb256, 256, 0, stream>>>(object, object_sample, totals, cap, G, W.pad_key, keys_in, vals_in);
    size_t temp_bytes = W.temp_bytes;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys_in, keys_out, vals_in, sidx, (int)cap, 0, W.end_bit, stream);
    if (e != cudaSuccess) return e;
    const DbArgs a{object, object_sample, totals, keys_out, sidx, G, eps * eps};
    db_core_kernel<<<nb128, 128, 0, stream>>>(a, min_samples, core, parent);
    db_hook_kernel<<<nb128, 128, 0, stream>>>(a, core, parent);
    db_verify_kernel<<<nb128, 128, 0, stream>>>(a, core, parent, status);
    db_flatten_kernel<<<nb256, 256, 0, stream>>>(cap, totals, core, parent, is_root);
    temp_bytes = W.temp_bytes;
    e = cub::DeviceScan::ExclusiveSum(temp, temp_bytes, is_root, rank, (int)cap + 1, stream);
    if (e != cudaSuccess) return e;
    db_label_kernel<<<nb128, 128, 0, stream>>>(a, core, parent, t);
    return cudaGetLastError();
}

// ---------------------------------------------------------------- msc_dbscan: the pipeline on one sample
// the per-sample words of the one sample
struct DbSample {
    uint32_t totals[3];  // [2] = rows
    uint32_t object_off;
    int32_t noise_first;
    uint32_t status;
};

// the caller's rows (any pitch >= 3) as float4 rows of sample 0, and the sample's words
__global__ void __launch_bounds__(256) db_prep_kernel(const float* __restrict__ pts, uint32_t n, int pitch, float4* __restrict__ rows,
                                                     uint32_t* __restrict__ sample, DbSample* __restrict__ one) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *one = DbSample{{0u, 0u, n}, 0u, 0x7fffffff, 0u};
    if (i >= n) return;
    const float* p = pts + (size_t)i * pitch;
    rows[i] = make_float4(p[0], p[1], p[2], 0.0f);
    sample[i] = 0u;
}

// rows, sample ids, the sample's words, cluster-table scratch the label kernel writes (slots [n, 11], first [n]), then DBSCAN's buffers
struct DbSampleWs {
    size_t rows, sample, one, slots, first;
    DbWs db;
};

static cudaError_t db_sample_layout(uint32_t n, const DbGrid& G, DbSampleWs* W) {
    size_t o = 0;
    W->rows = o; o = al256(o + (size_t)n * 16);
    W->sample = o; o = al256(o + (size_t)n * 4);
    W->one = o; o = al256(o + sizeof(DbSample));
    W->slots = o; o = al256(o + (size_t)n * 44);
    W->first = o; o = al256(o + (size_t)n * 4);
    return db_layout(o, n, 1, G, &W->db);
}

}  // namespace msc

extern "C" {

size_t msc_dbscan_workspace_bytes(uint32_t n, const int32_t dims[3]) {
    using namespace msc;
    if (!dims || n >= 0x7fffffffu) return 0;
    DbGrid G{};
    G.ncells = (uint64_t)dims[0] * dims[1] * dims[2];
    DbSampleWs W;
    return db_sample_layout(n, G, &W) == cudaSuccess ? W.db.end : 0;
}

// Synchronous on `stream`: one copy of the cluster count and the status word at the end.
int msc_dbscan(const float* pts, uint32_t n, int32_t pitch, double eps, int32_t min_samples, const double origin[3], double cell,
               const int32_t dims[3], int32_t* labels, int32_t* n_clusters_host, void* workspace, size_t workspace_bytes, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(origin && dims && (n == 0 || (pts && labels)) && workspace, "null argument");
    MSC_REQUIRE(pitch >= 3 && eps > 0.0 && cell >= eps && min_samples >= 1, "bad parameters (cell must be >= eps)");
    MSC_REQUIRE(dims[0] > 0 && dims[1] > 0 && dims[2] > 0, "bad grid dims");
    // CUB's item counts are int, and its scan covers n + 1 items
    MSC_REQUIRE(n < 0x7fffffffu, "msc_dbscan: too many points (%u)", n);
    const size_t ncells = (size_t)dims[0] * dims[1] * dims[2];
    MSC_REQUIRE(ncells < ((size_t)1 << 31), "grid too large");
    const DbGrid G{origin[0], origin[1], origin[2], 1.0 / cell, dims[0], dims[1], dims[2], ncells};
    DbSampleWs W;
    MSC_CUDA(db_sample_layout(n, G, &W));
    MSC_REQUIRE(workspace_bytes >= W.db.end, "workspace too small: need %zu bytes", W.db.end);
    if (n_clusters_host) *n_clusters_host = 0;
    if (n == 0) return MSC_OK;
    cudaStream_t stream = (cudaStream_t)stream_v;
    unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
    float4* rows = (float4*)(ws + W.rows);
    uint32_t* sample = (uint32_t*)(ws + W.sample);
    DbSample* one = (DbSample*)(ws + W.one);
    db_prep_kernel<<<(n + 255) / 256, 256, 0, stream>>>(pts, n, pitch, rows, sample, one);
    const ClusterTable t{&one->object_off, (const uint32_t*)(ws + W.db.rank), (uint32_t*)(ws + W.slots), (uint32_t*)(ws + W.first), labels,
                         &one->noise_first};
    MSC_CUDA(db_enqueue(W.db, ws, G, rows, sample, one->totals, eps, (uint32_t)min_samples, t, &one->status, stream));
    uint32_t k = 0, status = 0;
    MSC_CUDA(cudaMemcpyAsync(&k, t.rank + n, 4, cudaMemcpyDeviceToHost, stream));
    MSC_CUDA(cudaMemcpyAsync(&status, &one->status, 4, cudaMemcpyDeviceToHost, stream));
    MSC_CUDA(cudaStreamSynchronize(stream));
    if (status & kDbUnmerged) {
        set_error("msc_dbscan: the component merge left an edge unmerged");
        return MSC_ERR_LAUNCH;
    }
    if (n_clusters_host) *n_clusters_host = (int32_t)k;
    return MSC_OK;
}

}  // extern "C"
