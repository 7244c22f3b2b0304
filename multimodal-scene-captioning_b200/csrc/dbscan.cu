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
// The device version: counting sort of the points into a grid of cells slightly larger than eps, neighbour counts over the
// 27 surrounding cells, atomic-min union-find over core-core edges (the root of a component is its smallest index), rank of
// the roots by an exclusive scan, and a final labelling pass.  Everything is float64 with -fmad=false, so the neighbour
// relation -- and therefore every label -- is identical to scikit-learn's whenever scikit-learn uses a tree (n >= 12 points).
// For n <= 11 scikit-learn brute-forces the neighbour search with a BLAS expansion |a|^2 - 2ab + |b|^2 that can drop a pair at
// exactly eps; this file keeps the rule above there too, so labels can differ from scikit-learn's only through such pairs.
#include "msc_common.cuh"

namespace msc {

struct DbscanGrid {
    double ox, oy, oz, inv_cell;
    int nx, ny, nz;
};

__device__ __forceinline__ void point_cell(const DbscanGrid& G, const float* p, int* cx, int* cy, int* cz) {
    *cx = min(max((int)floor(((double)p[0] - G.ox) * G.inv_cell), 0), G.nx - 1);
    *cy = min(max((int)floor(((double)p[1] - G.oy) * G.inv_cell), 0), G.ny - 1);
    *cz = min(max((int)floor(((double)p[2] - G.oz) * G.inv_cell), 0), G.nz - 1);
}

__global__ void __launch_bounds__(256) db_count_kernel(const float* __restrict__ pts, uint32_t n, int pitch, DbscanGrid G, uint32_t* __restrict__ cell_of,
                                                      uint32_t* __restrict__ cell_count) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int cx, cy, cz;
    point_cell(G, pts + (size_t)i * pitch, &cx, &cy, &cz);
    const uint32_t c = ((uint32_t)cz * G.ny + cy) * G.nx + cx;
    cell_of[i] = c;
    atomicAdd(&cell_count[c], 1u);
}

// single-block exclusive scan of `n` u32 (n up to a few million); total to out_total
__global__ void __launch_bounds__(1024) db_scan_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t n, uint32_t* __restrict__ out_total) {
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = (i < n) ? in[i] : 0u;
        uint32_t x = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += y; }
        if (lane == 31) s_warp[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = s_warp[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, w, d); if (lane >= d) w += y; }
            s_warp[lane] = w;
        }
        __syncthreads();
        const uint32_t excl = s_carry + (warp ? s_warp[warp - 1] : 0u) + x - v;
        if (i < n) out[i] = excl;
        __syncthreads();
        if (threadIdx.x == 0) s_carry += s_warp[31];
        __syncthreads();
    }
    if (threadIdx.x == 0 && out_total) *out_total = s_carry;
}

__global__ void __launch_bounds__(256) db_scatter_kernel(uint32_t n, const uint32_t* __restrict__ cell_of, const uint32_t* __restrict__ cell_start,
                                                        uint32_t* __restrict__ cursor, uint32_t* __restrict__ sorted) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t c = cell_of[i];
    sorted[cell_start[c] + atomicAdd(&cursor[c], 1u)] = i;
}

// visit every neighbour j of point i (squared distance <= eps2 in float64, x -> y -> z) and call f(j)
template <class F>
__device__ __forceinline__ void for_each_neighbour(const float* __restrict__ pts, int pitch, const DbscanGrid& G, double eps2,
                                                   const uint32_t* __restrict__ cell_start, const uint32_t* __restrict__ cell_count,
                                                   const uint32_t* __restrict__ sorted, uint32_t i, F f) {
    const float* p = pts + (size_t)i * pitch;
    const double px = (double)p[0], py = (double)p[1], pz = (double)p[2];
    int cx, cy, cz;
    point_cell(G, p, &cx, &cy, &cz);
    for (int z = max(cz - 1, 0); z <= min(cz + 1, G.nz - 1); ++z)
        for (int y = max(cy - 1, 0); y <= min(cy + 1, G.ny - 1); ++y)
            for (int x = max(cx - 1, 0); x <= min(cx + 1, G.nx - 1); ++x) {
                const uint32_t c = ((uint32_t)z * G.ny + y) * G.nx + x;
                const uint32_t b = cell_start[c], e = b + cell_count[c];
                for (uint32_t k = b; k < e; ++k) {
                    const uint32_t j = sorted[k];
                    const float* q = pts + (size_t)j * pitch;
                    const double dx = px - (double)q[0], dy = py - (double)q[1], dz = pz - (double)q[2];
                    double d = dx * dx;
                    d = d + dy * dy;
                    d = d + dz * dz;
                    if (d <= eps2) f(j);
                }
            }
}

__global__ void __launch_bounds__(128) db_core_kernel(const float* __restrict__ pts, uint32_t n, int pitch, DbscanGrid G, double eps2, uint32_t min_samples,
                                                     const uint32_t* __restrict__ cell_start, const uint32_t* __restrict__ cell_count,
                                                     const uint32_t* __restrict__ sorted, uint8_t* __restrict__ core, uint32_t* __restrict__ parent) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t cnt = 0;
    for_each_neighbour(pts, pitch, G, eps2, cell_start, cell_count, sorted, i, [&](uint32_t) { ++cnt; });
    core[i] = cnt >= min_samples ? 1 : 0;
    parent[i] = i;
}

__device__ __forceinline__ uint32_t db_find(const uint32_t* parent, uint32_t a) {
    uint32_t p = ((const volatile uint32_t*)parent)[a];
    while (p != a) { a = p; p = ((const volatile uint32_t*)parent)[a]; }
    return a;
}

// one round of hooking over core-core edges: the larger root is hung under the smaller one (atomicMin), so a component's
// root converges to its smallest index.  *changed is set when any hook happened.
__global__ void __launch_bounds__(128) db_hook_kernel(const float* __restrict__ pts, uint32_t n, int pitch, DbscanGrid G, double eps2,
                                                     const uint32_t* __restrict__ cell_start, const uint32_t* __restrict__ cell_count,
                                                     const uint32_t* __restrict__ sorted, const uint8_t* __restrict__ core, uint32_t* __restrict__ parent,
                                                     uint32_t* __restrict__ changed) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !core[i]) return;
    for_each_neighbour(pts, pitch, G, eps2, cell_start, cell_count, sorted, i, [&](uint32_t j) {
        if (j >= i || !core[j]) return;
        uint32_t a = db_find(parent, i), b = db_find(parent, j);
        while (a != b) {
            const uint32_t hi = max(a, b), lo = min(a, b);
            const uint32_t old = atomicMin(&parent[hi], lo);
            *changed = 1u;
            if (old == hi) break;   // hi was a root and now hangs under lo
            a = db_find(parent, old);  // hi already had a smaller parent: merge that tree with lo
            b = db_find(parent, lo);
        }
    });
}

__global__ void __launch_bounds__(256) db_flatten_kernel(uint32_t n, const uint8_t* __restrict__ core, uint32_t* __restrict__ parent, uint32_t* __restrict__ is_root) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t r = i;
    if (core[i]) { r = db_find(parent, i); }
    is_root[i] = (core[i] && r == i) ? 1u : 0u;
    if (core[i]) parent[i] = r;  // roots keep pointing at themselves, so concurrent finds stay valid
}

__global__ void __launch_bounds__(128) db_label_kernel(const float* __restrict__ pts, uint32_t n, int pitch, DbscanGrid G, double eps2,
                                                      const uint32_t* __restrict__ cell_start, const uint32_t* __restrict__ cell_count,
                                                      const uint32_t* __restrict__ sorted, const uint8_t* __restrict__ core, const uint32_t* __restrict__ parent,
                                                      const uint32_t* __restrict__ root_rank, int32_t* __restrict__ labels) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (core[i]) { labels[i] = (int32_t)root_rank[parent[i]]; return; }
    uint32_t best = 0xffffffffu;
    for_each_neighbour(pts, pitch, G, eps2, cell_start, cell_count, sorted, i, [&](uint32_t j) {
        if (core[j]) best = min(best, root_rank[parent[j]]);
    });
    labels[i] = (best == 0xffffffffu) ? -1 : (int32_t)best;
}

struct DbscanWs {
    size_t cell_count, cell_start, cursor, cell_of, sorted, parent, is_root, root_rank, core, flag, total;
};
static DbscanWs db_layout(uint32_t n, size_t ncells) {
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    DbscanWs W;
    size_t o = 0;
    W.cell_count = o; o = al(o + ncells * 4);
    W.cell_start = o; o = al(o + ncells * 4);
    W.cursor = o; o = al(o + ncells * 4);
    W.cell_of = o; o = al(o + (size_t)n * 4);
    W.sorted = o; o = al(o + (size_t)n * 4);
    W.parent = o; o = al(o + (size_t)n * 4);
    W.is_root = o; o = al(o + (size_t)n * 4);
    W.root_rank = o; o = al(o + (size_t)n * 4);
    W.core = o; o = al(o + (size_t)n);
    W.flag = o; o = al(o + 256);
    W.total = o;
    return W;
}

}  // namespace msc

extern "C" {

size_t msc_dbscan_workspace_bytes(uint32_t n, const int32_t dims[3]) {
    if (!dims) return 0;
    return msc::db_layout(n, (size_t)dims[0] * dims[1] * dims[2]).total;
}

// Synchronous on `stream` (the component merge iterates until a device flag stays clear).
int msc_dbscan(const float* pts, uint32_t n, int32_t pitch, double eps, int32_t min_samples, const double origin[3], double cell,
               const int32_t dims[3], int32_t* labels, int32_t* n_clusters_host, void* workspace, size_t workspace_bytes, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(origin && dims && (n == 0 || (pts && labels)) && workspace, "null argument");
    MSC_REQUIRE(pitch >= 3 && eps > 0.0 && cell >= eps && min_samples >= 1, "bad parameters (cell must be >= eps)");
    MSC_REQUIRE(dims[0] > 0 && dims[1] > 0 && dims[2] > 0, "bad grid dims");
    const size_t ncells = (size_t)dims[0] * dims[1] * dims[2];
    MSC_REQUIRE(ncells < ((size_t)1 << 31), "grid too large");
    const DbscanWs W = db_layout(n, ncells);
    MSC_REQUIRE(workspace_bytes >= W.total, "workspace too small: need %zu bytes", W.total);
    if (n_clusters_host) *n_clusters_host = 0;
    if (n == 0) return MSC_OK;
    cudaStream_t stream = (cudaStream_t)stream_v;
    unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
    uint32_t* cell_count = (uint32_t*)(ws + W.cell_count); uint32_t* cell_start = (uint32_t*)(ws + W.cell_start);
    uint32_t* cursor = (uint32_t*)(ws + W.cursor); uint32_t* cell_of = (uint32_t*)(ws + W.cell_of); uint32_t* sorted = (uint32_t*)(ws + W.sorted);
    uint32_t* parent = (uint32_t*)(ws + W.parent); uint32_t* is_root = (uint32_t*)(ws + W.is_root); uint32_t* root_rank = (uint32_t*)(ws + W.root_rank);
    uint8_t* core = (uint8_t*)(ws + W.core); uint32_t* flag = (uint32_t*)(ws + W.flag);
    DbscanGrid G{origin[0], origin[1], origin[2], 1.0 / cell, dims[0], dims[1], dims[2]};
    const double eps2 = eps * eps;
    const unsigned nb256 = (n + 255) / 256, nb128 = (n + 127) / 128;
    MSC_CUDA(cudaMemsetAsync(cell_count, 0, ncells * 4, stream));
    MSC_CUDA(cudaMemsetAsync(cursor, 0, ncells * 4, stream));
    db_count_kernel<<<nb256, 256, 0, stream>>>(pts, n, pitch, G, cell_of, cell_count);
    db_scan_kernel<<<1, 1024, 0, stream>>>(cell_count, cell_start, (uint32_t)ncells, nullptr);
    db_scatter_kernel<<<nb256, 256, 0, stream>>>(n, cell_of, cell_start, cursor, sorted);
    db_core_kernel<<<nb128, 128, 0, stream>>>(pts, n, pitch, G, eps2, (uint32_t)min_samples, cell_start, cell_count, sorted, core, parent);
    // atomic-min hooking converges in O(log n) sweeps in practice; a chain of n core points bounds it by n, so the cap grows with n and a
    // flag that is still set after it is an error, never a silently under-merged labelling
    const int max_sweeps = 64 + (int)(n / 1024 < 4096 ? n / 1024 : 4096);
    bool merged = false;
    for (int it = 0; it < max_sweeps && !merged; ++it) {
        MSC_CUDA(cudaMemsetAsync(flag, 0, 4, stream));
        db_hook_kernel<<<nb128, 128, 0, stream>>>(pts, n, pitch, G, eps2, cell_start, cell_count, sorted, core, parent, flag);
        uint32_t h = 0;
        MSC_CUDA(cudaMemcpyAsync(&h, flag, 4, cudaMemcpyDeviceToHost, stream));
        MSC_CUDA(cudaStreamSynchronize(stream));
        merged = h == 0;
    }
    if (!merged) {
        set_error("msc_dbscan: component merge did not converge in %d sweeps", max_sweeps);
        return MSC_ERR_LAUNCH;
    }
    db_flatten_kernel<<<nb256, 256, 0, stream>>>(n, core, parent, is_root);
    db_scan_kernel<<<1, 1024, 0, stream>>>(is_root, root_rank, n, flag + 1);
    db_label_kernel<<<nb128, 128, 0, stream>>>(pts, n, pitch, G, eps2, cell_start, cell_count, sorted, core, parent, root_rank, labels);
    uint32_t k = 0;
    MSC_CUDA(cudaMemcpyAsync(&k, flag + 1, 4, cudaMemcpyDeviceToHost, stream));
    MSC_CUDA(cudaStreamSynchronize(stream));
    MSC_CUDA(cudaGetLastError());
    if (n_clusters_host) *n_clusters_host = (int32_t)k;
    return MSC_OK;
}

}  // extern "C"
