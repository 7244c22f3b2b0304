// cluster_match.cu -- [EXT] which annotated box each LiDAR cluster lies in, for every sample of an msc_lidar_batch result in one
// stream-ordered pass.  Definition: include/msc_geom.h msc_cluster_match_batch; DESIGN.md section 4.8.
//
// Three launches:
//   cm_prep_kernel    prepared boxes (the record of fused_tables_kernel, box_record) into the workspace, accumulators zeroed;
//                     block 0 also scans the work items per sample, one per (tile of kCmBoxTile boxes) x (tile of kCmLabelTile labels);
//   cm_count_kernel   a persistent grid takes work items from a counter.  An item stages its boxes in shared memory, reads the sample's
//                     object rows and tests every row whose label is in its tile (noise rows: label tile 0 only) against every box of
//                     the tile (box_contains, the exact A.2 test), counting (box, label) hits in shared memory.  It then reduces its
//                     counters into per-box totals and 64-bit (count, ~index) argmax keys, and per-label argmax keys, with global
//                     atomics.  A row's first hit anywhere (an atomic exchange on a per-row flag) counts it once for in_any_box;
//   cm_finish_kernel  decodes the keys into the cluster and box tables.
// Every reduction is an integer sum or maximum, so the results do not depend on the grid, the tiling or the row order.
#include <algorithm>

#include "fused_common.cuh"

#include <cub/block/block_scan.cuh>

namespace msc {

constexpr int kCmThreads = 256;
constexpr int kCmBoxTile = 128;                 // boxes per work item
constexpr int kCmLabelTile = 64;                // labels per work item
constexpr int kCmCols = kCmLabelTile + 1;       // counter columns per box: noise, then the tile's labels (odd: conflict-free box rows)
constexpr int kCmCtasPerSm = 4;

struct CmArgs {
    int n_samples, n_boxes;
    uint32_t cap;
    const int32_t* sample_box_off;
    const double* boxes;
    const double* ego_pose;
    const double* lidar_calib;
    const float4* object;
    const int32_t* labels;
    const uint32_t* object_off;
    const uint32_t* counts;
    const int32_t* n_clusters;
    // workspace
    uint32_t* work_off;            // [S + 1] first work item of each sample; [S] = total
    uint32_t* work_next;           // [1] work counter
    float* boxp;                   // [n_boxes, kBoxStride]
    uint32_t* box_acc;             // [n_boxes, 3] rows, cluster_rows, clusters
    unsigned long long* box_key;   // [n_boxes] (points << 32) | ~label
    uint32_t* row_hit;             // [cap] the row lies in some box (set once)
    unsigned long long* cl_key;    // [cap] (points << 32) | ~box
    uint32_t* cl_any;              // [cap] rows of the cluster inside some box
    int32_t* out_cluster;
    int32_t* out_box;
};

// clusters of sample s as the kernels use them: within [0, object rows]
__device__ __forceinline__ int cm_clusters(const CmArgs& a, int s) {
    return min(max(a.n_clusters[s], 0), (int)a.counts[s * 3 + 2]);
}

__device__ __forceinline__ uint32_t cm_items(const CmArgs& a, int s) {
    const int nb = a.sample_box_off[s + 1] - a.sample_box_off[s];
    if (nb <= 0) return 0u;
    const int k = cm_clusters(a, s);
    return (uint32_t)((nb + kCmBoxTile - 1) / kCmBoxTile) * (uint32_t)max((k + kCmLabelTile - 1) / kCmLabelTile, 1);
}

// the last s in [0, n) with off[s] <= v (off non-decreasing, off[0] <= v)
template <typename T>
__device__ __forceinline__ int cm_last_le(const T* __restrict__ off, int n, T v) {
    int lo = 0, hi = n;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (off[mid] <= v) lo = mid; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(kCmThreads) cm_prep_kernel(const CmArgs a) {
    const size_t gid = (size_t)blockIdx.x * kCmThreads + threadIdx.x, nthreads = (size_t)gridDim.x * kCmThreads;
    for (size_t b = gid; b < (size_t)a.n_boxes; b += nthreads) {
        const int s = cm_last_le(a.sample_box_off, a.n_samples, (int32_t)b);
        const double* box = a.boxes + b * 10;
        double c[3] = {box[0], box[1], box[2]};
        double R[9];
        quat_to_rot(box + 6, R);
        frame_change(a.ego_pose + (size_t)s * 7, c, R);
        frame_change(a.lidar_calib + (size_t)s * 7, c, R);
        box_record(box, c, R, a.boxp + b * kBoxStride);
        a.box_acc[b * 3 + 0] = 0u; a.box_acc[b * 3 + 1] = 0u; a.box_acc[b * 3 + 2] = 0u;
        a.box_key[b] = 0ull;
    }
    for (size_t i = gid; i < (size_t)a.cap; i += nthreads) {
        a.row_hit[i] = 0u;
        a.cl_key[i] = 0ull;
        a.cl_any[i] = 0u;
    }
    if (blockIdx.x == 0) {
        using Scan = cub::BlockScan<uint32_t, kCmThreads>;
        __shared__ typename Scan::TempStorage tmp;
        __shared__ uint32_t s_carry;
        if (threadIdx.x == 0) { s_carry = 0u; *a.work_next = 0u; }
        __syncthreads();
        for (int base = 0; base < a.n_samples; base += kCmThreads) {
            const int s = base + threadIdx.x;
            const uint32_t v = s < a.n_samples ? cm_items(a, s) : 0u;
            uint32_t excl, total;
            Scan(tmp).ExclusiveSum(v, excl, total);
            if (s < a.n_samples) a.work_off[s] = s_carry + excl;
            __syncthreads();
            if (threadIdx.x == 0) s_carry += total;
            __syncthreads();
        }
        if (threadIdx.x == 0) a.work_off[a.n_samples] = s_carry;
    }
}

__global__ void __launch_bounds__(kCmThreads) cm_count_kernel(const CmArgs a) {
    __shared__ __align__(16) float s_box[kCmBoxTile * kBoxStride];
    __shared__ uint32_t s_cnt[kCmBoxTile * kCmCols];
    __shared__ uint32_t s_item;
    const int tid = threadIdx.x;
    const uint32_t n_items = a.work_off[a.n_samples];
    for (;;) {
        if (tid == 0) s_item = atomicAdd(a.work_next, 1u);
        __syncthreads();
        const uint32_t w = s_item;
        if (w >= n_items) break;  // uniform
        const int s = cm_last_le(a.work_off, a.n_samples, w);
        const int box0 = a.sample_box_off[s], nbs = a.sample_box_off[s + 1] - box0, K = cm_clusters(a, s);
        const uint32_t nbt = (uint32_t)((nbs + kCmBoxTile - 1) / kCmBoxTile), local = w - a.work_off[s];
        const int bt = (int)(local % nbt), lt = (int)(local / nbt);
        const int b0 = bt * kCmBoxTile, nb = min(kCmBoxTile, nbs - b0);
        const int l0 = lt * kCmLabelTile, nl = max(min(kCmLabelTile, K - l0), 0);
        const float* src = a.boxp + (size_t)(box0 + b0) * kBoxStride;
        for (int i = tid; i < nb * kBoxStride; i += kCmThreads) s_box[i] = src[i];
        for (int i = tid; i < nb * kCmCols; i += kCmThreads) s_cnt[i] = 0u;
        __syncthreads();
        const uint32_t off = a.object_off[s], n = a.counts[s * 3 + 2];
        for (uint32_t r = tid; r < n; r += kCmThreads) {
            const int lab = a.labels[off + r];
            int col;
            if (lab < 0) {
                if (lt != 0) continue;
                col = 0;
            } else {
                if (lab < l0 || lab >= l0 + nl) continue;
                col = lab - l0 + 1;
            }
            const float4 p = a.object[off + r];
            bool any = false;
            for (int b = 0; b < nb; ++b)
                if (box_contains(s_box, b, p.x, p.y, p.z)) {
                    atomicAdd(&s_cnt[b * kCmCols + col], 1u);
                    any = true;
                }
            if (any && col > 0 && atomicExch(&a.row_hit[off + r], 1u) == 0u) atomicAdd(&a.cl_any[off + lab], 1u);
        }
        __syncthreads();
        for (int b = tid; b < nb; b += kCmThreads) {  // per box of the tile: totals and the best label
            const uint32_t* c = s_cnt + b * kCmCols;
            uint32_t rows = 0, nz = 0, best = 0;
            int best_l = 0;
            for (int l = 0; l < nl; ++l) {
                const uint32_t v = c[1 + l];
                rows += v;
                nz += v != 0u;
                if (v > best) { best = v; best_l = l; }
            }
            const int gb = box0 + b0 + b;
            const uint32_t all = rows + (lt == 0 ? c[0] : 0u);
            if (all) atomicAdd(&a.box_acc[gb * 3 + 0], all);
            if (rows) atomicAdd(&a.box_acc[gb * 3 + 1], rows);
            if (nz) atomicAdd(&a.box_acc[gb * 3 + 2], nz);
            if (best) atomicMax(&a.box_key[gb], ((unsigned long long)best << 32) | (uint32_t)~(uint32_t)(l0 + best_l));
        }
        for (int l = tid; l < nl; l += kCmThreads) {  // per label of the tile: the best box
            uint32_t best = 0;
            int best_b = 0;
            for (int b = 0; b < nb; ++b) {
                const uint32_t v = s_cnt[b * kCmCols + 1 + l];
                if (v > best) { best = v; best_b = b; }
            }
            if (best) atomicMax(&a.cl_key[off + l0 + l], ((unsigned long long)best << 32) | (uint32_t)~(uint32_t)(b0 + best_b));
        }
        __syncthreads();  // s_box, s_cnt and s_item are reused by the next item
    }
}

__global__ void __launch_bounds__(kCmThreads) cm_finish_kernel(const CmArgs a) {
    const size_t i = (size_t)blockIdx.x * kCmThreads + threadIdx.x;
    if (i < (size_t)a.n_boxes) {
        const unsigned long long key = a.box_key[i];
        int32_t* o = a.out_box + i * 5;
        o[0] = (int32_t)a.box_acc[i * 3 + 0];
        o[1] = (int32_t)a.box_acc[i * 3 + 1];
        o[2] = (int32_t)a.box_acc[i * 3 + 2];
        o[3] = key ? (int32_t)~(uint32_t)key : -1;
        o[4] = (int32_t)(key >> 32);
    }
    if (i < (size_t)a.cap) {  // cluster slot object_off[s] + k, k < n_clusters[s]
        const int s = cm_last_le(a.object_off, a.n_samples, (uint32_t)i);
        if (a.object_off[s] > (uint32_t)i || (uint32_t)i - a.object_off[s] >= (uint32_t)cm_clusters(a, s)) return;
        const unsigned long long key = a.cl_key[i];
        int32_t* o = a.out_cluster + i * 3;
        o[0] = key ? (int32_t)~(uint32_t)key : -1;
        o[1] = (int32_t)(key >> 32);
        o[2] = (int32_t)a.cl_any[i];
    }
}

struct CmWs {
    size_t work_off, work_next, boxp, box_acc, box_key, row_hit, cl_key, cl_any, total;
};

static CmWs cm_layout(int n_samples, int n_boxes, uint32_t cap) {
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t S = (size_t)n_samples, B = (size_t)n_boxes, n = cap;
    CmWs W;
    size_t o = 0;
    W.work_off = o; o = al(o + (S + 1) * 4);
    W.work_next = o; o = al(o + 4);
    W.boxp = o; o = al(o + B * kBoxStride * 4);
    W.box_acc = o; o = al(o + B * 12);
    W.box_key = o; o = al(o + B * 8);
    W.row_hit = o; o = al(o + n * 4);
    W.cl_key = o; o = al(o + n * 8);
    W.cl_any = o; o = al(o + n * 4);
    W.total = o;
    return W;
}

static bool cm_sizes_ok(int32_t n_samples, int32_t n_boxes, uint32_t cap) {
    return n_samples >= 0 && n_boxes >= 0 && cap <= 0x7fffffffu;
}

}  // namespace msc

extern "C" {

size_t msc_cluster_match_batch_workspace_bytes(int32_t n_samples, int32_t n_boxes, uint32_t row_capacity) {
    using namespace msc;
    if (!cm_sizes_ok(n_samples, n_boxes, row_capacity)) return 0;
    return cm_layout(n_samples, n_boxes, row_capacity).total;
}

int msc_cluster_match_batch(const msc_batch_in* in, const msc_lidar_batch_out* rows, int32_t n_samples, const msc_cluster_match_out* out,
                            void* workspace, size_t workspace_bytes, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(in && rows && out, "msc_cluster_match_batch: null argument");
    MSC_REQUIRE(n_samples >= 0 && in->n_samples >= 0 && in->n_boxes >= 0, "msc_cluster_match_batch: negative count");
    MSC_REQUIRE(n_samples == in->n_samples, "msc_cluster_match_batch: n_samples %d differs from the batch's %d", (int)n_samples,
                (int)in->n_samples);
    if (n_samples == 0) return MSC_OK;
    const uint32_t cap = rows->row_capacity;
    MSC_REQUIRE(cm_sizes_ok(n_samples, in->n_boxes, cap), "msc_cluster_match_batch: row_capacity too large (%u)", cap);
    MSC_REQUIRE(in->sample_box_off && in->ego_pose && in->lidar_calib && (in->n_boxes == 0 || in->boxes),
                "msc_cluster_match_batch: null input array");
    MSC_REQUIRE(rows->counts && rows->object_off && rows->n_clusters && (cap == 0 || (rows->object && rows->labels)),
                "msc_cluster_match_batch: null msc_lidar_batch output");
    MSC_REQUIRE((cap == 0 || out->cluster) && (in->n_boxes == 0 || out->box), "msc_cluster_match_batch: null output");
    const CmWs W = cm_layout(n_samples, in->n_boxes, cap);
    MSC_REQUIRE(workspace, "msc_cluster_match_batch: null workspace");
    MSC_REQUIRE(workspace_bytes >= W.total, "msc_cluster_match_batch: workspace too small: need %zu bytes, got %zu", W.total, workspace_bytes);
    MSC_REQUIRE(((uintptr_t)workspace & 255) == 0, "msc_cluster_match_batch: workspace must be 256-byte aligned");
    int dev = 0, sms = 0;
    MSC_CUDA(cudaGetDevice(&dev));
    MSC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    cudaStream_t stream = (cudaStream_t)stream_v;
    unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);

    CmArgs a;
    a.n_samples = n_samples; a.n_boxes = in->n_boxes; a.cap = cap;
    a.sample_box_off = in->sample_box_off; a.boxes = in->boxes; a.ego_pose = in->ego_pose; a.lidar_calib = in->lidar_calib;
    a.object = reinterpret_cast<const float4*>(rows->object); a.labels = rows->labels; a.object_off = rows->object_off;
    a.counts = rows->counts; a.n_clusters = rows->n_clusters;
    a.work_off = (uint32_t*)(ws + W.work_off); a.work_next = (uint32_t*)(ws + W.work_next); a.boxp = (float*)(ws + W.boxp);
    a.box_acc = (uint32_t*)(ws + W.box_acc); a.box_key = (unsigned long long*)(ws + W.box_key); a.row_hit = (uint32_t*)(ws + W.row_hit);
    a.cl_key = (unsigned long long*)(ws + W.cl_key); a.cl_any = (uint32_t*)(ws + W.cl_any);
    a.out_cluster = out->cluster; a.out_box = out->box;

    const size_t n_fill = std::max<size_t>(std::max<size_t>((size_t)in->n_boxes, cap), 1);
    const unsigned prep_blocks = (unsigned)std::min<size_t>((n_fill + kCmThreads - 1) / kCmThreads, (size_t)sms * 16);
    cm_prep_kernel<<<prep_blocks, kCmThreads, 0, stream>>>(a);
    cm_count_kernel<<<(unsigned)(sms * kCmCtasPerSm), kCmThreads, 0, stream>>>(a);
    cm_finish_kernel<<<(unsigned)((n_fill + kCmThreads - 1) / kCmThreads), kCmThreads, 0, stream>>>(a);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

}  // extern "C"
