// lidar_images.cu -- the LiDAR agent's images for many samples / clusters per call: the finished 800 x 800 BEV of every sample of a
// window of an msc_lidar_batch result (LiDARAgent._generate_multi_layer_bev, lidar_agent.py:539-634) and the finished 512 x 512
// 4-view image of every cluster of a view list (LiDARAgent._generate_cluster_visualization, :241-356).
//
// The cv2 overlays (ego cross, rings, labels, axes, titles) are drawn with the default LINE_8 and no anti-aliasing: the pixels they set
// and the colours they set them to do not depend on what is underneath.  The host derives that fixed (pixel, BGR) list -- the stamp --
// once per image geometry from its own drawing code, and the last kernel of each call writes it over the raster (DESIGN.md section 4.7).
#include <cub/block/block_scan.cuh>

#include "lidar_common.cuh"

namespace msc {

constexpr uint32_t kBevTableShort = 1u;   // msc_keyframe_bev_batch status: a cell count has no entry in the density table
constexpr uint32_t kViewTooLarge = 1u;    // msc_cluster_views_batch status: a view holds more points than max_view_points
constexpr int kBevRasterBlocks = 148 * 8;

struct BevWindow {
    const float4* ground;
    const float4* object;
    const uint32_t* ground_off;
    const uint32_t* object_off;
    const uint32_t* counts;
    int first, n, res;
    float bev_range;
    uint32_t* count;    // [n, res, res] rows per cell, rows flipped like the output
    uint32_t* winner;   // [n, res, res] 0 empty, 1 ground, 2 + i object row i of the sample
    uint32_t* smp;      // [n, 4] ordered-int min / max object height, largest cell count, -
    float* height;      // [n, res, res] output, flipped
};

// window sample of row `row`: the last s in [first, first + n) whose slice starts at or before it (an empty sample shares its
// offset with the next one, which then owns the row)
__device__ __forceinline__ int window_sample(const uint32_t* __restrict__ off, int first, int n, uint32_t row) {
    int lo = first, hi = first + n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= row) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// one pass over the ground then the object rows of the window (grid-stride, warp-uniform trip count): the raster of
// kf_bev_raster_kernel on each row's own grid, writing the flipped row (cv2.flip(..., 0), lidar_agent.py:618-620)
__global__ void __launch_bounds__(256) bev_batch_raster_kernel(const BevWindow W) {
    const int last = W.first + W.n - 1;
    const uint32_t g0 = W.ground_off[W.first], o0 = W.object_off[W.first];
    const uint32_t ng = W.ground_off[last] + W.counts[last * 3 + 1] - g0;
    const uint32_t total = ng + W.object_off[last] + W.counts[last * 3 + 2] - o0;
    const int res = W.res;
    const float two_r = __fmul_rn(2.0f, W.bev_range), resf = (float)res;
    const size_t plane = (size_t)res * res;
    const uint32_t lane = threadIdx.x & 31;
    for (uint32_t base = blockIdx.x * blockDim.x + threadIdx.x - lane; base < total; base += gridDim.x * blockDim.x) {
        const uint32_t i = base + lane;
        int s = -1;
        uint32_t cnt = 0, zlo = 0xffffffffu, zhi = 0u;
        if (i < total) {
            const bool is_obj = i >= ng;
            const uint32_t row = is_obj ? o0 + (i - ng) : g0 + i;
            s = window_sample(is_obj ? W.object_off : W.ground_off, W.first, W.n, row);
            const float4 p = is_obj ? W.object[row] : W.ground[row];
            int ix, iy;
            bev_xy(p, W.bev_range, two_r, resf, res, &ix, &iy);
            const size_t cell = (size_t)(s - W.first) * plane + (size_t)(res - 1 - iy) * res + ix;
            cnt = atomicAdd(&W.count[cell], 1u) + 1u;  // the cell's final count is the largest of these
            if (p.z > 0.0f) atomicMax(reinterpret_cast<int*>(W.height) + cell, __float_as_int(p.z));
            atomicMax(&W.winner[cell], is_obj ? (2u + (row - W.object_off[s])) : 1u);
            if (is_obj) { zlo = f2ord(p.z); zhi = zlo; }
        }
        // per-sample maxima: one set of atomics per warp whose rows are one sample's (nearly all), else one per row
        const int s0 = __shfl_sync(0xffffffffu, s, 0);
        if (__all_sync(0xffffffffu, s == s0)) {
            cnt = __reduce_max_sync(0xffffffffu, cnt);
            zlo = __reduce_min_sync(0xffffffffu, zlo);
            zhi = __reduce_max_sync(0xffffffffu, zhi);
            if (lane != 0) s = -1;
        }
        if (s >= 0) {
            uint32_t* m = W.smp + (size_t)(s - W.first) * 4;
            atomicMax(&m[2], cnt);
            if (zlo != 0xffffffffu) { atomicMin(&m[0], zlo); atomicMax(&m[1], zhi); }
        }
    }
}

// one thread per output pixel: semantic colour from the winner and density lut[c] / lut[cmax] * 255 in float32 (lidar_agent.py:563-564
// through finish_bev_layers' table); the height plane is already final
__global__ void __launch_bounds__(256) bev_batch_finish_kernel(const BevWindow W, const float* __restrict__ lut, uint32_t lut_len,
                                                              uint8_t* __restrict__ semantic, uint8_t* __restrict__ density,
                                                              uint32_t* __restrict__ status) {
    const size_t plane = (size_t)W.res * W.res;
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= plane) return;
    const int i = blockIdx.y;
    const size_t c = (size_t)i * plane + p;
    const uint32_t* m = W.smp + (size_t)i * 4;
    uint8_t b, g, r;
    bev_colour(W.winner[c], W.object + W.object_off[W.first + i], m, &b, &g, &r);
    semantic[c * 3 + 0] = b; semantic[c * 3 + 1] = g; semantic[c * 3 + 2] = r;
    const uint32_t cmax = m[2];
    uint8_t d = 0;
    if (cmax >= lut_len) {
        if (p == 0) atomicOr(status, kBevTableShort);
    } else if (cmax > 0) {
        d = (uint8_t)__float2int_rz(__fmul_rn(__fdiv_rn(lut[W.count[c]], lut[cmax]), 255.0f));
    }
    density[c] = d;
}

// stamp [m, 2] = (pixel, B | G << 8 | R << 16) written over image blockIdx.y of `out`
__global__ void __launch_bounds__(256) stamp_kernel(const uint32_t* __restrict__ stamp, uint32_t m, uint8_t* __restrict__ out, uint32_t image_px) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const uint32_t px = stamp[2 * j], col = stamp[2 * j + 1];
    if (px >= image_px) return;
    uint8_t* o = out + ((size_t)blockIdx.y * image_px + px) * 3;
    o[0] = (uint8_t)col; o[1] = (uint8_t)(col >> 8); o[2] = (uint8_t)(col >> 16);
}

// ---------------------------------------------------------------- cluster views
// one CTA per view: its point count; a view above max_points sets the status and counts as empty
__global__ void __launch_bounds__(256) view_count_kernel(const int32_t* __restrict__ labels, const int32_t* __restrict__ views, uint32_t max_points,
                                                        int32_t* __restrict__ off, uint32_t* __restrict__ status) {
    __shared__ uint32_t s_n;
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    const int32_t* v = views + 3 * blockIdx.x;
    const int32_t e = v[1], lab = v[2];
    uint32_t c = 0;
    for (int32_t r = v[0] + (int32_t)threadIdx.x; r < e; r += blockDim.x) c += labels[r] == lab;
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_n, c);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t n = s_n;
        if (n > max_points) { atomicOr(status, kViewTooLarge); n = 0; }
        off[blockIdx.x] = (int32_t)n;
    }
}

// single block: counts off[0..n) -> exclusive offsets off[0..n]
__global__ void __launch_bounds__(1024) view_scan_kernel(int32_t* __restrict__ off, int n) {
    using Scan = cub::BlockScan<int32_t, 1024>;
    __shared__ typename Scan::TempStorage tmp;
    int32_t carry = 0;
    for (int base = 0; base < n; base += 1024) {
        const int i = base + threadIdx.x;
        const int32_t x = i < n ? off[i] : 0;
        int32_t ex, sum;
        Scan(tmp).ExclusiveSum(x, ex, sum);
        if (i < n) off[i] = carry + ex;
        carry += sum;
        __syncthreads();
    }
    if (threadIdx.x == 0) off[n] = carry;
}

// one CTA per view: its rows in row order into order[off[v] ..], and the mean and pixel scale of ops.cluster_views (lidar_agent.py
// :255-264): the mean is NumPy's float32 sum along axis 0 -- sequential in row order -- over n; max_range the largest per-axis
// fl(fl(max - c) - fl(min - c)) (rounding is monotone, so the extremes of the centred points are the centred extremes)
__global__ void __launch_bounds__(256) view_gather_kernel(const float4* __restrict__ rows, const int32_t* __restrict__ labels,
                                                         const int32_t* __restrict__ views, const int32_t* __restrict__ off,
                                                         uint32_t* __restrict__ order, float* __restrict__ center_scale) {
    __shared__ float s_xyz[3][256];
    __shared__ uint32_t s_warp[8], s_mm[6];
    const int v = blockIdx.x;
    const int32_t o = off[v], n = off[v + 1] - o;
    float* cs = center_scale + 4 * v;
    if (n == 0) {  // an oversized view (the status is set); the splat reads no point of it
        if (threadIdx.x < 4) cs[threadIdx.x] = threadIdx.x == 3 ? 1.0f : 0.0f;
        return;
    }
    const int32_t b = views[3 * v], e = views[3 * v + 1], lab = views[3 * v + 2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < 6) s_mm[threadIdx.x] = threadIdx.x < 3 ? 0xffffffffu : 0u;
    float sx = 0.0f, sy = 0.0f, sz = 0.0f;
    uint32_t done = 0;
    for (int32_t base = b; base < e; base += 256) {
        const int32_t r = base + (int32_t)threadIdx.x;
        const bool hit = r < e && labels[r] == lab;
        const uint32_t bal = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        uint32_t before = 0, tile = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) { before += w < warp ? s_warp[w] : 0u; tile += s_warp[w]; }
        if (hit) {
            const uint32_t k = before + __popc(bal & ((1u << lane) - 1u));
            const float4 p = rows[r];
            order[o + done + k] = (uint32_t)r;
            s_xyz[0][k] = p.x; s_xyz[1][k] = p.y; s_xyz[2][k] = p.z;
            const uint32_t q[3] = {f2ord(p.x), f2ord(p.y), f2ord(p.z)};
#pragma unroll
            for (int a = 0; a < 3; ++a) { atomicMin(&s_mm[a], q[a]); atomicMax(&s_mm[3 + a], q[a]); }
        }
        __syncthreads();
        if (threadIdx.x == 0)
            for (uint32_t k = 0; k < tile; ++k) { sx = __fadd_rn(sx, s_xyz[0][k]); sy = __fadd_rn(sy, s_xyz[1][k]); sz = __fadd_rn(sz, s_xyz[2][k]); }
        done += tile;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const float nf = (float)n;
        const float c[3] = {__fdiv_rn(sx, nf), __fdiv_rn(sy, nf), __fdiv_rn(sz, nf)};
        float mr = 0.0f;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float ra = __fsub_rn(__fsub_rn(ord2f(s_mm[3 + a]), c[a]), __fsub_rn(ord2f(s_mm[a]), c[a]));
            if (a == 0 || ra > mr) mr = ra;  // Python's max(a, b, c)
        }
        cs[0] = c[0]; cs[1] = c[1]; cs[2] = c[2];
        cs[3] = mr > 0.0f ? __fdiv_rn(89.6f, mr) : 1.0f;  // (256 * 0.35) / np.float32 evaluates in float32
    }
}

struct ViewsWs {
    size_t keys, irange, center_scale, off, views, order, end;
};
inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }
inline ViewsWs views_layout(int n_views, int max_view_points) {
    ViewsWs w;
    const size_t n = (size_t)n_views;
    w.keys = 0;
    w.irange = align256(w.keys + n * kGrid * kGrid * 4);
    w.center_scale = align256(w.irange + n * 32);
    w.off = align256(w.center_scale + n * 16);
    w.views = align256(w.off + (n + 1) * 4);
    w.order = align256(w.views + n * 12);
    w.end = align256(w.order + n * (size_t)max_view_points * 4);
    return w;
}
inline size_t bev_ws_bytes(int res, int n) {
    const size_t plane = (size_t)res * res * n * 4;
    return align256(plane) * 2 + align256((size_t)n * 16);
}

}  // namespace msc

extern "C" {

size_t msc_keyframe_bev_batch_workspace_bytes(int32_t bev_res, int32_t n) {
    if (bev_res <= 0 || bev_res > 8192 || n < 0 || n > 65535) return 0;
    return msc::bev_ws_bytes(bev_res, n);
}

int msc_keyframe_bev_batch(const msc_params* params, const msc_lidar_batch_out* rows, int32_t n_samples, int32_t first, int32_t n,
                           const float* lut, int32_t lut_len, const uint32_t* stamp, int32_t stamp_len, uint8_t* semantic, float* height,
                           uint8_t* density, uint32_t* status, void* workspace, size_t workspace_bytes, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(params && rows, "null argument");
    const int res = params->bev_res;
    MSC_REQUIRE(res > 0 && res <= 8192, "bev_res out of range");
    MSC_REQUIRE(first >= 0 && n >= 0 && n <= 65535 && (int64_t)first + n <= n_samples, "window [first, first + n) outside the batch");
    MSC_REQUIRE(lut_len >= 1 && stamp_len >= 0, "negative sizes");
    if (n == 0) return MSC_OK;
    MSC_REQUIRE(rows->ground_off && rows->object_off && rows->counts && ((rows->ground && rows->object) || rows->row_capacity == 0),
                "null row buffer");
    MSC_REQUIRE(lut && (stamp || stamp_len == 0) && semantic && height && density && status && workspace, "null buffer");
    MSC_REQUIRE(workspace_bytes >= bev_ws_bytes(res, n), "workspace too small: need %zu bytes", bev_ws_bytes(res, n));
    cudaStream_t stream = (cudaStream_t)stream_v;
    const size_t plane = (size_t)res * res;
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    const size_t grid_bytes = align256(plane * n * 4);
    BevWindow W{reinterpret_cast<const float4*>(rows->ground), reinterpret_cast<const float4*>(rows->object), rows->ground_off, rows->object_off,
                rows->counts, first, n, res, params->bev_range, reinterpret_cast<uint32_t*>(ws), reinterpret_cast<uint32_t*>(ws + grid_bytes),
                reinterpret_cast<uint32_t*>(ws + 2 * grid_bytes), height};
    MSC_CUDA(cudaMemsetAsync(ws, 0, 2 * grid_bytes, stream));
    MSC_CUDA(cudaMemsetAsync(W.smp, 0, (size_t)n * 16, stream));
    MSC_CUDA(cudaMemset2DAsync(W.smp, 16, 0xff, 4, (size_t)n, stream));  // min height: ordered +inf
    MSC_CUDA(cudaMemsetAsync(height, 0, plane * n * 4, stream));
    bev_batch_raster_kernel<<<kBevRasterBlocks, 256, 0, stream>>>(W);
    const dim3 grid((unsigned)((plane + 255) / 256), (unsigned)n);
    bev_batch_finish_kernel<<<grid, 256, 0, stream>>>(W, lut, (uint32_t)lut_len, semantic, density, status);
    if (stamp_len > 0)
        stamp_kernel<<<dim3((unsigned)((stamp_len + 255) / 256), (unsigned)n), 256, 0, stream>>>(stamp, (uint32_t)stamp_len, semantic, (uint32_t)plane);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

size_t msc_cluster_views_batch_workspace_bytes(int32_t n_views, int32_t max_view_points) {
    if (n_views < 0 || n_views > 65535 || max_view_points < 0 || max_view_points >= (1 << 24)) return 0;
    return msc::views_layout(n_views, max_view_points).end;
}

int msc_cluster_views_batch(const float* rows, const int32_t* labels, const int32_t* views, int32_t n_views, int32_t max_view_points,
                            const uint32_t* stamp, int32_t stamp_len, uint8_t* out_bgr, uint32_t* status, void* workspace,
                            size_t workspace_bytes, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(n_views >= 0 && n_views <= 65535, "n_views out of range");
    MSC_REQUIRE(max_view_points >= 0 && max_view_points < (1 << 24), "max_view_points out of range for the 24-bit draw-order key");
    MSC_REQUIRE(stamp_len >= 0, "negative stamp length");
    if (n_views == 0) return MSC_OK;
    MSC_REQUIRE(rows && labels && views && (stamp || stamp_len == 0) && out_bgr && status && workspace, "null buffer");
    for (int v = 0; v < n_views; ++v)
        MSC_REQUIRE(views[3 * v] >= 0 && views[3 * v] < views[3 * v + 1], "view %d: empty or inverted row range [%d, %d)", v, views[3 * v],
                    views[3 * v + 1]);
    const ViewsWs L = views_layout(n_views, max_view_points);
    MSC_REQUIRE(workspace_bytes >= L.end, "workspace too small: need %zu bytes", L.end);
    cudaStream_t stream = (cudaStream_t)stream_v;
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    uint32_t* keys = reinterpret_cast<uint32_t*>(ws + L.keys);
    uint32_t* irange = reinterpret_cast<uint32_t*>(ws + L.irange);
    float* cs = reinterpret_cast<float*>(ws + L.center_scale);
    int32_t* off = reinterpret_cast<int32_t*>(ws + L.off);
    int32_t* dviews = reinterpret_cast<int32_t*>(ws + L.views);
    uint32_t* order = reinterpret_cast<uint32_t*>(ws + L.order);
    const float4* pts = reinterpret_cast<const float4*>(rows);
    MSC_CUDA(cudaMemcpyAsync(dviews, views, (size_t)n_views * 12, cudaMemcpyHostToDevice, stream));
    MSC_CUDA(cudaMemsetAsync(keys, 0, (size_t)n_views * kGrid * kGrid * 4, stream));
    MSC_CUDA(cudaMemsetAsync(irange, 0, (size_t)n_views * 32, stream));  // pairs (min as ordered uint = 0xffffffff, max = 0)
    MSC_CUDA(cudaMemset2DAsync(irange, 8, 0xff, 4, (size_t)n_views * 4, stream));
    view_count_kernel<<<n_views, 256, 0, stream>>>(labels, dviews, (uint32_t)max_view_points, off, status);
    view_scan_kernel<<<1, 1024, 0, stream>>>(off, n_views);
    view_gather_kernel<<<n_views, 256, 0, stream>>>(pts, labels, dviews, off, order, cs);
    if (max_view_points > 0) {
        const dim3 grid((unsigned)((max_view_points * 4 + 255) / 256), (unsigned)n_views);
        cluster_splat_kernel<<<grid, 256, 0, stream>>>(pts, order, off, n_views, cs, keys, irange);
    }
    cluster_colour_kernel<<<dim3((kGrid * kGrid + 255) / 256, (unsigned)n_views), 256, 0, stream>>>(pts, order, off, keys, irange, out_bgr);
    if (stamp_len > 0)
        stamp_kernel<<<dim3((unsigned)((stamp_len + 255) / 256), (unsigned)n_views), 256, 0, stream>>>(stamp, (uint32_t)stamp_len, out_bgr,
                                                                                                        kGrid * kGrid);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

}  // extern "C"
