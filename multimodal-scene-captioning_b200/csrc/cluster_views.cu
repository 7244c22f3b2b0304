// cluster_views.cu -- the per-cluster 4-view raster the reference sends to its VLM
// (LiDARAgent._generate_cluster_visualization, lidar_agent.py:241-356), SURVEY.md section 8(f) rank 1.
//
// The reference draws, per cluster, four 256x256 views into a 512x512 grid with one cv2.circle(radius 2, filled) per
// point in a Python loop; later points overwrite earlier ones, later views overwrite earlier views where discs bleed
// over a quadrant border.  On the device that is: per point and view, atomicMax of the draw order into a per-pixel
// key grid over the 13-pixel footprint of cv2's filled radius-2 circle (|dx|+|dy| <= 2, clipped to the 512x512 grid),
// then one pass that turns each pixel's winner into its grey value.  Axes, titles (cv2.line / cv2.putText) and the
// batch mosaic stay on the host: they are drawn after the points and never overlap another view's discs.
#include "lidar_common.cuh"

namespace msc {

__device__ __forceinline__ uint32_t f2ord_cv(float f) {
    uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float ord2f_cv(uint32_t u) {
    uint32_t b = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
    return __uint_as_float(b);
}

// pixel of point p in view v (lidar_agent.py:276-280 for the axis views, :322-336 for the isometric one)
__device__ __forceinline__ bool view_pixel(int v, float cx, float cy, float cz, float scale, int* px, int* py) {
    if (v < 3) {
        const float a = (v == 2) ? cy : cx;               // (0,1) (0,2) (1,2)
        const float b = (v == 0) ? cy : cz;
        *px = __float2int_rz(__fadd_rn(__fmul_rn(a, scale), 128.0f));   // float32 arithmetic, astype(int) truncates
        *py = __float2int_rz(__fadd_rn(__fmul_rn(b, scale), 128.0f));
    } else {
        const double c = 0.8660254037844387, s = 0.49999999999999994;   // np.cos(np.pi/6), np.sin(np.pi/6)
        const double x = (double)cx, y = (double)cy, z = (double)cz;
        const double r1y = y * c - z * s, r1z = y * s + z * c;          // centered @ rot_x.T
        const double r2x = x * c + r1z * s, r2z = -x * s + r1z * c;     // ... @ rot_y.T
        const double sc = (double)scale;
        *px = __double2int_rz((r2x + r1y * 0.5) * sc + 128.0);
        *py = __double2int_rz((r2z - r1y * 0.5) * sc + 128.0);
    }
    return *px >= 0 && *px < kView && *py >= 0 && *py < kView;
}

// one thread per (point of a cluster, view): intensity range of the view's valid points + disc splat of the draw order
__global__ void __launch_bounds__(256) cluster_splat_kernel(const float4* __restrict__ pts, const uint32_t* __restrict__ order,
                                                           const int32_t* __restrict__ cluster_off, int n_clusters, const float* __restrict__ center_scale,
                                                           uint32_t* __restrict__ keys, uint32_t* __restrict__ irange) {
    const int cl = blockIdx.y;
    const int n = cluster_off[cl + 1] - cluster_off[cl];
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * 4) return;
    const int rank = t >> 2, v = t & 3;
    const float4 p = pts[order[cluster_off[cl] + rank]];
    const float* cs = center_scale + cl * 4;
    const float cx = __fsub_rn(p.x, cs[0]), cy = __fsub_rn(p.y, cs[1]), cz = __fsub_rn(p.z, cs[2]);  // :256
    int px, py;
    if (!view_pixel(v, cx, cy, cz, cs[3], &px, &py)) return;
    const uint32_t io = f2ord_cv(p.w);
    atomicMin(&irange[(cl * 4 + v) * 2 + 0], io);   // :287 intensities.min() / .max() over the valid points of this view
    atomicMax(&irange[(cl * 4 + v) * 2 + 1], io);
    const int gx = (v & 1) * kView + px;                       // quadrant_x = 0,1,0,1
    const int gy = (v >> 1) * kView + (kView - py - 1);        // quadrant_y = 0,0,1,1 ; y flipped (:296)
    const uint32_t key = ((uint32_t)(v + 1) << 24) | (uint32_t)(rank + 1);  // later view, then later point, wins
    uint32_t* g = keys + (size_t)cl * kGrid * kGrid;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
        const int w = 2 - (dy < 0 ? -dy : dy);
        const int y = gy + dy;
        if (y < 0 || y >= kGrid) continue;
        for (int dx = -w; dx <= w; ++dx) {
            const int x = gx + dx;
            if (x >= 0 && x < kGrid) atomicMax(&g[y * kGrid + x], key);
        }
    }
}

// one thread per pixel: white background, else the winner's intensity normalised over its view (:287-288, float32)
__global__ void __launch_bounds__(256) cluster_colour_kernel(const float4* __restrict__ pts, const uint32_t* __restrict__ order,
                                                            const int32_t* __restrict__ cluster_off, const uint32_t* __restrict__ keys,
                                                            const uint32_t* __restrict__ irange, uint8_t* __restrict__ out) {
    const int cl = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= kGrid * kGrid) return;
    const uint32_t key = keys[(size_t)cl * kGrid * kGrid + i];
    uint8_t g = 255;
    if (key) {
        const int v = (int)(key >> 24) - 1, rank = (int)(key & 0xffffffu) - 1;
        const float inten = pts[order[cluster_off[cl] + rank]].w;
        const float lo = ord2f_cv(irange[(cl * 4 + v) * 2]), hi = ord2f_cv(irange[(cl * 4 + v) * 2 + 1]);
        const float nrm = __fmul_rn(__fdiv_rn(__fsub_rn(inten, lo), __fadd_rn(__fsub_rn(hi, lo), 1e-6f)), 255.0f);
        g = (uint8_t)__float2int_rz(nrm);  // astype(np.uint8) of a value in [0, 255)
    }
    uint8_t* o = out + ((size_t)cl * kGrid * kGrid + i) * 3;
    o[0] = g; o[1] = g; o[2] = g;
}

}  // namespace msc

extern "C" int msc_cluster_views(const float* pts_xyzi, const uint32_t* order, const int32_t* cluster_off, int32_t n_clusters,
                                 int32_t max_cluster_points, const float* center_scale, uint32_t* keys, uint32_t* irange, uint8_t* out_bgr,
                                 void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(n_clusters >= 0 && max_cluster_points >= 0, "negative counts");
    if (n_clusters == 0) return MSC_OK;
    MSC_REQUIRE(pts_xyzi && order && cluster_off && center_scale && keys && irange && out_bgr, "null argument");
    MSC_REQUIRE(max_cluster_points < (1 << 24), "cluster too large for the 24-bit draw-order key");
    cudaStream_t stream = (cudaStream_t)stream_v;
    MSC_CUDA(cudaMemsetAsync(keys, 0, (size_t)n_clusters * kGrid * kGrid * 4, stream));
    // irange pairs: (min as ordered uint = 0xffffffff, max = 0)
    MSC_CUDA(cudaMemsetAsync(irange, 0, (size_t)n_clusters * 8 * 4, stream));
    MSC_CUDA(cudaMemset2DAsync(irange, 8, 0xff, 4, (size_t)n_clusters * 4, stream));
    if (max_cluster_points > 0) {
        dim3 grid((unsigned)((max_cluster_points * 4 + 255) / 256), (unsigned)n_clusters);
        cluster_splat_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const float4*>(pts_xyzi), order, cluster_off, n_clusters, center_scale, keys,
                                                        irange);
    }
    dim3 grid2((kGrid * kGrid + 255) / 256, (unsigned)n_clusters);
    cluster_colour_kernel<<<grid2, 256, 0, stream>>>(reinterpret_cast<const float4*>(pts_xyzi), order, cluster_off, keys, irange, out_bgr);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}
