// camera_depth.cu -- [EXT] row e7: LiDAR returns projected into the camera images (devkit map_pointcloud_to_image), batched.
// Per (sample, camera) a downsampled depth map (minimum depth per ds x ds pixel block) and the number of returns that land in the
// image; per (box, camera) the LiDAR support of the box's projected extent.  Definition: include/msc_geom.h msc_camera_depth_batch.
//
// Three launches, stream-ordered:
//   camera_depth_fill_kernel     depth <- +inf bits, cam_points <- 0;
//   camera_depth_kernel          one pass over the raw sweeps: CTA (s, part) of X CTAs per sample composes sample s's camera matrices
//                                once, then takes every X-th 1024-point tile of the sample's sweeps (tiles numbered across the sweeps),
//                                stages its rows in shared memory with 16-byte loads, transforms and projects each point and stores
//                                its depth with a 32-bit atomicMin on the bits of the positive f32 depth (bit order = value order);
//                                cam_points is a warp reduction into shared counters, added to global once per CTA;
//   camera_depth_support_kernel  one warp per (box, camera): the box projection of msc_project_boxes (project_box_z), then a scan of
//                                the extent's depth blocks with four warp-reduced counts.
// Minimum and sums are order-independent, so the results do not depend on X, the tile size or the scheduling.
#include <algorithm>

#include "msc_common.cuh"

namespace msc {

constexpr int kDepthThreads = 256;
constexpr int kDepthPPT = 4;                              // points per thread per tile
constexpr int kDepthTile = kDepthThreads * kDepthPPT;     // points per tile (a multiple of 4: tiles start 16-byte aligned)
constexpr int kDepthTileVec = kDepthTile * 5 / 4;         // float4s of a full tile
constexpr int kDepthPointsPerCta = 16384;                 // sizes X from the batch's points-per-sample hint
constexpr uint32_t kInfBits = 0x7f800000u;

struct DepthArgs {
    const float* points;
    const int32_t* sample_sweep_off;
    const uint32_t* sweep_start;
    const uint32_t* sweep_count;
    const double* sweep_pose;
    const double* ego_pose;
    const double* lidar_calib;
    const double* cam_ego_pose;
    const double* cam_calib;
    const double* cam_K;
    uint32_t* depth_bits;
    uint32_t* cam_points;
    float rc, min_dist, u_hi, v_hi, u_guard, v_guard;
    int n_cams, ds, hb, wb, ctas_per_sample;
};

// cam_from_ref, f64 without FMA in this order: ref -> ego (lidar_calib: c' = R c + t), ego -> global (ego_pose, same form),
// global -> camera ego (cam_ego_pose, frame_change), camera ego -> camera (cam_calib, frame_change); then P = K [R | t] rounded once.
__device__ __forceinline__ void rigid_apply(const double* __restrict__ pose7, double c[3], double R[9]) {
    double Q[9];
    quat_to_rot(pose7 + 3, Q);
    double c2[3], R2[9];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        c2[r] = ((Q[r * 3 + 0] * c[0] + Q[r * 3 + 1] * c[1]) + Q[r * 3 + 2] * c[2]) + pose7[r];
#pragma unroll
        for (int k = 0; k < 3; ++k) R2[r * 3 + k] = (Q[r * 3 + 0] * R[0 * 3 + k] + Q[r * 3 + 1] * R[1 * 3 + k]) + Q[r * 3 + 2] * R[2 * 3 + k];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) c[k] = c2[k];
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = R2[k];
}

__device__ __noinline__ void camera_matrix(const double* __restrict__ ego_pose, const double* __restrict__ lidar_calib,
                                           const double* __restrict__ cam_ego_pose, const double* __restrict__ cam_calib,
                                           const double* __restrict__ K, float* P12) {
    double c[3] = {lidar_calib[0], lidar_calib[1], lidar_calib[2]};
    double R[9];
    quat_to_rot(lidar_calib + 3, R);
    rigid_apply(ego_pose, c, R);
    frame_change(cam_ego_pose, c, R);
    frame_change(cam_calib, c, R);
    for (int r = 0; r < 3; ++r) {
        for (int k = 0; k < 3; ++k) P12[r * 4 + k] = (float)((K[r * 3 + 0] * R[0 * 3 + k] + K[r * 3 + 1] * R[1 * 3 + k]) + K[r * 3 + 2] * R[2 * 3 + k]);
        P12[r * 4 + 3] = (float)((K[r * 3 + 0] * c[0] + K[r * 3 + 1] * c[1]) + K[r * 3 + 2] * c[2]);
    }
}

__global__ void __launch_bounds__(kDepthThreads) camera_depth_fill_kernel(uint32_t* __restrict__ depth_bits, size_t n,
                                                                          uint32_t* __restrict__ cam_points, int n_cp) {
    const size_t stride = (size_t)gridDim.x * kDepthThreads;
    for (size_t i = (size_t)blockIdx.x * kDepthThreads + threadIdx.x; i < n; i += stride) depth_bits[i] = kInfBits;
    if (blockIdx.x == 0)
        for (int i = threadIdx.x; i < n_cp; i += kDepthThreads) cam_points[i] = 0;
}

__global__ void __launch_bounds__(kDepthThreads) camera_depth_kernel(const DepthArgs a) {
    __shared__ float4 s_rows[kDepthTileVec];
    __shared__ float4 s_P[MSC_MAX_CAMS * 3];
    __shared__ uint32_t s_cnt[MSC_MAX_CAMS];
    const int X = a.ctas_per_sample;
    const int s = blockIdx.x / X, part = blockIdx.x - s * X;
    const int C = a.n_cams, tid = threadIdx.x, lane = tid & 31;
    if (tid < C) {
        const size_t sc = (size_t)s * C + tid;
        camera_matrix(a.ego_pose + (size_t)s * 7, a.lidar_calib + (size_t)s * 7, a.cam_ego_pose + sc * 7, a.cam_calib + sc * 7,
                      a.cam_K + sc * 9, reinterpret_cast<float*>(&s_P[tid * 3]));
        s_cnt[tid] = 0;
    }
    const int sw0 = a.sample_sweep_off[s], sw1 = a.sample_sweep_off[s + 1];
    const float* s_f = reinterpret_cast<const float*>(s_rows);
    __syncthreads();
    uint32_t base = 0;  // number of the sample's first tile of sweep j (tiles are numbered across the sample's sweeps)
    for (int j = sw0; j < sw1; ++j) {
        const uint32_t cnt = a.sweep_count[j], start = a.sweep_start[j];
        const uint32_t nt = (cnt + kDepthTile - 1) / kDepthTile;
        const double* M = a.sweep_pose + (size_t)j * 12;
        double m[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) m[k] = M[k];
        // first tile t of this sweep with (base + t) % X == part
        for (uint32_t t = ((uint32_t)part + (uint32_t)X - base % (uint32_t)X) % (uint32_t)X; t < nt; t += (uint32_t)X) {
            const uint32_t n = min((uint32_t)kDepthTile, cnt - t * kDepthTile);
            const uint32_t nvec = (n * 5 + 3) / 4;  // ends within 16 bytes of the last row (msc_batch_in layout rule)
            const float4* src = reinterpret_cast<const float4*>(a.points + ((size_t)start + (size_t)t * kDepthTile) * 5);
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const uint32_t i = tid + k * kDepthThreads;
                if (i < nvec) s_rows[i] = __ldcs(src + i);
            }
            __syncthreads();
            float px[kDepthPPT], py[kDepthPPT], pz[kDepthPPT];
            bool ok[kDepthPPT];
#pragma unroll
            for (int k = 0; k < kDepthPPT; ++k) {
                const uint32_t i = tid + k * kDepthThreads;
                const float x = s_f[5 * i], y = s_f[5 * i + 1], z = s_f[5 * i + 2];
                ok[k] = (i < n) && !(fabsf(x) < a.rc && fabsf(y) < a.rc);  // remove_close in the sweep's own frame
                const double xd = (double)x, yd = (double)y, zd = (double)z;
                px[k] = (float)__fma_rn(m[0], xd, __fma_rn(m[1], yd, __fma_rn(m[2], zd, m[3])));
                py[k] = (float)__fma_rn(m[4], xd, __fma_rn(m[5], yd, __fma_rn(m[6], zd, m[7])));
                pz[k] = (float)__fma_rn(m[8], xd, __fma_rn(m[9], yd, __fma_rn(m[10], zd, m[11])));
            }
            __syncthreads();  // s_rows is free for the next tile
            for (int c = 0; c < C; ++c) {
                const float4 p0 = s_P[c * 3], p1 = s_P[c * 3 + 1], p2 = s_P[c * 3 + 2];
                uint32_t* img = a.depth_bits + (size_t)(s * C + c) * (size_t)a.hb * (size_t)a.wb;
                uint32_t hits = 0;
#pragma unroll
                for (int k = 0; k < kDepthPPT; ++k) {
                    const float w = __fmaf_rn(p2.x, px[k], __fmaf_rn(p2.y, py[k], __fmaf_rn(p2.z, pz[k], p2.w)));
                    if (!(ok[k] && w > a.min_dist)) continue;  // w > 0 from here on (min_dist >= 0)
                    const float ua = __fmaf_rn(p0.x, px[k], __fmaf_rn(p0.y, py[k], __fmaf_rn(p0.z, pz[k], p0.w)));
                    const float vb = __fmaf_rn(p1.x, px[k], __fmaf_rn(p1.y, py[k], __fmaf_rn(p1.z, pz[k], p1.w)));
                    // conservative rejects before the divisions: a < RN(w/2) gives RN(a/w) <= 1 (also for subnormal w), and
                    // a > RN(2W w) gives RN(a/w) >= W - 1; NaN passes them and fails the exact test below
                    if (ua < __fmul_rn(0.5f, w) || ua > __fmul_rn(a.u_guard, w) || vb < __fmul_rn(0.5f, w) || vb > __fmul_rn(a.v_guard, w)) continue;
                    const float u = __fdiv_rn(ua, w), v = __fdiv_rn(vb, w);
                    if (!(u > 1.0f && u < a.u_hi && v > 1.0f && v < a.v_hi)) continue;
                    const int bx = __float2int_rz(u) / a.ds, by = __float2int_rz(v) / a.ds;
                    atomicMin(img + (size_t)by * a.wb + bx, __float_as_uint(w));
                    ++hits;
                }
                hits = __reduce_add_sync(0xffffffffu, hits);
                if (lane == 0 && hits) atomicAdd(&s_cnt[c], hits);
            }
        }
        base += nt;
    }
    __syncthreads();
    if (tid < C && s_cnt[tid]) atomicAdd(&a.cam_points[(size_t)s * C + tid], s_cnt[tid]);
}

struct SupportArgs {
    int n_samples, n_boxes, n_cams, ds, hb, wb, image_w, image_h;
    double margin;
    const int32_t* sample_box_off;
    const double* boxes;
    const double* cam_ego_pose;
    const double* cam_calib;
    const double* cam_K;
    const float* depth;
    uint32_t* box_support;
};

__global__ void __launch_bounds__(128) camera_depth_support_kernel(const SupportArgs a) {
    const int g = (int)((blockIdx.x * 128u + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (g >= a.n_boxes * a.n_cams) return;  // uniform per warp
    const int b = g / a.n_cams, c = g - b * a.n_cams;
    int lo = 0, hi = a.n_samples;  // the sample s with sample_box_off[s] <= b < sample_box_off[s + 1]
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (a.sample_box_off[mid] <= b) lo = mid; else hi = mid - 1;
    }
    const int s = lo;
    const size_t sc = (size_t)s * a.n_cams + c;
    uint8_t vis;
    float ext[4];
    double z[2];
    project_box_z<true>(a.boxes + (size_t)b * 10, a.cam_ego_pose + sc * 7, a.cam_calib + sc * 7, a.cam_K + sc * 9, (double)a.image_w,
                        (double)a.image_h, &vis, ext, z);
    uint32_t n_blocks = 0, n_hit = 0, n_front = 0, n_on = 0;
    if (vis) {
        const int bx0 = __float2int_rz(ext[0]) / a.ds, bx1 = min(__float2int_rz(ext[2]), a.image_w - 1) / a.ds;
        const int by0 = __float2int_rz(ext[1]) / a.ds, by1 = min(__float2int_rz(ext[3]), a.image_h - 1) / a.ds;
        n_blocks = (uint32_t)(bx1 - bx0 + 1) * (uint32_t)(by1 - by0 + 1);
        const double zf = z[0] - a.margin, zo = z[1] + a.margin;
        const float* img = a.depth + sc * (size_t)a.hb * (size_t)a.wb;
        for (int by = by0; by <= by1; ++by)
            for (int bx = bx0 + lane; bx <= bx1; bx += 32) {
                const float d = img[(size_t)by * a.wb + bx];
                if (d < INFINITY) {
                    ++n_hit;
                    if ((double)d < zf) ++n_front;
                    else if ((double)d <= zo) ++n_on;
                }
            }
        n_hit = __reduce_add_sync(0xffffffffu, n_hit);
        n_front = __reduce_add_sync(0xffffffffu, n_front);
        n_on = __reduce_add_sync(0xffffffffu, n_on);
    }
    if (lane == 0) {
        uint32_t* o = a.box_support + (size_t)g * 4;
        o[0] = n_blocks; o[1] = n_hit; o[2] = n_front; o[3] = n_on;
    }
}

}  // namespace msc

extern "C" {

int msc_camera_depth_batch(const msc_params* params, const msc_depth_params* dp, const msc_batch_in* in, const msc_depth_out* out,
                           void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(params && dp && in && out, "msc_camera_depth_batch: null argument");
    MSC_REQUIRE(dp->downsample >= 1, "msc_camera_depth_batch: downsample must be >= 1 (got %d)", (int)dp->downsample);
    MSC_REQUIRE(params->n_cams >= 1 && params->n_cams <= MSC_MAX_CAMS, "msc_camera_depth_batch: n_cams must be in 1..%d (got %d)",
                MSC_MAX_CAMS, (int)params->n_cams);
    MSC_REQUIRE(params->image_w > 2 && params->image_h > 2, "msc_camera_depth_batch: image_w and image_h must be > 2 (got %d x %d)",
                (int)params->image_w, (int)params->image_h);
    MSC_REQUIRE(params->image_w <= (1 << 24) && params->image_h <= (1 << 24), "msc_camera_depth_batch: image_w and image_h must be <= 2^24");
    MSC_REQUIRE(dp->min_dist >= 0.0f, "msc_camera_depth_batch: min_dist must be >= 0 (got %g)", (double)dp->min_dist);
    MSC_REQUIRE(dp->support_margin >= 0.0f, "msc_camera_depth_batch: support_margin must be >= 0 and not NaN (got %g)",
                (double)dp->support_margin);
    MSC_REQUIRE(in->n_samples >= 0 && in->n_boxes >= 0, "msc_camera_depth_batch: negative counts");
    if (in->n_samples == 0) return MSC_OK;
    MSC_REQUIRE(out->depth && out->cam_points, "msc_camera_depth_batch: depth and cam_points must not be NULL");
    MSC_REQUIRE(in->points && in->sample_sweep_off && in->sweep_start && in->sweep_count && in->sweep_pose && in->ego_pose &&
                    in->lidar_calib && in->cam_ego_pose && in->cam_calib && in->cam_K,
                "msc_camera_depth_batch: null input array");
    const bool support = out->box_support != nullptr && in->n_boxes > 0;
    MSC_REQUIRE(!support || (in->boxes && in->sample_box_off), "msc_camera_depth_batch: box_support needs boxes and sample_box_off");
    cudaStream_t stream = (cudaStream_t)stream_v;
    const int S = in->n_samples, C = params->n_cams, ds = dp->downsample;
    const int hb = (int)(((int64_t)params->image_h + ds - 1) / ds), wb = (int)(((int64_t)params->image_w + ds - 1) / ds);
    const size_t n_depth = (size_t)S * C * (size_t)hb * (size_t)wb;
    const int64_t hint = in->points_per_sample_hint > 0 ? in->points_per_sample_hint : 347200;  // 0: a 10-sweep sample
    const int X = (int)std::min<int64_t>(std::max<int64_t>((hint + kDepthPointsPerCta - 1) / kDepthPointsPerCta, 1), 4096);
    MSC_REQUIRE((int64_t)S * X <= 0x7fffffff, "msc_camera_depth_batch: too many samples for one call");

    const size_t fill_blocks = std::min<size_t>((n_depth + kDepthThreads - 1) / kDepthThreads, 148 * 16);
    camera_depth_fill_kernel<<<(unsigned)std::max<size_t>(fill_blocks, 1), kDepthThreads, 0, stream>>>(
        reinterpret_cast<uint32_t*>(out->depth), n_depth, out->cam_points, S * C);
    MSC_CUDA(cudaGetLastError());

    DepthArgs a;
    a.points = in->points; a.sample_sweep_off = in->sample_sweep_off; a.sweep_start = in->sweep_start; a.sweep_count = in->sweep_count;
    a.sweep_pose = in->sweep_pose; a.ego_pose = in->ego_pose; a.lidar_calib = in->lidar_calib; a.cam_ego_pose = in->cam_ego_pose;
    a.cam_calib = in->cam_calib; a.cam_K = in->cam_K;
    a.depth_bits = reinterpret_cast<uint32_t*>(out->depth); a.cam_points = out->cam_points;
    a.rc = params->remove_close_radius; a.min_dist = dp->min_dist;
    a.u_hi = (float)(params->image_w - 1); a.v_hi = (float)(params->image_h - 1);
    a.u_guard = 2.0f * (float)params->image_w; a.v_guard = 2.0f * (float)params->image_h;
    a.n_cams = C; a.ds = ds; a.hb = hb; a.wb = wb; a.ctas_per_sample = X;
    camera_depth_kernel<<<(unsigned)(S * X), kDepthThreads, 0, stream>>>(a);
    MSC_CUDA(cudaGetLastError());

    if (support) {
        MSC_REQUIRE((int64_t)in->n_boxes * C <= 0x7fffffff / 32, "msc_camera_depth_batch: too many boxes for one call");
        SupportArgs sa;
        sa.n_samples = S; sa.n_boxes = in->n_boxes; sa.n_cams = C; sa.ds = ds; sa.hb = hb; sa.wb = wb;
        sa.image_w = params->image_w; sa.image_h = params->image_h; sa.margin = (double)dp->support_margin;
        sa.sample_box_off = in->sample_box_off; sa.boxes = in->boxes; sa.cam_ego_pose = in->cam_ego_pose; sa.cam_calib = in->cam_calib;
        sa.cam_K = in->cam_K; sa.depth = out->depth; sa.box_support = out->box_support;
        const int warps = in->n_boxes * C;
        camera_depth_support_kernel<<<(warps + 3) / 4, 128, 0, stream>>>(sa);
        MSC_CUDA(cudaGetLastError());
    }
    return MSC_OK;
}

}  // extern "C"
