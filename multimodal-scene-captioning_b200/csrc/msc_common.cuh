// msc_common.cuh -- shared device/host helpers for libmsc_geom (sm_100a only).
//
// Arithmetic contract (DESIGN.md "exact arithmetic"): every .cu in this directory is compiled with
// -fmad=false, so + - * / sqrt are single IEEE-754 round-to-nearest operations and a fused
// multiply-add exists only where __fma_rn / __fmaf_rn is written.  That is what makes integer outputs
// (counts, flags, cells, categories) bit-identical to the scalar definition of the path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/msc_geom.h"

namespace msc {

// ---------------------------------------------------------------- host-side error plumbing
void set_error(const char* fmt, ...);
#define MSC_REQUIRE(cond, ...)                \
    do {                                      \
        if (!(cond)) {                        \
            msc::set_error(__VA_ARGS__);      \
            return MSC_ERR_BAD_ARGUMENT;      \
        }                                     \
    } while (0)
#define MSC_CUDA(call)                                                                      \
    do {                                                                                    \
        cudaError_t e__ = (call);                                                           \
        if (e__ != cudaSuccess) {                                                           \
            msc::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return MSC_ERR_LAUNCH;                                                          \
        }                                                                                   \
    } while (0)

// ---------------------------------------------------------------- mbarrier + bulk-copy (TMA) PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_parity(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "MSC_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra MSC_DONE_%=;\n"
        "bra MSC_WAIT_%=;\n"
        "MSC_DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// L2 eviction policy for data that is read exactly once (the raw sweeps).
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// 1-D bulk asynchronous copy global -> shared (TMA unit; SASS UBLKCP), completion on an mbarrier.
// dst/src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

// ---------------------------------------------------------------- f64 pose algebra (no FMA; see header)
// unit quaternion (w,x,y,z) -> row-major rotation, normalising first
__device__ __forceinline__ void quat_to_rot(const double* __restrict__ q, double R[9]) {
    double w = q[0], x = q[1], y = q[2], z = q[3];
    double n = sqrt(((w * w + x * x) + y * y) + z * z);
    w = w / n; x = x / n; y = y / n; z = z / n;
    double xx = x * x, yy = y * y, zz = z * z, xy = x * y, xz = x * z, yz = y * z, wx = w * x, wy = w * y, wz = w * z;
    R[0] = 1.0 - 2.0 * (yy + zz); R[1] = 2.0 * (xy - wz);       R[2] = 2.0 * (xz + wy);
    R[3] = 2.0 * (xy + wz);       R[4] = 1.0 - 2.0 * (xx + zz); R[5] = 2.0 * (yz - wx);
    R[6] = 2.0 * (xz - wy);       R[7] = 2.0 * (yz + wx);       R[8] = 1.0 - 2.0 * (xx + yy);
}
// devkit Box.translate(-t); Box.rotate(q^-1): c <- R(q)^T (c - t), R <- R(q)^T R
__device__ __forceinline__ void frame_change(const double* __restrict__ pose7, double c[3], double R[9]) {
    double P[9];
    quat_to_rot(pose7 + 3, P);
    double d0 = c[0] - pose7[0], d1 = c[1] - pose7[1], d2 = c[2] - pose7[2];
    c[0] = (P[0] * d0 + P[3] * d1) + P[6] * d2;
    c[1] = (P[1] * d0 + P[4] * d1) + P[7] * d2;
    c[2] = (P[2] * d0 + P[5] * d1) + P[8] * d2;
    double T[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int k = 0; k < 3; ++k) T[r * 3 + k] = (P[0 * 3 + r] * R[0 * 3 + k] + P[1 * 3 + r] * R[1 * 3 + k]) + P[2 * 3 + r] * R[2 * 3 + k];
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = T[k];
}

// BEV cell index (lidar_agent.py:547-552): clip(trunc((c + r) / (2r) * res), 0, res-1), float32 steps
__device__ __forceinline__ int bev_index(float c, float r, float two_r, float resf, int res_m1) {
    float t = __fmul_rn(__fdiv_rn(__fadd_rn(c, r), two_r), resf);
    int i = __float2int_rz(t);
    return min(max(i, 0), res_m1);
}

// 4-way bearing bins of scenegraph_agent.py:194-201 as exact predicates (0 front, 1 left, 2 back, 3 right)
// At the origin the reference's atan2 follows the sign of dx: (-0, +-0) is +-180 degrees (left), (+0, +-0) is 0 (right).
__device__ __forceinline__ uint8_t bearing4(double dx, double dy) {
    if (dx == 0.0 && dy == 0.0) return signbit(dx) ? 1 : 3;
    if (dy > 0.0 && dx <= dy && -dx < dy) return 0;
    if (dx < 0.0 && dy <= -dx && dy > dx) return 1;
    if (dy < 0.0 && dx >= dy && dx < -dy) return 2;
    return 3;
}

// box -> camera projection of one (box, camera) pair, devkit box_in_image(BoxVisibility.ANY) (App. A.3)
__device__ __forceinline__ void project_box(const double* __restrict__ box, const double* __restrict__ cam_ego_pose,
                                            const double* __restrict__ cam_calib, const double* __restrict__ K,
                                            double W, double H, uint8_t* visible, float* extent4) {
    double c[3] = {box[0], box[1], box[2]};
    double R[9];
    quat_to_rot(box + 6, R);
    frame_change(cam_ego_pose, c, R);
    frame_change(cam_calib, c, R);
    const double hl = box[4] / 2.0, hw = box[3] / 2.0, hh = box[5] / 2.0;
    bool any_vis = false, all_front = true;
    double umin = INFINITY, vmin = INFINITY, umax = -INFINITY, vmax = -INFINITY;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const double lx = (k < 4) ? hl : -hl;
        const double ly = (k == 0 || k == 3 || k == 4 || k == 7) ? hw : -hw;
        const double lz = (k == 0 || k == 1 || k == 4 || k == 5) ? hh : -hh;
        double X = ((R[0] * lx + R[1] * ly) + R[2] * lz) + c[0];
        double Y = ((R[3] * lx + R[4] * ly) + R[5] * lz) + c[1];
        double Z = ((R[6] * lx + R[7] * ly) + R[8] * lz) + c[2];
        double pu = (K[0] * X + K[1] * Y) + K[2] * Z;
        double pv = (K[3] * X + K[4] * Y) + K[5] * Z;
        double pw = (K[6] * X + K[7] * Y) + K[8] * Z;
        double u = pu / pw, v = pv / pw;
        if ((u > 0.0) && (u < W) && (v > 0.0) && (v < H) && (Z > 1.0)) any_vis = true;
        if (!(Z > 0.1)) all_front = false;
        if (u < umin) umin = u;
        if (u > umax) umax = u;
        if (v < vmin) vmin = v;
        if (v > vmax) vmax = v;
    }
    bool ok = any_vis && all_front;
    *visible = ok ? 1 : 0;
    if (ok) {
        if (umin < 0.0) umin = 0.0;
        if (vmin < 0.0) vmin = 0.0;
        if (umax > W) umax = W;
        if (vmax > H) vmax = H;
        extent4[0] = (float)umin; extent4[1] = (float)vmin; extent4[2] = (float)umax; extent4[3] = (float)vmax;
    } else {
        extent4[0] = extent4[1] = extent4[2] = extent4[3] = 0.0f;
    }
}

}  // namespace msc
