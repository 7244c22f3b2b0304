// fused_common.cuh -- types and device helpers shared by the table kernels (fused_evidence.cu) and the two streaming kernels
// (stream4.cu: config 10, the default; fused_stream.cu: config 7, the TMA-ring generation, which also serves fov_keep_mask != 0).
#pragma once
#include "msc_common.cuh"

namespace msc {

constexpr int kBoxStride = 20;      // floats per box record: 80 B stride makes the four LDS.128 conflict-free

constexpr uint32_t kCullEmpty = 0xffffffffu;  // no candidate box in this cell
constexpr uint32_t kCullAll = 0xfefefefeu;    // more than four boxes touch the cell: test every box
constexpr int kAccWords = 9;                  // per-box accumulators: count, min s, 3 axis words, 3 carry words, pad; the odd
                                              // stride spreads the same word of different boxes over all 32 banks
constexpr int kMaxWarps = 32;
constexpr int kInnerMax = 50;  // fused_stream.cu: side of the fine (one BEV cell) edge-class grid around the sensor

struct FusedLayout {  // byte offsets into dynamic smem, computed on the host
    int32_t tiles_off, window_off, cull_off, boxp_off, boxacc_off, misc_off, queue_off, total_bytes;
    int32_t win_w, win_lo;         // window covers cells [win_lo, win_lo + win_w) in x and y
    int32_t cull_dim, cull_shift;  // cull cell = BEV cell >> cull_shift
    int32_t inner_off, inner_dim, inner_lo;  // fused_stream.cu: edge classes per BEV cell for cells [inner_lo, inner_lo + inner_dim)^2 (0: none)
    int32_t max_boxes;             // capacity of the smem box tables
    int32_t pcnt_off, isum_delta;  // stream4.cu: bytes from the window region's start to the cull-cell count words / from array A to array B
    int32_t win_stride;            // stream4.cu: words between window rows (win_w + 1: odd, so rays along y do not pile up in one bank)
};

struct FusedArgs {
    msc_params P;
    msc_batch_in in;
    msc_batch_out out;
    FusedLayout L;
    // host-precomputed scalars (exact): 2r, res, RN(1/2r), 2^centroid_shift, 2^intensity_shift
    float two_r, resf, rcp_two_r, cscale, iscale;
    int32_t centroid_bias;  // 2^(centroid_shift + 6): makes the quantised coordinate non-negative
    int32_t pad_;           // (unused; it keeps the parameter offsets of the members below, and ptxas schedules the PPT = 4 main loops of
                            // stream4.cu differently when they move)
    // Replicas of the small result tables (per-box tables, projection tables, stats): the kernels that produce a value also store it
    // through these pointers -- peer-mapped (symmetric) memory of the other GPUs of the box -- so the "gather" of a sharded batch is
    // part of the producing kernels (P2P stores over NVLink / NVSwitch), not a collective after them.  bev_* members are ignored.
    int32_t n_replicas;
    msc_batch_out replica[MSC_MAX_REPLICAS];
};

// Packed pairs of f32 (Blackwell FADD2 / FMUL2 / FFMA2: two IEEE round-to-nearest operations per lane and issue slot; each half is
// bit-identical to the scalar instruction, so the arithmetic contract of msc_common.cuh is unchanged).
__device__ __forceinline__ unsigned long long f2_pack(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2_unpack(unsigned long long v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ unsigned long long f2_add(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long f2_mul(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long f2_fma(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
// ---------------------------------------------------------------- shared-memory, mbarrier and bulk-copy (TMA) PTX
// Every address is a 32-bit shared-state-space address: both streaming kernels derive theirs from one opaque base register, so their
// loops carry no generic-address arithmetic.
__device__ __forceinline__ uint32_t lds8(uint32_t saddr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t saddr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t saddr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(saddr));
    return v;
}
__device__ __forceinline__ float4 lds128(uint32_t saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void lds_f64x2(uint32_t saddr, double& a, double& b) {
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(a), "=d"(b) : "r"(saddr));
}
__device__ __forceinline__ void red_shared_add(uint32_t saddr, uint32_t v) {
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t atom_shared_add(uint32_t saddr, uint32_t v) {
    uint32_t old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(saddr), "r"(v) : "memory");
    return old;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait_parity(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "MSC_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra MSC_DONE_%=;\n"
        "bra MSC_WAIT_%=;\n"
        "MSC_DONE_%=:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// L2 eviction policy for data that is read exactly once (the raw sweeps).
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// 1-D bulk asynchronous copy global -> shared (TMA unit; SASS UBLKCP) of `bytes` (a multiple of 16; both addresses 16-byte aligned),
// announced on mbarrier `bar` first, whose phase completes when the bytes have landed.  One lane issues it.
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar), "l"(policy)
                 : "memory");
}

// ---------------------------------------------------------------- pieces both streaming kernels share
// One point of box accumulators acc_s (kAccWords words): count, min s^2 (es2 bits: non-negative floats order as unsigned), and the
// biased fixed-point coordinates.  Centroid sums are one 32-bit word per axis plus a carry word that takes a rare second atomic when
// the word wraps (the coordinate is a 24-bit value, so that is at most once per 256 points): order-independent integers.
__device__ __forceinline__ void box_accumulate(uint32_t acc_s, uint32_t es2, uint32_t fx, uint32_t fy, uint32_t fz) {
    red_shared_add(acc_s, 1u);
    asm volatile("red.shared.min.u32 [%0], %1;" ::"r"(acc_s + 4u), "r"(es2) : "memory");
    const uint32_t ox = atom_shared_add(acc_s + 8u, fx), oy = atom_shared_add(acc_s + 12u, fy), oz = atom_shared_add(acc_s + 16u, fz);
    if (ox > ~fx) red_shared_add(acc_s + 20u, 1u);
    if (oy > ~fy) red_shared_add(acc_s + 24u, 1u);
    if (oz > ~fz) red_shared_add(acc_s + 28u, 1u);
}
// Centroid coordinate of a box with cnt > 0 member points from the biased 64-bit sum of its fixed-point coordinates: exact integers and
// one f64 division, which makes it bit-identical to the scalar definition.  (A box without members has the centroid 0 and the nearest
// distance +inf.)
__device__ __forceinline__ float box_centroid(const FusedArgs& A, uint32_t cnt, unsigned long long biased) {
    const long long sum = (long long)biased - (long long)cnt * (long long)A.centroid_bias;
    return (float)((double)sum / ((double)cnt * (double)A.cscale));
}
// Zero-fill one sample's global BEV layers: ncell (count, isum) pairs and ncell max heights, 16-byte stores by `nthreads` threads.
__device__ __forceinline__ void zero_bev_layers(uint32_t* ci, float* h, size_t ncell, uint32_t tid, uint32_t nthreads) {
    uint4* c4 = reinterpret_cast<uint4*>(ci);
    for (size_t i = tid; i < ncell / 2; i += nthreads) c4[i] = make_uint4(0, 0, 0, 0);
    uint4* h4 = reinterpret_cast<uint4*>(h);
    for (size_t i = tid; i < ncell / 4; i += nthreads) h4[i] = make_uint4(0, 0, 0, 0);
}
// Edge-table entry (apex.x, apex.y, a, b) of one edge of camera wedge wq (in_wedge's form): q = p - apex, the point passes iff
// fma(a, q.y, -(b * q.x)) >= 0, with (a, b) = (w4, w5) for the right edge and (-w2, -w3) for the left one.
__device__ __forceinline__ float4 wedge_edge_entry(const float* wq, bool left) {
    float4 E;
    E.x = wq[0]; E.y = wq[1];
    if (left) { E.z = -wq[2]; E.w = -wq[3]; } else { E.z = wq[4]; E.w = wq[5]; }
    return E;
}
// Camera c's 8-bit counter of a pair of byte-counter words (cam_lo: cameras 0-3, cam_hi: 4-7).
__device__ __forceinline__ uint32_t cam_byte(uint32_t cam_lo, uint32_t cam_hi, int c) { return ((c < 4 ? cam_lo : cam_hi) >> ((c & 3) * 8)) & 0xffu; }

struct TableLayout {  // offsets (bytes) into the workspace
    size_t counter_off, boxprep_off, wedge_off, cullids_off;
    size_t boxscr_off, splitstats_off;  // merge scratch of samples processed in parts: per-box (count | min << 32, 3 biased sums) u64 x 4, per-sample stats + ticket
    size_t tileoff_off;                 // stream4.cu: [n_samples + 1] exclusive prefix of warp tiles per sample
    size_t cls_off;                     // stream4.cu: per-CTA class words, [max CTAs][cull_dim^2 + kInnerMax^2] u32
    size_t total;
};

// fused_stream.cu (config 7): launch shape (1024 threads x 2 points per lane), shared-memory layout (win_w < 0: does not fit), launcher
constexpr int kStreamThreads = 1024, kStreamTilePts = 64;
FusedLayout stream_layout(int smem_bytes, int res, int cull_dim, int cull_shift, int box_cap, int opt_window, int inner_dim);
int launch_stream_kernel(const FusedArgs& args, const TableLayout& T, unsigned char* ws, int grid, bool fov, bool fast, cudaStream_t stream);
// stream4.cu (config 10)
int stream4_threads(int ppt);
FusedLayout stream4_layout(int smem_bytes, int ppt, int res, int cull_dim, int cull_shift, int box_cap, int opt_window, int inner_dim);
bool stream4_is_standard(const FusedArgs& a, int smem_bytes, int ppt, int opt_window);
int stream4_std_boxes();
int launch_stream4_partition(const FusedArgs& args, const TableLayout& T, unsigned char* ws, int grid, cudaStream_t stream, int* launches);
int launch_stream4_kernel(const FusedArgs& args, const TableLayout& T, unsigned char* ws, int grid, int ppt, bool fov, bool fast, bool standard,
                          cudaStream_t stream);

// Per-edge classes of one cell against one wedge: bit0 = the wedge may contain points of the cell,
// bit1 = the right edge is undecided inside the cell, bit2 = the left edge is.  Same extremes over the cell and the same guard band
// as classify_cell(); an edge every point of the cell passes needs no exact test, an edge every point fails empties the wedge.
__device__ __forceinline__ uint32_t classify_cell_edges(const float* __restrict__ wq, float x0, float x1, float y0, float y1) {
    // both cross products are affine in (x, y): over the rectangle they range over (value at the centre) -/+ (extent), which costs a
    // third of four corner evaluations.  The float evaluation error of the exact test is < 1e-4 for |p| < 128 m and << guard for |p|
    // up to the 1200 m "absorbing" edge cells, far inside the 2e-3 guard band.
    const float guard = 2e-3f;
    const float hx = 0.5f * (x1 - x0), hy = 0.5f * (y1 - y0);
    const float qx = 0.5f * (x0 + x1) - wq[0], qy = 0.5f * (y0 + y1) - wq[1];
    const float cr = wq[4] * qy - wq[5] * qx, cr_e = fabsf(wq[4]) * hy + fabsf(wq[5]) * hx;
    const float cl = qx * wq[3] - qy * wq[2], cl_e = fabsf(wq[3]) * hx + fabsf(wq[2]) * hy;
    if (cr + cr_e < -guard || cl + cl_e < -guard) return 0u;  // outside
    return 1u | ((cr - cr_e > guard) ? 0u : 2u) | ((cl - cl_e > guard) ? 0u : 4u);
}

// Class word of entry i of a sample's class tables (i < cull_dim^2: cull cell i; beyond: fine cell i - cull_dim^2, one BEV cell of the
// inner_dim x inner_dim square around the sensor), from the sample's camera wedges wq[MSC_MAX_CAMS][6] (any address space):
// bit c = camera c's wedge may contain points of the cell, bit 8 + c = its right edge is undecided inside the cell, bit 16 + c = its left
// edge is.  Every point whose bev_cell() index falls in the cell lies in the padded rectangle; first / last cells absorb what is clipped
// into them.  Both streaming kernels evaluate this per sample in their prologue (5,000 cells x 6 cameras: < 1 % of a sample's work).
__device__ __forceinline__ uint32_t edge_class_word(const FusedArgs& A, const float* __restrict__ wq, int i) {
    const msc_params& P = A.P;
    const int ncc = A.L.cull_dim * A.L.cull_dim;
    const float big = 4.0f * P.bev_range + 1000.0f, pad = 2e-3f;
    float x0, x1, y0, y1;
    if (i >= ncc) {
        const int j = i - ncc, jy = j / A.L.inner_dim, jx = j - jy * A.L.inner_dim;
        const float cell_b = A.two_r / A.resf;
        const int ix = A.L.inner_lo + jx, iy = A.L.inner_lo + jy, last_b = P.bev_res - 1;
        x0 = (ix == 0) ? -big : (-P.bev_range + (float)ix * cell_b - pad); x1 = (ix == last_b) ? big : (-P.bev_range + (float)(ix + 1) * cell_b + pad);
        y0 = (iy == 0) ? -big : (-P.bev_range + (float)iy * cell_b - pad); y1 = (iy == last_b) ? big : (-P.bev_range + (float)(iy + 1) * cell_b + pad);
    } else {
        const int gy = i / A.L.cull_dim, gx = i - gy * A.L.cull_dim;
        const float cell_m = (A.two_r / A.resf) * (float)(1 << A.L.cull_shift);
        const int last = A.L.cull_dim - 1;
        x0 = (gx == 0) ? -big : (-P.bev_range + (float)gx * cell_m - pad); x1 = (gx == last) ? big : (-P.bev_range + (float)(gx + 1) * cell_m + pad);
        y0 = (gy == 0) ? -big : (-P.bev_range + (float)gy * cell_m - pad); y1 = (gy == last) ? big : (-P.bev_range + (float)(gy + 1) * cell_m + pad);
    }
    uint32_t eb = 0;
    for (int c = 0; c < P.n_cams; ++c) {
        const uint32_t k = classify_cell_edges(wq + c * 6, x0, x1, y0, y1);
        eb |= ((k & 1u) << c) | (((k >> 1) & 1u) << (8 + c)) | (((k >> 2) & 1u) << (16 + c));  // in-bit, right / left edge undecided
    }
    return eb;
}

// exact wedge test (the definition): q = p - apex, cross(e_right, q) >= 0 and cross(q, e_left) >= 0
__device__ __forceinline__ bool in_wedge(const float* __restrict__ wq, float x, float y) {
    const float qx = __fsub_rn(x, wq[0]), qy = __fsub_rn(y, wq[1]);
    const float cr = __fmaf_rn(wq[4], qy, -__fmul_rn(wq[5], qx));
    const float cl = __fmaf_rn(-wq[2], qy, __fmul_rn(wq[3], qx));  // same shape as cr: product on the x term, fma on the y term
    return (cr >= 0.0f) && (cl >= 0.0f);
}

// Conservative oriented rasterisation of a prepared box's xy footprint (a zonotope spanned by the projected edge
// vectors) into the cull grid.  Every member point lies in the corner hull up to float rounding (<< the 2 mm
// margin) and bev_cell() is monotonic, so a member can never fall in an unmarked cell.
// cull_words: first id word of cell 0; STRIDE words between cells (2: the smem (ids, classes) pairs, 1: the workspace id table).
// The cells of the box's bounding rectangle are dealt round-robin to `nworkers` callers (worker = 0 .. nworkers - 1).
template <int STRIDE>
static __device__ __noinline__ void rasterise_box(const FusedArgs& A, const float* __restrict__ o, int b, uint32_t* __restrict__ cull_words,
                                                  int worker = 0, int nworkers = 1) {
    const msc_params& P = A.P;
    const FusedLayout& L = A.L;
    const float margin = 2e-3f;
    const float cx = o[16], cy = o[17];
    const float ex[3] = {o[3], o[6], o[9]}, ey[3] = {o[4], o[7], o[10]};
    const float rx = 0.5f * (fabsf(ex[0]) + fabsf(ex[1]) + fabsf(ex[2])) + margin;
    const float ry = 0.5f * (fabsf(ey[0]) + fabsf(ey[1]) + fabsf(ey[2])) + margin;
    const int res_m1 = P.bev_res - 1;
    const int cx0 = bev_cell<false>(cx - rx, P.bev_range, A.two_r, A.rcp_two_r, A.resf, res_m1) >> L.cull_shift;
    const int cx1 = bev_cell<false>(cx + rx, P.bev_range, A.two_r, A.rcp_two_r, A.resf, res_m1) >> L.cull_shift;
    const int cy0 = bev_cell<false>(cy - ry, P.bev_range, A.two_r, A.rcp_two_r, A.resf, res_m1) >> L.cull_shift;
    const int cy1 = bev_cell<false>(cy + ry, P.bev_range, A.two_r, A.rcp_two_r, A.resf, res_m1) >> L.cull_shift;
    const float cell_m = (A.two_r / A.resf) * (float)(1 << L.cull_shift);
    const int last = L.cull_dim - 1;
    const int nx_cells = cx1 - cx0 + 1, n_cells = nx_cells * (cy1 - cy0 + 1);
    for (int ci = worker; ci < n_cells; ci += nworkers) {
        {
            const int gy = cy0 + ci / nx_cells, gx = cx0 + ci % nx_cells;
            // edge cells absorb everything clipped into them: never reject those
            bool reject = false;
            if (gx > 0 && gx < last && gy > 0 && gy < last) {
                const float mx = -P.bev_range + ((float)gx + 0.5f) * cell_m, my = -P.bev_range + ((float)gy + 0.5f) * cell_m;
                const float dx = cx - mx, dy = cy - my;
                const float hc = 0.5f * cell_m + margin;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float nx = -ey[k], ny = ex[k];  // normal of projected edge k
                    const float nn = fabsf(nx) + fabsf(ny);
                    if (nn > 1e-6f) {
                        const float dist = fabsf(dx * nx + dy * ny);
                        float rb = 0.0f;
#pragma unroll
                        for (int j = 0; j < 3; ++j) rb += 0.5f * fabsf(ex[j] * nx + ey[j] * ny);
                        if (dist > (rb + hc * nn) * 1.0001f + margin * nn) reject = true;
                    }
                }
            }
            if (reject) continue;
            uint32_t* slot = cull_words + (size_t)(gy * L.cull_dim + gx) * STRIDE;
            for (;;) {
                const uint32_t old = *reinterpret_cast<volatile uint32_t*>(slot);
                if (old == kCullAll) break;
                uint32_t nw = kCullAll;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (nw == kCullAll && ((old >> (8 * k)) & 0xffu) == 0xffu) nw = (old & ~(0xffu << (8 * k))) | ((uint32_t)b << (8 * k));
                if (atomicCAS(slot, old, nw) == old) break;
            }
        }
    }
}

// Prepared box record o[kBoxStride] (App. A.2) of a box already moved into the sensor frame -- centre c and rotation R, f64 without FMA
// from the global frame through ego_pose (frame_change) and lidar_calib (frame_change) -- with box = center3, size (w, l, h), quat: the
// devkit points_in_box vectors rounded to f32 (corner 0, the three edge vectors, their squared lengths) and the centre, for the cull
// rasterisation.  fused_tables_kernel and csrc/cluster_match.cu share it; the frame changes stay at the call sites, because
// fused_tables_kernel's instruction schedule changes when they move into a helper.
__device__ __forceinline__ void box_record(const double* box, const double c[3], const double R[9], float* o) {
    const double w = box[3], l = box[4], h = box[5];
    const double hl = l / 2.0, hw = w / 2.0, hh = h / 2.0;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        o[r] = (float)(((R[r * 3 + 0] * hl + R[r * 3 + 1] * hw) + R[r * 3 + 2] * hh) + c[r]);
        o[3 + r] = (float)(-(l * R[r * 3 + 0]));
        o[6 + r] = (float)(-(w * R[r * 3 + 1]));
        o[9 + r] = (float)(-(h * R[r * 3 + 2]));
    }
    o[12] = __fmaf_rn(o[5], o[5], __fmaf_rn(o[4], o[4], __fmul_rn(o[3], o[3])));
    o[13] = __fmaf_rn(o[8], o[8], __fmaf_rn(o[7], o[7], __fmul_rn(o[6], o[6])));
    o[14] = __fmaf_rn(o[11], o[11], __fmaf_rn(o[10], o[10], __fmul_rn(o[9], o[9])));
    o[15] = 0.0f;
    o[16] = (float)c[0]; o[17] = (float)c[1]; o[18] = (float)c[2]; o[19] = 0.0f;
}

// A.2 exact membership test of one point against one prepared box (closed intervals, float32 with fmaf chains).
__device__ __forceinline__ bool box_contains(const float* __restrict__ boxp, int b, float xr, float yr, float zr) {
    const float4* bp = reinterpret_cast<const float4*>(boxp + b * kBoxStride);
    const float4 b0 = bp[0], b1 = bp[1], b2 = bp[2], b3 = bp[3];
    const float v0 = __fsub_rn(xr, b0.x), v1 = __fsub_rn(yr, b0.y), v2 = __fsub_rn(zr, b0.z);
    const float iv = __fmaf_rn(b1.y, v2, __fmaf_rn(b1.x, v1, __fmul_rn(b0.w, v0)));
    const float jv = __fmaf_rn(b2.x, v2, __fmaf_rn(b1.w, v1, __fmul_rn(b1.z, v0)));
    const float kv = __fmaf_rn(b2.w, v2, __fmaf_rn(b2.z, v1, __fmul_rn(b2.y, v0)));
    return iv >= 0.0f && iv <= b3.x && jv >= 0.0f && jv <= b3.y && kv >= 0.0f && kv <= b3.z;
}
}  // namespace msc
