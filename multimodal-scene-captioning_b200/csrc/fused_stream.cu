// fused_stream.cu -- second generation of the streaming kernel (launch shape "config" 7).  Superseded as the default by stream4.cu
// (config 10); it still serves fov_keep_mask != 0 (a FOV *filter* needs the per-point wedge classes before the BEV update) and is the
// shape every change to stream4.cu is compared with bit for bit (tools/sweep_configs.py).
//
// Same arithmetic, per point, as fused_evidence.cu (SURVEY.md App. A + lidar_agent.py:103-132, :547-560); what
// changed is the control structure, because the first generation was instruction-issue bound (ncu: 80 % of issue
// slots, 353 warp instructions per 32 points, 20 of 32 lanes active):
//   * the per-point phase after the transform is straight-line code: dropped / out-of-window points add into a per-lane
//     sink word instead of branching around the window atomics, and the rare periphery / max-height reductions share
//     one region whose base pointers are read back from smem;
//   * camera wedges are classified per EDGE and per cull cell: a point in a cell that straddles one image-column
//     ray evaluates that one cross product (one LDS.128), not both edges of the wedge from six scalar loads; the test
//     is branch-free, two rounds are peeled for all lanes and a loop takes the few points that need more;
//   * one tile cursor (the tile in flight) instead of separate producer / consumer cursors, 32-bit shared addresses
//     from one opaque base register, the warp index made warp-uniform for the compiler;
//   * candidate-box ids per cull cell come from a pre-kernel (fused_evidence.cu: fused_cullids_kernel), so the
//     per-sample prologue only copies tables; crowded cells ("test every box") go through the candidate queue.
// 530 warp instructions per 64-point warp tile instead of 706 (profiles/r1b_stream_evidence_ncu_full.txt).
#include "fused_common.cuh"

namespace msc {

constexpr int kStreamPoseSmem = 12;  // sweeps whose transforms are staged per sample; later ones use a per-warp slot

// Launch shape: NT threads = NT/32 warps; every warp owns two ring slots of 32*PPT points and a 64-entry candidate queue.
// POSE_REG keeps the current sweep's 3x4 f64 transform in registers (shapes with a 128-register budget).
template <int NT, int PPT, bool POSE_REG>
struct StreamShape {
    static constexpr int kThreads = NT, kWarps = NT / 32, kPts = PPT;
    static constexpr bool kPoseReg = POSE_REG;
    static constexpr int kTilePts = 32 * PPT;
    static constexpr int kTileFloats = kTilePts * 5;
    static constexpr int kTileBytes = kTilePts * 20;
    static constexpr int kRingBytes = kWarps * 2 * kTileBytes;
    static constexpr int kQueueBytes = kWarps * 64 * 16;
    static_assert(kTileBytes % 16 == 0 && kWarps <= kMaxWarps, "shape");
};

struct StreamMisc {  // small per-CTA state at misc_off
    uint64_t full_bar[kMaxWarps * 2];  // [warp][slot]: TMA bytes landed in that warp's ring slot
    float4 edge_pad;                   // the branch-free edge test of a point with nothing to test reads the entry before edge[0]
    float4 edge[2 * MSC_MAX_CAMS];     // [c] right edge, [8 + c] left edge of camera c: (apex.x, apex.y, A, B)
    uint32_t dummy[64];                // per-lane sink of the window updates of dropped / out-of-window points
    uint32_t stats[MSC_STATS_STRIDE];
    uint32_t sweep_start[kStreamPoseSmem], sweep_count[kStreamPoseSmem];
    int32_t sample;
    int32_t pad_[3];
    unsigned long long* ci64;           // this sample's (count, isum) layer as 64-bit cells, and its max-height layer:
    int* h32;                           // read back by the few lanes per warp that update the periphery
    double pose[kStreamPoseSmem * 12];  // this sample's 3x4 sweep transforms
    double wpose[kMaxWarps * 12];       // per-warp slot for sweeps beyond kStreamPoseSmem
    float wq[MSC_MAX_CAMS * 6];         // this sample's camera wedges (fused_tables_kernel), source of the per-cell edge classes
};

// launch shape: 1024 threads x 2 points per lane
using Shape0 = StreamShape<kStreamThreads, kStreamTilePts / 32, false>;

// Shared-memory layout (bytes): the warps' ring slots, their candidate queues, (box ids, edge classes) per cull cell, the box tables, the
// per-CTA state, the fine edge classes around the sensor, and last the BEV window of (count, isum) cells, the largest even side that fits.
FusedLayout stream_layout(int smem_bytes, int res, int cull_dim, int cull_shift, int box_cap, int opt_window, int inner_dim) {
    FusedLayout L{};
    L.cull_dim = cull_dim; L.cull_shift = cull_shift; L.max_boxes = box_cap < 1 ? 1 : box_cap;
    int off = 0;
    L.tiles_off = off; off += (Shape0::kRingBytes + 127) & ~127;
    L.queue_off = off; off += (Shape0::kQueueBytes + 127) & ~127;
    L.cull_off = off; off += (cull_dim * cull_dim * 8 + 127) & ~127;
    L.boxp_off = off; off += L.max_boxes * kBoxStride * 4;
    L.boxacc_off = off; off += L.max_boxes * kAccWords * 4; off = (off + 127) & ~127;
    L.misc_off = off; off += ((int)sizeof(StreamMisc) + 127) & ~127;
    L.inner_dim = inner_dim; L.inner_lo = (res - inner_dim) / 2;
    L.inner_off = off; off += (inner_dim * inner_dim * 4 + 127) & ~127;
    L.window_off = off;
    const int avail = smem_bytes - off;
    if (avail < 0) { L.win_w = -1; return L; }
    int w = 0;
    while ((w + 2) * (w + 2) * 8 <= avail && (w + 2) <= res) w += 2;
    if (opt_window > 0 && opt_window < w) w = opt_window & ~1;
    if (((res - w) / 2) & 1) w -= 2;  // keep win_lo even so flush rows stay 16-byte aligned
    if (w < 0) w = 0;
    L.win_w = w;
    L.win_lo = (res - w) / 2;
    L.total_bytes = off + w * w * 8;
    return L;
}

template <class C, bool FOV, bool FASTDIV, bool KEEPMASK>
__global__ void __launch_bounds__(C::kThreads, 1) stream_evidence_kernel(const __grid_constant__ FusedArgs A, const TableLayout T,
                                                                         unsigned char* __restrict__ ws) {
    constexpr int NT = C::kThreads, W = C::kWarps, PPT = C::kPts, TP = C::kTilePts, TF = C::kTileFloats;
    constexpr bool MREG = C::kPoseReg;
    extern __shared__ __align__(128) unsigned char smem[];
    const msc_params& P = A.P;
    const FusedLayout& L = A.L;
    uint2* const window = reinterpret_cast<uint2*>(smem + L.window_off);
    uint2* const cull = reinterpret_cast<uint2*>(smem + L.cull_off);            // .x box ids, .y edge classes
    float* const boxp = reinterpret_cast<float*>(smem + L.boxp_off);            // [max_boxes][kBoxStride]
    uint32_t* const boxacc = reinterpret_cast<uint32_t*>(smem + L.boxacc_off);  // [max_boxes][kAccWords]
    StreamMisc* const misc = reinterpret_cast<StreamMisc*>(smem + L.misc_off);
    uint32_t* const work_counter = reinterpret_cast<uint32_t*>(ws + T.counter_off);
    const float* const g_boxprep = reinterpret_cast<const float*>(ws + T.boxprep_off);
    const float* const g_wedges = reinterpret_cast<const float*>(ws + T.wedge_off);
    const uint32_t* const g_cullids = reinterpret_cast<const uint32_t*>(ws + T.cullids_off);

    const int tid = threadIdx.x, lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // warp-uniform as far as the compiler is concerned
    uint32_t smem_s = smem_u32(smem);
    asm volatile("" : "+r"(smem_s));  // opaque: one live register instead of a re-derived generic->shared conversion per use
    const uint32_t misc_s = smem_s + (uint32_t)L.misc_off;
    const uint32_t ring_s = smem_s + (uint32_t)L.tiles_off + (uint32_t)warp * (uint32_t)(2 * TF * 4);  // this warp's two slots
    const uint32_t bar_s = misc_s + (uint32_t)warp * 16u;                                               // its two mbarriers
    const uint32_t queue_s = smem_s + (uint32_t)L.queue_off + (uint32_t)warp * (64u * 16u);              // its candidate queue
    const uint32_t edge_s = misc_s + (uint32_t)offsetof(StreamMisc, edge);
    const uint32_t sink_s = misc_s + (uint32_t)offsetof(StreamMisc, dummy) + (uint32_t)lane * 8u;
    const uint32_t window_s = smem_s + (uint32_t)L.window_off;
    const float* const ring = reinterpret_cast<const float*>(smem + L.tiles_off) + (size_t)warp * (2 * TF);
    const int res = P.bev_res, res_m1 = P.bev_res - 1;
    const size_t ncell = (size_t)res * (size_t)res;
    const int n_cams = P.n_cams;
    const uint64_t policy = l2_policy_evict_first();
    uint32_t lt_mask = (1u << lane) - 1u;
    asm volatile("" : "+r"(lt_mask));  // keep it in its register (the compiler would re-derive it from %tid at every use)

    if (lane == 0) {
        mbar_init(smem_u32(&misc->full_bar[warp * 2 + 0]), 1);
        mbar_init(smem_u32(&misc->full_bar[warp * 2 + 1]), 1);
        mbar_fence_init();
    }
    uint32_t wk = 0;  // tiles this warp has consumed since launch: slot = wk & 1, mbarrier parity = (wk >> 1) & 1
    __syncthreads();

    for (;;) {
        // ------------------------------------------------------------ fetch a sample
        if (tid == 0) misc->sample = (int32_t)atomicAdd(work_counter, 1u);
        __syncthreads();
        const int sample = misc->sample;
        if (sample >= A.in.n_samples) break;

        const int sw0 = A.in.sample_sweep_off[sample], sw1 = A.in.sample_sweep_off[sample + 1];
        const int n_sw = sw1 - sw0;
        if (tid < kStreamPoseSmem && tid < n_sw) {
            misc->sweep_start[tid] = A.in.sweep_start[sw0 + tid];
            misc->sweep_count[tid] = A.in.sweep_count[sw0 + tid];
        }
        for (int i = tid; i < min(n_sw, kStreamPoseSmem) * 12; i += NT) misc->pose[i] = A.in.sweep_pose[(size_t)sw0 * 12 + i];
        if (tid < MSC_STATS_STRIDE) misc->stats[tid] = 0u;
        if (FOV && tid < MSC_MAX_CAMS * 6) misc->wq[tid] = g_wedges[(size_t)sample * MSC_MAX_CAMS * 6 + tid];
        if (tid == 0) {
            misc->ci64 = reinterpret_cast<unsigned long long*>(A.out.bev_ci) + (size_t)sample * ncell;
            misc->h32 = reinterpret_cast<int*>(A.out.bev_height) + (size_t)sample * ncell;
        }
        __syncthreads();

        // Warp `warp` owns tiles warp, warp + W, warp + 2W, ... of every sweep.  One cursor describes the tile in flight.
        int n_si = -1;
        uint32_t n_first = 0, n_cnt = 0, n_base = 0;
        auto next_tile = [&]() -> bool {
            n_first += (uint32_t)(W * TP);
            while (n_first >= n_cnt) {  // next sweep that still has a tile for this warp
                if (++n_si >= n_sw) return false;
                if (n_si < kStreamPoseSmem) { n_cnt = misc->sweep_count[n_si]; n_base = misc->sweep_start[n_si]; }
                else { n_cnt = A.in.sweep_count[sw0 + n_si]; n_base = A.in.sweep_start[sw0 + n_si]; }
                n_first = (uint32_t)(warp * TP);
            }
            return true;
        };
        auto issue = [&](uint32_t slot) {  // whole warp (uniform control flow); one lane talks to the TMA unit
            const uint32_t npts = min((uint32_t)TP, n_cnt - n_first);
            const uint32_t bytes = (npts * 20u + 15u) & ~15u;
            const float* src = A.in.points + ((size_t)n_base + n_first) * 5;
            if (lane == 0) bulk_load(ring_s + slot * (uint32_t)(TF * 4), src, bytes, bar_s + slot * 8u, policy);
        };
        bool more = next_tile();
        if (more) issue(wk & 1u);  // overlaps the prologue below

        // ------------------------------------------------------------ prologue: zero accumulators, copy tables to smem
        const int bx0 = A.in.sample_box_off[sample];
        int n_boxes = A.in.sample_box_off[sample + 1] - bx0;
        const bool box_overflow = n_boxes > L.max_boxes;  // caller under-declared max_boxes_per_sample
        if (box_overflow) n_boxes = L.max_boxes;
        const size_t cell_base = (size_t)sample * ncell;
        uint32_t* const g_ci = A.out.bev_ci + cell_base * 2;
        float* const g_h = A.out.bev_height + cell_base;
        {
            uint4* w4 = reinterpret_cast<uint4*>(window);
            const int n_w4 = (L.win_w * L.win_w * 8) / 16;
            for (int i = tid; i < n_w4; i += NT) w4[i] = make_uint4(0, 0, 0, 0);
            const int n_cull = L.cull_dim * L.cull_dim;
            const uint32_t* ids = g_cullids + (size_t)sample * n_cull;  // candidate boxes per cull cell (fused_cullids_kernel)
            // edge classes of the sample's camera wedges per cull cell, and per BEV cell around the sensor (fine table)
            for (int i = tid; i < n_cull; i += NT) cull[i] = make_uint2(ids[i], (FOV && n_cams > 0) ? edge_class_word(A, misc->wq, i) : 0u);
            if (FOV) {
                const int n_inner = L.inner_dim * L.inner_dim;
                uint32_t* inner = reinterpret_cast<uint32_t*>(smem + L.inner_off);
                for (int i = tid; i < n_inner; i += NT) inner[i] = edge_class_word(A, misc->wq, n_cull + i);
            }
            for (int i = tid; i < n_boxes * kAccWords; i += NT) boxacc[i] = ((i % kAccWords) == 1) ? 0x7f800000u : 0u;
            const float4* bsrc = reinterpret_cast<const float4*>(g_boxprep + (size_t)bx0 * kBoxStride);
            for (int i = tid; i < n_boxes * (kBoxStride / 4); i += NT) reinterpret_cast<float4*>(boxp)[i] = bsrc[i];
            if (FOV && tid < 2 * MSC_MAX_CAMS) {
                const int c = tid & (MSC_MAX_CAMS - 1);
                float4 E = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                if (c < n_cams) {
                    E = wedge_edge_entry(g_wedges + ((size_t)sample * MSC_MAX_CAMS + c) * 6, tid >= MSC_MAX_CAMS);
                }
                misc->edge[tid] = E;
                if (tid == 0) misc->edge_pad = E;
            }
            // zero-fill this sample's global layers (window cells are overwritten by the flush; filling them too
            // keeps the stores fully coalesced)
            zero_bev_layers(g_ci, g_h, ncell, tid, NT);
        }
        __threadfence();
        __syncthreads();

        // ------------------------------------------------------------ main loop: this warp's tiles, no cross-warp sync
        uint32_t c_close = 0, c_kept = 0, c_ground = 0;  // per-thread counters (flushed once per sample)
        uint32_t cam_lo = 0, cam_hi = 0;                 // eight 8-bit per-camera counters, spilled every <= 255 points
        uint32_t cam_pts = 0;
        uint32_t q_head = 0, q_tail = 0;  // warp-uniform (every lane derives them from the same ballots); < 32 pending between points
        // every lane tests one queued point against its candidate boxes; the (usually single) containing box is accumulated
        // once after the loop, a second containing box (overlapping annotations) inside it
        auto drain_queue = [&](uint32_t n_take) {
            const float4 e = lds128(queue_s + (((q_head + (uint32_t)lane) & 63u) << 4));
            if ((uint32_t)lane < n_take) {
                uint32_t ids = __float_as_uint(e.w);
                const float es2 = __fadd_rn(__fmul_rn(e.x, e.x), __fmul_rn(e.y, e.y));
                // box_accumulate() with the fixed-point coordinates evaluated once per point
                const uint32_t fx = (uint32_t)(__float2int_rn(__fmul_rn(e.x, A.cscale)) + A.centroid_bias);
                const uint32_t fy = (uint32_t)(__float2int_rn(__fmul_rn(e.y, A.cscale)) + A.centroid_bias);
                const uint32_t fz = (uint32_t)(__float2int_rn(__fmul_rn(e.z, A.cscale)) + A.centroid_bias);
                auto accumulate = [&](int b) {
                    box_accumulate(smem_s + (uint32_t)L.boxacc_off + (uint32_t)b * (uint32_t)(kAccWords * 4), __float_as_uint(es2), fx, fy, fz);
                };
                int hit = -1;
                if (ids == kCullAll) {  // crowded cell (more than four boxes): test every box
                    for (int b = 0; b < n_boxes; ++b)
                        if (box_contains(boxp, b, e.x, e.y, e.z)) {
                            if (hit >= 0) accumulate(b); else hit = b;
                        }
                } else {
                    do {
                        const int b = (int)(ids & 0xffu);
                        if (box_contains(boxp, b, e.x, e.y, e.z)) {
                            if (hit >= 0) accumulate(b); else hit = b;
                        }
                        ids = (ids >> 8) | 0xff000000u;
                    } while ((ids & 0xffu) != 0xffu);
                }
                if (hit >= 0) accumulate(hit);
            }
            q_head += n_take;
        };
        uint32_t pose_s = 0;
        int pose_si = -1;
        double M[MREG ? 12 : 1];
        while (more) {
            // ---- the tile in flight becomes the current one; its successor takes the slot consumed in the previous iteration
            const uint32_t npts = min((uint32_t)TP, n_cnt - n_first);
            if (n_si != pose_si) {
                pose_si = n_si;
                if (n_si < kStreamPoseSmem) {
                    pose_s = misc_s + (uint32_t)offsetof(StreamMisc, pose) + (uint32_t)n_si * 96u;
                } else {
                    __syncwarp();
                    if (lane < 12) misc->wpose[warp * 12 + lane] = A.in.sweep_pose[(size_t)(sw0 + n_si) * 12 + lane];
                    __syncwarp();
                    pose_s = misc_s + (uint32_t)offsetof(StreamMisc, wpose) + (uint32_t)warp * 96u;
                }
                if (MREG) {
#pragma unroll
                    for (int i = 0; i < 12; i += 2) lds_f64x2(pose_s + i * 8, M[MREG ? i : 0], M[MREG ? i + 1 : 0]);
                }
            }
            more = next_tile();
            if (more) issue((wk + 1u) & 1u);
            mbar_wait_parity(bar_s + (wk & 1u) * 8u, (wk >> 1) & 1u);
            const float* tp = ring + (wk & 1u) * TF + lane * 5;

            // ---- phase A: branch-free over the lane's points so their dependency chains interleave
            float xr[PPT], yr[PPT], zr[PPT], inten[PPT];
            bool keep[PPT];
            {
                double xd[PPT], yd[PPT], zd[PPT];
#pragma unroll
                for (int u = 0; u < PPT; ++u) {
                    const bool valid = (uint32_t)lane + (uint32_t)u * 32u < npts;
                    const float x = tp[u * 160 + 0], y = tp[u * 160 + 1], z = tp[u * 160 + 2];
                    inten[u] = tp[u * 160 + 3];
                    // A.1 remove_close (square, sweep's own sensor frame)
                    const bool close = (fabsf(x) < P.remove_close_radius) & (fabsf(y) < P.remove_close_radius);
                    keep[u] = valid & !close;
                    xd[u] = (double)x; yd[u] = (double)y; zd[u] = (double)z;
                    if (keep[u]) ++c_close;
                }
                __syncwarp();  // every lane has read its rows: the slot may be refilled at the top of the next iteration
                // A.1 f64 matrix x f32 point -> f32, one matrix row at a time
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    double m0, m1, m2, m3;
                    if (MREG) {
                        m0 = M[MREG ? r * 4 + 0 : 0]; m1 = M[MREG ? r * 4 + 1 : 0]; m2 = M[MREG ? r * 4 + 2 : 0]; m3 = M[MREG ? r * 4 + 3 : 0];
                    } else {
                        lds_f64x2(pose_s + r * 32, m0, m1);
                        lds_f64x2(pose_s + r * 32 + 16, m2, m3);
                    }
#pragma unroll
                    for (int u = 0; u < PPT; ++u) {
                        const float v = (float)__fma_rn(m0, xd[u], __fma_rn(m1, yd[u], __fma_rn(m2, zd[u], m3)));
                        if (r == 0) xr[u] = v; else if (r == 1) yr[u] = v; else zr[u] = v;
                    }
                }
            }
            uint32_t cand[PPT], cell[PPT], wc_s[PPT], in_bits[PPT], st[PPT];
#pragma unroll
            for (int u = 0; u < PPT; ++u) {
                // lidar_agent.py:106-110, sqrt-free (thresholds on s are exact, geometry.sqrt_thresholds)
                const float s2 = __fadd_rn(__fmul_rn(xr[u], xr[u]), __fmul_rn(yr[u], yr[u]));
                keep[u] = keep[u] && (s2 >= P.s_lo) && (s2 <= P.s_hi) && (zr[u] < P.z_max) && (zr[u] > P.z_min);
                // BEV cell, lidar_agent.py:547-552 (garbage for dropped points is clamped and never used)
                const int ix = bev_cell<FASTDIV>(xr[u], P.bev_range, A.two_r, A.rcp_two_r, A.resf, res_m1);
                const int iy = bev_cell<FASTDIV>(yr[u], P.bev_range, A.two_r, A.rcp_two_r, A.resf, res_m1);
                const uint32_t ce_s = smem_s + (uint32_t)L.cull_off + (uint32_t)(((iy >> L.cull_shift) * L.cull_dim + (ix >> L.cull_shift)) << 3);
                cand[u] = lds32(ce_s);
                if (FOV) {
                    // edge classes: from the fine grid (one BEV cell) around the sensor, where a 2 m cull cell is crossed by several
                    // image-column rays, else from the cull cell; one load either way
                    const uint32_t jx = (uint32_t)(ix - L.inner_lo), jy = (uint32_t)(iy - L.inner_lo);
                    const bool fine = jx < (uint32_t)L.inner_dim && jy < (uint32_t)L.inner_dim;
                    const uint32_t cls_s = fine ? smem_s + (uint32_t)L.inner_off + ((jy * (uint32_t)L.inner_dim + jx) << 2) : ce_s + 4u;
                    const uint32_t cls = lds32(cls_s);
                    in_bits[u] = cls & 0xffu;
                    st[u] = keep[u] ? (cls >> 8) : 0u;  // bit c: right edge of camera c undecided in this cell, bit 8 + c: left edge
                } else {
                    in_bits[u] = 0u; st[u] = 0u;
                }
                cell[u] = (uint32_t)iy * (uint32_t)res + (uint32_t)ix;
                const uint32_t wx = (uint32_t)(ix - L.win_lo), wy = (uint32_t)(iy - L.win_lo);
                const bool inwin = wx < (uint32_t)L.win_w && wy < (uint32_t)L.win_w;
                wc_s[u] = inwin ? window_s + ((wy * (uint32_t)L.win_w + wx) << 3) : 0u;  // 0: periphery, one 64-bit global RED
            }
            // ---- phase B: one exact cross product per image-column ray a point's cull cell straddles.  The test is branch-free
            // (a point with nothing left to test reads the table entry before edge[0] and clears no bit); one round covers
            // nearly every point, a loop takes the rest.
            if (FOV) {
                uint32_t pass[PPT];
                auto edge_test = [&](int u) {
                    const uint32_t sbits = st[u];
                    const uint32_t low = sbits & (0u - sbits);        // lowest set bit (0 if none)
                    const int e = 31 - __clz((int)low);               // its index; -1: nothing to test
                    st[u] = sbits ^ low;
                    const float4 E = lds128(edge_s + (uint32_t)(e * 16));
                    const float qx = __fsub_rn(xr[u], E.x), qy = __fsub_rn(yr[u], E.y);
                    const float cr = __fmaf_rn(E.z, qy, -__fmul_rn(E.w, qx));
                    if (!(cr >= 0.0f)) pass[u] &= ~low;
                };
#pragma unroll
                for (int u = 0; u < PPT; ++u) pass[u] = 0xffffu;
#pragma unroll
                for (int u = 0; u < PPT; ++u) edge_test(u);  // one round for every lane; with the fine grid a second ray is rare
                uint32_t left_over = 0;
#pragma unroll
                for (int u = 0; u < PPT; ++u) left_over |= st[u];
                while (left_over) {
                    left_over = 0;
#pragma unroll
                    for (int u = 0; u < PPT; ++u) { edge_test(u); left_over |= st[u]; }
                }
#pragma unroll
                for (int u = 0; u < PPT; ++u) in_bits[u] &= pass[u] & (pass[u] >> 8);  // a camera keeps its bit iff both of its edges passed
            }
            // ---- phase C: straight-line accumulation; dropped points update a per-lane sink word instead of branching
            uint32_t q[PPT];
            bool periphery = false;
#pragma unroll
            for (int u = 0; u < PPT; ++u) {
                if (FOV) {
                    if (!keep[u]) in_bits[u] = 0u;
                    // spread 8 bits into 8 byte counters (no carries: the multiplier's partial products do not overlap)
                    cam_lo += ((in_bits[u] & 0xfu) * 0x00204081u) & 0x01010101u;
                    cam_hi += ((in_bits[u] >> 4) * 0x00204081u) & 0x01010101u;
                    if (KEEPMASK && (in_bits[u] & P.fov_keep_mask) == 0u) keep[u] = false;  // fov_keep_mask != 0: a FOV filter, not only counts
                }
                if (keep[u]) ++c_kept;
                if (keep[u] && zr[u] < P.ground_z) ++c_ground;  // lidar_agent.py:128
                // Q8 intensity, clamp [0, 65535]; NaN -> 0
                q[u] = min(__float2uint_rn(__fmul_rn(inten[u], A.iscale)), 65535u);  // the conversion saturates at 0 and maps NaN to 0
                const bool to_window = keep[u] && wc_s[u] != 0u;
                const uint32_t wa = to_window ? wc_s[u] : sink_s;
                red_shared_add(wa, 1u);
                red_shared_add(wa + 4u, q[u]);
                periphery = periphery || (keep[u] && (wc_s[u] == 0u || zr[u] > 0.0f));
                if (!keep[u]) cand[u] = kCullEmpty;
            }
            if (periphery) {  // a few lanes per warp: cells outside the window (one 64-bit RED) and the max-height layer (z > 0 only)
                unsigned long long* const ci64 = *reinterpret_cast<unsigned long long* volatile*>(&misc->ci64);
                int* const h32 = *reinterpret_cast<int* volatile*>(&misc->h32);
#pragma unroll
                for (int u = 0; u < PPT; ++u) {
                    if (keep[u] && wc_s[u] == 0u)
                        asm volatile("red.global.add.u64 [%0], %1;" ::"l"(ci64 + cell[u]), "l"(1ull | ((unsigned long long)q[u] << 32)) : "memory");
                    if (keep[u] && zr[u] > 0.0f)  // :560, 0-initialised max
                        asm volatile("red.global.max.s32 [%0], %1;" ::"l"(h32 + cell[u]), "r"(__float_as_int(zr[u])) : "memory");
                }
            }
            // ---- phase D: points that have candidate boxes go to this warp's queue; whenever 32 are pending every lane tests
            // one of them (dense), instead of a handful of lanes looping while the rest of the warp idles
#pragma unroll
            for (int u = 0; u < PPT; ++u) {
                const bool has = cand[u] != kCullEmpty;
                const uint32_t m = __ballot_sync(0xffffffffu, has);
                if (has) {
                    const uint32_t slot = (q_tail + __popc(m & lt_mask)) & 63u;
                    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(queue_s + (slot << 4)), "f"(xr[u]), "f"(yr[u]), "f"(zr[u]),
                                 "f"(__uint_as_float(cand[u]))
                                 : "memory");
                }
                q_tail += __popc(m);
                if (q_tail - q_head >= 32u) {
                    __syncwarp();  // the entries stored above are visible to the lanes that test them
                    drain_queue(32u);
                }
            }
            ++wk;
            if (FOV) {
                cam_pts += PPT;
                if (cam_pts > 255u - PPT) {  // spill the byte counters before any of them can wrap
#pragma unroll
                    for (int c = 0; c < MSC_MAX_CAMS; ++c) {
                        const uint32_t v = cam_byte(cam_lo, cam_hi, c);
                        if (v) atomicAdd(&misc->stats[5 + c], v);
                    }
                    cam_lo = cam_hi = cam_pts = 0;
                }
            }
        }
        while (q_tail != q_head) {
            __syncwarp();
            drain_queue(min(q_tail - q_head, 32u));
        }

        // ------------------------------------------------------------ epilogue
        {
            uint32_t v[3 + MSC_MAX_CAMS];
            v[0] = c_close; v[1] = c_kept; v[2] = c_ground;
#pragma unroll
            for (int c = 0; c < MSC_MAX_CAMS; ++c) v[3 + c] = FOV ? cam_byte(cam_lo, cam_hi, c) : 0u;
#pragma unroll
            for (int i = 0; i < 3 + (FOV ? MSC_MAX_CAMS : 0); ++i) {
                const uint32_t r = __reduce_add_sync(0xffffffffu, v[i]);
                if (lane == 0 && r) atomicAdd(&misc->stats[i < 3 ? 1 + i : 2 + i], r);
            }
        }
        __syncthreads();  // every tile of the sample is accumulated
        {
            // window flush: coalesced 16-byte stores of (count, isum) pairs, two cells per store
            const int half_w = L.win_w >> 1;  // win_w and win_lo are even -> 16-byte aligned rows
            uint32_t flags = 0;
            for (int i = tid; i < L.win_w * half_w; i += NT) {
                const int wy = i / half_w, wx2 = i - wy * half_w;
                const uint4 v = reinterpret_cast<const uint4*>(window)[wy * half_w + wx2];
                const size_t cell = (size_t)(wy + L.win_lo) * (size_t)res + (size_t)(wx2 * 2 + L.win_lo);
                *reinterpret_cast<uint4*>(g_ci + cell * 2) = v;
                flags |= (v.x >= 65536u || v.z >= 65536u) ? 1u : 0u;
            }
            // per-box results
            for (int b = tid; b < n_boxes; b += NT) {
                const uint32_t* acc = boxacc + b * kAccWords;
                const uint32_t cnt = acc[0];
                const size_t o = (size_t)(bx0 + b);
                A.out.box_count[o] = cnt;
                if (cnt == 0) {
                    A.out.box_nearest[o] = INFINITY;
                    A.out.box_centroid[o * 3 + 0] = 0.0f; A.out.box_centroid[o * 3 + 1] = 0.0f; A.out.box_centroid[o * 3 + 2] = 0.0f;
                } else {
                    A.out.box_nearest[o] = __fsqrt_rn(__uint_as_float(acc[1]));
#pragma unroll
                    for (int k = 0; k < 3; ++k)
                        A.out.box_centroid[o * 3 + k] = box_centroid(A, cnt, (unsigned long long)acc[2 + k] + ((unsigned long long)acc[5 + k] << 32));
                }
            }
            if (flags) atomicOr(&misc->stats[13], flags);
        }
        __syncthreads();
        if (tid < MSC_STATS_STRIDE) {
            uint32_t v = misc->stats[tid];
            if (tid == 0) {
                v = 0;
                for (int s = sw0; s < sw1; ++s) v += A.in.sweep_count[s];
            }
            if (tid == 4) v = misc->stats[2] - misc->stats[3];  // n_object = n_kept - n_ground
            if (tid == 13 && box_overflow) v |= 0x80000000u;
            A.out.stats[(size_t)sample * MSC_STATS_STRIDE + tid] = v;
        }
        // (the __syncthreads after the next sample fetch orders these reads before the smem is re-zeroed)
    }
}

template <class C, bool FOV, bool FASTDIV, bool KEEPMASK>
static int launch_one(const FusedArgs& args, const TableLayout& T, unsigned char* ws, int grid, cudaStream_t stream) {
    auto kern = stream_evidence_kernel<C, FOV, FASTDIV, KEEPMASK>;
    MSC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, args.L.total_bytes));
    kern<<<grid, C::kThreads, args.L.total_bytes, stream>>>(args, T, ws);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

int launch_stream_kernel(const FusedArgs& args, const TableLayout& T, unsigned char* ws, int grid, bool fov, bool fast, cudaStream_t stream) {
    using C = Shape0;
    if (fov && args.P.fov_keep_mask != 0u)
        return fast ? launch_one<C, true, true, true>(args, T, ws, grid, stream) : launch_one<C, true, false, true>(args, T, ws, grid, stream);
    if (fov) return fast ? launch_one<C, true, true, false>(args, T, ws, grid, stream) : launch_one<C, true, false, false>(args, T, ws, grid, stream);
    return fast ? launch_one<C, false, true, false>(args, T, ws, grid, stream) : launch_one<C, false, false, false>(args, T, ws, grid, stream);
}

}  // namespace msc
