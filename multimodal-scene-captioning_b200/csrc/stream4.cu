// stream4.cu -- fourth generation of the streaming kernel (launch shape "config" 10, the default).
//
// Same arithmetic per point as fused_stream.cu (SURVEY.md App. A + lidar_agent.py:103-132, :547-560); results are bit-identical
// (tools/sweep_configs.py).  Every variant of this kernel saturates two units together: instruction issue and the LSU data pipe
// (shared-memory wavefronts).  What this generation does about both, and about batches that do not fill the device:
//   * work is partitioned STATICALLY in warp tiles (128 rows of one sweep): fused_tables_kernel prefix-sums the tiles of every sample,
//     CTA b of G owns global tiles [b * total / G, (b + 1) * total / G).  A sample that straddles CTA boundaries (a single keyframe,
//     a shard that is not a multiple of the SM count) is processed in parts that merge with integer reductions; the part that takes
//     the last ticket finalises the sample.  Every SM gets the same share of the points whatever the batch size.
//   * raw rows reach shared memory through the TMA unit (cp.async.bulk into the warp's own tile slot, completion on the warp's own
//     mbarrier): the bulk copy costs the LSU data pipe nothing.  The lanes read the slot in passes of 32 * PPT rows; the next tile's
//     copy is issued as soon as the last pass has its rows in registers.  (Measured alternatives: two 64-row slots with two mbarriers,
//     4.6 % slower; commit b7fc82f, rows straight into registers with 128-bit loads -- fewer instructions, no slot, and slower: the
//     strided loads re-touch every 128-byte line five times on that pipe.)
//   * dropped points are counted by WHERE their atomic lands (one sink word per lane for remove_close, another for the range /
//     height gate), periphery points count into their cull cell's word (which returns the cell's edge code like a window word does):
//     n_after_close, n_kept and the decided share of the per-camera counts all come out of the epilogue's sums.
//   * the edge code a count word returns says whether an image-column ray crosses the point's cell at all (19 % of the kept points);
//     those points wait in a per-warp edge queue and are tested 32 at a time, one per lane: ONE branch-free cross product selected by
//     the code; cells crossed by exactly two rays of different cameras get pair codes (assigned per sample as they occur) and a
//     second test under a warp vote; anything else is a cold path.  (Testing every point in line -- a pad entry for code 0 -- issued
//     the same number of instructions but 6 % more shared-memory wavefronts.)
//   * cull-cell ids are a 4-byte table of their own; class words live in a per-CTA slice of the workspace (the hot loop never reads
//     them); window rows have an odd stride (a ray along y does not pile up in one bank).
//   * the shared-memory layout is a constexpr function used by the host and by the kernel: the instantiation for the standard
//     configuration (STD) takes every offset and threshold as a compile-time constant instead of re-reading the constant bank and
//     re-deriving table addresses per tile (at 64 registers per thread nothing of that survives in registers).
//   * the result tables of a shard can be REPLICATED to the other GPUs of the box by the finalising code itself (P2P stores through
//     A.replica[]): the gather of a sharded batch without a collective.
#include "fused_common.cuh"

namespace msc {

// Two launch shapes: PPT = 2 points per lane and pass (1024 threads x 64 registers, the default: more warps to hide latency) and PPT = 4
// (512 threads x 128 registers: fewer instructions per point, half the warps).
__host__ __device__ constexpr int s4_threads(int ppt) { return ppt == 4 ? 512 : 1024; }
constexpr int kS4MaxWarps = 32;
// candidate queue per warp.  PPT = 4: 128 entries, drained 64 at a time (two per lane), checked every two point slots (<= 63 pending + 64
// pushed); PPT = 2: 64 entries, drained 32 at a time, checked after every point slot (<= 31 pending + 32 pushed)
__host__ __device__ constexpr int s4_queue_entries(int ppt) { return ppt == 4 ? 128 : 64; }
constexpr int kS4PoseSmem = 10;   // sweeps whose transforms / extents are staged per sample (BASELINE configs 3-5: 10); later ones are read from global memory
constexpr int kS4SinkWords = 64;  // per array: [0, 32) remove_close sink of lane l, [32, 64) range / height sink of lane l
constexpr uint32_t kS4CodeShift = 27, kS4CountMask = (1u << kS4CodeShift) - 1u, kS4CodeMulti = 31u;

constexpr int kS4PairCodes = 14;  // codes 17..30: cells crossed by exactly two rays of different cameras, assigned per sample as they occur

struct S4Misc {  // small per-CTA state at misc_off
    // [code]: the exact test of an image-column ray, wedge_edge_entry(); 0 = pad (the test fails: a = NaN); 1 + c right edge, 9 + c left
    // edge of camera c; 17 + i the first / second edge of pair i (edge2 is a pad for every other code); 31 = several edges, resolved on a
    // cold path from the cell's class word
    float4 edge1[32], edge2[32];
    uint2 inc1[32], inc2[32];  // byte-counter increments (cameras 0-3, 4-7) of the entry's camera
    uint32_t pairs[16];  // pair i: 0 = free, else 0x100 | e1 | e2 << 4 (edge numbers 0-7 right, 8-15 left)
    uint32_t stats[MSC_STATS_STRIDE];
    uint32_t sweep_start[kS4PoseSmem], sweep_count[kS4PoseSmem];
    int32_t ticket, pad_[3];
    double pose[kS4PoseSmem * 12];  // this sample's 3x4 sweep transforms
    double wpose[kS4MaxWarps * 12];  // per-warp slot for sweeps beyond kS4PoseSmem
    float wq[MSC_MAX_CAMS * 6];     // this sample's camera wedges (fused_tables_kernel), source of the per-cell edge classes
};

int stream4_threads(int ppt) { return s4_threads(ppt); }

// Shared-memory layout (bytes).  One block per warp first -- its tile slot of raw rows, its candidate queue, its edge queue, its mbarrier:
// one base register reaches all of them with immediate offsets -- then the cull-cell ids, the small per-CTA state, the window region
//   array A = [64 sink words][win_w^2 count | code << 27][cull_dim^2 periphery count | code << 27]
//   array B = [64 sink words][win_w^2 Q8 intensity sums]
// and, last, the box tables (their size is the only part that depends on the batch).  constexpr: the kernel instantiation for the
// standard configuration takes every offset from here as a compile-time constant (immediate operands instead of constant-bank loads
// and address arithmetic), the host uses the same function for every configuration.
constexpr int kS4TileRows = 128;  // rows of a warp tile for both launch shapes: one bulk copy, one wait, one cursor step per 128 rows
// edge queue per warp: points of cells that an image-column ray crosses wait here (x, y: 8 bytes; the cell's edge code: 1 byte) until 32
// are pending, then every lane runs the exact cross products of one of them.  Checked after every point slot (<= 31 pending + 32 pushed)
constexpr int kS4EdgeEntries = 64;
__host__ __device__ constexpr int s4_warp_block_bytes(int ppt) {  // (a multiple of 16)
    return kS4TileRows * 20 + s4_queue_entries(ppt) * 16 + kS4EdgeEntries * 8 + kS4EdgeEntries + 16;
}
__host__ __device__ constexpr FusedLayout s4_layout(int smem_bytes, int ppt, int res, int cull_dim, int cull_shift, int box_cap, int opt_window,
                                                    int inner_dim) {
    FusedLayout L{};
    L.cull_dim = cull_dim; L.cull_shift = cull_shift; L.max_boxes = box_cap < 1 ? 1 : box_cap;
    L.inner_dim = inner_dim; L.inner_lo = (res - inner_dim) / 2; L.inner_off = 0;
    int off = 0;
    L.tiles_off = off; L.queue_off = off; off += (s4_threads(ppt) / 32) * s4_warp_block_bytes(ppt);
    L.cull_off = off; off += (cull_dim * cull_dim * 4 + 127) & ~127;
    L.misc_off = off; off += ((int)sizeof(S4Misc) + 127) & ~127;
    L.window_off = off;
    const int n_cull_r = (kS4SinkWords + cull_dim * cull_dim + 3) & ~3;  // sink words + cull-cell words of array A, rounded
    const int box_bytes = ((L.max_boxes * kBoxStride * 4 + L.max_boxes * kAccWords * 4) + 127) & ~127;
    const int avail = smem_bytes - off - box_bytes - (n_cull_r + kS4SinkWords) * 4;
    // window rows are stored with an ODD stride (win_w + 1 words): the 32 points of a warp slot lie along one ray from the sensor, and
    // with a stride that is a multiple of 32 (96!) a ray along y would put all of them in one bank
    int w = 0;
    while ((w + 2) * (w + 3) * 8 <= avail && (w + 2) <= res) w += 2;
    if (opt_window > 0 && opt_window < w) w = opt_window & ~1;
    if (((res - w) / 2) & 1) w -= 2;  // keep win_lo even so flush rows stay 16-byte aligned in the global layer
    if (w < 0) w = 0;
    L.win_w = avail < 0 ? -1 : w;
    L.win_lo = (res - w) / 2;
    L.win_stride = w + 1;
    const int n_store = w * (w + 1);
    L.pcnt_off = (kS4SinkWords + n_store) * 4;
    L.isum_delta = (n_store + n_cull_r) * 4;  // word of array A -> the same word of array B
    off += (n_store + n_cull_r) * 4 + (kS4SinkWords + n_store) * 4;
    L.boxp_off = off; off += L.max_boxes * kBoxStride * 4;
    L.boxacc_off = off; off += L.max_boxes * kAccWords * 4;
    L.total_bytes = (off + 127) & ~127;
    return L;
}
// The standard configuration (BASELINE configs 2-5): 200 x 200 grid over +-50 m, 2 m cull cells, the reference's thresholds, up to
// kS4StdBoxes boxes per sample, the B200's 227 KB of shared memory.
constexpr int kS4StdSmem = 232448, kS4StdRes = 200, kS4StdCullDim = 50, kS4StdCullShift = 2, kS4StdBoxes = 128, kS4StdInner = kInnerMax;
struct S4StdParams {  // msc_params / FusedArgs members the main loop reads, as the standard configuration has them (bit patterns of
    // msc_geom.layout.GeomParams() / geometry.sqrt_thresholds)
    static constexpr float remove_close_radius = 1.0f, s_lo = 0x1.000004p+0f, s_hi = 0x1.387ffep+11f, z_min = -3.0f, z_max = 5.0f,
                           ground_z = -0x1.666666p+0f, bev_range = 50.0f, two_r = 100.0f, rcp_two_r = 0x1.47ae14p-7f, resf = 200.0f, iscale = 256.0f;
};
bool stream4_is_standard(const FusedArgs& a, int smem_bytes, int ppt, int opt_window) {
    const msc_params& P = a.P;
    typedef S4StdParams S;
    if (ppt != 2 || smem_bytes != kS4StdSmem || opt_window != 0) return false;
    if (P.bev_res != kS4StdRes || a.L.cull_dim != kS4StdCullDim || a.L.cull_shift != kS4StdCullShift || a.L.max_boxes > kS4StdBoxes) return false;
    return P.remove_close_radius == S::remove_close_radius && P.s_lo == S::s_lo && P.s_hi == S::s_hi && P.z_min == S::z_min && P.z_max == S::z_max &&
           P.ground_z == S::ground_z && P.bev_range == S::bev_range && a.two_r == S::two_r && a.rcp_two_r == S::rcp_two_r && a.resf == S::resf &&
           a.iscale == S::iscale;
}
FusedLayout stream4_layout(int smem_bytes, int ppt, int res, int cull_dim, int cull_shift, int box_cap, int opt_window, int inner_dim) {
    return s4_layout(smem_bytes, ppt, res, cull_dim, cull_shift, box_cap, opt_window, inner_dim);
}
int stream4_std_boxes() { return kS4StdBoxes; }

// predicated global reductions (one instruction each, no branch-around sequence)
__device__ __forceinline__ void s4_red_global_u64_if(unsigned long long* p, unsigned long long v, bool pred) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %2, 0;\n@p red.global.add.u64 [%0], %1;\n}" ::"l"(p), "l"(v), "r"((uint32_t)pred) : "memory");
}
__device__ __forceinline__ void s4_red_global_max_if(int* p, int v, bool pred) {
    asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %2, 0;\n@p red.global.max.s32 [%0], %1;\n}" ::"l"(p), "r"(v), "r"((uint32_t)pred) : "memory");
}
// bev_cell() of x and y in one packed pass (same operations, same order, per half); the clip is a float -> unsigned conversion (negative
// and NaN -> 0, like max(trunc, 0)) followed by one unsigned min
template <bool FASTDIV>
__device__ __forceinline__ void s4_bev_cell_xy(float x, float y, float r, float two_r, float rcp_two_r, float resf, uint32_t res_m1, uint32_t& ix, uint32_t& iy) {
    const unsigned long long a = f2_add(f2_pack(x, y), f2_pack(r, r));
    unsigned long long q;
    if (FASTDIV) {
        const unsigned long long rc = f2_pack(rcp_two_r, rcp_two_r);
        const unsigned long long q0 = f2_mul(a, rc);
        const unsigned long long rem = f2_fma(f2_pack(-two_r, -two_r), q0, a);
        q = f2_fma(rem, rc, q0);
    } else {
        float ax, ay;
        f2_unpack(a, ax, ay);
        q = f2_pack(__fdiv_rn(ax, two_r), __fdiv_rn(ay, two_r));
    }
    float tx, ty;
    f2_unpack(f2_mul(q, f2_pack(resf, resf)), tx, ty);
    ix = min(__float2uint_rz(tx), res_m1);
    iy = min(__float2uint_rz(ty), res_m1);
}
// cameras whose wedge contains every point of the cell
__device__ __forceinline__ uint32_t s4_decided_in(uint32_t cls) { return cls & ~(cls >> 8) & ~(cls >> 16) & 0xffu; }

// ------------------------------------------------------------------------------------------------ partition pre-kernels
// Samples that straddle a CTA boundary of the static partition merge their parts with reductions: zero their output layers and merge
// scratch first.  Block b looks at boundary b + 1 of a G-CTA launch; the first boundary inside a sample does the work.
__global__ void __launch_bounds__(256) stream4_straddle_kernel(const __grid_constant__ FusedArgs A, const TableLayout T, unsigned char* __restrict__ ws, int G) {
    const uint32_t* const tile_off = reinterpret_cast<const uint32_t*>(ws + T.tileoff_off);
    const int n = A.in.n_samples;
    const uint32_t total = tile_off[n];
    const uint32_t b = blockIdx.x + 1u;
    const uint32_t g = (uint32_t)((unsigned long long)b * total / (uint32_t)G);
    const uint32_t gp = (uint32_t)((unsigned long long)(b - 1u) * total / (uint32_t)G);
    // sample s with tile_off[s] < g < tile_off[s + 1]
    int lo = 0, hi = n;  // last s with tile_off[s] < g
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (tile_off[mid] < g) lo = mid; else hi = mid; }
    const int s = lo;
    if (n == 0 || !(tile_off[s] < g && g < tile_off[s + 1])) return;
    if (b > 1u && gp > tile_off[s]) return;  // an earlier boundary lies inside the same sample
    const size_t ncell = (size_t)A.P.bev_res * (size_t)A.P.bev_res;
    zero_bev_layers(A.out.bev_ci + (size_t)s * ncell * 2, A.out.bev_height + (size_t)s * ncell, ncell, threadIdx.x, blockDim.x);
    uint32_t* st = reinterpret_cast<uint32_t*>(ws + T.splitstats_off) + (size_t)s * MSC_STATS_STRIDE;
    if (threadIdx.x < MSC_STATS_STRIDE) st[threadIdx.x] = 0u;
    unsigned long long* scr = reinterpret_cast<unsigned long long*>(ws + T.boxscr_off);
    for (int gb = A.in.sample_box_off[s] + (int)threadIdx.x; gb < A.in.sample_box_off[s + 1]; gb += blockDim.x) {
        scr[(size_t)gb * 4 + 0] = 0x7f800000ull << 32;  // count 0 | min +inf
        scr[(size_t)gb * 4 + 1] = 0ull; scr[(size_t)gb * 4 + 2] = 0ull; scr[(size_t)gb * 4 + 3] = 0ull;
    }
}

// ------------------------------------------------------------------------------------------------ the streaming kernel
template <bool FOV, bool FASTDIV, int PPT, bool STD>
__global__ void __launch_bounds__(s4_threads(PPT), 1) stream4_kernel(const __grid_constant__ FusedArgs A, const TableLayout T,
                                                                     unsigned char* __restrict__ ws) {
    constexpr int NT = s4_threads(PPT), W = NT / 32, TP = kS4TileRows, TSH = 7, SUB = kS4TileRows / (32 * PPT), kS4QueueEntries = s4_queue_entries(PPT);
    extern __shared__ __align__(128) unsigned char smem[];
    // STD: every layout offset and every threshold of the main loop is a compile-time constant (the host selects this instantiation only
    // when the call's layout and parameters equal them bit for bit, stream4_is_standard); otherwise they are kernel arguments
    constexpr FusedLayout SL = s4_layout(kS4StdSmem, PPT, kS4StdRes, kS4StdCullDim, kS4StdCullShift, kS4StdBoxes, 0, kS4StdInner);
    struct PV { float remove_close_radius, s_lo, s_hi, z_min, z_max, ground_z, bev_range; int bev_res, n_cams; };
    const FusedLayout L = STD ? SL : A.L;
    const PV P = STD ? PV{S4StdParams::remove_close_radius, S4StdParams::s_lo, S4StdParams::s_hi, S4StdParams::z_min, S4StdParams::z_max,
                          S4StdParams::ground_z, S4StdParams::bev_range, kS4StdRes, A.P.n_cams}
                     : PV{A.P.remove_close_radius, A.P.s_lo, A.P.s_hi, A.P.z_min, A.P.z_max, A.P.ground_z, A.P.bev_range, A.P.bev_res, A.P.n_cams};
    const float two_r = STD ? S4StdParams::two_r : A.two_r, rcp_two_r = STD ? S4StdParams::rcp_two_r : A.rcp_two_r, resf = STD ? S4StdParams::resf : A.resf,
                iscale = STD ? S4StdParams::iscale : A.iscale;
    const int n_cull = L.cull_dim * L.cull_dim;
    uint32_t* const cullids = reinterpret_cast<uint32_t*>(smem + L.cull_off);   // [n_cull] candidate box ids of the cull cell
    // class words (camera in-bits and undecided-edge bits) of the cull cells and of the fine cells around the sensor: only the prologue
    // (which turns them into edge codes), the epilogue and the cold multi-edge path read them, so they live in a per-CTA slice of the
    // workspace (L1 / L2 hits) and leave 20 KB of shared memory to the BEV window
    uint32_t* const cullcls = reinterpret_cast<uint32_t*>(ws + T.cls_off) + (size_t)blockIdx.x * (size_t)(n_cull + kInnerMax * kInnerMax);  // [n_cull]
    uint32_t* const inner = cullcls + n_cull;                                   // [inner_dim^2] fine classes (one per BEV cell around the sensor)
    float* const boxp = reinterpret_cast<float*>(smem + L.boxp_off);            // [max_boxes][kBoxStride]
    uint32_t* const boxacc = reinterpret_cast<uint32_t*>(smem + L.boxacc_off);  // [max_boxes][kAccWords]
    S4Misc* const misc = reinterpret_cast<S4Misc*>(smem + L.misc_off);
    const int win_w = L.win_w, win_lo = L.win_lo, win_stride = L.win_stride;
    const int n_win = win_w * win_stride;  // words of a window array (rows padded to the odd stride)
    // window region: array A = [64 sink][n_win count | code << 27][n_cull periphery count | code << 27], array B = [64 sink][n_win Q8
    // intensity sums] (a periphery point adds its intensity to the lane's sink word of array B)
    uint32_t* const arrA = reinterpret_cast<uint32_t*>(smem + L.window_off);
    uint32_t* const arrB = arrA + (L.isum_delta >> 2);
    uint32_t* const wcount = arrA + kS4SinkWords;
    uint32_t* const pcnt = wcount + n_win;
    uint32_t* const wisum = arrB + kS4SinkWords;
    const float* const g_boxprep = reinterpret_cast<const float*>(ws + T.boxprep_off);
    const float* const g_wedges = reinterpret_cast<const float*>(ws + T.wedge_off);
    const uint32_t* const g_cullids = reinterpret_cast<const uint32_t*>(ws + T.cullids_off);

    const int tid = threadIdx.x, lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // warp-uniform as far as the compiler is concerned
    uint32_t smem_s = smem_u32(smem);
    asm volatile("" : "+r"(smem_s));  // opaque: one live register instead of a re-derived generic->shared conversion per use
    const uint32_t misc_s = smem_s + (uint32_t)L.misc_off;
    constexpr uint32_t kSlotBytes = (uint32_t)TP * 20u, kWarpBlock = (uint32_t)s4_warp_block_bytes(PPT);
    const uint32_t ring_s = smem_s + (uint32_t)L.tiles_off + (uint32_t)warp * kWarpBlock;  // this warp's block: ONE slot of 128 raw rows,
    const uint32_t queue_s = ring_s + kSlotBytes;                                          // its candidate queue
    const uint32_t eq_s = queue_s + (uint32_t)(kS4QueueEntries * 16);                      // its edge queue: (x, y) pairs,
    const uint32_t eqc_s = eq_s + (uint32_t)(kS4EdgeEntries * 8);                          // their edge codes (bytes)
    const uint32_t bar_s = eqc_s + (uint32_t)kS4EdgeEntries;                               // and its mbarrier
    const uint64_t policy = l2_policy_evict_first();
    const uint32_t edge1_s = misc_s + (uint32_t)offsetof(S4Misc, edge1);
    constexpr uint32_t kEdge2 = (uint32_t)(offsetof(S4Misc, edge2) - offsetof(S4Misc, edge1)), kInc1 = (uint32_t)(offsetof(S4Misc, inc1) - offsetof(S4Misc, edge1)),
                       kInc2 = (uint32_t)(offsetof(S4Misc, inc2) - offsetof(S4Misc, edge1));
    const uint32_t cull_s = smem_s + (uint32_t)L.cull_off;
    const uint32_t arrA_s = smem_s + (uint32_t)L.window_off;
    const uint32_t sink_close_s = arrA_s + (uint32_t)lane * 4u, sink_gate_s = arrA_s + 128u + (uint32_t)lane * 4u;
    const uint32_t wcount_s = arrA_s + (uint32_t)kS4SinkWords * 4u;
    const uint32_t pcnt_s = arrA_s + (uint32_t)L.pcnt_off;     // (host-computed: (kS4SinkWords + n_win) * 4)
    const uint32_t isum_delta = (uint32_t)L.isum_delta;        // word of array A -> the same word of array B (host-computed: arr_words * 4)
    const int res = P.bev_res, res_m1 = P.bev_res - 1;
    const size_t ncell = (size_t)res * (size_t)res;
    const int n_cams = P.n_cams;
    const int n_inner = L.inner_dim * L.inner_dim;

    if (lane == 0) {
        mbar_init(bar_s, 1);
        mbar_fence_init();
    }
    uint32_t wk = 0;  // tiles this warp has consumed since launch: mbarrier parity = wk & 1
    __syncthreads();

    // ------------------------------------------------------------ this CTA's share of the batch: a range of global tiles
    const uint32_t* const tile_off = reinterpret_cast<const uint32_t*>(ws + T.tileoff_off);  // [n_samples + 1]
    const int n_samples = A.in.n_samples;
    const uint32_t G = gridDim.x, cta = blockIdx.x;
    const uint32_t total = tile_off[n_samples];
    const uint32_t g0 = (uint32_t)((unsigned long long)cta * total / G), g1 = (uint32_t)((unsigned long long)(cta + 1) * total / G);
    auto cta_of = [&](uint32_t r) -> uint32_t { return (uint32_t)((((unsigned long long)r + 1ull) * G + total - 1ull) / total) - 1u; };
    int s_begin;
    {   // first sample whose tiles start at or after g0, or the one before it when that one straddles g0
        int lo = 0, hi = n_samples;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (tile_off[mid] < g0) lo = mid + 1; else hi = mid; }
        s_begin = (lo > 0 && (lo == n_samples || tile_off[lo] > g0)) ? lo - 1 : lo;
    }
    for (int sample = s_begin; sample < n_samples; ++sample) {
        const uint32_t off = tile_off[sample], tiles_s = tile_off[sample + 1] - off;
        if (off >= g1 && !(cta == G - 1u && off >= total)) break;  // (the last CTA also owns empty samples at the very end)
        uint32_t lr0 = 0, lr1 = 0, n_parts = 1;
        if (tiles_s == 0) {
            if (off < g0) continue;  // an empty sample belongs to the CTA whose range holds its offset
        } else {
            lr0 = max(g0, off) - off;
            lr1 = min(g1, off + tiles_s) - off;
            if (lr0 >= lr1) continue;
            // CTAs that own at least one tile of the sample.  With at least one tile per CTA the owners are contiguous; with fewer tiles
            // than CTAs every tile has an owner of its own (and the CTAs in between own nothing)
            n_parts = total >= G ? cta_of(off + tiles_s - 1u) - cta_of(off) + 1u : tiles_s;
        }
        __syncthreads();  // the previous sample's epilogue has read the per-CTA state that is re-initialised below

        const int sw0 = A.in.sample_sweep_off[sample], sw1 = A.in.sample_sweep_off[sample + 1];
        const int n_sw = sw1 - sw0;
        if (tid < kS4PoseSmem && tid < n_sw) {
            misc->sweep_start[tid] = A.in.sweep_start[sw0 + tid];
            misc->sweep_count[tid] = A.in.sweep_count[sw0 + tid];
        }
        for (int i = tid; i < min(n_sw, kS4PoseSmem) * 12; i += NT) misc->pose[i] = A.in.sweep_pose[(size_t)sw0 * 12 + i];
        if (tid < MSC_STATS_STRIDE) { misc->stats[tid] = 0u; misc->pairs[tid] = 0u; }
        if (FOV && tid < MSC_MAX_CAMS * 6) misc->wq[tid] = g_wedges[(size_t)sample * MSC_MAX_CAMS * 6 + tid];
        __syncthreads();

        // ---- tile cursor: this part owns local tiles [lr0, lr1) of the sample, warp `warp` takes lr0 + warp, + W, ...; a tile is 128
        // rows of ONE sweep (the last tile of a sweep is partial), lane l owns rows 4 l .. 4 l + 3 of it.
        uint32_t t = lr0 + (uint32_t)warp;  // local tile index of the tile whose rows are in flight
        int n_si = -1;                      // its sweep
        uint32_t s_tb = 0, s_te = 0, s_cnt = 0, s_base = 0;  // tiles [s_tb, s_te) belong to sweep n_si: s_cnt rows from row s_base
        auto seek_sweep = [&]() {  // (precondition: t < lr1 <= tiles of the sample)
            while (t >= s_te) {
                ++n_si;
                if (n_si < kS4PoseSmem) { s_cnt = misc->sweep_count[n_si]; s_base = misc->sweep_start[n_si]; }
                else { s_cnt = A.in.sweep_count[sw0 + n_si]; s_base = A.in.sweep_start[sw0 + n_si]; }
                s_tb = s_te;
                s_te += (s_cnt + (uint32_t)(TP - 1)) >> TSH;
            }
        };
        // Raw rows travel global -> shared memory with the TMA unit (cp.async.bulk, completion on the warp's own mbarrier): the copy
        // costs the LSU data pipe nothing -- five strided 64/128-bit loads per lane re-touch every 128-byte line five times there, and that
        // pipe is what the kernel saturates first -- and no registers.  ONE slot of 128 rows per warp: the lanes read the slot in SUB
        // passes of 32 * PPT rows; as soon as the last pass has read its rows the slot is free and the next tile's copy goes out, so it
        // has the whole last pass (>= half a tile of work) to land.  One copy, one wait and one cursor step per 128 rows.
        auto issue = [&]() {  // whole warp (uniform control flow); one lane talks to the TMA unit
            const uint32_t first = (t - s_tb) << TSH;
            const uint32_t npts = min((uint32_t)TP, s_cnt - first);
            const uint32_t bytes = (npts * 20u + 15u) & ~15u;
            const float* src = A.in.points + ((size_t)s_base + first) * 5;
            if (lane == 0) bulk_load(ring_s, src, bytes, bar_s, policy);
        };
        bool more = t < lr1;
        if (more) { seek_sweep(); issue(); }  // overlaps the prologue below

        // ------------------------------------------------------------ prologue: accumulators, tables -> smem
        const int bx0 = A.in.sample_box_off[sample];
        int n_boxes = A.in.sample_box_off[sample + 1] - bx0;
        const bool box_overflow = n_boxes > L.max_boxes;  // caller under-declared max_boxes_per_sample
        if (box_overflow) n_boxes = L.max_boxes;
        const size_t cell_base = (size_t)sample * ncell;
        uint32_t* const g_ci = A.out.bev_ci + cell_base * 2;
        float* const g_h = A.out.bev_height + cell_base;
        // class word of BEV cell (ix, iy): fine table inside [inner_lo, inner_lo + inner_dim)^2, else the cull cell's
        auto class_of = [&](int ix, int iy) -> uint32_t {
            if (!FOV) return 0u;
            const uint32_t jx = (uint32_t)(ix - L.inner_lo), jy = (uint32_t)(iy - L.inner_lo);
            if (jx < (uint32_t)L.inner_dim && jy < (uint32_t)L.inner_dim) return inner[jy * (uint32_t)L.inner_dim + jx];
            return cullcls[(iy >> L.cull_shift) * L.cull_dim + (ix >> L.cull_shift)];
        };
        // edge code of a cell from its class word (bits 0-7 in-bits, 8-15 right edge undecided, 16-23 left edge undecided): 0 = every
        // camera decided, 1 + e = exactly edge e undecided, 17 + i = exactly the two edges of pair i (different cameras; pairs get their
        // numbers as cells meet them), 31 = anything else
        auto code_of = [&](uint32_t cls) -> uint32_t {
            const uint32_t und = (cls >> 8) & 0xffffu;
            if (und == 0u) return 0u;
            const uint32_t e1 = (uint32_t)__ffs((int)und) - 1u, rest = und & (und - 1u);
            if (rest == 0u) return e1 + 1u;
            const uint32_t e2 = (uint32_t)__ffs((int)rest) - 1u;
            if ((rest & (rest - 1u)) || ((e1 ^ e2) & 7u) == 0u) return kS4CodeMulti;  // three or more rays, or both rays of one camera
            const uint32_t key = 0x100u | e1 | (e2 << 4);
            for (int i = 0; i < kS4PairCodes; ++i) {
                const uint32_t old = atomicCAS(&misc->pairs[i], 0u, key);
                if (old == 0u || old == key) return 17u + (uint32_t)i;
            }
            return kS4CodeMulti;
        };
        {
            const uint32_t* ids = g_cullids + (size_t)sample * n_cull;  // candidate boxes per cull cell (fused_cullids_kernel)
            // edge classes of the sample's camera wedges per cull cell, and per BEV cell around the sensor (fine table)
            for (int i = tid; i < n_cull; i += NT) {
                const uint32_t cls = FOV ? edge_class_word(A, misc->wq, i) : 0u;
                cullids[i] = ids[i];
                cullcls[i] = cls;
                pcnt[i] = code_of(cls) << kS4CodeShift;
            }
            if (FOV)
                for (int i = tid; i < n_inner; i += NT) inner[i] = edge_class_word(A, misc->wq, n_cull + i);
            if (tid < kS4SinkWords) { arrA[tid] = 0u; arrB[tid] = 0u; }
            for (int i = tid; i < n_win; i += NT) wisum[i] = 0u;
            for (int i = tid; i < n_boxes * kAccWords; i += NT) boxacc[i] = ((i % kAccWords) == 1) ? 0x7f800000u : 0u;
            const float4* bsrc = reinterpret_cast<const float4*>(g_boxprep + (size_t)bx0 * kBoxStride);
            for (int i = tid; i < n_boxes * (kBoxStride / 4); i += NT) reinterpret_cast<float4*>(boxp)[i] = bsrc[i];
            // zero-fill this sample's global layers (a straddling sample was zero-filled by stream4_straddle_kernel)
            if (n_parts == 1) zero_bev_layers(g_ci, g_h, ncell, tid, NT);
        }
        __threadfence();
        __syncthreads();  // class tables are in smem
        for (int i = tid; i < n_win; i += NT) {
            const int wy = i / win_stride, wx = i - wy * win_stride;
            wcount[i] = wx < win_w ? code_of(class_of(wx + win_lo, wy + win_lo)) << kS4CodeShift : 0u;
        }
        __syncthreads();  // every pair that occurs has its code
        if (tid < 64) {
            const int code = tid & 31, second = tid >> 5;
            int e = -1;  // edge tested by this entry
            if (code >= 1 && code <= 2 * MSC_MAX_CAMS) e = second ? -1 : code - 1;
            else if (code >= 17 && code < 17 + kS4PairCodes && misc->pairs[code - 17]) e = (int)((misc->pairs[code - 17] >> (second ? 4 : 0)) & 0xfu);
            float4 E = make_float4(0.0f, 0.0f, __int_as_float(0x7fc00000), 0.0f);  // pad: the test fails
            uint2 inc = make_uint2(0u, 0u);
            const int c = e & (MSC_MAX_CAMS - 1);
            if (FOV && e >= 0 && c < n_cams) {
                E = wedge_edge_entry(misc->wq + c * 6, e >= MSC_MAX_CAMS);
                inc.x = c < 4 ? 1u << (8 * c) : 0u;
                inc.y = c < 4 ? 0u : 1u << (8 * (c - 4));
            }
            (second ? misc->edge2 : misc->edge1)[code] = E;
            (second ? misc->inc2 : misc->inc1)[code] = inc;
        }
        __syncthreads();

        // ------------------------------------------------------------ main loop: this warp's tiles, no cross-warp sync
        uint32_t c_ground = 0;             // per-thread counter (flushed once per sample)
        uint32_t cam_lo = 0, cam_hi = 0;  // eight 8-bit per-camera counters of the exact edge tests (a point adds at most 1 per camera),
        uint32_t pstate = 0;              // spilled into the sample's smem counters before 255 points have been added since the last spill
        // (measured alternative: 4-bit counters in one register with one-word increments -- three LSU wavefronts fewer per tile, a spill
        // every 7 tiles instead of every 127: 0.4 % slower)
        uint32_t q_head = 0, q_tail = 0;   // warp-uniform (every lane derives them from the same ballots)
        // Every lane tests TWO queued points (entries head + lane and head + 32 + lane) against their candidate boxes, one candidate of
        // each per trip, so two independent box tests are in flight per lane; the (usually single) containing box is accumulated once
        // after the loop, a second containing box (overlapping annotations) inside it.
        // (The 80-register shape drains 32 entries at a time, one per lane: eight 128-bit loads in flight per lane do not fit.)
        constexpr uint32_t kDrain = PPT == 4 ? 64u : 32u;
        auto drain_queue = [&](uint32_t n_take) {  // n_take <= kDrain
            const float4 e0 = lds128(queue_s + (((q_head + (uint32_t)lane) & (uint32_t)(kS4QueueEntries - 1)) << 4));
            float4 e1 = e0;
            if (kDrain == 64u) e1 = lds128(queue_s + (((q_head + 32u + (uint32_t)lane) & (uint32_t)(kS4QueueEntries - 1)) << 4));
            uint32_t ids0 = (uint32_t)lane < n_take ? __float_as_uint(e0.w) : kCullEmpty;
            uint32_t ids1 = (kDrain == 64u && (uint32_t)lane + 32u < n_take) ? __float_as_uint(e1.w) : kCullEmpty;
            auto accumulate = [&](int b, const float4& e) {
                const float es2 = __fadd_rn(__fmul_rn(e.x, e.x), __fmul_rn(e.y, e.y));
                const uint32_t fx = (uint32_t)(__float2int_rn(__fmul_rn(e.x, A.cscale)) + A.centroid_bias);
                const uint32_t fy = (uint32_t)(__float2int_rn(__fmul_rn(e.y, A.cscale)) + A.centroid_bias);
                const uint32_t fz = (uint32_t)(__float2int_rn(__fmul_rn(e.z, A.cscale)) + A.centroid_bias);
                box_accumulate(smem_s + (uint32_t)L.boxacc_off + (uint32_t)b * (uint32_t)(kAccWords * 4), __float_as_uint(es2), fx, fy, fz);
            };
            int hit0 = -1, hit1 = -1;
            const bool crowded0 = ids0 == kCullAll, crowded1 = ids1 == kCullAll;  // more than four boxes touch the cell: test every box (below)
            if (crowded0) ids0 = kCullEmpty;
            if (crowded1) ids1 = kCullEmpty;
            if (kDrain == 64u) {
                while ((ids0 & ids1 & 0xffu) != 0xffu) {  // (an entry that has run out of candidates re-tests box 0 and ignores the answer)
                    const uint32_t b0 = ids0 & 0xffu, b1 = ids1 & 0xffu;
                    const bool in0 = box_contains(boxp, (int)(b0 == 0xffu ? 0u : b0), e0.x, e0.y, e0.z) && b0 != 0xffu;
                    const bool in1 = box_contains(boxp, (int)(b1 == 0xffu ? 0u : b1), e1.x, e1.y, e1.z) && b1 != 0xffu;
                    if (in0) { if (hit0 >= 0) accumulate((int)b0, e0); else hit0 = (int)b0; }
                    if (in1) { if (hit1 >= 0) accumulate((int)b1, e1); else hit1 = (int)b1; }
                    ids0 = (ids0 >> 8) | 0xff000000u;
                    ids1 = (ids1 >> 8) | 0xff000000u;
                }
            } else {
                while ((ids0 & 0xffu) != 0xffu) {
                    const int b0 = (int)(ids0 & 0xffu);
                    if (box_contains(boxp, b0, e0.x, e0.y, e0.z)) { if (hit0 >= 0) accumulate(b0, e0); else hit0 = b0; }
                    ids0 = (ids0 >> 8) | 0xff000000u;
                }
            }
            if (crowded0 || crowded1) {
                for (int b = 0; b < n_boxes; ++b) {
                    if (crowded0 && box_contains(boxp, b, e0.x, e0.y, e0.z)) { if (hit0 >= 0) accumulate(b, e0); else hit0 = b; }
                    if (crowded1 && box_contains(boxp, b, e1.x, e1.y, e1.z)) { if (hit1 >= 0) accumulate(b, e1); else hit1 = b; }
                }
            }
            // (Aggregating the hits of one box over the warp first, __match_any_sync + __reduce_*_sync, is bit-identical and 76 % slower:
            // DESIGN.md section 5.)
            if (hit0 >= 0) accumulate(hit0, e0);
            if (hit1 >= 0) accumulate(hit1, e1);
            q_head += n_take;
        };
        // ---- exact cross products for the points of cells that image-column rays cross, 32 queued points at a time (one per lane): the
        // first ray of the point's edge code for every lane (a pad entry's test fails), the second ray (codes 17..30) and the cold path
        // (code 31: cells crossed by three or more rays, or by both rays of one camera, next to a camera) under warp votes.  The camera's
        // byte counter takes the entry's increment: at most one per camera and call.
        uint32_t e_head = 0, e_tail = 0;  // warp-uniform
        auto drain_edges = [&](uint32_t n_take) {  // n_take <= 32
            const uint32_t slot = (e_head + (uint32_t)lane) & (uint32_t)(kS4EdgeEntries - 1);
            const uint2 pw = lds64(eq_s + (slot << 3));
            const float px = __uint_as_float(pw.x), py = __uint_as_float(pw.y);
            const uint32_t code = (uint32_t)lane < n_take ? lds8(eqc_s + slot) : 0u;
            {
                const float4 E = lds128(edge1_s + (code << 4));
                const uint2 inc = lds64(edge1_s + kInc1 + (code << 3));
                const float qx = __fsub_rn(px, E.x), qy = __fsub_rn(py, E.y);
                const float cr = __fmaf_rn(E.z, qy, -__fmul_rn(E.w, qx));
                if (cr >= 0.0f) { cam_lo += inc.x; cam_hi += inc.y; }
            }
            if (__any_sync(0xffffffffu, code > 2u * MSC_MAX_CAMS)) {
                const float4 E2 = lds128(edge1_s + kEdge2 + (code << 4));
                const uint2 inc2 = lds64(edge1_s + kInc2 + (code << 3));
                const float qx2 = __fsub_rn(px, E2.x), qy2 = __fsub_rn(py, E2.y);
                const float cr2 = __fmaf_rn(E2.z, qy2, -__fmul_rn(E2.w, qx2));
                if (cr2 >= 0.0f) { cam_lo += inc2.x; cam_hi += inc2.y; }
            }
            if (__any_sync(0xffffffffu, code == kS4CodeMulti)) {
                if (code == kS4CodeMulti) {
                    // the class the point's code came from: its cull cell's outside the window, else its BEV cell's
                    uint32_t cix, ciy;
                    s4_bev_cell_xy<FASTDIV>(px, py, P.bev_range, two_r, rcp_two_r, resf, (uint32_t)res_m1, cix, ciy);
                    const bool pp = max(cix - (uint32_t)win_lo, ciy - (uint32_t)win_lo) >= (uint32_t)win_w;
                    const uint32_t cls = pp ? cullcls[(ciy >> L.cull_shift) * L.cull_dim + (cix >> L.cull_shift)] : class_of((int)cix, (int)ciy);
                    uint32_t und = (cls >> 8) & 0xffffu, pass = 0xffffu;
                    while (und) {
                        const int e = __ffs((int)und) - 1;
                        und &= und - 1u;
                        const float4 E = lds128(edge1_s + ((uint32_t)(e + 1) << 4));
                        const float qx = __fsub_rn(px, E.x), qy = __fsub_rn(py, E.y);
                        const float cr = __fmaf_rn(E.z, qy, -__fmul_rn(E.w, qx));
                        if (!(cr >= 0.0f)) pass &= ~(1u << e);
                    }
                    // cameras with an undecided edge in this cell whose every undecided edge passed
                    const uint32_t any_und = ((cls >> 8) | (cls >> 16)) & 0xffu;
                    const uint32_t in = cls & any_und & pass & (pass >> 8);
                    cam_lo += ((in & 0xfu) * 0x00204081u) & 0x01010101u;  // bit c -> byte c
                    cam_hi += ((in >> 4) * 0x00204081u) & 0x01010101u;
                }
            }
            e_head += n_take;
            if (++pstate == 255u) {  // spill the byte counters before any of them can wrap
#pragma unroll
                for (int c = 0; c < MSC_MAX_CAMS; ++c) {
                    const uint32_t v = cam_byte(cam_lo, cam_hi, c);
                    if (v) red_shared_add(misc_s + (uint32_t)offsetof(S4Misc, stats) + (uint32_t)(5 + c) * 4u, v);
                }
                cam_lo = cam_hi = pstate = 0;
            }
        };
        while (more) {
            // the transform of the tile that is consumed now (n_si is still its sweep: the cursor advances further down); recomputed per
            // tile rather than carried in registers
            uint32_t pose_s = misc_s + (uint32_t)offsetof(S4Misc, pose) + (uint32_t)n_si * 96u;
            if (n_si >= kS4PoseSmem) {  // more sweeps than are staged: through this warp's slot (re-read per tile: rare and slow, but correct)
                __syncwarp();
                if (lane < 12) misc->wpose[warp * 12 + lane] = A.in.sweep_pose[(size_t)(sw0 + n_si) * 12 + lane];
                __syncwarp();
                pose_s = misc_s + (uint32_t)offsetof(S4Misc, wpose) + (uint32_t)warp * 96u;
            }
            // ---- the tile in flight becomes the current one
            const uint32_t npts = min((uint32_t)TP, s_cnt - ((t - s_tb) << TSH));
            mbar_wait_parity(bar_s, wk & 1u);
#pragma unroll 1
          for (int sub = 0; sub < SUB; ++sub) {  // SUB passes of 32 * PPT rows over the slot
            // ---- phase A: branch-free over the lane's points so their dependency chains interleave.  Lane l owns rows l, l + 32, ... of
            // the tile (a 5-word stride between lanes: bank-conflict free, and the 32 lanes of a slot hold 32 different rings)
            float xr[PPT], yr[PPT], zr[PPT];
            uint32_t q[PPT];
            bool close[PPT];
            {
                double xd[PPT], yd[PPT], zd[PPT];
                const uint32_t row_s = ring_s + (uint32_t)sub * (uint32_t)(PPT * 640) + (uint32_t)lane * 20u;
                const bool partial = npts < (uint32_t)TP;  // (warp-uniform)
#pragma unroll
                for (int u = 0; u < PPT; ++u) {
                    float x = __uint_as_float(lds32(row_s + u * 640u));
                    const float y = __uint_as_float(lds32(row_s + u * 640u + 4u)), z = __uint_as_float(lds32(row_s + u * 640u + 8u));
                    const float inten = __uint_as_float(lds32(row_s + u * 640u + 12u));
                    // last tile of a sweep: rows past its end hold stale data -> NaN fails every compare below
                    if (partial && (uint32_t)lane + (uint32_t)(u + sub * PPT) * 32u >= npts) x = __int_as_float(0x7fc00000);
                    // A.1 remove_close (square, sweep's own sensor frame)
                    close[u] = (fabsf(x) < P.remove_close_radius) & (fabsf(y) < P.remove_close_radius);
                    // Q8 intensity, clamp [0, 65535], NaN -> 0: fmaxf drops NaN and negatives, the FFMA rounds v * 2^shift to nearest even
                    // in the low mantissa bits of 2^23 + v * 2^shift (exact while below 2^23; larger values clamp anyway)
                    q[u] = min(__float_as_uint(__fmaf_rn(fmaxf(inten, 0.0f), iscale, 8388608.0f)) - 0x4b000000u, 65535u);
                    xd[u] = (double)x; yd[u] = (double)y; zd[u] = (double)z;
                }
                if (sub == SUB - 1) {  // every row of the slot has been read: the successor's copy goes out now
                    __syncwarp();
                    ++wk;
                    t += (uint32_t)W;
                    more = t < lr1;
                    if (more) { seek_sweep(); issue(); }
                }
                // A.1 f64 matrix x f32 point -> f32, one matrix row at a time
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    double m0, m1, m2, m3;
                    lds_f64x2(pose_s + r * 32, m0, m1);
                    lds_f64x2(pose_s + r * 32 + 16, m2, m3);
#pragma unroll
                    for (int u = 0; u < PPT; ++u) {
                        const float v = (float)__fma_rn(m0, xd[u], __fma_rn(m1, yd[u], __fma_rn(m2, zd[u], m3)));
                        if (r == 0) xr[u] = v; else if (r == 1) yr[u] = v; else zr[u] = v;
                    }
                }
            }
            // ---- the candidates queued by earlier tiles are tested while the conversions and the f64 chain above are in flight
            if (q_tail - q_head >= kDrain) {
                __syncwarp();  // the entries stored by the previous iteration are visible to the lanes that test them
                do drain_queue(kDrain); while (q_tail - q_head >= kDrain);
            }
            // ---- phase B: filter, BEV cell, cull entry, count word
            uint32_t cand[PPT], code[PPT];
            // this sample's (count, isum) layer as 64-bit cells and its max-height layer: re-derived from the sample index per tile (two
            // wide multiply-adds; holding the two pointers would cost four of the 64 registers, reading them back from smem LSU wavefronts)
            const unsigned long long cell0 = (unsigned long long)(uint32_t)sample * (unsigned long long)(uint32_t)(res * res);
            unsigned long long* const ci64g = reinterpret_cast<unsigned long long*>(A.out.bev_ci) + cell0;
            int* const h32g = reinterpret_cast<int*>(A.out.bev_height) + cell0;
#pragma unroll
            for (int u = 0; u < PPT; ++u) {
                // lidar_agent.py:106-110, sqrt-free (thresholds on s are exact, geometry.sqrt_thresholds)
                const float s2 = __fadd_rn(__fmul_rn(xr[u], xr[u]), __fmul_rn(yr[u], yr[u]));
                const bool keep = !close[u] && (s2 >= P.s_lo) && (s2 <= P.s_hi) && (zr[u] < P.z_max) && (zr[u] > P.z_min);
                // BEV cell, lidar_agent.py:547-552 (garbage for dropped points is clamped and never used)
                uint32_t ix, iy;
                s4_bev_cell_xy<FASTDIV>(xr[u], yr[u], P.bev_range, two_r, rcp_two_r, resf, (uint32_t)res_m1, ix, iy);
                const uint32_t ci = (iy >> L.cull_shift) * (uint32_t)L.cull_dim + (ix >> L.cull_shift);
                const uint32_t ids = lds32(cull_s + (ci << 2));
                const uint32_t wx = ix - (uint32_t)win_lo, wy = iy - (uint32_t)win_lo;
                const bool inwin = max(wx, wy) < (uint32_t)win_w;
                // ---- phase C: the atomic that counts the point returns its cell's edge code.  Window cells count into the window, cells
                // outside it into their cull cell's word, dropped points into one of the lane's two sink words (code 0)
                uint32_t wa = inwin ? wcount_s + ((wy * (uint32_t)win_stride + wx) << 2) : pcnt_s + (ci << 2);
                wa = keep ? wa : (close[u] ? sink_close_s : sink_gate_s);
                const uint32_t old = atom_shared_add(wa, 1u);
                red_shared_add((keep && !inwin) ? sink_close_s + isum_delta : wa + isum_delta, q[u]);
                if (keep && zr[u] < P.ground_z) ++c_ground;  // lidar_agent.py:128
                code[u] = old >> kS4CodeShift;
                cand[u] = keep ? ids : kCullEmpty;
                // cells outside the window take one 64-bit reduction on the global (count, isum) cell, the max-height layer one on the float
                // bits for z > 0 (lidar_agent.py:560, 0-initialised max); both predicated, no branch
                const uint32_t lin = iy * (uint32_t)res + ix;
                s4_red_global_u64_if(ci64g + lin, 1ull | ((unsigned long long)q[u] << 32), keep && !inwin);
                s4_red_global_max_if(h32g + lin, __float_as_int(zr[u]), keep && zr[u] > 0.0f);
            }
            // ---- phase D: points that have candidate boxes go to this warp's queue; whenever 32 are pending every lane tests
            // one of them (dense), instead of a handful of lanes looping while the rest of the warp idles.  The queue is drained at the top
            // of the next iteration (and here, half way, only if it could otherwise overflow).
#pragma unroll
            for (int u = 0; u < PPT; ++u) {
                uint32_t lt_mask;
                asm("mov.u32 %0, %%lanemask_lt;" : "=r"(lt_mask));
                if (FOV) {  // points of cells that a ray crosses (edge code != 0) go to the edge queue
                    const bool edge = code[u] != 0u;
                    const uint32_t me = __ballot_sync(0xffffffffu, edge);
                    if (edge) {
                        const uint32_t slot = (e_tail + __popc(me & lt_mask)) & (uint32_t)(kS4EdgeEntries - 1);
                        asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(eq_s + (slot << 3)), "f"(xr[u]), "f"(yr[u]) : "memory");
                        asm volatile("st.shared.u8 [%0], %1;" ::"r"(eqc_s + slot), "r"(code[u]) : "memory");
                    }
                    e_tail += __popc(me);
                    if (e_tail - e_head >= 32u) {
                        __syncwarp();
                        drain_edges(32u);
                    }
                }
                const bool has = cand[u] != kCullEmpty;
                const uint32_t m = __ballot_sync(0xffffffffu, has);
                if (has) {
                    const uint32_t slot = (q_tail + __popc(m & lt_mask)) & (uint32_t)(kS4QueueEntries - 1);
                    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(queue_s + (slot << 4)), "f"(xr[u]), "f"(yr[u]), "f"(zr[u]),
                                 "f"(__uint_as_float(cand[u]))
                                 : "memory");
                }
                q_tail += __popc(m);
                if (PPT == 4 ? (u == 1 && q_tail - q_head >= 64u) : (u == 0 && q_tail - q_head >= 32u)) {  // (so that the next slot(s) fit)
                    __syncwarp();
                    drain_queue(kDrain);
                }
            }
          }
        }
        while (q_tail != q_head) {
            __syncwarp();
            drain_queue(min(q_tail - q_head, kDrain));
        }
        if (FOV && e_tail != e_head) {  // (fewer than 32 are left)
            __syncwarp();
            drain_edges(e_tail - e_head);
        }

        // ------------------------------------------------------------ epilogue
        __syncthreads();  // every tile of this part is accumulated
        // Everything that leaves the CTA is additive (or a min): per-thread counters, then the sink / window / cull-cell words -- window
        // cells go to the global layers, the counts give n_removed and n_kept and, times the cameras that hold a whole cell, the decided
        // share of the per-camera counts.
        uint32_t kept = 0, removed = 0, flags = 0, camc[MSC_MAX_CAMS];
#pragma unroll
        for (int c = 0; c < MSC_MAX_CAMS; ++c) camc[c] = FOV ? cam_byte(cam_lo, cam_hi, c) : 0u;
        if (tid < 32) removed = arrA[tid];
        for (int i = tid; i < n_cull; i += NT) {  // periphery points, per cull cell
            const uint32_t c0 = pcnt[i] & kS4CountMask;
            if (c0 == 0u) continue;
            kept += c0;
            if (FOV) {
                const uint32_t d0 = s4_decided_in(cullcls[i]);
#pragma unroll
                for (int c = 0; c < MSC_MAX_CAMS; ++c) camc[c] += ((d0 >> c) & 1u) ? c0 : 0u;
            }
        }
        unsigned long long* const ci64 = reinterpret_cast<unsigned long long*>(g_ci);
        {
            const int half_w = win_w >> 1;  // win_w and win_lo are even -> 16-byte aligned rows of the global layer
            for (int i = tid; i < win_w * half_w; i += NT) {
                const int wy = i / half_w, wx = (i - wy * half_w) * 2;
                const uint2 c2 = make_uint2(wcount[wy * win_stride + wx], wcount[wy * win_stride + wx + 1]);
                const uint2 s2 = make_uint2(wisum[wy * win_stride + wx], wisum[wy * win_stride + wx + 1]);
                const uint32_t c0 = c2.x & kS4CountMask, c1 = c2.y & kS4CountMask;
                const int cx = wx + win_lo, cy = wy + win_lo;
                const size_t cell = (size_t)cy * (size_t)res + (size_t)cx;
                uint32_t t0 = c0, t1 = c1;  // the cells' counts once this part's points are in
                if (n_parts == 1) {
                    *reinterpret_cast<uint4*>(g_ci + cell * 2) = make_uint4(c0, s2.x, c1, s2.y);
                } else {  // a part of a straddling sample merges with atomics (stream4_straddle_kernel zero-filled the layers); the part whose
                    // add takes a cell to 65536 sees it in the returned count, so the flag does not depend on how the sample is split
                    if (c0) t0 += (uint32_t)atomicAdd(ci64 + cell, (unsigned long long)c0 | ((unsigned long long)s2.x << 32));
                    if (c1) t1 += (uint32_t)atomicAdd(ci64 + cell + 1, (unsigned long long)c1 | ((unsigned long long)s2.y << 32));
                }
                if ((c0 | c1) == 0u) continue;
                kept += c0 + c1;
                flags |= (t0 >= 65536u || t1 >= 65536u) ? 1u : 0u;
                if (FOV) {
                    const uint32_t d0 = s4_decided_in(class_of(cx, cy)), d1 = s4_decided_in(class_of(cx + 1, cy));
#pragma unroll
                    for (int c = 0; c < MSC_MAX_CAMS; ++c) camc[c] += (((d0 >> c) & 1u) ? c0 : 0u) + (((d1 >> c) & 1u) ? c1 : 0u);
                }
            }
        }
        {
            uint32_t v[4 + MSC_MAX_CAMS];
            v[0] = removed; v[1] = kept; v[2] = c_ground; v[3] = 0u;
#pragma unroll
            for (int c = 0; c < MSC_MAX_CAMS; ++c) v[4 + c] = camc[c];
#pragma unroll
            for (int i = 0; i < 4 + (FOV ? MSC_MAX_CAMS : 0); ++i) {
                if (i == 3) continue;
                const uint32_t r = __reduce_add_sync(0xffffffffu, v[i]);
                if (lane == 0 && r) atomicAdd(&misc->stats[1 + i], r);  // [1] removed, [2] kept, [3] ground, [5 + c] per camera
            }
            const uint32_t f = __reduce_or_sync(0xffffffffu, flags);
            if (lane == 0 && f) atomicOr(&misc->stats[13], f);
        }
        __syncthreads();
        uint32_t* const g_stats = A.out.stats + (size_t)sample * MSC_STATS_STRIDE;
        bool finalise = true;
        if (n_parts > 1) {
            unsigned long long* const scr = reinterpret_cast<unsigned long long*>(ws + T.boxscr_off) + (size_t)bx0 * 4;
            for (int b = tid; b < n_boxes; b += NT) {
                const uint32_t* acc = boxacc + b * kAccWords;
                if (acc[0]) {
                    uint32_t* s32 = reinterpret_cast<uint32_t*>(scr + (size_t)b * 4);
                    atomicAdd(s32, acc[0]);
                    atomicMin(s32 + 1, acc[1]);
#pragma unroll
                    for (int k = 0; k < 3; ++k) atomicAdd(scr + (size_t)b * 4 + 1 + k, (unsigned long long)acc[2 + k] + ((unsigned long long)acc[5 + k] << 32));
                }
            }
            uint32_t* const gsc = reinterpret_cast<uint32_t*>(ws + T.splitstats_off) + (size_t)sample * MSC_STATS_STRIDE;
            if (tid < MSC_STATS_STRIDE && tid != 15 && misc->stats[tid]) {
                if (tid == 13) atomicOr(gsc + tid, misc->stats[tid]); else atomicAdd(gsc + tid, misc->stats[tid]);
            }
            // the part that takes the last ticket sees every other part's reductions and finalises the sample
            __threadfence();
            __syncthreads();
            if (tid == 0) misc->ticket = (int32_t)atomicAdd(gsc + 15, 1u);
            __syncthreads();
            finalise = misc->ticket == (int32_t)n_parts - 1;
            if (finalise) {
                __threadfence();
                if (tid < MSC_STATS_STRIDE && tid != 15) misc->stats[tid] = __ldcg(gsc + tid);
            }
        }
        if (finalise) {
            const unsigned long long* const scr = reinterpret_cast<const unsigned long long*>(ws + T.boxscr_off) + (size_t)bx0 * 4;
            for (int b = tid; b < n_boxes; b += NT) {
                uint32_t cnt, mn;
                unsigned long long sum3[3];
                if (n_parts == 1) {
                    const uint32_t* acc = boxacc + b * kAccWords;
                    cnt = acc[0]; mn = acc[1];
#pragma unroll
                    for (int k = 0; k < 3; ++k) sum3[k] = (unsigned long long)acc[2 + k] + ((unsigned long long)acc[5 + k] << 32);
                } else {
                    const unsigned long long w0 = __ldcg(scr + (size_t)b * 4);
                    cnt = (uint32_t)w0; mn = (uint32_t)(w0 >> 32);
#pragma unroll
                    for (int k = 0; k < 3; ++k) sum3[k] = __ldcg(scr + (size_t)b * 4 + 1 + k);
                }
                const size_t o = (size_t)(bx0 + b);
                float nearest = INFINITY, cen[3] = {0.0f, 0.0f, 0.0f};
                if (cnt != 0) {
                    nearest = __fsqrt_rn(__uint_as_float(mn));
#pragma unroll
                    for (int k = 0; k < 3; ++k) cen[k] = box_centroid(A, cnt, sum3[k]);
                }
                A.out.box_count[o] = cnt;
                A.out.box_nearest[o] = nearest;
                A.out.box_centroid[o * 3 + 0] = cen[0]; A.out.box_centroid[o * 3 + 1] = cen[1]; A.out.box_centroid[o * 3 + 2] = cen[2];
                for (int r = 0; r < A.n_replicas; ++r) {  // the same entry on the other GPUs of the box (P2P stores)
                    A.replica[r].box_count[o] = cnt;
                    A.replica[r].box_nearest[o] = nearest;
                    A.replica[r].box_centroid[o * 3 + 0] = cen[0]; A.replica[r].box_centroid[o * 3 + 1] = cen[1]; A.replica[r].box_centroid[o * 3 + 2] = cen[2];
                }
            }
            __syncthreads();  // (a straddling sample: misc->stats holds the merged counters)
            if (tid < MSC_STATS_STRIDE) {
                uint32_t v = misc->stats[tid];
                uint32_t n_in = 0;
                if (tid <= 1)
                    for (int s = sw0; s < sw1; ++s) n_in += A.in.sweep_count[s];
                if (tid == 0) v = n_in;
                if (tid == 1) v = n_in - v;                            // n_after_close = n_in - removed
                if (tid == 4) v = misc->stats[2] - misc->stats[3];     // n_object = n_kept - n_ground
                if (tid == 13 && box_overflow) v |= 0x80000000u;
                if (tid == 15) v = 0u;
                g_stats[tid] = v;
                for (int r = 0; r < A.n_replicas; ++r) A.replica[r].stats[(size_t)sample * MSC_STATS_STRIDE + tid] = v;
            }
        }
    }
}

template <bool FOV, bool FASTDIV, int PPT, bool STD>
static int s4_launch_one(const FusedArgs& args, const TableLayout& T, unsigned char* ws, int grid, cudaStream_t stream) {
    auto kern = stream4_kernel<FOV, FASTDIV, PPT, STD>;
    MSC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, args.L.total_bytes));
    kern<<<grid, s4_threads(PPT), args.L.total_bytes, stream>>>(args, T, ws);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

// the partition pre-kernel (zero-fill of the samples that straddle CTA boundaries; the tile prefix per sample comes from fused_tables_kernel)
int launch_stream4_partition(const FusedArgs& args, const TableLayout& T, unsigned char* ws, int grid, cudaStream_t stream, int* launches) {
    if (grid > 1) {
        stream4_straddle_kernel<<<grid - 1, 256, 0, stream>>>(args, T, ws, grid);
        MSC_CUDA(cudaGetLastError());
        ++*launches;
    }
    return MSC_OK;
}

template <int PPT>
static int s4_launch_ppt(const FusedArgs& args, const TableLayout& T, unsigned char* ws, int grid, bool fov, bool fast, cudaStream_t stream) {
    if (fov) return fast ? s4_launch_one<true, true, PPT, false>(args, T, ws, grid, stream) : s4_launch_one<true, false, PPT, false>(args, T, ws, grid, stream);
    return fast ? s4_launch_one<false, true, PPT, false>(args, T, ws, grid, stream) : s4_launch_one<false, false, PPT, false>(args, T, ws, grid, stream);
}

// standard: the compile-time-constant instantiation (stream4_is_standard() held for this call: PPT 2, the Markstein division applies)
int launch_stream4_kernel(const FusedArgs& args, const TableLayout& T, unsigned char* ws, int grid, int ppt, bool fov, bool fast, bool standard,
                          cudaStream_t stream) {
    if (standard && ppt == 2 && fast)
        return fov ? s4_launch_one<true, true, 2, true>(args, T, ws, grid, stream) : s4_launch_one<false, true, 2, true>(args, T, ws, grid, stream);
    return ppt == 4 ? s4_launch_ppt<4>(args, T, ws, grid, fov, fast, stream) : s4_launch_ppt<2>(args, T, ws, grid, fov, fast, stream);
}

}  // namespace msc
