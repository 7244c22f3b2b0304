// fused_evidence.cu -- host side of the fused hot path (msc_fused_* entry points) and its three table kernels.
//
// The hot path is one pass over the raw sweeps of a batch of samples (stream4.cu; fused_stream.cu for fov_keep_mask != 0).
// Everything that does not touch points runs once per batch in small, fully parallel kernels and lands in the workspace:
// prepared boxes (devkit points_in_box vectors, App. A.2), box -> camera projection (A.3), camera wedges, the per-cell
// edge classes of the wedges, and the candidate-box ids of every cull cell.  Semantics: SURVEY.md App. A.
#include <mutex>

#include "fused_common.cuh"

namespace msc {

// ------------------------------------------------------------------------------------------------ table kernel
// Everything that does not touch points runs once per batch in a small, fully parallel kernel and lands in the
// workspace: prepared boxes (devkit points_in_box vectors, App. A.2), box -> camera projection (A.3), camera
// wedges, and the per-cull-cell wedge classes.  The streaming kernel then only copies its sample's rows to smem.


// camera wedge: apex = camera centre in the sensor xy-plane, edges = image columns 0 and W (f64, no FMA)
__device__ void compute_wedge(int image_w, const double* __restrict__ lcal, const double* __restrict__ ccal, const double* __restrict__ K,
                              float* __restrict__ wq) {
    double Rl[9], Rc[9];
    quat_to_rot(lcal + 3, Rl);
    quat_to_rot(ccal + 3, Rc);
    const double d0 = ccal[0] - lcal[0], d1 = ccal[1] - lcal[1], d2 = ccal[2] - lcal[2];
    const double ox = (Rl[0] * d0 + Rl[3] * d1) + Rl[6] * d2;
    const double oy = (Rl[1] * d0 + Rl[4] * d1) + Rl[7] * d2;
    const double fx = K[0], cxp = K[2];
    const double dl[3] = {(0.0 - cxp) / fx, 0.0, 1.0};
    const double dr[3] = {((double)image_w - cxp) / fx, 0.0, 1.0};
    double le[3], re[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        le[r] = (Rc[r * 3 + 0] * dl[0] + Rc[r * 3 + 1] * dl[1]) + Rc[r * 3 + 2] * dl[2];
        re[r] = (Rc[r * 3 + 0] * dr[0] + Rc[r * 3 + 1] * dr[1]) + Rc[r * 3 + 2] * dr[2];
    }
    wq[0] = (float)ox; wq[1] = (float)oy;
    wq[2] = (float)((Rl[0] * le[0] + Rl[3] * le[1]) + Rl[6] * le[2]);
    wq[3] = (float)((Rl[1] * le[0] + Rl[4] * le[1]) + Rl[7] * le[2]);
    wq[4] = (float)((Rl[0] * re[0] + Rl[3] * re[1]) + Rl[6] * re[2]);
    wq[5] = (float)((Rl[1] * re[0] + Rl[4] * re[1]) + Rl[7] * re[2]);
}

// grid: ceil(max(n_boxes_total, n_samples) * max(n_cams,1) / 256) blocks of 256 threads
__global__ void __launch_bounds__(256) fused_tables_kernel(const __grid_constant__ FusedArgs A, const TableLayout T, int n_boxes_total,
                                                          unsigned char* __restrict__ ws, uint32_t tile_pts) {
    const msc_params& P = A.P;
    const int n_cams = P.n_cams;
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    float* const boxprep = reinterpret_cast<float*>(ws + T.boxprep_off);
    float* const wedges = reinterpret_cast<float*>(ws + T.wedge_off);
    // (0) housekeeping that would otherwise be two memsets: the streaming kernel's work counter and the candidate-id table
    // (kCullEmpty everywhere; fused_cullids_kernel inserts into it after this kernel)
    {
        const size_t nthreads = (size_t)gridDim.x * blockDim.x;
        if (gid == 0) *reinterpret_cast<uint32_t*>(ws + T.counter_off) = 0u;
        uint32_t* ids = reinterpret_cast<uint32_t*>(ws + T.cullids_off);
        const size_t n_ids = (size_t)A.in.n_samples * (size_t)(A.L.cull_dim * A.L.cull_dim);
        for (size_t i = gid; i < n_ids; i += nthreads) ids[i] = kCullEmpty;
    }
    // sample of a global box index: binary search in sample_box_off
    auto sample_of_box = [&](int gb) {
        int lo = 0, hi = A.in.n_samples;
        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (A.in.sample_box_off[mid] <= gb) lo = mid; else hi = mid; }
        return lo;
    };
    // (1) prepared boxes: one thread per box
    if (gid < n_boxes_total) {
        const int sample = sample_of_box(gid);
        const double* box = A.in.boxes + (size_t)gid * 10;
        double c[3] = {box[0], box[1], box[2]};
        double R[9];
        quat_to_rot(box + 6, R);
        frame_change(A.in.ego_pose + (size_t)sample * 7, c, R);
        frame_change(A.in.lidar_calib + (size_t)sample * 7, c, R);
        box_record(box, c, R, boxprep + (size_t)gid * kBoxStride);
    }
    // (2) box -> camera projection (App. A.3): one thread per (box, camera)
    if (n_cams > 0 && gid < n_boxes_total * n_cams) {
        const int gb = gid / n_cams, c = gid - gb * n_cams;
        const int sample = sample_of_box(gb);
        project_box(A.in.boxes + (size_t)gb * 10, A.in.cam_ego_pose + ((size_t)sample * n_cams + c) * 7,
                    A.in.cam_calib + ((size_t)sample * n_cams + c) * 7, A.in.cam_K + ((size_t)sample * n_cams + c) * 9, (double)P.image_w,
                    (double)P.image_h, A.out.proj_visible + gid, A.out.proj_extent + (size_t)gid * 4);
        if (A.n_replicas > 0) {  // the same entry on the other GPUs of the box (P2P stores)
            const uint8_t vis = A.out.proj_visible[gid];
            const float4 ext = *reinterpret_cast<const float4*>(A.out.proj_extent + (size_t)gid * 4);
            for (int r = 0; r < A.n_replicas; ++r) {
                A.replica[r].proj_visible[gid] = vis;
                *reinterpret_cast<float4*>(A.replica[r].proj_extent + (size_t)gid * 4) = ext;
            }
        }
    }
    // (3) camera wedges: one thread per (sample, camera)
    if (n_cams > 0 && gid < A.in.n_samples * n_cams) {
        const int sample = gid / n_cams, c = gid - sample * n_cams;
        compute_wedge(P.image_w, A.in.lidar_calib + (size_t)sample * 7, A.in.cam_calib + ((size_t)sample * n_cams + c) * 7,
                      A.in.cam_K + ((size_t)sample * n_cams + c) * 9, wedges + ((size_t)sample * MSC_MAX_CAMS + c) * 6);
    }
    // (4) stream4.cu's static partition: tile_off[s] = warp tiles (tile_pts rows of one sweep) of samples [0, s); the first block scans
    // (it is scheduled first, so its serial passes over the sweep counts run beside the other blocks' projections, not after them)
    if (tile_pts != 0u && blockIdx.x == 0) {
        __shared__ uint32_t part[256];
        uint32_t* const tile_off = reinterpret_cast<uint32_t*>(ws + T.tileoff_off);
        const int n = A.in.n_samples, tid = threadIdx.x;
        const int per = (n + 255) / 256;
        const int s0 = min(tid * per, n), s1 = min(s0 + per, n);
        auto tiles_of = [&](int s) {
            uint32_t t = 0;
            for (int w = A.in.sample_sweep_off[s]; w < A.in.sample_sweep_off[s + 1]; ++w) t += (A.in.sweep_count[w] + tile_pts - 1u) / tile_pts;
            return t;
        };
        uint32_t sum = 0;
        for (int s = s0; s < s1; ++s) sum += tiles_of(s);
        part[tid] = sum;
        __syncthreads();
        for (int d = 1; d < 256; d <<= 1) {  // inclusive scan
            const uint32_t v = tid >= d ? part[tid - d] : 0u;
            __syncthreads();
            part[tid] += v;
            __syncthreads();
        }
        uint32_t run = part[tid] - sum;
        for (int s = s0; s < s1; ++s) { tile_off[s] = run; run += tiles_of(s); }
        if (tid == 255) tile_off[n] = part[255];
    }
}

// Candidate-box ids per (sample, cull cell): conservative oriented rasterisation of every box footprint, one warp per box (lanes
// share the cells of its bounding rectangle), into a workspace table the host pre-fills with kCullEmpty.
__global__ void __launch_bounds__(128) fused_cullids_kernel(const __grid_constant__ FusedArgs A, const TableLayout T, unsigned char* __restrict__ ws) {
    const int sample = blockIdx.x, lane = threadIdx.x & 31;
    const int bx0 = A.in.sample_box_off[sample];
    int n_boxes = A.in.sample_box_off[sample + 1] - bx0;
    if (n_boxes > A.L.max_boxes) n_boxes = A.L.max_boxes;  // caller under-declared max_boxes_per_sample: the streaming kernel drops these boxes too
    uint32_t* ids = reinterpret_cast<uint32_t*>(ws + T.cullids_off) + (size_t)sample * (size_t)(A.L.cull_dim * A.L.cull_dim);
    // the grid has a warp per DECLARED box; the loop covers samples that hold more (up to the room the streaming kernel has)
    const int stride = (int)(gridDim.y * blockDim.x) >> 5;
    for (int b = (int)(blockIdx.y * blockDim.x + threadIdx.x) >> 5; b < n_boxes; b += stride) {
        const float* o = reinterpret_cast<const float*>(ws + T.boxprep_off) + (size_t)(bx0 + b) * kBoxStride;
        rasterise_box<1>(A, o, b, ids, lane, 32);
    }
}


}  // namespace msc

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
constexpr int kTimeRing = 64;

// One context per caller (host thread / engine): options, the timing ring and the facts about the
// most recent call live here, not in process globals, so contexts on different host threads, streams or devices never share state.
struct msc_fused_ctx {
    int device = 0, sms = 0, smem_optin = 0;
    int opt_fov = 1;
    int opt_window = 0;        // 0 = auto (largest that fits)
    int opt_cull_shift = -1;   // -1 = auto (cull cell ~ 2 m)
    int opt_fastdiv = 1;       // allow the Markstein division for whitelisted divisors
    int opt_config = 0;        // 0 = auto: stream4.cu; 10 / 7 force stream4.cu / fused_stream.cu (fov_keep_mask != 0 always takes fused_stream.cu)
    int opt_grid = 0;          // stream4.cu: CTAs of the launch, 0 = auto (the SM count, fewer for batches of a few thousand rows)
    int opt_ppt = 2;           // stream4.cu: points per lane, 2 (1024 threads) or 4 (512 threads)
    int opt_std = 1;           // stream4.cu: allow the compile-time-constant instantiation for the standard configuration
    int last_standard = 0;
    int opt_time_kernel = 0;   // bracket the streaming kernel with CUDA events (msc_fused_kernel_times)
    int last_window = 0, last_smem = 0, last_fastdiv = 0, last_tile_pts = 0, last_threads = 0, last_launches = 0, last_grid = 0, last_config = 0;
    bool ev_made = false;
    cudaEvent_t ev0[kTimeRing], ev1[kTimeRing];
    long long ev_count = 0;  // calls timed so far
    std::mutex mu;           // serialises calls that share this context
};

namespace msc {

static int time_begin(msc_fused_ctx* X, cudaStream_t stream) {
    if (!X->opt_time_kernel) return MSC_OK;
    if (!X->ev_made) {
        for (int i = 0; i < kTimeRing; ++i) { MSC_CUDA(cudaEventCreate(&X->ev0[i])); MSC_CUDA(cudaEventCreate(&X->ev1[i])); }
        X->ev_made = true;
    }
    MSC_CUDA(cudaEventRecord(X->ev0[X->ev_count % kTimeRing], stream));
    return MSC_OK;
}
static int time_end(msc_fused_ctx* X, cudaStream_t stream) {
    if (!X->opt_time_kernel) return MSC_OK;
    MSC_CUDA(cudaEventRecord(X->ev1[X->ev_count % kTimeRing], stream));
    ++X->ev_count;
    return MSC_OK;
}

// divisors 2*bev_range for which tools/markstein_check.c has been run over the full float range
static bool fastdiv_verified(float two_r) {
    const float ok[] = {100.0f, 102.4f, 120.0f, 150.0f, 160.0f, 200.0f};
    for (float v : ok)
        if (two_r == v) return true;
    int e = 0;
    return frexpf(two_r, &e) == 0.5f;  // powers of two divide exactly either way
}

static void cull_geometry(const msc_params& P, int opt_cull_shift, int* shift, int* dim) {
    const float cell_m = 2.0f * P.bev_range / (float)P.bev_res;
    int sh = 0;
    if (opt_cull_shift >= 0) sh = opt_cull_shift;
    else {
        // auto: the largest power-of-two multiple of a BEV cell that is not above 2 m -- and coarser still until the cull grid has at
        // most 64 x 64 cells (its id and count tables sit in shared memory: 32 KB; e.g. 0.512 m cells would give a 100 x 100 grid)
        while ((float)(1 << (sh + 1)) * cell_m <= 2.0f + 1e-6f && sh < 10) ++sh;
        while ((((P.bev_res - 1) >> sh) + 1) > 64 && sh < 10) ++sh;
    }
    *shift = sh;
    *dim = ((P.bev_res - 1) >> sh) + 1;
}

constexpr int kMaxGrid = 256;  // upper bound of the streaming kernels' grid (one CTA per SM)

static TableLayout table_layout(const msc_params& P, int n_samples, int n_boxes, int cull_dim) {
    auto align = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t ns = (size_t)(n_samples > 0 ? n_samples : 1), nb = (size_t)(n_boxes > 0 ? n_boxes : 1);
    const size_t dim = (size_t)cull_dim;
    TableLayout T;
    size_t off = 0;
    T.counter_off = off; off = align(off + 256);
    T.boxprep_off = off; off = align(off + nb * kBoxStride * 4);
    T.wedge_off = off; off = align(off + ns * MSC_MAX_CAMS * 6 * 4);
    T.cullids_off = off; off = align(off + ns * dim * dim * 4);
    T.boxscr_off = off; off = align(off + nb * 32);
    T.splitstats_off = off; off = align(off + ns * MSC_STATS_STRIDE * 4);
    T.tileoff_off = off; off = align(off + (ns + 1) * 4);
    T.cls_off = off; off = align(off + (size_t)kMaxGrid * (dim * dim + (size_t)kInnerMax * kInnerMax) * 4);
    T.total = off;
    return T;
}

// tables (prepared boxes, projection, wedges, housekeeping -> workspace), then the candidate-box ids of every cull cell; the per-cell
// edge classes of the camera wedges are computed by the streaming kernels themselves, per sample, from the wedges
static int launch_tables(msc_fused_ctx* X, const FusedArgs& args, const TableLayout& T, unsigned char* ws, int n_boxes_total, int tile_pts,
                         int declared_max_boxes, cudaStream_t stream) {
    const int cams = args.P.n_cams > 0 ? args.P.n_cams : 1;
    long long work = (long long)n_boxes_total * cams;
    if ((long long)args.in.n_samples * cams > work) work = (long long)args.in.n_samples * cams;
    X->last_launches = 0;
    const unsigned blocks = (unsigned)((work + 255) / 256);
    fused_tables_kernel<<<blocks < 1 ? 1 : blocks, 256, 0, stream>>>(args, T, n_boxes_total, ws, (uint32_t)tile_pts);
    MSC_CUDA(cudaGetLastError());
    ++X->last_launches;
    if (n_boxes_total > 0 && args.L.max_boxes > 0) {
        int per_sample = declared_max_boxes < args.L.max_boxes ? declared_max_boxes : args.L.max_boxes;
        if (per_sample < 1) per_sample = 1;
        const dim3 cgrid((unsigned)args.in.n_samples, (unsigned)((per_sample + 3) / 4));  // a warp per declared box, one grid column per sample
        fused_cullids_kernel<<<cgrid, 128, 0, stream>>>(args, T, ws);
        MSC_CUDA(cudaGetLastError());
        ++X->last_launches;
    }
    return MSC_OK;
}

}  // namespace msc

extern "C" {

int msc_fused_create(msc_fused_ctx** out) {
    using namespace msc;
    MSC_REQUIRE(out, "null argument");
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        set_error("no CUDA device visible");
        return MSC_ERR_NO_DEVICE;
    }
    msc_fused_ctx* X = new (std::nothrow) msc_fused_ctx();
    MSC_REQUIRE(X, "out of host memory");
    cudaError_t e = cudaGetDevice(&X->device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&X->sms, cudaDevAttrMultiProcessorCount, X->device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&X->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, X->device);
    if (e != cudaSuccess) {
        set_error("device query failed: %s", cudaGetErrorString(e));
        delete X;
        return MSC_ERR_LAUNCH;
    }
    *out = X;
    return MSC_OK;
}

int msc_fused_destroy(msc_fused_ctx* X) {
    if (!X) return MSC_OK;
    if (X->ev_made)
        for (int i = 0; i < kTimeRing; ++i) { cudaEventDestroy(X->ev0[i]); cudaEventDestroy(X->ev1[i]); }
    delete X;
    return MSC_OK;
}

size_t msc_fused_workspace_bytes(const msc_fused_ctx* X, const msc_params* params, int32_t n_samples, int32_t n_boxes) {
    if (!params || params->bev_res <= 0) return 0;
    int cshift = 0, cdim = 0;
    msc::cull_geometry(*params, X ? X->opt_cull_shift : -1, &cshift, &cdim);
    return msc::table_layout(*params, n_samples, n_boxes, cdim).total;
}

int msc_fused_set_option(msc_fused_ctx* X, const char* key, int32_t value) {
    using namespace msc;
    MSC_REQUIRE(X && key, "null argument");
    std::lock_guard<std::mutex> lock(X->mu);
    if (!strcmp(key, "fov")) { X->opt_fov = value ? 1 : 0; return MSC_OK; }
    if (!strcmp(key, "window")) { X->opt_window = value; return MSC_OK; }
    if (!strcmp(key, "cull_shift")) { X->opt_cull_shift = value; return MSC_OK; }
    if (!strcmp(key, "fastdiv")) { X->opt_fastdiv = value ? 1 : 0; return MSC_OK; }
    if (!strcmp(key, "config")) { MSC_REQUIRE(value == 0 || value == 7 || value == 10, "config must be 0 (auto), 10 (stream4.cu) or 7 (fused_stream.cu)"); X->opt_config = value; return MSC_OK; }
    if (!strcmp(key, "grid")) { MSC_REQUIRE(value >= 0 && value <= kMaxGrid, "grid out of range"); X->opt_grid = value; return MSC_OK; }
    if (!strcmp(key, "ppt")) { MSC_REQUIRE(value == 2 || value == 4, "ppt must be 2 or 4"); X->opt_ppt = value; return MSC_OK; }
    if (!strcmp(key, "standard")) { X->opt_std = value ? 1 : 0; return MSC_OK; }
    if (!strcmp(key, "time_kernel")) { X->opt_time_kernel = value ? 1 : 0; return MSC_OK; }
    set_error("unknown option %s", key);
    return MSC_ERR_BAD_ARGUMENT;
}

int msc_fused_get_option(msc_fused_ctx* X, const char* key, int32_t* value) {
    using namespace msc;
    MSC_REQUIRE(X && key && value, "null argument");
    std::lock_guard<std::mutex> lock(X->mu);
    if (!strcmp(key, "fov")) { *value = X->opt_fov; return MSC_OK; }
    if (!strcmp(key, "window")) { *value = X->opt_window; return MSC_OK; }
    if (!strcmp(key, "cull_shift")) { *value = X->opt_cull_shift; return MSC_OK; }
    if (!strcmp(key, "fastdiv")) { *value = X->opt_fastdiv; return MSC_OK; }
    if (!strcmp(key, "config")) { *value = X->opt_config; return MSC_OK; }
    if (!strcmp(key, "grid")) { *value = X->opt_grid; return MSC_OK; }
    if (!strcmp(key, "ppt")) { *value = X->opt_ppt; return MSC_OK; }
    if (!strcmp(key, "standard")) { *value = X->opt_std; return MSC_OK; }
    if (!strcmp(key, "last_standard")) { *value = X->last_standard; return MSC_OK; }
    if (!strcmp(key, "time_kernel")) { *value = X->opt_time_kernel; return MSC_OK; }
    if (!strcmp(key, "last_window")) { *value = X->last_window; return MSC_OK; }
    if (!strcmp(key, "last_smem")) { *value = X->last_smem; return MSC_OK; }
    if (!strcmp(key, "last_fastdiv")) { *value = X->last_fastdiv; return MSC_OK; }
    if (!strcmp(key, "last_grid")) { *value = X->last_grid; return MSC_OK; }
    if (!strcmp(key, "last_config")) { *value = X->last_config; return MSC_OK; }
    if (!strcmp(key, "tile_pts")) { *value = X->last_tile_pts; return MSC_OK; }
    if (!strcmp(key, "threads")) { *value = X->last_threads; return MSC_OK; }
    if (!strcmp(key, "last_launches")) { *value = X->last_launches; return MSC_OK; }
    set_error("unknown option %s", key);
    return MSC_ERR_BAD_ARGUMENT;
}

int msc_fused_kernel_times(msc_fused_ctx* X, float* out_ms_host, int32_t n) {
    using namespace msc;
    MSC_REQUIRE(X && out_ms_host && n >= 0, "bad argument");
    std::lock_guard<std::mutex> lock(X->mu);
    const long long have = X->ev_count < kTimeRing ? X->ev_count : kTimeRing;
    const int take = (int)(n < have ? n : have);
    for (int i = 0; i < take; ++i) {
        const long long k = X->ev_count - take + i;
        MSC_CUDA(cudaEventSynchronize(X->ev1[k % kTimeRing]));
        MSC_CUDA(cudaEventElapsedTime(out_ms_host + i, X->ev0[k % kTimeRing], X->ev1[k % kTimeRing]));
    }
    return take;
}

int msc_fused_evidence_batch(msc_fused_ctx* X, const msc_params* params, const msc_batch_in* in, const msc_batch_out* out, void* workspace,
                             size_t workspace_bytes, void* stream_v) {
    return msc_fused_evidence_batch_replicated(X, params, in, out, 0, nullptr, workspace, workspace_bytes, stream_v);
}

int msc_fused_evidence_batch_replicated(msc_fused_ctx* X, const msc_params* params, const msc_batch_in* in, const msc_batch_out* out,
                                        int32_t n_replicas, const msc_batch_out* replicas, void* workspace, size_t workspace_bytes, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(X && params && in && out && workspace, "null argument");
    MSC_REQUIRE(n_replicas >= 0 && n_replicas <= MSC_MAX_REPLICAS && (n_replicas == 0 || replicas), "n_replicas out of range");
    MSC_REQUIRE(in->n_samples >= 0 && in->n_boxes >= 0, "negative counts");
    MSC_REQUIRE(params->n_cams >= 0 && params->n_cams <= MSC_MAX_CAMS, "n_cams out of range");
    MSC_REQUIRE(params->bev_res > 0 && params->bev_res <= 4096 && (params->bev_res & 1) == 0, "bev_res must be even and <= 4096");
    MSC_REQUIRE(params->centroid_shift >= 0 && params->centroid_shift <= 17, "centroid_shift out of range (the biased coordinate is a 24-bit value)");
    MSC_REQUIRE(params->intensity_shift >= 0 && params->intensity_shift <= 8, "intensity_shift out of range");
    // the biased fixed-point coordinate must fit 24 bits: |c| * 2^shift < 2^(shift + 6)  <=>  |c| < 64 m
    MSC_REQUIRE(params->range_max < 64.0f && params->z_max < 64.0f && params->z_min > -64.0f, "range_max / z limits must be below 64 m");
    MSC_REQUIRE(in->max_boxes_per_sample >= 0 && in->max_boxes_per_sample <= MSC_MAX_BOXES_FUSED, "more than %d boxes in one sample",
                MSC_MAX_BOXES_FUSED);
    MSC_REQUIRE(in->points_per_sample_hint >= 0, "negative points_per_sample_hint");
    MSC_REQUIRE((((uintptr_t)in->points) & 15) == 0, "points must be 16-byte aligned");
    MSC_REQUIRE((((uintptr_t)workspace) & 255) == 0, "workspace must be 256-byte aligned");
    std::lock_guard<std::mutex> lock(X->mu);
    int dev = 0;
    MSC_CUDA(cudaGetDevice(&dev));
    MSC_REQUIRE(dev == X->device, "context was created on device %d, current device is %d", X->device, dev);
    int cshift = 0, cdim = 0;
    cull_geometry(*params, X->opt_cull_shift, &cshift, &cdim);
    const TableLayout T = table_layout(*params, in->n_samples, in->n_boxes, cdim);
    MSC_REQUIRE(workspace_bytes >= T.total, "workspace too small: need %zu bytes", T.total);
    cudaStream_t stream = (cudaStream_t)stream_v;
    if (in->n_samples == 0) return MSC_OK;
    FusedArgs args;
    args.P = *params;
    args.in = *in;
    args.out = *out;
    args.two_r = 2.0f * params->bev_range;
    args.resf = (float)params->bev_res;
    args.rcp_two_r = 1.0f / args.two_r;
    args.cscale = (float)(1 << params->centroid_shift);
    args.iscale = (float)(1 << params->intensity_shift);
    args.centroid_bias = 1 << (params->centroid_shift + 6);
    args.n_replicas = n_replicas;
    for (int r = 0; r < n_replicas; ++r) args.replica[r] = replicas[r];
    const bool fov = X->opt_fov != 0 && params->n_cams > 0;
    const bool fast = X->opt_fastdiv != 0 && fastdiv_verified(args.two_r);
    // Kernel choice.  stream4.cu: raw rows through one TMA slot per warp, static partition of the batch in warp tiles (any batch size fills
    // the device evenly).  fused_stream.cu: the TMA-ring generation, one sample per CTA at a time -- the only one with the per-point wedge
    // classes a FOV *filter* (fov_keep_mask) needs.
    const bool keepmask = fov && params->fov_keep_mask != 0u;
    MSC_REQUIRE(!(keepmask && n_replicas > 0), "replicated result tables are not available with fov_keep_mask != 0");
    MSC_REQUIRE(!(X->opt_config == 7 && n_replicas > 0), "replicated result tables need the stream4.cu kernel (config 0 or 10)");
    int gen = keepmask ? 7 : X->opt_config;
    if (gen == 0) gen = 10;  // (on batches that fill the device the two kernels measure the same; stream4.cu also fills it on every other batch)
    const bool s4 = gen == 10;
    X->last_fastdiv = fast ? 1 : 0;
    unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
    // fine edge classes for the kInnerMax x kInnerMax BEV cells around the sensor, where several image-column rays cross a 2 m cull cell
    int inner = fov ? (params->bev_res < kInnerMax ? params->bev_res : kInnerMax) : 0;
    inner &= ~1;
    bool standard = false;
    int tile_pts, threads, grid;
    if (s4) {
        // the box tables are sized for the standard capacity when the batch fits it, so that the layout -- and with it the choice of
        // the compile-time-constant instantiation -- does not depend on the batch
        const int cap = in->max_boxes_per_sample <= stream4_std_boxes() ? stream4_std_boxes() : in->max_boxes_per_sample;
        args.L = stream4_layout(X->smem_optin, X->opt_ppt, params->bev_res, cdim, cshift, cap, X->opt_window, inner);
        standard = args.L.win_w >= 0 && fast && stream4_is_standard(args, X->smem_optin, X->opt_ppt, X->opt_window) && X->opt_std != 0;
        tile_pts = 128; threads = stream4_threads(X->opt_ppt);
        // every CTA gets the same number of warp tiles; a batch of a few thousand rows is not spread thinner than one tile per warp
        const long long pts = in->points_per_sample_hint > 0 ? in->points_per_sample_hint : 347200;
        const long long est_tiles = (long long)in->n_samples * ((pts + tile_pts - 1) / tile_pts);
        const long long g = X->opt_grid > 0 ? X->opt_grid : 2 * est_tiles / (threads / 32);  // (small batches: down to half a tile per warp)
        grid = (int)(g < 1 ? 1 : (g > X->sms ? X->sms : g));
        if (grid > kMaxGrid) grid = kMaxGrid;
    } else {
        args.L = stream_layout(X->smem_optin, params->bev_res, cdim, cshift, in->max_boxes_per_sample, X->opt_window, inner);
        tile_pts = kStreamTilePts; threads = kStreamThreads;
        grid = in->n_samples < X->sms ? in->n_samples : X->sms;
    }
    X->last_tile_pts = tile_pts; X->last_threads = threads;
    if (args.L.win_w < 0) {
        set_error("shared-memory layout does not fit (%d bytes available)", X->smem_optin);
        return MSC_ERR_UNSUPPORTED;
    }
    X->last_config = gen;
    X->last_window = args.L.win_w;
    X->last_smem = args.L.total_bytes;
    int rc;
    // (stream4.cu's static partition: the table kernel prefix-sums the warp tiles of every sample, a pre-kernel zero-fills the samples
    // that straddle CTAs)
    if ((rc = launch_tables(X, args, T, ws, in->n_boxes, s4 ? tile_pts : 0, in->max_boxes_per_sample, stream)) != MSC_OK) return rc;
    if (s4 && (rc = launch_stream4_partition(args, T, ws, grid, stream, &X->last_launches)) != MSC_OK) return rc;
    X->last_grid = grid;
    if ((rc = time_begin(X, stream)) != MSC_OK) return rc;
    rc = s4 ? launch_stream4_kernel(args, T, ws, grid, X->opt_ppt, fov, fast, standard, stream) : launch_stream_kernel(args, T, ws, grid, fov, fast, stream);
    X->last_standard = standard ? 1 : 0;
    if (rc != MSC_OK) return rc;
    ++X->last_launches;
    return time_end(X, stream);
}

}  // extern "C"
