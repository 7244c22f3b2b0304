// cluster_mosaic.cu -- the classifier mosaics of LiDARAgent._classify_batch_with_llm (lidar_agent.cluster_mosaic) from cluster views
// already on the device: one launch copies the views into their cells, a second writes each count's stamp (the '#idx' labels and the
// white of the empty cells, lidar_agent.mosaic_stamp) over them.
#include <algorithm>
#include <vector>

#include "msc_common.cuh"

namespace msc {

constexpr int kView = 512;
constexpr int kViewChunks = kView * 3 / 16;  // 16-byte chunks per view row

struct MosaicRec {
    int64_t off;           // first byte in out_bgr
    int32_t first, count;  // views
    int32_t cols, rows;
};

__host__ __device__ __forceinline__ int mosaic_cols(int count) { return count < 3 ? count : 3; }
__host__ __device__ __forceinline__ int mosaic_rows(int count) { return (count + 2) / 3; }

// grid (chunks, mosaics): 16-byte chunks of mosaic blockIdx.y; a chunk lies in one cell (a view row is 96 chunks)
__global__ void __launch_bounds__(256) mosaic_copy_kernel(const MosaicRec* __restrict__ rec, const uint4* __restrict__ views, uint8_t* __restrict__ out) {
    const MosaicRec m = rec[blockIdx.y];
    const int64_t chunks = (int64_t)m.rows * kView * m.cols * kViewChunks;
    uint4* dst = reinterpret_cast<uint4*>(out + m.off);
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < chunks; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t y = k / (m.cols * kViewChunks);
        const int xc = (int)(k - y * m.cols * kViewChunks);
        const int cell = (int)(y / kView) * m.cols + xc / kViewChunks;
        if (cell >= m.count) continue;  // empty cells: the stamp makes them white
        dst[k] = views[((int64_t)(m.first + cell) * kView + y % kView) * kViewChunks + xc % kViewChunks];
    }
}

__global__ void __launch_bounds__(256) mosaic_stamp_kernel(const MosaicRec* __restrict__ rec, const uint32_t* __restrict__ stamps,
                                                           const int32_t* __restrict__ stamp_off, uint8_t* __restrict__ out) {
    const MosaicRec m = rec[blockIdx.y];
    if (m.count < 2) return;
    const int32_t a = stamp_off[m.count], b = stamp_off[m.count + 1];
    for (int32_t j = a + (int32_t)(blockIdx.x * blockDim.x + threadIdx.x); j < b; j += gridDim.x * blockDim.x) {
        const uint32_t px = stamps[2 * j], col = stamps[2 * j + 1];
        uint8_t* o = out + m.off + (int64_t)px * 3;
        o[0] = (uint8_t)col; o[1] = (uint8_t)(col >> 8); o[2] = (uint8_t)(col >> 16);
    }
}

}  // namespace msc

extern "C" {

size_t msc_cluster_mosaics_workspace_bytes(int32_t n) {
    if (n < 0 || n > 65535) return 0;
    const size_t b = ((size_t)n * sizeof(msc::MosaicRec) + 12 * 4 + 255) & ~(size_t)255;
    return b > 256 ? b : 256;
}

int msc_cluster_mosaics(const uint8_t* views, int32_t n_views, const int32_t* groups, int32_t n, const uint32_t* stamps, const int32_t* stamp_off,
                        uint8_t* out_bgr, void* workspace, size_t workspace_bytes, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(n >= 0 && n <= 65535, "msc_cluster_mosaics: n out of range");
    if (n == 0) return MSC_OK;
    MSC_REQUIRE(views && groups && stamps && stamp_off && out_bgr && workspace, "msc_cluster_mosaics: a pointer argument is NULL");
    MSC_REQUIRE(((uintptr_t)workspace & 255) == 0 && ((uintptr_t)views & 15) == 0 && ((uintptr_t)out_bgr & 15) == 0,
                "msc_cluster_mosaics: workspace must be 256-byte aligned, views and out_bgr 16-byte aligned");
    const size_t need = msc_cluster_mosaics_workspace_bytes(n);
    MSC_REQUIRE(workspace_bytes >= need, "msc_cluster_mosaics: workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
    std::vector<unsigned char> host((size_t)n * sizeof(MosaicRec) + 12 * 4);
    MosaicRec* rec = reinterpret_cast<MosaicRec*>(host.data());
    int64_t off = 0;
    int32_t max_stamp = 0;
    for (int k = 2; k <= 10; ++k) {
        MSC_REQUIRE(stamp_off[k] >= 0 && stamp_off[k + 1] >= stamp_off[k], "msc_cluster_mosaics: stamp_off is not ascending");
        max_stamp = std::max(max_stamp, stamp_off[k + 1] - stamp_off[k]);
    }
    int64_t max_chunks = 0;
    for (int j = 0; j < n; ++j) {
        const int32_t f = groups[2 * j], c = groups[2 * j + 1];
        MSC_REQUIRE(c >= 1 && c <= 10 && f >= 0 && f <= n_views - c, "msc_cluster_mosaics: group %d (%d, %d) outside 1..10 views of %d", j, f, c, n_views);
        rec[j] = MosaicRec{off, f, c, mosaic_cols(c), mosaic_rows(c)};
        const int64_t bytes = (int64_t)rec[j].rows * kView * rec[j].cols * kView * 3;
        max_chunks = std::max(max_chunks, bytes / 16);
        off += bytes;
    }
    memcpy(host.data() + (size_t)n * sizeof(MosaicRec), stamp_off, 12 * 4);
    cudaStream_t st = (cudaStream_t)stream_v;
    // pageable source: staged before the call returns
    MSC_CUDA(cudaMemcpyAsync(workspace, host.data(), host.size(), cudaMemcpyHostToDevice, st));
    const MosaicRec* d_rec = reinterpret_cast<const MosaicRec*>(workspace);
    const int32_t* d_off = reinterpret_cast<const int32_t*>(reinterpret_cast<unsigned char*>(workspace) + (size_t)n * sizeof(MosaicRec));
    mosaic_copy_kernel<<<dim3((unsigned)std::min<int64_t>((max_chunks + 255) / 256, 1024), (unsigned)n), 256, 0, st>>>(
        d_rec, reinterpret_cast<const uint4*>(views), out_bgr);
    if (max_stamp)
        mosaic_stamp_kernel<<<dim3((unsigned)std::min<int32_t>((max_stamp + 255) / 256, 1024), (unsigned)n), 256, 0, st>>>(d_rec, stamps, d_off, out_bgr);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

}  // extern "C"
