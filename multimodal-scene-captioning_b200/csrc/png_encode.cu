// png_encode.cu -- PNG files of 8-bit RGB / grey images on the device, for a batch of images of any shapes in one stream-ordered call.
// What is fixed is the inflated IDAT payload: per row, Pillow's filter choice (ZipEncode.c) and the filtered bytes, so the file decodes
// to the same pixels and inflates to the same bytes as Pillow's.  The deflate stream is this encoder's own: one dynamic-Huffman block
// per image (one table over all the image's tiles), or stored blocks when those are not larger.
//
// Six launches and one descriptor copy, no allocation, no host synchronisation:
//   1. png_filter_kernel   one warp per row: the four candidate costs, Pillow's choice, the filter byte and the filtered row.
//   2. png_lz77_kernel     one CTA per 32 KiB tile of an image's filtered stream.  Per position two match candidates, neither past the
//                          tile's end: the run of bytes equal to their left neighbour (distance 1), and the latest earlier position with
//                          the same 4-byte hash (a shared-memory table seeded with the previous 32 KiB and updated 256 positions at a
//                          time with atomicMax, so the candidate does not depend on scheduling), taken when it is at least 4 bytes and
//                          2 longer than the run (it is not tried inside a run of 64 or more, where it rarely gains and costs compares).  A greedy parse whose per-thread entry points are iterated to a fixed point, the tile's
//                          tokens, its symbol histogram and its Adler-32 partial sums.
//   3. png_huffman_kernel  one CTA per image: histogram, length-limited codes (<= 15 bits; the code-length code <= 7), the block header,
//                          each tile's bit offset, the Adler-32; dynamic or stored, whichever is smaller; the file size.
//   4. png_outoff_kernel   scans the file sizes -> out_off, sets the status word.
//   5. png_pack_kernel     one CTA per tile of a dynamic image: its codes at its bit offset.
//   6. png_place_kernel    one CTA per image: signature, IHDR, IDAT (zlib header, deflate data, Adler-32) with its CRC-32, IEND.
// Every image owns fixed regions of the workspace, so its file never depends on the other images of the call or on the launch shape.
#include <algorithm>
#include <cstdio>
#include <vector>

#include <cub/block/block_scan.cuh>

#include "msc_common.cuh"

namespace msc {

constexpr int kPngTile = 32768;                 // stream bytes per LZ77 tile
constexpr int kLzThreads = 256;
constexpr int kLzSeg = kPngTile / kLzThreads;   // positions whose parse one thread owns
constexpr int kLzWords = kPngTile / 32;
constexpr int kSyms = 286 + 30;                 // literal / length, then distance symbols
constexpr int kMaxMatch = 258;
constexpr int kHashBits = 13;
constexpr int kWindow = 32768;                  // deflate's largest distance
constexpr int kFarRun = 64;                     // no hash candidate is tried inside a distance-1 run this long
constexpr int kStoredMax = 65535;               // bytes per stored block
constexpr int kHdrWords = 160;                  // >= 17 + 19 * 3 + 316 * 14 bits of block header
constexpr int64_t kPngFraming = 57;             // signature, IHDR, IDAT length / type / CRC, IEND

struct PngImg {
    const uint8_t* pixels;
    int64_t pitch;
    int32_t h, w, c, swap;
    int64_t raw;          // h * (1 + w c): the inflated IDAT payload
    int64_t stream_off;   // bytes into the stream area; the token area uses the same index, in u32
    int64_t region_off;   // u32 words into the region area (the deflate data)
    int64_t row_first;    // first row of the image among all rows of the call
    int32_t tile_first, n_tiles;
};

struct PngTile {
    uint32_t hist[kSyms];
    uint32_t ntok, ad_a, ad_b, pad_;
    uint64_t bit_off;     // first bit of the tile in the image's deflate data
};

struct PngRes {
    uint64_t bits;        // dynamic: deflate bits; stored: 0
    int64_t zlen;         // zlib stream bytes
    uint32_t adler;
    int32_t stored;
};

__device__ __forceinline__ int png_image_of(const PngImg* __restrict__ imgs, int n, int64_t key, bool by_row) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((by_row ? imgs[mid].row_first : (int64_t)imgs[mid].tile_first) <= key) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// byte x of a row as the PNG sees it (BGR read as RGB with swap)
__device__ __forceinline__ int png_px(const uint8_t* __restrict__ row, int x, int swap) {
    if (swap) {
        const int k = x % 3;
        x += 2 - 2 * k;
    }
    return row[x];
}

__device__ __forceinline__ uint32_t png_cost(int v) {
    v &= 255;
    return (uint32_t)(v < 128 ? v : 256 - v);
}

__device__ __forceinline__ int png_paeth(int a, int b, int c) {
    const int p = a + b - c, pa = abs(p - a), pb = abs(p - b), pc = abs(p - c);
    return (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
}

// one warp per row; candidates None (0), Up (2), Sub (1), Paeth (4) in that order, replaced only by a strictly smaller cost (so the
// early stop at cost 0 changes nothing), Average never
__global__ void __launch_bounds__(256) png_filter_kernel(const PngImg* __restrict__ imgs, int n, int64_t total_rows, uint8_t* __restrict__ stream) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < total_rows; r += nwarps) {
        const PngImg& I = imgs[png_image_of(imgs, n, r, true)];
        const int y = (int)(r - I.row_first), L = I.w * I.c, bpp = I.c, sw = I.swap;
        const uint8_t* cur = I.pixels + (int64_t)y * I.pitch;
        const uint8_t* prev = y ? cur - I.pitch : nullptr;
        uint32_t cost[4] = {0, 0, 0, 0};
        for (int x = lane; x < L; x += 32) {
            const int v = png_px(cur, x, sw), a = x >= bpp ? png_px(cur, x - bpp, sw) : 0;
            const int b = prev ? png_px(prev, x, sw) : 0, c = prev && x >= bpp ? png_px(prev, x - bpp, sw) : 0;
            cost[0] += png_cost(v);
            cost[1] += png_cost(v - b);
            cost[2] += png_cost(v - a);
            cost[3] += png_cost(v - png_paeth(a, b, c));
        }
        int best = 0;
        uint32_t bc = __reduce_add_sync(0xffffffffu, cost[0]);
        for (int k = 1; k < 4; ++k) {
            const uint32_t s = __reduce_add_sync(0xffffffffu, cost[k]);
            if (s < bc) { bc = s; best = k; }
        }
        uint8_t* out = stream + I.stream_off + (int64_t)y * (1 + L);
        if (lane == 0) out[0] = (uint8_t)(best == 0 ? 0 : best == 1 ? 2 : best == 2 ? 1 : 4);
        for (int x = lane; x < L; x += 32) {
            const int v = png_px(cur, x, sw), a = x >= bpp ? png_px(cur, x - bpp, sw) : 0;
            const int b = prev ? png_px(prev, x, sw) : 0, c = prev && x >= bpp ? png_px(prev, x - bpp, sw) : 0;
            const int f = best == 0 ? v : best == 1 ? v - b : best == 2 ? v - a : v - png_paeth(a, b, c);
            out[1 + x] = (uint8_t)f;
        }
    }
}

// deflate length / distance symbols (RFC 1951 3.2.5)
__device__ __forceinline__ void png_len_sym(int len, int& sym, int& nx, int& xv) {
    const int x = len - 3;
    if (len == kMaxMatch) { sym = 285; nx = 0; xv = 0; }
    else if (x < 8) { sym = 257 + x; nx = 0; xv = 0; }
    else {
        const int nb = 31 - __clz(x);
        sym = 257 + 4 * (nb - 1) + ((x >> (nb - 2)) & 3);
        nx = nb - 2;
        xv = x & ((1 << nx) - 1);
    }
}
__device__ __forceinline__ void png_dist_sym(int d, int& sym, int& nx, int& xv) {
    const int x = d - 1;
    if (x < 4) { sym = x; nx = 0; xv = 0; }
    else {
        const int nb = 31 - __clz(x);
        sym = 2 * nb + ((x >> (nb - 1)) & 1);
        nx = nb - 1;
        xv = x & ((1 << nx) - 1);
    }
}
__host__ __device__ __forceinline__ int png_len_extra(int s) { return s >= 265 && s < 285 ? (s - 261) / 4 : 0; }
__host__ __device__ __forceinline__ int png_dist_extra(int d) { return d < 4 ? 0 : d / 2 - 1; }

// length of the run of set bits from bit p of a tile mask (bits past the tile's end are clear), at most kMaxMatch
__device__ __forceinline__ int png_run(const uint32_t* __restrict__ m, int p) {
    int w = p >> 5;
    const uint32_t x = ~(m[w] >> (p & 31));
    int run = x ? __ffs(x) - 1 : 32;
    if (run < 32 - (p & 31)) return run;
    run = 32 - (p & 31);
    for (++w; w < kLzWords && run < kMaxMatch; ++w) {
        const uint32_t v = m[w];
        if (v != 0xffffffffu) return min(run + __ffs(~v) - 1, kMaxMatch);
        run += 32;
    }
    return min(run, kMaxMatch);
}

__device__ __forceinline__ uint32_t png_hash(const uint8_t* __restrict__ s, int64_t q) {
    const uint32_t key = (uint32_t)s[q] | (uint32_t)s[q + 1] << 8 | (uint32_t)s[q + 2] << 16 | (uint32_t)s[q + 3] << 24;
    return (key * 2654435761u) >> (32 - kHashBits);
}

// the match at tile position p: (length << 16) | distance, 0 for a literal.  s: the image's stream, t0: the tile's first byte, len: its
// length, mask: its distance-1 bits, cand: its hash candidates (distance, 0: none)
__device__ __forceinline__ uint32_t png_match(const uint8_t* __restrict__ s, int64_t t0, int len, const uint32_t* __restrict__ mask,
                                              const uint16_t* __restrict__ cand, int p) {
    const int r = png_run(mask, p);
    uint32_t best = r >= 3 ? (uint32_t)r << 16 | 1u : 0u;
    const int d = cand[p];
    if (d > 1 && r < kFarRun) {
        const int lim = min(kMaxMatch, len - p);
        const uint8_t* a = s + t0 + p;
        const uint8_t* b = a - d;
        int k = 0;
        while (k < lim && a[k] == b[k]) ++k;
        if (k >= 4 && k >= r + 2) best = (uint32_t)k << 16 | (uint32_t)d;
    }
    return best;
}

__global__ void __launch_bounds__(kLzThreads) png_lz77_kernel(const PngImg* __restrict__ imgs, int n, const uint8_t* __restrict__ stream,
                                                                uint32_t* __restrict__ tokens, PngTile* __restrict__ tiles) {
    __shared__ uint32_t mask[kLzWords];  // bit p: byte p equals byte p - 1
    __shared__ int32_t head[1 << kHashBits];
    extern __shared__ uint16_t cand[];   // kPngTile: distance of the hash candidate, 0: none
    __shared__ uint32_t hist[kSyms];
    __shared__ int entry[kLzThreads + 1];
    __shared__ uint64_t red[2][kLzThreads / 32];
    using Scan = cub::BlockScan<uint32_t, kLzThreads>;
    __shared__ typename Scan::TempStorage scan_tmp;

    const int tile = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const PngImg& I = imgs[png_image_of(imgs, n, tile, false)];
    const int64_t t0 = (int64_t)(tile - I.tile_first) * kPngTile;
    const int len = (int)min((int64_t)kPngTile, I.raw - t0);
    const uint8_t* __restrict__ s = stream + I.stream_off;

    // the equality mask, and the Adler-32 partial sums: a = sum b_i, b = sum (len - i) b_i over the tile
    uint32_t sa = 0, sb = 0;
    for (int p0 = 0; p0 < kPngTile; p0 += kLzThreads) {
        const int p = p0 + tid;
        const int64_t q = t0 + p;
        const int v = p < len ? s[q] : -1;
        if (p < len) { sa += (uint32_t)v; sb += (uint32_t)v * (uint32_t)(len - p); }
        const uint32_t b = __ballot_sync(0xffffffffu, p < len && q >= 1 && s[q - 1] == v);
        if (lane == 0) mask[p >> 5] = b;
    }
    for (int k = tid; k < kSyms; k += kLzThreads) hist[k] = 0;
    for (int k = tid; k < (1 << kHashBits); k += kLzThreads) head[k] = -1;
    entry[tid] = tid * kLzSeg;
    {
        // sb: 128 products below 2^23 per thread
        uint64_t a = __reduce_add_sync(0xffffffffu, sa), b = sb;
#pragma unroll
        for (int o = 16; o; o >>= 1) b += __shfl_xor_sync(0xffffffffu, b, o);
        if (lane == 0) { red[0][warp] = a; red[1][warp] = b; }
    }
    __syncthreads();

    // hash candidates: the table holds, per hash, the latest position (image stream index) of the previous 32 KiB and of the earlier
    // chunks of this tile; the positions of a chunk look it up, then enter themselves
    const int64_t hash_end = I.raw - 3;  // positions with 4 bytes to hash
    for (int64_t q = max((int64_t)0, t0 - kWindow) + tid; q < min(t0, hash_end); q += kLzThreads) atomicMax(&head[png_hash(s, q)], (int32_t)q);
    __syncthreads();
    for (int p0 = 0; p0 < len; p0 += kLzThreads) {
        const int p = p0 + tid;
        const int64_t q = t0 + p;
        const bool live = p < len && q < hash_end;
        const uint32_t h = live ? png_hash(s, q) : 0u;
        if (p < len) {
            const int32_t c = live ? head[h] : -1;
            cand[p] = (uint16_t)(c >= 0 && q - c <= kWindow ? q - c : 0);
        }
        __syncthreads();
        if (live) atomicMax(&head[h], (int32_t)q);
        __syncthreads();
    }

    // greedy parse: thread t parses from entry[t] until it passes its segment's end; its exit is thread t + 1's entry.  After round k
    // the entries of threads 0..k are those of the sequential parse, so the fixed point is reached in at most kLzThreads rounds.
    const int a0 = tid * kLzSeg, e0 = min(a0 + kLzSeg, len);
    uint32_t cnt = 0;
    for (;;) {
        int p = entry[tid];
        cnt = 0;
        while (p < e0) {
            const uint32_t m = png_match(s, t0, len, mask, cand, p);
            p += m ? (int)(m >> 16) : 1;
            ++cnt;
        }
        __syncthreads();
        // a thread whose segment starts past the tile's end has no successor that parses
        const bool changed = tid + 1 < kLzThreads && a0 + kLzSeg < len && entry[tid + 1] != p;
        if (changed) entry[tid + 1] = p;
        if (!__syncthreads_or(changed)) break;
    }
    uint32_t off, total;
    Scan(scan_tmp).ExclusiveSum(cnt, off, total);
    uint32_t* __restrict__ tok = tokens + I.stream_off + t0 + off;
    for (int p = entry[tid]; p < e0;) {
        const uint32_t m = png_match(s, t0, len, mask, cand, p);
        if (m) {
            int sym, nx, xv;
            png_len_sym((int)(m >> 16), sym, nx, xv);
            atomicAdd(&hist[sym], 1u);
            png_dist_sym((int)(m & 0xffffu), sym, nx, xv);
            atomicAdd(&hist[286 + sym], 1u);
            *tok++ = m;
            p += (int)(m >> 16);
        } else {
            const uint32_t v = s[t0 + p];
            atomicAdd(&hist[v], 1u);
            *tok++ = v;
            ++p;
        }
    }
    __syncthreads();
    PngTile& T = tiles[tile];
    for (int k = tid; k < kSyms; k += kLzThreads) T.hist[k] = hist[k];
    if (tid == 0) {
        uint64_t a = 0, b = 0;
        for (int w = 0; w < kLzThreads / 32; ++w) { a += red[0][w]; b += red[1][w]; }
        T.ntok = total;
        T.ad_a = (uint32_t)(a % 65521u);
        T.ad_b = (uint32_t)(b % 65521u);
    }
}

// ---------------------------------------------------------------- Huffman codes (one thread)
// Code lengths of the used symbols of freq[0 .. n): Huffman's construction on the symbols sorted by (frequency, symbol) with two
// queues (leaves first on ties), then lengths above `limit` folded back as in JPEG Annex K.3 (Kraft sum kept at 1), and the lengths
// handed out again from the most frequent symbol down.  Fewer than two used symbols get two codes of one bit, as zlib does.
__device__ void png_code_lengths(const uint32_t* freq, int n, int limit, uint8_t* len, uint16_t* order, uint32_t* wt, uint16_t* parent,
                                 int* bits) {
    int m = 0;
    for (int s = 0; s < n; ++s) {
        len[s] = 0;
        if (freq[s]) order[m++] = (uint16_t)s;
    }
    if (m < 2) {
        const int a = m ? order[0] : 0;
        len[a] = 1;
        len[a == 0 ? 1 : 0] = 1;
        return;
    }
    for (int i = 1; i < m; ++i) {  // insertion sort by (freq, symbol)
        const uint16_t v = order[i];
        int j = i - 1;
        while (j >= 0 && (freq[order[j]] > freq[v] || (freq[order[j]] == freq[v] && order[j] > v))) { order[j + 1] = order[j]; --j; }
        order[j + 1] = v;
    }
    for (int i = 0; i < m; ++i) wt[i] = freq[order[i]];
    int leaf = 0, node = m;
    for (int k = m; k < 2 * m - 1; ++k) {
        uint32_t w = 0;
        for (int t = 0; t < 2; ++t) {
            const bool take_leaf = leaf < m && (node >= k || wt[leaf] <= wt[node]);
            const int pick = take_leaf ? leaf++ : node++;
            parent[pick] = (uint16_t)k;
            w += wt[pick];
        }
        wt[k] = w;
    }
    for (int l = 0; l < max(m, limit + 1); ++l) bits[l] = 0;  // depths reach m - 1; lengths are read up to limit
    wt[2 * m - 2] = 0;  // depths, reusing wt: parents come after their children
    int maxd = 0;
    for (int k = 2 * m - 3; k >= 0; --k) {
        wt[k] = wt[parent[k]] + 1;
        if (k < m) { ++bits[wt[k]]; maxd = max(maxd, (int)wt[k]); }
    }
    for (int i = maxd; i > limit; --i) {
        while (bits[i] > 0) {
            int j = i - 2;
            while (bits[j] == 0) --j;
            bits[i] -= 2;
            bits[i - 1] += 1;
            bits[j + 1] += 2;
            bits[j] -= 1;
        }
    }
    int k = m - 1;
    for (int l = 1; l <= limit; ++l)
        for (int c = 0; c < bits[l]; ++c) len[order[k--]] = (uint8_t)l;
}

// canonical codes (RFC 1951 3.2.2), bit-reversed for LSB-first packing: (length << 16) | code
__device__ void png_canonical(const uint8_t* len, int n, uint32_t* code, int* count /* 32 */) {
    int* next = count + 16;
    for (int l = 0; l < 16; ++l) count[l] = 0;
    for (int s = 0; s < n; ++s) ++count[len[s]];
    count[0] = 0;
    int c = 0;
    for (int l = 1; l < 16; ++l) { c = (c + count[l - 1]) << 1; next[l] = c; }
    for (int s = 0; s < n; ++s) {
        const int l = len[s];
        code[s] = l ? (uint32_t)l << 16 | (__brev((uint32_t)next[l]++) >> (32 - l)) : 0u;
    }
}

struct PngBits {
    uint32_t* w;
    uint32_t pos;
    __device__ __forceinline__ void put(uint32_t v, int nb) {
        if (!nb) return;
        const uint32_t k = pos >> 5, o = pos & 31;
        w[k] |= v << o;
        if (o + nb > 32) w[k + 1] |= v >> (32 - o);
        pos += nb;
    }
};

__global__ void __launch_bounds__(256) png_huffman_kernel(const PngImg* __restrict__ imgs, PngTile* __restrict__ tiles, uint32_t* __restrict__ codes,
                                                          PngRes* __restrict__ res, uint64_t* __restrict__ size, uint32_t* __restrict__ region) {
    __shared__ uint32_t freq[kSyms], code[kSyms], wt[2 * 286], hdr[kHdrWords];
    __shared__ uint8_t len[kSyms + 2], cl_len[19];
    __shared__ uint16_t order[286], parent[2 * 286];
    __shared__ uint16_t rle[kSyms];
    __shared__ uint8_t seq[kSyms];
    __shared__ int bits[286];
    __shared__ uint32_t cl_freq[19], cl_code[19];
    __shared__ uint64_t s_bits;
    __shared__ uint32_t s_hbits;
    __shared__ int s_stored;
    const int i = blockIdx.x, tid = threadIdx.x;
    const PngImg& I = imgs[i];
    PngTile* __restrict__ T = tiles + I.tile_first;
    for (int k = tid; k < kSyms; k += blockDim.x) {
        uint32_t f = k == 256;
        for (int t = 0; t < I.n_tiles; ++t) f += T[t].hist[k];
        freq[k] = f;
    }
    for (int k = tid; k < kHdrWords; k += blockDim.x) hdr[k] = 0;
    __syncthreads();
    if (tid == 0) {
        png_code_lengths(freq, 286, 15, len, order, wt, parent, bits);
        png_code_lengths(freq + 286, 30, 15, len + 286, order, wt, parent, bits);
        int hlit = 286, hdist = 30;
        while (hlit > 257 && !len[hlit - 1]) --hlit;
        while (hdist > 1 && !len[286 + hdist - 1]) --hdist;
        // run-length code of the hlit + hdist lengths (one sequence): 16 repeats the previous length 3-6 times, 17 / 18 code 3-10 /
        // 11-138 zeros; rle entries are symbol | extra << 5
        const int N = hlit + hdist;
        for (int k = 0; k < N; ++k) seq[k] = k < hlit ? len[k] : len[286 + k - hlit];
        int nr = 0;
        for (int k = 0; k < 19; ++k) cl_freq[k] = 0;
        for (int k = 0; k < N;) {
            const int cur = seq[k];
            int run = 1;
            while (k + run < N && seq[k + run] == cur) ++run;
            int r = run;
            if (cur == 0) {
                while (r >= 11) { const int q = min(r, 138); rle[nr++] = (uint16_t)(18 | (q - 11) << 5); r -= q; }
                if (r >= 3) { rle[nr++] = (uint16_t)(17 | (r - 3) << 5); r = 0; }
            } else {
                rle[nr++] = (uint16_t)cur;
                --r;
                while (r >= 3) { const int q = min(r, 6); rle[nr++] = (uint16_t)(16 | (q - 3) << 5); r -= q; }
            }
            for (; r > 0; --r) rle[nr++] = (uint16_t)cur;
            k += run;
        }
        for (int k = 0; k < nr; ++k) ++cl_freq[rle[k] & 31];
        png_code_lengths(cl_freq, 19, 7, cl_len, order, wt, parent, bits);
        png_canonical(cl_len, 19, cl_code, bits);
        static const uint8_t perm[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        int hclen = 19;
        while (hclen > 4 && !cl_len[perm[hclen - 1]]) --hclen;
        PngBits hb{hdr, 0};
        hb.put(5, 3);  // BFINAL = 1, BTYPE = 2 (dynamic)
        hb.put((uint32_t)(hlit - 257), 5);
        hb.put((uint32_t)(hdist - 1), 5);
        hb.put((uint32_t)(hclen - 4), 4);
        for (int k = 0; k < hclen; ++k) hb.put(cl_len[perm[k]], 3);
        for (int k = 0; k < nr; ++k) {
            const int sym = rle[k] & 31, x = rle[k] >> 5;
            hb.put(cl_code[sym] & 0xffffu, (int)(cl_code[sym] >> 16));
            hb.put((uint32_t)x, sym == 16 ? 2 : sym == 17 ? 3 : sym == 18 ? 7 : 0);
        }
        s_hbits = hb.pos;
        png_canonical(len, 286, code, bits);
        png_canonical(len + 286, 30, code + 286, bits);
    }
    __syncthreads();
    for (int k = tid; k < kSyms; k += blockDim.x) codes[(int64_t)i * kSyms + k] = code[k];
    // bits of every tile, then their offsets
    for (int t = tid; t < I.n_tiles; t += blockDim.x) {
        uint64_t b = 0;
        for (int k = 0; k < kSyms; ++k) {
            const uint32_t h = T[t].hist[k];
            if (h) b += (uint64_t)h * ((code[k] >> 16) + (k < 286 ? png_len_extra(k) : png_dist_extra(k - 286)));
        }
        T[t].bit_off = b;
    }
    __syncthreads();
    if (tid == 0) {
        uint64_t pos = s_hbits, a = 0, b = 0;
        for (int t = 0; t < I.n_tiles; ++t) {
            const uint64_t tb = T[t].bit_off;
            T[t].bit_off = pos;
            pos += tb;
            const int64_t end = min((int64_t)(t + 1) * kPngTile, I.raw);
            a += T[t].ad_a;
            b += T[t].ad_b + (uint64_t)T[t].ad_a * (uint64_t)((I.raw - end) % 65521);
            b %= 65521u;
        }
        const uint64_t bits = pos + (code[256] >> 16);
        const int64_t nblk = (I.raw + kStoredMax - 1) / kStoredMax;
        const int64_t stored_bytes = I.raw + 5 * nblk;
        const int stored = (int64_t)((bits + 7) >> 3) >= stored_bytes;
        PngRes r;
        r.bits = stored ? 0 : bits;
        r.zlen = 2 + (stored ? stored_bytes : (int64_t)((bits + 7) >> 3)) + 4;
        r.adler = (uint32_t)(((b + (uint64_t)(I.raw % 65521)) % 65521u) << 16 | ((1 + a) % 65521u));
        r.stored = stored;
        res[i] = r;
        size[i] = (uint64_t)(kPngFraming + r.zlen);
        s_bits = bits;
        s_stored = stored;
    }
    __syncthreads();
    if (s_stored) return;
    uint32_t* __restrict__ reg = region + I.region_off;
    const uint64_t nw = (s_bits + 31) >> 5;
    for (uint64_t k = tid; k < nw; k += blockDim.x) reg[k] = k < kHdrWords ? hdr[k] : 0u;
    __syncthreads();
    if (tid == 0) {  // end of block
        const uint64_t p = s_bits - (code[256] >> 16);
        PngBits eb{reg + (p >> 5), (uint32_t)(p & 31)};
        eb.put(code[256] & 0xffffu, (int)(code[256] >> 16));
    }
}

// out_off = exclusive scan of the file sizes (n + 1 entries); status = 1 when they exceed the arena
__global__ void __launch_bounds__(256) png_outoff_kernel(int32_t n, const uint64_t* __restrict__ size, uint64_t out_bytes, int64_t* __restrict__ out_off,
                                                         int32_t* __restrict__ status) {
    using Scan = cub::BlockScan<uint64_t, 256>;
    __shared__ typename Scan::TempStorage tmp;
    uint64_t running = 0;
    for (int i0 = 0; i0 < n; i0 += 256) {
        const int i = i0 + threadIdx.x;
        uint64_t excl, agg;
        Scan(tmp).ExclusiveSum(i < n ? size[i] : 0ull, excl, agg);
        if (i < n) out_off[i] = (int64_t)(running + excl);
        running += agg;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out_off[n] = (int64_t)running;
        *status = running > out_bytes ? 1 : 0;
    }
}

// one CTA per tile of a dynamic image: each thread packs a contiguous run of the tile's tokens LSB-first at its bit offset; words it
// covers whole are stored, words shared with a neighbour are OR-ed into the region (zeroed by png_huffman_kernel)
__global__ void __launch_bounds__(kLzThreads) png_pack_kernel(const PngImg* __restrict__ imgs, int n, const uint32_t* __restrict__ tokens,
                                                              const PngTile* __restrict__ tiles, const uint32_t* __restrict__ codes,
                                                              const PngRes* __restrict__ res, uint32_t* __restrict__ region) {
    __shared__ uint32_t code[kSyms];
    using Scan = cub::BlockScan<uint32_t, kLzThreads>;
    __shared__ typename Scan::TempStorage scan_tmp;
    const int tile = blockIdx.x, tid = threadIdx.x;
    const int i = png_image_of(imgs, n, tile, false);
    if (res[i].stored) return;
    const PngImg& I = imgs[i];
    for (int k = tid; k < kSyms; k += kLzThreads) code[k] = codes[(int64_t)i * kSyms + k];
    __syncthreads();
    const PngTile& T = tiles[tile];
    const uint32_t* __restrict__ tok = tokens + I.stream_off + (int64_t)(tile - I.tile_first) * kPngTile;
    const uint32_t per = (T.ntok + kLzThreads - 1) / kLzThreads;
    const uint32_t k0 = min(T.ntok, per * tid), k1 = min(T.ntok, k0 + per);
    uint32_t nb = 0;
    for (uint32_t k = k0; k < k1; ++k) {
        const uint32_t t = tok[k];
        if (t < 256) nb += code[t] >> 16;
        else {
            int sym, nx, xv;
            png_len_sym((int)(t >> 16), sym, nx, xv);
            nb += (code[sym] >> 16) + nx;
            png_dist_sym((int)(t & 0xffffu), sym, nx, xv);
            nb += (code[286 + sym] >> 16) + nx;
        }
    }
    uint32_t off, total;
    Scan(scan_tmp).ExclusiveSum(nb, off, total);
    if (!nb) return;
    const uint64_t start = T.bit_off + off;
    uint32_t* __restrict__ reg = region + I.region_off;
    uint64_t w = start >> 5, acc = 0;
    int nbit = (int)(start & 31);
    const uint64_t first = w;
    auto put = [&](uint32_t v, int l) {
        acc |= (uint64_t)v << nbit;
        nbit += l;
        if (nbit >= 32) {
            if (w == first && (start & 31)) atomicOr(&reg[w], (uint32_t)acc);
            else reg[w] = (uint32_t)acc;
            ++w;
            acc >>= 32;
            nbit -= 32;
        }
    };
    for (uint32_t k = k0; k < k1; ++k) {
        const uint32_t t = tok[k];
        if (t < 256) put(code[t] & 0xffffu, (int)(code[t] >> 16));
        else {
            int sym, nx, xv;
            png_len_sym((int)(t >> 16), sym, nx, xv);
            put((code[sym] & 0xffffu) | (uint32_t)xv << (code[sym] >> 16), (int)(code[sym] >> 16) + nx);
            png_dist_sym((int)(t & 0xffffu), sym, nx, xv);
            put((code[286 + sym] & 0xffffu) | (uint32_t)xv << (code[286 + sym] >> 16), (int)(code[286 + sym] >> 16) + nx);
        }
    }
    if (nbit) atomicOr(&reg[w], (uint32_t)acc);
}

// ---------------------------------------------------------------- framing and CRC-32
__device__ __forceinline__ uint32_t png_multmodp(uint32_t a, uint32_t b) {  // a * b mod P, reflected (zlib crc32.c)
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}
__device__ __forceinline__ uint32_t png_x8n(uint64_t n) {  // x^(8 n) mod P
    uint32_t p = 1u << 31, sq = 1u << 23;
    for (; n; n >>= 1) {
        if (n & 1) p = png_multmodp(sq, p);
        sq = png_multmodp(sq, sq);
    }
    return p;
}

constexpr int kPlaceThreads = 512;
__constant__ uint8_t kPngSig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
__constant__ uint8_t kPngIend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xae, 0x42, 0x60, 0x82};

// byte k of image I's zlib stream
__device__ __forceinline__ uint8_t png_zbyte(const PngImg& I, const PngRes& R, const uint8_t* __restrict__ s, const uint8_t* __restrict__ reg, int64_t k) {
    if (k < 2) return k ? 0x9c : 0x78;
    if (k >= R.zlen - 4) return (uint8_t)(R.adler >> (8 * (R.zlen - 1 - k)));
    const int64_t j = k - 2;
    if (!R.stored) return reg[j];
    const int64_t blk = j / (kStoredMax + 5), o = j - blk * (kStoredMax + 5);
    const int64_t nblk = (I.raw + kStoredMax - 1) / kStoredMax;
    const uint32_t blen = (uint32_t)min((int64_t)kStoredMax, I.raw - blk * kStoredMax);
    switch (o) {
        case 0: return blk == nblk - 1;
        case 1: return (uint8_t)blen;
        case 2: return (uint8_t)(blen >> 8);
        case 3: return (uint8_t)~blen;
        case 4: return (uint8_t)(~blen >> 8);
        default: return s[blk * kStoredMax + o - 5];
    }
}

__global__ void __launch_bounds__(kPlaceThreads) png_place_kernel(const PngImg* __restrict__ imgs, int32_t n, const PngRes* __restrict__ res,
                                                                  const uint8_t* __restrict__ stream, const uint32_t* __restrict__ region,
                                                                  uint64_t out_bytes, const int64_t* __restrict__ out_off, uint8_t* __restrict__ out) {
    __shared__ uint32_t tab[256], crc_t[kPlaceThreads], xp_t[kPlaceThreads];
    if ((uint64_t)out_off[n] > out_bytes) return;
    const int i = blockIdx.x, tid = threadIdx.x;
    const PngImg& I = imgs[i];
    const PngRes R = res[i];
    {
        uint32_t c = tid;
        for (int k = 0; k < 8; ++k) c = c & 1 ? 0xedb88320u ^ (c >> 1) : c >> 1;
        if (tid < 256) tab[tid] = c;
    }
    __syncthreads();
    uint8_t* __restrict__ dst = out + out_off[i];
    const uint8_t* __restrict__ s = stream + I.stream_off;
    const uint8_t* __restrict__ reg = reinterpret_cast<const uint8_t*>(region + I.region_off);
    if (tid < 8) dst[tid] = kPngSig[tid];
    if (tid < 12) dst[45 + R.zlen + tid] = kPngIend[tid];
    if (tid == 0) {  // IHDR: length 13, type, width, height, depth 8, colour type, compression, filter, interlace 0; CRC
        uint8_t* h = dst + 8;
        for (int k = 0; k < 21; ++k) h[k] = 0;
        h[3] = 13; h[4] = 'I'; h[5] = 'H'; h[6] = 'D'; h[7] = 'R';
        h[10] = (uint8_t)(I.w >> 8); h[11] = (uint8_t)I.w; h[14] = (uint8_t)(I.h >> 8); h[15] = (uint8_t)I.h;
        h[16] = 8; h[17] = (uint8_t)(I.c == 3 ? 2 : 0);
        uint32_t c = 0xffffffffu;
        for (int k = 4; k < 21; ++k) c = tab[(c ^ h[k]) & 255] ^ (c >> 8);
        for (int k = 0; k < 4; ++k) h[21 + k] = (uint8_t)(~c >> (24 - 8 * k));
        for (int k = 0; k < 4; ++k) dst[33 + k] = (uint8_t)(R.zlen >> (24 - 8 * k));
    }
    // "IDAT" and the zlib stream: thread t writes and checksums bytes [t L, (t + 1) L), the partial CRCs are combined in order
    const int64_t total = 4 + R.zlen, per = (total + kPlaceThreads - 1) / kPlaceThreads;
    const int64_t b0 = min(total, per * tid), b1 = min(total, b0 + per);
    uint8_t* d = dst + 37;
    uint32_t c = 0xffffffffu;
    for (int64_t k = b0; k < b1; ++k) {
        const uint8_t v = k < 4 ? (uint8_t)(0x49444154u >> (24 - 8 * k)) : png_zbyte(I, R, s, reg, k - 4);
        d[k] = v;
        c = tab[(c ^ v) & 255] ^ (c >> 8);
    }
    crc_t[tid] = b1 > b0 ? ~c : 0u;
    xp_t[tid] = png_x8n((uint64_t)(b1 - b0));
    __syncthreads();
    if (tid == 0) {
        uint32_t crc = crc_t[0];
        for (int t = 1; t < kPlaceThreads; ++t) crc = png_multmodp(xp_t[t], crc) ^ crc_t[t];
        uint8_t* e = d + total;
        for (int k = 0; k < 4; ++k) e[k] = (uint8_t)(crc >> (24 - 8 * k));
    }
}

// ---------------------------------------------------------------- host
struct PngLayout {
    std::vector<PngImg> imgs;
    int64_t rows, tiles;
    size_t desc, tile, codes, res, size, stream, tokens, region, total;
};

static size_t png_al(size_t v) { return (v + 255) & ~(size_t)255; }

// false when an image is refused or the call does not fit the grid / size_t
static bool png_layout(int32_t n, const msc_png_image* im, PngLayout* L, char* why, size_t why_len) {
    L->imgs.resize((size_t)n);
    int64_t rows = 0, tiles = 0, sbytes = 0, rwords = 0;
    for (int32_t i = 0; i < n; ++i) {
        const msc_png_image& a = im[i];
        auto bad = [&](const char* what) { snprintf(why, why_len, "image %d: %s", (int)i, what); return false; };
        if (a.channels != 1 && a.channels != 3) return bad("channels must be 1 or 3");
        if (a.swap_rb && a.channels != 3) return bad("swap_rb needs 3 channels");
        if (a.height < 1 || a.height > 65535 || a.width < 1 || a.width > 65535) return bad("height and width must be in 1..65535");
        const int64_t raw = (int64_t)a.height * (1 + (int64_t)a.width * a.channels);
        const int64_t nblk = (raw + kStoredMax - 1) / kStoredMax;
        if (raw >= (int64_t)1 << 31 || 6 + raw + 5 * nblk > 0x7fffffff) return bad("the image is too large for one IDAT chunk");
        if (a.row_pitch < (int64_t)a.width * a.channels) return bad("row pitch below width * channels");
        if (!a.pixels) return bad("NULL pixels");
        PngImg& g = L->imgs[(size_t)i];
        g.pixels = a.pixels; g.pitch = a.row_pitch;
        g.h = a.height; g.w = a.width; g.c = a.channels; g.swap = a.swap_rb ? 1 : 0;
        g.raw = raw;
        g.stream_off = sbytes;
        g.region_off = rwords;
        g.row_first = rows;
        g.tile_first = (int32_t)tiles;
        g.n_tiles = (int32_t)((raw + kPngTile - 1) / kPngTile);
        rows += a.height;
        tiles += g.n_tiles;
        sbytes += (raw + 15) & ~(int64_t)15;
        rwords += ((raw + 5 * nblk + 3) / 4 + 2 + 3) & ~(int64_t)3;
        if (tiles > 0x7fffffff) return bad("too many tiles for one call");
    }
    L->rows = rows;
    L->tiles = tiles;
    size_t o = 0;
    L->desc = o; o = png_al(o + (size_t)n * sizeof(PngImg));
    L->tile = o; o = png_al(o + (size_t)tiles * sizeof(PngTile));
    L->codes = o; o = png_al(o + (size_t)n * kSyms * 4);
    L->res = o; o = png_al(o + (size_t)n * sizeof(PngRes));
    L->size = o; o = png_al(o + (size_t)n * 8);
    L->stream = o; o = png_al(o + (size_t)sbytes);
    L->tokens = o; o = png_al(o + (size_t)sbytes * 4);
    L->region = o; o = png_al(o + (size_t)rwords * 4);
    L->total = o > 256 ? o : 256;
    return true;
}

}  // namespace msc

extern "C" {

size_t msc_png_encode_workspace_bytes(int32_t n, const msc_png_image* images_host) {
    using namespace msc;
    if (n < 0 || (n > 0 && !images_host)) return 0;
    PngLayout L;
    char why[160];
    if (!png_layout(n, images_host, &L, why, sizeof(why))) return 0;
    return L.total;
}

int msc_png_encode_batch(int32_t n, const msc_png_image* images_host, uint8_t* out, size_t out_bytes, int64_t* out_off, int32_t* status,
                         void* workspace, size_t workspace_bytes, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(n >= 0, "msc_png_encode_batch: negative n");
    if (n == 0) return MSC_OK;
    MSC_REQUIRE(images_host && out && out_off && status && workspace, "msc_png_encode_batch: a pointer argument is NULL");
    MSC_REQUIRE(((uintptr_t)workspace & 255) == 0, "msc_png_encode_batch: workspace must be 256-byte aligned");
    PngLayout L;
    char why[160];
    MSC_REQUIRE(png_layout(n, images_host, &L, why, sizeof(why)), "msc_png_encode_batch: %s", why);
    MSC_REQUIRE(workspace_bytes >= L.total, "msc_png_encode_batch: workspace too small: need %zu bytes, got %zu", L.total, workspace_bytes);

    unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
    const PngImg* d_imgs = reinterpret_cast<const PngImg*>(ws + L.desc);
    PngTile* tiles = reinterpret_cast<PngTile*>(ws + L.tile);
    uint32_t* codes = reinterpret_cast<uint32_t*>(ws + L.codes);
    PngRes* res = reinterpret_cast<PngRes*>(ws + L.res);
    uint64_t* size = reinterpret_cast<uint64_t*>(ws + L.size);
    uint8_t* stream = ws + L.stream;
    uint32_t* tokens = reinterpret_cast<uint32_t*>(ws + L.tokens);
    uint32_t* region = reinterpret_cast<uint32_t*>(ws + L.region);
    cudaStream_t st = (cudaStream_t)stream_v;
    constexpr int kLzSmem = kPngTile * 2;
    MSC_CUDA(cudaFuncSetAttribute(png_lz77_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLzSmem));
    // pageable source: staged before the call returns
    MSC_CUDA(cudaMemcpyAsync(ws + L.desc, L.imgs.data(), (size_t)n * sizeof(PngImg), cudaMemcpyHostToDevice, st));
    const unsigned fgrid = (unsigned)std::min<int64_t>((L.rows + 7) / 8, 148 * 64);
    png_filter_kernel<<<fgrid, 256, 0, st>>>(d_imgs, n, L.rows, stream);
    png_lz77_kernel<<<(unsigned)L.tiles, kLzThreads, kLzSmem, st>>>(d_imgs, n, stream, tokens, tiles);
    png_huffman_kernel<<<(unsigned)n, 256, 0, st>>>(d_imgs, tiles, codes, res, size, region);
    png_outoff_kernel<<<1, 256, 0, st>>>(n, size, (uint64_t)out_bytes, out_off, status);
    png_pack_kernel<<<(unsigned)L.tiles, kLzThreads, 0, st>>>(d_imgs, n, tokens, tiles, codes, res, region);
    png_place_kernel<<<(unsigned)n, kPlaceThreads, 0, st>>>(d_imgs, n, res, stream, region, (uint64_t)out_bytes, out_off, out);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

}  // extern "C"
