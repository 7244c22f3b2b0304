// jpeg_decode.cu -- batched camera-frame decode with every stage on the device (DESIGN.md section 4.9): byte unstuffing and restart
// segmentation, a self-synchronising Huffman decode (Weissenberger & Schmidt, "Massively Parallel Huffman Decoding on GPUs", ICPP 2018),
// DC prediction, the integer IDCT, chroma upsampling and colour conversion -- for a whole batch of files in four launches.  The results
// equal msc_jpeg_entropy_decode_host (coefficients) and msc_jpeg_reconstruct (frames) of jpeg.cu bit for bit: the bit-level rules below
// restate jpeg.cu's BitReader / entropy_decode, and the IDCT / upsampling / colour arithmetic is jpeg_common.cuh's, shared with jpeg.cu.
//
//   jd_unstuff_kernel   one CTA per image: the scan's bytes -> a packed stream without stuffed zeros, cut at markers into restart
//                       segments; per segment its byte range and its first subsequence.
//   jd_huffman_kernel   one CTA per image: zero-fills the image's coefficients, then decodes its subsequences (kSubBits bits each) a
//                       window of kJdThreads at a time -- speculative decodes iterated to a fixed point, a scan of completed blocks, a
//                       final decode that writes -- and last the DC prediction per component.
//   jd_idct_kernel      one launch for every block of every component of every image (jpeg.cu's jpeg_idct_kernel, per-CTA descriptors).
//   jd_color_kernel     one launch for every row of every image (jpeg.cu's jpeg_color_kernel, per-CTA descriptors).
#include <cub/block/block_scan.cuh>
#include <vector>

#include "jpeg_common.cuh"
#include "msc_common.cuh"

namespace msc {

constexpr int kJdThreads = 256;         // threads of the unstuff, Huffman and reconstruction CTAs
constexpr int kJdBytes = 8;             // scan bytes per thread and tile of the unstuff pass
constexpr uint32_t kSubBits = 1024;     // bits per subsequence of the Huffman decode
constexpr uint32_t kNone = 0xffffffffu;
constexpr uint64_t kPoison = ~0ull;     // the state after an invalid code: never equal to a real state
constexpr int64_t kMaxScanBytes = 1 << 28;  // bit positions stay below 2^31

// per-image record in the workspace, written by the host from the plan
struct JdImage {
    msc_jpeg_desc d;
    int64_t scan;        // first scan byte in `files`
    int64_t coef;        // first coefficient in `coef` (a multiple of 8)
    int64_t out;         // first byte in `out`
    int64_t packed;      // workspace offsets: the unstuffed stream (scan_bytes + 16 bytes) ...
    int64_t seg;         // ... u32 seg_begin[n_seg], seg_end[n_seg] (bytes of the packed stream), sub_base[n_seg + 1] ...
    int64_t planes;      // ... and the component planes (d.plane_bytes)
    int32_t scan_bytes, n_seg, ri, bpm, total_mcus;
    int32_t huff[3][2];  // index of the DC / AC table of each component in the workspace table array
    int32_t idct_cta[4]; // first IDCT CTA of each component, relative to the image's first; [n_comp] = the image's count
    int32_t color_chunks;  // colour CTAs per row
    uint8_t slot_comp[8], slot_by[8], slot_bx[8];  // component and block position of each block slot of an MCU
};

// ------------------------------------------------------------------------------------------------ unstuff + segment
struct JdEvents {
    int s, m, n;  // last segment start, last marker, number of segment starts
};
struct JdEventsOp {
    __device__ __forceinline__ JdEvents operator()(const JdEvents& a, const JdEvents& b) const { return {max(a.s, b.s), max(a.m, b.m), a.n + b.n}; }
};

// A byte j of the scan (0 <= j < L; j = L is a virtual byte past the end) is
//   a marker      if it is FF and not followed by 00 (an FF in the last byte is a marker: jpeg.cu's BitReader reads zeros from there);
//   a segment start if bytes j-2, j-1 are FF D0..D7 (segment 0 starts at 0): segment k starts after the k-th restart marker;
//   data          if no marker lies between the last segment start and j (inclusive);
//   kept          if it is data of one of the first n_seg segments and not the 00 of a stuffed FF 00.
// Kept bytes go to the packed stream in order; segment k is packed bytes [seg_begin[k], seg_end[k]).
__global__ void __launch_bounds__(kJdThreads) jd_unstuff_kernel(const JdImage* __restrict__ imgs, const uint8_t* __restrict__ files, uint8_t* ws,
                                                                int32_t* status) {
    using Scan = cub::BlockScan<JdEvents, kJdThreads>;
    using Count = cub::BlockScan<uint32_t, kJdThreads>;
    __shared__ union {
        typename Scan::TempStorage scan;
        typename Count::TempStorage count;
    } tmp;
    const JdImage& I = imgs[blockIdx.x];
    const uint8_t* __restrict__ b = files + I.scan;
    const int L = I.scan_bytes, n_seg = I.n_seg;
    uint8_t* packed = ws + I.packed;
    uint32_t* seg_begin = reinterpret_cast<uint32_t*>(ws + I.seg);
    uint32_t* seg_end = seg_begin + n_seg;
    uint32_t* sub_base = seg_end + n_seg;
    for (int k = threadIdx.x; k < n_seg; k += kJdThreads) { seg_begin[k] = k ? kNone : 0u; seg_end[k] = kNone; }
    if (threadIdx.x == 0) status[blockIdx.x] = 0;
    __syncthreads();
    JdEvents carry = {0, -1, 0};
    uint32_t kept_total = 0;
    for (int t0 = 0; t0 <= L; t0 += kJdThreads * kJdBytes) {
        const int j0 = t0 + (int)threadIdx.x * kJdBytes;
        int w[kJdBytes + 3];  // bytes j0-2 .. j0+kJdBytes, -1 outside the scan
#pragma unroll
        for (int q = 0; q < kJdBytes + 3; ++q) {
            const int j = j0 - 2 + q;
            w[q] = (j >= 0 && j < L) ? (int)b[j] : -1;
        }
        auto is_start = [&](int q) { return w[q] == 0xFF && w[q + 1] >= 0xD0 && w[q + 1] <= 0xD7; };  // byte j0+q is a segment start
        auto is_marker = [&](int q) { return w[q + 2] == 0xFF && w[q + 3] != 0; };                      // byte j0+q is a marker
        JdEvents loc = {-1, -1, 0};
#pragma unroll
        for (int q = 0; q < kJdBytes; ++q) {
            if (j0 + q > L) break;
            if (is_start(q)) { loc.s = j0 + q; ++loc.n; }
            if (is_marker(q)) loc.m = j0 + q;
        }
        JdEvents pre, agg;
        Scan(tmp.scan).ExclusiveScan(loc, pre, JdEvents{-1, -1, 0}, JdEventsOp(), agg);
        __syncthreads();
        const JdEvents at = JdEventsOp()(carry, pre);  // events before byte j0
        // walk the thread's bytes; pass 0 counts kept bytes, pass 1 writes them and the segment bounds
        uint32_t pos = 0;
        for (int pass = 0; pass < 2; ++pass) {
            int s = at.s, m = at.m, ns = at.n;
            bool prev_ff = w[1] == 0xFF && m < s;  // byte j0-1 is a data FF: byte j0 is its stuffed 00
            uint32_t nk = 0;
#pragma unroll
            for (int q = 0; q < kJdBytes; ++q) {
                const int j = j0 + q;
                if (j > L) break;
                if (is_start(q)) {
                    s = j; ++ns;
                    if (pass && ns < n_seg) seg_begin[ns] = pos + nk;
                }
                if (is_marker(q)) {
                    if (pass && m < s && ns < n_seg) seg_end[ns] = pos + nk;  // the first marker of the segment ends its data
                    m = j;
                }
                const bool data = j < L && m < s;
                const bool kept = data && !prev_ff && ns < n_seg;
                prev_ff = data && w[q + 2] == 0xFF;
                if (kept) {
                    if (pass) packed[pos + nk] = (uint8_t)w[q + 2];
                    ++nk;
                }
            }
            if (pass == 0) {
                uint32_t tile_kept;
                Count(tmp.count).ExclusiveSum(nk, pos, tile_kept);
                __syncthreads();
                pos += kept_total;
                kept_total += tile_kept;
            }
        }
        carry = JdEventsOp()(carry, agg);
    }
    __syncthreads();
    // segment bounds, missing restart markers, and the first subsequence of every segment
    uint32_t run = 0;
    for (int k0 = 0; k0 < n_seg; k0 += kJdThreads) {
        const int k = k0 + (int)threadIdx.x;
        uint32_t nsub = 0;
        if (k < n_seg) {
            uint32_t a = seg_begin[k], e = seg_end[k];
            if (a == kNone) {  // jpeg.cu: "restart marker missing"
                status[blockIdx.x] = MSC_ERR_BAD_ARGUMENT;
                a = e = kept_total;
                seg_begin[k] = a;
            }
            if (e == kNone) e = kept_total;
            seg_end[k] = e;
            nsub = max(1u, ((e - a) * 8u + kSubBits - 1) / kSubBits);
        }
        uint32_t base, total;
        Count(tmp.count).ExclusiveSum(nsub, base, total);
        __syncthreads();
        if (k < n_seg) sub_base[k] = run + base;
        run += total;
    }
    if (threadIdx.x == 0) sub_base[n_seg] = run;
}

// ------------------------------------------------------------------------------------------------ Huffman decode
// Bits [pos, pos + 32) of a segment that ends at bit se: the packed bytes, zeros from se on (jpeg.cu: a marker or the end feeds zeros).
__device__ __forceinline__ uint32_t jd_peek(const uint32_t* __restrict__ words, uint32_t pos, uint32_t se) {
    if (pos >= se) return 0;
    const uint32_t wi = pos >> 5, sh = pos & 31;
    const uint64_t x = ((uint64_t)__byte_perm(words[wi], 0, 0x0123) << 32) | __byte_perm(words[wi + 1], 0, 0x0123);
    uint32_t v = (uint32_t)(x >> (32 - sh));
    const uint32_t left = se - pos;
    if (left < 32) v &= ~(0xffffffffu >> left);
    return v;
}

// jpeg.cu BitReader::decode on the 32 bits at the read position: the symbol and its code length, or -1 for an invalid code
__device__ __forceinline__ int jd_symbol(const msc_jpeg_huff& t, uint32_t bits, uint32_t* len) {
    const uint32_t e = t.look[bits >> 23];
    if (e) { *len = e >> 8; return (int)(e & 0xff); }
    uint32_t l = 10;
    int32_t code = (int32_t)(bits >> 22);
    while (l <= 16 && code > t.maxcode[l]) { ++l; code = (int32_t)(bits >> (32 - l)); }
    if (l > 16) return -1;
    *len = l;
    return t.vals[(code + t.valptr[l]) & 0xff];
}

__device__ __forceinline__ int32_t jd_extend(uint32_t bits, uint32_t len, uint32_t s) {
    if (s == 0) return 0;
    const int32_t v = (int32_t)((bits << len) >> (32 - s));
    return v < (1 << (s - 1)) ? v - (1 << s) + 1 : v;
}

__device__ __forceinline__ uint64_t jd_pack(uint32_t pos, uint32_t slot, uint32_t zz) { return ((uint64_t)pos << 16) | (slot << 8) | zz; }

struct JdSegment {
    const uint32_t* words;
    uint32_t se, sat;      // end bit of the segment's data; positions saturate at sat (past se the stream is all zeros)
};

struct JdWriter {           // the final decode: where the blocks of the subsequence go
    int16_t* coef;          // the image's coefficients
    const JdImage* I;
    uint32_t first_block;   // decode-order index of the segment's first block
    uint32_t quota;         // blocks of the segment
};

// Decode symbols from state (pos, slot, zz) until the first symbol boundary at or after `end` (WRITE: or until the segment's block
// quota is reached, counting from block index `blk` of the segment).  Returns the state there, or kPoison after an invalid code, a DC
// size above 15 or an AC run past 63.  *done: blocks completed.  Terminates: every symbol consumes at least one bit.
template <bool WRITE>
__device__ __forceinline__ uint64_t jd_run(uint64_t st, uint32_t end, const JdSegment& S, const msc_jpeg_huff (*tabs)[2], const uint8_t* slot_comp, uint32_t bpm,
                           uint32_t* done, const JdWriter W, uint32_t blk, const uint8_t* zigzag) {
    uint32_t pos = (uint32_t)(st >> 16), slot = (uint32_t)(st >> 8) & 0xff, zz = (uint32_t)st & 0xff;
    uint32_t n = 0;
    int16_t* dst = nullptr;
    auto locate = [&]() {  // natural-order coefficients of block blk of the segment
        const JdImage& I = *W.I;
        const uint32_t g = W.first_block + blk;
        const uint32_t m = g / bpm;
        const int c = slot_comp[slot];
        const msc_jpeg_comp& k = I.d.comp[c];
        const uint32_t my = m / (uint32_t)I.d.mcus_x, mx = m - my * (uint32_t)I.d.mcus_x;
        const uint32_t by = my * k.v + I.slot_by[slot], bx = mx * k.h + I.slot_bx[slot];
        dst = W.coef + k.coef_off + ((size_t)by * k.blocks_x + bx) * 64;
    };
    if (WRITE) locate();
    while (pos < end) {
        const int c = slot_comp[slot];
        const uint32_t bits = jd_peek(S.words, pos, S.se);
        uint32_t len;
        bool complete = false;
        if (zz == 0) {
            const int s = jd_symbol(tabs[c][0], bits, &len);
            if (s < 0 || s > 15) { *done = n; return kPoison; }
            if (WRITE) dst[0] = (int16_t)jd_extend(bits, len, (uint32_t)s);  // the difference; the prediction follows per component
            pos += len + (uint32_t)s;
            zz = 1;
        } else {
            const int rs = jd_symbol(tabs[c][1], bits, &len);
            if (rs < 0) { *done = n; return kPoison; }
            const uint32_t r = (uint32_t)rs >> 4, sz = (uint32_t)rs & 15;
            if (sz == 0) {
                if (r == 15) {
                    zz += 16;
                    complete = zz > 63;
                } else {
                    complete = true;  // EOB
                }
            } else {
                zz += r;
                if (zz > 63) { *done = n; return kPoison; }
                if (WRITE) dst[zigzag[zz]] = (int16_t)jd_extend(bits, len, sz);
                ++zz;
                complete = zz == 64;
            }
            pos += len + sz;
        }
        pos = min(pos, S.sat);
        if (complete) {
            zz = 0;
            slot = slot + 1 == bpm ? 0 : slot + 1;
            ++n;
            if (WRITE) {
                if (++blk >= W.quota) break;
                locate();
            }
        }
    }
    *done = n;
    return jd_pack(pos, slot, zz);
}

struct JdSegFlag {
    uint32_t first, v;  // a segment's first subsequence; completed blocks
};
struct JdSegOp {
    __device__ __forceinline__ JdSegFlag operator()(const JdSegFlag& a, const JdSegFlag& b) const { return {a.first | b.first, b.first ? b.v : a.v + b.v}; }
};

// Synchronisation (DESIGN.md section 4.9): subsequence i's entry state is exact when it starts its segment, and when it is the first of a
// window (the exact exit of the window before).  Every other entry starts as a guess; each round re-decodes the subsequences whose entry
// changed, from the previous subsequence's exit.  In round r the first r + 1 entries of the window are exact (induction), so the loop
// reaches a fixed point after at most kJdThreads rounds whatever the data, and at the fixed point every entry is exact.
__global__ void __launch_bounds__(kJdThreads, 4) jd_huffman_kernel(const JdImage* __restrict__ imgs, const msc_jpeg_huff* __restrict__ huff,
                                                                int16_t* coef_all, const uint8_t* __restrict__ ws, int32_t* status, const uint8_t* __restrict__ zig) {
    using Scan = cub::BlockScan<JdSegFlag, kJdThreads>;
    __shared__ uint8_t zigzag[64];
    __shared__ typename Scan::TempStorage tmp;
    __shared__ msc_jpeg_huff tabs[3][2];
    __shared__ uint64_t exits[kJdThreads];
    __shared__ uint8_t slot_comp[8];
    const JdImage& I = imgs[blockIdx.x];
    if (status[blockIdx.x] != 0) return;
    int16_t* coef = coef_all + I.coef;
    {  // the host decoder starts from zeros
        int4* z = reinterpret_cast<int4*>(coef);
        const int64_t n16 = I.d.coef_elems / 8;
        for (int64_t i = threadIdx.x; i < n16; i += kJdThreads) z[i] = make_int4(0, 0, 0, 0);
    }
    for (int c = 0; c < I.d.n_comp; ++c)
        for (int k = 0; k < 2; ++k) {
            const uint32_t* src = reinterpret_cast<const uint32_t*>(huff + I.huff[c][k]);
            uint32_t* dst = reinterpret_cast<uint32_t*>(&tabs[c][k]);
            for (int i = threadIdx.x; i < (int)(sizeof(msc_jpeg_huff) / 4); i += kJdThreads) dst[i] = src[i];
        }
    if (threadIdx.x < 8) slot_comp[threadIdx.x] = I.slot_comp[threadIdx.x];
    if (threadIdx.x < 64) zigzag[threadIdx.x] = zig[threadIdx.x];
    __syncthreads();
    const uint32_t* seg_begin = reinterpret_cast<const uint32_t*>(ws + I.seg);
    const uint32_t* seg_end = seg_begin + I.n_seg;
    const uint32_t* sub_base = seg_end + I.n_seg;
    const uint32_t* words = reinterpret_cast<const uint32_t*>(ws + I.packed);
    const uint32_t n_sub = sub_base[I.n_seg], bpm = (uint32_t)I.bpm;
    const uint32_t seg_mcus = I.ri ? (uint32_t)I.ri : (uint32_t)I.total_mcus;
    uint64_t carry_exit = 0;
    uint32_t carry_blocks = 0;
    for (uint32_t w0 = 0; w0 < n_sub; w0 += kJdThreads) {
        const uint32_t i = w0 + threadIdx.x;
        const bool live = i < n_sub;
        int k = 0;
        bool first = true, last = true;
        uint32_t start = 0, end = kNone;
        JdSegment S = {words, 0, 0};
        if (live) {
            int lo = 0, hi = I.n_seg - 1;  // the segment: the last k with sub_base[k] <= i
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (sub_base[mid] <= i) lo = mid; else hi = mid - 1;
            }
            k = lo;
            const uint32_t j = i - sub_base[k];
            first = j == 0;
            last = i + 1 == sub_base[k + 1];
            S.se = seg_end[k] * 8u;
            S.sat = S.se + 64u;
            start = seg_begin[k] * 8u + j * kSubBits;
            end = last ? kNone : start + kSubBits;
        }
        const bool known = first || threadIdx.x == 0;
        uint64_t entry = (!first && threadIdx.x == 0) ? carry_exit : jd_pack(start, 0, 0);
        uint64_t exit = kPoison;
        uint32_t cnt = 0;
        bool need = live && !last;
        for (;;) {
            if (need) {
                cnt = 0;
                exit = entry == kPoison ? kPoison : jd_run<false>(entry, end, S, tabs, slot_comp, bpm, &cnt, JdWriter{}, 0, zigzag);
            }
            exits[threadIdx.x] = exit;
            __syncthreads();
            const uint64_t ne = (live && !known) ? exits[threadIdx.x - 1] : entry;
            const bool changed = ne != entry;
            if (!__syncthreads_or(changed)) break;
            entry = ne;
            need = changed && !last;
        }
        // blocks completed before each subsequence, within its segment
        JdSegFlag pre, agg;
        Scan(tmp).ExclusiveScan(JdSegFlag{first ? 1u : 0u, last ? 0u : cnt}, pre, JdSegFlag{0, 0}, JdSegOp(), agg);
        const uint32_t blk = first ? 0u : (pre.first ? pre.v : carry_blocks + pre.v);
        if (live && entry != kPoison) {
            const uint32_t seg_first = (uint32_t)k * seg_mcus;
            const uint32_t quota = min(seg_mcus, (uint32_t)I.total_mcus - seg_first) * bpm;
            if (blk < quota) {
                const JdWriter W = {coef, &I, seg_first * bpm, quota};
                uint32_t done;
                if (jd_run<true>(entry, end, S, tabs, slot_comp, bpm, &done, W, blk, zigzag) == kPoison) status[blockIdx.x] = MSC_ERR_BAD_ARGUMENT;
            }
        }
        carry_exit = exits[kJdThreads - 1];
        carry_blocks = agg.first ? agg.v : carry_blocks + agg.v;
        __syncthreads();
    }
    __syncthreads();
    // DC prediction: a segmented scan per component over its blocks in decode order, reset at every restart segment (int32 running
    // sums stored truncated to int16, as the host decoder does)
    for (int c = 0; c < I.d.n_comp; ++c) {
        const msc_jpeg_comp& K = I.d.comp[c];
        const uint32_t per = (uint32_t)(K.h * K.v), n = (uint32_t)I.total_mcus * per;
        int16_t* base = coef + K.coef_off;
        uint32_t run = 0;
        for (uint32_t q0 = 0; q0 < n; q0 += kJdThreads) {
            const uint32_t q = q0 + threadIdx.x;
            int16_t* dc = nullptr;
            JdSegFlag v = {0, 0};
            if (q < n) {
                const uint32_t m = q / per, r = q - m * per;
                const uint32_t my = m / (uint32_t)I.d.mcus_x, mx = m - my * (uint32_t)I.d.mcus_x;
                const uint32_t by = my * K.v + r / K.h, bx = mx * K.h + r % K.h;
                dc = base + ((size_t)by * K.blocks_x + bx) * 64;
                v = {(r == 0 && m % seg_mcus == 0) ? 1u : 0u, (uint32_t)(int32_t)*dc};
            }
            JdSegFlag inc, agg;
            __syncthreads();
            Scan(tmp).InclusiveScan(v, inc, JdSegOp(), agg);
            if (dc) *dc = (int16_t)(inc.first ? inc.v : run + inc.v);
            run = agg.first ? agg.v : run + agg.v;
        }
    }
}

// ------------------------------------------------------------------------------------------------ reconstruction
__device__ __forceinline__ int jd_find(const int32_t* __restrict__ first, int n, int cta) {  // the last i with first[i] <= cta
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (first[mid] <= cta) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// jpeg.cu's jpeg_idct_kernel: 8 threads per 8x8 block, 32 blocks per CTA; the CTA's image and component come from the tables
__global__ void __launch_bounds__(256) jd_idct_kernel(const JdImage* __restrict__ imgs, const int32_t* __restrict__ idct_first, int n_img,
                                                      const int16_t* __restrict__ coef_all, uint8_t* ws) {
    __shared__ int wsm[32][64 + 1];
    const int im = jd_find(idct_first, n_img, blockIdx.x);
    const JdImage& I = imgs[im];
    const int rel = blockIdx.x - idct_first[im];
    int c = 0;
    while (c + 1 < I.d.n_comp && I.idct_cta[c + 1] <= rel) ++c;
    const msc_jpeg_comp& K = I.d.comp[c];
    const int lb = threadIdx.x >> 3, j = threadIdx.x & 7;
    const int b = (rel - I.idct_cta[c]) * 32 + lb;
    const bool live = b < K.blocks_x * K.blocks_y;
    int o[8];
    if (live) {  // pass 1: columns, dequantised input, results scaled up by 2^PASS1_BITS
        const int16_t* cf = coef_all + I.coef + K.coef_off + (size_t)b * 64 + j;
        const uint16_t* qt = K.qt;
        jd_butterfly(cf[0] * (int)qt[j], cf[8] * (int)qt[8 + j], cf[16] * (int)qt[16 + j], cf[24] * (int)qt[24 + j], cf[32] * (int)qt[32 + j],
                     cf[40] * (int)qt[40 + j], cf[48] * (int)qt[48 + j], cf[56] * (int)qt[56 + j], o, 13 - 2);
#pragma unroll
        for (int r = 0; r < 8; ++r) wsm[lb][r * 8 + j] = o[r];
    }
    __syncthreads();
    if (live) {  // pass 2: rows, descale by CONST_BITS + PASS1_BITS + 3, level shift + range limit
        const int* w = &wsm[lb][j * 8];
        jd_butterfly(w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], o, 13 + 2 + 3);
        const int bx = b % K.blocks_x, by = b / K.blocks_x;
        uint8_t* dst = ws + I.planes + K.plane_off + ((size_t)(by * 8 + j) * K.blocks_x + bx) * 8;
        uint2 pk;
        pk.x = (uint32_t)jd_idct_limit(o[0]) | ((uint32_t)jd_idct_limit(o[1]) << 8) | ((uint32_t)jd_idct_limit(o[2]) << 16) | ((uint32_t)jd_idct_limit(o[3]) << 24);
        pk.y = (uint32_t)jd_idct_limit(o[4]) | ((uint32_t)jd_idct_limit(o[5]) << 8) | ((uint32_t)jd_idct_limit(o[6]) << 16) | ((uint32_t)jd_idct_limit(o[7]) << 24);
        *reinterpret_cast<uint2*>(dst) = pk;
    }
}

// jpeg.cu's jpeg_color_kernel: one CTA per 256 pixels of a row
__global__ void __launch_bounds__(256) jd_color_kernel(const JdImage* __restrict__ imgs, const int32_t* __restrict__ color_first, int n_img,
                                                       const uint8_t* __restrict__ ws, uint8_t* out_all) {
    const int im = jd_find(color_first, n_img, blockIdx.x);
    const JdImage& I = imgs[im];
    const int rel = blockIdx.x - color_first[im];
    const int y = rel / I.color_chunks, x = (rel - y * I.color_chunks) * 256 + threadIdx.x;
    const int width = I.d.width;
    if (x >= width) return;
    const uint8_t* planes = ws + I.planes;
    uint8_t* out = out_all + I.out;
    const int Y = planes[I.d.comp[0].plane_off + (size_t)y * (I.d.comp[0].blocks_x * 8) + x];
    if (I.d.n_comp == 1) {
        out[(size_t)y * width + x] = (uint8_t)Y;
        return;
    }
    const msc_jpeg_comp& K = I.d.comp[1];
    const int stride = K.blocks_x * 8;
    const int cb = jd_chroma(planes + K.plane_off, stride, K.ds_w, K.ds_h, I.d.hmax, I.d.vmax, x, y) - 128;
    const int cr = jd_chroma(planes + I.d.comp[2].plane_off, stride, K.ds_w, K.ds_h, I.d.hmax, I.d.vmax, x, y) - 128;
    jd_ycc_rgb(Y, cb, cr, out + ((size_t)y * width + x) * 3);
}

// ------------------------------------------------------------------------------------------------ host
static size_t jd_al(size_t v) { return (v + 255) & ~(size_t)255; }

// a plan's descriptor as parse_headers builds it (the batch trusts its geometry for every address it forms)
static bool jd_plan_ok(const msc_jpeg_plan& p) {
    const msc_jpeg_desc& d = p.desc;
    if (d.n_comp != 1 && d.n_comp != 3) return false;
    if (d.width < 1 || d.width > 65535 || d.height < 1 || d.height > 65535) return false;
    if (p.scan_off < 0 || p.scan_bytes < 0 || p.scan_bytes >= kMaxScanBytes || p.restart_interval < 0) return false;
    if (d.n_comp == 1 && (d.hmax != 1 || d.vmax != 1 || d.comp[0].h != 1 || d.comp[0].v != 1)) return false;
    if (d.n_comp == 3) {
        const bool layout = (d.hmax == 1 && d.vmax == 1) || (d.hmax == 2 && d.vmax == 1) || (d.hmax == 2 && d.vmax == 2);
        if (!layout || d.comp[0].h != d.hmax || d.comp[0].v != d.vmax) return false;
        for (int c = 1; c < 3; ++c)
            if (d.comp[c].h != 1 || d.comp[c].v != 1) return false;
    }
    if (d.mcus_x != (d.width + 8 * d.hmax - 1) / (8 * d.hmax) || d.mcus_y != (d.height + 8 * d.vmax - 1) / (8 * d.vmax)) return false;
    int64_t coef = 0;
    for (int c = 0; c < d.n_comp; ++c) {
        const msc_jpeg_comp& k = d.comp[c];
        if (p.td[c] < 0 || p.td[c] > 3 || p.ta[c] < 0 || p.ta[c] > 3) return false;
        if (k.blocks_x != d.mcus_x * k.h || k.blocks_y != d.mcus_y * k.v || k.coef_off != coef || k.plane_off != coef) return false;
        if (k.ds_w != (d.width * k.h + d.hmax - 1) / d.hmax || k.ds_h != (d.height * k.v + d.vmax - 1) / d.vmax) return false;
        coef += (int64_t)k.blocks_x * k.blocks_y * 64;
    }
    return d.coef_elems == coef && d.plane_bytes == coef;
}

struct JdLayout {
    size_t zig, imgs, idct_first, color_first, huff, table_end, total;
    std::vector<int64_t> per_image;  // first workspace byte of each image's region
    int64_t idct_ctas = 0, color_ctas = 0;
};

static int jd_n_seg(const msc_jpeg_plan& p) {
    const int64_t mcus = (int64_t)p.desc.mcus_x * p.desc.mcus_y;
    return p.restart_interval ? (int)((mcus + p.restart_interval - 1) / p.restart_interval) : 1;
}

static size_t jd_image_bytes(const msc_jpeg_plan& p) {
    return jd_al((size_t)p.scan_bytes + 16) + jd_al(((size_t)3 * jd_n_seg(p) + 1) * 4) + jd_al((size_t)p.desc.plane_bytes);
}

static bool jd_layout(int32_t n, const msc_jpeg_plan* plans, JdLayout* L) {
    if (n < 0 || (n > 0 && !plans)) return false;
    size_t o = 0;
    L->zig = o; o = jd_al(o + 64);
    L->imgs = o; o = jd_al(o + (size_t)n * sizeof(JdImage));
    L->idct_first = o; o = jd_al(o + ((size_t)n + 1) * 4);
    L->color_first = o; o = jd_al(o + ((size_t)n + 1) * 4);
    L->huff = o; o = jd_al(o + (size_t)n * 6 * sizeof(msc_jpeg_huff));
    L->table_end = o;
    L->per_image.resize((size_t)n);
    for (int32_t i = 0; i < n; ++i) {
        const msc_jpeg_plan& p = plans[i];
        if (!jd_plan_ok(p)) return false;
        L->per_image[(size_t)i] = (int64_t)o;
        o += jd_image_bytes(p);
        const msc_jpeg_desc& d = p.desc;
        for (int c = 0; c < d.n_comp; ++c) L->idct_ctas += ((int64_t)d.comp[c].blocks_x * d.comp[c].blocks_y + 31) / 32;
        L->color_ctas += (int64_t)d.height * ((d.width + 255) / 256);
    }
    if (L->idct_ctas > 0x7fffffff || L->color_ctas > 0x7fffffff) return false;
    L->total = o > 256 ? o : 256;
    return true;
}

}  // namespace msc

extern "C" {

size_t msc_jpeg_decode_batch_workspace_bytes(int32_t n, const msc_jpeg_plan* plans_host) {
    msc::JdLayout L;
    return msc::jd_layout(n, plans_host, &L) ? L.total : 0;
}

int msc_jpeg_decode_batch(int32_t n, const msc_jpeg_plan* plans_host, const uint8_t* files, const int64_t* file_off_host, int16_t* coef,
                          const int64_t* coef_off_host, uint8_t* out, const int64_t* out_off_host, int32_t* status, void* workspace,
                          size_t workspace_bytes, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(n >= 0, "msc_jpeg_decode_batch: negative n");
    if (n == 0) return MSC_OK;
    MSC_REQUIRE(plans_host && files && file_off_host && coef && coef_off_host && out && out_off_host && status && workspace,
                "msc_jpeg_decode_batch: a pointer argument is NULL");
    MSC_REQUIRE(((uintptr_t)workspace & 255) == 0, "msc_jpeg_decode_batch: workspace must be 256-byte aligned");
    MSC_REQUIRE(((uintptr_t)coef & 15) == 0, "msc_jpeg_decode_batch: coef must be 16-byte aligned");
    JdLayout L;
    MSC_REQUIRE(jd_layout(n, plans_host, &L), "msc_jpeg_decode_batch: a plan is not a supported sequential JPEG (or the batch is too large)");
    MSC_REQUIRE(workspace_bytes >= L.total, "msc_jpeg_decode_batch: workspace too small: need %zu bytes, got %zu", L.total, workspace_bytes);
    for (int32_t i = 0; i < n; ++i)
        MSC_REQUIRE(file_off_host[i] >= 0 && coef_off_host[i] >= 0 && (coef_off_host[i] & 7) == 0 && out_off_host[i] >= 0,
                    "msc_jpeg_decode_batch: image %d: negative offset or coef offset not a multiple of 8", (int)i);

    std::vector<unsigned char> host(L.table_end, 0);
    memcpy(host.data() + L.zig, kZigzag, 64);
    JdImage* rec = reinterpret_cast<JdImage*>(host.data() + L.imgs);
    int32_t* idct_first = reinterpret_cast<int32_t*>(host.data() + L.idct_first);
    int32_t* color_first = reinterpret_cast<int32_t*>(host.data() + L.color_first);
    msc_jpeg_huff* huff = reinterpret_cast<msc_jpeg_huff*>(host.data() + L.huff);
    int n_huff = 0;
    auto intern = [&](const msc_jpeg_huff& t) {  // consecutive files usually share their tables
        for (int k = n_huff - 1; k >= 0 && k >= n_huff - 16; --k)
            if (!memcmp(&huff[k], &t, sizeof(t))) return k;
        huff[n_huff] = t;
        return n_huff++;
    };
    int32_t icta = 0, ccta = 0;
    for (int32_t i = 0; i < n; ++i) {
        const msc_jpeg_plan& p = plans_host[i];
        JdImage& R = rec[i];
        R.d = p.desc;
        R.scan = file_off_host[i] + p.scan_off;
        R.coef = coef_off_host[i];
        R.out = out_off_host[i];
        const int64_t base = L.per_image[(size_t)i];
        R.packed = base;
        R.seg = R.packed + (int64_t)jd_al((size_t)p.scan_bytes + 16);
        R.planes = R.seg + (int64_t)jd_al(((size_t)3 * jd_n_seg(p) + 1) * 4);
        R.scan_bytes = (int32_t)p.scan_bytes;
        R.n_seg = jd_n_seg(p);
        R.ri = p.restart_interval;
        R.total_mcus = p.desc.mcus_x * p.desc.mcus_y;
        int slot = 0;
        for (int c = 0; c < p.desc.n_comp; ++c) {
            R.huff[c][0] = intern(p.dc[p.td[c]]);
            R.huff[c][1] = intern(p.ac[p.ta[c]]);
            for (int by = 0; by < p.desc.comp[c].v; ++by)
                for (int bx = 0; bx < p.desc.comp[c].h; ++bx, ++slot) {
                    R.slot_comp[slot] = (uint8_t)c; R.slot_by[slot] = (uint8_t)by; R.slot_bx[slot] = (uint8_t)bx;
                }
        }
        R.bpm = slot;
        int32_t rel = 0;
        for (int c = 0; c < p.desc.n_comp; ++c) {
            R.idct_cta[c] = rel;
            rel += (p.desc.comp[c].blocks_x * p.desc.comp[c].blocks_y + 31) / 32;
        }
        R.idct_cta[p.desc.n_comp] = rel;
        R.color_chunks = (p.desc.width + 255) / 256;
        idct_first[i] = icta; icta += rel;
        color_first[i] = ccta; ccta += p.desc.height * R.color_chunks;
    }
    idct_first[n] = icta;
    color_first[n] = ccta;

    unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
    const JdImage* d_rec = reinterpret_cast<const JdImage*>(ws + L.imgs);
    cudaStream_t stream = (cudaStream_t)stream_v;
    // pageable source: staged before the call returns, so `host` may go out of scope
    MSC_CUDA(cudaMemcpyAsync(ws, host.data(), L.huff + (size_t)n_huff * sizeof(msc_jpeg_huff), cudaMemcpyHostToDevice, stream));
    jd_unstuff_kernel<<<(unsigned)n, kJdThreads, 0, stream>>>(d_rec, files, ws, status);
    jd_huffman_kernel<<<(unsigned)n, kJdThreads, 0, stream>>>(d_rec, reinterpret_cast<const msc_jpeg_huff*>(ws + L.huff), coef, ws, status, ws + L.zig);
    if (icta) jd_idct_kernel<<<(unsigned)icta, 256, 0, stream>>>(d_rec, reinterpret_cast<const int32_t*>(ws + L.idct_first), n, coef, ws);
    if (ccta) jd_color_kernel<<<(unsigned)ccta, 256, 0, stream>>>(d_rec, reinterpret_cast<const int32_t*>(ws + L.color_first), n, ws, out);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

}  // extern "C"
