// jpeg_encode.cu -- camera-frame JPEG encode on the device, byte-identical to Pillow's `Image.fromarray(rgb).save(buf, "JPEG", quality=q)`
// (the reference's CameraAgent._encode_image, camera_agent.py:128-137), i.e. libjpeg-turbo's default compression: JFIF 4:2:0, the
// Annex K quantisation tables scaled by jpeg_set_quality, 16-bit fixed-point RGB -> YCbCr (jccolor.c), h2v2 downsampling with the
// alternating 1 / 2 bias (jcsample.c), the slow-integer FDCT (jfdctint.c), round-half-away quantisation, the Annex K.3 Huffman tables,
// no restart markers.  Every step is integer arithmetic with fixed rounding, so equality is a matter of following it to the letter.
//
// A batch of same-sized images is encoded in six launches, none of which synchronises the host or allocates:
//   1. jpeg_enc_kernel<false>  per CTA of 42 MCUs: colour, edge replication, downsampling, FDCT, quantisation, then the Huffman code
//                              length of every block; writes the CTA's bit count and its first / last DC values.
//   2. jpeg_enc_offsets_kernel per image: adds the DC code lengths that depend on the previous CTA, scans -> each CTA's bit offset.
//   3. jpeg_enc_kernel<true>   recomputes the coefficients (cheaper than storing them), scans the block lengths inside the CTA and
//                              packs the CTA's bits in shared memory; words shared with a neighbouring CTA go to a side slot.
//   4. jpeg_enc_size_kernel    per image: merges the shared words, counts the 0xFF bytes of the scan -> file size.
//   5. jpeg_enc_outoff_kernel  scans the file sizes -> out_off, sets the status word.
//   6. jpeg_enc_place_kernel   per image: header, byte-stuffed scan, EOI into the arena (nothing when the arena is too small).
// Each image owns a fixed region of the workspace sized for its worst-case scan, so results never depend on scheduling or on the
// other images of the batch.
#include <initializer_list>

#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include "jpeg_common.cuh"
#include "msc_common.cuh"

namespace msc {

constexpr int kEncThreads = 256;
constexpr int kEncMcus = 42;                  // MCUs per CTA: 6 * 42 = 252 blocks, one per thread in the Huffman pass
constexpr int kEncBlocks = 6 * kEncMcus;
constexpr int kCoefStride = 66;               // int16 per block row in shared memory: an odd word stride, no bank conflicts
constexpr int kMaxBlockBits = 22 + 63 * 26;   // DC: 11-bit code + 11 bits; AC: 16-bit code + 10 bits per coefficient
constexpr int kCtaWords = (kEncBlocks * kMaxBlockBits + 31 + 7) / 32 + 1;
constexpr int kHeaderMax = 640;

struct EncGeom {
    int32_t width, height;
    int32_t mcus_x, mcus;          // per image
    int32_t blocks_x, blocks_y;    // luma blocks that hold image data: ceil(W / 8), ceil(H / 8)
    int32_t chroma_h;              // downsampled chroma rows, ceil(H / 2)
    int32_t ctas;                  // CTAs per image
    int64_t img_bytes;             // H * W * 3
    int64_t region_words;          // u32 words of scan workspace per image
};

struct EncTables {
    uint16_t div[2][64];   // 8 * quantisation value, natural order; [0] luma, [1] chroma
    uint8_t zz[64];        // zigzag position -> natural index
    uint32_t dc[2][12];    // (code length << 16) | code, per DC category
    uint32_t ac[2][256];   // (code length << 16) | code, per (run << 4 | size) symbol
};

struct EncHeader {
    int32_t len;
    uint8_t b[kHeaderMax];
};

// the tables as the kernels read them: staged in shared memory once per CTA, since the Huffman walk and the quantiser index them with
// per-thread indices (from the parameter bank those loads would serialise)
struct JeTables {
    uint32_t ac[2][256];
    uint32_t dc[2][12];
    uint16_t div[2][64];
    uint8_t zz[64];
    __device__ __forceinline__ void load(const EncTables& T) {
        for (int i = threadIdx.x; i < 512; i += blockDim.x) ac[i >> 8][i & 255] = T.ac[i >> 8][i & 255];
        for (int i = threadIdx.x; i < 128; i += blockDim.x) div[i >> 6][i & 63] = T.div[i >> 6][i & 63];
        for (int i = threadIdx.x; i < 24; i += blockDim.x) dc[i / 12][i % 12] = T.dc[i / 12][i % 12];
        for (int i = threadIdx.x; i < 64; i += blockDim.x) zz[i] = T.zz[i];
    }
};

struct EncCta {
    uint32_t bits;           // pass 1: bits of the CTA's blocks without the DC codes of its first Y, Cb and Cr block
    int16_t dc_first[3];     // Y0, Cb, Cr of the first MCU
    int16_t dc_last[3];      // Y3, Cb, Cr of the last MCU
};

__device__ __forceinline__ int je_descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }

// jfdctint.c (jpeg_fdct_islow), one 1-D pass: CONST_BITS 13, PASS1_BITS 2; the row pass scales up by 2^PASS1_BITS, the column pass
// descales by it, so the output is the DCT scaled by 8
template <bool ROWS>
__device__ __forceinline__ void je_fdct8(const int d[8], int o[8]) {
    constexpr int C = 13, P = 2, SH = ROWS ? C - P : C + P;
    int t0 = d[0] + d[7], t7 = d[0] - d[7], t1 = d[1] + d[6], t6 = d[1] - d[6];
    int t2 = d[2] + d[5], t5 = d[2] - d[5], t3 = d[3] + d[4], t4 = d[3] - d[4];
    const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    if (ROWS) {
        o[0] = (t10 + t11) * (1 << P);
        o[4] = (t10 - t11) * (1 << P);
    } else {
        o[0] = je_descale(t10 + t11, P);
        o[4] = je_descale(t10 - t11, P);
    }
    int z1 = (t12 + t13) * 4433;
    o[2] = je_descale(z1 + t13 * 6270, SH);
    o[6] = je_descale(z1 - t12 * 15137, SH);
    z1 = t4 + t7;
    int z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7;
    const int z5 = (z3 + z4) * 9633;
    t4 *= 2446; t5 *= 16819; t6 *= 25172; t7 *= 12299;
    z1 *= -7373; z2 *= -20995;
    z3 = z3 * -16069 + z5;
    z4 = z4 * -3196 + z5;
    o[7] = je_descale(t4 + z1 + z3, SH);
    o[5] = je_descale(t5 + z2 + z4, SH);
    o[3] = je_descale(t6 + z2 + z3, SH);
    o[1] = je_descale(t7 + z1 + z4, SH);
}

// N pixels (3 N bytes) of one image row from column x0, edge-replicated past the right edge; vector loads where the row allows
template <int N>  // 8 or 16
__device__ __forceinline__ void je_load_row(const uint8_t* __restrict__ row, int x0, int W, uint32_t (&w)[N * 3 / 4]) {
    const uint8_t* p = row + (size_t)x0 * 3;
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    if (x0 + N <= W && (a & (N - 1)) == 0) {  // N-byte loads: 16 bytes for 16 pixels, 8 for 8
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            if constexpr (N == 16) {
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(p) + k);
                w[4 * k] = v.x; w[4 * k + 1] = v.y; w[4 * k + 2] = v.z; w[4 * k + 3] = v.w;
            } else {
                const uint2 v = __ldg(reinterpret_cast<const uint2*>(p) + k);
                w[2 * k] = v.x; w[2 * k + 1] = v.y;
            }
        }
    } else {
#pragma unroll
        for (int k = 0; k < N * 3 / 4; ++k) w[k] = 0;
#pragma unroll
        for (int i = 0; i < N * 3; ++i) {
            const int x = min(x0 + i / 3, W - 1);
            w[i >> 2] |= (uint32_t)__ldg(row + (size_t)x * 3 + i % 3) << (8 * (i & 3));
        }
    }
}

template <int N>
__device__ __forceinline__ int je_byte(const uint32_t (&w)[N], int i) { return (int)((w[i >> 2] >> (8 * (i & 3))) & 255u); }

// jccolor.c rgb_ycc_convert: FIX(x) = (int)(x * 65536 + 0.5); Y rounds with ONE_HALF, Cb / Cr with CBCR_OFFSET + ONE_HALF - 1
__device__ __forceinline__ int je_y(int r, int g, int b) { return (19595 * r + 38470 * g + 7471 * b + 32768) >> 16; }
__device__ __forceinline__ int je_cb(int r, int g, int b) { return (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16; }
__device__ __forceinline__ int je_cr(int r, int g, int b) { return (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16; }

__device__ __forceinline__ int je_nbits(int v) { return v ? 32 - __clz(v < 0 ? -v : v) : 0; }

// bit sinks of the Huffman walk: one counts, one packs MSB-first into shared-memory words (atomicOr: the first and last word of a
// block are shared with its neighbours)
struct JeCount {
    uint32_t n = 0;
    __device__ __forceinline__ void put(uint32_t, int len) { n += (uint32_t)len; }
};
struct JePack {
    uint32_t* buf;
    uint32_t w;
    int n;
    uint64_t acc;
    __device__ __forceinline__ JePack(uint32_t* b, uint32_t pos) : buf(b), w(pos >> 5), n((int)(pos & 31)), acc(0) {}
    __device__ __forceinline__ void put(uint32_t bits, int len) {  // len <= 27
        acc = (acc << len) | bits;
        n += len;
        if (n >= 32) {
            n -= 32;
            atomicOr(&buf[w++], (uint32_t)(acc >> n));
            acc &= (1ull << n) - 1ull;
        }
    }
    __device__ __forceinline__ void flush() {
        if (n) atomicOr(&buf[w], (uint32_t)(acc << (32 - n)));
    }
};

// jchuff.c encode_one_block: DC difference, then run-length coded AC (ZRL only in front of a nonzero coefficient, EOB only when the
// block ends in zeros); a negative value v is sent as the low n bits of v - 1
template <class Sink>
__device__ __forceinline__ void je_block(const int16_t* __restrict__ c, int diff, bool with_dc, int tab, const JeTables& T, Sink& s) {
    if (with_dc) {
        const int n = je_nbits(diff);
        const uint32_t code = T.dc[tab][n];
        s.put(((code & 0xffffu) << n) | ((uint32_t)(diff < 0 ? diff - 1 : diff) & ((1u << n) - 1u)), (int)(code >> 16) + n);
    }
    int run = 0;
    for (int k = 1; k < 64; ++k) {
        const int v = c[T.zz[k]];
        if (v == 0) {
            ++run;
            continue;
        }
        for (; run > 15; run -= 16) {
            const uint32_t zrl = T.ac[tab][0xf0];
            s.put(zrl & 0xffffu, (int)(zrl >> 16));
        }
        const int n = je_nbits(v);
        const uint32_t code = T.ac[tab][(run << 4) + n];
        s.put(((code & 0xffffu) << n) | ((uint32_t)(v < 0 ? v - 1 : v) & ((1u << n) - 1u)), (int)(code >> 16) + n);
        run = 0;
    }
    if (run) {
        const uint32_t eob = T.ac[tab][0];
        s.put(eob & 0xffffu, (int)(eob >> 16));
    }
}

__device__ __forceinline__ uint32_t je_dc_bits(const JeTables& T, int tab, int diff) {
    const int n = je_nbits(diff);
    return (T.dc[tab][n] >> 16) + (uint32_t)n;
}

// One CTA = kEncMcus consecutive MCUs of one image.  Transform: 8 threads per block (thread j: row j, then column j), 32 blocks per
// round, quantised coefficients (natural order) staged in shared memory.  Huffman pass: one thread per block.
// PACK = false: per-CTA bit count and boundary DC values -> rec.  PACK = true: the CTA's bits at cta_off -> region / head / tail.
template <bool PACK>
__global__ void __launch_bounds__(kEncThreads) jpeg_enc_kernel(const EncGeom G, const EncTables T, const uint8_t* __restrict__ rgb,
                                                               EncCta* __restrict__ rec, const uint64_t* __restrict__ cta_off,
                                                               uint32_t* __restrict__ region, uint32_t* __restrict__ head,
                                                               uint32_t* __restrict__ tail) {
    __shared__ int16_t coef[kEncBlocks][kCoefStride];
    __shared__ int ws[32][64 + 1];
    __shared__ JeTables tabs;
    using Scan = cub::BlockScan<uint32_t, kEncThreads>;
    using Reduce = cub::BlockReduce<uint32_t, kEncThreads>;
    __shared__ union {
        typename Scan::TempStorage scan;
        typename Reduce::TempStorage reduce;
    } cubtmp;
    extern __shared__ uint32_t bitbuf[];  // PACK only: kCtaWords

    const int64_t cta = blockIdx.x;
    const int64_t img = cta / G.ctas;
    const int cc = (int)(cta - img * G.ctas);
    const int m0 = cc * kEncMcus;
    const int nm = min(kEncMcus, G.mcus - m0);
    const int nb = nm * 6;
    const uint8_t* __restrict__ src = rgb + img * G.img_bytes;
    const int W = G.width, H = G.height;
    const int tid = threadIdx.x, lb = tid >> 3, j = tid & 7;
    tabs.load(T);
    __syncthreads();

    for (int r = 0; r * 32 < nb; ++r) {
        const int k = r * 32 + lb;
        const int m = m0 + k / 6, p = k % 6;
        const int my = m / G.mcus_x, mx = m - my * G.mcus_x;
        const int yy = 2 * my + (p >> 1), xx = 2 * mx + (p & 1);
        const bool live = k < nb;
        const bool dummy = p < 4 && (yy >= G.blocks_y || xx >= G.blocks_x);  // jccoefct.c: zero AC, DC copied below
        if (live && !dummy) {
            int d[8], o[8];
            if (p < 4) {
                uint32_t w[6];
                je_load_row<8>(src + (size_t)min(8 * yy + j, H - 1) * W * 3, 8 * xx, W, w);
#pragma unroll
                for (int i = 0; i < 8; ++i) d[i] = je_y(je_byte(w, 3 * i), je_byte(w, 3 * i + 1), je_byte(w, 3 * i + 2)) - 128;
            } else {
                // h2v2_downsample of rows 2 cy, 2 cy + 1 (the last row repeated for odd heights): (a + b + c + d + bias) >> 2, bias 1, 2, ...
                const int cy = min(8 * my + j, G.chroma_h - 1);
                uint32_t w0[12], w1[12];
                je_load_row<16>(src + (size_t)(2 * cy) * W * 3, 16 * mx, W, w0);
                je_load_row<16>(src + (size_t)min(2 * cy + 1, H - 1) * W * 3, 16 * mx, W, w1);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    int s = 0;
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        const int e = 3 * (2 * i + q);
                        s += p == 4 ? je_cb(je_byte(w0, e), je_byte(w0, e + 1), je_byte(w0, e + 2)) + je_cb(je_byte(w1, e), je_byte(w1, e + 1), je_byte(w1, e + 2))
                                    : je_cr(je_byte(w0, e), je_byte(w0, e + 1), je_byte(w0, e + 2)) + je_cr(je_byte(w1, e), je_byte(w1, e + 1), je_byte(w1, e + 2));
                    }
                    d[i] = ((s + 1 + (i & 1)) >> 2) - 128;
                }
            }
            je_fdct8<true>(d, o);
#pragma unroll
            for (int i = 0; i < 8; ++i) ws[lb][j * 8 + i] = o[i];
        }
        __syncthreads();
        if (live) {
            if (dummy) {
#pragma unroll
                for (int i = 0; i < 8; ++i) coef[k][i * 8 + j] = 0;
            } else {
                int d[8], o[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) d[i] = ws[lb][i * 8 + j];
                je_fdct8<false>(d, o);
                const int tab = p < 4 ? 0 : 1;
#pragma unroll
                for (int i = 0; i < 8; ++i) {  // jcdctmgr.c quantize: divide by 8 * qval, rounding half away from zero
                    const int q = tabs.div[tab][i * 8 + j];
                    const int a = (abs(o[i]) + (q >> 1)) / q;
                    coef[k][i * 8 + j] = (int16_t)(o[i] < 0 ? -a : a);
                }
            }
        }
        __syncthreads();
    }
    if (tid < nm) {  // dummy blocks: right edge -> DC of the block to the left; bottom row -> DC of the MCU's block 1, for both
        const int m = m0 + tid, my = m / G.mcus_x, mx = m - my * G.mcus_x;
        int16_t* b = &coef[tid * 6][0];
        const bool right = 2 * mx + 1 >= G.blocks_x, bottom = 2 * my + 1 >= G.blocks_y;
        if (right) b[kCoefStride] = b[0];
        if (bottom) {
            b[2 * kCoefStride] = b[kCoefStride];
            b[3 * kCoefStride] = b[kCoefStride];
        } else if (right) {
            b[3 * kCoefStride] = b[2 * kCoefStride];
        }
    }
    __syncthreads();

    // Huffman pass: block tid.  DC predictor: the previous block of the same component (Y: the previous Y block; Cb / Cr: previous MCU)
    const int p = tid % 6;
    const int tab = p < 4 ? 0 : 1;
    const int comp = p < 4 ? 0 : p - 3;
    const bool live = tid < nb;
    const bool first_of_comp = tid < 6 && (p == 0 || p >= 4);
    int pred = 0;
    if (live && !first_of_comp) pred = coef[p == 0 ? tid - 3 : (p < 4 ? tid - 1 : tid - 6)][0];
    if (PACK && live && first_of_comp && cc > 0) pred = rec[cta - 1].dc_last[comp];
    const int dc = live ? coef[tid][0] : 0;

    JeCount cnt;
    if (live) je_block(&coef[tid][0], dc - pred, PACK || !first_of_comp, tab, tabs, cnt);
    if (!PACK) {
        const uint32_t total = Reduce(cubtmp.reduce).Sum(cnt.n);
        if (tid == 0) {
            EncCta e;
            e.bits = total;
            e.dc_first[0] = coef[0][0]; e.dc_first[1] = coef[4][0]; e.dc_first[2] = coef[5][0];
            e.dc_last[0] = coef[nb - 3][0]; e.dc_last[1] = coef[nb - 2][0]; e.dc_last[2] = coef[nb - 1][0];
            rec[cta] = e;
        }
        return;
    }
    uint32_t excl, total;
    Scan(cubtmp.scan).ExclusiveSum(cnt.n, excl, total);
    const uint64_t s = cta_off[cta];  // first bit of this CTA within its image's scan
    const uint32_t lead = (uint32_t)(s & 31);
    const bool last_cta = cc == G.ctas - 1;
    const uint32_t end = lead + total;
    const uint32_t end_pad = last_cta ? (end + 7) & ~7u : end;  // the scan's last byte is padded with 1-bits
    const int nw = (int)((end_pad + 31) >> 5);
    for (int w = tid; w < nw; w += kEncThreads) bitbuf[w] = 0;
    __syncthreads();
    if (live) {
        JePack pk(bitbuf, lead + excl);
        je_block(&coef[tid][0], dc - pred, true, tab, tabs, pk);
        pk.flush();
    }
    __syncthreads();
    if (tid == 0 && end_pad > end) {
        const int pad = (int)(end_pad - end);
        bitbuf[end >> 5] |= ((1u << pad) - 1u) << (32 - (int)(end & 31) - pad);
    }
    __syncthreads();
    uint32_t* dst = region + img * G.region_words + (s >> 5);
    for (int w = tid; w < nw; w += kEncThreads) {
        const uint32_t v = __byte_perm(bitbuf[w], 0, 0x0123);  // MSB-first words -> bytes in stream order
        if (w == 0 && lead) head[cta] = v;
        else if (w == nw - 1 && (end_pad & 31)) tail[cta] = v;
        else dst[w] = v;
    }
}

// per image: bit offset of every CTA (adding the DC codes of each CTA's first Y / Cb / Cr block) and the scan's bit count
__global__ void __launch_bounds__(kEncThreads) jpeg_enc_offsets_kernel(const EncGeom G, const EncTables T, const EncCta* __restrict__ rec,
                                                                       uint64_t* __restrict__ cta_off, uint64_t* __restrict__ img_bits) {
    using Scan = cub::BlockScan<uint64_t, kEncThreads>;
    __shared__ typename Scan::TempStorage tmp;
    __shared__ JeTables tabs;
    tabs.load(T);
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * G.ctas;
    uint64_t running = 0;
    for (int c0 = 0; c0 < G.ctas; c0 += kEncThreads) {
        const int c = c0 + threadIdx.x;
        uint64_t bits = 0;
        if (c < G.ctas) {
            const EncCta e = rec[base + c];
            int16_t prev[3] = {0, 0, 0};
            if (c > 0) {
                const EncCta q = rec[base + c - 1];
                prev[0] = q.dc_last[0]; prev[1] = q.dc_last[1]; prev[2] = q.dc_last[2];
            }
            bits = (uint64_t)e.bits + je_dc_bits(tabs, 0, e.dc_first[0] - prev[0]) + je_dc_bits(tabs, 1, e.dc_first[1] - prev[1]) +
                   je_dc_bits(tabs, 1, e.dc_first[2] - prev[2]);
        }
        uint64_t excl, agg;
        Scan(tmp).ExclusiveSum(bits, excl, agg);
        if (c < G.ctas) cta_off[base + c] = running + excl;
        running += agg;
        __syncthreads();
    }
    if (threadIdx.x == 0) img_bits[blockIdx.x] = running;
}

// 0xFF bytes among the first min(left, 4) bytes of a scan word (bytes in stream order)
__device__ __forceinline__ uint32_t je_ff_bytes(uint32_t v, uint64_t left) {
    const uint32_t mask = left >= 4 ? 0xffffffffu : (1u << (8 * left)) - 1u;
    return __popc(__vcmpeq4(v, 0xffffffffu) & mask) >> 3;
}

// per image: merge the words two CTAs share, then count the scan's 0xFF bytes -> the file size (header + stuffed scan + EOI)
__global__ void __launch_bounds__(kEncThreads) jpeg_enc_size_kernel(const EncGeom G, int32_t header_len, const uint64_t* __restrict__ cta_off,
                                                                    const uint64_t* __restrict__ img_bits, const uint32_t* __restrict__ head,
                                                                    const uint32_t* __restrict__ tail, uint32_t* region,
                                                                    uint64_t* __restrict__ size) {
    using Reduce = cub::BlockReduce<uint32_t, kEncThreads>;
    __shared__ typename Reduce::TempStorage tmp;
    const int64_t i = blockIdx.x, base = i * G.ctas;
    uint32_t* reg = region + i * G.region_words;
    const uint64_t nbytes = (img_bits[i] + 7) >> 3;
    for (int c = 1 + threadIdx.x; c < G.ctas; c += kEncThreads) {
        const uint64_t s = cta_off[base + c];
        if (s & 31) reg[s >> 5] = tail[base + c - 1] | head[base + c];
    }
    if (threadIdx.x == 0 && (nbytes & 3)) reg[nbytes >> 2] = tail[base + G.ctas - 1];
    __syncthreads();
    uint32_t ff = 0;
    for (uint64_t w = threadIdx.x; w < (nbytes + 3) >> 2; w += kEncThreads) {
        ff += je_ff_bytes(reg[w], nbytes - 4 * w);
    }
    ff = Reduce(tmp).Sum(ff);
    if (threadIdx.x == 0) size[i] = (uint64_t)header_len + nbytes + ff + 2;
}

// out_off = exclusive scan of the file sizes (n + 1 entries); status = 1 when they exceed the arena
__global__ void __launch_bounds__(kEncThreads) jpeg_enc_outoff_kernel(int32_t n, const uint64_t* __restrict__ size, uint64_t out_bytes,
                                                                      int64_t* __restrict__ out_off, int32_t* __restrict__ status) {
    using Scan = cub::BlockScan<uint64_t, kEncThreads>;
    __shared__ typename Scan::TempStorage tmp;
    uint64_t running = 0;
    for (int i0 = 0; i0 < n; i0 += kEncThreads) {
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

// per image: header, the scan with a 0x00 stuffed after every 0xFF, EOI.  Writes nothing when the batch does not fit the arena.
// Warp w owns a contiguous run of whole 32-word rows of the scan; per row, lane l reads word l (coalesced), and a warp scan of the
// lanes' stuffed lengths places their bytes side by side, so a warp's stores also cover one contiguous stretch.
constexpr int kPlaceThreads = 512, kPlaceWarps = kPlaceThreads / 32;
__global__ void __launch_bounds__(kPlaceThreads) jpeg_enc_place_kernel(const EncGeom G, const EncHeader Hd, int32_t n,
                                                                       const uint64_t* __restrict__ img_bits, const uint32_t* __restrict__ region,
                                                                       uint64_t out_bytes, const int64_t* __restrict__ out_off,
                                                                       uint8_t* __restrict__ out) {
    __shared__ uint32_t warp_ff[kPlaceWarps];
    if ((uint64_t)out_off[n] > out_bytes) return;
    const int64_t i = blockIdx.x;
    const uint64_t o = (uint64_t)out_off[i], nbytes = (img_bits[i] + 7) >> 3, fsize = (uint64_t)out_off[i + 1] - o;
    const uint32_t* __restrict__ scan = region + i * G.region_words;  // bytes in stream order
    uint8_t* __restrict__ dst = out + o;
    for (int t = threadIdx.x; t < Hd.len; t += kPlaceThreads) dst[t] = Hd.b[t];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t nwords = (nbytes + 3) >> 2, rows = (nwords + 31) >> 5, per_warp = 32 * ((rows + kPlaceWarps - 1) / kPlaceWarps);
    const uint64_t w0 = min(nwords, (uint64_t)warp * per_warp), w1 = min(nwords, w0 + per_warp);
    uint32_t ff = 0;
    for (uint64_t w = w0 + lane; w < w1; w += 32) ff += je_ff_bytes(scan[w], nbytes - 4 * w);
    ff = __reduce_add_sync(0xffffffffu, ff);
    if (lane == 0) warp_ff[warp] = ff;
    __syncthreads();
    uint64_t q = (uint64_t)Hd.len + 4 * w0;  // where this warp's first byte goes
    for (int k = 0; k < warp; ++k) q += warp_ff[k];
    for (uint64_t wb = w0; wb < w1; wb += 32) {
        const uint64_t w = wb + lane;
        uint32_t v = 0, nb = 0, len = 0;
        if (w < w1) {
            v = scan[w];
            nb = nbytes - 4 * w >= 4 ? 4u : (uint32_t)(nbytes - 4 * w);
            len = nb + je_ff_bytes(v, nbytes - 4 * w);
        }
        uint32_t incl = len;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += y;
        }
        uint64_t p = q + incl - len;
        for (uint32_t b = 0; b < nb; ++b) {
            const uint8_t x = (uint8_t)(v >> (8 * b));
            dst[p++] = x;
            if (x == 0xff) dst[p++] = 0;
        }
        q += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (threadIdx.x == 0) {
        dst[fsize - 2] = 0xff;
        dst[fsize - 1] = 0xd9;
    }
}

// ------------------------------------------------------------------------------------------------ host
// Annex K.3 tables (jcparam.c std_huff_tables): DC luma, AC luma, DC chroma, AC chroma
static const uint8_t kBitsDc0[16] = {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0};
static const uint8_t kBitsDc1[16] = {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0};
static const uint8_t kValsDc[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
static const uint8_t kBitsAc0[16] = {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d};
static const uint8_t kValsAc0[162] = {
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14, 0x32, 0x81, 0x91, 0xa1,
    0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26,
    0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56,
    0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85,
    0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa,
    0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6,
    0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9,
    0xfa};
static const uint8_t kBitsAc1[16] = {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77};
static const uint8_t kValsAc1[162] = {
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32, 0x81, 0x08, 0x14, 0x42,
    0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19,
    0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55,
    0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83,
    0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8,
    0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4,
    0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9,
    0xfa};
// Annex K.1 / K.2, natural order
static const uint8_t kStdLuma[64] = {16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22, 29,
                                     51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, 49, 64, 78, 87, 103, 121,
                                     120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
static const uint8_t kStdChroma[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99,
                                       99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                                       99, 99, 99, 99, 99, 99, 99, 99, 99, 99};

// Annex C: code of every symbol of a (bits, vals) table, as (length << 16) | code
static void je_codes(const uint8_t bits[16], const uint8_t* vals, uint32_t* table) {
    uint32_t code = 0;
    int k = 0;
    for (int l = 1; l <= 16; ++l) {
        for (int i = 0; i < bits[l - 1]; ++i) table[vals[k++]] = ((uint32_t)l << 16) | code++;
        code <<= 1;
    }
}

// jcparam.c jpeg_set_quality(q, force_baseline = TRUE)
static void je_qtable(const uint8_t std[64], int q, uint8_t out[64]) {
    const int scale = q < 50 ? 5000 / q : 200 - 2 * q;
    for (int i = 0; i < 64; ++i) {
        const int v = (std[i] * scale + 50) / 100;
        out[i] = (uint8_t)(v < 1 ? 1 : (v > 255 ? 255 : v));
    }
}

// SOI, APP0 (JFIF 1.01, no density, no thumbnail), DQT x2, SOF0 (4:2:0), DHT x4, SOS -- what Pillow writes for an RGB array
static int je_header(int h, int w, const uint8_t qt[2][64], uint8_t* b) {
    int n = 0;
    auto put = [&](std::initializer_list<int> v) { for (int x : v) b[n++] = (uint8_t)x; };
    put({0xff, 0xd8, 0xff, 0xe0, 0x00, 0x10, 'J', 'F', 'I', 'F', 0, 1, 1, 0, 0, 1, 0, 1, 0, 0});
    for (int t = 0; t < 2; ++t) {
        put({0xff, 0xdb, 0x00, 0x43, t});
        for (int k = 0; k < 64; ++k) b[n++] = qt[t][kZigzag[k]];
    }
    put({0xff, 0xc0, 0x00, 0x11, 8, h >> 8, h & 255, w >> 8, w & 255, 3, 1, 0x22, 0, 2, 0x11, 1, 3, 0x11, 1});
    const uint8_t* bits[4] = {kBitsDc0, kBitsAc0, kBitsDc1, kBitsAc1};
    const uint8_t* vals[4] = {kValsDc, kValsAc0, kValsDc, kValsAc1};
    const int cls[4] = {0x00, 0x10, 0x01, 0x11};
    for (int t = 0; t < 4; ++t) {
        int nv = 0;
        for (int l = 0; l < 16; ++l) nv += bits[t][l];
        const int len = 2 + 1 + 16 + nv;
        put({0xff, 0xc4, len >> 8, len & 255, cls[t]});
        for (int l = 0; l < 16; ++l) b[n++] = bits[t][l];
        for (int v = 0; v < nv; ++v) b[n++] = vals[t][v];
    }
    put({0xff, 0xda, 0x00, 0x0c, 3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0});
    return n;
}

struct JeLayout {
    EncGeom G;
    int64_t n_ctas;
    size_t rec, cta_off, head, tail, img_bits, size, region, total;
};

static bool je_mul(size_t a, size_t b, size_t* out) {
    if (a && b > SIZE_MAX / a) return false;
    *out = a * b;
    return true;
}

// false when the batch is too large for one call (CTA count beyond the grid limit or a workspace beyond size_t)
static bool je_layout(int32_t n, int32_t h, int32_t w, JeLayout* L) {
    EncGeom& G = L->G;
    G.width = w; G.height = h;
    G.mcus_x = (w + 15) / 16;
    const int mcus_y = (h + 15) / 16;
    G.mcus = G.mcus_x * mcus_y;
    G.blocks_x = (w + 7) / 8; G.blocks_y = (h + 7) / 8;
    G.chroma_h = (h + 1) / 2;
    G.ctas = (G.mcus + kEncMcus - 1) / kEncMcus;
    G.img_bytes = (int64_t)h * w * 3;
    const uint64_t bound_bits = (uint64_t)G.mcus * 6 * kMaxBlockBits + 8;
    G.region_words = (int64_t)(((bound_bits + 31) / 32 + 1 + 3) & ~3ull);
    L->n_ctas = (int64_t)n * G.ctas;
    if (L->n_ctas > 0x7fffffff) return false;
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t N = (size_t)n, C = (size_t)L->n_ctas;
    size_t o = 0, region_bytes;
    L->rec = o; o = al(o + C * sizeof(EncCta));
    L->cta_off = o; o = al(o + C * 8);
    L->head = o; o = al(o + C * 4);
    L->tail = o; o = al(o + C * 4);
    L->img_bits = o; o = al(o + N * 8);
    L->size = o; o = al(o + N * 8);
    L->region = o;
    if (!je_mul(N, (size_t)G.region_words * 4, &region_bytes) || region_bytes > SIZE_MAX - o - 256) return false;
    L->total = al(o + region_bytes) > 256 ? al(o + region_bytes) : 256;  // never 0, which reports arguments out of range
    return true;
}

static bool je_dims_ok(int32_t n, int32_t h, int32_t w) { return n >= 0 && h >= 1 && h <= 65535 && w >= 1 && w <= 65535; }

}  // namespace msc

extern "C" {

size_t msc_jpeg_encode_workspace_bytes(int32_t n_images, int32_t height, int32_t width, size_t out_bytes) {
    using namespace msc;
    (void)out_bytes;  // the scan is packed at its worst-case length before its stuffed size is known: the arena does not change the need
    JeLayout L;
    if (!je_dims_ok(n_images, height, width) || !je_layout(n_images, height, width, &L)) return 0;
    return L.total;
}

int msc_jpeg_encode_batch(int32_t n_images, int32_t height, int32_t width, int32_t quality, const uint8_t* rgb, uint8_t* out, size_t out_bytes,
                          int64_t* out_off, int32_t* status, void* workspace, size_t workspace_bytes, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(quality >= 1 && quality <= 100, "msc_jpeg_encode_batch: quality must be in 1..100 (got %d)", (int)quality);
    MSC_REQUIRE(height >= 1 && height <= 65535 && width >= 1 && width <= 65535,
                "msc_jpeg_encode_batch: height and width must be in 1..65535 (got %d x %d)", (int)height, (int)width);
    MSC_REQUIRE(n_images >= 0, "msc_jpeg_encode_batch: negative n_images");
    if (n_images == 0) return MSC_OK;
    MSC_REQUIRE(rgb && out && out_off && status && workspace, "msc_jpeg_encode_batch: a pointer argument is NULL");
    MSC_REQUIRE(((uintptr_t)workspace & 255) == 0, "msc_jpeg_encode_batch: workspace must be 256-byte aligned");
    JeLayout L;
    MSC_REQUIRE(je_layout(n_images, height, width, &L), "msc_jpeg_encode_batch: %d images of %d x %d are too many for one call",
                (int)n_images, (int)height, (int)width);
    MSC_REQUIRE(workspace_bytes >= L.total, "msc_jpeg_encode_batch: workspace too small: need %zu bytes, got %zu", L.total, workspace_bytes);

    EncTables T;
    uint8_t qt[2][64];
    je_qtable(kStdLuma, quality, qt[0]);
    je_qtable(kStdChroma, quality, qt[1]);
    for (int t = 0; t < 2; ++t)
        for (int i = 0; i < 64; ++i) T.div[t][i] = (uint16_t)(8 * qt[t][i]);
    memcpy(T.zz, kZigzag, 64);
    memset(T.dc, 0, sizeof(T.dc));
    memset(T.ac, 0, sizeof(T.ac));
    je_codes(kBitsDc0, kValsDc, T.dc[0]);
    je_codes(kBitsDc1, kValsDc, T.dc[1]);
    je_codes(kBitsAc0, kValsAc0, T.ac[0]);
    je_codes(kBitsAc1, kValsAc1, T.ac[1]);
    EncHeader Hd;
    Hd.len = je_header(height, width, qt, Hd.b);

    unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
    EncCta* rec = (EncCta*)(ws + L.rec);
    uint64_t* cta_off = (uint64_t*)(ws + L.cta_off);
    uint32_t* head = (uint32_t*)(ws + L.head);
    uint32_t* tail = (uint32_t*)(ws + L.tail);
    uint64_t* img_bits = (uint64_t*)(ws + L.img_bits);
    uint64_t* size = (uint64_t*)(ws + L.size);
    uint32_t* region = (uint32_t*)(ws + L.region);
    cudaStream_t stream = (cudaStream_t)stream_v;
    const EncGeom& G = L.G;
    const unsigned grid = (unsigned)L.n_ctas;
    const size_t pack_smem = (size_t)kCtaWords * 4;
    MSC_CUDA(cudaFuncSetAttribute(jpeg_enc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pack_smem));

    jpeg_enc_kernel<false><<<grid, kEncThreads, 0, stream>>>(G, T, rgb, rec, nullptr, nullptr, nullptr, nullptr);
    jpeg_enc_offsets_kernel<<<(unsigned)n_images, kEncThreads, 0, stream>>>(G, T, rec, cta_off, img_bits);
    jpeg_enc_kernel<true><<<grid, kEncThreads, pack_smem, stream>>>(G, T, rgb, rec, cta_off, region, head, tail);
    jpeg_enc_size_kernel<<<(unsigned)n_images, kEncThreads, 0, stream>>>(G, Hd.len, cta_off, img_bits, head, tail, region, size);
    jpeg_enc_outoff_kernel<<<1, kEncThreads, 0, stream>>>(n_images, size, (uint64_t)out_bytes, out_off, status);
    jpeg_enc_place_kernel<<<(unsigned)n_images, kPlaceThreads, 0, stream>>>(G, Hd, n_images, img_bits, region, (uint64_t)out_bytes, out_off, out);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

}  // extern "C"
