// jpeg.cu -- camera-image decode for the on-disk step (SURVEY.md section 8(f) rank 3): NuScenesLoader._load_camera
// (nuscenes_loader.py:136-144) is `np.array(Image.open(path))`, i.e. libjpeg(-turbo)'s default decompression.  This file restates that
// pipeline so that the result is BIT-IDENTICAL to it: the entropy (Huffman) decode -- inherently sequential per image -- runs on the host,
// one image per thread; everything per-sample runs on the device: dequantisation + the "slow integer" inverse DCT (jidctint.c),
// "fancy" (triangle-filter) chroma upsampling for 4:2:2 / 4:2:0 (jdsample.c), and the fixed-point YCbCr -> RGB conversion (jdcolor.c).
// All three are integer algorithms with fixed rounding, so equality with PIL is a matter of following them to the letter; the constants
// and rounding terms below are the ones the JPEG reference implementation publishes.
//
// Supported: baseline / extended-sequential Huffman JPEG, 8 bits, 1 component (grayscale) or 3 components (JFIF YCbCr) in one
// interleaved scan, sampling 4:4:4 / 4:2:2 (h2v1) / 4:2:0 (h2v2), restart intervals.  Progressive, arithmetic-coded, CMYK / Adobe-RGB
// files and other sampling layouts return MSC_ERR_UNSUPPORTED (nuScenes camera frames are baseline 4:2:0 JFIF).
#include <vector>

#include "jpeg_common.cuh"
#include "msc_common.cuh"

namespace msc {

// ------------------------------------------------------------------------------------------------ host: parse + Huffman decode
struct HuffTable {
    bool present = false;
    uint8_t bits[17] = {0};
    uint8_t vals[256] = {0};
    // decoding tables (JPEG Annex F.2.2.3): per code length the largest code, and the index of the first symbol of that length
    int32_t maxcode[18];
    int32_t valptr[17];
    uint16_t look[512];  // 9-bit lookahead: (length << 8) | symbol, 0 = longer than 9 bits
    void build() {
        int32_t code = 0, k = 0;
        int32_t huffcode[257];
        uint8_t huffsize[257];
        int p = 0;
        for (int l = 1; l <= 16; ++l)
            for (int i = 0; i < bits[l]; ++i) huffsize[p++] = (uint8_t)l;
        huffsize[p] = 0;
        int si = huffsize[0];
        p = 0;
        while (huffsize[p]) {
            while (huffsize[p] == si) { huffcode[p++] = code; ++code; }
            code <<= 1;
            ++si;
        }
        p = 0;
        for (int l = 1; l <= 16; ++l) {
            if (bits[l]) {
                valptr[l] = p - huffcode[p];
                p += bits[l];
                maxcode[l] = huffcode[p - 1];
            } else {
                maxcode[l] = -1;
            }
        }
        maxcode[17] = 0xFFFFF;
        memset(look, 0, sizeof(look));
        p = 0;
        for (int l = 1; l <= 9; ++l)
            for (int i = 0; i < bits[l]; ++i, ++p) {
                const int32_t first = huffcode[p] << (9 - l);
                for (int c = 0; c < (1 << (9 - l)); ++c) look[first + c] = (uint16_t)((l << 8) | vals[p]);
            }
        (void)k;
    }
};

struct BitReader {
    const uint8_t* p;
    const uint8_t* end;
    uint64_t acc = 0;
    int n = 0;         // valid bits in acc (msb-aligned at bit n-1)
    bool hit_marker = false;
    void fill() {
        while (n <= 56) {
            uint32_t b = 0;
            if (!hit_marker && p < end) {
                b = *p;
                if (b == 0xFF) {
                    if (p + 1 < end && p[1] == 0x00) { p += 2; }
                    else { hit_marker = true; b = 0; }  // a marker: feed zeros (the caller stops at the MCU count / restart boundary)
                } else {
                    ++p;
                }
            }
            acc = (acc << 8) | b;
            n += 8;
        }
    }
    inline uint32_t peek(int k) { if (n < k) fill(); return (uint32_t)((acc >> (n - k)) & ((1u << k) - 1u)); }
    inline void skip(int k) { n -= k; }
    inline int32_t receive_extend(int s) {
        if (s == 0) return 0;
        const int32_t v = (int32_t)peek(s);
        skip(s);
        return v < (1 << (s - 1)) ? v - (1 << s) + 1 : v;
    }
    inline int decode(const HuffTable& t) {
        if (n < 16) fill();
        const uint32_t l9 = (uint32_t)((acc >> (n - 9)) & 0x1ff);
        const uint16_t e = t.look[l9];
        if (e) { n -= e >> 8; return e & 0xff; }
        int32_t code = (int32_t)((acc >> (n - 10)) & 0x3ff);
        int l = 10;
        while (l <= 16 && code > t.maxcode[l]) {
            ++l;
            code = (int32_t)((acc >> (n - l)) & ((1u << l) - 1u));
        }
        if (l > 16) return -1;
        n -= l;
        return t.vals[(code + t.valptr[l]) & 0xff];
    }
    void reset_to(const uint8_t* q) { p = q; acc = 0; n = 0; hit_marker = false; }
};

struct ParsedJpeg {
    msc_jpeg_desc d;
    HuffTable dc[4], ac[4];
    int td[3] = {0, 0, 0}, ta[3] = {0, 0, 0};
    int restart_interval = 0;
    const uint8_t* scan = nullptr;
    const uint8_t* end = nullptr;
};

static inline uint32_t be16(const uint8_t* p) { return ((uint32_t)p[0] << 8) | p[1]; }

// headers up to the start of the (single) scan; returns an msc_status
static int parse_headers(const uint8_t* data, size_t nbytes, ParsedJpeg* J) {
    memset(&J->d, 0, sizeof(J->d));
    if (nbytes < 4 || data[0] != 0xFF || data[1] != 0xD8) { set_error("not a JPEG stream (no SOI)"); return MSC_ERR_BAD_ARGUMENT; }
    const uint8_t* p = data + 2;
    const uint8_t* end = data + nbytes;
    uint16_t qt[4][64];
    bool have_qt[4] = {false, false, false, false};
    int comp_id[3] = {0, 0, 0}, comp_tq[3] = {0, 0, 0};
    bool have_sof = false;
    while (p + 4 <= end) {
        if (p[0] != 0xFF) { set_error("JPEG: marker expected"); return MSC_ERR_BAD_ARGUMENT; }
        while (p < end && *p == 0xFF) ++p;  // fill bytes
        if (p >= end) break;
        const uint8_t m = *p++;
        if (m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) continue;
        if (m == 0xD9) break;
        if (p + 2 > end) break;
        const uint32_t len = be16(p);
        if (len < 2 || p + len > end) { set_error("JPEG: truncated segment"); return MSC_ERR_BAD_ARGUMENT; }
        const uint8_t* s = p + 2;
        const uint8_t* se = p + len;
        if (m == 0xDB) {  // DQT
            while (s < se) {
                const int pq = *s >> 4, tq = *s & 15;
                ++s;
                if (tq > 3 || s + (pq ? 128 : 64) > se) { set_error("JPEG: bad DQT"); return MSC_ERR_BAD_ARGUMENT; }
                for (int i = 0; i < 64; ++i) {
                    const uint16_t v = pq ? (uint16_t)be16(s + 2 * i) : s[i];
                    qt[tq][kZigzag[i]] = v;
                }
                s += pq ? 128 : 64;
                have_qt[tq] = true;
            }
        } else if (m == 0xC4) {  // DHT
            while (s < se) {
                const int tc = *s >> 4, th = *s & 15;
                ++s;
                if (tc > 1 || th > 3 || s + 16 > se) { set_error("JPEG: bad DHT"); return MSC_ERR_BAD_ARGUMENT; }
                HuffTable& t = tc ? J->ac[th] : J->dc[th];
                int total = 0;
                t.bits[0] = 0;
                for (int i = 1; i <= 16; ++i) { t.bits[i] = s[i - 1]; total += s[i - 1]; }
                s += 16;
                if (total > 256 || s + total > se) { set_error("JPEG: bad DHT"); return MSC_ERR_BAD_ARGUMENT; }
                memcpy(t.vals, s, (size_t)total);
                s += total;
                t.present = true;
                t.build();
            }
        } else if (m == 0xC0 || m == 0xC1) {  // SOF0 / SOF1: sequential Huffman
            if (len < 8) { set_error("JPEG: bad SOF"); return MSC_ERR_BAD_ARGUMENT; }
            if (s[0] != 8) { set_error("JPEG: %d-bit samples are not supported", (int)s[0]); return MSC_ERR_UNSUPPORTED; }
            J->d.height = (int32_t)be16(s + 1);
            J->d.width = (int32_t)be16(s + 3);
            J->d.n_comp = s[5];
            if (J->d.n_comp != 1 && J->d.n_comp != 3) { set_error("JPEG: %d components are not supported", J->d.n_comp); return MSC_ERR_UNSUPPORTED; }
            if (len < 8u + 3u * (uint32_t)J->d.n_comp || J->d.width <= 0 || J->d.height <= 0) { set_error("JPEG: bad SOF"); return MSC_ERR_BAD_ARGUMENT; }
            for (int c = 0; c < J->d.n_comp; ++c) {
                comp_id[c] = s[6 + 3 * c];
                J->d.comp[c].h = s[7 + 3 * c] >> 4;
                J->d.comp[c].v = s[7 + 3 * c] & 15;
                comp_tq[c] = s[8 + 3 * c] & 3;
            }
            have_sof = true;
        } else if (m == 0xC2 || (m >= 0xC5 && m <= 0xCF && m != 0xC8 && m != 0xCC)) {
            set_error("JPEG: progressive / lossless / arithmetic-coded files are not supported (SOF marker 0x%02x)", m);
            return MSC_ERR_UNSUPPORTED;
        } else if (m == 0xDD) {  // DRI
            if (len >= 4) J->restart_interval = (int)be16(s);
        } else if (m == 0xEE) {  // Adobe: a colour transform other than YCbCr is not handled
            if (len >= 14 && !memcmp(s, "Adobe", 5) && s[11] != 1 && J->d.n_comp == 3) { set_error("JPEG: Adobe colour transform %d is not supported", (int)s[11]); return MSC_ERR_UNSUPPORTED; }
        } else if (m == 0xDA) {  // SOS
            if (!have_sof) { set_error("JPEG: SOS before SOF"); return MSC_ERR_BAD_ARGUMENT; }
            const int ns = s[0];
            if (ns != J->d.n_comp) { set_error("JPEG: non-interleaved scans are not supported"); return MSC_ERR_UNSUPPORTED; }
            for (int i = 0; i < ns; ++i) {
                int c = -1;
                for (int k = 0; k < J->d.n_comp; ++k)
                    if (comp_id[k] == s[1 + 2 * i]) c = k;
                if (c != i) { set_error("JPEG: unexpected component order in SOS"); return MSC_ERR_UNSUPPORTED; }
                J->td[c] = s[2 + 2 * i] >> 4;
                J->ta[c] = s[2 + 2 * i] & 15;
                if (J->td[c] > 3 || J->ta[c] > 3 || !J->dc[J->td[c]].present || !J->ac[J->ta[c]].present) { set_error("JPEG: missing Huffman table"); return MSC_ERR_BAD_ARGUMENT; }
            }
            J->scan = se;
            J->end = end;
            break;
        }
        p += len;
    }
    if (!have_sof || !J->scan) { set_error("JPEG: no scan found"); return MSC_ERR_BAD_ARGUMENT; }
    msc_jpeg_desc& d = J->d;
    d.hmax = d.vmax = 1;
    for (int c = 0; c < d.n_comp; ++c) {
        if (d.comp[c].h < 1 || d.comp[c].v < 1) { set_error("JPEG: bad sampling factors"); return MSC_ERR_BAD_ARGUMENT; }
        d.hmax = d.comp[c].h > d.hmax ? d.comp[c].h : d.hmax;
        d.vmax = d.comp[c].v > d.vmax ? d.comp[c].v : d.vmax;
    }
    if (d.n_comp == 1) { d.comp[0].h = d.comp[0].v = 1; d.hmax = d.vmax = 1; }  // a single component is never subsampled (its factors are ignored)
    if (d.n_comp == 3) {
        const bool luma_ok = (d.comp[0].h == d.hmax && d.comp[0].v == d.vmax);
        const bool chroma_ok = d.comp[1].h == 1 && d.comp[1].v == 1 && d.comp[2].h == 1 && d.comp[2].v == 1;
        const bool layout_ok = (d.hmax == 1 && d.vmax == 1) || (d.hmax == 2 && d.vmax == 1) || (d.hmax == 2 && d.vmax == 2);
        if (!luma_ok || !chroma_ok || !layout_ok) { set_error("JPEG: sampling layout %dx%d/%dx%d/%dx%d is not supported", d.comp[0].h, d.comp[0].v, d.comp[1].h, d.comp[1].v, d.comp[2].h, d.comp[2].v); return MSC_ERR_UNSUPPORTED; }
    }
    d.mcus_x = (d.width + 8 * d.hmax - 1) / (8 * d.hmax);
    d.mcus_y = (d.height + 8 * d.vmax - 1) / (8 * d.vmax);
    size_t coef = 0, plane = 0;
    for (int c = 0; c < d.n_comp; ++c) {
        msc_jpeg_comp& k = d.comp[c];
        if (!have_qt[comp_tq[c]]) { set_error("JPEG: missing quantisation table"); return MSC_ERR_BAD_ARGUMENT; }
        memcpy(k.qt, qt[comp_tq[c]], sizeof(k.qt));
        k.blocks_x = d.mcus_x * k.h;
        k.blocks_y = d.mcus_y * k.v;
        k.ds_w = (d.width * k.h + d.hmax - 1) / d.hmax;
        k.ds_h = (d.height * k.v + d.vmax - 1) / d.vmax;
        k.coef_off = (int64_t)coef;
        k.plane_off = (int64_t)plane;
        coef += (size_t)k.blocks_x * k.blocks_y * 64;
        plane += (size_t)k.blocks_x * k.blocks_y * 64;
    }
    d.coef_elems = (int64_t)coef;
    d.plane_bytes = (int64_t)plane;
    return MSC_OK;
}

static int entropy_decode(ParsedJpeg& J, int16_t* coef) {
    const msc_jpeg_desc& d = J.d;
    memset(coef, 0, (size_t)d.coef_elems * sizeof(int16_t));
    BitReader br;
    br.p = J.scan;
    br.end = J.end;
    int32_t pred[3] = {0, 0, 0};
    int restart_left = J.restart_interval;
    int next_rst = 0;
    for (int my = 0; my < d.mcus_y; ++my) {
        for (int mx = 0; mx < d.mcus_x; ++mx) {
            if (J.restart_interval && restart_left == 0) {
                // byte-align, find the RSTn marker, reset the predictors
                const uint8_t* q = br.p;
                while (q + 1 < J.end && !(q[0] == 0xFF && q[1] >= 0xD0 && q[1] <= 0xD7)) ++q;
                if (q + 1 >= J.end) { set_error("JPEG: restart marker missing"); return MSC_ERR_BAD_ARGUMENT; }
                (void)next_rst;
                br.reset_to(q + 2);
                pred[0] = pred[1] = pred[2] = 0;
                restart_left = J.restart_interval;
            }
            for (int c = 0; c < d.n_comp; ++c) {
                const msc_jpeg_comp& k = d.comp[c];
                const HuffTable& dct = J.dc[J.td[c]];
                const HuffTable& act = J.ac[J.ta[c]];
                for (int by = 0; by < k.v; ++by)
                    for (int bx = 0; bx < k.h; ++bx) {
                        int16_t* blk = coef + k.coef_off + ((size_t)(my * k.v + by) * k.blocks_x + (size_t)(mx * k.h + bx)) * 64;
                        int s = br.decode(dct);
                        if (s < 0 || s > 15) { set_error("JPEG: corrupt DC code"); return MSC_ERR_BAD_ARGUMENT; }
                        pred[c] += br.receive_extend(s);
                        blk[0] = (int16_t)pred[c];
                        for (int kk = 1; kk < 64;) {
                            const int rs = br.decode(act);
                            if (rs < 0) { set_error("JPEG: corrupt AC code"); return MSC_ERR_BAD_ARGUMENT; }
                            const int r = rs >> 4, sz = rs & 15;
                            if (sz == 0) {
                                if (r == 15) { kk += 16; continue; }
                                break;  // EOB
                            }
                            kk += r;
                            if (kk > 63) { set_error("JPEG: corrupt AC run"); return MSC_ERR_BAD_ARGUMENT; }
                            blk[kZigzag[kk]] = (int16_t)br.receive_extend(sz);
                            ++kk;
                        }
                    }
            }
            if (J.restart_interval) --restart_left;
        }
    }
    return MSC_OK;
}

// ------------------------------------------------------------------------------------------------ device: IDCT, upsampling, colour
struct IdctParams {
    const int16_t* coef;
    uint8_t* plane;
    int blocks_x, n_blocks;
    uint16_t qt[64];
};

// 8 threads per 8x8 block: thread j does column j of pass 1 and row j of pass 2; 32 blocks per CTA
__global__ void __launch_bounds__(256) jpeg_idct_kernel(const IdctParams P) {
    __shared__ int ws[32][64 + 1];
    const int lb = threadIdx.x >> 3, j = threadIdx.x & 7;
    const int b = blockIdx.x * 32 + lb;
    const bool live = b < P.n_blocks;
    int o[8];
    if (live) {  // pass 1: columns, dequantised input, results scaled up by 2^PASS1_BITS
        const int16_t* c = P.coef + (size_t)b * 64 + j;
        jd_butterfly(c[0] * (int)P.qt[j], c[8] * (int)P.qt[8 + j], c[16] * (int)P.qt[16 + j], c[24] * (int)P.qt[24 + j], c[32] * (int)P.qt[32 + j],
                     c[40] * (int)P.qt[40 + j], c[48] * (int)P.qt[48 + j], c[56] * (int)P.qt[56 + j], o, 13 - 2);
#pragma unroll
        for (int r = 0; r < 8; ++r) ws[lb][r * 8 + j] = o[r];
    }
    __syncthreads();
    if (live) {  // pass 2: rows, descale by CONST_BITS + PASS1_BITS + 3, level shift + range limit
        const int* w = &ws[lb][j * 8];
        jd_butterfly(w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], o, 13 + 2 + 3);
        const int bx = b % P.blocks_x, by = b / P.blocks_x;
        uint8_t* dst = P.plane + ((size_t)(by * 8 + j) * P.blocks_x + bx) * 8;
        uint2 pk;
        pk.x = (uint32_t)jd_idct_limit(o[0]) | ((uint32_t)jd_idct_limit(o[1]) << 8) | ((uint32_t)jd_idct_limit(o[2]) << 16) | ((uint32_t)jd_idct_limit(o[3]) << 24);
        pk.y = (uint32_t)jd_idct_limit(o[4]) | ((uint32_t)jd_idct_limit(o[5]) << 8) | ((uint32_t)jd_idct_limit(o[6]) << 16) | ((uint32_t)jd_idct_limit(o[7]) << 24);
        *reinterpret_cast<uint2*>(dst) = pk;
    }
}

struct ColorParams {
    const uint8_t* y;
    const uint8_t* cb;
    const uint8_t* cr;
    uint8_t* out;
    int width, height, n_comp;
    int y_stride, c_stride;  // plane row strides (blocks_x * 8)
    int c_w, c_h;            // downsampled_width / height of the chroma planes
    int hsub, vsub;          // 1 or 2
};

__global__ void __launch_bounds__(256) jpeg_color_kernel(const ColorParams P) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= P.width || y >= P.height) return;
    const int Y = P.y[(size_t)y * P.y_stride + x];
    if (P.n_comp == 1) {
        P.out[(size_t)y * P.width + x] = (uint8_t)Y;
        return;
    }
    const int cb = jd_chroma(P.cb, P.c_stride, P.c_w, P.c_h, P.hsub, P.vsub, x, y) - 128;
    const int cr = jd_chroma(P.cr, P.c_stride, P.c_w, P.c_h, P.hsub, P.vsub, x, y) - 128;
    jd_ycc_rgb(Y, cb, cr, P.out + ((size_t)y * P.width + x) * 3);
}

}  // namespace msc

extern "C" {

int msc_jpeg_info(const uint8_t* jpeg_host, size_t nbytes, msc_jpeg_desc* desc) {
    using namespace msc;
    MSC_REQUIRE(jpeg_host && desc, "null argument");
    ParsedJpeg J;
    const int rc = parse_headers(jpeg_host, nbytes, &J);
    if (rc != MSC_OK) return rc;
    *desc = J.d;
    return MSC_OK;
}

int msc_jpeg_entropy_decode_host(const uint8_t* jpeg_host, size_t nbytes, const msc_jpeg_desc* desc, int16_t* coef_host) {
    using namespace msc;
    MSC_REQUIRE(jpeg_host && desc && coef_host, "null argument");
    ParsedJpeg J;
    int rc = parse_headers(jpeg_host, nbytes, &J);
    if (rc != MSC_OK) return rc;
    MSC_REQUIRE(J.d.coef_elems == desc->coef_elems && J.d.width == desc->width && J.d.height == desc->height, "descriptor does not belong to this stream");
    return entropy_decode(J, coef_host);
}

int msc_jpeg_decode_plan(const uint8_t* jpeg_host, size_t nbytes, msc_jpeg_plan* plan) {
    using namespace msc;
    MSC_REQUIRE(jpeg_host && plan, "null argument");
    ParsedJpeg J;
    const int rc = parse_headers(jpeg_host, nbytes, &J);
    if (rc != MSC_OK) return rc;
    memset(plan, 0, sizeof(*plan));
    plan->desc = J.d;
    plan->scan_off = (int64_t)(J.scan - jpeg_host);
    plan->scan_bytes = (int64_t)(J.end - J.scan);
    plan->restart_interval = J.restart_interval;
    for (int c = 0; c < 3; ++c) { plan->td[c] = J.td[c]; plan->ta[c] = J.ta[c]; }
    for (int t = 0; t < 4; ++t) {
        const HuffTable* src[2] = {&J.dc[t], &J.ac[t]};
        msc_jpeg_huff* dst[2] = {&plan->dc[t], &plan->ac[t]};
        for (int k = 0; k < 2; ++k) {
            if (!src[k]->present) continue;
            memcpy(dst[k]->look, src[k]->look, sizeof(dst[k]->look));
            for (int l = 1; l <= 17; ++l) dst[k]->maxcode[l] = src[k]->maxcode[l];  // (entry 0 is unused; valptr is set for used lengths only)
            for (int l = 1; l <= 16; ++l) dst[k]->valptr[l] = src[k]->bits[l] ? src[k]->valptr[l] : 0;
            memcpy(dst[k]->vals, src[k]->vals, sizeof(dst[k]->vals));
        }
    }
    return MSC_OK;
}

int msc_jpeg_reconstruct(const msc_jpeg_desc* desc, const int16_t* coef, uint8_t* planes, uint8_t* out, void* stream_v) {
    using namespace msc;
    MSC_REQUIRE(desc && coef && planes && out, "null argument");
    MSC_REQUIRE(desc->n_comp == 1 || desc->n_comp == 3, "bad descriptor");
    cudaStream_t stream = (cudaStream_t)stream_v;
    for (int c = 0; c < desc->n_comp; ++c) {
        const msc_jpeg_comp& k = desc->comp[c];
        IdctParams P;
        P.coef = coef + k.coef_off;
        P.plane = planes + k.plane_off;
        P.blocks_x = k.blocks_x;
        P.n_blocks = k.blocks_x * k.blocks_y;
        memcpy(P.qt, k.qt, sizeof(P.qt));
        jpeg_idct_kernel<<<(P.n_blocks + 31) / 32, 256, 0, stream>>>(P);
        MSC_CUDA(cudaGetLastError());
    }
    ColorParams C;
    C.y = planes + desc->comp[0].plane_off;
    C.cb = desc->n_comp == 3 ? planes + desc->comp[1].plane_off : nullptr;
    C.cr = desc->n_comp == 3 ? planes + desc->comp[2].plane_off : nullptr;
    C.out = out;
    C.width = desc->width; C.height = desc->height; C.n_comp = desc->n_comp;
    C.y_stride = desc->comp[0].blocks_x * 8;
    C.c_stride = desc->n_comp == 3 ? desc->comp[1].blocks_x * 8 : 0;
    C.c_w = desc->n_comp == 3 ? desc->comp[1].ds_w : 0;
    C.c_h = desc->n_comp == 3 ? desc->comp[1].ds_h : 0;
    C.hsub = desc->hmax; C.vsub = desc->vmax;
    const dim3 grid((unsigned)((desc->width + 255) / 256), (unsigned)desc->height);
    jpeg_color_kernel<<<grid, 256, 0, stream>>>(C);
    MSC_CUDA(cudaGetLastError());
    return MSC_OK;
}

}  // extern "C"
