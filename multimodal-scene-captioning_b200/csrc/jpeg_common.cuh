// jpeg_common.cuh -- tables and integer arithmetic shared by the JPEG decoders (jpeg.cu, jpeg_decode.cu) and the encoder (jpeg_encode.cu).
#pragma once
#include <stdint.h>

namespace msc {

// zigzag position -> natural (row-major) index of an 8x8 block (ITU-T T.81 Figure A.6)
static const uint8_t kZigzag[64] = {0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
                                    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// ------------------------------------------------------------------------------------------------ decode: IDCT, upsampling, colour
// jidctint.c (jpeg_idct_islow): CONST_BITS 13, PASS1_BITS 2, the thirteen FIX() constants
__device__ __forceinline__ int jd_descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }
// IDCT_range_limit(cinfo)[x & RANGE_MASK] with the table of jdmaster.c:prepare_range_limit_table (centre 128, 10-bit wrap)
__device__ __forceinline__ uint8_t jd_idct_limit(int x) {
    const int v = x & 1023;
    return (uint8_t)(v < 128 ? 128 + v : v < 512 ? 255 : v < 896 ? 0 : v - 896);
}

// one 1-D pass of jpeg_idct_islow over d0..d7, descaled by `shift`
__device__ __forceinline__ void jd_butterfly(int d0, int d1, int d2, int d3, int d4, int d5, int d6, int d7, int o[8], int shift) {
    constexpr int C298 = 2446, C390 = 3196, C541 = 4433, C765 = 6270, C899 = 7373, C1175 = 9633, C1501 = 12299, C1847 = 15137, C1961 = 16069,
                  C2053 = 16819, C2562 = 20995, C3072 = 25172;
    // even part
    int z2 = d2, z3 = d6;
    int z1 = (z2 + z3) * C541;
    int tmp2 = z1 + z3 * (-C1847);
    int tmp3 = z1 + z2 * C765;
    z2 = d0; z3 = d4;
    int tmp0 = (z2 + z3) << 13;
    int tmp1 = (z2 - z3) << 13;
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    // odd part
    tmp0 = d7; tmp1 = d5; tmp2 = d3; tmp3 = d1;
    z1 = tmp0 + tmp3; z2 = tmp1 + tmp2; z3 = tmp0 + tmp2;
    int z4 = tmp1 + tmp3;
    const int z5 = (z3 + z4) * C1175;
    tmp0 *= C298; tmp1 *= C2053; tmp2 *= C3072; tmp3 *= C1501;
    z1 *= -C899; z2 *= -C2562; z3 *= -C1961; z4 *= -C390;
    z3 += z5; z4 += z5;
    tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
    o[0] = jd_descale(tmp10 + tmp3, shift); o[7] = jd_descale(tmp10 - tmp3, shift);
    o[1] = jd_descale(tmp11 + tmp2, shift); o[6] = jd_descale(tmp11 - tmp2, shift);
    o[2] = jd_descale(tmp12 + tmp1, shift); o[5] = jd_descale(tmp12 - tmp1, shift);
    o[3] = jd_descale(tmp13 + tmp0, shift); o[4] = jd_descale(tmp13 - tmp0, shift);
}

// one chroma sample at full resolution: jdsample.c fullsize / h2v1_fancy / h2v2_fancy (fancy only when downsampled_width > 2, else replication)
__device__ __forceinline__ int jd_chroma(const uint8_t* __restrict__ pl, int stride, int cw, int ch, int hsub, int vsub, int x, int y) {
    if (hsub == 1) return pl[(size_t)y * stride + x];
    const int ix = x >> 1;
    if (cw <= 2) return pl[(size_t)(vsub == 2 ? (y >> 1) : y) * stride + ix];  // h2v1_upsample / h2v2_upsample: plain replication
    if (vsub == 1) {  // h2v1_fancy_upsample: 3/4 nearer + 1/4 further, rounding 1 on the left sample of a pair, 2 on the right one
        const uint8_t* r = pl + (size_t)y * stride;
        const int v = r[ix];
        if ((x & 1) == 0) return ix == 0 ? v : (v * 3 + r[ix - 1] + 1) >> 2;
        return ix == cw - 1 ? v : (v * 3 + r[ix + 1] + 2) >> 2;
    }
    // h2v2_fancy_upsample: column sums 3 * nearer row + further row, then the same filter horizontally with rounding 8 / 7 and >> 4
    const int iy = y >> 1;
    int ny = (y & 1) ? iy + 1 : iy - 1;  // further row: above for the upper output row of a pair, below for the lower one
    ny = ny < 0 ? 0 : (ny > ch - 1 ? ch - 1 : ny);  // (context rows at the image edges duplicate the edge row, jdmainct.c)
    const uint8_t* r0 = pl + (size_t)iy * stride;
    const uint8_t* r1 = pl + (size_t)ny * stride;
    const int cs = r0[ix] * 3 + r1[ix];
    if ((x & 1) == 0) {
        if (ix == 0) return (cs * 4 + 8) >> 4;
        return (cs * 3 + (r0[ix - 1] * 3 + r1[ix - 1]) + 8) >> 4;
    }
    if (ix == cw - 1) return (cs * 4 + 7) >> 4;
    return (cs * 3 + (r0[ix + 1] * 3 + r1[ix + 1]) + 7) >> 4;
}

__device__ __forceinline__ uint8_t jd_clamp(int v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

// jdcolor.c build_ycc_rgb_table + ycc_rgb_convert: SCALEBITS 16, FIX(1.40200) = 91881, FIX(1.77200) = 116130, FIX(0.71414) = 46802,
// FIX(0.34414) = 22554, ONE_HALF = 32768.  cb, cr are centred (sample - 128).
__device__ __forceinline__ void jd_ycc_rgb(int Y, int cb, int cr, uint8_t* o) {
    const int r = Y + ((91881 * cr + 32768) >> 16);
    const int b = Y + ((116130 * cb + 32768) >> 16);
    const int g = Y + (((-22554) * cb + 32768 + (-46802) * cr) >> 16);
    o[0] = jd_clamp(r); o[1] = jd_clamp(g); o[2] = jd_clamp(b);
}

}  // namespace msc
