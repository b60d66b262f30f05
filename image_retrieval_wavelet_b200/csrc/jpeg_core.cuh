// JPEG decode core: the per-sample arithmetic of libjpeg 6.2 (libjpeg-turbo, as Pillow decodes with it), restated for
// the device.  Huffman decode step (8-bit lookahead table, then maxcode / valoffset), dequantisation + "islow" IDCT
// (jidctint.c: CONST_BITS 13, PASS1_BITS 2, the post-IDCT range-limit table), fancy upsampling (jdsample.c h2v1 / h2v2,
// edges at the component's downsampled size; replication when the chroma is at most 2 samples wide) and the fixed-point
// YCbCr -> RGB of jdcolor.c.
//
// Everything is __host__ __device__ and indexed per (subsequence / block / pixel), so that tests/ run the very code the
// kernels run on the CPU (csrc/hostsim.cpp).  Layouts of the records the worker builds (transforms/jpeg.py) and of the
// launch records the host builds (jpeg.cu) are defined here once.
#pragma once
#include <stddef.h>
#include <stdint.h>

#ifndef __CUDACC__
#define __host__
#define __device__
#define __forceinline__ inline
#endif

namespace b200 {

// Huffman record (1024 bytes): uint16 look[256] = (length << 8) | symbol of every code of <= 8 bits by its 8-bit prefix
// (0: longer code), int32 maxcode[18], int32 valoffset[18], uint8 huffval[256].
constexpr int kJpegHuffBytes = 1024, kJpegQuantBytes = 128;
constexpr int kJpegLookOff = 0, kJpegMaxcodeOff = 512, kJpegValoffOff = 584, kJpegHuffvalOff = 656;

// One device-decoded or raw image of a launch.
struct JpegImage {
    long long in_off, in_bytes;     // byte range of the clean entropy stream (or raw HWC pixels) in `in`
    long long out_off;              // byte offset of the HWC RGB output
    long long coef_off[3];          // int16 offset of each component's coefficient plane [bh][bw][64] in the workspace
    long long plane_off[3];         // byte offset of each component's sample plane [bh * 8][bw * 8] in the workspace
    long long block0;               // first block of the image on the IDCT grid
    long long pix0;                 // first pixel of the image on the colour grid
    int kind, H, W, ncomp, hmax, vmax, mcus_x, bpm;
    int bw[3], bh[3];               // component planes in blocks (whole MCUs)
    int dw, dh;                     // downsampled width / height of the chroma components (libjpeg)
    int q_off[3], dc_off[3], ac_off[3];   // byte offsets of the component's tables in the table block
};

// One restart interval (the whole scan when there are none): its bits are [0, nbits) of the clean stream from byte
// `byte0` of `in`; it holds nmcu MCUs from MCU mcu0; its subsequences are [sub0, sub0 + nsub) of the launch.
struct JpegInterval {
    long long byte0;
    long long sub0;
    unsigned nbits;
    int image, mcu0, nmcu, nsub;
};

// Decoder state at a symbol boundary: bit position in the interval, block of the MCU, coefficient index (0: DC next).
__host__ __device__ __forceinline__ unsigned long long jpeg_state(unsigned p, int z, int k) {
    return static_cast<unsigned long long>(p) | (static_cast<unsigned long long>(z) << 32) | (static_cast<unsigned long long>(k) << 40);
}
__host__ __device__ __forceinline__ unsigned jpeg_state_p(unsigned long long s) { return static_cast<unsigned>(s); }
__host__ __device__ __forceinline__ int jpeg_state_z(unsigned long long s) { return static_cast<int>((s >> 32) & 0xff); }
__host__ __device__ __forceinline__ int jpeg_state_k(unsigned long long s) { return static_cast<int>((s >> 40) & 0xff); }

// MSB-first bit reader over [0, nbits) of an interval; bits past the end read as 0 (libjpeg inserts zeros there).
struct JpegBits {
    const uint8_t *data;
    unsigned nbytes;
    unsigned next;                  // next byte to load
    unsigned long long buf;         // left-aligned
    int have;                       // valid bits in buf
    unsigned pos;                   // bits consumed

    __host__ __device__ __forceinline__ void seek(const uint8_t *d, unsigned nbits, unsigned p) {
        data = d, nbytes = (nbits + 7) >> 3, next = p >> 3, buf = 0, have = 0, pos = p;
        fill();
        buf <<= (p & 7), have -= (p & 7);
    }
    __host__ __device__ __forceinline__ void fill() {
        while (have <= 56) {
            const unsigned long long b = next < nbytes ? data[next] : 0u;
            ++next;
            buf |= b << (56 - have);
            have += 8;
        }
    }
    __host__ __device__ __forceinline__ unsigned peek16() const { return static_cast<unsigned>(buf >> 48); }
    __host__ __device__ __forceinline__ void skip(int n) {
        buf <<= n, have -= n, pos += n;
        if (have < 32) fill();
    }
    __host__ __device__ __forceinline__ int take(int n) {          // 0 <= n <= 16
        const int v = n ? static_cast<int>(buf >> (64 - n)) : 0;
        skip(n);
        return v;
    }
};

__host__ __device__ __forceinline__ int jpeg_extend(int v, int s) { return (s && v < (1 << (s - 1))) ? v - (1 << s) + 1 : v; }

// One Huffman symbol (jdhuff.c: lookahead, then the code lengths 9..16 against maxcode; an invalid code gives 0).
__host__ __device__ __forceinline__ int jpeg_huff_decode(JpegBits &b, const uint8_t *rec) {
    const unsigned p16 = b.peek16();
    const unsigned e = reinterpret_cast<const uint16_t *>(rec + kJpegLookOff)[p16 >> 8];
    if (e) {
        b.skip(static_cast<int>(e >> 8));
        return static_cast<int>(e & 0xff);
    }
    const int *maxcode = reinterpret_cast<const int *>(rec + kJpegMaxcodeOff);
    int l = 9;
    while (l <= 16 && static_cast<int>(p16 >> (16 - l)) > maxcode[l]) ++l;
    if (l > 16) {
        b.skip(16);
        return 0;
    }
    const int code = static_cast<int>(p16 >> (16 - l));
    b.skip(l);
    return rec[kJpegHuffvalOff + ((code + reinterpret_cast<const int *>(rec + kJpegValoffOff)[l]) & 0xff)];
}

__host__ __device__ __forceinline__ int jpeg_natural(int k) {       // zigzag index -> natural, k up to 79 (jpeg_natural_order)
    static constexpr unsigned char nat[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                       41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                       30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    return k < 64 ? nat[k] : 63;
}

// Component of block z of an MCU (3 components: hmax * vmax luma blocks, then Cb, then Cr).
__host__ __device__ __forceinline__ int jpeg_comp(const JpegImage &im, int z) {
    const int nl = im.hmax * im.vmax;
    return im.ncomp == 1 ? 0 : (z < nl ? 0 : z - nl + 1);
}

// Where block z of MCU m lands: int16 offset of its 64 coefficients.
__host__ __device__ __forceinline__ long long jpeg_block_coef(const JpegImage &im, long long m, int z) {
    const int c = jpeg_comp(im, z);
    const long long my = m / im.mcus_x, mx = m - my * im.mcus_x;
    long long by = my, bx = mx;
    if (c == 0 && im.ncomp == 3) by = my * im.vmax + z / im.hmax, bx = mx * im.hmax + z % im.hmax;
    return im.coef_off[c] + (by * im.bw[c] + bx) * 64;
}

// Decode of one subsequence from state `s` at a symbol boundary, symbol by symbol while the position is below `stop`.
// Speculative pass (WRITE = false): sums[0] = blocks completed, sums[1 + c] = sum of component c's DC differences.
// Final pass (WRITE = true): also stops once `block_limit` blocks of the interval are done; the coefficients of the block
// in progress (`block`, interval-relative, counted on) are stored, the DC made absolute from the predictors pred[c].
// Returns the state at the first symbol boundary at or past `stop`.
template <bool WRITE>
__host__ __device__ __forceinline__ unsigned long long jpeg_decode_run(const JpegImage &im, const JpegInterval &iv, const uint8_t *in,
                                                              const uint8_t *tab, unsigned long long s, unsigned stop,
                                                              unsigned *sums, long long block, long long block_limit,
                                                              int *pred, int16_t *coef) {
    JpegBits b;
    b.seek(in + iv.byte0, iv.nbits, jpeg_state_p(s));
    int z = jpeg_state_z(s), k = jpeg_state_k(s);
    const int bpm = im.bpm;
    // per-component values in scalars (a run-time index into a small array would put it in local memory)
    int p0 = WRITE ? pred[0] : 0, p1 = WRITE ? pred[1] : 0, p2 = WRITE ? pred[2] : 0;
    unsigned nblk = 0;
    while (b.pos < stop && (!WRITE || block < block_limit)) {
        const int c = jpeg_comp(im, z);
        int16_t *blk = nullptr;
        if (WRITE) blk = coef + jpeg_block_coef(im, iv.mcu0 + block / bpm, z);
        if (k == 0) {
            const int sz = jpeg_huff_decode(b, tab + im.dc_off[c]);
            const int diff = jpeg_extend(b.take(sz), sz);
            const int v = (c == 0 ? p0 : (c == 1 ? p1 : p2)) + diff;
            if (c == 0) p0 = v; else if (c == 1) p1 = v; else p2 = v;
            if (WRITE) blk[0] = static_cast<int16_t>(v);
            k = 1;
        } else {
            const int sym = jpeg_huff_decode(b, tab + im.ac_off[c]);
            const int r = sym >> 4, sz = sym & 15;
            if (sz) {
                k += r;
                const int v = jpeg_extend(b.take(sz), sz);
                if (WRITE) blk[jpeg_natural(k)] = static_cast<int16_t>(v);
                ++k;
            } else {
                k = r == 15 ? k + 16 : 64;                 // ZRL, or end of block
            }
        }
        if (k >= 64) {
            k = 0;
            if (++z == bpm) z = 0;
            if (WRITE) ++block; else ++nblk;
        }
    }
    if (!WRITE) sums[0] = nblk, sums[1] = static_cast<unsigned>(p0), sums[2] = static_cast<unsigned>(p1), sums[3] = static_cast<unsigned>(p2);
    return jpeg_state(b.pos, z, k);
}

// ---- dequantisation + islow IDCT (jidctint.c), as two 8-point passes so that a kernel runs them on 8 threads
constexpr int kFix0298 = 2446, kFix0390 = 3196, kFix0541 = 4433, kFix0765 = 6270, kFix0899 = 7373, kFix1175 = 9633,
              kFix1501 = 12299, kFix1847 = 15137, kFix1961 = 16069, kFix2053 = 16819, kFix2562 = 20995, kFix3072 = 25172;

__host__ __device__ __forceinline__ void jpeg_idct_1d(const int *v, int stride, int pre, int *o) {
    int z2 = v[2 * stride], z3 = v[6 * stride];
    int z1 = (z2 + z3) * kFix0541;
    const int tmp2 = z1 - z3 * kFix1847, tmp3 = z1 + z2 * kFix0765;
    z2 = v[0] + pre, z3 = v[4 * stride];
    const int tmp0 = (z2 + z3) * 8192, tmp1 = (z2 - z3) * 8192;
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    int t0 = v[7 * stride], t1 = v[5 * stride], t2 = v[3 * stride], t3 = v[1 * stride];
    z1 = t0 + t3, z2 = t1 + t2, z3 = t0 + t2;
    int z4 = t1 + t3;
    const int z5 = (z3 + z4) * kFix1175;
    t0 *= kFix0298, t1 *= kFix2053, t2 *= kFix3072, t3 *= kFix1501;
    z1 *= -kFix0899, z2 *= -kFix2562, z3 = z3 * -kFix1961 + z5, z4 = z4 * -kFix0390 + z5;
    t0 += z1 + z3, t1 += z2 + z4, t2 += z2 + z3, t3 += z1 + z4;
    o[0] = tmp10 + t3, o[7] = tmp10 - t3, o[1] = tmp11 + t2, o[6] = tmp11 - t2;
    o[2] = tmp12 + t1, o[5] = tmp12 - t1, o[3] = tmp13 + t0, o[4] = tmp13 - t0;
}

// Pass 1, column `col`: dequantised coefficients -> ws[row * 8 + col] (>> CONST_BITS - PASS1_BITS, rounded).
__host__ __device__ __forceinline__ void jpeg_idct_col(const int16_t *coef, const uint16_t *q, int col, int *ws) {
    int v[8], o[8];
    for (int r = 0; r < 8; ++r) v[r] = static_cast<int>(coef[r * 8 + col]) * static_cast<int>(q[r * 8 + col]);
    jpeg_idct_1d(v, 1, 0, o);
    for (int r = 0; r < 8; ++r) ws[r * 8 + col] = (o[r] + (1 << 10)) >> 11;
}

// libjpeg's range-limit table on an IDCT output x (centred on 0), indexed by x & 1023.
__host__ __device__ __forceinline__ uint8_t jpeg_range_limit(int x) {
    const int v = x & 1023;
    return static_cast<uint8_t>(v < 128 ? v + 128 : (v < 512 ? 255 : (v < 896 ? 0 : v - 896)));
}

// Pass 2, row `row` of ws -> 8 samples (>> CONST_BITS + PASS1_BITS + 3, rounding folded into the DC term).
__host__ __device__ __forceinline__ void jpeg_idct_row(const int *ws, int row, uint8_t *out) {
    int o[8];
    jpeg_idct_1d(ws + row * 8, 1, 1 << 4, o);
    for (int c = 0; c < 8; ++c) out[c] = jpeg_range_limit(o[c] >> 18);
}

// ---- upsampling + colour conversion of one output pixel
__host__ __device__ __forceinline__ int jpeg_clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// Chroma sample of output pixel (y, x) from plane p (row pitch `pitch`), libjpeg's upsampler for the image's sampling.
__host__ __device__ __forceinline__ int jpeg_chroma(const JpegImage &im, const uint8_t *p, int pitch, int y, int x) {
    if (im.hmax == 1) return p[static_cast<size_t>(y) * pitch + x];
    const int j = x >> 1, last = im.dw - 1;
    if (im.dw <= 2) return p[static_cast<size_t>(y / im.vmax) * pitch + j];
    if (im.vmax == 1) {
        const uint8_t *r = p + static_cast<size_t>(y) * pitch;
        const int c = 3 * r[j];
        if (x & 1) return j == last ? r[j] : (c + r[j + 1] + 2) >> 2;
        return j == 0 ? r[0] : (c + r[j - 1] + 1) >> 2;
    }
    const int i = y >> 1, n = jpeg_clampi((y & 1) ? i + 1 : i - 1, 0, im.dh - 1);
    const uint8_t *r0 = p + static_cast<size_t>(i) * pitch, *r1 = p + static_cast<size_t>(n) * pitch;
    const int s = 3 * r0[j] + r1[j];
    if (x & 1) return j == last ? (4 * s + 7) >> 4 : (3 * s + 3 * r0[j + 1] + r1[j + 1] + 7) >> 4;
    return j == 0 ? (4 * s + 8) >> 4 : (3 * s + 3 * r0[j - 1] + r1[j - 1] + 8) >> 4;
}

__host__ __device__ __forceinline__ uint8_t jpeg_clamp8(int v) { return static_cast<uint8_t>(v < 0 ? 0 : (v > 255 ? 255 : v)); }

// RGB of output pixel (y, x) of a device-decoded image; `ws` is the workspace the sample planes live in.
__host__ __device__ __forceinline__ void jpeg_pixel(const JpegImage &im, const uint8_t *ws, int y, int x, uint8_t *rgb) {
    const int pitch0 = im.bw[0] * 8;
    const int Y = ws[im.plane_off[0] + static_cast<size_t>(y) * pitch0 + x];
    if (im.ncomp == 1) {
        rgb[0] = rgb[1] = rgb[2] = static_cast<uint8_t>(Y);
        return;
    }
    const int pitch = im.bw[1] * 8;
    const int cb = jpeg_chroma(im, ws + im.plane_off[1], pitch, y, x) - 128, cr = jpeg_chroma(im, ws + im.plane_off[2], pitch, y, x) - 128;
    rgb[0] = jpeg_clamp8(Y + ((91881 * cr + 32768) >> 16));
    rgb[1] = jpeg_clamp8(Y + ((-22554 * cb + 32768 - 46802 * cr) >> 16));
    rgb[2] = jpeg_clamp8(Y + ((116130 * cb + 32768) >> 16));
}

// Image of a global index (block or pixel) by binary search over the images' first indices (ascending).
template <typename Get>
__host__ __device__ __forceinline__ int jpeg_find(int n, long long idx, Get first) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (first(mid) <= idx) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// ---- the programs of the three launches, per subsequence / block / pixel (the kernels in jpeg.cu, the simulator in
// hostsim.cpp).  Workspace arrays per subsequence: entry / exit state, sums (blocks, DC differences of 3 components;
// exclusive prefix over the launch after the scan), dirty flag (entry changed since the last speculative decode).
struct JpegArgs {
    const uint8_t *in;
    uint8_t *out;
    uint8_t *ws;
    const JpegImage *images;
    const JpegInterval *ivs;
    const uint8_t *tab;
    unsigned long long *entry, *exit;
    unsigned *sums;
    unsigned char *dirty;
    int16_t *coef;
    int n_img, n_int;
    long long n_sub, n_blocks, n_pix;
    unsigned sub_bits;
};

__host__ __device__ __forceinline__ int jpeg_sub_interval(const JpegArgs &a, long long i) {
    return jpeg_find(a.n_int, i, [&](int j) { return a.ivs[j].sub0; });
}
__host__ __device__ __forceinline__ unsigned jpeg_sub_end(const JpegArgs &a, const JpegInterval &iv, long long i) {
    const unsigned long long e = static_cast<unsigned long long>(i - iv.sub0 + 1) * a.sub_bits;
    return e < iv.nbits ? static_cast<unsigned>(e) : iv.nbits;
}

// Every subsequence starts speculatively at its first bit, block 0 of an MCU, DC next; the first of an interval is right.
__host__ __device__ __forceinline__ void jpeg_sub_init(const JpegArgs &a, long long i) {
    const JpegInterval &iv = a.ivs[jpeg_sub_interval(a, i)];
    a.entry[i] = jpeg_state(static_cast<unsigned>((i - iv.sub0) * a.sub_bits), 0, 0);
    a.dirty[i] = 1;
}

// Decode a dirty subsequence from its entry state to the first symbol boundary past its end: exit state and sums.
__host__ __device__ __forceinline__ void jpeg_sub_speculate(const JpegArgs &a, long long i) {
    if (!a.dirty[i]) return;
    const JpegInterval &iv = a.ivs[jpeg_sub_interval(a, i)];
    a.exit[i] = jpeg_decode_run<false>(a.images[iv.image], iv, a.in, a.tab, a.entry[i], jpeg_sub_end(a, iv, i), a.sums + 4 * i, 0, 0,
                                       nullptr, nullptr);
    a.dirty[i] = 0;
}

// Synchronisation: the next subsequence of the interval must start exactly where this one's decode crossed into it.
// Returns true when its entry changed (it is decoded again next round).  Once every entry equals its predecessor's exit,
// entry 0 of each interval being true makes every entry true: the final decode is the sequential one.
__host__ __device__ __forceinline__ bool jpeg_sub_sync(const JpegArgs &a, long long i) {
    const JpegInterval &iv = a.ivs[jpeg_sub_interval(a, i)];
    if (i + 1 >= iv.sub0 + iv.nsub || a.exit[i] == a.entry[i + 1]) return false;
    a.entry[i + 1] = a.exit[i];
    a.dirty[i + 1] = 1;
    return true;
}

// Final decode of subsequence i after the scan (sums = exclusive prefix): coefficients into their blocks, DC absolute.
__host__ __device__ __forceinline__ void jpeg_sub_write(const JpegArgs &a, long long i) {
    const JpegInterval &iv = a.ivs[jpeg_sub_interval(a, i)];
    const JpegImage &im = a.images[iv.image];
    const unsigned *base = a.sums + 4 * iv.sub0, *here = a.sums + 4 * i;
    int pred[3];
    for (int c = 0; c < 3; ++c) pred[c] = static_cast<int>(here[1 + c] - base[1 + c]);
    const bool last = i + 1 == iv.sub0 + iv.nsub;
    jpeg_decode_run<true>(im, iv, a.in, a.tab, a.entry[i], last ? 0xffffffffu : jpeg_sub_end(a, iv, i), nullptr,
                          static_cast<long long>(here[0] - base[0]), static_cast<long long>(iv.nmcu) * im.bpm, pred, a.coef);
}

// IDCT work item: block g of the launch -> its image, coefficients, quantisation table and sample-plane position.
struct JpegBlockRef {
    const int16_t *coef;
    const uint16_t *q;
    uint8_t *dst;       // row 0 of the block's 8 x 8 samples
    int pitch;
};
__host__ __device__ __forceinline__ JpegBlockRef jpeg_block(const JpegArgs &a, long long g) {
    const int m = jpeg_find(a.n_img, g, [&](int j) { return a.images[j].block0; });
    const JpegImage &im = a.images[m];
    long long local = g - im.block0;
    int c = 0;
    while (c + 1 < im.ncomp && local >= static_cast<long long>(im.bw[c]) * im.bh[c]) local -= static_cast<long long>(im.bw[c]) * im.bh[c], ++c;
    const long long by = local / im.bw[c], bx = local - by * im.bw[c];
    JpegBlockRef r;
    r.coef = a.coef + im.coef_off[c] + local * 64;
    r.q = reinterpret_cast<const uint16_t *>(a.tab + im.q_off[c]);
    r.pitch = im.bw[c] * 8;
    r.dst = a.ws + im.plane_off[c] + (by * 8) * r.pitch + bx * 8;
    return r;
}

// Output pixel p of the launch (images in order): RGB of a decoded image, or the worker-decoded pixel copied.
__host__ __device__ __forceinline__ void jpeg_out_pixel(const JpegArgs &a, long long p) {
    const int m = jpeg_find(a.n_img, p, [&](int j) { return a.images[j].pix0; });
    const JpegImage &im = a.images[m];
    const long long local = p - im.pix0;
    uint8_t *o = a.out + im.out_off + local * 3;
    if (im.kind != 0) {
        const uint8_t *src = a.in + im.in_off + local * 3;
        o[0] = src[0], o[1] = src[1], o[2] = src[2];
        return;
    }
    const int y = static_cast<int>(local / im.W), x = static_cast<int>(local - static_cast<long long>(y) * im.W);
    jpeg_pixel(im, a.ws, y, x, o);
}

}  // namespace b200
