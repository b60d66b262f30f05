// Host-side planner of b200_jpeg_decode_u8 (shared by the CUDA launcher and the CPU simulator used in tests): checks the
// descriptors and tables the worker built, and lays out the launch records and the workspace.
#pragma once
#include <algorithm>
#include <cstring>
#include <vector>

#include "b200ret.h"
#include "jpeg_core.cuh"

namespace b200 {

constexpr unsigned kJpegSubBits = 1024;        // bits per subsequence of the parallel entropy decode
constexpr int kJpegThreads = 256;
constexpr int kJpegMaxCtas = 4096;             // upper bound of the cooperative grid (cta totals in the workspace)

struct JpegPlan {
    std::vector<JpegImage> images;
    std::vector<JpegInterval> ivs;
    long long n_sub = 0, n_blocks = 0, n_pix = 0;
    size_t off_head = 0, off_cta = 0, off_coef = 0, zero_bytes = 0;         // [0, zero_bytes) is cleared per call
    size_t off_images = 0, off_ivs = 0, off_tab = 0, stage_bytes = 0;       // one H2D copy of [off_images, +stage_bytes)
    size_t off_entry = 0, off_exit = 0, off_sums = 0, off_dirty = 0, off_planes = 0, bytes = 0;
};

inline size_t jpeg_round256(size_t v) { return (v + 255) / 256 * 256; }

// B200_OK or the error the entry point returns; no CUDA call.  out_offsets may be NULL (workspace query).
inline int jpeg_plan(const b200_jpeg_desc *desc, const unsigned char *tables, size_t tables_bytes, int n,
                     const long long *out_offsets, unsigned sub_bits, JpegPlan &p) {
    if (n < 0 || (n > 0 && (!desc || !tables)) || sub_bits < 8 || sub_bits > (1u << 30)) return B200_ERR_INVALID_ARG;
    if (tables_bytes >= (1ull << 31)) return B200_ERR_UNSUPPORTED;                  // table offsets are int on the device
    p = JpegPlan();
    p.images.resize(n);
    long long coef = 0, planes = 0;
    auto table_ok = [&](long long off, size_t len, int align) {
        return off >= 0 && off % align == 0 && static_cast<size_t>(off) + len <= tables_bytes;
    };
    for (int i = 0; i < n; ++i) {
        const b200_jpeg_desc &d = desc[i];
        JpegImage &im = p.images[i];
        std::memset(&im, 0, sizeof(im));
        if (d.kind != B200_JPEG_HUFFMAN && d.kind != B200_JPEG_RAW) return B200_ERR_INVALID_ARG;
        if (d.height < 1 || d.width < 1 || d.in_offset < 0 || d.in_bytes < 0) return B200_ERR_INVALID_ARG;
        if (out_offsets && out_offsets[i] < 0) return B200_ERR_INVALID_ARG;
        if (d.height * d.width > (1LL << 31)) return B200_ERR_UNSUPPORTED;
        im.kind = static_cast<int>(d.kind), im.H = static_cast<int>(d.height), im.W = static_cast<int>(d.width);
        im.in_off = d.in_offset, im.in_bytes = d.in_bytes, im.out_off = out_offsets ? out_offsets[i] : 0;
        im.pix0 = p.n_pix, im.block0 = p.n_blocks;
        p.n_pix += d.height * d.width;
        if (d.kind == B200_JPEG_RAW) {
            if (d.in_bytes != d.height * d.width * 3) return B200_ERR_INVALID_ARG;
            continue;
        }
        if (d.height > 65535 || d.width > 65535 || d.restart_interval < 0 || d.restart_interval > 65535) return B200_ERR_INVALID_ARG;
        if (d.ncomp != 1 && d.ncomp != 3) return B200_ERR_UNSUPPORTED;
        const bool samp_ok = d.ncomp == 1 ? (d.hmax == 1 && d.vmax == 1)
                                          : ((d.hmax == 1 && d.vmax == 1) || (d.hmax == 2 && d.vmax == 1) || (d.hmax == 2 && d.vmax == 2));
        if (!samp_ok) return B200_ERR_UNSUPPORTED;
        im.ncomp = static_cast<int>(d.ncomp), im.hmax = static_cast<int>(d.hmax), im.vmax = static_cast<int>(d.vmax);
        im.mcus_x = static_cast<int>((d.width + 8 * d.hmax - 1) / (8 * d.hmax));
        const long long mcus_y = (d.height + 8 * d.vmax - 1) / (8 * d.vmax), mcus = mcus_y * im.mcus_x;
        im.bpm = im.ncomp == 1 ? 1 : im.hmax * im.vmax + 2;
        im.dw = static_cast<int>((d.width + d.hmax - 1) / d.hmax), im.dh = static_cast<int>((d.height + d.vmax - 1) / d.vmax);
        for (int c = 0; c < im.ncomp; ++c) {
            if (!table_ok(d.quant[c], kJpegQuantBytes, 2) || !table_ok(d.dc[c], kJpegHuffBytes, 4) || !table_ok(d.ac[c], kJpegHuffBytes, 4))
                return B200_ERR_INVALID_ARG;
            im.q_off[c] = static_cast<int>(d.quant[c]), im.dc_off[c] = static_cast<int>(d.dc[c]), im.ac_off[c] = static_cast<int>(d.ac[c]);
            im.bw[c] = c == 0 ? im.mcus_x * im.hmax : im.mcus_x;
            im.bh[c] = static_cast<int>(c == 0 ? mcus_y * im.vmax : mcus_y);
            const long long blocks = static_cast<long long>(im.bw[c]) * im.bh[c];
            im.coef_off[c] = coef, im.plane_off[c] = planes;
            coef += blocks * 64, planes += static_cast<long long>(jpeg_round256(static_cast<size_t>(blocks) * 64));
            p.n_blocks += blocks;
        }
        const long long ri = d.restart_interval, n_int = ri ? (mcus + ri - 1) / ri : 1;
        if (!table_ok(d.intervals, static_cast<size_t>(n_int) * 8, 8)) return B200_ERR_INVALID_ARG;
        const long long *starts = reinterpret_cast<const long long *>(tables + d.intervals);
        for (long long r = 0; r < n_int; ++r) {
            const long long s0 = starts[r], s1 = r + 1 < n_int ? starts[r + 1] : d.in_bytes;
            if ((r == 0 && s0 != 0) || s1 < s0 || s1 > d.in_bytes) return B200_ERR_INVALID_ARG;
            if ((s1 - s0) * 8 >= (1LL << 31)) return B200_ERR_UNSUPPORTED;
            JpegInterval iv;
            iv.byte0 = d.in_offset + s0, iv.nbits = static_cast<unsigned>((s1 - s0) * 8), iv.image = i;
            iv.mcu0 = static_cast<int>(r * (ri ? ri : mcus)), iv.nmcu = static_cast<int>(ri ? std::min(ri, mcus - r * ri) : mcus);
            iv.nsub = static_cast<int>(iv.nbits > 0 ? (iv.nbits + sub_bits - 1) / sub_bits : 1);
            iv.sub0 = p.n_sub;
            p.n_sub += iv.nsub;
            p.ivs.push_back(iv);
        }
    }
    size_t o = 0;
    auto take = [&](size_t nb) {
        const size_t at = o;
        o = jpeg_round256(o + nb);
        return at;
    };
    p.off_head = take(256);
    p.off_cta = take(static_cast<size_t>(kJpegMaxCtas) * 16);
    p.off_coef = take(static_cast<size_t>(coef) * 2);
    p.zero_bytes = o;
    p.off_images = take(p.images.size() * sizeof(JpegImage));
    p.off_ivs = take(p.ivs.size() * sizeof(JpegInterval));
    p.off_tab = take(tables_bytes);
    p.stage_bytes = o - p.off_images;
    p.off_entry = take(static_cast<size_t>(p.n_sub) * 8);
    p.off_exit = take(static_cast<size_t>(p.n_sub) * 8);
    p.off_sums = take(static_cast<size_t>(p.n_sub) * 16);
    p.off_dirty = take(static_cast<size_t>(p.n_sub));
    p.off_planes = o;
    for (JpegImage &im : p.images)
        for (int c = 0; c < im.ncomp; ++c) im.plane_off[c] += static_cast<long long>(p.off_planes);
    p.bytes = p.off_planes + static_cast<size_t>(planes);
    return B200_OK;
}

// The launch records and tables as the device sees them: [off_images, off_images + stage_bytes) of the workspace.
inline void jpeg_stage(const JpegPlan &p, const unsigned char *tables, size_t tables_bytes, std::vector<unsigned char> &stage) {
    stage.assign(p.stage_bytes, 0);
    std::memcpy(stage.data(), p.images.data(), p.images.size() * sizeof(JpegImage));
    std::memcpy(stage.data() + (p.off_ivs - p.off_images), p.ivs.data(), p.ivs.size() * sizeof(JpegInterval));
    std::memcpy(stage.data() + (p.off_tab - p.off_images), tables, tables_bytes);
}

inline JpegArgs jpeg_args(const JpegPlan &p, const uint8_t *in, uint8_t *out, uint8_t *ws, unsigned sub_bits) {
    JpegArgs a;
    a.in = in, a.out = out, a.ws = ws;
    a.images = reinterpret_cast<const JpegImage *>(ws + p.off_images);
    a.ivs = reinterpret_cast<const JpegInterval *>(ws + p.off_ivs);
    a.tab = ws + p.off_tab;
    a.entry = reinterpret_cast<unsigned long long *>(ws + p.off_entry);
    a.exit = reinterpret_cast<unsigned long long *>(ws + p.off_exit);
    a.sums = reinterpret_cast<unsigned *>(ws + p.off_sums);
    a.dirty = ws + p.off_dirty;
    a.coef = reinterpret_cast<int16_t *>(ws + p.off_coef);
    a.n_img = static_cast<int>(p.images.size()), a.n_int = static_cast<int>(p.ivs.size());
    a.n_sub = p.n_sub, a.n_blocks = p.n_blocks, a.n_pix = p.n_pix, a.sub_bits = sub_bits;
    return a;
}

}  // namespace b200
