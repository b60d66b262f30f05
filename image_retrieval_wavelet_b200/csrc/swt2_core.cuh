// HP-SWT core: undecimated separable wavelet stencil over one shared-memory tile.
//
// Replaces pywt.swt2 as called by SWTTransform._apply_wavelet
// (/root/reference/main/transforms/custom_transforms.py:163-166): level l (dilation s = 2^(l-1)) is the periodised FIR
//      y[n] = sum_t h[t] * x[(n + s * (F/2 - t)) mod N]
// along axis -2 and then axis -1 with (dec_lo | dec_hi); level l+1 consumes level l's LL; only the level-L bands
// (cA, cH, cV, cD) are kept.
//
// Per tile: (1) the tile plus its composite halo is staged once, wrapped and converted to float32, in shared memory;
// (2) every level is a horizontal pass (shared -> shared) and a vertical pass (shared -> shared, or -> global for the
// last level), both fully unrolled over the taps with compile-time F and dilation: a horizontal unit is 4 adjacent
// pixels of one row (aligned 128-bit shared loads), a vertical unit is 4 columns x kSwtR rows of one residue class, so
// each staged row is loaded once for kSwtR outputs; (3) the four sub-bands leave the SM once, as 128-bit streaming
// stores.  No intermediate plane ever goes to global memory.  The kernels are issue-bound before they are HBM-bound, so
// the unit -> (row, column) maps use precomputed multiply-high divisions and no per-pixel modulo.
//
// Everything here is __host__ __device__ and expressed per (tid, nthreads) so that tests/ can run the very same
// indexing code on the CPU (csrc/hostsim.cpp) — there is no CPU product path.
#pragma once
#include <stddef.h>
#include <stdint.h>

#ifndef __CUDACC__
#include <cmath>
#define __host__
#define __device__
#define __forceinline__ inline
#endif

namespace b200 {

constexpr int kSwtGuard = 32;   // floats of slack before/after each buffer (garbage column groups may touch it)
constexpr int kSwtR = 4;        // output rows per vertical work unit
constexpr int kSwtMaxLevelFast = 3;

struct SwtGeom {
    int B, C, H, W;          // planes = B*C
    int level, F;
    int in_is_u8;
    int TH, TW;              // output tile (TW % 4 == 0; fast path: TH % (kSwtR * 2^(level-1)) == 0)
    int tiles_y, tiles_x;
    int top, left;           // rows/cols needed before the tile = (2^L - 1) * (F/2 - 1)
    int bot, right;          // rows/cols needed after the tile  = (2^L - 1) * F/2
    int padL;                // left halo rounded up to a multiple of 4: tile column 0 sits at buffer column padL
    int RH, RWp;             // staged rows, padded row stride in floats (multiple of 4)
    int RHv;                 // rows of the last level's horizontal outputs = TH + 2^(L-1) * (F-1)
    int threads;             // CTA size
    int off_b;               // float offset of buffer B from the start of shared memory
    uint32_t m_load;         // multiply-high reciprocals of the unit -> row divisors (0: divisor 1)
    uint32_t m_load8;        // same for the uint8 staging units (8 buffer columns each)
    int u8_stage;            // uint8 staging: 1 = 8-pixel units, 0 = the 4-pixel units shared with float32 (chosen from W)
    uint32_t m_lvl[kSwtMaxLevelFast];
    float lo[20], hi[20];
    // host only, behind the taps: ptxas merges the kernels' tap loads at 16-byte boundaries of the parameter block, so
    // lo / hi keep the offset (12 mod 16) the kernels were measured with
    int nbuf;                // generic program: 3 full buffers; fast program: buffer A + buffer B (off_b)
    int smem_floats;
};

// Pass form of the fast path, a function of (F, level) alone (measurements: swt2_plan.h, DESIGN.md §4.1).
// 2: register-window intermediate levels (swt_rw_ll) + two-pass last level; 0: two-pass levels.
__host__ __device__ constexpr int swt_rw_form(int F, int level) { return level >= 2 && F <= 4 ? 2 : 0; }
// 1: sliding last vertical pass (swt_vpass_final_slide; TH % (kVsR * 2^(level-1)) == 0); 0: blocked (swt_vpass_final).
__host__ __device__ constexpr int swt_vs_form(int F, int level) { return level == 1 && F == 8 ? 1 : 0; }

__host__ __device__ __forceinline__ uint32_t swt_magic(uint32_t d) {      // host planner only (64-bit division)
    return d <= 1 ? 0u : static_cast<uint32_t>(((1ull << 32) + d - 1) / d);
}
// u / d for u * d < 2^32, m = swt_magic(d)
__host__ __device__ __forceinline__ uint32_t swt_div(uint32_t u, uint32_t m) {
#ifdef __CUDA_ARCH__
    return m ? __umulhi(u, m) : u;
#else
    return m ? static_cast<uint32_t>((static_cast<unsigned long long>(u) * m) >> 32) : u;
#endif
}

// uint8 -> float32 / 255, bit-identical to IEEE division (np.array(img).astype(float32) / 255.0,
// custom_transforms.py:147) for all 256 inputs: 1/255 split into float32 hi + lo, q = fma(x, hi, x * lo) carries
// ~48 bits of x/255 into a single rounding, and no x/255 lies within 2^-33 (relative) of a float32 rounding boundary.
// Checked exhaustively (tests/test_host_logic.py through the simulator, and against the oracle on the device).
__host__ __device__ __forceinline__ float swt_u8_float(float x) {      // x = float(b), b = 0..255
    const float hi = 0.003921568859368562698f;        // fl32(1/255)
    const float lo = -2.319175823606301e-10f;         // fl32(1/255 - hi)
#ifdef __CUDA_ARCH__
    return __fmaf_rn(x, hi, __fmul_rn(x, lo));
#else
    const float t = x * lo;
    return std::fmaf(x, hi, t);
#endif
}
__host__ __device__ __forceinline__ float swt_u8_unit(uint32_t b) { return swt_u8_float(static_cast<float>(b)); }

// a0 += c*x0, a1 += c*x1.  PACKED: one FFMA2 on sm_100 (two independent IEEE FMAs — same bits as the scalar form).
// Measured on B200: packing pays for the long filters' last vertical pass (db4 level 1: +4 %), and costs 5-15 % on the
// short ones (register-pair constraints), so the callers enable it for F >= 6 only.
template <bool PACKED>
__host__ __device__ __forceinline__ void swt_fma2(float c, float x0, float x1, float &a0, float &a1) {
#if defined(__CUDA_ARCH__) && __CUDA_ARCH__ >= 1000
    if constexpr (PACKED) {
        const float2 r = __ffma2_rn(make_float2(c, c), make_float2(x0, x1), make_float2(a0, a1));
        a0 = r.x, a1 = r.y;
        return;
    }
#endif
    a0 += c * x0, a1 += c * x1;
}

// a += cl*x, d += ch*x (one pixel, both filters): the packed form multiplies the (lo, hi) tap pair by a broadcast x
template <bool PACKED>
__host__ __device__ __forceinline__ void swt_fma_pair(float cl, float ch, float x, float &a, float &d) {
#if defined(__CUDA_ARCH__) && __CUDA_ARCH__ >= 1000
    if constexpr (PACKED) {
        const float2 r = __ffma2_rn(make_float2(cl, ch), make_float2(x, x), make_float2(a, d));
        a = r.x, d = r.y;
        return;
    }
#endif
    a += cl * x, d += ch * x;
}

template <int VEC>
__host__ __device__ __forceinline__ void swt_ld_vec(const float *p, float *d) {
#ifdef __CUDA_ARCH__
    if constexpr (VEC == 4) {
        const float4 v = *reinterpret_cast<const float4 *>(p);
        d[0] = v.x, d[1] = v.y, d[2] = v.z, d[3] = v.w;
    } else {
        const float2 v = *reinterpret_cast<const float2 *>(p);
        d[0] = v.x, d[1] = v.y;
    }
#else
    for (int e = 0; e < VEC; ++e) d[e] = p[e];
#endif
}
template <int VEC>
__host__ __device__ __forceinline__ void swt_st_vec(float *p, const float *s) {
#ifdef __CUDA_ARCH__
    if constexpr (VEC == 4)
        *reinterpret_cast<float4 *>(p) = make_float4(s[0], s[1], s[2], s[3]);
    else
        *reinterpret_cast<float2 *>(p) = make_float2(s[0], s[1]);
#else
    for (int e = 0; e < VEC; ++e) p[e] = s[e];
#endif
}

// periodic index; branch-free when i is within one period of [0, n) (always, unless the image is smaller than the halo)
__host__ __device__ __forceinline__ int swt_wrap(int i, int n) {
    i += i < 0 ? n : 0;
    i -= i >= n ? n : 0;
    if (i < 0 || i >= n) {
        i %= n;
        i += i < 0 ? n : 0;
    }
    return i;
}

// ---------------------------------------------------------------------------------------------- tile load
// Rows [ty*TH - top, ...) x buffer columns [0, RWp) of the staging buffer; buffer column padL is global column
// tx*TW.  Every buffer cell gets the periodically wrapped pixel (cells outside the halo are never used).  A unit is 4
// buffer columns of one row.  kSwtLoadBatch units are in flight per thread: `ld.issue` starts the global reads of 4
// consecutive in-row pixels (widest aligned accesses) for the whole batch before `ld.finish` converts any of them, so
// the global-memory latency is paid once per batch; units that wrap around the image edge go pixel by pixel (`ld.one`).
constexpr int kSwtLoadBatch = 4;

template <typename Ld>
__host__ __device__ __forceinline__ void swt_load_tile(const SwtGeom &g, const void *in_plane, float *buf, int ty, int tx,
                                                       int tid, int nthreads, Ld ld) {
    const int r_first = ty * g.TH - g.top;
    const int gc_base = tx * g.TW - g.padL;            // global column of buffer column 0
    const int groups = g.RWp / 4;
    const uint32_t units = static_cast<uint32_t>(g.RH) * groups;
    for (uint32_t base = tid; base < units; base += kSwtLoadBatch * nthreads) {
        uint32_t raw[kSwtLoadBatch][4];
        size_t off[kSwtLoadBatch];
        int dst[kSwtLoadBatch], gcs[kSwtLoadBatch];
#pragma unroll
        for (int b = 0; b < kSwtLoadBatch; ++b) {
            const uint32_t u = base + b * nthreads;
            dst[b] = -1;
            if (u < units) {
                const int i = static_cast<int>(swt_div(u, g.m_load));
                const int m = static_cast<int>(u) - i * groups;
                const int gr = swt_wrap(r_first + i, g.H);
                // a unit that lies entirely beyond one image edge is the same 4 pixels one period away: only the (at
                // most two per row) units that straddle an edge go pixel by pixel
                int gc = gc_base + 4 * m;
                gc -= gc >= g.W ? g.W : 0;
                gc += gc + 3 < 0 ? g.W : 0;
                gcs[b] = gc;
                off[b] = static_cast<size_t>(gr) * g.W;
                dst[b] = i * g.RWp + 4 * m;
                if (gc >= 0 && gc + 3 < g.W) ld.issue(in_plane, off[b] + gc, g.in_is_u8, raw[b]);
            }
        }
#pragma unroll
        for (int b = 0; b < kSwtLoadBatch; ++b) {
            if (dst[b] < 0) continue;
            float v[4];
            if (gcs[b] >= 0 && gcs[b] + 3 < g.W) {
                ld.finish(raw[b], off[b] + gcs[b], g.in_is_u8, v);
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) v[e] = ld.one(in_plane, off[b] + swt_wrap(gcs[b] + e, g.W), g.in_is_u8);
            }
            swt_st_vec<4>(buf + dst[b], v);
        }
    }
}

// uint8 planes: a unit is kSwtU8Chunk = 8 consecutive buffer columns of one row.  The 8 pixels are read as the three
// aligned 32-bit words that cover them and funnel-shifted into place (a 518-wide row starts on any byte boundary),
// converted with swt_u8_unit and stored as two 128-bit words.  One row / column decomposition, one wrap and one edge
// test per 8 pixels instead of per 4 — the staging phase was 38 % of the issued instructions of the db4 level-1 kernel
// (profiles/r1x_swt_full.md) — and kSwtU8Batch units (3 loads each) are in flight per thread.  Units that straddle an image
// edge go pixel by pixel; units entirely beyond an edge read the same pixels one period away.
constexpr int kSwtU8Chunk = 8;

// kSwtU8Batch = units in flight per thread: 2 under the short filters, 4 (12 loads) under F >= 6 (measured: db4 518^2
// 924 -> 917 us with 4, db2 518^2 726 -> 771 us)
template <int kSwtU8Batch, typename Ld>
__host__ __device__ __forceinline__ void swt_load_tile_u8(const SwtGeom &g, const uint8_t *plane, float *buf, int ty, int tx,
                                                          int tid, int nthreads, Ld ld) {
    const int r_first = ty * g.TH - g.top;
    const int gc_base = tx * g.TW - g.padL;
    const int chunks = (g.RWp + kSwtU8Chunk - 1) / kSwtU8Chunk;
    const uint32_t units = static_cast<uint32_t>(g.RH) * chunks;
    for (uint32_t base = tid; base < units; base += kSwtU8Batch * nthreads) {
        uint32_t raw[kSwtU8Batch][3];
        size_t off[kSwtU8Batch];
        int dst[kSwtU8Batch], gcs[kSwtU8Batch];
        bool full[kSwtU8Batch];            // RWp is a multiple of 4, not of 8: the last unit of a row may own 4 columns only
#pragma unroll
        for (int b = 0; b < kSwtU8Batch; ++b) {
            const uint32_t u = base + b * nthreads;
            dst[b] = -1;
            full[b] = false;
            if (u < units) {
                const int i = static_cast<int>(swt_div(u, g.m_load8));
                const int m = static_cast<int>(u) - i * chunks;
                const int gr = swt_wrap(r_first + i, g.H);
                int gc = gc_base + kSwtU8Chunk * m;
                gc -= gc >= g.W ? g.W : 0;
                gc += gc + (kSwtU8Chunk - 1) < 0 ? g.W : 0;
                gcs[b] = gc;
                off[b] = static_cast<size_t>(gr) * g.W;
                dst[b] = i * g.RWp + kSwtU8Chunk * m;
                full[b] = kSwtU8Chunk * (m + 1) <= g.RWp;
                if (gc >= 0 && gc + (kSwtU8Chunk - 1) < g.W) ld.issue_u8x8(plane, off[b] + gc, raw[b]);
            }
        }
#pragma unroll
        for (int b = 0; b < kSwtU8Batch; ++b) {
            if (dst[b] < 0) continue;
            float v[kSwtU8Chunk];
            if (gcs[b] >= 0 && gcs[b] + (kSwtU8Chunk - 1) < g.W) {
                ld.finish_u8x8(raw[b], off[b] + gcs[b], v);
            } else {
#pragma unroll
                for (int e = 0; e < kSwtU8Chunk; ++e) v[e] = ld.one(plane, off[b] + swt_wrap(gcs[b] + e, g.W), 1);
            }
            swt_st_vec<4>(buf + dst[b], v);
            if (full[b]) swt_st_vec<4>(buf + dst[b] + 4, v + 4);
        }
    }
}

// ---------------------------------------------------------------------------------------------- horizontal pass
// dst(row - dr0, col - dc0) = sum_t h[t] * src(row, col + S*(F/2 - t)) for rows [r0, r1) and `ncg` column groups of 4
// starting at buffer column 4*c0g; dlo uses dec_lo, dhi (BOTH) dec_hi.
template <int F, int S, bool BOTH>
__host__ __device__ __forceinline__ void swt_hpass(const SwtGeom &g, const float *src, int sstride, float *dlo, float *dhi,
                                                   int dstride, int r0, int r1, int c0g, int ncg, uint32_t magic, int dr0,
                                                   int dc0, int tid, int nthreads) {
    constexpr int omin = -S * (F / 2 - 1);
    constexpr int omax = S * (F / 2);
    constexpr int amin = -(((-omin) + 3) / 4) * 4;                       // omin floored to a multiple of 4 (omin <= 0)
    constexpr int nvec = (3 + omax - amin) / 4 + 1;
    const uint32_t units = static_cast<uint32_t>(r1 - r0) * ncg;
    for (uint32_t u = tid; u < units; u += nthreads) {
        const int rr = static_cast<int>(swt_div(u, magic));
        const int cg = static_cast<int>(u) - rr * ncg;
        const int row = r0 + rr, j0 = 4 * (c0g + cg);
        const float *p = src + row * sstride + j0 + amin;
        float w[nvec * 4];
#pragma unroll
        for (int i = 0; i < nvec; ++i) swt_ld_vec<4>(p + 4 * i, w + 4 * i);
        float a[4], d[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            float sa = 0.f, sd = 0.f;
#pragma unroll
            for (int t = 0; t < F; ++t) {
                const float x = w[v + S * (F / 2 - t) - amin];
                if constexpr (BOTH)
                    swt_fma_pair<(F >= 6)>(g.lo[t], g.hi[t], x, sa, sd);
                else
                    sa += g.lo[t] * x;
            }
            a[v] = sa, d[v] = sd;
        }
        const int o = (row - dr0) * dstride + (j0 - dc0);
        swt_st_vec<4>(dlo + o, a);
        if (BOTH) swt_st_vec<4>(dhi + o, d);
    }
}

// ---------------------------------------------------------------------------------------------- vertical passes
// A unit is (column group, residue class rho mod S, block of kSwtR rows of that class): the kSwtR + F - 1 source rows
// are loaded once; out[m] = sum_t h[t] * w[m + F-1-t].
// Intermediate level: LL only, shared -> shared, output rows [r0, r1) (any count; rows past r1 are computed from
// clamped loads and dropped).
template <int F, int S>
__host__ __device__ __forceinline__ void swt_vpass_ll(const SwtGeom &g, const float *src, float *dst, int stride, int r0, int r1,
                                                      int c0g, int ncg, uint32_t magic, int tid, int nthreads) {
    constexpr int R = kSwtR;
    const int per_class = (r1 - r0 + S - 1) / S;
    const int nblk = (per_class + R - 1) / R;
    const uint32_t units = static_cast<uint32_t>(ncg) * S * nblk;
    for (uint32_t u = tid; u < units; u += nthreads) {
        const int rest = static_cast<int>(swt_div(u, magic));
        const int cg = static_cast<int>(u) - rest * ncg;
        const int rho = rest % S, b = rest / S;
        const int first = r0 + rho + S * R * b;
        const int j0 = 4 * (c0g + cg);
        float w[R + F - 1][4];
#pragma unroll
        for (int m = 0; m < R + F - 1; ++m) {
            int rr = first - S * (F / 2 - 1) + S * m;
            rr = rr < g.RH - 1 ? rr : g.RH - 1;
            swt_ld_vec<4>(src + rr * stride + j0, w[m]);
        }
#pragma unroll
        for (int m = 0; m < R; ++m) {
            const int i = first + S * m;
            float a[4];
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                float s = 0.f;
#pragma unroll
                for (int t = 0; t < F; ++t) s += g.lo[t] * w[m + F - 1 - t][v];
                a[v] = s;
            }
            if (i < r1) swt_st_vec<4>(dst + i * stride + j0, a);
        }
    }
}

// Last level: hl / hh are the compact horizontal outputs (RHv rows x stride TWp, row 0 = tile row 0 - S*(F/2-1));
// the four bands of the TH x TW tile go to global memory (out_plane: [4][H][W]) through `store(p, v, n)`.
// ALIGNED: W % 4 == 0 — every column group is 4 wide and every output row 16-byte aligned, so the stores need neither the
// width nor the alignment test (16 stores per unit; the tests were ~5 instructions each).
template <int F, int S, bool ALIGNED, typename Store>
__host__ __device__ __forceinline__ void swt_vpass_final(const SwtGeom &g, const float *hl, const float *hh, int stride,
                                                         float *out_plane, int row_g0, int col_g0, int ncg, uint32_t magic,
                                                         int tid, int nthreads, Store store) {
    constexpr int R = F == 8 ? kSwtR / 2 : kSwtR;        // F = 8: 2 rows per unit keep the kernel at 80 registers without spills
    const int nblk = g.TH / (S * R);
    const uint32_t units = static_cast<uint32_t>(ncg) * S * nblk;
    const size_t plane = static_cast<size_t>(g.H) * g.W;
    for (uint32_t u = tid; u < units; u += nthreads) {
        const int rest = static_cast<int>(swt_div(u, magic));
        const int cg = static_cast<int>(u) - rest * ncg;
        const int rho = rest % S, b = rest / S;
        const int o0 = rho + S * R * b;                     // first tile-local output row of the unit
        const int gc = col_g0 + 4 * cg;
        if (gc >= g.W || row_g0 + o0 >= g.H) continue;
        const int n = g.W - gc >= 4 ? 4 : g.W - gc;          // W is even: n is 4 or 2
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const float *src = (half ? hh : hl) + o0 * stride + 4 * cg;
            float w[R + F - 1][4];
#pragma unroll
            for (int m = 0; m < R + F - 1; ++m) swt_ld_vec<4>(src + S * m * stride, w[m]);
#pragma unroll
            for (int m = 0; m < R; ++m) {
                float a[4], d[4];
                if constexpr (F >= 6) {          // packed FFMA2 over pixel pairs (see swt_fma2)
#pragma unroll
                    for (int v = 0; v < 4; ++v) a[v] = 0.f, d[v] = 0.f;
#pragma unroll
                    for (int t = 0; t < F; ++t) {
                        const float *x = w[m + F - 1 - t];
                        swt_fma2<true>(g.lo[t], x[0], x[1], a[0], a[1]);      // lo along H
                        swt_fma2<true>(g.lo[t], x[2], x[3], a[2], a[3]);
                        swt_fma2<true>(g.hi[t], x[0], x[1], d[0], d[1]);      // hi along H
                        swt_fma2<true>(g.hi[t], x[2], x[3], d[2], d[3]);
                    }
                } else {
#pragma unroll
                    for (int v = 0; v < 4; ++v) {
                        float sa = 0.f, sd = 0.f;
#pragma unroll
                        for (int t = 0; t < F; ++t) {
                            const float x = w[m + F - 1 - t][v];
                            sa += g.lo[t] * x;                  // lo along H
                            sd += g.hi[t] * x;                  // hi along H
                        }
                        a[v] = sa, d[v] = sd;
                    }
                }
                const int gr = row_g0 + o0 + S * m;
                if (gr < g.H) {
                    // hl (lo along W): cA (LL) = plane 0, cH 'da' (LH) = plane 1; hh: cV 'ad' (HL) = plane 2, cD (HH) = plane 3
                    float *o = out_plane + (half ? 2 * plane : 0) + static_cast<size_t>(gr) * g.W + gc;
                    if constexpr (ALIGNED) {
                        store.vec4(o, a);
                        store.vec4(o + plane, d);
                    } else {
                        store(o, a, n);
                        store(o + plane, d, n);
                    }
                }
            }
        }
    }
}

// Sliding form of the last level's vertical pass (swt_vs_form): a unit is 4 columns x kVsR output rows of one residue class of
// ONE sub-band (band = 2 * (hh ? 1 : 0) + (dec_hi along H ? 1 : 0) = its output plane).  The unit walks its
// kVsR + F - 1 source rows top to bottom through a register window of F rows: every row is loaded once per kVsR outputs
// whatever F is (the blocked form above re-loads (R + F - 1) / R rows per output with R = 2 for the 8-tap filters: 4.5
// loads and 36 bytes of shared-memory reads per pixel), the output pointer advances by one image row per step instead
// of being rebuilt from (row, column) for each of the unit's stores (20 of the blocked form's 36 instructions per pixel
// were address arithmetic, db4 level 1), and one band per unit keeps window + taps + accumulators at F * 4 + F + 4
// registers, so the 8-tap kernels fit the 64-register budget of four 256-thread CTAs per SM.
constexpr int kVsR = 8;

template <int F, int S, bool ALIGNED, typename Store>
__host__ __device__ __forceinline__ void swt_vpass_final_slide(const SwtGeom &g, const float *hl, const float *hh, int stride,
                                                               float *out_plane, int row_g0, int col_g0, int ncg,
                                                               uint32_t magic, int tid, int nthreads, Store store) {
    constexpr int R = kVsR;
    const int nblk = g.TH / (S * R);
    const uint32_t units = 4u * static_cast<uint32_t>(ncg) * S * nblk;
    const size_t plane = static_cast<size_t>(g.H) * g.W;
    const int step = S * stride;
    const size_t ostep = static_cast<size_t>(S) * g.W;
#pragma unroll 1
    for (uint32_t u = tid; u < units; u += nthreads) {
        const int rest = static_cast<int>(swt_div(u, magic));
        const int cg = static_cast<int>(u) - rest * ncg;
        const int band = rest & 3, rb = rest >> 2;
        const int rho = rb % S, b = rb / S;
        const int o0 = rho + S * R * b;                     // first tile-local output row of the unit
        const int gc = col_g0 + 4 * cg;
        const int rows_left = g.H - (row_g0 + o0);          // output m exists iff S * m < rows_left
        if (gc >= g.W || rows_left <= 0) continue;
        const int n = g.W - gc >= 4 ? 4 : g.W - gc;          // W is even: n is 4 or 2
        const float *p = ((band & 2) ? hh : hl) + o0 * stride + 4 * cg;
        // hl (lo along W): cA (LL) = plane 0, cH 'da' (LH) = plane 1; hh: cV 'ad' (HL) = plane 2, cD (HH) = plane 3
        float *o = out_plane + band * plane + static_cast<size_t>(row_g0 + o0) * g.W + gc;
        float f[F];                                          // this band's taps along H
#pragma unroll
        for (int t = 0; t < F; ++t) f[t] = (band & 1) ? g.hi[t] : g.lo[t];
        float win[F][4];
#pragma unroll
        for (int k = 0; k < F - 1; ++k) swt_ld_vec<4>(p + k * step, win[k]);
        p += (F - 1) * step;
#pragma unroll
        for (int m = 0; m < R; ++m) {
            swt_ld_vec<4>(p, win[(m + F - 1) % F]);
            p += step;
            float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int t = 0; t < F; ++t) {
                const float *x = win[(m + F - 1 - t) % F];
                swt_fma2<(F >= 6)>(f[t], x[0], x[1], a[0], a[1]);
                swt_fma2<(F >= 6)>(f[t], x[2], x[3], a[2], a[3]);
            }
            if (S * m < rows_left) {
                if constexpr (ALIGNED)
                    store.vec4(o, a);
                else
                    store(o, a, n);
            }
            o += ostep;
        }
    }
}

// ---------------------------------------------------------------------------------------------- register-window passes
// An intermediate level as ONE pass (swt_rw_form 2): a unit is 4 adjacent columns x kRwR output rows of one residue
// class mod S.  The unit walks its kRwR + F - 1 source rows top to bottom; each row is filtered horizontally in registers
// (aligned 128-bit shared loads, FFMA2 over pixel pairs) into a window of the last F filtered rows, and every new row
// completes one output row, which is filtered vertically straight out of that window.  The horizontal outputs never go
// to shared memory (the two-pass form above stores and re-loads a plane of them per level, with the unit -> (row,
// column) index arithmetic of two more sweeps), at the price of (kRwR + F - 1) / kRwR times the horizontal FMAs.
constexpr int kRwR = 8;

// Keeps the compiler from hoisting the shared loads of later rows of a (fully unrolled) unit above this point: without
// it ptxas front-loads every row of the unit and spills the window.
__host__ __device__ __forceinline__ void swt_rw_fence() {
#ifdef __CUDA_ARCH__
    asm volatile("" ::: "memory");
#endif
}

// h[v] = sum_t f[t] * row[j0 + v + S * (F/2 - t)], v = 0..3 (j0 % 4 == 0)
template <int F, int S>
__host__ __device__ __forceinline__ void swt_rw_hrow(const float *row, int j0, const float *f, float *h) {
    h[0] = h[1] = h[2] = h[3] = 0.f;
    if constexpr (S % 4 == 0) {                                  // every tap is an aligned 4-vector of its own
#pragma unroll
        for (int t = 0; t < F; ++t) {
            float x[4];
            swt_ld_vec<4>(row + j0 + S * (F / 2 - t), x);
            swt_fma2<true>(f[t], x[0], x[1], h[0], h[1]);
            swt_fma2<true>(f[t], x[2], x[3], h[2], h[3]);
        }
    } else {
        constexpr int omin = -S * (F / 2 - 1), omax = S * (F / 2);
        constexpr int amin = -(((-omin) + 3) / 4) * 4;           // omin floored to a multiple of 4 (omin <= 0)
        constexpr int nvec = (3 + omax - amin) / 4 + 1;
        float w[nvec * 4];
#pragma unroll
        for (int i = 0; i < nvec; ++i) swt_ld_vec<4>(row + j0 + amin + 4 * i, w + 4 * i);
#pragma unroll
        for (int t = 0; t < F; ++t) {
            const int o = S * (F / 2 - t) - amin;
            swt_fma2<true>(f[t], w[o], w[o + 1], h[0], h[1]);
            swt_fma2<true>(f[t], w[o + 2], w[o + 3], h[2], h[3]);
        }
    }
}

// Intermediate level: LL only, shared -> shared.  dst(i, j) for rows [r0, r1) and `ncg` column groups from 4 * c0g
// (rows past r1 are computed from clamped loads and dropped).
template <int F, int S>
__host__ __device__ __forceinline__ void swt_rw_ll(const SwtGeom &g, const float *src, float *dst, int stride, int r0, int r1,
                                                   int c0g, int ncg, uint32_t magic, int tid, int nthreads) {
    constexpr int R = kRwR;
    const int per_class = (r1 - r0 + S - 1) / S;
    const int nblk = (per_class + R - 1) / R;
    const uint32_t units = static_cast<uint32_t>(ncg) * S * nblk;
#pragma unroll 1
    for (uint32_t u = tid; u < units; u += nthreads) {
        const int rest = static_cast<int>(swt_div(u, magic));
        const int cg = static_cast<int>(u) - rest * ncg;
        const int rho = rest % S, b = rest / S;
        const int first = r0 + rho + S * R * b;                 // first output row of the unit
        const int j0 = 4 * (c0g + cg);
        float win[F][4];
#pragma unroll
        for (int k = 0; k < R + F - 1; ++k) {
            int rr = first - S * (F / 2 - 1) + S * k;
            rr = rr < g.RH - 1 ? rr : g.RH - 1;
            swt_rw_hrow<F, S>(src + rr * stride, j0, g.lo, win[k % F]);
            if (k >= F - 1) {
                const int m = k - (F - 1), i = first + S * m;
                float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int t = 0; t < F; ++t) {
                    const float *x = win[(m + F - 1 - t) % F];
                    swt_fma2<true>(g.lo[t], x[0], x[1], a[0], a[1]);
                    swt_fma2<true>(g.lo[t], x[2], x[3], a[2], a[3]);
                }
                if (i < r1) swt_st_vec<4>(dst + i * stride + j0, a);
            }
            swt_rw_fence();
        }
    }
}

// ---------------------------------------------------------------------------------------------- tile programs
// The per-CTA program is written once, as a sequence of phases handed to `exec`: on the device a phase runs as
// phase(threadIdx.x, blockDim.x) followed by __syncthreads(); the CPU simulator runs it for tid = 0..nthreads-1.
struct SwtTileId {
    int plane, ty, tx;
};

// valid column range of the approximation after `lvl` intermediate levels, as column groups of the staging buffer
__host__ __device__ __forceinline__ void swt_level_cols(const SwtGeom &g, int lvl, int &c0g, int &ncg) {
    const int span = (1 << lvl) - 1;
    const int cb = g.padL - g.left + span * (g.F / 2 - 1);
    const int ce = g.padL + g.TW + g.right - span * (g.F / 2);
    c0g = cb / 4;
    ncg = (ce + 3) / 4 - c0g;
}

// One program per (F, LEVEL): the pass form follows from them (swt_rw_form, swt_vs_form), so that each kernel is
// compiled and register-allocated for one form only.
template <int F, int LEVEL, typename Exec, typename Store, typename Ld>
__host__ __device__ __forceinline__ void swt_tile_program(const SwtGeom &g, const void *in, float *out, SwtTileId id,
                                                          float *smem, Exec exec, Store store, Ld ld) {
    constexpr int RW = swt_rw_form(F, LEVEL), VS = swt_vs_form(F, LEVEL);
    const size_t plane_px = static_cast<size_t>(g.H) * g.W;
    const void *in_plane = g.in_is_u8 ? static_cast<const void *>(static_cast<const uint8_t *>(in) + id.plane * plane_px)
                                      : static_cast<const void *>(static_cast<const float *>(in) + id.plane * plane_px);
    float *out_plane = out + static_cast<size_t>(id.plane) * 4 * plane_px;
    float *a = smem + kSwtGuard;
    float *b = smem + g.off_b;
    // float32 planes whose tile rows are 16-byte aligned and do not wrap in x are staged by the bulk-copy (TMA) engine,
    // one row per copy, completion on an mbarrier kept in the (otherwise unused) leading guard; everything else —
    // uint8 input (needs the /255 conversion), image-edge tiles — goes through the register path.
    // RW == 2 at level 2: the one register-window pass must END in buffer A (the two-pass last level needs the larger
    // buffer B for its horizontal outputs), so the tile is staged into B
    float *stage = (RW == 2 && LEVEL == 2) ? b : a;
    exec([&](int tid, int n) {
        if (g.in_is_u8 && g.u8_stage >= 1)
            swt_load_tile_u8<((F >= 6 && VS == 0) ? 4 : 2)>(g, static_cast<const uint8_t *>(in_plane), stage, id.ty, id.tx, tid, n, ld);
        else if (!ld.bulk_stage(g, in_plane, stage, smem, id.ty, id.tx, tid, n))
            swt_load_tile(g, in_plane, stage, id.ty, id.tx, tid, n, ld);
    });
    constexpr int hb = F / 2 - 1, ha = F / 2;          // halo of a dilation-1 step
    int vb = 0, ve = g.RH;                             // valid rows of the current approximation
    int c0g, ncg;
    // The intermediate levels leave the approximation in `cur` and the free buffer in `other`: a register-window level
    // is one pass that swaps them, a two-pass level filters cur -> other (horizontal) -> cur (vertical).
    float *cur = stage, *other = stage == a ? b : a;
    if constexpr (LEVEL >= 2) {
        swt_level_cols(g, 1, c0g, ncg);
        if constexpr (RW != 0) {
            vb += hb, ve -= ha;
            exec([&](int tid, int n) { swt_rw_ll<F, 1>(g, cur, other, g.RWp, vb, ve, c0g, ncg, g.m_lvl[0], tid, n); });
            float *t = cur;
            cur = other, other = t;
        } else {
            exec([&](int tid, int n) { swt_hpass<F, 1, false>(g, cur, g.RWp, other, nullptr, g.RWp, vb, ve, c0g, ncg, g.m_lvl[0], 0, 0, tid, n); });
            vb += hb, ve -= ha;
            exec([&](int tid, int n) { swt_vpass_ll<F, 1>(g, other, cur, g.RWp, vb, ve, c0g, ncg, g.m_lvl[0], tid, n); });
        }
    }
    if constexpr (LEVEL >= 3) {
        swt_level_cols(g, 2, c0g, ncg);
        if constexpr (RW != 0) {
            vb += 2 * hb, ve -= 2 * ha;
            exec([&](int tid, int n) { swt_rw_ll<F, 2>(g, cur, other, g.RWp, vb, ve, c0g, ncg, g.m_lvl[1], tid, n); });
            float *t = cur;
            cur = other, other = t;
        } else {
            exec([&](int tid, int n) { swt_hpass<F, 2, false>(g, cur, g.RWp, other, nullptr, g.RWp, vb, ve, c0g, ncg, g.m_lvl[1], 0, 0, tid, n); });
            vb += 2 * hb, ve -= 2 * ha;
            exec([&](int tid, int n) { swt_vpass_ll<F, 2>(g, other, cur, g.RWp, vb, ve, c0g, ncg, g.m_lvl[1], tid, n); });
        }
    }
    constexpr int S = 1 << (LEVEL - 1);
    const int twp = (g.TW + 3) / 4 * 4;
    float *hl = other, *hh = other + static_cast<size_t>(g.RHv) * twp;
    const int r0 = g.top - S * hb;
    exec([&](int tid, int n) {
        swt_hpass<F, S, true>(g, cur, g.RWp, hl, hh, twp, r0, r0 + g.RHv, g.padL / 4, twp / 4, g.m_lvl[LEVEL - 1], r0, g.padL, tid, n);
    });
    exec([&](int tid, int n) {
        if constexpr (VS != 0) {
            if ((g.W & 3) == 0)
                swt_vpass_final_slide<F, S, true>(g, hl, hh, twp, out_plane, id.ty * g.TH, id.tx * g.TW, twp / 4, g.m_lvl[LEVEL - 1], tid, n, store);
            else
                swt_vpass_final_slide<F, S, false>(g, hl, hh, twp, out_plane, id.ty * g.TH, id.tx * g.TW, twp / 4, g.m_lvl[LEVEL - 1], tid, n, store);
        } else {
            if ((g.W & 3) == 0)
                swt_vpass_final<F, S, true>(g, hl, hh, twp, out_plane, id.ty * g.TH, id.tx * g.TW, twp / 4, g.m_lvl[LEVEL - 1], tid, n, store);
            else
                swt_vpass_final<F, S, false>(g, hl, hh, twp, out_plane, id.ty * g.TH, id.tx * g.TW, twp / 4, g.m_lvl[LEVEL - 1], tid, n, store);
        }
    });
}

// Generic fallback (any even F <= 20, level <= 4): runtime taps, one pixel per work item, three buffers.
__host__ __device__ __forceinline__ void swt_gen_hpass(const SwtGeom &g, const float *src, float *dlo, float *dhi, int S,
                                                       int r0, int r1, int c0, int c1, int tid, int n) {
    const int w = c1 - c0;
    for (int idx = tid; idx < (r1 - r0) * w; idx += n) {
        const int i = r0 + idx / w, j = c0 + idx % w;
        float a = 0.f, d = 0.f;
        for (int t = 0; t < g.F; ++t) {
            const float x = src[i * g.RWp + j + S * (g.F / 2 - t)];
            a += g.lo[t] * x;
            d += g.hi[t] * x;
        }
        dlo[i * g.RWp + j] = a;
        if (dhi) dhi[i * g.RWp + j] = d;
    }
}
__host__ __device__ __forceinline__ void swt_gen_vpass_ll(const SwtGeom &g, const float *tlo, float *dst, int S, int r0,
                                                          int r1, int c0, int c1, int tid, int n) {
    const int w = c1 - c0;
    for (int idx = tid; idx < (r1 - r0) * w; idx += n) {
        const int i = r0 + idx / w, j = c0 + idx % w;
        float a = 0.f;
        for (int t = 0; t < g.F; ++t) a += g.lo[t] * tlo[(i + S * (g.F / 2 - t)) * g.RWp + j];
        dst[i * g.RWp + j] = a;
    }
}
__host__ __device__ __forceinline__ void swt_gen_vpass_final(const SwtGeom &g, const float *tlo, const float *thi,
                                                             float *out_plane, int S, int row_g0, int col_g0, int tid,
                                                             int n) {
    const size_t plane = static_cast<size_t>(g.H) * g.W;
    for (int idx = tid; idx < g.TH * g.TW; idx += n) {
        const int i = g.top + idx / g.TW, j = g.padL + idx % g.TW;
        const int gr = row_g0 + i, gc = col_g0 + j;
        if (gr >= g.H || gc >= g.W) continue;
        float a = 0.f, b = 0.f, c = 0.f, d = 0.f;
        for (int t = 0; t < g.F; ++t) {
            const float xl = tlo[(i + S * (g.F / 2 - t)) * g.RWp + j], xh = thi[(i + S * (g.F / 2 - t)) * g.RWp + j];
            a += g.lo[t] * xl, b += g.hi[t] * xl, c += g.lo[t] * xh, d += g.hi[t] * xh;
        }
        float *o = out_plane + static_cast<size_t>(gr) * g.W + gc;
        o[0] = a, o[plane] = b, o[2 * plane] = c, o[3 * plane] = d;
    }
}

template <typename Exec, typename Ld>
__host__ __device__ __forceinline__ void swt_generic_program(const SwtGeom &g, const void *in, float *out, SwtTileId id,
                                                             float *smem, Exec exec, Ld ld) {
    const size_t plane_px = static_cast<size_t>(g.H) * g.W;
    const void *in_plane = g.in_is_u8 ? static_cast<const void *>(static_cast<const uint8_t *>(in) + id.plane * plane_px)
                                      : static_cast<const void *>(static_cast<const float *>(in) + id.plane * plane_px);
    float *out_plane = out + static_cast<size_t>(id.plane) * 4 * plane_px;
    const size_t buf_floats = static_cast<size_t>(g.RH) * g.RWp + 2 * kSwtGuard;
    float *x = smem + kSwtGuard, *tlo = x + buf_floats, *thi = tlo + buf_floats;
    exec([&](int tid, int n) { swt_load_tile(g, in_plane, x, id.ty, id.tx, tid, n, ld); });
    const int hb = g.F / 2 - 1, ha = g.F / 2;
    int vb = 0, ve = g.RH, cb = g.padL - g.left, ce = g.padL + g.TW + g.right;
    for (int lv = 1; lv < g.level; ++lv) {
        const int S = 1 << (lv - 1);
        cb += S * hb, ce -= S * ha;
        exec([&](int tid, int n) { swt_gen_hpass(g, x, tlo, nullptr, S, vb, ve, cb, ce, tid, n); });
        vb += S * hb, ve -= S * ha;
        exec([&](int tid, int n) { swt_gen_vpass_ll(g, tlo, x, S, vb, ve, cb, ce, tid, n); });
    }
    const int S = 1 << (g.level - 1);
    exec([&](int tid, int n) { swt_gen_hpass(g, x, tlo, thi, S, vb, ve, g.padL, g.padL + g.TW, tid, n); });
    exec([&](int tid, int n) {
        swt_gen_vpass_final(g, tlo, thi, out_plane, S, id.ty * g.TH - g.top, id.tx * g.TW - g.padL, tid, n);
    });
}

}  // namespace b200
