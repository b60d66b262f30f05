// SURVEY §8 (f3): the pixel step in front of the SWT, on the device.
//
//   b200_resize_u8  <- BaseWaveletTransform.fix_size            /root/reference/main/transforms/custom_transforms.py:132-139
//                      (PIL `image.resize((new_w, new_h), resample=Image.BICUBIC)` up to a multiple of 2^level: 518 -> 520
//                      for levels 2-3) and the PIL resize behind torchvision's Resize in the eval transforms
//                      (config/transform/NAME.yaml: Resize(256) -> CenterCrop(224), bilinear with antialiasing).
//   b200_resize_crop_u8 <- that eval transform, Resize(size) -> CenterCrop(crop) of torchvision on every PIL image of a
//                      batch, for a ragged batch of decoded HWC images in one launch: only the crop window of each resized
//                      image is computed (resize_crop_kernel below).
//   b200_resize_random_crop_u8 <- the training transform, Resize(size) -> RandomResizedCrop(crop) -> RandomHorizontalFlip of
//                      torchvision on every PIL image of a batch, with the boxes and flips drawn by the caller: two launches
//                      of resize_crop_kernel, the box of each resized image (a window of the first resize), then a full
//                      resize of that box to the crop size stored mirrored where the flip is drawn.
//
// The arithmetic is Pillow's (third-party, pinned `pillow==8.2.0` in requirements.txt:5; src/libImaging/Resample.c, the
// 8-bit path, unchanged through the 12.x release installed here), restated:
//   * per output coordinate, the window [xmin, xmin + n) of input samples and its weights
//       w(x) = filter((x + xmin - center + 0.5) / filterscale), center = (xx + 0.5) * in/out, support = filter support *
//       max(in/out, 1), normalised to sum 1 in double precision (precompute_coeffs), then rounded to 22-bit fixed point
//       (normalize_coeffs_8bpc);
//   * a horizontal pass into a uint8 intermediate, then a vertical pass (ImagingResampleInner: a pass is skipped when
//       its size does not change), each output = clip8((2^21 + sum pixel * weight) >> 22).
// The tables are built on the host in the same double arithmetic (a few hundred entries) and copied to the caller's
// workspace; the two kernels are one thread per 4 output bytes, HBM-bound at ~2 bytes moved per pixel and pass.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <tuple>
#include <vector>

#include "common.cuh"

namespace b200 {

constexpr int kResizePrecisionBits = 32 - 8 - 2;
constexpr int kResizeMaxTaps = 64;

static double resize_filter(int filter, double x) {
    if (x < 0.0) x = -x;
    if (filter == B200_RESIZE_BILINEAR) return x < 1.0 ? 1.0 - x : 0.0;
    const double a = -0.5;                                   // bicubic, Keys a = -0.5 (Resample.c: bicubic_filter)
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}
static double resize_support(int filter) { return filter == B200_RESIZE_BILINEAR ? 1.0 : 2.0; }

static int resize_ksize(int in_size, int out_size, int filter) {
    double filterscale = static_cast<double>(in_size) / out_size;
    if (filterscale < 1.0) filterscale = 1.0;
    return static_cast<int>(std::ceil(resize_support(filter) * filterscale)) * 2 + 1;
}

// Resample.c precompute_coeffs + normalize_coeffs_8bpc: bounds[2*xx] = first input sample, bounds[2*xx+1] = count,
// kk[xx*ksize + x] = 22-bit fixed-point weights (zero beyond the count).  Every output coordinate's entry depends on that
// coordinate alone, so the rows [first, first + count) of the table are built by themselves (a crop window); count < 0:
// the whole axis.
static void resize_coeffs(int in_size, int out_size, int filter, int ksize, std::vector<int> &bounds, std::vector<int> &kk,
                          int first = 0, int count = -1) {
    if (count < 0) count = out_size;
    const double scale = static_cast<double>(in_size) / out_size;
    const double filterscale = scale < 1.0 ? 1.0 : scale;
    const double support = resize_support(filter) * filterscale;
    bounds.assign(static_cast<size_t>(count) * 2, 0);
    kk.assign(static_cast<size_t>(count) * ksize, 0);
    std::vector<double> k(ksize);
    for (int i = 0; i < count; ++i) {
        const int xx = first + i;
        const double center = (xx + 0.5) * scale;
        const double ss = 1.0 / filterscale;
        double ww = 0.0;
        int xmin = static_cast<int>(center - support + 0.5);
        if (xmin < 0) xmin = 0;
        int xmax = static_cast<int>(center + support + 0.5);
        if (xmax > in_size) xmax = in_size;
        xmax -= xmin;
        for (int x = 0; x < xmax; ++x) {
            const double w = resize_filter(filter, (x + xmin - center + 0.5) * ss);
            k[x] = w;
            ww += w;
        }
        for (int x = 0; x < xmax; ++x) {
            if (ww != 0.0) k[x] /= ww;
            const double v = k[x] * (1 << kResizePrecisionBits);
            kk[static_cast<size_t>(i) * ksize + x] = v < 0 ? static_cast<int>(-0.5 + v) : static_cast<int>(0.5 + v);
        }
        bounds[2 * i] = xmin, bounds[2 * i + 1] = xmax;
    }
}

__device__ __forceinline__ uint32_t resize_clip8(int acc) {
    const int v = acc >> kResizePrecisionBits;
    return static_cast<uint32_t>(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// Launch shape of both passes: blockDim = (column groups of 4 output bytes, kResizeRows rows); one CTA covers
// kResizeRows consecutive rows so that the weight rows it reads stay in L1; no division anywhere on the device.
constexpr int kResizeRows = 4;

// out[row][xx] from in[row][xmin .. xmin + n): one thread = 4 adjacent output columns of one row
__global__ void __launch_bounds__(1024) resize_h_kernel(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, long long rows,
                                                        int W, int Wout, int ksize, const int2 *__restrict__ bounds,
                                                        const int *__restrict__ kk) {
    const long long row = static_cast<long long>(blockIdx.x) * kResizeRows + threadIdx.y;
    if (row >= rows) return;
    const uint8_t *src = in + row * W;
    uint8_t *dst_row = out + row * Wout;
    for (int x0 = 4 * threadIdx.x; x0 < Wout; x0 += 4 * blockDim.x) {
        uint32_t px[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            px[e] = 0;
            const int xx = x0 + e;
            if (xx < Wout) {
                const int2 b = __ldg(bounds + xx);
                const int *k = kk + static_cast<size_t>(xx) * ksize;
                int acc = 1 << (kResizePrecisionBits - 1);
                for (int x = 0; x < b.y; ++x) acc += static_cast<int>(__ldg(src + b.x + x)) * __ldg(k + x);
                px[e] = resize_clip8(acc);
            }
        }
        uint8_t *dst = dst_row + x0;
        if (x0 + 3 < Wout && (reinterpret_cast<uintptr_t>(dst) & 3) == 0) {
            *reinterpret_cast<uint32_t *>(dst) = px[0] | (px[1] << 8) | (px[2] << 16) | (px[3] << 24);
        } else {
            for (int e = 0; e < 4 && x0 + e < Wout; ++e) dst[e] = static_cast<uint8_t>(px[e]);
        }
    }
}

// out[p][yy][x] from in[p][ymin .. ymin + n)[x]: one thread = 4 adjacent columns of one output row; grid = (row blocks, planes)
__global__ void __launch_bounds__(1024) resize_v_kernel(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int H, int Hout,
                                                        int W, int ksize, const int2 *__restrict__ bounds,
                                                        const int *__restrict__ kk) {
    const int yy = static_cast<int>(blockIdx.x) * kResizeRows + threadIdx.y;
    if (yy >= Hout) return;
    const size_t p = blockIdx.y;
    const int2 b = __ldg(bounds + yy);
    const int *k = kk + static_cast<size_t>(yy) * ksize;
    const uint8_t *src_row = in + (p * H + b.x) * W;
    uint8_t *dst_row = out + (p * Hout + yy) * W;
    for (int x0 = 4 * threadIdx.x; x0 < W; x0 += 4 * blockDim.x) {
        const uint8_t *src = src_row + x0;
        const bool vec = x0 + 3 < W && (reinterpret_cast<uintptr_t>(src) & 3) == 0 && (W & 3) == 0;
        int acc[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[e] = 1 << (kResizePrecisionBits - 1);
        for (int y = 0; y < b.y; ++y) {
            const int w = __ldg(k + y);
            const uint8_t *r = src + static_cast<size_t>(y) * W;
            if (vec) {
                const uint32_t v = __ldg(reinterpret_cast<const uint32_t *>(r));
                acc[0] += static_cast<int>(v & 0xffu) * w, acc[1] += static_cast<int>((v >> 8) & 0xffu) * w;
                acc[2] += static_cast<int>((v >> 16) & 0xffu) * w, acc[3] += static_cast<int>(v >> 24) * w;
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (x0 + e < W) acc[e] += static_cast<int>(__ldg(r + e)) * w;
            }
        }
        uint8_t *dst = dst_row + x0;
        if (vec && (reinterpret_cast<uintptr_t>(dst) & 3) == 0) {
            *reinterpret_cast<uint32_t *>(dst) =
                resize_clip8(acc[0]) | (resize_clip8(acc[1]) << 8) | (resize_clip8(acc[2]) << 16) | (resize_clip8(acc[3]) << 24);
        } else {
            for (int e = 0; e < 4 && x0 + e < W; ++e) dst[e] = static_cast<uint8_t>(resize_clip8(acc[e]));
        }
    }
}

static dim3 resize_block(int width) {
    const int groups = (width + 3) / 4;
    const int tx = groups >= 256 ? 256 : (groups + 31) / 32 * 32;
    return dim3(tx, kResizeRows);
}

// ---- fused form: one CTA per 32 x 128 output tile of one plane.  The input window of the tile is staged once in shared
// memory (aligned 32-bit loads; a row of a 518-wide plane starts on any byte, so every staged row keeps its own byte
// offset), the horizontal pass writes the uint8 intermediate of exactly the rows the tile's vertical windows need into
// shared memory, the vertical pass writes the tile.  Same integer arithmetic per pixel as the two-kernel form (and as
// Pillow), but the intermediate never reaches HBM: 1 byte read + 1 byte written per pixel.  An axis whose size does not
// change runs with identity tables (window 1, weight 2^22: (2^21 + p * 2^22) >> 22 == p exactly).
constexpr int kRzTH = 32, kRzTW = 128, kRzThreads = 256;

struct ResizeFusedArgs {
    const uint8_t *in;
    uint8_t *out;
    const int2 *hb, *vb;
    const int *hk, *vk;
    int H, W, Hout, Wout, ksh, ksv;
    int max_rows, max_words;          // staged rows / 32-bit words per staged row (upper bounds over all tiles)
    long long plane0;                 // first plane of this launch (gridDim.z <= 65535 planes per launch)
};

// KSH / KSV > 0: the window length is a compile-time constant (tables are zero beyond each window's count, so the
// fixed-length sums are the same integers), taps unrolled and the thread's weights held in registers; 0: run-time counts.
template <int KSH, int KSV>
__global__ void __launch_bounds__(kRzThreads) resize_fused_kernel(const __grid_constant__ ResizeFusedArgs a) {
    extern __shared__ __align__(16) unsigned char rz_smem[];
    int2 *s_hb = reinterpret_cast<int2 *>(rz_smem);                                          // [kRzTW]
    int2 *s_vb = s_hb + kRzTW;                                                               // [kRzTH]
    uint32_t *s_in = reinterpret_cast<uint32_t *>(s_vb + kRzTH);                             // [max_rows][max_words]
    int *s_hk = reinterpret_cast<int *>(s_in + a.max_rows * a.max_words);                    // [kRzTW][ksh]
    int *s_vk = s_hk + kRzTW * a.ksh;                                                        // [kRzTH][ksv]
    int *s_off = s_vk + kRzTH * a.ksv;                                                       // [max_rows] byte offset of column xlo in the staged row
    uint8_t *s_tmp = reinterpret_cast<uint8_t *>(s_off + a.max_rows);                        // [max_rows + pad][kRzTW]
    const int tid = static_cast<int>(threadIdx.x);
    const int x0 = static_cast<int>(blockIdx.x) * kRzTW, y0 = static_cast<int>(blockIdx.y) * kRzTH;
    const size_t p = static_cast<size_t>(a.plane0) + blockIdx.z;
    const int nx = a.Wout - x0 < kRzTW ? a.Wout - x0 : kRzTW, ny = a.Hout - y0 < kRzTH ? a.Hout - y0 : kRzTH;
    // windows are monotone in the output coordinate: the tile's input window is [first.x, last.x + last.y)
    const int2 bx0 = __ldg(a.hb + x0), bx1 = __ldg(a.hb + x0 + nx - 1), by0 = __ldg(a.vb + y0), by1 = __ldg(a.vb + y0 + ny - 1);
    const int xlo = bx0.x, cols = bx1.x + bx1.y - bx0.x, ylo = by0.x, rows = by1.x + by1.y - by0.x;
    const int ksh = KSH ? KSH : a.ksh, ksv = KSV ? KSV : a.ksv;
    for (int i = tid; i < kRzTW * ksh; i += kRzThreads) s_hk[i] = i < nx * ksh ? __ldg(a.hk + static_cast<size_t>(x0) * ksh + i) : 0;
    for (int i = tid; i < kRzTH * ksv; i += kRzThreads) s_vk[i] = i < ny * ksv ? __ldg(a.vk + static_cast<size_t>(y0) * ksv + i) : 0;
    for (int i = tid; i < kRzTW; i += kRzThreads) s_hb[i] = i < nx ? __ldg(a.hb + x0 + i) : make_int2(xlo, 0);
    for (int i = tid; i < kRzTH; i += kRzThreads) s_vb[i] = i < ny ? __ldg(a.vb + y0 + i) : make_int2(ylo, 0);
    // stage: warp w takes rows w, w + 8, ...; its lanes the aligned words of the row
    const size_t plane_off = p * a.H * a.W;
    const int lane = tid & 31, warp = tid >> 5;
    for (int r = warp; r < rows; r += kRzThreads / 32) {
        const size_t base = plane_off + static_cast<size_t>(ylo + r) * a.W + xlo;
        const uint32_t *src = reinterpret_cast<const uint32_t *>(a.in + (base & ~static_cast<size_t>(3)));
        const int words = (static_cast<int>(base & 3) + cols + 3) >> 2;
        for (int w = lane; w < words; w += 32) s_in[r * a.max_words + w] = __ldg(src + w);
        if (lane == 0) s_off[r] = static_cast<int>(base & 3) - xlo;
    }
    __syncthreads();
    // horizontal pass: thread = one output column (weights in registers when KSH > 0), rows 2 apart
    {
        const int xx = tid & (kRzTW - 1);
        const int2 b = s_hb[xx];
        const int *k = s_hk + xx * ksh;
        int kr[KSH ? KSH : 1];
        if constexpr (KSH > 0) {
#pragma unroll
            for (int x = 0; x < KSH; ++x) kr[x] = k[x];
        }
        if (xx < nx) {
            for (int r = tid / kRzTW; r < rows; r += kRzThreads / kRzTW) {
                const uint8_t *row = reinterpret_cast<const uint8_t *>(s_in + r * a.max_words) + s_off[r] + b.x;
                int acc = 1 << (kResizePrecisionBits - 1);
                if constexpr (KSH > 0) {
#pragma unroll
                    for (int x = 0; x < KSH; ++x) acc += static_cast<int>(row[x]) * kr[x];
                } else {
                    for (int x = 0; x < b.y; ++x) acc += static_cast<int>(row[x]) * k[x];
                }
                s_tmp[r * kRzTW + xx] = static_cast<uint8_t>(resize_clip8(acc));
            }
        }
    }
    __syncthreads();
    // vertical pass: thread = 4 adjacent columns, rows 8 apart
    {
        const int g4 = 4 * (tid & 31);
        if (g4 < nx) {
            for (int yy = tid >> 5; yy < ny; yy += kRzThreads / 32) {
                const int2 b = s_vb[yy];
                const int *k = s_vk + yy * ksv;
                const uint8_t *col = s_tmp + (b.x - ylo) * kRzTW + g4;
                int acc[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) acc[e] = 1 << (kResizePrecisionBits - 1);
                auto tap = [&](int y) {
                    const uint32_t v = *reinterpret_cast<const uint32_t *>(col + y * kRzTW);
                    const int w = k[y];
                    acc[0] += static_cast<int>(v & 0xffu) * w, acc[1] += static_cast<int>((v >> 8) & 0xffu) * w;
                    acc[2] += static_cast<int>((v >> 16) & 0xffu) * w, acc[3] += static_cast<int>(v >> 24) * w;
                };
                if constexpr (KSV > 0) {
#pragma unroll
                    for (int y = 0; y < KSV; ++y) tap(y);
                } else {
                    for (int y = 0; y < b.y; ++y) tap(y);
                }
                uint8_t *dst = a.out + (p * a.Hout + y0 + yy) * a.Wout + x0 + g4;
                if (g4 + 3 < nx && (reinterpret_cast<uintptr_t>(dst) & 3) == 0) {
                    *reinterpret_cast<uint32_t *>(dst) =
                        resize_clip8(acc[0]) | (resize_clip8(acc[1]) << 8) | (resize_clip8(acc[2]) << 16) | (resize_clip8(acc[3]) << 24);
                } else {
                    for (int e = 0; e < 4 && g4 + e < nx; ++e) dst[e] = static_cast<uint8_t>(resize_clip8(acc[e]));
                }
            }
        }
    }
}

using resize_fused_fn = void (*)(const ResizeFusedArgs);
static resize_fused_fn resize_pick_fused(int ksh, int ksv) {
    if (ksh == 5 && ksv == 5) return resize_fused_kernel<5, 5>;      // fix_size: bicubic, both axes grow
    if (ksh == 1 && ksv == 5) return resize_fused_kernel<1, 5>;      // one axis unchanged (identity window)
    if (ksh == 5 && ksv == 1) return resize_fused_kernel<5, 1>;
    return resize_fused_kernel<0, 0>;
}

// upper bounds of the input window of any tile: max over tiles of (last.x + last.y - first.x)
static int resize_max_window(const std::vector<int> &bounds, int out_size, int tile) {
    int m = 1;
    for (int t0 = 0; t0 < out_size; t0 += tile) {
        const int t1 = (t0 + tile < out_size ? t0 + tile : out_size) - 1;
        const int span = bounds[2 * t1] + bounds[2 * t1 + 1] - bounds[2 * t0];
        if (span > m) m = span;
    }
    return m;
}
static void resize_identity(int size, std::vector<int> &bounds, std::vector<int> &kk) {
    bounds.resize(static_cast<size_t>(size) * 2);
    kk.assign(size, 1 << kResizePrecisionBits);
    for (int i = 0; i < size; ++i) bounds[2 * i] = i, bounds[2 * i + 1] = 1;
}

struct ResizeLayout {
    int ksh, ksv;
    size_t off_tmp, off_hb, off_hk, off_vb, off_vk, bytes;
};
static ResizeLayout resize_layout(long long planes, int H, int W, int Hout, int Wout, int filter) {
    ResizeLayout l{};
    const bool need_h = Wout != W, need_v = Hout != H;
    l.ksh = need_h ? resize_ksize(W, Wout, filter) : 1;         // an unchanged axis runs with identity tables in the fused form
    l.ksv = need_v ? resize_ksize(H, Hout, filter) : 1;
    size_t o = 0;
    auto take = [&](size_t n) {
        const size_t at = o;
        o = round_up<size_t>(o + n, 256);
        return at;
    };
    l.off_tmp = take(need_h && need_v ? static_cast<size_t>(planes) * H * Wout : 0);      // two-kernel form only
    l.off_hb = take(static_cast<size_t>(Wout) * 8);
    l.off_hk = take(static_cast<size_t>(Wout) * l.ksh * 4);
    l.off_vb = take(static_cast<size_t>(Hout) * 8);
    l.off_vk = take(static_cast<size_t>(Hout) * l.ksv * 4);
    l.bytes = o;
    return l;
}

// ---- resize + crop of a ragged batch: torchvision Resize(size) -> CenterCrop(crop) (b200_resize_crop_u8) and the two
// resamplings of Resize(size) -> RandomResizedCrop(crop) -> RandomHorizontalFlip (b200_resize_random_crop_u8) on PIL
// images.  A crop of a resize is the resize evaluated inside the crop window: output (y, x) of image i is resized sample
// (top_i + y, left_i + x), whose window and weights are those rows of the full-axis tables.  So the host builds just the
// Hc_i (Wc_i) table rows of each axis, shared by every image with the same (input size, resized size, crop origin, crop
// size), and one launch covers the batch: image i's planar [C][Hc_i][Wc_i] output at its own byte offset, one CTA per
// kRcTH x kRcTW tile of one channel.  The CTA walks its tile in sub-blocks of sub_h x sub_w output samples, chosen per
// image on the host as the one that stages the fewest source bytes per output sample within kRcSmemBudget: one sub-block
// (the whole tile) for reductions up to ~2x, tall narrow ones for large photos (a short sub-block would recompute the
// horizontal pass of its vertical window for every few output rows).  Per sub-block: stage channel c of the source window in
// shared memory (aligned 32-bit loads of the interleaved HWC rows, de-interleaved while stored), horizontal pass into a
// shared uint8 intermediate, vertical pass, store.  The grid is one-dimensional: images in descending order of staged
// bytes (a large photo's tiles start in the first wave instead of trailing behind the small images), then tiles, then
// channels, so the C CTAs of a tile are adjacent and the interleaved source words they all load come from L2 after the
// first.  Images may have different output sizes, so each descriptor records its first CTA and a CTA finds its descriptor
// by a binary search over them.  With `flip` set the vertical pass stores output column x at Wc - 1 - x
// (RandomHorizontalFlip): the output is mirrored, never the source, as Pillow's weight tables need not be bit-symmetric.
constexpr int kRcTH = 32, kRcTW = 128, kRcThreads = 256;
constexpr int kRcSmemBudget = 32 * 1024;

struct CropDesc {
    long long in_off;         // byte offset of the image in `in`
    long long out_off;        // byte offset of the image's planar [C][Hc][Wc] output in `out`
    int cta0;                 // first CTA of the image (descriptors in launch order: ascending)
    int W;                    // input width (row pitch W * C bytes)
    int Hc, Wc, flip;         // output size; flip: output column x is stored at Wc - 1 - x
    int hb, hk, ksh;          // tables (int index into the table block): bounds / weights of crop column 0, taps
    int vb, vk, ksv;          // the same for crop row 0
    int sub_h, sub_w;         // sub-block of the tile (powers of two dividing kRcTH / kRcTW; sub_w >= 4)
    int max_rows, stride;     // staged source rows / bytes per staged row, upper bounds over the image's sub-blocks
};

__host__ __device__ inline size_t crop_smem_bytes(int sub_h, int sub_w, int ksh, int ksv, int max_rows, int stride) {
    return static_cast<size_t>(sub_w + sub_h) * 8 + static_cast<size_t>(ksh * sub_w + sub_h * ksv) * 4 +
           static_cast<size_t>(max_rows) * (stride + sub_w);
}

// kGeneral = false: every crop of the launch is Hc_all x Wc_all and none is mirrored (every eval launch).  That form is
// the launch-argument kernel the eval path always had: the descriptor search, the shared-memory stash of the store
// operands and the mirrored stores are compiled out, so the eval transform keeps its speed.
template <int C, bool kGeneral>
__global__ void __launch_bounds__(kRcThreads, 4) resize_crop_kernel(const uint8_t *__restrict__ in, uint8_t *__restrict__ out,
                                                                 const CropDesc *__restrict__ descs, const int *__restrict__ tab,
                                                                 int n, int Hc_all, int Wc_all) {
    extern __shared__ __align__(16) unsigned char rc_smem[];
    const int cta = static_cast<int>(blockIdx.x);
    int Hc = Hc_all, Wc = Wc_all, rank, c, bx, by;
    if (!kGeneral || Hc_all > 0) {
        // one crop size for the launch: the tile and channel follow from the CTA index and the launch arguments alone,
        // without waiting for the descriptor
        const int tiles_x = (Wc + kRcTW - 1) / kRcTW, tiles_y = (Hc + kRcTH - 1) / kRcTH;
        const unsigned t = static_cast<unsigned>(cta) / C, tt = t / tiles_x;
        c = static_cast<int>(cta - t * C), bx = static_cast<int>(t - tt * tiles_x);
        by = static_cast<int>(tt % tiles_y), rank = static_cast<int>(tt / tiles_y);
    } else {
        // the last descriptor whose first CTA is <= cta lies in [lo, lo + span): each warp narrows it 32-fold per step
        // (its lanes probe 32 evenly spaced descriptors at once), two dependent loads for up to 1024 descriptors
        const int lane = static_cast<int>(threadIdx.x) & 31;
        int lo = 0, span = n;
        while (span > 1) {
            const int step = (span + 31) >> 5, probe = lo + lane * step;
            const unsigned le = __ballot_sync(0xffffffffu, probe < lo + span && __ldg(&descs[probe].cta0) <= cta);
            const int k = 31 - __clz(le);                                // lane 0 holds: descs[lo].cta0 <= cta
            lo += k * step, span = min(step, span - k * step);
        }
        rank = lo, Hc = descs[lo].Hc, Wc = descs[lo].Wc;
        const int tiles_x = (Wc + kRcTW - 1) / kRcTW;
        const unsigned local = static_cast<unsigned>(cta - descs[lo].cta0), t = local / C, tt = t / tiles_x;
        c = static_cast<int>(local - t * C), bx = static_cast<int>(t - tt * tiles_x), by = static_cast<int>(tt);
    }
    const CropDesc &d = descs[rank];
    const int2 *hb = reinterpret_cast<const int2 *>(tab + d.hb), *vb = reinterpret_cast<const int2 *>(tab + d.vb);
    const int *hk = tab + d.hk, *vk = tab + d.vk;
    const int sh = d.sub_h, sw = d.sub_w, ksh = d.ksh, ksv = d.ksv, stride = d.stride, max_rows = d.max_rows;
    const size_t in_off = static_cast<size_t>(d.in_off), pitch = static_cast<size_t>(d.W) * C;
    int2 *s_hb = reinterpret_cast<int2 *>(rc_smem);                     // [sw] (first sample - xlo, count)
    int2 *s_vb = s_hb + sw;                                              // [sh] (first row - ylo, count)
    int *s_hk = reinterpret_cast<int *>(s_vb + sh);                      // [ksh][sw]: tap-major, lanes read adjacent words
    int *s_vk = s_hk + ksh * sw;                                         // [sh][ksv]
    uint8_t *s_in = reinterpret_cast<uint8_t *>(s_vk + sh * ksv);        // [max_rows][stride] channel c of the window
    uint8_t *s_tmp = s_in + max_rows * stride;                           // [max_rows][sw] horizontal pass
    const int tid = static_cast<int>(threadIdx.x), lane = tid & 31, warp = tid >> 5;
    // general form: what only the stores need waits in shared memory, not in registers: the kernel is at its 64-register
    // cap (4 CTAs per SM), and values live across the staging and horizontal loops slow them down
    __shared__ uint8_t *s_out;
    __shared__ int s_wc, s_flip;
    if (kGeneral && tid == 0) s_out = out + d.out_off + static_cast<size_t>(c) * Hc * Wc, s_wc = Wc, s_flip = d.flip;
    const size_t plane_off = kGeneral ? 0 : static_cast<size_t>(d.out_off) + static_cast<size_t>(c) * Hc * Wc;
    const int x0 = bx * kRcTW, y0 = by * kRcTH;
    const int nx = Wc - x0 < kRcTW ? Wc - x0 : kRcTW, ny = Hc - y0 < kRcTH ? Hc - y0 : kRcTH;
    const int sw_log = __ffs(sw) - 1, ng = sw >> 2, ng_log = sw_log - 2;
    for (int sy = 0; sy < ny; sy += sh) {
        for (int sx = 0; sx < nx; sx += sw) {
            const int mh = ny - sy < sh ? ny - sy : sh, mw = nx - sx < sw ? nx - sx : sw;
            const int xa = x0 + sx, ya = y0 + sy;
            // windows are monotone in the output coordinate: the sub-block's window is [first.x, last.x + last.y)
            const int2 bx0 = __ldg(hb + xa), bx1 = __ldg(hb + xa + mw - 1), by0 = __ldg(vb + ya), by1 = __ldg(vb + ya + mh - 1);
            const int xlo = bx0.x, cols = bx1.x + bx1.y - xlo, ylo = by0.x, rows = by1.x + by1.y - ylo;
            __syncthreads();                                             // the previous sub-block is done with shared memory
            for (int i = tid; i < sw; i += kRcThreads) {
                const int2 b = i < mw ? __ldg(hb + xa + i) : make_int2(xlo, 0);
                s_hb[i] = make_int2(b.x - xlo, b.y);
            }
            for (int i = tid; i < sh; i += kRcThreads) {
                const int2 b = i < mh ? __ldg(vb + ya + i) : make_int2(ylo, 0);
                s_vb[i] = make_int2(b.x - ylo, b.y);
            }
            for (int i = tid; i < ksh * sw; i += kRcThreads) {
                const int t = i >> sw_log, j = i & (sw - 1);
                s_hk[i] = j < mw ? __ldg(hk + static_cast<size_t>(xa + j) * ksh + t) : 0;
            }
            for (int i = tid; i < sh * ksv; i += kRcThreads) s_vk[i] = i < mh * ksv ? __ldg(vk + static_cast<size_t>(ya) * ksv + i) : 0;
            // stage: warp w takes source rows w, w + 8, ...; its lanes the aligned words covering bytes
            // [xlo * C, (xlo + cols) * C) of the row, keeping the bytes of channel c
            const int nbytes = cols * C;
            for (int r = warp; r < rows; r += kRcThreads / 32) {
                const size_t start = in_off + static_cast<size_t>(ylo + r) * pitch + static_cast<size_t>(xlo) * C;
                const uint32_t *src = reinterpret_cast<const uint32_t *>(in + (start & ~static_cast<size_t>(3)));
                const int lead = static_cast<int>(start & 3), words = (lead + nbytes + 3) >> 2;
                uint8_t *dst = s_in + r * stride;
                for (int w = lane; w < words; w += 32) {
                    const uint32_t v = __ldg(src + w);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int p = 4 * w + e - lead;
                        if (p >= 0 && p < nbytes && p % C == c) dst[p / C] = static_cast<uint8_t>(v >> (8 * e));
                    }
                }
            }
            __syncthreads();
            // horizontal pass: thread = one output column of the sub-block, rows kRcThreads / sw apart
            {
                const int j = tid & (sw - 1);
                if (j < mw) {
                    const int2 b = s_hb[j];
                    for (int r = tid >> sw_log; r < rows; r += kRcThreads >> sw_log) {
                        const uint8_t *row = s_in + r * stride + b.x;
                        int acc = 1 << (kResizePrecisionBits - 1);
                        for (int x = 0; x < b.y; ++x) acc += static_cast<int>(row[x]) * s_hk[x * sw + j];
                        s_tmp[r * sw + j] = static_cast<uint8_t>(resize_clip8(acc));
                    }
                }
            }
            __syncthreads();
            // vertical pass: thread = 4 adjacent columns, rows kRcThreads / (sw / 4) apart
            {
                const int g4 = 4 * (tid & (ng - 1));
                if (g4 < mw) {
                    uint8_t *const out_plane = kGeneral ? s_out : out + plane_off;
                    const int wo = kGeneral ? s_wc : Wc, flip = kGeneral ? s_flip : 0;
                    const int xo = xa + g4, xs = flip ? wo - 4 - xo : xo;       // first column / lowest address of the 4
                    for (int yy = tid >> ng_log; yy < mh; yy += kRcThreads >> ng_log) {
                        const int2 b = s_vb[yy];
                        const int *k = s_vk + yy * ksv;
                        const uint8_t *col = s_tmp + b.x * sw + g4;
                        int acc[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) acc[e] = 1 << (kResizePrecisionBits - 1);
                        for (int y = 0; y < b.y; ++y) {
                            const uint32_t v = *reinterpret_cast<const uint32_t *>(col + y * sw);
                            const int w = k[y];
                            acc[0] += static_cast<int>(v & 0xffu) * w, acc[1] += static_cast<int>((v >> 8) & 0xffu) * w;
                            acc[2] += static_cast<int>((v >> 16) & 0xffu) * w, acc[3] += static_cast<int>(v >> 24) * w;
                        }
                        const uint32_t v = resize_clip8(acc[0]) | (resize_clip8(acc[1]) << 8) | (resize_clip8(acc[2]) << 16) |
                                           (resize_clip8(acc[3]) << 24);
                        uint8_t *row = out_plane + static_cast<size_t>(ya + yy) * wo;
                        if (g4 + 3 < mw && (reinterpret_cast<uintptr_t>(row + xs) & 3) == 0) {
                            *reinterpret_cast<uint32_t *>(row + xs) = flip ? __byte_perm(v, 0, 0x0123) : v;
                        } else {
                            for (int e = 0; e < 4 && g4 + e < mw; ++e) row[flip ? wo - 1 - xo - e : xo + e] = static_cast<uint8_t>(v >> (8 * e));
                        }
                    }
                }
            }
        }
    }
}

using resize_crop_fn = void (*)(const uint8_t *, uint8_t *, const CropDesc *, const int *, int, int, int);
static resize_crop_fn resize_pick_crop(int C, bool general) {
    switch (C) {
        case 1: return general ? resize_crop_kernel<1, true> : resize_crop_kernel<1, false>;
        case 2: return general ? resize_crop_kernel<2, true> : resize_crop_kernel<2, false>;
        case 3: return general ? resize_crop_kernel<3, true> : resize_crop_kernel<3, false>;
        default: return general ? resize_crop_kernel<4, true> : resize_crop_kernel<4, false>;
    }
}

// One axis table: rows [first, first + count) of in_size -> out_size (identity tables when the size does not change:
// window 1, weight 2^22).
struct CropAxisKey {
    int in_size, out_size, first, count;
};
static int crop_ksize(int in_size, int out_size, int filter) { return in_size == out_size ? 1 : resize_ksize(in_size, out_size, filter); }

// One output image of a launch: the source image (H x W, at byte in_off of the input), its resized size, the crop window
// (top, left, Hc, Wc) inside the resized image, and where its planar output goes.
struct CropGeom {
    int H, W, RH, RW, top, left, Hc, Wc, flip;
    long long in_off, out_off;
};

// B200_OK, or the error the entry points return for this image (no CUDA call).
static int crop_check_geom(const CropGeom &g, int C, int filter) {
    if (g.H < 1 || g.W < 1 || g.RH < 1 || g.RW < 1 || g.top < 0 || g.left < 0 || g.Hc < 1 || g.Wc < 1) return B200_ERR_INVALID_ARG;
    if (g.top > g.RH - g.Hc || g.left > g.RW - g.Wc) return B200_ERR_INVALID_ARG;      // the crop must lie inside the resized image
    if (static_cast<long long>(g.W) * C > 0x7fffffffLL) return B200_ERR_UNSUPPORTED;
    if (crop_ksize(g.W, g.RW, filter) > kResizeMaxTaps || crop_ksize(g.H, g.RH, filter) > kResizeMaxTaps) return B200_ERR_UNSUPPORTED;
    return B200_OK;
}

static long long crop_ctas(const std::vector<CropGeom> &g, int C) {
    long long ctas = 0;
    for (const CropGeom &e : g) ctas += static_cast<long long>(C) * ceil_div(e.Wc, kRcTW) * ceil_div(e.Hc, kRcTH);
    return ctas;
}

// Host-side layout of one launch: the descriptor block, then one table block per distinct axis key (bounds, then weights;
// every table starts on a 16-byte boundary).
struct CropLayout {
    std::vector<CropAxisKey> keys;
    std::vector<int> key_off, key_ks;   // int offset of each key's bounds in the table block, its window length
    std::vector<int> h_key, v_key;      // per image: horizontal / vertical key
    size_t table_ints = 0, off_tab = 0, bytes = 0;
};
static int crop_find_or_add(CropLayout &l, std::map<std::tuple<int, int, int, int>, int> &seen, const CropAxisKey &k,
                            int filter) {
    const auto t = std::make_tuple(k.in_size, k.out_size, k.first, k.count);
    const auto it = seen.find(t);
    if (it != seen.end()) return it->second;
    seen.emplace(t, static_cast<int>(l.keys.size()));
    const int ks = crop_ksize(k.in_size, k.out_size, filter);
    l.keys.push_back(k);
    l.key_off.push_back(static_cast<int>(l.table_ints));
    l.key_ks.push_back(ks);
    l.table_ints += round_up<size_t>(static_cast<size_t>(k.count) * 2, 4) + round_up<size_t>(static_cast<size_t>(k.count) * ks, 4);
    return static_cast<int>(l.keys.size()) - 1;
}

static CropLayout crop_layout(const std::vector<CropGeom> &g, int filter) {
    CropLayout l;
    std::map<std::tuple<int, int, int, int>, int> seen;
    const size_t n = g.size();
    l.h_key.resize(n), l.v_key.resize(n);
    for (size_t i = 0; i < n; ++i) {
        l.h_key[i] = crop_find_or_add(l, seen, CropAxisKey{g[i].W, g[i].RW, g[i].left, g[i].Wc}, filter);
        l.v_key[i] = crop_find_or_add(l, seen, CropAxisKey{g[i].H, g[i].RH, g[i].top, g[i].Hc}, filter);
    }
    l.off_tab = round_up<size_t>(n * sizeof(CropDesc), 256);
    l.bytes = l.off_tab + l.table_ints * 4;
    return l;
}

// The tables, staging plans and descriptors of one launch, written to `stage` (l.bytes, zeroed): descriptors in launch
// order, the images that stage the most source bytes first.  Returns the dynamic shared memory the launch needs, or 0
// when no sub-block of some image fits kRcSmemBudget.
static size_t crop_stage(const std::vector<CropGeom> &g, int C, int filter, const CropLayout &l, unsigned char *stage) {
    const int n = static_cast<int>(g.size());
    int *tab = reinterpret_cast<int *>(stage + l.off_tab);
    std::vector<std::vector<int>> key_bounds(l.keys.size());
    for (size_t k = 0; k < l.keys.size(); ++k) {
        const CropAxisKey &key = l.keys[k];
        std::vector<int> kk;
        if (key.in_size == key.out_size) {
            key_bounds[k].resize(static_cast<size_t>(key.count) * 2);
            kk.assign(key.count, 1 << kResizePrecisionBits);
            for (int i = 0; i < key.count; ++i) key_bounds[k][2 * i] = key.first + i, key_bounds[k][2 * i + 1] = 1;
        } else {
            resize_coeffs(key.in_size, key.out_size, filter, l.key_ks[k], key_bounds[k], kk, key.first, key.count);
        }
        std::memcpy(tab + l.key_off[k], key_bounds[k].data(), key_bounds[k].size() * 4);
        std::memcpy(tab + l.key_off[k] + round_up<size_t>(static_cast<size_t>(key.count) * 2, 4), kk.data(), kk.size() * 4);
    }
    // staging plan per (horizontal, vertical) key pair: the sub-block that fits kRcSmemBudget and stages the fewest source
    // bytes per output sample (then the larger one)
    std::map<std::pair<int, int>, std::pair<CropDesc, double>> plans;
    std::vector<std::pair<double, int>> order(n);                       // (-staged bytes of the image, image)
    std::vector<CropDesc> by_image(n);
    size_t smem = 0;
    for (int i = 0; i < n; ++i) {
        const int hk = l.h_key[i], vk = l.v_key[i], Hc = g[i].Hc, Wc = g[i].Wc;
        auto it = plans.find(std::make_pair(hk, vk));
        if (it == plans.end()) {
            CropDesc p{};
            p.hb = l.key_off[hk], p.hk = l.key_off[hk] + static_cast<int>(round_up<size_t>(static_cast<size_t>(Wc) * 2, 4));
            p.vb = l.key_off[vk], p.vk = l.key_off[vk] + static_cast<int>(round_up<size_t>(static_cast<size_t>(Hc) * 2, 4));
            p.ksh = l.key_ks[hk], p.ksv = l.key_ks[vk];
            double best = 0.0;
            for (int sw = kRcTW; sw >= 4; sw /= 2) {
                const int stride = round_up(resize_max_window(key_bounds[hk], Wc, sw), 4);
                for (int sh = kRcTH; sh >= 1; sh /= 2) {
                    const int rows = resize_max_window(key_bounds[vk], Hc, sh);
                    if (crop_smem_bytes(sh, sw, p.ksh, p.ksv, rows, stride) > static_cast<size_t>(kRcSmemBudget)) continue;
                    const double per_sample = static_cast<double>(rows) * stride / (static_cast<double>(sh) * sw);
                    if (best == 0.0 || per_sample < best)
                        best = per_sample, p.sub_h = sh, p.sub_w = sw, p.max_rows = rows, p.stride = stride;
                }
            }
            if (best == 0.0) return 0;
            it = plans.emplace(std::make_pair(hk, vk), std::make_pair(p, best)).first;
        }
        CropDesc d = it->second.first;
        d.in_off = g[i].in_off, d.out_off = g[i].out_off, d.W = g[i].W, d.Hc = Hc, d.Wc = Wc, d.flip = g[i].flip;
        by_image[i] = d;
        order[i] = std::make_pair(-it->second.second * Hc * Wc, i);
        const size_t need = crop_smem_bytes(d.sub_h, d.sub_w, d.ksh, d.ksv, d.max_rows, d.stride);
        if (need > smem) smem = need;
    }
    std::stable_sort(order.begin(), order.end());
    CropDesc *descs = reinterpret_cast<CropDesc *>(stage);
    int cta = 0;
    for (int r = 0; r < n; ++r) {
        CropDesc &d = descs[r];
        d = by_image[order[r].second];
        d.cta0 = cta;
        cta += C * ceil_div(d.Wc, kRcTW) * ceil_div(d.Hc, kRcTH);
    }
    return smem;
}

// One launch over descriptors and tables already in device memory at `block` (descriptors at 0, tables at off_tab).  When
// all crops of the launch have one size, it goes to the kernel as launch arguments; the general form of the kernel runs
// unless that holds and no crop is mirrored.
static int crop_launch(int C, const uint8_t *in, uint8_t *out, const unsigned char *block, size_t off_tab,
                       const std::vector<CropGeom> &g, long long ctas, size_t smem, cudaStream_t st) {
    const int n = static_cast<int>(g.size());
    int Hc = g[0].Hc, Wc = g[0].Wc;
    bool flip = false;
    for (const CropGeom &e : g) {
        if (e.Hc != Hc || e.Wc != Wc) Hc = Wc = 0;
        flip = flip || e.flip;
    }
    resize_crop_fn fn = resize_pick_crop(C, Hc == 0 || flip);
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
    fn<<<static_cast<unsigned>(ctas), kRcThreads, smem, st>>>(in, out, reinterpret_cast<const CropDesc *>(block),
                                                              reinterpret_cast<const int *>(block + off_tab), n,
                                                              Hc, Wc);
    B200_LAUNCH_CHECK("resize_crop_kernel");
    return B200_OK;
}

// ---- b200_resize_crop_u8: geom rows H, W, RH, RW, top, left; every crop Hc x Wc, none mirrored.
static int crop_check(int n, const int *geom, int C, int Hc, int Wc, int filter) {
    if (n < 0 || C < 1 || C > 4 || Hc < 1 || Wc < 1) return B200_ERR_INVALID_ARG;
    if (filter != B200_RESIZE_BICUBIC && filter != B200_RESIZE_BILINEAR) return B200_ERR_INVALID_ARG;
    if (n > 0 && !geom) return B200_ERR_INVALID_ARG;
    if (static_cast<long long>(n) * C > 0x7fffffffLL) return B200_ERR_UNSUPPORTED;
    for (int i = 0; i < n; ++i) {
        const int *g = geom + 6 * i;
        const int rc = crop_check_geom(CropGeom{g[0], g[1], g[2], g[3], g[4], g[5], Hc, Wc, 0, 0, 0}, C, filter);
        if (rc != B200_OK) return rc;
    }
    return B200_OK;
}

static std::vector<CropGeom> crop_geoms(int n, const int *geom, const long long *offsets, int C, int Hc, int Wc) {
    std::vector<CropGeom> g(n);
    for (int i = 0; i < n; ++i) {
        const int *r = geom + 6 * i;
        g[i] = CropGeom{r[0], r[1], r[2], r[3], r[4], r[5], Hc, Wc, 0, offsets ? offsets[i] : 0,
                        static_cast<long long>(i) * C * Hc * Wc};
    }
    return g;
}

// ---- b200_resize_random_crop_u8: geom rows H, W, RH, RW, top, left, h, w, flip.  Launch 1 computes each image's window
// (top, left, h, w) of the first resize into a planar [C][h][w] uint8 intermediate (each image 4-byte aligned); launch 2
// resizes every intermediate plane in full to Ho x Wo as a one-channel image, mirrored when flip is set.
static int random_crop_check(int n, const int *geom, int C, int Ho, int Wo, int filter) {
    if (n < 0 || C < 1 || C > 4 || Ho < 1 || Wo < 1) return B200_ERR_INVALID_ARG;
    if (filter != B200_RESIZE_BICUBIC && filter != B200_RESIZE_BILINEAR) return B200_ERR_INVALID_ARG;
    if (n > 0 && !geom) return B200_ERR_INVALID_ARG;
    if (static_cast<long long>(n) * C > 0x7fffffffLL) return B200_ERR_UNSUPPORTED;
    for (int i = 0; i < n; ++i) {
        const int *g = geom + 9 * i;
        if (g[8] != 0 && g[8] != 1) return B200_ERR_INVALID_ARG;
        int rc = crop_check_geom(CropGeom{g[0], g[1], g[2], g[3], g[4], g[5], g[6], g[7], 0, 0, 0}, C, filter);
        if (rc == B200_OK) rc = crop_check_geom(CropGeom{g[6], g[7], Ho, Wo, 0, 0, Ho, Wo, 0, 0, 0}, 1, filter);
        if (rc != B200_OK) return rc;
    }
    return B200_OK;
}

struct RandomCropLayout {
    std::vector<CropGeom> g1, g2;       // launch 1 (one per image, C channels), launch 2 (one per image and channel)
    CropLayout l1, l2;
    size_t off_l2 = 0, off_tmp = 0, bytes = 0;
};
static RandomCropLayout random_crop_layout(int n, const int *geom, const long long *offsets, int C, int Ho, int Wo, int filter) {
    RandomCropLayout r;
    r.g1.resize(n), r.g2.resize(static_cast<size_t>(n) * C);
    long long tmp = 0;
    for (int i = 0; i < n; ++i) {
        const int *g = geom + 9 * i;
        const int h = g[6], w = g[7];
        r.g1[i] = CropGeom{g[0], g[1], g[2], g[3], g[4], g[5], h, w, 0, offsets ? offsets[i] : 0, tmp};
        for (int c = 0; c < C; ++c)
            r.g2[static_cast<size_t>(i) * C + c] = CropGeom{h, w, Ho, Wo, 0, 0, Ho, Wo, g[8], tmp + static_cast<long long>(c) * h * w,
                                                            (static_cast<long long>(i) * C + c) * Ho * Wo};
        tmp += round_up<long long>(static_cast<long long>(C) * h * w, 4);
    }
    r.l1 = crop_layout(r.g1, filter), r.l2 = crop_layout(r.g2, filter);
    r.off_l2 = round_up<size_t>(r.l1.bytes, 256);
    r.off_tmp = round_up<size_t>(r.off_l2 + r.l2.bytes, 256);
    r.bytes = r.off_tmp + static_cast<size_t>(tmp);
    return r;
}

}  // namespace b200

using namespace b200;

extern "C" {

size_t b200_resize_workspace_bytes(long long planes, int H, int W, int Hout, int Wout, int filter) {
    if (planes < 1 || H < 1 || W < 1 || Hout < 1 || Wout < 1) return 0;
    if (filter != B200_RESIZE_BICUBIC && filter != B200_RESIZE_BILINEAR) return 0;
    return resize_layout(planes, H, W, Hout, Wout, filter).bytes;
}

int b200_resize_u8(const uint8_t *in, uint8_t *out, long long planes, int H, int W, int Hout, int Wout, int filter,
                   void *workspace, size_t workspace_bytes, b200_stream_t stream) {
    if (!in || !out || planes < 1 || H < 1 || W < 1 || Hout < 1 || Wout < 1) return B200_ERR_INVALID_ARG;
    if (filter != B200_RESIZE_BICUBIC && filter != B200_RESIZE_BILINEAR) return B200_ERR_INVALID_ARG;
    cudaStream_t st = as_stream(stream);
    const bool need_h = Wout != W, need_v = Hout != H;
    if (!need_h && !need_v) {                                   // PIL returns a copy
        B200_CUDA_TRY(cudaMemcpyAsync(out, in, static_cast<size_t>(planes) * H * W, cudaMemcpyDeviceToDevice, st));
        return B200_OK;
    }
    const ResizeLayout l = resize_layout(planes, H, W, Hout, Wout, filter);
    if (l.ksh > kResizeMaxTaps || l.ksv > kResizeMaxTaps) return B200_ERR_UNSUPPORTED;      // > ~15x reduction
    if (!workspace || workspace_bytes < l.bytes) return B200_ERR_WORKSPACE;
    unsigned char *w = static_cast<unsigned char *>(workspace);
    std::vector<int> hbnd, hkk, vbnd, vkk;
    if (need_h) resize_coeffs(W, Wout, filter, l.ksh, hbnd, hkk); else resize_identity(W, hbnd, hkk);
    if (need_v) resize_coeffs(H, Hout, filter, l.ksv, vbnd, vkk); else resize_identity(H, vbnd, vkk);
    // one H2D copy for the four tables (they are adjacent in the workspace); a pageable-source cudaMemcpyAsync stages
    // the host data before it returns, so the staging vector may die at scope exit
    {
        std::vector<unsigned char> stage(l.bytes - l.off_hb, 0);
        std::memcpy(stage.data(), hbnd.data(), hbnd.size() * 4);
        std::memcpy(stage.data() + (l.off_hk - l.off_hb), hkk.data(), hkk.size() * 4);
        std::memcpy(stage.data() + (l.off_vb - l.off_hb), vbnd.data(), vbnd.size() * 4);
        std::memcpy(stage.data() + (l.off_vk - l.off_hb), vkk.data(), vkk.size() * 4);
        B200_CUDA_TRY(cudaMemcpyAsync(w + l.off_hb, stage.data(), stage.size(), cudaMemcpyHostToDevice, st));
    }
    {   // fused form whenever the largest tile window fits shared memory and the input allows aligned 32-bit loads
        ResizeFusedArgs fa;
        fa.in = in, fa.out = out;
        fa.hb = reinterpret_cast<const int2 *>(w + l.off_hb), fa.vb = reinterpret_cast<const int2 *>(w + l.off_vb);
        fa.hk = reinterpret_cast<const int *>(w + l.off_hk), fa.vk = reinterpret_cast<const int *>(w + l.off_vk);
        fa.H = H, fa.W = W, fa.Hout = Hout, fa.Wout = Wout, fa.ksh = l.ksh, fa.ksv = l.ksv;
        // fixed-length windows read up to ksize - 1 samples past a window's own count (zero weights): pad rows and columns
        fa.max_rows = resize_max_window(vbnd, Hout, kRzTH);
        fa.max_words = (resize_max_window(hbnd, Wout, kRzTW) + 3 + 3 + l.ksh) / 4 + 1;
        const size_t smem = static_cast<size_t>(fa.max_rows) * fa.max_words * 4 + static_cast<size_t>(fa.max_rows + l.ksv) * kRzTW +
                            static_cast<size_t>(kRzTW) * l.ksh * 4 + static_cast<size_t>(kRzTH) * l.ksv * 4 + (kRzTW + kRzTH) * 8 +
                            static_cast<size_t>(fa.max_rows) * 4;
        const char *force = std::getenv("B200_RESIZE_FUSED");
        const bool want = !(force && force[0] == '0');
        if (want && smem <= 160 * 1024 && (reinterpret_cast<uintptr_t>(in) & 3) == 0 && ceil_div(Hout, kRzTH) <= 65535) {
            resize_fused_fn fn = resize_pick_fused(l.ksh, l.ksv);
            B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               static_cast<int>(smem)));
            for (long long p0 = 0; p0 < planes; p0 += 65535) {
                const unsigned np = static_cast<unsigned>(planes - p0 < 65535 ? planes - p0 : 65535);
                fa.plane0 = p0;
                fn<<<dim3(ceil_div(Wout, kRzTW), ceil_div(Hout, kRzTH), np), kRzThreads, smem, st>>>(fa);
                B200_LAUNCH_CHECK("resize_fused_kernel");
            }
            return B200_OK;
        }
    }
    const uint8_t *src = in;
    if (need_h) {
        uint8_t *dst = need_v ? w + l.off_tmp : out;
        const long long rows = planes * H;
        const long long blocks = ceil_div<long long>(rows, kResizeRows);
        if (blocks > 0x7fffffffLL) return B200_ERR_UNSUPPORTED;
        resize_h_kernel<<<static_cast<unsigned>(blocks), resize_block(Wout), 0, st>>>(
            src, dst, rows, W, Wout, l.ksh, reinterpret_cast<const int2 *>(w + l.off_hb), reinterpret_cast<const int *>(w + l.off_hk));
        B200_LAUNCH_CHECK("resize_h_kernel");
        src = dst;
    }
    if (need_v) {
        const size_t in_plane = static_cast<size_t>(H) * Wout, out_plane = static_cast<size_t>(Hout) * Wout;
        for (long long p0 = 0; p0 < planes; p0 += 65535) {
            const unsigned np = static_cast<unsigned>(planes - p0 < 65535 ? planes - p0 : 65535);
            resize_v_kernel<<<dim3(ceil_div(Hout, kResizeRows), np), resize_block(Wout), 0, st>>>(
                src + p0 * in_plane, out + p0 * out_plane, H, Hout, Wout, l.ksv, reinterpret_cast<const int2 *>(w + l.off_vb),
                reinterpret_cast<const int *>(w + l.off_vk));
            B200_LAUNCH_CHECK("resize_v_kernel");
        }
    }
    return B200_OK;
}

size_t b200_resize_crop_workspace_bytes(int n, const int *geom_host, int C, int Hc, int Wc, int filter) {
    if (n < 1 || crop_check(n, geom_host, C, Hc, Wc, filter) != B200_OK) return 0;
    return crop_layout(crop_geoms(n, geom_host, nullptr, C, Hc, Wc), filter).bytes;
}

int b200_resize_crop_u8(const uint8_t *in, const long long *offsets_host, const int *geom_host, int n, int C, int Hc, int Wc,
                        int filter, uint8_t *out, void *workspace, size_t workspace_bytes, b200_stream_t stream) {
    const int rc = crop_check(n, geom_host, C, Hc, Wc, filter);
    if (rc != B200_OK) return rc;
    if (n == 0) return B200_OK;
    if (!in || !out || !offsets_host) return B200_ERR_INVALID_ARG;
    if (reinterpret_cast<uintptr_t>(in) & 3) return B200_ERR_ALIGNMENT;
    for (int i = 0; i < n; ++i) {
        if (offsets_host[i] < 0) return B200_ERR_INVALID_ARG;
        if (offsets_host[i] & 3) return B200_ERR_ALIGNMENT;
    }
    const std::vector<CropGeom> g = crop_geoms(n, geom_host, offsets_host, C, Hc, Wc);
    const long long ctas = crop_ctas(g, C);
    if (ctas > 0x7fffffffLL) return B200_ERR_UNSUPPORTED;
    const CropLayout l = crop_layout(g, filter);
    if (l.table_ints > 0x7fffffffULL) return B200_ERR_UNSUPPORTED;              // descriptors index the tables with int
    if (!workspace || workspace_bytes < l.bytes) return B200_ERR_WORKSPACE;
    // descriptors + tables, staged on the host and copied with one cudaMemcpyAsync (a pageable-source copy stages the host
    // data before it returns, so the vector may die at scope exit)
    std::vector<unsigned char> stage(l.bytes, 0);
    const size_t smem = crop_stage(g, C, filter, l, stage.data());
    if (smem == 0) return B200_ERR_UNSUPPORTED;
    cudaStream_t st = as_stream(stream);
    unsigned char *w = static_cast<unsigned char *>(workspace);
    B200_CUDA_TRY(cudaMemcpyAsync(w, stage.data(), stage.size(), cudaMemcpyHostToDevice, st));
    return crop_launch(C, in, out, w, l.off_tab, g, ctas, smem, st);
}

size_t b200_resize_random_crop_workspace_bytes(int n, const int *geom_host, int C, int Ho, int Wo, int filter) {
    if (n < 1 || random_crop_check(n, geom_host, C, Ho, Wo, filter) != B200_OK) return 0;
    return random_crop_layout(n, geom_host, nullptr, C, Ho, Wo, filter).bytes;
}

int b200_resize_random_crop_u8(const uint8_t *in, const long long *offsets_host, const int *geom_host, int n, int C, int Ho,
                               int Wo, int filter, uint8_t *out, void *workspace, size_t workspace_bytes, b200_stream_t stream) {
    const int rc = random_crop_check(n, geom_host, C, Ho, Wo, filter);
    if (rc != B200_OK) return rc;
    if (n == 0) return B200_OK;
    if (!in || !out || !offsets_host) return B200_ERR_INVALID_ARG;
    if (reinterpret_cast<uintptr_t>(in) & 3) return B200_ERR_ALIGNMENT;
    for (int i = 0; i < n; ++i) {
        if (offsets_host[i] < 0) return B200_ERR_INVALID_ARG;
        if (offsets_host[i] & 3) return B200_ERR_ALIGNMENT;
    }
    const RandomCropLayout r = random_crop_layout(n, geom_host, offsets_host, C, Ho, Wo, filter);
    const long long ctas1 = crop_ctas(r.g1, C), ctas2 = crop_ctas(r.g2, 1);
    if (ctas1 > 0x7fffffffLL || ctas2 > 0x7fffffffLL) return B200_ERR_UNSUPPORTED;
    if (r.l1.table_ints > 0x7fffffffULL || r.l2.table_ints > 0x7fffffffULL) return B200_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < r.bytes) return B200_ERR_WORKSPACE;
    // both launches' descriptors and tables in one staging buffer and one cudaMemcpyAsync; the intermediate follows them
    std::vector<unsigned char> stage(r.off_l2 + r.l2.bytes, 0);
    const size_t smem1 = crop_stage(r.g1, C, filter, r.l1, stage.data());
    const size_t smem2 = crop_stage(r.g2, 1, filter, r.l2, stage.data() + r.off_l2);
    if (smem1 == 0 || smem2 == 0) return B200_ERR_UNSUPPORTED;
    cudaStream_t st = as_stream(stream);
    unsigned char *w = static_cast<unsigned char *>(workspace);
    B200_CUDA_TRY(cudaMemcpyAsync(w, stage.data(), stage.size(), cudaMemcpyHostToDevice, st));
    const int rc1 = crop_launch(C, in, w + r.off_tmp, w, r.l1.off_tab, r.g1, ctas1, smem1, st);
    if (rc1 != B200_OK) return rc1;
    return crop_launch(1, w + r.off_tmp, out, w + r.off_l2, r.l2.off_tab, r.g2, ctas2, smem2, st);
}

}  // extern "C"
