// HP-SWT kernels: batched stationary wavelet transform, all four sub-bands of the coarsest level in one pass.
//
//   b200_swt2_fwd   <- BaseWaveletTransform.__call__ + SWTTransform._apply_wavelet
//                      (/root/reference/main/transforms/custom_transforms.py:145-166; pywt.swt2 + coeffs[0])
//   b200_raw_stack  <- RawStackTransform._apply_wavelet (custom_transforms.py:172-188)
//
// HBM-bound: 1 (uint8) or 4 (float32) bytes read and 16 bytes written per image-channel pixel, independent of the
// filter length and level because every intermediate stays in shared memory / registers (swt2_core.cuh).  One CTA
// per (plane, tile); tile shape from swt_plan(); outputs leave the SM as 128-bit (W % 4 == 0) or 64-bit streaming
// stores, each warp writing whole 128-byte lines of one band row.
#include "common.cuh"
#include "swt2_plan.h"

namespace b200 {

struct SwtDeviceExec {
    template <typename Fn>
    __device__ __forceinline__ void operator()(Fn fn) const {
        fn(static_cast<int>(threadIdx.x), static_cast<int>(blockDim.x));
        __syncthreads();
    }
};

// Global-memory readers of the staging phase: 4 consecutive in-row pixels with the widest access the address allows
// (rows of a 518-wide uint8 image start on 2-byte boundaries every other row), uint8 converted with swt_u8_unit.
struct DevLoad {
    // Stages the whole tile with cp.async.bulk (one row per copy) when the plane is float32, rows are 16-byte aligned
    // (W % 4 == 0) and the staged columns [tx*TW - padL, + RWp) lie inside the image; returns false otherwise.
    // Called by every thread of the CTA with the same arguments; on return the tile is visible to the caller (the
    // phase's __syncthreads() publishes it to the rest).
    __device__ __forceinline__ bool bulk_stage(const SwtGeom &g, const void *plane, float *buf, float *smem, int ty, int tx,
                                               int tid, int nthreads) const {
        const int gc0 = tx * g.TW - g.padL;
        if (g.in_is_u8 || (g.W & 3) || gc0 < 0 || gc0 + g.RWp > g.W) return false;
        uint64_t *bar = reinterpret_cast<uint64_t *>(smem);          // leading guard floats: never written otherwise
        const uint32_t row_bytes = static_cast<uint32_t>(g.RWp) * 4u;
        if (tid == 0) {
            mbar_init(bar, 1);
            mbar_fence_init();
            mbar_expect_tx(bar, row_bytes * static_cast<uint32_t>(g.RH));
        }
        __syncthreads();
        const float *src = static_cast<const float *>(plane);
        const int r_first = ty * g.TH - g.top;
        for (int i = tid; i < g.RH; i += nthreads) {
            const int gr = swt_wrap(r_first + i, g.H);
            bulk_g2s(buf + i * g.RWp, src + static_cast<size_t>(gr) * g.W + gc0, row_bytes, bar);
        }
        mbar_wait(bar, 0);
        return true;
    }
    // starts the reads of 4 consecutive in-row pixels at element offset `off` of the plane
    __device__ __forceinline__ void issue(const void *plane, size_t off, int is_u8, uint32_t *raw) const {
        if (is_u8) {
            const uint8_t *p = static_cast<const uint8_t *>(plane) + (off & ~static_cast<size_t>(3));
            raw[0] = __ldg(reinterpret_cast<const uint32_t *>(p));
            raw[1] = (off & 3) ? __ldg(reinterpret_cast<const uint32_t *>(p + 4)) : 0u;   // the 4 pixels straddle two words
        } else {
            const float *p = static_cast<const float *>(plane) + off;
            if ((off & 3) == 0) {
                const uint4 u = ldg_stream_u4(p);
                raw[0] = u.x, raw[1] = u.y, raw[2] = u.z, raw[3] = u.w;
            } else if ((off & 1) == 0) {
                const uint2 a = __ldg(reinterpret_cast<const uint2 *>(p)), b = __ldg(reinterpret_cast<const uint2 *>(p + 2));
                raw[0] = a.x, raw[1] = a.y, raw[2] = b.x, raw[3] = b.y;
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) raw[e] = __ldg(reinterpret_cast<const uint32_t *>(p) + e);
            }
        }
    }
    __device__ __forceinline__ void finish(const uint32_t *raw, size_t off, int is_u8, float *v) const {
        if (is_u8) {
            const uint32_t w = __funnelshift_r(raw[0], raw[1], 8u * (static_cast<uint32_t>(off) & 3u));
            v[0] = swt_u8_unit(w & 0xffu), v[1] = swt_u8_unit((w >> 8) & 0xffu);
            v[2] = swt_u8_unit((w >> 16) & 0xffu), v[3] = swt_u8_unit(w >> 24);
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) v[e] = __uint_as_float(raw[e]);
        }
    }
    // 8 consecutive uint8 pixels at byte offset `off`: the three aligned words that cover them ...
    __device__ __forceinline__ void issue_u8x8(const uint8_t *plane, size_t off, uint32_t *raw) const {
        const uint32_t *p = reinterpret_cast<const uint32_t *>(plane + (off & ~static_cast<size_t>(3)));
        raw[0] = __ldg(p);
        raw[1] = __ldg(p + 1);
        raw[2] = (off & 3) ? __ldg(p + 2) : 0u;      // an aligned run needs (and may own) two words only
    }
    // ... funnel-shifted into two little-endian words of 4 pixels and converted (float(b) by the 2^23 trick: PRMT puts
    // the byte under the exponent of 8388608.0f, one exact subtraction recovers it — no I2F, no separate extraction)
    __device__ __forceinline__ void finish_u8x8(const uint32_t *raw, size_t off, float *v) const {
        const uint32_t sh = 8u * (static_cast<uint32_t>(off) & 3u);
        const uint32_t w0 = __funnelshift_r(raw[0], raw[1], sh), w1 = __funnelshift_r(raw[1], raw[2], sh);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const uint32_t bits = __byte_perm(e < 4 ? w0 : w1, 0x4B000000u, 0x7440u | static_cast<uint32_t>(e & 3));
            v[e] = swt_u8_float(__uint_as_float(bits) - 8388608.0f);
        }
    }
    __device__ __forceinline__ float one(const void *plane, size_t off, int is_u8) const {
        return is_u8 ? swt_u8_unit(__ldg(static_cast<const uint8_t *>(plane) + off)) : __ldg(static_cast<const float *>(plane) + off);
    }
};
// n = 4: one 128-bit streaming store when the address allows, else two 64-bit ones; n = 2: one 64-bit store
struct DevStore {
    __device__ __forceinline__ void vec4(float *p, const float *v) const { stg_stream_f4(p, make_float4(v[0], v[1], v[2], v[3])); }
    __device__ __forceinline__ void operator()(float *p, const float *v, int n) const {
        if (n == 4 && (reinterpret_cast<uintptr_t>(p) & 15) == 0) {
            stg_stream_f4(p, make_float4(v[0], v[1], v[2], v[3]));
        } else {
            stg_stream_f2(p, make_float2(v[0], v[1]));
            if (n == 4) stg_stream_f2(p + 2, make_float2(v[2], v[3]));
        }
    }
};

__device__ __forceinline__ SwtTileId swt_block_tile() {
    SwtTileId id;
    id.tx = static_cast<int>(blockIdx.x), id.ty = static_cast<int>(blockIdx.y), id.plane = static_cast<int>(blockIdx.z);
    return id;
}

// Register budgets are part of the design: a 256-thread CTA at 64 registers fits 4 per SM, at 65-72 only 3 — measured
// 0.74 vs 0.64 of the HBM roofline for haar level 2 — so F <= 4 and the sliding F = 8 level-1 kernel are pinned to 64
// registers and F = 6, 8 to 80 (F = 8 with 2 output rows per vertical unit; F = 10 spills there).
template <int F, int LEVEL>
__global__ void __launch_bounds__(256, ((F <= 4 || swt_vs_form(F, LEVEL)) ? 4 : (F <= 8 ? 3 : 2)))
    swt2_tile_kernel(const __grid_constant__ SwtGeom g, const void *__restrict__ in, float *__restrict__ out) {
    extern __shared__ __align__(16) float swt_smem[];
    swt_tile_program<F, LEVEL>(g, in, out, swt_block_tile(), swt_smem, SwtDeviceExec{}, DevStore{}, DevLoad{});
}

__global__ void __launch_bounds__(256) swt2_generic_kernel(const __grid_constant__ SwtGeom g, const void *__restrict__ in,
                                                           float *__restrict__ out) {
    extern __shared__ __align__(16) float swt_smem[];
    swt_generic_program(g, in, out, swt_block_tile(), swt_smem, SwtDeviceExec{}, DevLoad{});
}

// RawStackTransform: out[b][c][copy][h][w] = in[b][c][h][w] (/255 for uint8), `copies` identical planes.
template <bool U8>
__global__ void __launch_bounds__(256) raw_stack_kernel(const void *__restrict__ in, float *__restrict__ out, long long planes,
                                                        long long plane_px, int copies) {
    const long long total = planes * plane_px;
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += stride) {
        const long long p = i / plane_px, o = i - p * plane_px;
        const float x = U8 ? swt_u8_unit(static_cast<const uint8_t *>(in)[i]) : static_cast<const float *>(in)[i];   // == b / 255.0f
        float *dst = out + p * copies * plane_px + o;
        for (int c = 0; c < copies; ++c) dst[c * plane_px] = x;
    }
}

using swt_fn = void (*)(const SwtGeom, const void *, float *);

// the fast-path kernel of (F, level): the only 15 instantiations of swt2_tile_kernel
template <int F>
static swt_fn pick_level(int level) {
    switch (level) {
        case 1: return swt2_tile_kernel<F, 1>;
        case 2: return swt2_tile_kernel<F, 2>;
        case 3: return swt2_tile_kernel<F, 3>;
    }
    return nullptr;
}
static swt_fn pick_swt(int F, int level) {
    switch (F) {
        case 2: return pick_level<2>(level);
        case 4: return pick_level<4>(level);
        case 6: return pick_level<6>(level);
        case 8: return pick_level<8>(level);
        case 10: return pick_level<10>(level);
    }
    return nullptr;
}

int swt2_launch(const void *in, int in_is_u8, float *out, int B, int C, int H, int W, const float *lo, const float *hi, int F,
                int level, cudaStream_t st) {
    SwtGeom g;
    const int rc = swt_plan(g, B, C, H, W, F, level, in_is_u8, lo, hi, sm_count());
    if (rc == -1) return B200_ERR_INVALID_ARG;
    if (rc) return B200_ERR_UNSUPPORTED;
    const size_t smem = swt_smem_bytes(g);
    const long long planes = static_cast<long long>(B) * C;
    if (planes > 0x7fffffffll || g.tiles_y > 65535) return B200_ERR_UNSUPPORTED;
    swt_fn fn = swt_fast_path(F, level) ? pick_swt(F, level) : swt2_generic_kernel;
    if (!fn) return B200_ERR_UNSUPPORTED;
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
    // tiles of one plane are adjacent in launch order (x fastest): CTAs that run together write neighbouring rows
    const size_t plane_px = static_cast<size_t>(H) * W;
    for (long long p0 = 0; p0 < planes; p0 += 65535) {
        const unsigned np = static_cast<unsigned>(planes - p0 < 65535 ? planes - p0 : 65535);
        const void *src = in_is_u8 ? static_cast<const void *>(static_cast<const uint8_t *>(in) + p0 * plane_px)
                                   : static_cast<const void *>(static_cast<const float *>(in) + p0 * plane_px);
        fn<<<dim3(g.tiles_x, g.tiles_y, np), g.threads, smem, st>>>(g, src, out + p0 * 4 * plane_px);
        B200_LAUNCH_CHECK("swt2_tile_kernel");
    }
    return B200_OK;
}

}  // namespace b200

using namespace b200;

extern "C" {

int b200_swt2_fwd(const void *in, int in_is_u8, float *out, int B, int C, int H, int W, const float *dec_lo,
                  const float *dec_hi, int F, int level, b200_stream_t stream) {
    if (!in || !out || !dec_lo || !dec_hi || B < 1 || C < 1 || H < 1 || W < 1) return B200_ERR_INVALID_ARG;
    if (F < 2 || (F & 1) || level < 1) return B200_ERR_INVALID_ARG;
    if (F > B200_SWT_MAX_FILTER || level > B200_SWT_MAX_LEVEL) return B200_ERR_UNSUPPORTED;
    if (H % (1 << level) || W % (1 << level)) return B200_ERR_INVALID_ARG;   // pywt.swt2 raises ValueError here
    if ((reinterpret_cast<uintptr_t>(out) & 15) || (reinterpret_cast<uintptr_t>(in) & (in_is_u8 ? 3 : 15)))
        return B200_ERR_ALIGNMENT;
    return swt2_launch(in, in_is_u8, out, B, C, H, W, dec_lo, dec_hi, F, level, as_stream(stream));
}

int b200_raw_stack(const void *in, int in_is_u8, float *out, int B, int C, int H, int W, int copies, b200_stream_t stream) {
    if (!in || !out || B < 1 || C < 1 || H < 1 || W < 1 || copies < 1) return B200_ERR_INVALID_ARG;
    const long long planes = static_cast<long long>(B) * C, px = static_cast<long long>(H) * W;
    const long long blocks = ceil_div<long long>(planes * px, 256);
    const int grid = static_cast<int>(blocks < sm_count() * 16ll ? blocks : sm_count() * 16ll);
    if (in_is_u8)
        raw_stack_kernel<true><<<grid, 256, 0, as_stream(stream)>>>(in, out, planes, px, copies);
    else
        raw_stack_kernel<false><<<grid, 256, 0, as_stream(stream)>>>(in, out, planes, px, copies);
    B200_LAUNCH_CHECK("raw_stack_kernel");
    return B200_OK;
}

}  // extern "C"
