// Tensor-core scorer of the continuous-embedding k-NN (get_knn, /root/reference/main/engine/get_knn.py:9-71, inner
// product branch :63-66 / faiss IndexFlatIP :35-52): S[q][n] = <Q[q], R[n]> for float32 inputs on the 5th-generation
// tensor cores, float32-grade accuracy through the split  x = hi + lo  (two bfloat16 each, |x - hi - lo| <= 2^-17 |x|):
//      <q, r>  ~=  <q_hi, r_hi> + <q_hi, r_lo> + <q_lo, r_hi>          (the dropped lo.lo term is <= 2^-16 of hi.hi)
// three tcgen05.mma chains accumulated in the same float32 TMEM accumulator.
//
// One persistent CTA per SM, warp-specialised:
//   warp 0      TMA producer: cp.async.bulk.tensor (128-byte swizzle) of the hi/lo tiles of Q (128 rows) and R (256 rows)
//               for one 64-wide K block per stage, 2 stages of 96 KB, mbarrier full/empty ring
//   warp 1      MMA issuer (one elected lane): 3 products x 4 K-steps of tcgen05.mma.kind::f16 M128 N256 K16 per stage,
//               tcgen05.commit releases the stage / publishes the accumulator; owns the TMEM allocation (512 columns =
//               two 128x256 float32 accumulators, so the epilogue of tile i overlaps the main loop of tile i+1)
//   warps 2..5  epilogue: tcgen05.ld 32 lanes x 32 columns -> registers -> 128-bit global stores of the score tile
// Tiles are walked Q-block fastest so that the R tile of a column block is shared through L2 by the CTAs running together.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "knn_tc.h"
#include "tc_common.cuh"

namespace b200 {

constexpr int kTcBM = 128, kTcBN = 256, kTcBK = 64;            // K block: 64 bf16 = one 128-byte swizzle row
constexpr int kTcStages = 2;
constexpr uint32_t kTcABytes = kTcBM * 128, kTcBBytes = kTcBN * 128;
constexpr uint32_t kTcStageBytes = 2 * kTcABytes + 2 * kTcBBytes;          // hi + lo of both operands: 96 KB
constexpr uint32_t kTcSmemBytes = kTcStages * kTcStageBytes + 1024 /*alignment*/ + 256 /*barriers*/;
constexpr int kTcThreads = 192;

// ---- float32 -> (hi, lo) bfloat16, rows padded with zeros to Dp (multiple of kTcBK)
__global__ void __launch_bounds__(256) knn_split_bf16_kernel(const float *__restrict__ x, long long rows, int D, int Dp,
                                                             __nv_bfloat16 *__restrict__ hi, __nv_bfloat16 *__restrict__ lo) {
    const long long total = rows * (Dp / 2);
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long r = i / (Dp / 2);
        const int c = static_cast<int>(i - r * (Dp / 2)) * 2;
        float a = 0.f, b = 0.f;
        if (c < D) a = x[r * D + c];
        if (c + 1 < D) b = x[r * D + c + 1];
        const __nv_bfloat16 ah = __float2bfloat16_rn(a), bh = __float2bfloat16_rn(b);
        const __nv_bfloat16 al = __float2bfloat16_rn(a - __bfloat162float(ah)), bl = __float2bfloat16_rn(b - __bfloat162float(bh));
        reinterpret_cast<__nv_bfloat162 *>(hi)[i] = __halves2bfloat162(ah, bh);
        reinterpret_cast<__nv_bfloat162 *>(lo)[i] = __halves2bfloat162(al, bl);
    }
}

// kind::f16: D float32, A/B bfloat16, both K-major, M = 128, N = 256
constexpr uint32_t kTcIdesc = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(kTcBN >> 3) << 17) |
                              (static_cast<uint32_t>(kTcBM >> 4) << 24);

// Epilogue modes: `filt.thr == nullptr`: the score tile is stored to S (row stride ldS).  Otherwise the scores never
// reach memory: a score that reaches its query's threshold thr[m] is appended — (order-preserving key << 32 | ~index) —
// to that query's candidate list (cand[m][..cap], cand_cnt[m] counts every hit, also beyond cap), i.e. the top-k
// selection is fused into the GEMM and the 2.3 GB score matrix of the COCO shape is never written.
struct TcFilter {
    const float *thr;
    unsigned long long *cand;
    uint32_t *cand_cnt;
    uint32_t cap;
    const uint32_t *gate;            // or null: when given and zero the kernel returns at once (fallback launches)
};

__global__ void __launch_bounds__(kTcThreads, 1) knn_scores_tc_kernel(const __grid_constant__ TcMaps maps, float *__restrict__ S,
                                                                       int M, long long N, long long ldS, int Dp,
                                                                       const TcFilter filt) {
    extern __shared__ unsigned char tc_smem_raw[];
    if (filt.gate && *filt.gate == 0u) return;
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kTcStages * kTcStageBytes);
    uint64_t *full = bars, *empty = bars + kTcStages, *acc_full = bars + 2 * kTcStages, *acc_empty = bars + 2 * kTcStages + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * kTcStages + 4);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_m = (M + kTcBM - 1) / kTcBM;
    const long long tiles_n = (N + kTcBN - 1) / kTcBN;
    const long long tiles = tiles_m * tiles_n;
    const int nkb = Dp / kTcBK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kTcStages; ++s) mbar_init(&full[s], 1), mbar_init(&empty[s], 1);
        for (int a = 0; a < 2; ++a) mbar_init(&acc_full[a], 1), mbar_init(&acc_empty[a], 128);
        mbar_fence_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t s = 0, ph = 0;
            for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
                const int m0 = static_cast<int>(t % tiles_m) * kTcBM;
                const int n0 = static_cast<int>(t / tiles_m) * kTcBN;
                for (int kb = 0; kb < nkb; ++kb) {
                    mbar_wait_guarded(&empty[s], ph ^ 1u);
                    unsigned char *st = smem + s * kTcStageBytes;
                    mbar_expect_tx(&full[s], kTcStageBytes);
                    tma_load_2d(st, &maps.q_hi, &full[s], kb * kTcBK, m0);
                    tma_load_2d(st + kTcABytes, &maps.q_lo, &full[s], kb * kTcBK, m0);
                    tma_load_2d(st + 2 * kTcABytes, &maps.r_hi, &full[s], kb * kTcBK, n0);
                    tma_load_2d(st + 2 * kTcABytes + kTcBBytes, &maps.r_lo, &full[s], kb * kTcBK, n0);
                    if (++s == kTcStages) s = 0, ph ^= 1u;
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            uint32_t s = 0, ph = 0, it = 0;
            for (long long t = blockIdx.x; t < tiles; t += gridDim.x, ++it) {
                const uint32_t ab = it & 1u, aph = (it >> 1) & 1u;
                mbar_wait_guarded(&acc_empty[ab], aph ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + ab * kTcBN;
                for (int kb = 0; kb < nkb; ++kb) {
                    mbar_wait_guarded(&full[s], ph);
                    tc_fence_after();
                    const uint32_t st = smem_u32(smem + s * kTcStageBytes);
                    const uint64_t a_hi = tc_smem_desc(st), a_lo = tc_smem_desc(st + kTcABytes);
                    const uint64_t b_hi = tc_smem_desc(st + 2 * kTcABytes), b_lo = tc_smem_desc(st + 2 * kTcABytes + kTcBBytes);
#pragma unroll
                    for (int k = 0; k < kTcBK / 16; ++k) {          // 32 bytes (16 bf16) per K-step: +2 in 16-byte units
                        tc_mma_bf16(d_tmem, a_hi + 2 * k, b_hi + 2 * k, kTcIdesc, (kb | k) != 0);
                        tc_mma_bf16(d_tmem, a_hi + 2 * k, b_lo + 2 * k, kTcIdesc, 1u);
                        tc_mma_bf16(d_tmem, a_lo + 2 * k, b_hi + 2 * k, kTcIdesc, 1u);
                    }
                    tc_commit(&empty[s]);                            // stage reusable once these MMAs have read it
                    if (++s == kTcStages) s = 0, ph ^= 1u;
                }
                tc_commit(&acc_full[ab]);                            // accumulator complete
            }
        }
    } else {
        const int quarter = warp & 3;                                // TMEM lanes 32*quarter .. +31 belong to this warp
        uint32_t it = 0;
        for (long long t = blockIdx.x; t < tiles; t += gridDim.x, ++it) {
            const uint32_t ab = it & 1u, aph = (it >> 1) & 1u;
            const int m0 = static_cast<int>(t % tiles_m) * kTcBM;
            const long long n0 = (t / tiles_m) * kTcBN;
            mbar_wait_guarded(&acc_full[ab], aph);
            tc_fence_after();
            const int m = m0 + quarter * 32 + lane;
            float *row = S + static_cast<size_t>(m) * ldS + n0;
            const uint32_t taddr = tmem_base + ab * kTcBN + (static_cast<uint32_t>(quarter * 32) << 16);
            const float th = (filt.thr && m < M) ? filt.thr[m] : 0.f;
            // the TMEM read of chunk c + 1 is in flight while chunk c is stored / filtered (two register buffers)
            uint32_t ra[32], rb[32];
            tc_ld32(taddr, ra);
            tc_ld_wait();
            auto consume = [&](const uint32_t (&r)[32], int c) {
                const long long nb = n0 + c * 32;
                if (filt.thr) {
                    if (m < M) {
                        uint32_t hit = 0;
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (__uint_as_float(r[j]) >= th) hit |= 1u << j;
                        if (nb + 32 > N) hit &= nb < N ? (0xffffffffu >> (32 - static_cast<int>(N - nb))) : 0u;
                        if (hit) {
                            uint32_t pos = atomicAdd(filt.cand_cnt + m, static_cast<uint32_t>(__popc(hit)));
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                if ((hit >> j) & 1u) {
                                    if (pos < filt.cap)
                                        filt.cand[static_cast<size_t>(m) * filt.cap + pos] =
                                            (static_cast<unsigned long long>(rank_key(__uint_as_float(r[j]), true)) << 32) |
                                            (0xffffffffu - static_cast<uint32_t>(nb + j));
                                    ++pos;
                                }
                            }
                        }
                    }
                } else if (m < M) {
                    if (nb + 32 <= N) {
#pragma unroll
                        for (int j = 0; j < 32; j += 4)
                            *reinterpret_cast<uint4 *>(row + c * 32 + j) = make_uint4(r[j], r[j + 1], r[j + 2], r[j + 3]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (nb + j < N) row[c * 32 + j] = __uint_as_float(r[j]);
                    }
                }
            };
#pragma unroll 1
            for (int c = 0; c < kTcBN / 32; c += 2) {
                tc_ld32(taddr + (c + 1) * 32, rb);
                consume(ra, c);
                tc_ld_wait();
                if (c + 2 < kTcBN / 32) tc_ld32(taddr + (c + 2) * 32, ra);
                consume(rb, c + 1);
                tc_ld_wait();
            }
            tc_fence_before();
            mbar_arrive(&acc_empty[ab]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ---- host side ---------------------------------------------------------------------------------------------------
size_t knn_tc_extra_workspace(int Q, long long N, int D) {
    const size_t Dp = round_up<size_t>(D, kTcBK);
    return round_up<size_t>(2 * (static_cast<size_t>(Q) + static_cast<size_t>(N)) * Dp * sizeof(__nv_bfloat16), 1024) + 1024;
}

int knn_tc_prepare(const float *queries, const float *refs, int Q, long long N, int D, void *extra, long long sample_stride,
                   TcContext *ctx, cudaStream_t st) {
    const int Dp = static_cast<int>(round_up<size_t>(D, kTcBK));
    unsigned char *base = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(extra) + 1023) & ~static_cast<uintptr_t>(1023));
    __nv_bfloat16 *q_hi = reinterpret_cast<__nv_bfloat16 *>(base);
    __nv_bfloat16 *q_lo = q_hi + static_cast<size_t>(Q) * Dp;
    __nv_bfloat16 *r_hi = q_lo + static_cast<size_t>(Q) * Dp;
    __nv_bfloat16 *r_lo = r_hi + static_cast<size_t>(N) * Dp;
    ctx->Q = Q, ctx->Dp = Dp, ctx->N = N, ctx->Ns = 0;
    const CUtensorMapDataType bf16 = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    if (!make_tensor_map(&ctx->full.q_hi, bf16, q_hi, Q, Dp, kTcBM) || !make_tensor_map(&ctx->full.q_lo, bf16, q_lo, Q, Dp, kTcBM) ||
        !make_tensor_map(&ctx->full.r_hi, bf16, r_hi, N, Dp, kTcBN) || !make_tensor_map(&ctx->full.r_lo, bf16, r_lo, N, Dp, kTcBN))
        return B200_ERR_UNSUPPORTED;
    if (sample_stride > 0) {
        ctx->Ns = N / sample_stride;
        ctx->sample.q_hi = ctx->full.q_hi, ctx->sample.q_lo = ctx->full.q_lo;
        if (!make_tensor_map(&ctx->sample.r_hi, bf16, r_hi, ctx->Ns, Dp, kTcBN, sample_stride) ||
            !make_tensor_map(&ctx->sample.r_lo, bf16, r_lo, ctx->Ns, Dp, kTcBN, sample_stride))
            return B200_ERR_UNSUPPORTED;
    }
    const int sms = sm_count();
    knn_split_bf16_kernel<<<sms * 8, 256, 0, st>>>(queries, Q, D, Dp, q_hi, q_lo);
    B200_LAUNCH_CHECK("knn_split_bf16_kernel");
    knn_split_bf16_kernel<<<sms * 8, 256, 0, st>>>(refs, N, D, Dp, r_hi, r_lo);
    B200_LAUNCH_CHECK("knn_split_bf16_kernel");
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(knn_scores_tc_kernel), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(kTcSmemBytes)));
    return B200_OK;
}

int knn_tc_scores(const TcContext *ctx, int sample, float *S, long long ldS, const float *thr, unsigned long long *cand,
                  uint32_t *cand_cnt, uint32_t cap, const uint32_t *gate, cudaStream_t st) {
    const long long n = sample ? ctx->Ns : ctx->N;
    const int sms = sm_count();
    const long long tiles = static_cast<long long>((ctx->Q + kTcBM - 1) / kTcBM) * ((n + kTcBN - 1) / kTcBN);
    const int grid = static_cast<int>(tiles < sms ? tiles : sms);
    TcFilter f;
    f.thr = thr, f.cand = cand, f.cand_cnt = cand_cnt, f.cap = cap, f.gate = gate;
    knn_scores_tc_kernel<<<grid, kTcThreads, kTcSmemBytes, st>>>(sample ? ctx->sample : ctx->full, S, ctx->Q, n, ldS, ctx->Dp, f);
    B200_LAUNCH_CHECK("knn_scores_tc_kernel");
    return B200_OK;
}

}  // namespace b200
