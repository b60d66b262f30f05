// Continuous-embedding k-NN: get_knn / get_knn_torch / get_knn_faiss
//   /root/reference/main/engine/get_knn.py:9-71  (queries @ references.T + topk(largest), or cdist + topk(smallest);
//   faiss IndexFlatIP / IndexFlatL2 on the reference's GPU path).
//
// v0 (this file): exact float32.  (1) a register-tiled SGEMM writes the Q x N score matrix to the caller's
// workspace, (2) one CTA per query selects the k best by an MSB-first radix select over order-preserving keys and
// sorts the survivors with a bitonic network; ties go to the smaller index.  For inner products the tensor-core
// (tcgen05) scorer of knn_tc.cu replaces step (1), and where the shape allows (knn_fused_rank) filters candidates in its
// epilogue instead of writing the matrix.  The exact path serves L2, B200_KNN_TC=0 and drivers without the tensor-map
// encoder, and is the tensor-core path's parity reference.
// The same scorer with the kEpiRealHamming epilogue is b200_real_hamming_dist: the reference's float32
// 0.5 * (B - q @ r.T) of real-valued codes (accuracy_calculator.py:183-186), in a summation order a CPU oracle restates.
#include <cmath>
#include <cstdlib>

#include "common.cuh"
#include "knn_tc.h"

namespace b200 {

constexpr int kBM = 128, kBN = 128, kBK = 16;
constexpr int kKnnMaxK = 4096;
constexpr int kKnnSample = 1024;     // sampled keys per row for the one-pass threshold
constexpr int kKnnCand = 8192;       // candidate capacity of the one-pass path (64 KB of shared memory)

__global__ void __launch_bounds__(256) row_sqnorm_kernel(const float *__restrict__ x, long long rows, int D,
                                                         float *__restrict__ out) {
    const long long warp = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= rows) return;
    float s = 0.f;
    for (int j = lane; j < D; j += 32) {
        const float v = x[warp * D + j];
        s += v * v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[warp] = s;
}

// Epilogue modes of knn_scores_kernel.  The mode is a template parameter so that kEpiScore (inner product, or L2 when
// the runtime flag l2 is set) compiles to the same code whether or not the other mode exists.
enum KnnEpilogue : int {
    kEpiScore = 0,          // S = <q,r>   (l2: sqrt(max(|q|^2 + |r|^2 - 2<q,r>, 0)))
    kEpiRealHamming = 1,    // S = 0.5f * ((float)nbits - <q,r>): calc_hamming_dist of real-valued codes
};

// S[q][n] from acc = <Q[q], R[n]>, one fmaf chain over the dimensions in index order (the k0 tiles, then kk ascending),
// starting from +0.0f.     Q: [M][D], R: [N][D], D % 4 == 0; row stride ldS.  nbits: kEpiRealHamming only.
template <int kEpi>
__global__ void __launch_bounds__(256) knn_scores_kernel(const float *__restrict__ Qm, const float *__restrict__ Rm,
                                                         float *__restrict__ S, int M, long long N, long long ldS, int D, int l2,
                                                         const float *__restrict__ qn, const float *__restrict__ rn, float nbits) {
    __shared__ __align__(16) float As[kBK][kBM + 4];
    __shared__ __align__(16) float Bs[kBK][kBN + 4];
    const int tid = threadIdx.x;
    const long long n0 = static_cast<long long>(blockIdx.x) * kBN;
    const int m0 = blockIdx.y * kBM;
    const int lrow = tid >> 1, lk = (tid & 1) * 8;
    const int tx = tid & 15, ty = tid >> 4;
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    const bool a_ok = m0 + lrow < M;
    const bool b_ok = n0 + lrow < N;
    const float *ap = Qm + static_cast<size_t>(a_ok ? m0 + lrow : 0) * D + lk;
    const float *bp = Rm + static_cast<size_t>(b_ok ? n0 + lrow : 0) * D + lk;
    for (int k0 = 0; k0 < D; k0 += kBK) {
        float4 a0 = make_float4(0, 0, 0, 0), a1 = a0, b0 = a0, b1 = a0;
        if (a_ok && k0 + lk < D) a0 = *reinterpret_cast<const float4 *>(ap + k0);
        if (a_ok && k0 + lk + 4 < D) a1 = *reinterpret_cast<const float4 *>(ap + k0 + 4);
        if (b_ok && k0 + lk < D) b0 = *reinterpret_cast<const float4 *>(bp + k0);
        if (b_ok && k0 + lk + 4 < D) b1 = *reinterpret_cast<const float4 *>(bp + k0 + 4);
        __syncthreads();
        As[lk + 0][lrow] = a0.x, As[lk + 1][lrow] = a0.y, As[lk + 2][lrow] = a0.z, As[lk + 3][lrow] = a0.w;
        As[lk + 4][lrow] = a1.x, As[lk + 5][lrow] = a1.y, As[lk + 6][lrow] = a1.z, As[lk + 7][lrow] = a1.w;
        Bs[lk + 0][lrow] = b0.x, Bs[lk + 1][lrow] = b0.y, Bs[lk + 2][lrow] = b0.z, Bs[lk + 3][lrow] = b0.w;
        Bs[lk + 4][lrow] = b1.x, Bs[lk + 5][lrow] = b1.y, Bs[lk + 6][lrow] = b1.z, Bs[lk + 7][lrow] = b1.w;
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kBK; ++kk) {
            float a[8], b[8];
            *reinterpret_cast<float4 *>(a) = *reinterpret_cast<const float4 *>(&As[kk][ty * 8]);
            *reinterpret_cast<float4 *>(a + 4) = *reinterpret_cast<const float4 *>(&As[kk][ty * 8 + 4]);
            *reinterpret_cast<float4 *>(b) = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 8]);
            *reinterpret_cast<float4 *>(b + 4) = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 8 + 4]);
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = m0 + ty * 8 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const long long n = n0 + tx * 8 + j;
            if (n >= N) continue;
            float v = acc[i][j];
            if (kEpi == kEpiRealHamming) {
                v = __fmul_rn(0.5f, __fsub_rn(nbits, v));       // two roundings, as the reference's float32 ops
            } else if (l2) {
                const float d2 = qn[m] + rn[n] - 2.f * v;
                v = d2 != d2 ? d2 : sqrtf(fmaxf(d2, 0.f));        // fmaxf would turn NaN into distance 0
            }
            S[static_cast<size_t>(m) * ldS + n] = v;
        }
    }
}

// MSB-first radix select, one digit: given the 256-bin histogram of the keys that still match the prefix, the largest
// digit d whose suffix count (bins d..255) reaches `need`, and how many keys are still wanted inside bin d.  Run by the
// first warp: lane l owns the 8 bins 255-8l .. 248-8l, a shuffle scan over the lanes replaces the serial walk over 256
// bins (which was a third of the select kernel's time).  Returns through *digit / *need_out (lane 0's view is written).
__device__ __forceinline__ void radix_pick_digit(const uint32_t *hist, uint32_t need, int lane, uint32_t *digit, uint32_t *need_out) {
    uint32_t local[8], s = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        local[i] = hist[255 - 8 * lane - i];
        s += local[i];
    }
    uint32_t incl = s;                                   // inclusive prefix over lanes = suffix count over bins
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    const uint32_t reach = __ballot_sync(0xffffffffu, incl >= need);
    const int owner = reach ? __ffs(static_cast<int>(reach)) - 1 : 31;   // no lane reaches: fewer keys than wanted -> digit 0
    if (lane == owner) {
        uint32_t left = need - (incl - s), d = 255u - 8u * owner;
        int i = 0;
        for (; i < 7; ++i) {                             // no lane reaches (fewer keys than wanted): walk on to digit 0
            if (reach && local[i] >= left) break;
            left -= local[i];
        }
        *digit = d - static_cast<uint32_t>(i);
        *need_out = left;
    }
}

__host__ __device__ constexpr int pow2_ceil(int k) { int p = 1; while (p < k) p <<= 1; return p; }

// a[0 .. n) descending, n a power of two, by 256 threads (a in shared memory; ends with __syncthreads)
template <typename T>
__device__ __forceinline__ void bitonic_sort_desc(T *a, int n, int tid) {
    for (int size = 2; size <= n; size <<= 1) {
        for (int st = size >> 1; st > 0; st >>= 1) {
            for (int i = tid; i < n / 2; i += 256) {
                const int lo = 2 * i - (i & (st - 1)), hi = lo + st;
                const bool desc = ((lo & size) == 0);
                const T x = a[lo], y = a[hi];
                if ((x < y) == desc) a[lo] = y, a[hi] = x;
            }
            __syncthreads();
        }
    }
}

// The k best of cnt distinct (key << 32 | ~idx) pairs in shared memory, best first, to idx_out / score_out [0 .. k): the
// exact k-th largest pair by an MSB-first radix select, then only the k winners, zero-padded to P = pow2_ceil(k) in
// top [P], are sorted.  hist [256], need, pref and top_cnt are the caller's shared scratch; 256 threads.
__device__ __forceinline__ void select_top_pairs(const unsigned long long *pairs, uint32_t cnt, int k, int P, unsigned long long *top,
                                                 int64_t *idx_out, float *score_out, bool largest, uint32_t *hist, uint32_t *need,
                                                 unsigned long long *pref, uint32_t *top_cnt, int tid) {
    if (tid == 0) *pref = 0ull, *need = static_cast<uint32_t>(k);
    __syncthreads();
    for (int shift = 56; shift >= 0; shift -= 8) {
        hist[tid] = 0;
        __syncthreads();
        const unsigned long long pf = *pref;
        for (uint32_t i = tid; i < cnt; i += 256) {
            const unsigned long long pr = pairs[i];
            if (shift == 56 || (pr >> (shift + 8)) == (pf >> (shift + 8))) atomicAdd(&hist[(pr >> shift) & 255ull], 1u);
        }
        __syncthreads();
        if (tid < 32) {
            __shared__ uint32_t s_digit;
            radix_pick_digit(hist, *need, tid, &s_digit, need);
            __syncwarp();
            if (tid == 0) *pref = pf | (static_cast<unsigned long long>(s_digit) << shift);
        }
        __syncthreads();
    }
    const unsigned long long kth = *pref;
    if (tid == 0) *top_cnt = 0;
    for (int i = tid; i < P; i += 256) top[i] = 0ull;
    __syncthreads();
    for (uint32_t i = tid; i < cnt; i += 256) {
        const unsigned long long pr = pairs[i];
        if (pr >= kth) top[atomicAdd(top_cnt, 1u)] = pr;             // exactly k of them
    }
    __syncthreads();
    bitonic_sort_desc(top, P, tid);
    for (int i = tid; i < k; i += 256) {
        const unsigned long long pr = top[i];
        idx_out[i] = static_cast<int64_t>(0xffffffffu - static_cast<uint32_t>(pr));
        score_out[i] = rank_key_inv(static_cast<uint32_t>(pr >> 32), largest);
    }
}

// One CTA (256 threads) per query row: the k largest keys (rank_key: larger scores first, or smaller distances for L2;
// NaN last), ties to the smaller index, sorted best-first.
// Lists longer than kKnnMaxK come out in passes of <= kKnnMaxK ranks: pass p only sees the entries that rank strictly
// after the last entry of pass p - 1 (k_done > 0: that entry is idx_out / score_out[k_done - 1] of the row), writes ranks
// k_done .. k_done + k - 1 of the ldo-wide output rows.  gate (or null): the launch does nothing while *gate == 0.
__global__ void __launch_bounds__(256) knn_select_kernel(const float *__restrict__ S, long long N, long long ldS, int k, int l2,
                                                         int fast_rank, int64_t *__restrict__ idx_out,
                                                         float *__restrict__ score_out, long long ldo, int k_done,
                                                         const uint32_t *__restrict__ gate) {
    extern __shared__ __align__(16) unsigned char knn_smem[];
    unsigned long long *s_pair = reinterpret_cast<unsigned long long *>(knn_smem);    // [P] (key << 32 | ~idx)
    __shared__ uint32_t s_hist[256];
    __shared__ uint32_t s_prefix, s_need, s_cnt_gt;
    __shared__ uint32_t s_scan[256];
    if (gate && *gate == 0u) return;
    const int tid = threadIdx.x;
    const float *row = S + static_cast<size_t>(blockIdx.x) * ldS;
    int64_t *orow_idx = idx_out + static_cast<size_t>(blockIdx.x) * ldo + k_done;          // where this pass writes its ranks
    float *orow_score = score_out + static_cast<size_t>(blockIdx.x) * ldo + k_done;
    const int P = pow2_ceil(k);
    // entries at or before the previous pass' last one are out of the game: their key reads as 0 ... but 0 is also a
    // legal key (NaN), so eligibility is carried separately
    unsigned long long bound = ~0ull;                     // exclusive upper bound on (key << 32 | ~idx)
    if (k_done > 0) {
        bound = (static_cast<unsigned long long>(rank_key(orow_score[-1], !l2)) << 32) | (0xffffffffu - static_cast<uint32_t>(orow_idx[-1]));
    }
    const uint32_t bkey = static_cast<uint32_t>(bound >> 32), bnidx = static_cast<uint32_t>(bound);
    auto eligible = [&](uint32_t u, long long n) {
        return k_done == 0 || u < bkey || (u == bkey && (0xffffffffu - static_cast<uint32_t>(n)) < bnidx);
    };
    auto key_of = [&](long long n) { return rank_key(row[n], !l2); };
    // ---- fast path: a threshold from a sorted sample that, with overwhelming probability, is not above the k-th
    // largest key and admits at most kKnnCand candidates; ONE pass over the row collects every key >= threshold, the
    // candidates are sorted exactly (ties by index).  Any miss (too few / too many candidates) falls through to the
    // exact 4-pass radix select below — the result is identical either way.
    if (fast_rank > 0) {
        __shared__ uint32_t s_samp[kKnnSample];
        const long long stride = N / kKnnSample;
        for (int i = tid; i < kKnnSample; i += 256) s_samp[i] = key_of(static_cast<long long>(i) * stride);
        __syncthreads();
        bitonic_sort_desc(s_samp, kKnnSample, tid);
        const uint32_t thr = s_samp[fast_rank - 1];
        if (tid == 0) s_cnt_gt = 0;
        __syncthreads();
        auto push = [&](uint32_t u, long long n) {
            if (u >= thr && eligible(u, n)) {
                const uint32_t pos = atomicAdd(&s_cnt_gt, 1u);
                if (pos < static_cast<uint32_t>(kKnnCand))
                    s_pair[pos] = (static_cast<unsigned long long>(u) << 32) | (0xffffffffu - static_cast<uint32_t>(n));
            }
        };
        // the row starts 16-byte aligned (ldS % 4 == 0): four 128-bit loads in flight per thread
        const float4 *row4 = reinterpret_cast<const float4 *>(row);
        const long long n4 = N / 4;
        for (long long base = tid; base < n4; base += 256 * 4) {
            float4 v[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const long long i = base + b * 256;
                v[b] = i < n4 ? __ldg(row4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            // keys of the 16 values, one bit per value that reaches the threshold, ONE counter bump for the thread
            uint32_t keys[16], mask = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const float e[4] = {v[b].x, v[b].y, v[b].z, v[b].w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    keys[4 * b + j] = rank_key(e[j], !l2);
                    if (base + b * 256 < n4 && keys[4 * b + j] >= thr && eligible(keys[4 * b + j], 4 * (base + b * 256) + j))
                        mask |= 1u << (4 * b + j);
                }
            }
            if (mask) {
                uint32_t pos = atomicAdd(&s_cnt_gt, static_cast<uint32_t>(__popc(mask)));
#pragma unroll
                for (int t = 0; t < 16; ++t) {
                    if ((mask >> t) & 1u) {
                        const long long n = 4 * (base + (t >> 2) * 256) + (t & 3);
                        if (pos < static_cast<uint32_t>(kKnnCand))
                            s_pair[pos] = (static_cast<unsigned long long>(keys[t]) << 32) | (0xffffffffu - static_cast<uint32_t>(n));
                        ++pos;
                    }
                }
            }
        }
        for (long long n = 4 * n4 + tid; n < N; n += 256) push(key_of(n), n);
        __syncthreads();
        const uint32_t cnt = s_cnt_gt;
        __syncthreads();
        if (cnt >= static_cast<uint32_t>(k) && cnt <= static_cast<uint32_t>(kKnnCand)) {
            __shared__ unsigned long long s_pref;
            select_top_pairs(s_pair, cnt, k, P, s_pair + kKnnCand, orow_idx, orow_score, !l2, s_hist, &s_need, &s_pref, &s_cnt_gt, tid);
            return;
        }
    }
    // ---- radix select of the k-th largest key
    if (tid == 0) s_prefix = 0, s_need = static_cast<uint32_t>(k);
    __syncthreads();
    for (int shift = 24; shift >= 0; shift -= 8) {
        s_hist[tid] = 0;
        __syncthreads();
        const uint32_t prefix = s_prefix;
        const uint32_t mask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
        for (long long n = tid; n < N; n += 256) {
            const uint32_t u = key_of(n);
            if ((u & mask) == prefix && eligible(u, n)) atomicAdd(&s_hist[(u >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (tid < 32) {
            __shared__ uint32_t s_digit;
            radix_pick_digit(s_hist, s_need, tid, &s_digit, &s_need);     // s_need: keys with this digit (and prefix) still wanted
            __syncwarp();
            if (tid == 0) s_prefix = prefix | (s_digit << shift);
        }
        __syncthreads();
    }
    const uint32_t T = s_prefix;                 // k-th largest key
    const uint32_t need_eq = s_need;             // entries equal to T to take, in index order
    if (tid == 0) s_cnt_gt = 0;
    for (int i = tid; i < P; i += 256) s_pair[i] = 0ull;
    __syncthreads();
    const uint32_t n_gt = static_cast<uint32_t>(k) - need_eq;
    uint32_t eq_base = 0;
    for (long long n0 = 0; n0 < N; n0 += 256) {
        const long long n = n0 + tid;
        uint32_t u = 0;
        bool gt = false, eq = false;
        if (n < N) {
            u = key_of(n);
            const bool el = eligible(u, n);
            gt = el && u > T, eq = el && u == T;
        }
        if (gt) {
            const uint32_t pos = atomicAdd(&s_cnt_gt, 1u);
            s_pair[pos] = (static_cast<unsigned long long>(u) << 32) | (0xffffffffu - static_cast<uint32_t>(n));
        }
        // ordered compaction of the == T entries: warp ballots + per-warp totals (index order is preserved)
        const uint32_t ballot = __ballot_sync(0xffffffffu, eq);
        const int lane = tid & 31, wid = tid >> 5;
        if (lane == 0) s_scan[wid] = __popc(ballot);
        __syncthreads();
        uint32_t before = eq_base, chunk_total = 0;
        for (int w = 0; w < 8; ++w) {
            const uint32_t c = s_scan[w];
            if (w < wid) before += c;
            chunk_total += c;
        }
        eq_base += chunk_total;                  // identical in every thread: no shared running counter
        if (eq) {
            const uint32_t pos = before + __popc(ballot & ((1u << lane) - 1u));
            if (pos < need_eq)
                s_pair[n_gt + pos] = (static_cast<unsigned long long>(u) << 32) | (0xffffffffu - static_cast<uint32_t>(n));
        }
        __syncthreads();                         // s_scan is rewritten by the next chunk
    }
    __syncthreads();
    bitonic_sort_desc(s_pair, P, tid);                // padding zeros sink to the end
    for (int i = tid; i < k; i += 256) {
        const unsigned long long pr = s_pair[i];
        const uint32_t u = static_cast<uint32_t>(pr >> 32);
        const uint32_t n = 0xffffffffu - static_cast<uint32_t>(pr);
        orow_idx[i] = static_cast<int64_t>(n);
        orow_score[i] = rank_key_inv(u, !l2);
    }
}

// Top-k of a candidate list written by the filtering epilogue of the tensor-core scorer (knn_tc.cu): one CTA per query;
// cnt pairs (key << 32 | ~idx), all distinct, staged in shared memory for select_top_pairs.  A list that is too short
// (threshold above the k-th neighbour) or overflowed raises *fail: the caller's gated launches then redo the whole call
// through the score matrix.
__global__ void __launch_bounds__(256) knn_select_cand_kernel(const unsigned long long *__restrict__ cand, const uint32_t *__restrict__ cand_cnt,
                                                              uint32_t cap, int k, int64_t *__restrict__ idx_out,
                                                              float *__restrict__ score_out, uint32_t *__restrict__ fail) {
    extern __shared__ __align__(16) unsigned char knn_smem[];
    unsigned long long *s_pair = reinterpret_cast<unsigned long long *>(knn_smem);    // [cap], then the top array [P]
    __shared__ uint32_t s_hist[256];
    __shared__ uint32_t s_need, s_cnt;
    __shared__ unsigned long long s_pref;
    const int tid = threadIdx.x;
    const uint32_t cnt = cand_cnt[blockIdx.x];
    if (cnt < static_cast<uint32_t>(k) || cnt > cap) {
        if (tid == 0) *fail = 1u;
        return;
    }
    const int P = pow2_ceil(k);
    const unsigned long long *list = cand + static_cast<size_t>(blockIdx.x) * cap;
    for (uint32_t i = tid; i < cnt; i += 256) s_pair[i] = list[i];
    select_top_pairs(s_pair, cnt, k, P, s_pair + cap, idx_out + static_cast<size_t>(blockIdx.x) * k,
                     score_out + static_cast<size_t>(blockIdx.x) * k, true, s_hist, &s_need, &s_pref, &s_cnt, tid);
}

// thr[q] = rank-th largest score of the sample row (the last of the sorted top-`rank` list the select kernel wrote)
__global__ void __launch_bounds__(256) knn_threshold_kernel(const float *__restrict__ top, int rank, int Q, float *__restrict__ thr,
                                                            uint32_t *__restrict__ cand_cnt, uint32_t *__restrict__ fail) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q == 0) *fail = 0u;
    if (q < Q) {
        thr[q] = top[static_cast<size_t>(q) * rank + rank - 1];
        cand_cnt[q] = 0u;
    }
}

}  // namespace b200

using namespace b200;

extern "C" {

// tensor-core scorer: inner-product metrics, unless B200_KNN_TC=0
static bool knn_use_tc(int metric_l2) {
    if (metric_l2) return false;       // |q|^2 + |r|^2 - 2<q,r> cancels for near neighbours: keep exact float32 products
    const char *e = getenv("B200_KNN_TC");
    return !(e && e[0] == '0');
}
static long long knn_ld(long long N) { return round_up<long long>(N, 4); }

constexpr uint32_t kKnnFusedCap = 8192;      // candidate pairs per query of the fused path (64 KB of shared memory in the select)
constexpr int kKnnSampleStride = 16;         // the threshold pass scores every 16th reference row

// sample rank whose score is, with ~5 sigma confidence, not above the k-th neighbour's; 0: the fused path does not apply
static int knn_fused_rank(long long N, int k) {
    const long long ns = N / kKnnSampleStride;
    if (ns < 4 * kKnnSample || k > kKnnMaxK) return 0;
    const double ks = static_cast<double>(k) / kKnnSampleStride;
    const double r = ks + 5.0 * sqrt(ks) + 2.0;
    const double expect = r * kKnnSampleStride;                                   // candidates per query
    if (r > kKnnMaxK || expect + 5.0 * sqrt(r) * kKnnSampleStride > 0.9 * kKnnFusedCap) return 0;
    return static_cast<int>(r + 0.5);
}

size_t b200_knn_workspace_bytes(int Q, long long N, int D, int k) {
    (void)k;
    if (Q < 1 || N < 1) return 0;
    // score matrix (always provisioned: the fused path falls back to it), norms, fused-path scratch, bf16 copies
    const size_t fused = round_up<size_t>(static_cast<size_t>(Q) * kKnnFusedCap * sizeof(unsigned long long), 256) +
                         round_up<size_t>(static_cast<size_t>(Q) * (kKnnMaxK * 12 + 16), 256) + 256;
    return round_up<size_t>(static_cast<size_t>(Q) * knn_ld(N) * sizeof(float), 256) + round_up<size_t>((Q + N) * sizeof(float), 256) +
           fused + knn_tc_extra_workspace(Q, N, D);
}

// ranks k_done .. of every row from the score matrix, kKnnMaxK per launch
static int knn_select_passes(const float *S, long long N, long long ldS, int Q, int k, int metric_l2, int64_t *idx, float *score,
                             const uint32_t *gate, cudaStream_t st) {
    B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(knn_select_kernel), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>((kKnnCand + kKnnMaxK) * sizeof(unsigned long long))));
    for (int done = 0; done < k; done += kKnnMaxK) {
        const int kp = k - done < kKnnMaxK ? k - done : kKnnMaxK;
        const int P = pow2_ceil(kp);
        // one-pass threshold path: sample rank r such that P(threshold above the last wanted rank) ~ 4 sigma, and the
        // expected number of eligible keys >= threshold (plus 4 sigma) fits the candidate buffer; else the radix select alone
        int fast_rank = 0;
        if (N >= 16 * kKnnSample) {
            const double p = static_cast<double>(done + kp) / static_cast<double>(N), m = kKnnSample;
            const double r = p * m + 4.0 * sqrt(p * m) + 2.0;
            const double expect = r / m * static_cast<double>(N) - done;
            if (r < m / 2 && expect + 4.0 * sqrt(r) / m * static_cast<double>(N) <= kKnnCand) fast_rank = static_cast<int>(r + 0.5);
        }
        const size_t smem = static_cast<size_t>(fast_rank ? kKnnCand + P : P) * sizeof(unsigned long long);
        knn_select_kernel<<<Q, 256, smem, st>>>(S, N, ldS, kp, metric_l2, fast_rank, idx, score, k, done, gate);
        B200_LAUNCH_CHECK("knn_select_kernel");
    }
    return B200_OK;
}

// Top-k of every row of a score matrix that is already on the device: idx int64 [Q][k] (column numbers), score [Q][k];
// largest != 0: largest first, else smallest first; ties to the smaller column.  The merge step of a sharded k-NN: the
// per-shard lists concatenated shard by shard are such a matrix (column order = global index order among equal scores).
int b200_select_topk_f32(const float *S, int Q, long long N, long long ldS, int k, int largest, int64_t *idx, float *score,
                         b200_stream_t stream) {
    if (!S || !idx || !score || Q < 1 || N < 1 || k < 1 || k > N || ldS < N) return B200_ERR_INVALID_ARG;
    if ((ldS & 3) || (reinterpret_cast<uintptr_t>(S) & 15) || N >= (1ll << 32) - 1) return B200_ERR_ALIGNMENT;
    return knn_select_passes(S, N, ldS, Q, k, largest ? 0 : 1, idx, score, nullptr, as_stream(stream));
}

int b200_knn_topk(const float *refs, const float *queries, int Q, long long N, int D, int k, int metric_l2, int64_t *idx,
                  float *score, void *workspace, size_t workspace_bytes, b200_stream_t stream) {
    if (!refs || !queries || !idx || !score || Q < 1 || N < 1 || D < 1 || k < 1) return B200_ERR_INVALID_ARG;
    if (k > N) return B200_ERR_INVALID_ARG;
    if ((D & 3) || N >= (1ll << 32) - 1) return B200_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < b200_knn_workspace_bytes(Q, N, D, k)) return B200_ERR_WORKSPACE;
    if ((reinterpret_cast<uintptr_t>(refs) | reinterpret_cast<uintptr_t>(queries)) & 15) return B200_ERR_ALIGNMENT;
    cudaStream_t st = as_stream(stream);
    const long long ldS = knn_ld(N);
    unsigned char *w = static_cast<unsigned char *>(workspace);
    float *S = reinterpret_cast<float *>(w);
    size_t off = round_up<size_t>(static_cast<size_t>(Q) * ldS * sizeof(float), 256);
    float *qn = reinterpret_cast<float *>(w + off);
    float *rn = qn + Q;
    off += round_up<size_t>((Q + N) * sizeof(float), 256);
    unsigned long long *cand = reinterpret_cast<unsigned long long *>(w + off);
    off += round_up<size_t>(static_cast<size_t>(Q) * kKnnFusedCap * sizeof(unsigned long long), 256);
    unsigned char *fz = w + off;                               // fused scratch: sample top list (idx, score), thr, counters
    off += round_up<size_t>(static_cast<size_t>(Q) * (kKnnMaxK * 12 + 16), 256) + 256;
    void *extra = w + off;
    if (knn_use_tc(metric_l2)) {
        TcContext ctx;
        const int rank = knn_fused_rank(N, k);
        const int rc = knn_tc_prepare(queries, refs, Q, N, D, extra, rank ? kKnnSampleStride : 0, &ctx, st);
        if (rc == B200_OK) {
            const uint32_t *gate = nullptr;
            if (rank) {
                // ---- fused path: threshold from a sampled pass, then the full GEMM keeps only the candidates
                const long long ns = N / kKnnSampleStride, lds = knn_ld(ns);
                int64_t *top_idx = reinterpret_cast<int64_t *>(fz);
                float *top_score = reinterpret_cast<float *>(fz + static_cast<size_t>(Q) * rank * 8);
                float *thr = top_score + static_cast<size_t>(Q) * rank;
                uint32_t *cand_cnt = reinterpret_cast<uint32_t *>(thr + Q);
                uint32_t *fail = cand_cnt + Q;
                if (int e = knn_tc_scores(&ctx, 1, S, lds, nullptr, nullptr, nullptr, 0, nullptr, st)) return e;      // sample scores in S
                if (int e = knn_select_passes(S, ns, lds, Q, rank, 0, top_idx, top_score, nullptr, st)) return e;
                knn_threshold_kernel<<<ceil_div(Q, 256), 256, 0, st>>>(top_score, rank, Q, thr, cand_cnt, fail);
                B200_LAUNCH_CHECK("knn_threshold_kernel");
                if (int e = knn_tc_scores(&ctx, 0, nullptr, 0, thr, cand, cand_cnt, kKnnFusedCap, nullptr, st)) return e;
                const size_t smem = (static_cast<size_t>(kKnnFusedCap) + pow2_ceil(k)) * sizeof(unsigned long long);
                B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(knn_select_cand_kernel),
                                                   cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   static_cast<int>((kKnnFusedCap + kKnnMaxK) * sizeof(unsigned long long))));
                knn_select_cand_kernel<<<Q, 256, smem, st>>>(cand, cand_cnt, kKnnFusedCap, k, idx, score, fail);
                B200_LAUNCH_CHECK("knn_select_cand_kernel");
                // any list too short / overflowed: the launches below redo the call through the score matrix, else they return at once
                gate = fail;
            }
            if (int e = knn_tc_scores(&ctx, 0, S, ldS, nullptr, nullptr, nullptr, 0, gate, st)) return e;
            return knn_select_passes(S, N, ldS, Q, k, 0, idx, score, gate, st);
        }
        if (rc != B200_ERR_UNSUPPORTED) return rc;
    }
    if (metric_l2) {
        row_sqnorm_kernel<<<ceil_div(Q, 8), 256, 0, st>>>(queries, Q, D, qn);
        B200_LAUNCH_CHECK("row_sqnorm_kernel");
        row_sqnorm_kernel<<<static_cast<unsigned>(ceil_div<long long>(N, 8)), 256, 0, st>>>(refs, N, D, rn);
        B200_LAUNCH_CHECK("row_sqnorm_kernel");
    }
    const dim3 grid(static_cast<unsigned>(ceil_div<long long>(N, kBN)), ceil_div(Q, kBM));
    knn_scores_kernel<kEpiScore><<<grid, 256, 0, st>>>(queries, refs, S, Q, N, ldS, D, metric_l2, qn, rn, 0.f);
    B200_LAUNCH_CHECK("knn_scores_kernel");
    return knn_select_passes(S, N, ldS, Q, k, metric_l2, idx, score, nullptr, st);
}

int b200_real_hamming_dist(const float *q, const float *db, int Q, long long N, int D, int nbits, float *dist, long long ldS,
                           b200_stream_t stream) {
    if (Q < 0 || N < 0 || D < 1 || nbits < 1 || nbits > D || ldS < N) return B200_ERR_INVALID_ARG;
    if (Q > 0 && N > 0 && (!q || !db || !dist)) return B200_ERR_INVALID_ARG;
    if ((D & 3) || ceil_div(Q, kBM) > 65535) return B200_ERR_UNSUPPORTED;
    if ((ldS & 3) || ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(db) | reinterpret_cast<uintptr_t>(dist)) & 15))
        return B200_ERR_ALIGNMENT;
    if (Q == 0 || N == 0) return B200_OK;
    const dim3 grid(static_cast<unsigned>(ceil_div<long long>(N, kBN)), ceil_div(Q, kBM));
    knn_scores_kernel<kEpiRealHamming><<<grid, 256, 0, as_stream(stream)>>>(q, db, dist, Q, N, ldS, D, 0, nullptr, nullptr,
                                                                             static_cast<float>(nbits));
    B200_LAUNCH_CHECK("knn_scores_kernel");
    return B200_OK;
}

}  // extern "C"
