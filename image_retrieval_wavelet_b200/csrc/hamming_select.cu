// Select pipeline of the Hamming mAP@k / top-k evaluator: the B200 form of
//   CustomCalculator.calculate_maphashing   /root/reference/main/engine/accuracy_calculator.py:203-231
// for the usual case that the k ranks that count are a small part of the database (COCO: 5000 of 117 218 rows).
//
// The three-stage counting sort (hamming_map.cu) pays ~25 instructions for EVERY (row, query) pair: score, label
// test, histogram bump, one byte of stash.  But a row can only matter when its distance is at most d*(q), the
// distance of the query's k-th neighbour — 4 % of the rows on the COCO shape.  So:
//   (P) a sampled histogram (every sel_stride-th 32-row group, ~k/256 of the rows, distances only, one global plane)
//       gives each query a bound b(q): the smallest distance whose sampled count, scaled up, covers k with a
//       5-sigma margin                                                           (select_sample/bound kernels)
//   (A) ONE pass over the packed database: XOR + POPC + compare per pair (16 instructions at 128 bits, no label
//       read, no counters in shared memory); a thread owns a query and appends the few rows within its bound —
//       (row, distance, relevance) in index order — to its per-(query, segment) candidate list, chunks of a global
//       pool                                                                     (hamming_select_kernel)
//   (B) one WARP per query counting-sorts its own list: histogram by distance, scan, d*, then a second walk in index
//       order gives every row its rank (distance base + running count, ties by index) and hit ordinal; AP terms are
//       the same exact 2^-40 fixed-point float32 quotients as the three-stage path    (hamming_select_rank_kernel)
// Exactness does not rest on the sample: a list shorter than k means the bound was too tight, and that query is redone
// with the bound lifted to "all rows" (second round of A and B, empty otherwise); if the candidate pool overflows
// (collapsed codes: every row ties) a device flag hands the whole problem to the three-stage path, whose kernels are
// launched behind that flag and return at once otherwise.  No host synchronisation anywhere: the sequence is
// CUDA-graph capturable.
#include "common.cuh"
#include "hamming_core.cuh"
#include "hamming_plan.h"
#include "tc_common.cuh"

namespace b200 {

// flags: uint32 [64] at plan->off_sel_flags
constexpr int kFlagCursor = 0;     // next free pool chunk (one pool)
constexpr int kFlagSubCursor = 32; // [32..63] next free chunk of sub-pool i (the pool split 32 ways: a CTA allocates from sub-pool
                                   // (segment x groups + group) % 32 — ~500 k same-address atomics on c3 become 32 streams)
constexpr int kSubPools = 32;
constexpr int kFlagFallback = 1;   // != 0: the select pipeline gave up, the three-stage path computes everything
constexpr int kFlagRetry = 2;      // number of queries whose list was shorter than k (round 1 redoes them)
constexpr int kFlagEst = 4;        // [4..5] uint64: estimated total number of candidates (from the sample)
constexpr uint32_t kBoundInactive = 1u << 30, kBoundRetry = 1u << 31;

struct SelArgs {
    const uint64_t *q_codes, *q_labels, *db_codes, *db_labels;
    uint32_t *bound;          // [Qpad]: bits 0-15 distance bound, bit 30 padding query, bit 31 redo with the bound lifted
    U32x2 *head;              // [Qpad][S] per list: (number of candidates, pool chunk of its first chunk)
    uint32_t *table;          // [Qpad][S][maxc] pool chunk of the c-th chunk of a list, c >= 1
    uint32_t *pool;           // [pool_chunks][chunk] entries: row-in-segment | distance << 16 | relevant << 24
    uint32_t *flags;
    uint32_t *status;         // or null: set to 1 when this launch sequence cannot finish by itself (a retry round or the fallback is needed)
    double *ap;               // [Q] or null
    uint32_t *tsum;           // [Q] or null
    uint32_t *rank_idx;       // [Q][k] or null
    uint16_t *rank_dist;      // [Q][k] or null
    unsigned long long est_cap;
    long long index_base;
    int Q, N, S, seg_len, tile, Qpad, ch_shift, maxc, bins, round;
    int stage;                // rank kernel: shared memory for the staged form was requested (S <= kStageMaxSeg)
    int seg0;                 // select kernel: first segment of this launch (a streamed evaluation launches segment ranges)
    int stage_cap;            // rank kernel: entries of shared memory of the staged form (<= kStageCap)
    uint32_t nsub, sub_chunks; // pool split: number of sub-pools (1 or kSubPools) and chunks of each
    uint32_t *mask;           // tensor-core filter: [32-row group][Qpad] hit masks (bit i: row 32 g + i is within the query's bound)
    uint32_t pool_chunks, k;
};

// Population count of NW 32-bit words.  POPC is a quarter-rate XU instruction (16 lanes/clk/SM) and the one pipe this
// kernel saturates, so word triples first go through a carry-save adder (two LOP3 on the full-rate ALU pipe):
// popc(a) + popc(b) + popc(c) = popc(a ^ b ^ c) + 2 popc(maj(a, b, c)) — 3 POPC instead of 4 for 128-bit codes, 4
// instead of 8 for 256-bit codes.
__device__ __forceinline__ void csa(uint32_t a, uint32_t b, uint32_t c, uint32_t &sum, uint32_t &carry) {
    sum = a ^ b ^ c;
    carry = (a & b) | (c & (a | b));          // one LOP3 each
}
template <int NW>
__device__ __forceinline__ uint32_t popc_words(const uint32_t *x) {
    if constexpr (NW == 2) {
        return __popc(x[0]) + __popc(x[1]);
    } else if constexpr (NW == 4) {
        uint32_t s, c;
        csa(x[0], x[1], x[2], s, c);
        return __popc(s) + __popc(x[3]) + 2u * __popc(c);
    } else {
        static_assert(NW == 8, "codes are 1, 2 or 4 uint64 words");
        uint32_t s1, c1, s2, c2, s3, c3, s4, c4;
        csa(x[0], x[1], x[2], s1, c1);
        csa(x[3], x[4], x[5], s2, c2);
        csa(s1, s2, x[6], s3, c3);
        csa(c1, c2, c3, s4, c4);
        return __popc(s3) + __popc(x[7]) + 2u * __popc(s4) + 4u * __popc(c4);
    }
}

template <int CW>
__device__ __forceinline__ uint32_t code_dist(const uint32_t *s_codes, int j, const uint32_t *qc) {
    uint32_t x[2 * CW];
    if constexpr (CW == 1) {
        const U32x2 v = reinterpret_cast<const U32x2 *>(s_codes)[j];
        x[0] = v.x ^ qc[0], x[1] = v.y ^ qc[1];
    } else {
#pragma unroll
        for (int i = 0; i < CW / 2; ++i) {
            const U32x4 v = reinterpret_cast<const U32x4 *>(s_codes)[j * (CW / 2) + i];
            x[4 * i] = v.x ^ qc[4 * i], x[4 * i + 1] = v.y ^ qc[4 * i + 1], x[4 * i + 2] = v.z ^ qc[4 * i + 2], x[4 * i + 3] = v.w ^ qc[4 * i + 3];
        }
    }
    return popc_words<2 * CW>(x);
}

// ------------------------------------------------------------------------------------------------ (P) sample
// Sample row r is database row 32 * stride * (r / 32) + r % 32 (whole 32-row groups, read in place: 512 contiguous bytes
// at 128 bits).  One THREAD owns one query; a CTA scores one segment of the sample, staged through shared memory like
// the select kernel's tiles, and counts distances in a private column of 16|16-bit shared counters (one conflict-free
// shared atomic per pair: a segment has at most 65535 rows); the columns are then added to the ONE global plane
// hist[bins][Qpad] (zeroed with the flags).  No labels, no per-segment planes: the bound needs distance counts only.
// (Round 2, first form: stage A's kernel of the three-stage path on a gathered copy of the sample — label test, stash
// logic and an 11-plane 29 MB histogram that the bound kernel read back: 54 + 26 us on c3 for 1/19 of the pairs.)
constexpr int kSampleTile = 256;      // rows per staged tile (multiple of 32)

template <int CW>
__global__ void __launch_bounds__(512) select_sample_kernel(const uint64_t *__restrict__ q_codes, const uint64_t *__restrict__ db_codes,
                                                            uint32_t *__restrict__ hist, long long smp_rows, int stride, int seg_len,
                                                            int Q, int Qpad, int bins) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint32_t *s_codes = reinterpret_cast<uint32_t *>(smem_raw);                          // [kSampleTile][2 CW]
    uint32_t *s_h = s_codes + static_cast<size_t>(kSampleTile) * 2 * CW;                 // [(bins + 1) / 2][T]
    // block (T, R): thread (t, r) scores rows r, r + R, ... of every tile for query t — R warps share a query's column,
    // which keeps an SM busy with few CTAs (a column block is zeroed and merged once per CTA)
    const int T = blockDim.x, R = blockDim.y, t = threadIdx.x, r = threadIdx.y;
    const int tid = r * T + t, nthreads = T * R;
    const int q = blockIdx.x * T + t;
    const int words = (bins + 1) >> 1;
    for (int i = tid; i < words * T; i += nthreads) s_h[i] = 0u;
    uint32_t qc[2 * CW];
    {
        const int qq = q < Q ? q : Q - 1;
        const uint32_t *pc = reinterpret_cast<const uint32_t *>(q_codes) + static_cast<size_t>(qq) * 2 * CW;
#pragma unroll
        for (int i = 0; i < 2 * CW; ++i) qc[i] = pc[i];
    }
    const long long seg_begin = static_cast<long long>(blockIdx.y) * seg_len;             // multiples of 32
    const long long seg_end = seg_begin + seg_len < smp_rows ? seg_begin + seg_len : smp_rows;
    for (long long tile0 = seg_begin; tile0 < seg_end; tile0 += kSampleTile) {
        const int n = static_cast<int>(kSampleTile < seg_end - tile0 ? kSampleTile : seg_end - tile0);      // a multiple of 32
        __syncthreads();                          // zeroed counters / the previous tile's readers
        // 16-byte pieces; group g of the tile = sample rows tile0 + 32 g ..., database rows from (tile0 / 32 + g) * stride * 32
        constexpr int kPiecesPerGroup = CW >= 2 ? 32 * (CW / 2) : 16;
        const int pieces = (n / 32) * kPiecesPerGroup;
        for (int i = tid; i < pieces; i += nthreads) {
            const int g = i / kPiecesPerGroup, o = i - g * kPiecesPerGroup;
            const uint4 *src = reinterpret_cast<const uint4 *>(db_codes + ((tile0 >> 5) + g) * stride * 32 * CW) + o;
            reinterpret_cast<uint4 *>(s_codes)[i] = __ldg(src);
        }
        __syncthreads();
#pragma unroll 4
        for (int j = r; j < n; j += R) {
            const uint32_t d = code_dist<CW>(s_codes, j, qc);
            atomicAdd(s_h + (d >> 1) * T + t, 1u << ((d & 1u) * 16u));
        }
    }
    __syncthreads();
    if (q >= Q) return;
    for (int w = r; w < words; w += R) {
        const uint32_t c = s_h[w * T + t];
        if (c & 0xffffu) atomicAdd(hist + static_cast<size_t>(2 * w) * Qpad + q, c & 0xffffu);
        if (c >> 16) atomicAdd(hist + static_cast<size_t>(2 * w + 1) * Qpad + q, c >> 16);
    }
}

// hist: uint32 [bins][Qpad] sampled rows of (distance, query).
// CTA = 32 queries (x) x 32 distance lanes (y): the counts are fetched in parallel over the distances, then the y == 0
// warp walks the distances of its 32 queries.
__global__ void __launch_bounds__(1024) select_bound_kernel(const uint32_t *__restrict__ hist, int bins, int Qpad, int Q,
                                                            uint32_t target, float inv_frac, uint32_t *__restrict__ bound,
                                                            uint32_t *__restrict__ flags) {
    __shared__ uint32_t s_tot[B200_MAX_CODE_BITS + 1][32];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int q = blockIdx.x * 32 + tx;                    // < Qpad: Qpad is a multiple of 32
    for (int d = ty; d < bins; d += 32) s_tot[d][tx] = hist[static_cast<size_t>(d) * Qpad + q];
    __syncthreads();
    if (ty != 0) return;
    unsigned long long est = 0;
    if (q >= Q) {
        bound[q] = kBoundInactive;
    } else {
        uint32_t cum = 0, b = static_cast<uint32_t>(bins - 1);
        for (int d = 0; d < bins; ++d) {
            cum += s_tot[d][tx];
            if (cum >= target) {
                b = static_cast<uint32_t>(d);
                break;
            }
        }
        bound[q] = b;
        est = static_cast<unsigned long long>(static_cast<float>(cum) * inv_frac);      // expected list length of this query
    }
    for (int o = 16; o > 0; o >>= 1) est += __shfl_down_sync(0xffffffffu, est, o);
    if (tx == 0) atomicAdd(reinterpret_cast<unsigned long long *>(flags + kFlagEst), est);
}

// ------------------------------------------------------------------------------------------------ (A) select
template <int LW, bool EQ>
__device__ __forceinline__ bool label_rel(const uint32_t *s_labs, int j, const uint32_t *ql) {
    uint32_t l[2 * LW];
    if constexpr (LW == 1) {
        const U32x2 v = reinterpret_cast<const U32x2 *>(s_labs)[j];
        l[0] = v.x, l[1] = v.y;
    } else {
#pragma unroll
        for (int i = 0; i < LW / 2; ++i) {
            const U32x4 v = reinterpret_cast<const U32x4 *>(s_labs)[j * (LW / 2) + i];
            l[4 * i] = v.x, l[4 * i + 1] = v.y, l[4 * i + 2] = v.z, l[4 * i + 3] = v.w;
        }
    }
    if constexpr (EQ) return ql[0] == l[0] && ql[1] == l[1];
    uint32_t any = 0;
#pragma unroll
    for (int i = 0; i < 2 * LW; ++i) any |= ql[i] & l[i];
    return any != 0;
}

// One THREAD owns one query (code, labels, bound in registers); the CTA walks one database segment staged through
// shared memory tile by tile, so a row is one broadcast shared-memory read for the warp.  32 rows are scored back to
// back (LDS + 4 XOR + 2 CSA + 3 POPC + 2 adds + compare per row at 128 bits; the distances are kept as packed bytes),
// then each thread appends its few candidates of the group — row order — to its (query, segment) list.
// Measured alternative (round 2, kept out): lanes = rows, loop over queries, one ballot per 32 pairs and a
// warp-uniform append per non-empty ballot — 13 instructions per 32 pairs to score, but 45 per append with only ~2
// candidate lanes each (87 % of the ballots are non-empty at 6 % candidates): 1.69 ms against 0.73 ms on c3.
// MASKED: the append half of the tensor-core form (A') — which rows are within the bound comes from the filter kernel's hit
// masks; only those rows are scored here (the distance their list entry carries).
template <int CW, int LW, bool EQ, bool MASKED = false>
__global__ void __launch_bounds__(128) hamming_select_kernel(const __grid_constant__ SelArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint32_t *s_codes = reinterpret_cast<uint32_t *>(smem_raw);
    uint32_t *s_labs = s_codes + static_cast<size_t>(a.tile) * 2 * CW;
    const int T = blockDim.x, t = threadIdx.x;
    const int q = blockIdx.x * T + t, seg = blockIdx.y + a.seg0;
    volatile uint32_t *vflags = a.flags;
    {
        // one thread decides for the CTA (another CTA may raise the fallback flag at any moment)
        bool quit = false;
        if (t == 0) {
            quit = vflags[kFlagFallback] != 0u;
            if (a.round == 0) {
                const unsigned long long est = *reinterpret_cast<volatile unsigned long long *>(a.flags + kFlagEst);
                if (est > a.est_cap) {         // the lists would not fit the pool: every CTA sees the same total and leaves
                    vflags[kFlagFallback] = 1u;
                    if (a.status) *a.status = 1u;
                    quit = true;
                }
            } else if (vflags[kFlagRetry] == 0u) {
                quit = true;
            }
        }
        if (__syncthreads_or(quit)) return;
    }
    const uint32_t bw = a.bound[q];
    const bool active = a.round == 0 ? !(bw & kBoundInactive) : (bw & kBoundRetry) != 0;
    if (!__syncthreads_or(active)) return;
    const int bnd = !active ? -1 : (a.round == 0 ? static_cast<int>(bw & 0xffffu) : 0xffff);
    const bool warp_active = __any_sync(0xffffffffu, active);

    uint32_t qc[2 * CW], ql[2 * LW];
    {
        const int qq = q < a.Q ? q : a.Q - 1;
        const uint32_t *pc = reinterpret_cast<const uint32_t *>(a.q_codes) + static_cast<size_t>(qq) * 2 * CW;
        const uint32_t *pl = reinterpret_cast<const uint32_t *>(a.q_labels) + static_cast<size_t>(qq) * 2 * LW;
#pragma unroll
        for (int i = 0; i < 2 * CW; ++i) qc[i] = pc[i];
#pragma unroll
        for (int i = 0; i < 2 * LW; ++i) ql[i] = pl[i];
    }
    const int seg_begin = seg * a.seg_len;
    const int seg_end = seg_begin + a.seg_len < a.N ? seg_begin + a.seg_len : a.N;
    uint32_t *tab = a.table + (static_cast<size_t>(q) * a.S + seg) * a.maxc;       // [c] pool chunk c of this list (c >= 1)
    uint32_t first = 0;
    const uint32_t chmask = (1u << a.ch_shift) - 1u;
    uint32_t fill = 0, base = 0;
    bool dead = false;

    // The 32 distances of the current group, packed 4 per word, are parked in this thread's 32 bytes of shared memory (two
    // 128-bit stores per group) so that the candidate loop below can fetch "distance of row i" with one byte load instead
    // of a select chain over 8 registers — and can run over the whole 32-bit mask at once: the warp iterates
    // max-over-lanes(popcount) times, and one loop over 32 rows has a smaller maximum than two loops over 16.
    unsigned char *s_d = reinterpret_cast<unsigned char *>(s_labs + static_cast<size_t>(a.tile) * 2 * LW) + static_cast<size_t>(t) * 32;

    // candidates of the 32 scored rows (bit i of m = tile row row0 + i), lowest row first
    auto append = [&](uint32_t m, int row0, int seg_row0) {
        while (m) {
            const int i = __ffs(static_cast<int>(m)) - 1;
            m &= m - 1u;
            const int j = row0 + i;
            const uint32_t d = MASKED ? code_dist<CW>(s_codes, j, qc) : static_cast<uint32_t>(s_d[i]);
            const bool rel = label_rel<LW, EQ>(s_labs, j, ql);
            if ((fill & chmask) == 0u) {
                uint32_t c;
                if (a.nsub > 1) {
                    const uint32_t sub = (static_cast<uint32_t>(seg) * gridDim.x + blockIdx.x) & (kSubPools - 1);
                    const uint32_t local = atomicAdd(a.flags + kFlagSubCursor + sub, 1u);
                    c = local < a.sub_chunks ? sub * a.sub_chunks + local : 0xffffffffu;
                } else {
                    c = atomicAdd(a.flags + kFlagCursor, 1u);
                }
                if (c >= a.pool_chunks) {
                    dead = true;
                    vflags[kFlagFallback] = 1u;
                    if (a.status) *a.status = 1u;
                } else {
                    if (fill == 0u)
                        first = c;
                    else
                        tab[fill >> a.ch_shift] = c;
                    base = c << a.ch_shift;
                }
            }
            if (!dead) a.pool[static_cast<size_t>(base) + (fill & chmask)] = static_cast<uint32_t>(seg_row0 + j) | (d << 16) | (static_cast<uint32_t>(rel) << 24);
            ++fill;
        }
    };

    for (int tile0 = seg_begin; tile0 < seg_end; tile0 += a.tile) {
        const int n = a.tile < seg_end - tile0 ? a.tile : seg_end - tile0;
        uint32_t mw[8];                       // MASKED: this query's hit masks of the tile's (<= 8) 32-row groups, requested ahead of the staging
        if constexpr (MASKED) {
#pragma unroll
            for (int g = 0; g < 8; ++g) mw[g] = 32 * g < n ? a.mask[static_cast<size_t>((tile0 >> 5) + g) * a.Qpad + q] : 0u;
        }
        {
            const uint4 *gc = reinterpret_cast<const uint4 *>(a.db_codes + static_cast<size_t>(tile0) * CW);
            const uint4 *gl = reinterpret_cast<const uint4 *>(a.db_labels + static_cast<size_t>(tile0) * LW);
            const int nc = (n * CW + 1) / 2, nl = (n * LW + 1) / 2;
            for (int i = t; i < nc; i += T) reinterpret_cast<uint4 *>(s_codes)[i] = ldg_stream_u4(gc + i);
            for (int i = t; i < nl; i += T) reinterpret_cast<uint4 *>(s_labs)[i] = ldg_stream_u4(gl + i);
        }
        __syncthreads();
        if constexpr (MASKED) {
#pragma unroll
            for (int g = 0; g < 8; ++g)
                if (mw[g]) append(mw[g], 32 * g, tile0 - seg_begin);
        } else if (warp_active) {
            int j = 0;
            for (; j + 32 <= n; j += 32) {
                uint32_t m = 0, w[8];
#pragma unroll
                for (int b = 0; b < 8; ++b) {
                    uint32_t d[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        d[i] = code_dist<CW>(s_codes, j + 4 * b + i, qc);
                        if (static_cast<int>(d[i]) <= bnd) m |= 1u << (4 * b + i);
                    }
                    w[b] = d[0] | (d[1] << 8) | (d[2] << 16) | (d[3] << 24);
                }
                if (m) {                        // (a thread only reads its own 32 bytes: no barrier)
                    reinterpret_cast<U32x4 *>(s_d)[0] = U32x4{w[0], w[1], w[2], w[3]};
                    reinterpret_cast<U32x4 *>(s_d)[1] = U32x4{w[4], w[5], w[6], w[7]};
                    append(m, j, tile0 - seg_begin);
                }
            }
            for (; j < n; ++j) {                 // the last, partial group of a segment
                const uint32_t d = code_dist<CW>(s_codes, j, qc);
                if (static_cast<int>(d) <= bnd) {
                    s_d[0] = static_cast<unsigned char>(d);
                    append(1u, j, tile0 - seg_begin);
                }
            }
        }
        __syncthreads();
    }
    if (active) a.head[static_cast<size_t>(q) * a.S + seg] = U32x2{dead ? 0u : fill, first};
}

// ------------------------------------------------------------------------------------------------ (A') select on the tensor cores
// Runs where the plan allows it (plan_select_tc in hamming_plan.h).  The scoring moves off the POPC pipe: for +-1 codes <q, r> = B - 2 d, so the distances of 128
// queries x 256 rows are ONE tcgen05.mma chain over the codes expanded to e4m3 bytes (+1 = 0x38, -1 = 0xB8, padding
// columns 0; float32 accumulation of at most 256 terms of +-1 is exact).  Two kernels:
//   hamming_select_tc_kernel (FILTER)  warp 0 TMA producer (query tile 128 x 128 B + row tile 256 x 128 B per 128-column K
//               block and stage, 128-byte swizzle, 3 stages of 48 KB); warp 1 MMA issuer (4 x tcgen05.mma.kind::f8f6f4
//               M128 N256 K32 per stage into one of two TMEM accumulators); warps 2..5 epilogue: thread = query (TMEM
//               lane), tcgen05.ld 32 columns at a time, dot >= B - 2 bound -> one bit; the 32-bit hit mask of every
//               (32-row group, query) goes to mask[group][Qpad] (a warp stores 128 contiguous bytes).  Persistent over
//               work units (query tile, segment), query tile fastest: the CTAs running together share a segment's rows in L2.
//   hamming_select_append_kernel (APPEND)  the SIMT select kernel above with its scoring loop replaced by a read of the
//               thread's hit masks: only the rows within the bound (4-6 % on c3) are scored again (XOR + POPC from the
//               staged tile: the distance the list entry carries), label-tested and appended — in row order, to the same
//               lists, so the rank kernel does not know which form ran.
// First form (measured, replaced): the appends in the filter's epilogue — 4 warps per SM (one per TMEM lane quarter) with
// nothing to hide the latency of the per-candidate chain: 1.42 ms on c3 against 0.64 ms for the SIMT kernel (DESIGN 4.2).
constexpr int kStcBM = 128, kStcBN = 256, kStcBK = 128;
constexpr int kStcStages = 3;
constexpr uint32_t kStcABytes = kStcBM * 128, kStcBBytes = kStcBN * 128, kStcStageBytes = kStcABytes + kStcBBytes;
constexpr int kStcThreads = 192;
constexpr uint32_t kStcSmemBytes = kStcStages * kStcStageBytes + 1024 /*alignment*/ + 256 /*barriers*/;
// kind::f8f6f4: D float32, A / B e4m3 (format 0), both K-major, M = 128, N = 256
constexpr uint32_t kStcIdesc = (1u << 4) | (static_cast<uint32_t>(kStcBN >> 3) << 17) | (static_cast<uint32_t>(kStcBM >> 4) << 24);

__device__ __forceinline__ void tc_mma_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// codes: uint64 [rows][cw] -> e4m3 bytes [rows][Bp]: column b = bit b % 64 of word b / 64 (set: +1, clear: -1), 0 from column B on
__global__ void __launch_bounds__(256) select_expand_fp8_kernel(const uint64_t *__restrict__ codes, long long rows, int cw, int B, int Bp,
                                                                uint4 *__restrict__ out) {
    const int per_row = Bp >> 4;
    const long long n16 = rows * per_row;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n16; i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long r = i / per_row;
        const int bit0 = static_cast<int>(i - r * per_row) << 4;
        uint32_t bits = 0;
        if (bit0 < cw * 64) bits = static_cast<uint32_t>(codes[r * cw + (bit0 >> 6)] >> (bit0 & 63)) & 0xffffu;
        const int valid = B - bit0 < 0 ? 0 : (B - bit0 > 16 ? 16 : B - bit0);
        uint32_t w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint32_t v = 0;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int j = 4 * k + e;
                const uint32_t byte = j < valid ? (((bits >> j) & 1u) ? 0x38u : 0xB8u) : 0u;
                v |= byte << (8 * e);
            }
            w[k] = v;
        }
        out[i] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

struct StcMaps {
    CUtensorMap q, db;
};

__global__ void __launch_bounds__(kStcThreads, 1) hamming_select_tc_kernel(const __grid_constant__ StcMaps maps, const __grid_constant__ SelArgs a,
                                                                           int B, int nkb) {
    extern __shared__ unsigned char stc_smem_raw[];
    __shared__ uint32_t s_quit;
    volatile uint32_t *vflags = a.flags;
    if (threadIdx.x == 0) {
        // one thread decides for the CTA (another CTA may raise the fallback flag at any moment)
        bool quit = vflags[kFlagFallback] != 0u;
        if (a.round == 0) {
            const unsigned long long est = *reinterpret_cast<volatile unsigned long long *>(a.flags + kFlagEst);
            if (est > a.est_cap) {             // the lists would not fit the pool: every CTA sees the same total and leaves
                vflags[kFlagFallback] = 1u;
                if (a.status) *a.status = 1u;
                quit = true;
            }
        } else if (vflags[kFlagRetry] == 0u) {
            quit = true;
        }
        s_quit = quit ? 1u : 0u;
    }
    __syncthreads();
    if (s_quit) return;

    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(stc_smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kStcStages * kStcStageBytes);
    uint64_t *full = bars, *empty = bars + kStcStages, *acc_full = bars + 2 * kStcStages, *acc_empty = bars + 2 * kStcStages + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * kStcStages + 4);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_m = a.Qpad / kStcBM;
    const int units = tiles_m * a.S;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStcStages; ++s) mbar_init(&full[s], 1), mbar_init(&empty[s], 1);
        for (int b = 0; b < 2; ++b) mbar_init(&acc_full[b], 1), mbar_init(&acc_empty[b], 128);
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
            for (int u = blockIdx.x; u < units; u += gridDim.x) {
                const int m0 = (u % tiles_m) * kStcBM, seg = u / tiles_m;
                const int seg_begin = seg * a.seg_len;
                const int seg_end = seg_begin + a.seg_len < a.N ? seg_begin + a.seg_len : a.N;
                for (int n0 = seg_begin; n0 < seg_end; n0 += kStcBN) {
                    for (int kb = 0; kb < nkb; ++kb) {
                        mbar_wait_guarded(&empty[s], ph ^ 1u);
                        unsigned char *st = smem + s * kStcStageBytes;
                        mbar_expect_tx(&full[s], kStcStageBytes);
                        tma_load_2d(st, &maps.q, &full[s], kb * kStcBK, m0);
                        tma_load_2d(st + kStcABytes, &maps.db, &full[s], kb * kStcBK, n0);
                        if (++s == kStcStages) s = 0, ph ^= 1u;
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            uint32_t s = 0, ph = 0, it = 0;
            for (int u = blockIdx.x; u < units; u += gridDim.x) {
                const int seg = u / tiles_m;
                const int seg_begin = seg * a.seg_len;
                const int seg_end = seg_begin + a.seg_len < a.N ? seg_begin + a.seg_len : a.N;
                for (int n0 = seg_begin; n0 < seg_end; n0 += kStcBN, ++it) {
                    const uint32_t ab = it & 1u, aph = (it >> 1) & 1u;
                    mbar_wait_guarded(&acc_empty[ab], aph ^ 1u);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + ab * kStcBN;
                    for (int kb = 0; kb < nkb; ++kb) {
                        mbar_wait_guarded(&full[s], ph);
                        tc_fence_after();
                        const uint32_t st = smem_u32(smem + s * kStcStageBytes);
                        const uint64_t da = tc_smem_desc(st), db = tc_smem_desc(st + kStcABytes);
#pragma unroll
                        for (int k = 0; k < kStcBK / 32; ++k)         // 32 bytes (32 e4m3) per K-step: +2 in 16-byte units
                            tc_mma_f8(d_tmem, da + 2 * k, db + 2 * k, kStcIdesc, (kb | k) != 0);
                        tc_commit(&empty[s]);                          // stage reusable once these MMAs have read it
                        if (++s == kStcStages) s = 0, ph ^= 1u;
                    }
                    tc_commit(&acc_full[ab]);                          // accumulator complete
                }
            }
        }
    } else {
        const int quarter = warp & 3;                                  // TMEM lanes 32 * quarter .. + 31 belong to this warp
        const int tq = quarter * 32 + lane;                            // this thread's query row of the tile
        const float Bf = static_cast<float>(B);
        uint32_t it = 0;
        for (int u = blockIdx.x; u < units; u += gridDim.x) {
            const int m0 = (u % tiles_m) * kStcBM, seg = u / tiles_m;
            const int seg_begin = seg * a.seg_len;
            const int seg_end = seg_begin + a.seg_len < a.N ? seg_begin + a.seg_len : a.N;
            const int q = m0 + tq;
            const uint32_t bw = a.bound[q];
            const bool active = a.round == 0 ? !(bw & kBoundInactive) : (bw & kBoundRetry) != 0;
            // within the bound  <=>  d <= bound  <=>  dot >= B - 2 bound
            const float thr = !active ? 3.0e38f : (a.round == 0 ? Bf - 2.f * static_cast<float>(bw & 0xffffu) : -3.0e38f);
            for (int n0 = seg_begin; n0 < seg_end; n0 += kStcBN, ++it) {
                const uint32_t ab = it & 1u, aph = (it >> 1) & 1u;
                const int rows = kStcBN < seg_end - n0 ? kStcBN : seg_end - n0;
                uint32_t *out = a.mask + static_cast<size_t>(n0 >> 5) * a.Qpad + q;      // a warp stores 128 contiguous bytes per group
                mbar_wait_guarded(&acc_full[ab], aph);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ab * kStcBN + (static_cast<uint32_t>(quarter * 32) << 16);
                uint32_t ra[32], rb[32];
                tc_ld32(taddr, ra);
                tc_ld_wait();
                auto consume = [&](const uint32_t (&r)[32], int c) {
                    uint32_t h[4] = {0u, 0u, 0u, 0u};                  // four independent chains
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (__uint_as_float(r[j]) >= thr) h[j & 3] |= 1u << j;
                    uint32_t hit = (h[0] | h[1]) | (h[2] | h[3]);
                    const int left = rows - c * 32;                    // columns of this chunk that are rows of the segment
                    if (left < 32) hit &= left > 0 ? (0xffffffffu >> (32 - left)) : 0u;
                    out[static_cast<size_t>(c) * a.Qpad] = hit;
                };
#pragma unroll 1
                for (int c = 0; c < kStcBN / 32; c += 2) {
                    tc_ld32(taddr + (c + 1) * 32, rb);
                    consume(ra, c);
                    tc_ld_wait();
                    if (c + 2 < kStcBN / 32) tc_ld32(taddr + (c + 2) * 32, ra);
                    consume(rb, c + 1);
                    tc_ld_wait();
                }
                tc_fence_before();
                mbar_arrive(&acc_empty[ab]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

static bool make_map_u8(CUtensorMap *map, const void *base, long long rows, int Bp, int box_rows) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return false;
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(Bp), static_cast<cuuint64_t>(rows)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(Bp)};
    const cuuint32_t box[2] = {static_cast<cuuint32_t>(kStcBK), static_cast<cuuint32_t>(box_rows)};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// ------------------------------------------------------------------------------------------------ (B) rank
// One CTA per query, kRankWarps warps.  Pass 1: every warp histograms a contiguous (index-order) part of the query's
// candidates by distance; a CTA-wide scan gives each (warp, distance) its rank / ordinal base and the cut-off distance
// d*; pass 2: every warp walks its part again with private running counters.
//
// STAGED form (a.stage, the usual case): the query's whole candidate set is first copied into shared memory, in index
// order, in three rounds of independent loads — the S list heads, the chunk id of every 128-entry block, the entries
// (coalesced, 4 in flight per thread) — and both passes run on the flat shared array; warp w owns entries
// [w * total / 8, (w + 1) * total / 8).  What the first form waited for was the dependent chain list head -> chunk ->
// entries, once per list and pass with one warp's worth of loads in flight: 41 us per CTA for 7.7k candidates on c3
// (0.28 ms for the kernel), almost all of it memory latency.
// CHUNKED form (a query with more than kStageCap candidates — a lifted bound in round 1 — or more than kStageMaxSeg
// segments): warp w owns a contiguous range of the segments and streams its lists from the pool, heads of 32 segments
// per coalesced load and the next block's entries requested before the current block is visited.
constexpr int kRankWarps = 8;
constexpr int kStageMaxSeg = 256;                         // lists per query the staged form handles (one thread each)
constexpr int kStageCap = 12288;                          // most entries of shared memory per CTA (48 KB: three CTAs per SM)
// entries the staged form gets for top-k k: 1.8 k + 512 (the sampled bound lists ~1.3-1.5 k candidates per query, a longer
// list takes the chunked form) in steps of 512 — c3 (k = 5000): 9728 entries = 55 KB per CTA with the counters, FOUR CTAs per
// SM instead of three
inline int rank_stage_cap(uint32_t k) {
    const long long cap = (static_cast<long long>(k) * 9 / 5 + 512 + 511) / 512 * 512;
    return static_cast<int>(cap < 1024 ? 1024 : (cap > kStageCap ? kStageCap : cap));
}
__host__ __device__ inline int rank_stage_max_blk(int cap) { return cap / 128 + kStageMaxSeg; }

// shared memory (uint32 words): per warp cnt[binsP] + peer[binsP]; the relevance bitmap of the k ranks; the staged form's arrays
__host__ __device__ inline size_t rank_counter_words(int bins, uint32_t k) {
    return static_cast<size_t>(kRankWarps) * 2 * ((bins + 31) & ~31) + ((static_cast<size_t>(k) + 31) >> 5);
}
inline size_t rank_smem_bytes(int bins, uint32_t k, int stage_cap) {
    size_t words = rank_counter_words(bins, k);
    if (stage_cap) words += stage_cap + 2 * rank_stage_max_blk(stage_cap) + 2 * kStageMaxSeg + 4;
    return words * sizeof(uint32_t);
}

template <bool EMIT>
__global__ void __launch_bounds__(kRankWarps * 32) hamming_select_rank_kernel(const __grid_constant__ SelArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint32_t s_scan[kRankWarps][2];
    __shared__ uint32_t s_dstar, s_quit, s_total, s_nblk;
    __shared__ unsigned long long s_sum[kRankWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, t = threadIdx.x;
    const int q = blockIdx.x;
    volatile uint32_t *vflags = a.flags;
    if (t == 0) {
        // one thread decides for the CTA (the fallback flag may be raised concurrently)
        const uint32_t bw = a.bound[q];
        s_quit = vflags[kFlagFallback] != 0u || (a.round != 0 && (vflags[kFlagRetry] == 0u || !(bw & kBoundRetry)));
        s_dstar = 0xffffffffu;
    }
    const int binsP = (a.bins + 31) & ~31;                      // <= 256 = blockDim
    uint32_t *cnt = reinterpret_cast<uint32_t *>(smem_raw) + static_cast<size_t>(warp) * binsP;           // this warp's counters
    // lanes of the current 32 entries per distance (pass 2): __match_any_sync costs ~84 issue cycles per warp on sm_100
    // (tools/ubench_match.cu), a shared atomicOr per lane + one load gives the same mask for a fraction of that
    uint32_t *peer = reinterpret_cast<uint32_t *>(smem_raw) + static_cast<size_t>(kRankWarps) * binsP + static_cast<size_t>(warp) * binsP;
    // bit r of s_rel: the row of rank r + 1 is relevant.  Pass 2 only places the rows; hit ordinals and AP terms come from
    // the bitmap afterwards, densely (one division per relevant rank, no per-entry relevant counters)
    uint32_t *s_rel = reinterpret_cast<uint32_t *>(smem_raw) + static_cast<size_t>(kRankWarps) * 2 * binsP;
    const uint32_t relw = (a.k + 31u) >> 5;
    for (int d = lane; d < binsP; d += 32) cnt[d] = 0u, peer[d] = 0u;
    for (uint32_t i = t; i < relw; i += kRankWarps * 32) s_rel[i] = 0u;
    __syncthreads();
    if (s_quit) return;
    const U32x2 *heads = a.head + static_cast<size_t>(q) * a.S;
    const uint32_t *table = a.table + static_cast<size_t>(q) * a.S * a.maxc;
    const int CH = 1 << a.ch_shift;

    // ---- staging (see above).  s_ent: the entries; s_bid / s_bmeta: per 128-entry block its pool chunk and
    // (destination | length - 1 << 14 | in-chunk offset / 128 << 21 | segment << 24); s_off: entry offset of each list.
    uint32_t *s_ent = reinterpret_cast<uint32_t *>(smem_raw) + rank_counter_words(a.bins, a.k);
    uint32_t *s_bid = s_ent + a.stage_cap, *s_bmeta = s_bid + rank_stage_max_blk(a.stage_cap);
    uint32_t *s_off = s_bmeta + rank_stage_max_blk(a.stage_cap);   // [S + 1]
    bool staged = a.stage != 0;
    uint32_t total_e = 0;
    if (staged) {
        uint32_t n = 0, first = 0;
        if (t < a.S) {
            const U32x2 h = heads[t];
            n = h.x, first = h.y;
        }
        const uint32_t nb = (n + 127u) >> 7;
        uint32_t ie = n, ib = nb;                               // inclusive scans over the lists: entries, blocks
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t te = __shfl_up_sync(0xffffffffu, ie, o), tb = __shfl_up_sync(0xffffffffu, ib, o);
            if (lane >= o) ie += te, ib += tb;
        }
        if (lane == 31) s_scan[warp][0] = ie, s_scan[warp][1] = ib;
        __syncthreads();
        uint32_t oe = 0, ob = 0, te = 0, tb = 0;
#pragma unroll
        for (int w = 0; w < kRankWarps; ++w) {
            if (w < warp) oe += s_scan[w][0], ob += s_scan[w][1];
            te += s_scan[w][0], tb += s_scan[w][1];
        }
        __syncthreads();                                        // s_scan is reused by the distance scan below
        staged = te <= static_cast<uint32_t>(a.stage_cap);      // (then tb <= the block arrays' size: at most one partial block per list)
        total_e = te;
        if (staged) {
            const uint32_t e0 = oe + ie - n, b0 = ob + ib - nb;  // exclusive
            if (t < a.S) s_off[t] = e0;
            if (t == 0) s_off[a.S] = te, s_total = te, s_nblk = tb;
            for (uint32_t bb = 0; bb < nb; ++bb) {
                const uint32_t i0 = bb << 7, c = i0 >> a.ch_shift;
                const uint32_t id = c == 0u ? first : table[static_cast<size_t>(t) * a.maxc + c];
                const uint32_t len = n - i0 < 128u ? n - i0 : 128u;
                s_bid[b0 + bb] = id;
                s_bmeta[b0 + bb] = (e0 + i0) | ((len - 1u) << 14) | (((i0 & static_cast<uint32_t>(CH - 1)) >> 7) << 21) | (static_cast<uint32_t>(t) << 24);
            }
            __syncthreads();
            // a thread copies 4 consecutive entries per step (one 128-bit load: a block starts on a 512-byte boundary of
            // the pool; what lies past a list's end inside its chunk is readable and dropped), 4 steps in flight
            const uint32_t slots = s_nblk << 5;
            for (uint32_t x0 = t; x0 < slots; x0 += 4u * kRankWarps * 32) {
                U32x4 v[4];
                uint32_t dst[4], cntv[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t x = x0 + static_cast<uint32_t>(j) * kRankWarps * 32;
                    cntv[j] = 0u;
                    if (x < slots) {
                        const uint32_t blk = x >> 5, i = (x & 31u) << 2;
                        const uint32_t meta = s_bmeta[blk], len = ((meta >> 14) & 127u) + 1u;
                        if (i < len) {
                            cntv[j] = len - i < 4u ? len - i : 4u;
                            dst[j] = (meta & 0x3fffu) + i;
                            v[j] = *reinterpret_cast<const U32x4 *>(a.pool + (static_cast<size_t>(s_bid[blk]) << a.ch_shift) + (((meta >> 21) & 7u) << 7) + i);
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (cntv[j] > 0u) s_ent[dst[j]] = v[j].x;
                    if (cntv[j] > 1u) s_ent[dst[j] + 1] = v[j].y;
                    if (cntv[j] > 2u) s_ent[dst[j] + 2] = v[j].z;
                    if (cntv[j] > 3u) s_ent[dst[j] + 3] = v[j].w;
                }
            }
            __syncthreads();
        }
    }
    const uint32_t e_lo = static_cast<uint32_t>(static_cast<unsigned long long>(warp) * total_e / kRankWarps);
    const uint32_t e_hi = static_cast<uint32_t>(static_cast<unsigned long long>(warp + 1) * total_e / kRankWarps);
    // flat walk of this warp's staged entries, 32 per visit; the segment of an entry (EMIT only) by bisection of s_off
    auto walk_flat = [&](auto visit) {
        for (uint32_t e0 = e_lo; e0 < e_hi; e0 += 32u) {
            const uint32_t e = e0 + lane;
            visit(e < e_hi ? s_ent[e] : 0xffffffffu, [&]() {
                int lo = 0, hi = a.S - 1;                       // last list whose offset is <= e
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if (s_off[mid] <= e)
                        lo = mid;
                    else
                        hi = mid - 1;
                }
                return lo;
            });
        }
    };

    const int seg_lo = static_cast<int>(static_cast<long long>(warp) * a.S / kRankWarps);
    const int seg_hi = static_cast<int>(static_cast<long long>(warp + 1) * a.S / kRankWarps);
    // Chunked walk: this warp's lists in index order as a stream of blocks of <= 128 consecutive entries (a chunk is a
    // multiple of 128 entries, so a block never straddles chunks); `visit` gets 32 entries per call (absent ones =
    // 0xffffffff).
    auto walk = [&](auto visit) {
        int seg = seg_lo - 1, batch0 = seg_lo;
        uint32_t hn = 0, hid = 0;                 // this lane's head of segment batch0 + lane
        uint32_t n = 0, id0 = 0, i0 = 0;          // current list: length, first chunk, next entry
        auto refill = [&]() {
            const int sg = batch0 + lane;
            const U32x2 h = sg < seg_hi ? heads[sg] : U32x2{0u, 0u};
            hn = h.x, hid = h.y;
        };
        if (seg_lo < seg_hi) refill();
        // next block of the stream: pointer to its first entry, its length (0: the stream has ended) and its segment
        auto next_block = [&](const uint32_t *&ptr, uint32_t &m, int &bseg) {
            while (i0 >= n) {
                ++seg;
                if (seg >= seg_hi) {
                    m = 0;
                    return;
                }
                if (seg - batch0 >= 32) {
                    batch0 += 32;
                    refill();
                }
                n = __shfl_sync(0xffffffffu, hn, seg - batch0);
                id0 = __shfl_sync(0xffffffffu, hid, seg - batch0);
                i0 = 0;
            }
            const uint32_t c = i0 >> a.ch_shift;
            const uint32_t id = c == 0u ? id0 : table[static_cast<size_t>(seg) * a.maxc + c];
            ptr = a.pool + (static_cast<size_t>(id) << a.ch_shift) + (i0 & static_cast<uint32_t>(CH - 1));
            m = n - i0 < 128u ? n - i0 : 128u;
            bseg = seg;
            i0 += 128u;
        };
        auto load = [&](const uint32_t *ptr, uint32_t m, uint32_t (&e)[4]) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t i = 32u * j + lane;
                e[j] = i < m ? ptr[i] : 0xffffffffu;
            }
        };
        const uint32_t *ptr = nullptr;
        uint32_t m = 0, e[4];
        int bseg = 0;
        next_block(ptr, m, bseg);
        if (m) load(ptr, m, e);
        while (m) {
            uint32_t cur[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) cur[j] = e[j];
            const uint32_t cm = m;
            const int cseg = bseg;
            next_block(ptr, m, bseg);
            if (m) load(ptr, m, e);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (32u * j < cm) visit(cur[j], [&]() { return cseg; });
        }
    };

    // pass 1: histogram of this warp's entries by distance
    auto count = [&](uint32_t e, auto) {
        if (e != 0xffffffffu) atomicAdd(cnt + ((e >> 16) & 0xffu), 1u);      // same-address lanes are serialised by the hardware: a few cycles each
    };
    if (staged)
        walk_flat(count);
    else
        walk(count);
    __syncwarp();
    __syncthreads();

    // CTA scan: thread d (< binsP <= 256) owns distance d.  Totals over the warps, exclusive scan over the distances,
    // then every warp's counters become its rank bases.
    uint32_t *all = reinterpret_cast<uint32_t *>(smem_raw);
    uint32_t tot_a = 0;
    if (t < binsP) {
#pragma unroll
        for (int w = 0; w < kRankWarps; ++w) tot_a += all[w * binsP + t];
    }
    uint32_t ia = tot_a;                                        // inclusive scan within the warp ...
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t ta = __shfl_up_sync(0xffffffffu, ia, o);
        if (lane >= o) ia += ta;
    }
    if (lane == 31) s_scan[warp][0] = ia;
    __syncthreads();
    uint32_t off_a = 0, total = 0;                              // ... plus the warps before it
#pragma unroll
    for (int w = 0; w < kRankWarps; ++w) {
        if (w < warp) off_a += s_scan[w][0];
        total += s_scan[w][0];
    }
    if (total < a.k) {
        // the bound missed the k-th neighbour (only possible in round 0: a lifted bound lists every row, and k <= rows)
        if (t == 0) {
            a.bound[q] |= kBoundRetry;
            atomicAdd(a.flags + kFlagRetry, 1u);
            if (a.status) *a.status = 1u;
        }
        return;
    }
    ia += off_a;
    if (t < binsP) {
        if (ia >= a.k && ia - tot_a < a.k) s_dstar = static_cast<uint32_t>(t);      // the one distance where the count crosses k
        uint32_t run_a = ia - tot_a;                            // exclusive: rows at smaller distances
#pragma unroll
        for (int w = 0; w < kRankWarps; ++w) {
            const uint32_t ca = all[w * binsP + t];
            all[w * binsP + t] = run_a;
            run_a += ca;
        }
    }
    __syncthreads();
    const uint32_t dstar = s_dstar;

    // pass 2: ranks in index order
    const uint32_t lt = (1u << lane) - 1u;
    auto rank_visit = [&](uint32_t e, auto seg_of) {
        const uint32_t d = (e >> 16) & 0xffu;
        const bool take = e != 0xffffffffu && d <= dstar;
        if (!__any_sync(0xffffffffu, take)) return;
        if (take) atomicOr(peer + d, 1u << lane);
        __syncwarp();
        const uint32_t peers = take ? peer[d] : 0u;           // the taken lanes with this lane's distance
        const uint32_t rank0 = take ? cnt[d] + __popc(peers & lt) : 0xffffffffu;      // rank - 1
        __syncwarp();
        if (take && (peers >> lane) == 1u) {                  // last lane of its distance group
            cnt[d] += __popc(peers);
            peer[d] = 0u;
        }
        __syncwarp();
        if (rank0 < a.k) {
            if (e >> 24) atomicOr(s_rel + (rank0 >> 5), 1u << (rank0 & 31u));
            if (EMIT) {
                const size_t o = static_cast<size_t>(q) * a.k + rank0;
                if (a.rank_idx)
                    a.rank_idx[o] = static_cast<uint32_t>(a.index_base + static_cast<long long>(seg_of()) * a.seg_len + (e & 0xffffu));
                if (a.rank_dist) a.rank_dist[o] = static_cast<uint16_t>(d);
            }
        }
    };
    if (staged)
        walk_flat(rank_visit);
    else
        walk(rank_visit);
    __syncthreads();

    // AP from the bitmap: thread t owns a contiguous run of its words; hit ordinal = relevant ranks before the run
    // (CTA scan of the runs' popcounts) + position within it; the terms are exact 2^-40 fixed-point integers, so the
    // order of the sums does not matter
    const uint32_t wpt = (relw + kRankWarps * 32 - 1) / (kRankWarps * 32);
    const uint32_t w_lo = t * wpt < relw ? t * wpt : relw, w_hi = (t + 1) * wpt < relw ? (t + 1) * wpt : relw;
    uint32_t mine = 0;
    for (uint32_t w = w_lo; w < w_hi; ++w) mine += __popc(s_rel[w]);
    uint32_t ih = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t th = __shfl_up_sync(0xffffffffu, ih, o);
        if (lane >= o) ih += th;
    }
    if (lane == 31) s_scan[warp][1] = ih;
    __syncthreads();
    uint32_t ordinal = ih - mine, hits_all = 0;
#pragma unroll
    for (int w = 0; w < kRankWarps; ++w) {
        if (w < warp) ordinal += s_scan[w][1];
        hits_all += s_scan[w][1];
    }
    unsigned long long sum = 0;
    for (uint32_t w = w_lo; w < w_hi; ++w) {
        uint32_t bits = s_rel[w];
        while (bits) {
            const uint32_t b = static_cast<uint32_t>(__ffs(static_cast<int>(bits))) - 1u;
            bits &= bits - 1u;
            sum += ap_term(++ordinal, 32u * w + b + 1u);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) s_sum[warp] = sum;
    __syncthreads();
    if (t == 0) {
        unsigned long long ts = 0;
        for (int w = 0; w < kRankWarps; ++w) ts += s_sum[w];
        if (a.ap) a.ap[q] = hits_all ? (static_cast<double>(ts) / 1099511627776.0) / static_cast<double>(hits_all) : 0.0;
        if (a.tsum) a.tsum[q] = hits_all;
    }
}

// ------------------------------------------------------------------------------------------------ dispatch
using sel_fn = void (*)(const SelArgs);
template <int CW>
static sel_fn pick_sel2(int lw, bool eq) {
    if (eq) return hamming_select_kernel<CW, 1, true>;
    switch (lw) {
        case 1: return hamming_select_kernel<CW, 1, false>;
        case 2: return hamming_select_kernel<CW, 2, false>;
        case 4: return hamming_select_kernel<CW, 4, false>;
    }
    return nullptr;
}
static sel_fn pick_sel(int cw, int lw, bool eq) {
    switch (cw) {
        case 1: return pick_sel2<1>(lw, eq);
        case 2: return pick_sel2<2>(lw, eq);
        case 4: return pick_sel2<4>(lw, eq);
    }
    return nullptr;
}
template <int CW>
static sel_fn pick_app2(int lw, bool eq) {
    if (eq) return hamming_select_kernel<CW, 1, true, true>;
    switch (lw) {
        case 1: return hamming_select_kernel<CW, 1, false, true>;
        case 2: return hamming_select_kernel<CW, 2, false, true>;
        case 4: return hamming_select_kernel<CW, 4, false, true>;
    }
    return nullptr;
}
static sel_fn pick_app(int cw, int lw, bool eq) {        // the MASKED (append-only) form
    switch (cw) {
        case 1: return pick_app2<1>(lw, eq);
        case 2: return pick_app2<2>(lw, eq);
        case 4: return pick_app2<4>(lw, eq);
    }
    return nullptr;
}

using stc_fn = void (*)(const StcMaps, const SelArgs, int, int);

// The select pipeline in three phases, so that a caller whose database arrives in pieces (b200_maphashing_host: row
// chunks over PCIe) can score the segments of a chunk while the next chunk is still in flight:
//   select_begin     flags + sample plane zeroed, sample histogram, bound.  sample_codes: the packed sample rows gathered
//                    in a compact buffer (row r = database row 32 stride (r / 32) + r % 32), or null = read in place
//   select_segments  round-0 select kernel on segments [seg0, seg1)
//   select_finish    rank; status == null: the retry round (select over all segments + rank) as well
// hamming_select_run = the three in a row.
static int sel_args(const b200_map_plan *p, const uint64_t *qc, const uint64_t *ql, const uint64_t *dc, const uint64_t *dl, void *ws,
                    double *ap, uint32_t *tsum, uint32_t *rank_idx, uint16_t *rank_dist, uint32_t *status, SelArgs *out) {
    unsigned char *w = static_cast<unsigned char *>(ws);
    SelArgs a;
    a.q_codes = qc, a.q_labels = ql, a.db_codes = dc, a.db_labels = dl;
    a.bound = reinterpret_cast<uint32_t *>(w + p->off_sel_bound);
    a.head = reinterpret_cast<U32x2 *>(w + p->off_sel_count);
    a.table = reinterpret_cast<uint32_t *>(w + p->off_sel_table);
    a.pool = reinterpret_cast<uint32_t *>(w + p->off_sel_pool);
    a.flags = reinterpret_cast<uint32_t *>(w + p->off_sel_flags);
    a.status = status;
    a.ap = ap, a.tsum = tsum, a.rank_idx = rank_idx, a.rank_dist = rank_dist;
    a.est_cap = static_cast<unsigned long long>(p->Q) * (4ull * static_cast<unsigned long long>(p->k) + 1024ull);   // = the pool's budget (hamming_plan.h)
    a.index_base = 0;
    a.Q = p->Q, a.N = static_cast<int>(p->N), a.S = p->sel_S, a.seg_len = p->sel_seg_len, a.tile = p->tile, a.Qpad = p->Qpad;
    a.ch_shift = 0;
    while ((1 << a.ch_shift) < p->sel_chunk) ++a.ch_shift;
    a.maxc = p->sel_maxc, a.bins = p->bins;
    a.pool_chunks = static_cast<uint32_t>(p->sel_pool_chunks), a.k = static_cast<uint32_t>(p->k);
    a.stage = (p->sel_S <= kStageMaxSeg && (p->sel_chunk >> 7) <= 8) ? 1 : 0;
    a.stage_cap = a.stage ? rank_stage_cap(a.k) : 0;
    a.round = 0, a.seg0 = 0, a.mask = nullptr;
    a.nsub = a.pool_chunks >= 64u * kSubPools ? kSubPools : 1u;
    a.sub_chunks = a.pool_chunks / a.nsub;
    *out = a;
    return B200_OK;
}

int select_begin(const b200_map_plan *p, const uint64_t *qc, const uint64_t *dc, const uint64_t *sample_codes, void *ws, cudaStream_t st) {
    unsigned char *w = static_cast<unsigned char *>(ws);
    const int cw = b200_code_words(p->B);
    uint32_t *flags = reinterpret_cast<uint32_t *>(w + p->off_sel_flags);
    // (P) sample -> bound
    uint32_t *smp_hist = reinterpret_cast<uint32_t *>(w + p->off_smp_hist);
    const size_t hist_bytes = static_cast<size_t>(p->bins) * p->Qpad * sizeof(uint32_t);
    if (p->off_smp_hist == p->off_sel_flags + 64 * sizeof(uint32_t)) {
        B200_CUDA_TRY(cudaMemsetAsync(flags, 0, 64 * sizeof(uint32_t) + hist_bytes, st));      // one node: flags + sample plane
    } else {
        B200_CUDA_TRY(cudaMemsetAsync(flags, 0, 64 * sizeof(uint32_t), st));
        B200_CUDA_TRY(cudaMemsetAsync(smp_hist, 0, hist_bytes, st));
    }
    {
        using smp_fn = void (*)(const uint64_t *, const uint64_t *, uint32_t *, long long, int, int, int, int, int);
        smp_fn sf = cw == 1 ? select_sample_kernel<1> : (cw == 2 ? select_sample_kernel<2> : (cw == 4 ? select_sample_kernel<4> : nullptr));
        if (!sf) return B200_ERR_UNSUPPORTED;
        const size_t ssmem = static_cast<size_t>(kSampleTile) * cw * 8 + static_cast<size_t>((p->bins + 1) / 2) * p->sel_T * sizeof(uint32_t);
        if (ssmem > 48 * 1024)
            B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(sf), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(ssmem)));
        sf<<<dim3(p->Qpad / p->sel_T, p->smp_S), dim3(p->sel_T, 512 / p->sel_T), ssmem, st>>>(
            qc, sample_codes ? sample_codes : dc, smp_hist, p->smp_rows, sample_codes ? 1 : p->sel_stride, p->smp_seg_len, p->Q, p->Qpad, p->bins);
        B200_LAUNCH_CHECK("select_sample_kernel");
    }
    stage_mark("sample_hist", st);
    {
        const double frac = static_cast<double>(p->smp_rows) / static_cast<double>(p->N);
        const double kf = static_cast<double>(p->k) * frac;
        const uint32_t target = static_cast<uint32_t>(kf + 5.0 * sqrt(kf) + 2.0);
        select_bound_kernel<<<p->Qpad / 32, dim3(32, 32), 0, st>>>(smp_hist, p->bins, p->Qpad, p->Q, target, static_cast<float>(1.0 / frac),
                                                                   reinterpret_cast<uint32_t *>(w + p->off_sel_bound), flags);
        B200_LAUNCH_CHECK("select_bound_kernel");
    }
    stage_mark("bound", st);
    return B200_OK;
}

int select_segments(const b200_map_plan *p, const uint64_t *qc, const uint64_t *ql, const uint64_t *dc, const uint64_t *dl, void *ws,
                    uint32_t *status, int seg0, int seg1, cudaStream_t st) {
    if (seg1 <= seg0) return B200_OK;
    SelArgs a;
    if (int rc = sel_args(p, qc, ql, dc, dl, ws, nullptr, nullptr, nullptr, nullptr, status, &a)) return rc;
    const int cw = b200_code_words(p->B);
    sel_fn fn = pick_sel(cw, p->LW, p->label_mode == B200_LABELS_EQUAL);
    if (!fn) return B200_ERR_UNSUPPORTED;
    const size_t smem = static_cast<size_t>(p->tile) * (cw + p->LW) * 8 + static_cast<size_t>(32) * p->sel_T;      // tile + parked distances
    a.seg0 = seg0;
    fn<<<dim3(p->Qpad / p->sel_T, seg1 - seg0), p->sel_T, smem, st>>>(a);
    B200_LAUNCH_CHECK("hamming_select_kernel");
    return B200_OK;
}

// ap / tsum (mAP) or rank_idx / rank_dist (top-k list) — whichever are given.  Leaves flags[kFlagFallback] for the caller's gate.
// status != null: round 0 only — the caller looks at *status afterwards and redoes the evaluation with the complete
// sequence (status == null) when it is set.  round0_selected: select_segments has already covered every segment.
int select_finish(const b200_map_plan *p, const uint64_t *qc, const uint64_t *ql, const uint64_t *dc, const uint64_t *dl, void *ws,
                  double *ap, uint32_t *tsum, uint32_t *rank_idx, uint16_t *rank_dist, uint32_t *status, bool round0_selected,
                  cudaStream_t st) {
    unsigned char *w = static_cast<unsigned char *>(ws);
    const int cw = b200_code_words(p->B);
    SelArgs a;
    if (int rc = sel_args(p, qc, ql, dc, dl, ws, ap, tsum, rank_idx, rank_dist, status, &a)) return rc;
    sel_fn fn = pick_sel(cw, p->LW, p->label_mode == B200_LABELS_EQUAL);
    if (!fn) return B200_ERR_UNSUPPORTED;
    // tensor-core form of the select pass (A'): filter kernel -> hit masks -> append kernel, where the plan carved its
    // workspace and the caller has not run round 0 already; the SIMT kernel when the driver cannot encode tensor maps
    const int Bp = (p->B + kStcBK - 1) / kStcBK * kStcBK;
    stc_fn tf = hamming_select_tc_kernel;
    sel_fn af = pick_app(cw, p->LW, p->label_mode == B200_LABELS_EQUAL);
    bool use_tc = !round0_selected && plan_select_tc(*p) && encode_tiled_fn() != nullptr;
    StcMaps maps;
    if (use_tc) {
        unsigned char *db8 = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(w + p->off_smp_codes) + 1023) & ~static_cast<uintptr_t>(1023));
        unsigned char *q8 = db8 + round_up<size_t>(static_cast<size_t>(p->N) * Bp, 1024);
        a.mask = reinterpret_cast<uint32_t *>(q8 + round_up<size_t>(static_cast<size_t>(p->Qpad) * Bp, 1024));
        if (!make_map_u8(&maps.q, q8, p->Q, Bp, kStcBM) || !make_map_u8(&maps.db, db8, p->N, Bp, kStcBN)) {
            use_tc = false;
        } else {
            const int sms = sm_count();
            select_expand_fp8_kernel<<<sms * 8, 256, 0, st>>>(dc, p->N, cw, p->B, Bp, reinterpret_cast<uint4 *>(db8));
            B200_LAUNCH_CHECK("select_expand_fp8_kernel");
            select_expand_fp8_kernel<<<(p->Q * (Bp / 16) + 255) / 256, 256, 0, st>>>(qc, p->Q, cw, p->B, Bp, reinterpret_cast<uint4 *>(q8));
            B200_LAUNCH_CHECK("select_expand_fp8_kernel");
            B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(tf), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               static_cast<int>(kStcSmemBytes)));
            stage_mark("expand", st);
        }
    }
    const size_t smem = static_cast<size_t>(p->tile) * (cw + p->LW) * 8 + static_cast<size_t>(32) * p->sel_T;      // tile + parked distances
    const bool emit = rank_idx != nullptr || rank_dist != nullptr;
    sel_fn rf = emit ? hamming_select_rank_kernel<true> : hamming_select_rank_kernel<false>;
    const size_t rsmem = rank_smem_bytes(p->bins, a.k, a.stage_cap);
    if (rsmem > 48 * 1024)
        B200_CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(rf), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(rsmem)));
    for (int round = 0; round < (status ? 1 : 2); ++round) {
        a.round = round;
        if (round == 0 && round0_selected) {
            // (the caller's select_segments launches did this round's select pass)
        } else if (use_tc) {
            const int units = (p->Qpad / kStcBM) * p->sel_S, sms = sm_count();
            tf<<<units < sms ? units : sms, kStcThreads, kStcSmemBytes, st>>>(maps, a, p->B, Bp / kStcBK);
            B200_LAUNCH_CHECK("hamming_select_tc_kernel");
            stage_mark(round ? "filter_round1" : "filter", st);
            af<<<dim3(p->Qpad / p->sel_T, p->sel_S), p->sel_T, smem, st>>>(a);
            B200_LAUNCH_CHECK("hamming_select_kernel (append)");
        } else {
            fn<<<dim3(p->Qpad / p->sel_T, p->sel_S), p->sel_T, smem, st>>>(a);
            B200_LAUNCH_CHECK("hamming_select_kernel");
        }
        stage_mark(round ? "select_round1" : "select", st);
        rf<<<p->Q, kRankWarps * 32, rsmem, st>>>(a);
        B200_LAUNCH_CHECK("hamming_select_rank_kernel");
        stage_mark(round ? "rank_round1" : "rank", st);
    }
    return B200_OK;
}

int hamming_select_run(const b200_map_plan *p, const uint64_t *qc, const uint64_t *ql, const uint64_t *dc, const uint64_t *dl,
                       void *ws, double *ap, uint32_t *tsum, uint32_t *rank_idx, uint16_t *rank_dist, uint32_t *status,
                       cudaStream_t st) {
    if (int rc = select_begin(p, qc, dc, nullptr, ws, st)) return rc;
    return select_finish(p, qc, ql, dc, dl, ws, ap, tsum, rank_idx, rank_dist, status, false, st);
}

}  // namespace b200

extern "C" int b200_map_select_status(const b200_map_plan *plan, const void *workspace, uint32_t *out4, b200_stream_t stream) {
    using namespace b200;
    if (!plan || !workspace || !out4 || !plan->select) return B200_ERR_INVALID_ARG;
    uint32_t f[64];                                             // the whole flags block, sub-pool cursors included
    B200_CUDA_TRY(cudaMemcpyAsync(f, static_cast<const unsigned char *>(workspace) + plan->off_sel_flags, sizeof(f),
                                  cudaMemcpyDeviceToHost, as_stream(stream)));
    B200_CUDA_TRY(cudaStreamSynchronize(as_stream(stream)));
    const unsigned long long est = static_cast<unsigned long long>(f[kFlagEst]) | (static_cast<unsigned long long>(f[kFlagEst + 1]) << 32);
    out4[0] = f[kFlagCursor], out4[1] = f[kFlagFallback], out4[2] = f[kFlagRetry];
    for (int i = 0; i < kSubPools; ++i) out4[0] += f[kFlagSubCursor + i];
    out4[3] = static_cast<uint32_t>(est / static_cast<unsigned long long>(plan->Q > 0 ? plan->Q : 1));
    return B200_OK;
}
