// Host-side launch planner of the Hamming mAP stages (shared by the CUDA launcher and the CPU simulator in tests).
#pragma once
#include <cstddef>
#include <cstdlib>

#include "b200ret.h"

namespace b200 {

template <typename T>
inline T plan_ceil_div(T a, T b) { return (a + b - 1) / b; }
template <typename T>
inline T plan_round_up(T a, T b) { return plan_ceil_div(a, b) * b; }

// largest stash (1 byte + 1 bit per (row, query) pair) a plan carves, in MB
constexpr size_t kMapStashMaxMB = 24576;

// Tensor-core form of the select pass (hamming_select.cu (A'): tcgen05 filter -> hit masks -> SIMT append; c3 select
// 0.61 -> 0.53 ms, c5 5.8 -> 3.7 ms) for a select plan: full 128-query groups, e4m3 copies of the codes (rows padded to
// 128-byte K blocks) and the hit masks (4 B per (32-row group, query)) bounded in the workspace.  Needs only Q, N, B and
// the query groups, so map_plan_init decides it before the select geometry, which it then fits to the form: 128-query
// select groups and segments of whole 256-row tiles.  The plan carves the e4m3 + mask block and the launcher runs the form
// exactly when this holds.
inline bool plan_select_tc(const b200_map_plan &p) {
    const size_t bp = static_cast<size_t>((p.B + 127) / 128) * 128;
    const size_t groups = static_cast<size_t>(plan_ceil_div<long long>(p.N, 256)) * 8;
    return p.T == 128 && p.Qpad % 128 == 0 && groups * p.Qpad * sizeof(uint32_t) <= (4ull << 30) &&
           static_cast<size_t>(p.N) * bp <= (8ull << 30);
}

// waves: how many machine-filling sets of segments to cut the database into (1: one CTA per SM slot; the host-buffer
// pipeline asks for one wave per H2D chunk so that stage A of a chunk fills the GPU while the next chunk is in flight)
// allow_select: the caller can run the select pipeline (device library, single shard); the simulator and sub-plans pass false
inline int map_plan_init(b200_map_plan *plan, int Q, long long N, long long N_total, int B, int LW, int label_mode,
                         long long k, int num_sms, int waves = 1, bool allow_select = false) {

    if (!plan || Q < 1 || N < 0 || N_total < N || B < 1 || k < 1) return B200_ERR_INVALID_ARG;
    if (label_mode != B200_LABELS_OVERLAP && label_mode != B200_LABELS_EQUAL) return B200_ERR_INVALID_ARG;
    if (B > B200_MAX_CODE_BITS || N >= (1ll << 31) - 65536 || N_total >= (1ll << 32) - 2) return B200_ERR_UNSUPPORTED;
    if (!(LW == 1 || LW == 2 || LW == 4) || (label_mode == B200_LABELS_EQUAL && LW != 1)) return B200_ERR_UNSUPPORTED;
    b200_map_plan p = {};
    p.Q = Q, p.N = N, p.N_total = N_total, p.B = B, p.LW = LW, p.label_mode = label_mode;
    p.k = k > N_total ? (N_total > 0 ? N_total : 1) : k;
    p.bins = B + 1;
    p.wide = p.k > 65534 ? 1 : 0;
    p.tile = 256;
    const int cw = b200_code_words(B);
    const size_t ctr_global = p.wide ? 8 : 4;                       // histogram entry in the workspace
    const size_t ctr = (p.wide && p.k < N_total) ? 8 : 4;           // shared-memory counter of the widest stage
    const size_t tile_bytes = static_cast<size_t>(p.tile) * (cw + LW) * 8;
    const size_t smem_cap = 227 * 1024;
    // queries per CTA: as many as keep >= 2 CTAs per SM resident, 128 at most (finer CTAs balance better)
    p.T = 128;
    while (p.T > 32 && 2 * (p.bins * ctr * p.T + tile_bytes + 1024) > smem_cap) p.T >>= 1;
    if (p.bins * ctr * p.T + tile_bytes + 1024 > smem_cap) return B200_ERR_UNSUPPORTED;
    while (p.T > 32 && p.T / 2 >= Q) p.T >>= 1;
    p.groups = static_cast<int>(plan_ceil_div<long long>(Q, p.T));
    p.Qpad = p.groups * p.T;
    const size_t smem = p.bins * ctr * p.T + tile_bytes;
    int per_sm = static_cast<int>(smem_cap / (smem + 1024));
    if (per_sm > 2048 / p.T) per_sm = 2048 / p.T;
    if (per_sm > 32) per_sm = 32;
    if (per_sm < 1) per_sm = 1;
    const long long capacity = static_cast<long long>(num_sms) * per_sm;
    // segments: fill the machine once, but keep a segment long enough to amortise the per-CTA counter setup
    const long long min_seg = 4ll * p.bins > 256 ? 4ll * p.bins : 256;
    long long S = capacity / p.groups;
    if (S < 1) S = 1;
    S *= waves < 1 ? 1 : waves;
    const long long s_cap = plan_ceil_div<long long>(N > 0 ? N : 1, min_seg);
    if (S > s_cap) S = s_cap;
    // stash mode: stage B re-reads 1 byte + 1 bit per (row, query) pair instead of scoring the pair again
    const size_t stash_d_bytes = static_cast<size_t>(plan_ceil_div<long long>(N > 0 ? N : 1, 16)) * p.Qpad * 16;
    const size_t stash_r_bytes = static_cast<size_t>(plan_ceil_div<long long>(N > 0 ? N : 1, 32)) * p.Qpad * 4;
    {
        // worth it when most rows are outside the top k (stage B then skips them at 1 byte each).  When k covers the
        // database every row is walked anyway: measured on c3_all, re-scoring in 4-row batches (2.25 ms) beats walking the
        // stash row by row (3.67 ms) and stage A is spared the stores.  B200_MAP_STASH=0/1 forces.
        const char *on = std::getenv("B200_MAP_STASH");
        const bool want = on ? on[0] != '0' : 4 * p.k <= N_total;
        p.stash = (B <= 254 && N > 0 && want && (stash_d_bytes + stash_r_bytes) / (1024 * 1024) < kMapStashMaxMB) ? 1 : 0;
    }
    const long long seg_unit = p.stash ? 32 : 2;
    long long seg = plan_round_up<long long>(plan_ceil_div<long long>(N > 0 ? N : 1, S), seg_unit);
    // stage A, the all-rows walk and the stash rank path count a segment in 16|16-bit shared counters, wide plan or not
    if (seg > 65534) seg = 65534 / seg_unit * seg_unit;
    S = plan_ceil_div<long long>(N > 0 ? N : 1, seg);
    if (S > 65535) return B200_ERR_UNSUPPORTED;   // gridDim.y
    p.S = static_cast<int>(S);
    p.seg_len = static_cast<int>(seg);
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t o = off; off = plan_round_up<size_t>(off + bytes, 256); return o; };
    p.off_hist = carve(static_cast<size_t>(p.S) * p.bins * p.Qpad * ctr_global);
    p.off_tot = carve(static_cast<size_t>(p.bins) * p.Qpad * 2 * sizeof(uint32_t));
    p.off_dstar = carve(static_cast<size_t>(p.Qpad) * sizeof(uint32_t));
    p.off_psum = carve(static_cast<size_t>(p.S) * p.Qpad * sizeof(double));
    p.off_phits = carve(static_cast<size_t>(p.S) * p.Qpad * sizeof(uint32_t));
    p.off_stash_d = carve(p.stash ? stash_d_bytes : 0);
    p.off_stash_r = carve(p.stash ? stash_r_bytes : 0);
    // ---- select mode (see b200ret.h)
    {
        const char *on = std::getenv("B200_MAP_SELECT");
        const bool forced = on && on[0] != '0';
        bool want = allow_select && N == N_total && !p.wide && B <= 254 && N >= 64 && p.k >= 2 && 2 * p.k <= N &&
                    p.k <= 131072;                       // the rank kernel keeps one bit per rank in shared memory
        if (on ? !forced : !(8 * p.k <= N && N >= 32768 && p.k >= 512)) want = false;
        if (want) {
            p.select = 1;
            // sample: enough rows that ~256 of the true top k are in it (relative sigma of the estimate <= 1/16)
            long long stride = p.k / 256;
            stride = stride < 1 ? 1 : (stride > 64 ? 64 : stride);
            if (const char *e = std::getenv("B200_SEL_STRIDE")) stride = std::atoll(e) > 0 ? std::atoll(e) : stride;     // tests
            const long long groups32 = N / 32;                    // whole 32-row groups only
            if (stride > groups32) stride = groups32;
            p.sel_stride = static_cast<int>(stride);
            p.smp_rows = 32 * plan_ceil_div<long long>(groups32, stride);
            // select CTAs = (query groups of sel_T) x segments: about 12 per SM (measured on c3 / c5: 8 -> 12-16 per SM is
            // 5-10 % faster, the candidate density differs between query groups and finer CTAs balance it), with segments of
            // >= 1024 rows so that the per-(query, segment) candidate lists stay long (the rank kernel pays per list); when
            // a GPU has few queries (a slice of a multi-GPU run) the groups shrink to 64 / 32 queries instead of the segments
            const bool stc = plan_select_tc(p);
            const long long cps = stc ? 20 : 12;       // (the append half is latency-bound: finer CTAs, 12 -> 20 per SM: 0.42 -> 0.37 ms on c3)
            const long long want = static_cast<long long>(num_sms) * cps;
            // (few query groups — a slice of a multi-GPU run: 512-row segments; 628 queries of c3: select 0.102 -> 0.088 ms,
            // rank 0.044 -> 0.050 ms)
            const long long min_seg = (p.Qpad / p.T) * plan_ceil_div<long long>(N, 1024) < 6ll * num_sms ? 512 : 1024;
            const long long cap_s = plan_ceil_div<long long>(N, min_seg);
            int tsel = p.T;
            // (groups shrink to 64 / 32 queries only when full groups could not give every SM one CTA: measured on a 628-
            // query slice of c3, 128 / 64 / 32 queries per CTA: 0.101 / 0.105 / 0.132 ms)
            if (!stc)
                while (tsel > 32 && (p.Qpad / tsel) * cap_s < num_sms) tsel >>= 1;
            p.sel_T = tsel;
            long long sS = plan_ceil_div<long long>(want, p.Qpad / tsel);
            if (sS > cap_s) sS = cap_s;
            long long sseg = plan_round_up<long long>(plan_ceil_div<long long>(N, sS), stc ? 256 : 64);      // (whole 256-row tiles of the tensor-core kernel)
            const long long sseg_cap = stc ? 65280 : 65472;       // row-in-segment is a 16-bit field of a candidate entry
            if (sseg > sseg_cap) sseg = sseg_cap;
            sS = plan_ceil_div<long long>(N, sseg);
            if (sS > 65535) p.select = 0;
            p.sel_S = static_cast<int>(sS), p.sel_seg_len = static_cast<int>(sseg);
            p.sel_maxc = 64;                                      // chunks a list can have
            int ch = 128;                                         // a warp reads a chunk 128 entries at a time
            while (static_cast<long long>(ch) * p.sel_maxc < sseg) ch <<= 1;
            p.sel_chunk = ch;
            // pool: half a chunk of slack per (query, segment) list + 4k candidates per query + 16 lifted-bound retries
            const long long lists = static_cast<long long>(p.Qpad) * sS;
            p.sel_pool_chunks = lists + plan_ceil_div<long long>(static_cast<long long>(Q) * (4 * p.k + 1024), ch) +
                                16 * (plan_ceil_div<long long>(N, ch) + sS);
            if (p.sel_pool_chunks >= (1ll << 31)) p.select = 0;
            // sample histogram (select_sample_kernel): (query groups of sel_T) x segments of the sample, about two CTAs per
            // SM (a CTA zeroes and merges a bins x sel_T column block: worth ~150 rows of scoring), segments of whole
            // 32-row groups, at least 128 and at most 65504 rows (16-bit shared counters)
            // (all CTAs are resident at once — 512 threads, <= 4 per SM — so the segment count is the one in [2, 4] CTAs per
            // SM that loads the SMs most evenly: 40 groups x 11 segments = 2.97 per SM on c3)
            const long long sgroups = p.Qpad / tsel;
            long long mS = plan_ceil_div<long long>(2ll * num_sms, sgroups);
            {
                double best = 1e30;
                const long long hi = plan_ceil_div<long long>(4ll * num_sms, sgroups);
                for (long long c = mS; c <= hi; ++c) {
                    const double per_sm = static_cast<double>(c * sgroups) / num_sms;
                    const double ratio = static_cast<double>(plan_ceil_div<long long>(c * sgroups, num_sms)) / per_sm;
                    if (ratio < best - 1e-9) best = ratio, mS = c;
                }
            }
            const long long m_cap = plan_ceil_div<long long>(p.smp_rows, 128);
            if (mS > m_cap) mS = m_cap;
            if (mS < 1) mS = 1;
            long long mseg = plan_round_up<long long>(plan_ceil_div<long long>(p.smp_rows, mS), 32);
            if (mseg > 65504) mseg = 65504;
            mS = plan_ceil_div<long long>(p.smp_rows, mseg);
            if (mS > 65535) p.select = 0;
            p.smp_S = static_cast<int>(mS), p.smp_seg_len = static_cast<int>(mseg);
        }
        if (p.select) {
            p.off_sel_flags = carve(64 * sizeof(uint32_t));
            p.off_smp_hist = carve(static_cast<size_t>(p.bins) * p.Qpad * sizeof(uint32_t));      // right behind the flags: one memset zeroes both
            p.off_sel_bound = carve(static_cast<size_t>(p.Qpad) * sizeof(uint32_t));
            p.off_sel_count = carve(static_cast<size_t>(p.Qpad) * p.sel_S * 2 * sizeof(uint32_t));      // list heads: (length, first chunk)
            p.off_sel_table = carve(static_cast<size_t>(p.Qpad) * p.sel_S * p.sel_maxc * sizeof(uint32_t));
            p.off_sel_pool = carve(static_cast<size_t>(p.sel_pool_chunks) * p.sel_chunk * sizeof(uint32_t));
            p.off_smp_codes = off;                                // == workspace_bytes: no tensor-core form for this plan
            if (plan_select_tc(p)) {
                // e4m3 copies of the codes for the tensor-core filter (rows padded to 128-byte K blocks) + its hit masks: one
                // uint32 per (32-row group, query), whole 256-row tiles
                const size_t bp = static_cast<size_t>((B + 127) / 128) * 128;
                const size_t groups = static_cast<size_t>(plan_ceil_div<long long>(N, 256)) * 8;
                p.off_smp_codes = carve(plan_round_up<size_t>(static_cast<size_t>(N) * bp, 1024) +
                                        plan_round_up<size_t>(static_cast<size_t>(p.Qpad) * bp, 1024) + 2048 + groups * p.Qpad * sizeof(uint32_t));
            }
        }
    }
    p.workspace_bytes = off;
    *plan = p;
    return B200_OK;
}

}  // namespace b200
