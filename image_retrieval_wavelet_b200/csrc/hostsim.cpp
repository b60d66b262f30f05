// CPU simulator of the kernels' per-CTA programs — TEST SUPPORT ONLY (built into libb200ret_sim.so, never into
// libb200ret.so, never loaded by the package).  It executes the very same __host__ __device__ tile programs and
// launch planners as the CUDA kernels, one CTA after the other, every phase for tid = 0..nthreads-1, so the
// indexing / halo / scan logic can be checked against the oracle in a container without a GPU.  It says nothing
// about memory-model or warp-level behaviour: the `-m gpu` tests remain the parity tests proper.
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "b200ret.h"
#include "hamming_core.cuh"
#include "hamming_plan.h"
#include "swt2_plan.h"

namespace b200 {

struct HostExec {
    int nthreads;
    std::vector<unsigned char> *store;
    template <typename Fn>
    void operator()(Fn fn) const {
        for (int t = 0; t < nthreads; ++t) fn(t, nthreads);
    }
    template <typename State>
    State *state(State *) const {
        store->assign(sizeof(State) * static_cast<size_t>(nthreads), 0);
        return reinterpret_cast<State *>(store->data());
    }
    int slot(int t) const { return t; }
};

struct HostLoad {
    bool bulk_stage(const SwtGeom &, const void *, float *, float *, int, int, int, int) const { return false; }   // device only
    void issue(const void *plane, size_t off, int is_u8, uint32_t *raw) const {
        for (int e = 0; e < 4; ++e) {
            if (is_u8)
                raw[e] = static_cast<const uint8_t *>(plane)[off + e];
            else
                std::memcpy(raw + e, static_cast<const float *>(plane) + off + e, 4);
        }
    }
    void finish(const uint32_t *raw, size_t, int is_u8, float *v) const {
        for (int e = 0; e < 4; ++e) {
            if (is_u8)
                v[e] = swt_u8_unit(raw[e]);
            else
                std::memcpy(v + e, raw + e, 4);
        }
    }
    void issue_u8x8(const uint8_t *plane, size_t off, uint32_t *raw) const {      // same three aligned words as the device
        const uint8_t *p = plane + (off & ~static_cast<size_t>(3));
        std::memcpy(raw, p, 8);
        raw[2] = 0;
        if (off & 3) std::memcpy(raw + 2, p + 8, 4);
    }
    void finish_u8x8(const uint32_t *raw, size_t off, float *v) const {
        const uint32_t sh = 8u * (static_cast<uint32_t>(off) & 3u);
        const uint64_t lo = raw[0] | (static_cast<uint64_t>(raw[1]) << 32), hi = raw[1] | (static_cast<uint64_t>(raw[2]) << 32);
        const uint32_t w[2] = {static_cast<uint32_t>(lo >> sh), static_cast<uint32_t>(hi >> sh)};
        for (int e = 0; e < 8; ++e) v[e] = swt_u8_unit((w[e / 4] >> (8 * (e & 3))) & 0xffu);
    }
    float one(const void *plane, size_t off, int is_u8) const {
        return is_u8 ? swt_u8_unit(static_cast<const uint8_t *>(plane)[off]) : static_cast<const float *>(plane)[off];
    }
};
struct HostStore {
    void vec4(float *p, const float *v) const {
        for (int e = 0; e < 4; ++e) p[e] = v[e];
    }
    void operator()(float *p, const float *v, int n) const {
        for (int e = 0; e < n; ++e) p[e] = v[e];
    }
};
struct HostLoadTile {
    void operator()(uint32_t *dst, const uint64_t *src, int n16, int t, int nt) const {
        for (int i = t; i < n16; i += nt) std::memcpy(dst + 4 * i, reinterpret_cast<const unsigned char *>(src) + 16 * i, 16);
    }
};

template <int F>
static void run_swt_level(const SwtGeom &g, const void *in, float *out, SwtTileId id, float *smem, HostExec ex) {
    switch (g.level) {
        case 1: swt_tile_program<F, 1>(g, in, out, id, smem, ex, HostStore{}, HostLoad{}); break;
        case 2: swt_tile_program<F, 2>(g, in, out, id, smem, ex, HostStore{}, HostLoad{}); break;
        case 3: swt_tile_program<F, 3>(g, in, out, id, smem, ex, HostStore{}, HostLoad{}); break;
    }
}

// The pass form the launcher runs: swt_rw_form (-1: the generic program), swt_vs_form, and the uint8 staging units.
static void swt_plan_forms(const SwtGeom &g, int *rw, int *vs, int *u8_stage) {
    const bool fast = swt_fast_path(g.F, g.level);
    *rw = fast ? swt_rw_form(g.F, g.level) : -1;
    *vs = fast ? swt_vs_form(g.F, g.level) : 0;
    *u8_stage = g.u8_stage;
}

template <int CW, int LW, bool EQ>
static void run_walk3(bool wide, int phase, bool all, const MapArgs &a, int gx, int gy, int T, unsigned char *smem, HostExec ex) {
    if (!phase) {
        if (wide)
            hamming_hist_program<CW, LW, EQ, true>(a, gx, gy, T, smem, ex, HostLoadTile{});
        else
            hamming_hist_program<CW, LW, EQ, false>(a, gx, gy, T, smem, ex, HostLoadTile{});
    } else if (wide) {
        if (all)
            hamming_walk_program<CW, LW, EQ, true, true>(a, gx, gy, T, smem, ex, HostLoadTile{});
        else
            hamming_walk_program<CW, LW, EQ, true, false>(a, gx, gy, T, smem, ex, HostLoadTile{});
    } else {
        if (all)
            hamming_walk_program<CW, LW, EQ, false, true>(a, gx, gy, T, smem, ex, HostLoadTile{});
        else
            hamming_walk_program<CW, LW, EQ, false, false>(a, gx, gy, T, smem, ex, HostLoadTile{});
    }
}
template <int CW>
static void run_walk2(int lw, bool eq, bool wide, int phase, bool all, const MapArgs &a, int gx, int gy, int T,
                      unsigned char *smem, HostExec ex) {
    if (eq) return run_walk3<CW, 1, true>(wide, phase, all, a, gx, gy, T, smem, ex);
    switch (lw) {
        case 1: return run_walk3<CW, 1, false>(wide, phase, all, a, gx, gy, T, smem, ex);
        case 2: return run_walk3<CW, 2, false>(wide, phase, all, a, gx, gy, T, smem, ex);
        case 4: return run_walk3<CW, 4, false>(wide, phase, all, a, gx, gy, T, smem, ex);
    }
}
static void run_walk(const b200_map_plan &p, int phase, const MapArgs &a, std::vector<unsigned char> &smem,
                     std::vector<unsigned char> &states) {
    const int cw = b200_code_words(p.B);
    const bool eq = p.label_mode == B200_LABELS_EQUAL;
    const char *tpq_env = std::getenv("B200_MAP_TPQ");
    const int tpq_req = tpq_env ? std::atoi(tpq_env) : 2;
    const int tpq = phase == 0 ? (tpq_req >= 1 && tpq_req <= 4 ? tpq_req : 2) : 1;      // stage A: threads per query, like the launcher
    HostExec ex{p.T * tpq, &states};
    for (int gy = 0; gy < p.S; ++gy)
        for (int gx = 0; gx < p.groups; ++gx) {
            std::fill(smem.begin(), smem.end(), 0xCD);      // poison: nothing may rely on zeroed shared memory
            const bool all = p.k >= p.N_total;
            if (phase == 1 && p.stash) {                    // stage B from the stash: no scoring
                if (p.wide) {
                    if (all) hamming_rank_program<true, true>(a, gx, gy, p.T, smem.data(), ex);
                    else hamming_rank_program<true, false>(a, gx, gy, p.T, smem.data(), ex);
                } else {
                    if (all) hamming_rank_program<false, true>(a, gx, gy, p.T, smem.data(), ex);
                    else hamming_rank_program<false, false>(a, gx, gy, p.T, smem.data(), ex);
                }
                continue;
            }
            switch (cw) {
                case 1: run_walk2<1>(p.LW, eq, p.wide, phase, all, a, gx, gy, p.T, smem.data(), ex); break;
                case 2: run_walk2<2>(p.LW, eq, p.wide, phase, all, a, gx, gy, p.T, smem.data(), ex); break;
                case 4: run_walk2<4>(p.LW, eq, p.wide, phase, all, a, gx, gy, p.T, smem.data(), ex); break;
            }
        }
}

static MapArgs make_args(const b200_map_plan &p, const uint64_t *qc, const uint64_t *ql, const uint64_t *dc, const uint64_t *dl,
                         unsigned char *ws, uint32_t *rank_idx, uint16_t *rank_dist, long long index_base) {
    MapArgs a;
    a.gate = nullptr;
    a.q_codes = qc, a.q_labels = ql, a.db_codes = dc, a.db_labels = dl;
    a.hist = ws + p.off_hist;
    a.dstar = reinterpret_cast<const uint32_t *>(ws + p.off_dstar);
    a.psum = reinterpret_cast<unsigned long long *>(ws + p.off_psum);
    a.phits = reinterpret_cast<uint32_t *>(ws + p.off_phits);
    a.rank_idx = rank_idx, a.rank_dist = rank_dist, a.index_base = index_base;
    a.seg_base = 0;
    a.stash_d = p.stash ? reinterpret_cast<U32x4 *>(ws + p.off_stash_d) : nullptr;
    a.stash_r = p.stash ? reinterpret_cast<uint32_t *>(ws + p.off_stash_r) : nullptr;
    a.Q = p.Q, a.N = static_cast<int>(p.N), a.bins = p.bins, a.seg_len = p.seg_len, a.tile = p.tile, a.Qpad = p.Qpad;
    a.k = static_cast<uint32_t>(p.k);
    return a;
}

}  // namespace b200

using namespace b200;

extern "C" {

// Same planner, same tile programs as b200_swt2_fwd; host pointers.
int sim_swt2_fwd(const void *in, int in_is_u8, float *out, int B, int C, int H, int W, const float *lo, const float *hi, int F,
                 int level, int num_sms, int *plan_out /* TH, TW, rw form, threads, vs form, RH, RWp, u8_stage or NULL */) {
    SwtGeom g;
    const int rc = swt_plan(g, B, C, H, W, F, level, in_is_u8, lo, hi, num_sms);
    if (rc == -1) return B200_ERR_INVALID_ARG;
    if (rc) return B200_ERR_UNSUPPORTED;
    if (plan_out) {
        plan_out[0] = g.TH, plan_out[1] = g.TW, plan_out[3] = g.threads, plan_out[5] = g.RH, plan_out[6] = g.RWp;
        swt_plan_forms(g, plan_out + 2, plan_out + 4, plan_out + 7);
    }
    std::vector<float> smem(swt_smem_bytes(g) / sizeof(float));
    std::vector<unsigned char> states;
    HostExec ex{g.threads, &states};
    for (int plane = 0; plane < B * C; ++plane)
        for (int ty = 0; ty < g.tiles_y; ++ty)
            for (int tx = 0; tx < g.tiles_x; ++tx) {
                const SwtTileId id{plane, ty, tx};
                for (auto &x : smem) x = -1.0e30f;                  // poison
                if (swt_fast_path(F, level)) {
                    switch (F) {
                        case 2: run_swt_level<2>(g, in, out, id, smem.data(), ex); break;
                        case 4: run_swt_level<4>(g, in, out, id, smem.data(), ex); break;
                        case 6: run_swt_level<6>(g, in, out, id, smem.data(), ex); break;
                        case 8: run_swt_level<8>(g, in, out, id, smem.data(), ex); break;
                        case 10: run_swt_level<10>(g, in, out, id, smem.data(), ex); break;
                    }
                } else {
                    swt_generic_program(g, in, out, id, smem.data(), ex, HostLoad{});
                }
            }
    return B200_OK;
}

// The uint8 -> [0, 1] conversion of the staging phase (must equal b / 255.0f bit for bit).
float sim_u8_unit(unsigned b) { return swt_u8_unit(b); }

// Planner only: TH, TW, rw form, threads, vs form, RH, RWp, smem bytes, CTAs, u8_stage (forms: swt_plan_forms).
int sim_swt2_plan(int B, int C, int H, int W, int F, int level, int in_is_u8, int num_sms, long long *plan_out) {
    SwtGeom g;
    float z[20] = {0};
    const int rc = swt_plan(g, B, C, H, W, F, level, in_is_u8, z, z, num_sms);
    if (rc) return rc;
    int rw, vs, u8_stage;
    swt_plan_forms(g, &rw, &vs, &u8_stage);
    plan_out[0] = g.TH, plan_out[1] = g.TW, plan_out[2] = rw, plan_out[3] = g.threads, plan_out[4] = vs;
    plan_out[5] = g.RH, plan_out[6] = g.RWp, plan_out[7] = static_cast<long long>(swt_smem_bytes(g));
    plan_out[8] = static_cast<long long>(B) * C * g.tiles_y * g.tiles_x, plan_out[9] = u8_stage;
    return 0;
}

// Hamming mAP over packed inputs with the database split into n_shards contiguous shards, each running the same
// stage programs and planner as one GPU would (totals "all-gathered" through host memory).  n_shards == 1 and
// force_ext == 0 is exactly b200_hamming_map.  rank_idx / rank_dist (may be NULL): [Q][k] global ranked list.
int sim_hamming_map(const uint64_t *qc, const uint64_t *ql, const uint64_t *dc, const uint64_t *dl, int Q, long long N, int B,
                    int LW, int label_mode, long long k, int n_shards, int force_ext, int num_sms, double *ap, uint32_t *tsum,
                    double *map_out, uint32_t *rank_idx, uint16_t *rank_dist, int *plan_out /* T, S, seg_len, wide */) {
    if (n_shards < 1) return B200_ERR_INVALID_ARG;
    const int cw = b200_code_words(B);
    const long long per = (N + n_shards - 1) / n_shards;
    struct Shard {
        b200_map_plan plan;
        long long base;
        std::vector<uint64_t> codes, labels;
        std::vector<unsigned char> ws;
    };
    std::vector<Shard> sh(n_shards);
    long long k_eff = 0;
    for (int r = 0; r < n_shards; ++r) {
        Shard &s = sh[r];
        s.base = std::min<long long>(N, per * r);
        const long long n = std::min<long long>(N, per * (r + 1)) - s.base;
        const int rc = map_plan_init(&s.plan, Q, n, N, B, LW, label_mode, k, num_sms);
        if (rc) return rc;
        k_eff = s.plan.k;
        const long long padded = (n + 1) / 2 * 2;
        s.codes.assign(static_cast<size_t>(padded) * cw + 2, 0);
        s.labels.assign(static_cast<size_t>(padded) * LW + 2, 0);
        if (n) {
            std::memcpy(s.codes.data(), dc + s.base * cw, sizeof(uint64_t) * n * cw);
            std::memcpy(s.labels.data(), dl + s.base * LW, sizeof(uint64_t) * n * LW);
        }
        s.ws.assign(s.plan.workspace_bytes, 0xCD);
    }
    if (plan_out) {
        plan_out[0] = sh[0].plan.T, plan_out[1] = sh[0].plan.S, plan_out[2] = sh[0].plan.seg_len, plan_out[3] = sh[0].plan.wide + 2 * sh[0].plan.stash;
    }
    if (rank_idx) std::memset(rank_idx, 0xFF, sizeof(uint32_t) * static_cast<size_t>(Q) * k_eff);
    if (rank_dist) std::memset(rank_dist, 0xFF, sizeof(uint16_t) * static_cast<size_t>(Q) * k_eff);
    std::vector<unsigned char> smem(227 * 1024), states;
    // stage A + shard totals
    const bool use_ext = n_shards > 1 || force_ext;
    const size_t tot_items = static_cast<size_t>(sh[0].plan.bins) * sh[0].plan.Qpad;
    std::vector<U32x2> gathered(use_ext ? tot_items * n_shards : 0);
    for (int r = 0; r < n_shards; ++r) {
        Shard &s = sh[r];
        MapArgs a = make_args(s.plan, qc, ql, s.codes.data(), s.labels.data(), s.ws.data(), nullptr, nullptr, 0);
        run_walk(s.plan, 0, a, smem, states);
        if (use_ext) {
            if (s.plan.Qpad != sh[0].plan.Qpad) return B200_ERR_UNSUPPORTED;
            U32x2 *tot = reinterpret_cast<U32x2 *>(s.ws.data() + s.plan.off_tot);
            for (size_t i = 0; i < tot_items; ++i) {
                if (s.plan.wide)
                    hamming_totals_item<true>(s.ws.data() + s.plan.off_hist, s.plan.S, tot_items, i, tot);
                else
                    hamming_totals_item<false>(s.ws.data() + s.plan.off_hist, s.plan.S, tot_items, i, tot);
            }
            std::memcpy(gathered.data() + tot_items * r, tot, sizeof(U32x2) * tot_items);
        }
    }
    // stage S + stage B + per-shard reduction
    std::vector<unsigned long long> sums(static_cast<size_t>(n_shards) * Q);
    std::vector<uint32_t> hits(static_cast<size_t>(n_shards) * Q);
    for (int r = 0; r < n_shards; ++r) {
        Shard &s = sh[r];
        const b200_map_plan &p = s.plan;
        HostExec ex{kScanQ * kScanY, &states};
        uint32_t *dstar = reinterpret_cast<uint32_t *>(s.ws.data() + p.off_dstar);
        for (int gx = 0; gx < p.Qpad / kScanQ; ++gx) {
            std::fill(smem.begin(), smem.end(), 0xCD);
            if (p.wide)
                hamming_scan_program<true>(s.ws.data() + p.off_hist, p.S, p.bins, p.Qpad, static_cast<uint32_t>(p.k),
                                           use_ext ? gathered.data() : nullptr, n_shards, r, dstar, gx, smem.data(), ex);
            else
                hamming_scan_program<false>(s.ws.data() + p.off_hist, p.S, p.bins, p.Qpad, static_cast<uint32_t>(p.k),
                                            use_ext ? gathered.data() : nullptr, n_shards, r, dstar, gx, smem.data(), ex);
        }
        MapArgs a = make_args(p, qc, ql, s.codes.data(), s.labels.data(), s.ws.data(), rank_idx, rank_dist, s.base);
        run_walk(p, 1, a, smem, states);
        for (int q = 0; q < Q; ++q)
            ap_reduce_item(a.psum, a.phits, p.S, p.Qpad, q, sums.data() + static_cast<size_t>(r) * Q,
                           hits.data() + static_cast<size_t>(r) * Q);
    }
    double total = 0.0;
    for (int q = 0; q < Q; ++q) {
        ap_finalize_item(sums.data(), hits.data(), n_shards, Q, q, ap, tsum);
        total += ap[q];
    }
    if (map_out) *map_out = total / Q;
    return B200_OK;
}

// ---- stage-level entry points: same signatures as the C-ABI (include/b200ret.h) minus the stream, host memory.
// They let the sharded evaluator's collective choreography (image_retrieval_wavelet_b200/engine/dist.py) run under
// torch.distributed's gloo backend on CPU with the real stage programs.
int sim_map_plan_init(b200_map_plan *plan, int Q, long long N, long long N_total, int B, int LW, int label_mode, long long k,
                      int num_sms) {
    return map_plan_init(plan, Q, N, N_total, B, LW, label_mode, k, num_sms);
}

int sim_hamming_hist(const b200_map_plan *p, const uint64_t *qc, const uint64_t *ql, const uint64_t *dc, const uint64_t *dl,
                     void *workspace) {
    std::vector<unsigned char> smem(227 * 1024), states;
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    MapArgs a = make_args(*p, qc, ql, dc, dl, ws, nullptr, nullptr, 0);
    run_walk(*p, 0, a, smem, states);
    const size_t items = static_cast<size_t>(p->bins) * p->Qpad;
    U32x2 *tot = reinterpret_cast<U32x2 *>(ws + p->off_tot);
    for (size_t i = 0; i < items; ++i) {
        if (p->wide)
            hamming_totals_item<true>(ws + p->off_hist, p->S, items, i, tot);
        else
            hamming_totals_item<false>(ws + p->off_hist, p->S, items, i, tot);
    }
    return B200_OK;
}

int sim_hamming_scan(const b200_map_plan *p, void *workspace, const uint32_t *tot_all_shards, int n_shards, int shard) {
    std::vector<unsigned char> smem(227 * 1024), states;
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    HostExec ex{kScanQ * kScanY, &states};
    uint32_t *dstar = reinterpret_cast<uint32_t *>(ws + p->off_dstar);
    const U32x2 *ext = reinterpret_cast<const U32x2 *>(tot_all_shards);
    for (int gx = 0; gx < p->Qpad / kScanQ; ++gx) {
        std::fill(smem.begin(), smem.end(), 0xCD);
        if (p->wide)
            hamming_scan_program<true>(ws + p->off_hist, p->S, p->bins, p->Qpad, static_cast<uint32_t>(p->k), ext, n_shards, shard,
                                       dstar, gx, smem.data(), ex);
        else
            hamming_scan_program<false>(ws + p->off_hist, p->S, p->bins, p->Qpad, static_cast<uint32_t>(p->k), ext, n_shards, shard,
                                        dstar, gx, smem.data(), ex);
    }
    return B200_OK;
}

int sim_hamming_ap(const b200_map_plan *p, const uint64_t *qc, const uint64_t *ql, const uint64_t *dc, const uint64_t *dl,
                   void *workspace, uint32_t *rank_idx, uint16_t *rank_dist, long long index_base) {
    std::vector<unsigned char> smem(227 * 1024), states;
    MapArgs a = make_args(*p, qc, ql, dc, dl, static_cast<unsigned char *>(workspace), rank_idx, rank_dist, index_base);
    run_walk(*p, 1, a, smem, states);
    return B200_OK;
}

int sim_ap_reduce(const b200_map_plan *p, void *workspace, uint64_t *sum_q, uint32_t *hits_q) {
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    for (int q = 0; q < p->Q; ++q)
        ap_reduce_item(reinterpret_cast<const unsigned long long *>(ws + p->off_psum),
                       reinterpret_cast<const uint32_t *>(ws + p->off_phits), p->S, p->Qpad, q,
                       reinterpret_cast<unsigned long long *>(sum_q), hits_q);
    return B200_OK;
}

int sim_ap_finalize(const uint64_t *sums, const uint32_t *hits, int n_parts, long long stride, int Q, double *ap, uint32_t *tsum,
                    double *map_out) {
    double total = 0.0;
    for (int q = 0; q < Q; ++q) {
        ap_finalize_item(reinterpret_cast<const unsigned long long *>(sums), hits, n_parts, stride, q, ap, tsum);
        total += ap[q];
    }
    if (map_out) *map_out = Q ? total / Q : 0.0;
    return B200_OK;
}

}  // extern "C"
