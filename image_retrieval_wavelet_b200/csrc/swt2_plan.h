// Host-side tile planner for the SWT kernel (shared by the CUDA launcher and the CPU host simulator used in tests).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstddef>

#include "swt2_core.cuh"

namespace b200 {

inline bool swt_fast_path(int F, int level) {
    return F >= 2 && F <= 10 && (F % 2) == 0 && level >= 1 && level <= kSwtMaxLevelFast;
}

inline size_t swt_smem_bytes(const SwtGeom &g) { return static_cast<size_t>(g.smem_floats) * sizeof(float); }

// Fills the geometry that follows from (TH, TW): staging region, buffers, division constants.
inline void swt_fill_geometry(SwtGeom &g, int th, int tw, bool fast) {
    g.TH = th, g.TW = tw;
    g.tiles_y = (g.H + th - 1) / th;
    g.tiles_x = (g.W + tw - 1) / tw;
    g.RH = th + g.top + g.bot;
    g.RWp = (g.padL + tw + g.right + 3) / 4 * 4;
    const int S = 1 << (g.level - 1);
    g.RHv = th + S * (g.F - 1);
    const size_t buf = static_cast<size_t>(g.RH) * g.RWp;
    if (fast) {
        g.nbuf = 2;
        g.off_b = static_cast<int>(kSwtGuard + buf + kSwtGuard);
        const size_t b_floats = std::max<size_t>(g.level > 1 ? buf : 0, static_cast<size_t>(2) * g.RHv * tw);
        g.smem_floats = static_cast<int>(g.off_b + b_floats + kSwtGuard);
    } else {
        g.nbuf = 3;
        g.off_b = 0;
        g.smem_floats = static_cast<int>(3 * (buf + 2 * kSwtGuard));
    }
    g.m_load = swt_magic(static_cast<uint32_t>(g.RWp / 4));
    g.m_load8 = swt_magic(static_cast<uint32_t>((g.RWp + kSwtU8Chunk - 1) / kSwtU8Chunk));
    for (int l = 0; l < kSwtMaxLevelFast; ++l) g.m_lvl[l] = 0;
    if (fast) {
        for (int l = 1; l < g.level; ++l) {
            int c0g, ncg;
            swt_level_cols(g, l, c0g, ncg);
            g.m_lvl[l - 1] = swt_magic(static_cast<uint32_t>(ncg));
        }
        g.m_lvl[g.level - 1] = swt_magic(static_cast<uint32_t>(tw / 4));
    }
}

// Chooses the output tile.  Cost = estimated issued instructions per output pixel (staging, intermediate levels over
// their halo-amplified regions, last level) x tail imbalance over the SMs x a penalty when fewer than two CTAs fit an
// SM's shared memory.  TW is a multiple of 4 (a tile may overhang the image: overhanging columns are staged wrapped
// and never stored); TH a multiple of kSwtR * 2^(level-1) on the fast path.
inline int swt_plan(SwtGeom &g, int B, int C, int H, int W, int F, int level, int in_is_u8, const float *lo, const float *hi,
                    int num_sms) {
    if (B < 1 || C < 1 || H < 1 || W < 1 || F < 2 || (F & 1) || F > 20 || level < 1 || level > 4) return -1;
    if (H % (1 << level) || W % (1 << level)) return -1;
    g = SwtGeom{};
    g.B = B, g.C = C, g.H = H, g.W = W, g.level = level, g.F = F, g.in_is_u8 = in_is_u8;
    for (int i = 0; i < 20; ++i) g.lo[i] = i < F ? lo[i] : 0.f, g.hi[i] = i < F ? hi[i] : 0.f;
    const bool fast = swt_fast_path(F, level);
    const int span = (1 << level) - 1;
    g.top = g.left = span * (F / 2 - 1);
    g.bot = g.right = span * (F / 2);
    g.padL = (g.left + 3) / 4 * 4;
    g.threads = 256;
    const int S = 1 << (level - 1);
    // Pass forms (swt2_core.cuh: swt_rw_form, swt_vs_form), measured on B200 (round 2):
    // - hybrid (register-window intermediate levels, swt_rw_ll; 256x3x520x520 uint8, fraction of the HBM roofline,
    //   two-pass -> hybrid): haar level 2 0.75 -> 0.79, db2 level 2 0.56 -> 0.61, haar level 3 0.53 -> 0.64, db2 level 3
    //   0.40 -> 0.43; the 8-tap filters lose 3-9 % (the 15 / 8 horizontal FMAs of an 8-row window outweigh the saved
    //   shared-memory round trip).  An all-register form (register-window last level too) lost everywhere: 128
    //   registers leave 16 warps per SM (db4 level 1: 0.58 -> 0.42).
    // - sliding last vertical pass (swt_vpass_final_slide; C4 grid, blocked -> sliding): db4 / sym4 level 1 0.581 ->
    //   0.605 of the HBM roofline (the 8-tap kernel drops from 80 to 64 registers: 7 % fewer instructions, 36 % fewer
    //   shared-memory wavefronts); the short filters lose (haar level 1 0.81 -> 0.62: their blocked pass has 4 output
    //   rows per unit already and twice the stores per unit), bior4.4 loses (0.52 -> 0.47) and so do levels 2 / 3 with
    //   every tile tried (db4 level 2 0.395 -> 0.33-0.37: TH must be a multiple of 8 * 2^(level-1)).
    const bool vs = fast && swt_vs_form(F, level);
    const int th_unit = fast ? (vs ? kVsR : kSwtR) * S : 1;
    const long long planes = static_cast<long long>(B) * C;
    double best = 1e30;
    int bth = 0, btw = 0;
    for (int nx = 1; nx <= 64; ++nx) {
        int tw = ((W + nx - 1) / nx + 3) / 4 * 4;
        if (nx > 1 && tw < 32) break;
        for (int th0 : {128, 96, 64, 48, 32, 24, 16, 8, 4, 2, 1}) {
            int th = (std::min(th0, H) + th_unit - 1) / th_unit * th_unit;
            if (th > 128) continue;
            SwtGeom t = g;
            swt_fill_geometry(t, th, tw, fast);
            const size_t bytes = swt_smem_bytes(t);
            if (bytes > 200 * 1024) continue;
            const double area = static_cast<double>(th) * tw;
            // issued thread-instructions of each phase, with the phase's units rounded up to whole CTA sweeps
            auto phase = [&](double units, double per_unit) { return std::ceil(units / g.threads) * g.threads * per_unit; };
            double cost = phase(static_cast<double>(t.RH) * (t.RWp / 4), 30.0);      // staging
            if (fast) {
                for (int l = 1; l < level; ++l) {                                     // intermediate levels (LL only)
                    const int sp = (1 << l) - 1, sp0 = (1 << (l - 1)) - 1, sl = 1 << (l - 1);
                    int c0g, ncg;
                    swt_level_cols(t, l, c0g, ncg);
                    const double rows_h = t.RH - sp0 * (F - 1), rows_v = t.RH - sp * (F - 1);
                    cost += phase(rows_h * ncg, 4.0 * F + 14.0);
                    cost += phase(static_cast<double>(ncg) * sl * std::ceil(std::ceil(rows_v / sl) / kSwtR), kSwtR * 4.0 * F + kSwtR + F + 12.0);
                }
                cost += phase(static_cast<double>(t.RHv) * (tw / 4), 8.0 * F + 16.0);                      // last level, horizontal
                cost += phase(static_cast<double>(tw / 4) * (th / kSwtR), kSwtR * 16.0 * F + 2.0 * (kSwtR + F) + 12.0 * kSwtR);   // vertical + stores
            } else {
                cost += 40.0 * F * level * t.RH * t.RWp;
            }
            cost = cost / area + 2500.0 / area;                                      // + per-CTA launch / barrier bubbles
            cost *= static_cast<double>(t.tiles_y) * th / H * (static_cast<double>(t.tiles_x) * tw / W);   // overhang
            const double ctas = static_cast<double>(planes) * t.tiles_y * t.tiles_x;
            const int per_sm = static_cast<int>(std::min(8.0, std::floor(227.0 * 1024 / static_cast<double>(bytes + 1024))));
            cost *= 1.0 + 0.5 * num_sms * std::min(per_sm, 4) / ctas;                 // tail: about half a wave
            if (per_sm < 2) cost *= 1.35;                                             // nothing hides the staging phase
            else if (per_sm < 3) cost *= 1.08;
            if (cost < best) best = cost, bth = th, btw = tw;
        }
    }
    // Measured on B200 (tile-shape sweeps, profiles/): small CTAs whose staging / horizontal / vertical phases interleave
    // across many resident CTAs beat what the instruction-count model above predicts.  Level 1: 128 threads, 16-row
    // (F <= 4) or 48-row tiles about 112 / 76 columns wide; deeper levels: 256 threads, 48 x ~76 tiles.  The model's
    // choice stays as the fallback when the preferred tile does not fit.
    if (fast) {
        const int want_th = (level == 1 && F <= 4) ? 16 : ((level == 1 && F == 8) ? 32 : 48);      // db4 level 1: 32x76 0.53, 48x76 0.48
        const int want_tw = (level == 1 && F <= 4) ? 112 : 76;
        const int nx = (W + want_tw - 1) / want_tw;
        const int tw = ((W + nx - 1) / nx + 3) / 4 * 4;
        const int th = (std::min(want_th, H) + th_unit - 1) / th_unit * th_unit;
        SwtGeom t = g;
        swt_fill_geometry(t, th, tw, fast);
        if (swt_smem_bytes(t) <= 110 * 1024) {
            bth = th, btw = tw;
            g.threads = level == 1 ? 128 : 256;
        }
    }
    if (bth == 0) return -2;
    swt_fill_geometry(g, bth, btw, fast);
    // uint8 staging units (swt2_core.cuh): 8 pixels per unit, except where rows are 4-byte aligned AND the kernel is a
    // short level-1 filter — there a 4-pixel unit is already one aligned load and the finer units balance better
    // (measured on B200, same box: 224x224 haar 32.7 vs 33.7 us, 520x520 db2 668 vs 680 us; 518-wide rows and long
    // filters gain 5-11 % from the 8-pixel units: db4 983 -> 932 us, bior4.4 1133 -> 1024 us, haar 635 -> 606 us)
    g.u8_stage = in_is_u8 ? ((W % 4 == 0 && level == 1 && F <= 4) ? 0 : 1) : 0;
    if (vs) {
        // the sliding pass has 4 * (TW / 4) * TH / kVsR units: the CTA size that leaves the fewest idle lanes in its sweeps
        const int units = 4 * ((g.TW + 3) / 4) * (g.TH / kVsR);
        double best_eff = 0;
        int best_t = g.threads;
        for (int t = 128; t <= 256; t += 32) {
            const int sweeps = (units + t - 1) / t;
            const double eff = static_cast<double>(units) / (static_cast<double>(sweeps) * t) - (t == g.threads ? 0.0 : 1e-3);
            if (eff > best_eff) best_eff = eff, best_t = t;
        }
        g.threads = best_t;
    }
    return 0;
}

}  // namespace b200
