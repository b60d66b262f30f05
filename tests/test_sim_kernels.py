"""The kernels' tile programs, executed on the CPU by the simulator (csrc/hostsim.cpp: same __host__ __device__ code
and planners as the CUDA build), against the oracle.  This is what can be checked without a GPU: indexing, halos, tile
planning, counter packing, scan and shard logic.  Device-only behaviour is covered by the -m gpu tests."""
import numpy as np
import pytest

from oracle import c_oracle, eval_ref, filters
from simlib import correlated_codes, multi_hot, pm1, sim_map, sim_swt

SWT_CASES = [
    ((2, 3, 224, 224), "haar", 1, np.uint8),      # BASELINE config C1 shape (small batch)
    ((1, 2, 32, 40), "db2", 2, np.float32),
    ((1, 1, 64, 72), "sym4", 3, np.float32),
    ((1, 1, 518, 518), "haar", 1, np.uint8),      # W % 4 != 0: 64-bit vector path
    ((1, 1, 520, 520), "db4", 3, np.uint8),       # C4 worst halo (49 rows/cols)
    ((1, 2, 48, 36), "bior4.4", 2, np.uint8),     # F = 10, biorthogonal
    ((1, 1, 30, 34), "db2", 1, np.float32),
    ((1, 1, 32, 32), "db7", 2, np.float32),       # F = 14: generic program
    ((1, 1, 16, 16), "db3", 1, np.uint8),
    ((1, 1, 8, 8), "db4", 3, np.float32),         # image smaller than the dilated filter: multiple wraps
    ((1, 1, 64, 64), "haar", 4, np.float32),      # level 4: generic program
    ((3, 1, 136, 200), "coif1", 3, np.uint8),
    ((1, 1, 2, 2), "haar", 1, np.uint8),          # minimum size
    ((1, 1, 24, 36), "sym4", 1, np.float32),      # sliding last pass: float32, smaller than one tile
    ((1, 1, 66, 94), "bior4.4", 1, np.uint8),     # F = 10 level 1: W % 4 = 2
    ((2, 1, 40, 36), "db2", 2, np.uint8),         # hybrid, uint8
    ((1, 1, 8, 8), "db2", 3, np.uint8),           # hybrid: smaller than one tile
]


@pytest.mark.parametrize("shape,name,level,dtype", SWT_CASES)
def test_swt_tile_program(sim, shape, name, level, dtype):
    rng = np.random.default_rng(sum(shape) + level)
    x = rng.integers(0, 256, shape).astype(np.uint8) if dtype == np.uint8 else rng.random(shape, dtype=np.float32)
    lo, hi = filters.filter_bank(name)
    rc, out, plan = sim_swt(sim, x, lo, hi, level)
    assert rc == 0
    ref = c_oracle.swt2(x, lo, hi, level)
    assert not np.isnan(out).any(), "some output pixel was never written"
    for band in range(4):
        tol = 1e-5 * max(np.abs(ref[:, :, band]).max(), 1e-30)
        assert np.abs(out[:, :, band] - ref[:, :, band]).max() <= tol, (band, plan)


# (F, level, W, uint8) -> (rw form, vs form, u8_stage); rw -1: the generic program
FORM_CASES = [
    ((2, 1, 224, 1), (0, 0, 0)), ((4, 1, 224, 1), (0, 0, 0)), ((6, 1, 224, 1), (0, 0, 1)), ((10, 1, 224, 0), (0, 0, 0)),   # two-pass
    ((2, 1, 518, 1), (0, 0, 1)), ((4, 1, 518, 0), (0, 0, 0)), ((10, 1, 518, 1), (0, 0, 1)),
    ((8, 1, 518, 1), (0, 1, 1)), ((8, 1, 224, 1), (0, 1, 1)), ((8, 1, 224, 0), (0, 1, 0)),                                 # sliding
    ((2, 2, 520, 1), (2, 0, 1)), ((4, 2, 520, 0), (2, 0, 0)), ((2, 3, 520, 1), (2, 0, 1)), ((4, 3, 256, 1), (2, 0, 1)),    # hybrid
    ((6, 2, 520, 1), (0, 0, 1)), ((8, 2, 520, 1), (0, 0, 1)), ((10, 2, 520, 0), (0, 0, 0)),                                # two-pass
    ((6, 3, 520, 0), (0, 0, 0)), ((8, 3, 520, 1), (0, 0, 1)), ((10, 3, 520, 1), (0, 0, 1)),
    ((12, 1, 224, 1), (-1, 0, 1)), ((20, 2, 224, 0), (-1, 0, 0)), ((2, 4, 224, 1), (-1, 0, 1)), ((4, 4, 224, 0), (-1, 0, 0)),  # generic
]


@pytest.mark.parametrize("case,forms", FORM_CASES)
def test_swt_plan_picks_the_form_of_filter_and_level(sim, case, forms):
    """The pass form is a function of (F, level) alone: hybrid for levels 2-3 under F <= 4, the sliding last pass for
    F = 8 at level 1, two-pass otherwise on the fast path; uint8 staging in 4-pixel units only for 4-byte aligned rows
    under a short level-1 filter."""
    import ctypes

    F, level, W, u8 = case
    plan = (ctypes.c_longlong * 10)()
    assert sim.sim_swt2_plan(4, 3, 224, W, F, level, u8, 148, plan) == 0
    assert (plan[2], plan[4], plan[9]) == forms, list(plan)
    if forms[0] >= 0:                                      # fast path: TH is a whole number of vertical units
        assert plan[0] % ((8 if forms[1] else 4) << (level - 1)) == 0, list(plan)


def _swt_rolled(sim, x, name, level, dy, dx):
    """x rolled by (dy, dx) through its planned pass form: parity with the rolled oracle and, for a non-zero roll, the
    rolled sub-bands of x bit for bit (the periodic SWT commutes with circular shifts, and every pixel is computed in the
    same order wherever tiles, staging units and register windows cut the image)."""
    lo, hi = filters.filter_bank(name)
    rc, out, plan = sim_swt(sim, np.roll(x, (dy, dx), axis=(2, 3)), lo, hi, level)
    assert rc == 0
    assert not np.isnan(out).any(), "some output pixel was never written"
    ref = np.roll(c_oracle.swt2(x, lo, hi, level), (dy, dx), axis=(3, 4))
    for band in range(4):
        assert np.abs(out[:, :, band] - ref[:, :, band]).max() <= 1e-5 * max(np.abs(ref[:, :, band]).max(), 1e-30), (band, plan)
    if dy or dx:
        rc0, out0, _ = sim_swt(sim, x, lo, hi, level)
        assert rc0 == 0 and np.array_equal(np.roll(out0, (dy, dx), axis=(3, 4)).view(np.uint32), out.view(np.uint32)), plan
    return out, plan


@pytest.mark.parametrize("shift", [0, 1, 2])
@pytest.mark.parametrize("shape,name,level,dtype", [((1, 2, 70, 518), "haar", 1, np.uint8), ((1, 1, 66, 94), "db4", 1, np.uint8),
                                                     ((2, 1, 40, 36), "db2", 2, np.float32), ((1, 1, 72, 88), "sym4", 3, np.uint8),
                                                     ((1, 1, 64, 80), "haar", 3, np.float32), ((1, 2, 48, 36), "bior4.4", 2, np.uint8),
                                                     ((1, 1, 8, 8), "db4", 3, np.float32), ((1, 1, 130, 518), "db2", 1, np.uint8)])
def test_swt_pass_forms_agree(sim, shift, shape, name, level, dtype):
    """Every pass form the planner picks (two-pass, sliding last pass, hybrid: test_swt_plan_picks_the_form_of_filter_and_level)
    on the image rolled by (shift, shift): same sub-bands as the oracle, including x / y wrap, W % 4 = 2 and tiny images."""
    rng = np.random.default_rng(sum(shape) + level)
    x = rng.integers(0, 256, shape).astype(np.uint8) if dtype == np.uint8 else rng.random(shape, dtype=np.float32)
    _swt_rolled(sim, x, name, level, shift, shift)


@pytest.mark.parametrize("dx", [0, 1])
@pytest.mark.parametrize("dy", [0, 2])
@pytest.mark.parametrize("shape,name,level,dtype", [((1, 2, 70, 518), "haar", 1, np.uint8), ((1, 1, 66, 94), "db4", 1, np.uint8),
                                                     ((2, 1, 40, 36), "db2", 2, np.float32), ((1, 1, 72, 88), "sym4", 3, np.uint8),
                                                     ((1, 2, 48, 36), "bior4.4", 2, np.uint8), ((1, 1, 8, 8), "db4", 3, np.float32),
                                                     ((1, 1, 130, 518), "sym4", 1, np.uint8)])
def test_swt_sliding_last_pass_agrees(sim, dx, dy, shape, name, level, dtype):
    """The last vertical pass: sliding (register window of F rows, one band per unit) for 8-tap filters at level 1,
    blocked (R + F - 1 rows per R outputs, both bands of a half per unit) otherwise — same sub-bands on the image rolled by
    (dy, dx), for tiles that overhang the image bottom, W % 4 = 2 rows and images smaller than one tile."""
    rng = np.random.default_rng(sum(shape) + level)
    x = rng.integers(0, 256, shape).astype(np.uint8) if dtype == np.uint8 else rng.random(shape, dtype=np.float32)
    _swt_rolled(sim, x, name, level, dy, dx)


@pytest.mark.parametrize("dx", [0, 1])
@pytest.mark.parametrize("shape,name,level", [((1, 2, 70, 518), "haar", 1), ((1, 1, 66, 94), "db4", 1), ((2, 1, 40, 36), "db2", 2),
                                              ((1, 1, 24, 10), "haar", 1), ((1, 2, 70, 518), "db2", 1), ((2, 1, 40, 10), "db2", 1)])
def test_swt_uint8_staging_units_agree(sim, dx, shape, name, level):
    """uint8 staging on rows that start on every byte alignment (the image rolled by dx), with x/y wrap, narrow images and
    the short last unit of a row.  Where both staging forms apply (level 1, F <= 4) they give identical bits: x (W % 4 = 2)
    is staged in 8-pixel units of three aligned words, [x, x] side by side (W % 4 = 0) in the 4-pixel units shared with
    float32, and the periodic transform of [x, x] is [swt(x), swt(x)]."""
    x = np.random.default_rng(len(name) + shape[3]).integers(0, 256, shape).astype(np.uint8)
    out, plan = _swt_rolled(sim, x, name, level, 0, dx)
    lo, hi = filters.filter_bank(name)
    if level == 1 and len(lo) <= 4:
        xr = np.roll(x, dx, axis=3)
        rc, out2, plan2 = sim_swt(sim, np.concatenate([xr, xr], axis=-1), lo, hi, 1)
        assert rc == 0 and plan[7] == 1 and plan2[7] == 0, (plan, plan2)
        assert np.array_equal(out2.view(np.uint32), np.concatenate([out, out], axis=-1).view(np.uint32))


@pytest.mark.parametrize("sms", [1, 16, 148, 1000])
def test_swt_planner_variants_agree(sim, sms):
    """Different SM counts make the planner pick different tiles; the result must not change."""
    x = np.random.default_rng(7).integers(0, 256, (1, 2, 56, 88)).astype(np.uint8)
    lo, hi = filters.filter_bank("db2")
    ref = c_oracle.swt2(x, lo, hi, 2)
    rc, out, plan = sim_swt(sim, x, lo, hi, 2, sms)
    assert rc == 0 and np.abs(out - ref).max() <= 1e-5 * np.abs(ref).max(), plan


def test_u8_conversion_is_bit_identical_to_division(sim):
    """custom_transforms.py:147 divides by 255.0 in float32; the kernels use a 2-instruction FMA form instead."""
    import ctypes

    sim.sim_u8_unit.restype = ctypes.c_float
    got = np.array([sim.sim_u8_unit(ctypes.c_uint(b)) for b in range(256)], dtype=np.float32)
    assert np.array_equal(got.view(np.uint32), (np.arange(256, dtype=np.float32) / np.float32(255.0)).view(np.uint32))


def test_swt_rejects_bad_arguments(sim):
    x = np.zeros((1, 1, 6, 8), np.uint8)
    lo, hi = filters.filter_bank("haar")
    assert sim_swt(sim, x, lo, hi, 2)[0] != 0                    # 6 % 4 != 0
    assert sim_swt(sim, x, lo[:1], hi[:1], 1)[0] != 0            # odd filter length


MAP_CASES = [
    # Q, N, bits, labels (-1: 1-D integer labels), k
    (37, 500, 64, 24, 50),
    (37, 500, 64, 24, None),
    (20, 3000, 32, 20, 700),
    (20, 3000, 128, 80, 3000),
    (9, 2000, 96, 130, 100),
    (16, 70000, 64, 24, 66000),      # wide counters (k > 65534)
    (16, 70000, 64, 24, 5000),       # narrow counters, many segments
    (5, 1, 64, 8, 1),
    (5, 2, 64, 8, 5),
    (33, 1000, 200, 200, None),      # 4 code words, 4 label words
    (40, 5000, 48, -1, 300),         # equality labels
    (3, 777, 17, 3, 10),             # odd everything
    (7, 1029, 256, 12, 64),          # B = 256: distances need 9 bits, never stashed
    (6, 333, 254, 5, None),          # largest stashable code width, partial last groups (333 % 32, 333 % 4)
]


@pytest.mark.parametrize("nq,n,bits,nlab,k", MAP_CASES)
@pytest.mark.parametrize("shards,ext,sms,stash", [(1, 0, 148, 1), (1, 1, 148, 0), (3, 0, 148, 1), (8, 0, 4, 1), (2, 0, 148, 0)])
def test_hamming_map_stage_programs(sim, monkeypatch, nq, n, bits, nlab, k, shards, ext, sms, stash):
    """stash = 1: stage B ranks from the (distance, relevance) stash stage A wrote; 0: stage B scores again."""
    monkeypatch.setenv("B200_MAP_STASH", str(stash))
    rng = np.random.default_rng(nq * 1000 + n + bits)
    q, r = pm1(rng, nq, bits), pm1(rng, n, bits)
    if n > nq:
        r[:nq] = q
        r[:nq, :3] *= -1                                 # near-duplicates: short distances exist
    if nlab > 0:
        ql, rl = multi_hot(rng, nq, nlab, 0.1), multi_hot(rng, n, nlab, 0.1)
    else:
        ql, rl = rng.integers(0, 6, nq), rng.integers(0, 6, n)
    m0, ap0, ts0, rank0, dist0 = eval_ref.maphashing_exact(q, ql, r, rl, k, return_details=True)
    m, ap, ts, ri, rd, plan = sim_map(sim, q, ql, r, rl, k, shards, ext, sms, want_rank=True)
    assert plan[3] // 2 == (stash if bits <= 254 else 0), plan                 # the mode under test is the one that ran
    assert np.array_equal(ts.astype(np.int64), ts0), plan                      # hits in the top-k: bit-exact
    assert np.array_equal(ri.astype(np.int64), rank0), plan                    # ranked indices: bit-exact
    assert np.array_equal(rd.astype(np.int64), dist0), plan                    # distances: bit-exact
    assert np.abs(ap - ap0).max() <= 1e-6 and abs(m - m0) <= 1e-6              # AP: fp32 quotients, fp64 sums


@pytest.mark.parametrize("tpq", ["1", "2", "3", "4"])
@pytest.mark.parametrize("nq,n,bits,nlab,k,stash", [(37, 500, 64, 24, 50, 1), (6, 333, 254, 5, None, 0), (20, 3000, 128, 80, 700, 1),
                                                    (3, 777, 17, 3, 10, 1)])
def test_stage_a_threads_per_query(sim, monkeypatch, tpq, nq, n, bits, nlab, k, stash):
    """Stage A with 1-4 threads per query (B200_MAP_TPQ): the threads of a query take alternate 32-row groups of every
    tile — including the partial last group, which exactly one of them owns — and share one counter column."""
    monkeypatch.setenv("B200_MAP_TPQ", tpq)
    monkeypatch.setenv("B200_MAP_STASH", str(stash))
    rng = np.random.default_rng(nq + n + bits)
    q, r = pm1(rng, nq, bits), pm1(rng, n, bits)
    ql, rl = multi_hot(rng, nq, nlab, 0.1), multi_hot(rng, n, nlab, 0.1)
    m0, ap0, ts0, rank0, dist0 = eval_ref.maphashing_exact(q, ql, r, rl, k, return_details=True)
    m, ap, ts, ri, rd, plan = sim_map(sim, q, ql, r, rl, k, 1, 0, 148, want_rank=True)
    assert np.array_equal(ts.astype(np.int64), ts0) and np.array_equal(ri.astype(np.int64), rank0), plan
    assert np.array_equal(rd.astype(np.int64), dist0) and np.abs(ap - ap0).max() <= 1e-6 and abs(m - m0) <= 1e-6


def test_hamming_map_on_reference_goldens(sim, golden):
    """The stage programs against outputs of the real reference code (stable tie order)."""
    for name in golden["cases"]:
        q, r, ql, rl = (golden[f"{name}/{k}"] for k in ("q", "r", "ql", "rl"))
        tk, inc = (int(v) for v in golden[f"{name}/topk"])
        topk = None if tk == -1 else ("max_bin_count" if tk == -2 else tk)
        topk = eval_ref.resolve_topk_ref(topk, rl, bool(inc))
        m, *_ = sim_map(sim, q.astype(np.float32), ql, r.astype(np.float32), rl, topk, 2, 0, 8)
        assert abs(m - float(golden[f"{name}/map_reference_stable"])) <= 1e-6, name


def test_hamming_map_constant_codes_closed_form(sim):
    """MAP-1: one code for everybody => ranking is the index order; AP follows from the labels alone."""
    rng = np.random.default_rng(11)
    ql, rl = multi_hot(rng, 12, 20, 0.15), multi_hot(rng, 150, 20, 0.15)
    q, r = np.ones((12, 64), np.float32), np.ones((150, 64), np.float32)
    m, ap, ts, ri, rd, _ = sim_map(sim, q, ql, r, rl, 40, want_rank=True)
    assert np.array_equal(ri, np.tile(np.arange(40, dtype=np.uint32), (12, 1))) and (rd == 0).all()
    for i in range(12):
        rel = (ql[i] @ rl[:40].T) > 0
        assert abs(ap[i] - eval_ref.ap_from_ranked_relevance(rel)[0]) <= 1e-6


def test_hamming_map_correlated_codes_are_informative(sim):
    rng = np.random.default_rng(12)
    rl = multi_hot(rng, 2000, 24, 0.1)
    ql = multi_hot(rng, 30, 24, 0.1)
    q, r = correlated_codes(rng, ql, rl, 64)
    m, ap, ts, *_ = sim_map(sim, q, ql, r, rl, 500)
    density = ((ql @ rl.T) > 0).mean()
    assert m > density + 0.1
    assert abs(m - eval_ref.maphashing_exact(q, ql, r, rl, 500)) <= 1e-6


def test_wide_plan_keeps_segments_within_16_bit_counters(sim):
    """k > 65534 (wide plan) on a database whose rows all share one code: every row of a segment lands in ONE
    (segment, distance) bucket, so a segment longer than 65534 rows would wrap the 16|16-bit shared counters of stage A
    and of the all-rows stage B.  The planner must cap the segment length in wide mode too."""
    rng = np.random.default_rng(5)
    nq, n, bits = 32, 150000, 64
    ql, rl = multi_hot(rng, nq, 10, 0.2), multi_hot(rng, n, 10, 0.2)
    q, r = np.ones((nq, bits), np.float32), np.ones((n, bits), np.float32)
    m, ap, ts, _, _, plan = sim_map(sim, q, ql, r, rl, None, 1, 0, 1)          # one SM: the planner wants ONE long segment
    assert plan[3] % 2 == 1 and plan[2] <= 65534, plan                         # wide, yet capped
    for i in (0, 7, 31):
        rel = (ql[i] @ rl.T) > 0
        want, hits = eval_ref.ap_from_ranked_relevance(rel)
        assert int(ts[i]) == hits and abs(ap[i] - want) <= 1e-6, (i, plan)
