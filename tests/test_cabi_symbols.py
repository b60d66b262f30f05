"""The C-ABI library loads and exports every symbol that include/b200ret.h declares; the ctypes table mirrors the header.
No compute call is made here (there is no GPU in the build container)."""
import ctypes
import os
import re

from image_retrieval_wavelet_b200 import _cabi, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "b200ret.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", text))
    inline = set(re.findall(r"static inline \w+ (b200_[a-z0-9_]+)\s*\(", text))
    return names - inline


def test_library_exports_every_declared_symbol():
    lib_path = build.build_lib()
    lib = ctypes.CDLL(lib_path)
    declared = _declared()
    assert len(declared) >= 25
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/b200ret.h but not exported"


def test_ctypes_table_matches_header():
    assert set(_cabi.SIGNATURES) == _declared()


def test_error_strings_and_version_need_no_device():
    lib = _cabi.load()
    assert lib.b200_version() >= 100
    assert lib.b200_error_string(0) == b"ok"
    assert b"unsupported" in lib.b200_error_string(_cabi.ERR_UNSUPPORTED)
    assert lib.b200_launch_count() == 0 or lib.b200_launch_count() > 0


def test_argument_validation_happens_before_any_cuda_call():
    """Invalid arguments are rejected on the host side, so these calls are safe without a device."""
    lib = _cabi.load()
    plan = _cabi.MapPlan()
    assert lib.b200_map_plan_init(ctypes.byref(plan), 0, 10, 10, 64, 1, 0, 5) == _cabi.ERR_INVALID_ARG        # Q = 0
    assert lib.b200_map_plan_init(ctypes.byref(plan), 4, 10, 10, 300, 1, 0, 5) == _cabi.ERR_UNSUPPORTED       # B > 256
    assert lib.b200_map_plan_init(ctypes.byref(plan), 4, 10, 10, 64, 3, 0, 5) == _cabi.ERR_UNSUPPORTED        # LW = 3
    assert lib.b200_swt2_fwd(None, 1, None, 1, 3, 8, 8, None, None, 2, 1, None) == _cabi.ERR_INVALID_ARG
    assert lib.b200_pack_codes(None, 5, 64, None, None, None) == _cabi.ERR_INVALID_ARG
    assert lib.b200_pack_codes(None, 0, 64, None, None, None) == _cabi.OK                                      # empty is fine
    assert lib.b200_knn_workspace_bytes(0, 10, 8, 1) == 0


def test_plan_struct_layout_matches_the_library():
    lib = _cabi.load()
    plan = _cabi.MapPlan()
    assert lib.b200_map_plan_init(ctypes.byref(plan), 5000, 117000, 117000, 128, 2, 0, 5000) == 0
    assert (plan.Q, plan.N, plan.B, plan.LW, plan.k, plan.bins) == (5000, 117000, 128, 2, 5000, 129)
    assert plan.wide == 0 and plan.T in (32, 64, 128) and plan.Qpad % 32 == 0 and plan.Qpad >= 5000
    assert plan.S * plan.seg_len >= 117000 and plan.seg_len % 2 == 0 and plan.seg_len <= 65534
    assert plan.off_hist < plan.off_tot < plan.off_dstar < plan.off_psum < plan.off_phits < plan.workspace_bytes
    assert lib.b200_map_plan_init(ctypes.byref(plan), 10000, 1000000, 1000000, 64, 2, 0, 1000000) == 0
    assert plan.wide == 1 and plan.k == 1000000


def test_select_planner_rules_for_query_slices():
    """hamming_plan.h (round 2): 128-query groups are kept as long as every SM can get a CTA; a GPU holding only a slice of
    the queries takes 512-row segments instead of smaller groups; every plan covers the database with whole segments whose
    row-in-segment fits 16 bits."""
    lib = _cabi.load()
    seen = {}
    for q, n, bits, lw, k in ((5000, 117000, 128, 2, 5000), (628, 117000, 128, 2, 5000), (1252, 117000, 128, 2, 5000),
                              (8, 40000, 64, 1, 600), (10000, 1000000, 64, 2, 5000), (1250, 1000000, 64, 2, 5000)):
        plan = _cabi.MapPlan()
        assert lib.b200_map_plan_init(ctypes.byref(plan), q, n, n, bits, lw, 0, k) == 0
        assert plan.select == 1
        assert plan.sel_S * plan.sel_seg_len >= n > (plan.sel_S - 1) * plan.sel_seg_len
        assert plan.sel_seg_len % 64 == 0 and 512 <= plan.sel_seg_len <= 65472 and plan.sel_S <= 65535
        assert plan.sel_T in (32, 64, 128) and plan.sel_T <= plan.T and plan.Qpad % plan.sel_T == 0
        assert plan.smp_rows % 32 == 0 and plan.smp_rows * plan.sel_stride >= 32 * (n // 32)
        seen[(q, n)] = (plan.sel_T, plan.sel_seg_len)
    assert seen[(5000, 117000)][0] == 128 and seen[(5000, 117000)][1] >= 1024
    assert seen[(628, 117000)] == (128, 512)                    # a slice of an 8-GPU run: full groups, short segments
    assert seen[(1252, 117000)] == (128, 1024)
    assert seen[(1250, 1000000)][0] == 128
    assert seen[(8, 40000)][0] == 32                            # too few queries for one CTA per SM: the groups shrink


def _plan_for(q, n, bits, lw, k):
    plan = _cabi.MapPlan()
    assert _cabi.load().b200_map_plan_init(ctypes.byref(plan), q, n, n, bits, lw, 0, k) == 0
    return plan


def test_plan_decides_the_tensor_core_form(monkeypatch):
    """hamming_plan.h: the tensor-core form of the select pass gets its workspace (e4m3 copies + hit masks, off_smp_codes <
    workspace_bytes) and 256-row tiles when the queries come in groups of 128 and the masks stay below 4 GB; small query
    sets and huge databases keep the SIMT kernel (off_smp_codes == workspace_bytes).  Every plan with that workspace has
    the geometry the tensor-core kernels are written for."""
    monkeypatch.delenv("B200_MAP_SELECT", raising=False)
    monkeypatch.delenv("B200_SEL_STRIDE", raising=False)
    p = _plan_for(5000, 117000, 128, 2, 5000)
    assert p.select == 1 and p.off_smp_codes < p.workspace_bytes and p.sel_seg_len % 256 == 0 and p.sel_T == 128
    masks = (117000 + 255) // 256 * 8 * p.Qpad * 4
    assert p.workspace_bytes - p.off_smp_codes >= 117000 * 128 + p.Qpad * 128 + masks
    p64 = _plan_for(10000, 1000000, 64, 2, 5000)                    # 64-bit codes are padded to one 128-byte K block
    assert p64.off_smp_codes < p64.workspace_bytes and p64.workspace_bytes - p64.off_smp_codes >= 1000000 * 128
    small = _plan_for(40, 70001, 64, 1, 5000)                       # fewer than 128 queries: SIMT kernel
    assert small.select == 1 and small.off_smp_codes == small.workspace_bytes
    huge = _plan_for(10000, 50000000, 64, 2, 5000)                  # the hit masks would take 63 GB: SIMT kernel
    assert huge.select == 1 and huge.off_smp_codes == huge.workspace_bytes
    tc = 0
    for q in (40, 64, 128, 130, 256, 300, 628, 1252, 5000, 10000):
        for n in (40000, 70001, 117000, 1000000, 50000000):
            for bits in (64, 128, 200):
                for k in (600, 5000):
                    pl = _plan_for(q, n, bits, 2, k)
                    if pl.select and pl.off_smp_codes != pl.workspace_bytes:
                        tc += 1
                        assert pl.sel_T == 128 and pl.Qpad % 128 == 0, (q, n, bits, k)
                        assert pl.sel_seg_len % 256 == 0 and pl.sel_seg_len <= 65280, (q, n, bits, k)
    assert tc >= 100


def test_plan_ignores_former_tuning_overrides(monkeypatch):
    """Only B200_MAP_SELECT, B200_SEL_STRIDE and B200_MAP_STASH reach the planner: the select geometry, the tensor-core
    form and the stash budget it once let the environment override are set to values that would change every plan
    below, and the plans stay the same field for field."""
    for name in ("B200_MAP_SELECT", "B200_SEL_STRIDE", "B200_MAP_STASH"):
        monkeypatch.delenv(name, raising=False)
    shapes = ((5000, 117000, 128, 2, 5000), (628, 117000, 128, 2, 5000), (40, 70001, 64, 1, 5000), (10000, 1000000, 64, 2, 5000),
              (256, 40000, 128, 1, 600))
    before = [_plan_for(*s) for s in shapes]
    # B200_ + name: the select CTAs per SM, minimum segment, query group, segment counts, tensor-core switch, stash budget
    hostile = {"SEL_CTAS_PER_SM": "1", "SEL_MIN_SEG": "64", "SEL_T": "32", "SEL_SEGMENTS": "3", "SMP_SEGMENTS": "1",
               "SEL_TC": "0", "MAP_STASH_MAX_MB": "0"}
    for name, value in hostile.items():
        monkeypatch.setenv("B200_" + name, value)
    for s, p0 in zip(shapes, before):
        p1 = _plan_for(*s)
        for field, _ in _cabi.MapPlan._fields_:
            assert getattr(p1, field) == getattr(p0, field), (s, field)
