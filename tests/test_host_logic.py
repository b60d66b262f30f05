"""Host-side logic of the drop-in mirrors that needs no device: metric discovery, include/exclude handling, exclude-list
assembly, constructor contracts, and loud failure without CUDA."""
import os

import numpy as np
import pytest
import torch

from image_retrieval_wavelet_b200 import _cabi
from image_retrieval_wavelet_b200.engine import CustomCalculator, get_accuracy_calculator
from image_retrieval_wavelet_b200.engine import accuracy_calculator as ac
from image_retrieval_wavelet_b200.transforms import DWTTransform, RawStackTransform, SWTTransform

no_cuda = not torch.cuda.is_available()


def test_metric_discovery_by_prefix():
    c = CustomCalculator(k=50, distance_metric="hamming", with_faiss=False)
    m = c.get_curr_metrics()
    for name in ("maphashing", "map", "bit_balance", "worst_bit_balance", "recall_at_1", "recall_at_1000", "rpr", "pr",
                 "mean_average_precision", "r_precision", "precision_at_1"):
        assert name in m
    assert c.num_top_k == 50 and c.distance_metric == "hamming" and c.with_faiss is False
    assert "map" in c.requires_knn() and "maphashing" not in c.requires_knn() and "bit_balance" not in c.requires_knn()


def test_exclude_list_assembly_matches_reference():
    """accuracy_calculator.py:373-394: caller excludes are merged with the base list and are effective."""
    c = get_accuracy_calculator(k=19581, exclude=["map", "rpr"])
    active = set(c.get_curr_metrics())
    assert "map" not in active and "rpr" not in active and "NMI" not in active and "pr_rc_hashing" not in active
    assert "recall_at_1" not in active and "mean_reciprocal_rank" not in active
    assert {"maphashing", "bit_balance", "worst_bit_balance"} <= active
    c2 = get_accuracy_calculator(k=5, with_AP=False, exclude_ranks=[100])
    assert "mean_average_precision" not in c2.get_curr_metrics()


def test_unknown_metric_names_are_rejected():
    with pytest.raises(ValueError):
        CustomCalculator(exclude=["recall_classic"])          # evaluate.py:46-52 documents exactly this
    with pytest.raises(ValueError):
        CustomCalculator(k=-3)
    with pytest.raises(TypeError):
        CustomCalculator(exclude="map")


def test_include_filters_current_metrics():
    c = CustomCalculator(k="max_bin_count")
    assert list(c.get_function_dict(include=["maphashing"]).keys()) == ["maphashing"]
    assert "maphashing" not in c.get_function_dict(exclude=["maphashing"])


def test_determine_k():
    c = CustomCalculator(k=None)
    assert c.determine_k(torch.tensor([3, 9]), 100, True) == 99
    assert CustomCalculator(k="max_bin_count").determine_k(torch.tensor([3, 9]), 100, True) == 8
    assert CustomCalculator(k=7).determine_k(torch.tensor([3, 9]), 100, False) == 7


def test_label_match_helpers_on_cpu_tensors():
    ql = torch.tensor([0, 1, 1, 2])
    rl = torch.tensor([1, 1, 1, 0, 3])
    uniq, counts = ac.get_label_match_counts(ql, rl, torch.eq)
    assert uniq.tolist() == [0, 1, 2] and counts.tolist() == [1, 3, 0]
    lone, mask = ac.get_lone_query_labels(ql, (uniq, counts), False, torch.eq)
    assert lone.tolist() == [2] and mask.tolist() == [True, True, True, False]
    lone, mask = ac.get_lone_query_labels(ql, (uniq, counts), True, torch.eq)
    assert lone.tolist() == [0, 2]


def test_transform_constructors_and_repr():
    t = SWTTransform(level=2, wavelet="db4")
    assert repr(t) == "SWTTransform(shape='C,S,H,W', wavelet=db4, level=2)"
    assert repr(RawStackTransform(copies=4)) == "RawStackTransform(shape='C,4,H,W', copies=4)"
    assert (t.level, t.wavelet) == (2, "db4")
    d = DWTTransform(level=3, wavelet="haar")
    assert repr(d) == "DWTTransform(shape='C,S,H/8,W/8', wavelet=haar, level=3)" and (d.level, d.wavelet) == (3, "haar")


def test_fix_size_matches_reference():
    from PIL import Image

    t = SWTTransform(level=3)
    assert t.fix_size(Image.new("RGB", (518, 518))).size == (520, 520)
    assert t.fix_size(Image.new("RGB", (224, 224))).size == (224, 224)
    assert SWTTransform(level=1).fix_size(Image.new("RGB", (31, 17))).size == (32, 18)


@pytest.mark.skipif(not no_cuda, reason="checks the behaviour of a CPU-only box")
def test_no_silent_cpu_fallback():
    from PIL import Image

    with pytest.raises(_cabi.B200Error):
        SWTTransform()(Image.new("RGB", (8, 8)))
    with pytest.raises(_cabi.B200Error):
        DWTTransform()(Image.new("RGB", (8, 8)))
    from image_retrieval_wavelet_b200.engine import DSCH
    from image_retrieval_wavelet_b200.transforms import dwt2, resize_u8

    codes, labels = torch.ones(4, 8), torch.ones(4, 3)
    for fn in (lambda: DSCH.mean_average_precision(codes, codes, labels, labels, 2), lambda: DSCH.pr_curve(codes, codes, labels, labels),
               lambda: DSCH.p_topK(codes, codes, labels, labels, K=[1]), lambda: DSCH.calc_hamming_dist(codes[0], codes),
               lambda: DSCH.get_precision_recall_by_Hamming_Radius(codes.numpy(), labels.numpy(), codes.numpy(), labels.numpy()),
               lambda: resize_u8(torch.zeros(1, 8, 8, dtype=torch.uint8), (16, 16)), lambda: dwt2(torch.zeros(1, 8, 8))):
        with pytest.raises(_cabi.B200Error):
            fn()
    c = CustomCalculator(k=5)
    with pytest.raises(_cabi.B200Error):
        c.calculate_maphashing(torch.ones(2, 8), torch.ones(2, 3), torch.ones(4, 8), torch.ones(4, 3), 2)
    with pytest.raises(_cabi.B200Error):
        c.get_accuracy(np.ones((2, 8)), np.ones((2, 3)), np.ones((4, 8)), np.ones((4, 3)), False, include=["maphashing"])


def test_query_bounds_cover_every_query_once_in_16_byte_slices():
    from image_retrieval_wavelet_b200.engine.map_engine import query_bounds

    for nq in (1, 3, 5, 64, 625, 5000, 10001):
        for world in (1, 2, 3, 4, 8):
            b = query_bounds(nq, world)
            assert len(b) == world and b[0][0] == 0 and b[-1][1] == nq
            assert all(x[1] == y[0] for x, y in zip(b[:-1], b[1:]))          # contiguous, in order, possibly empty at the end
            assert all(x[0] % 4 == 0 for x in b if x[1] > x[0])              # non-empty hit-count slices start on 16-byte boundaries


class _FakeDataset:
    """The slice of the reference's dataset interface build_fast_eval_subset / make_subset touch."""

    def __init__(self, n, n_tags, seed):
        import random

        rng = random.Random(seed)
        self.paths = [f"img{i}.jpg" for i in range(n)]
        self.labels = [sorted(rng.sample(range(n_tags), rng.randint(1, 3))) for _ in range(n)]
        self.super_labels = None
        self._at_R = 17
        self.get_instance_dict()

    def get_instance_dict(self):
        self.instance_dict = {}
        for i, tags in enumerate(self.labels):
            for t in tags:
                self.instance_dict.setdefault(t, []).append(i)

    def get_super_dict(self):
        pass

    def __len__(self):
        return len(self.paths)


def test_build_fast_eval_subset_mirror():
    """batch_map.py:39-91: deterministic, de-duplicated, at most `size` images, groups below min_per_class skipped; against
    the recorded selections of tests/golden/subset_golden.npz, and against the reference's own function when its tree is
    readable."""
    from image_retrieval_wavelet_b200.engine import build_fast_eval_subset

    ds = _FakeDataset(300, 12, 1)
    ds.instance_dict[99] = [5]                          # a singleton group: never eligible
    a, b = build_fast_eval_subset(ds, 64, seed=3), build_fast_eval_subset(ds, 64, seed=3)
    assert a.paths == b.paths and len(a.paths) == 64 and len(set(a.paths)) == 64 and not hasattr(a, "_at_R")
    assert build_fast_eval_subset(ds, 64, seed=4).paths != a.paths
    assert len(build_fast_eval_subset(ds, 10 ** 6).paths) == 300
    with pytest.raises(ValueError):
        build_fast_eval_subset(ds, 8, min_per_class=10 ** 6)
    with pytest.raises(AttributeError):
        build_fast_eval_subset(object(), 8)
    want = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "subset_golden.npz"))
    for size, seed in ((64, 3), (17, 0), (10 ** 6, 9)):
        got = [ds.paths.index(p) for p in build_fast_eval_subset(ds, size, seed=seed).paths]
        assert got == want[f"size{size}_seed{seed}"].tolist(), (size, seed)
    from oracle import ref_loader

    if ref_loader.available():
        import importlib.util
        import sys
        import types

        ref_loader.load_reference()                     # stubs + main.engine.accuracy_calculator
        spec = importlib.util.spec_from_file_location("main.engine.make_subset", os.path.join(ref_loader.REF, "main/engine/make_subset.py"))
        ms = importlib.util.module_from_spec(spec)
        sys.modules["main.engine.make_subset"] = ms
        spec.loader.exec_module(ms)
        spec = importlib.util.spec_from_file_location("main.engine.batch_map", os.path.join(ref_loader.REF, "main/engine/batch_map.py"))
        bm = importlib.util.module_from_spec(spec)
        sys.modules["main.engine.batch_map"] = bm
        spec.loader.exec_module(bm)
        assert isinstance(bm, types.ModuleType)
        for size, seed in ((64, 3), (17, 0), (10 ** 6, 9)):
            assert bm.build_fast_eval_subset(ds, size, seed=seed).paths == build_fast_eval_subset(ds, size, seed=seed).paths


def test_nvtx_range_is_a_harmless_context_manager(monkeypatch):
    """The NVTX ranges around the host-side phases (SURVEY 5 tracing) must never change control flow: usable without a
    GPU, nestable, exceptions pass through, B200_NVTX=0 makes them no-ops."""
    from image_retrieval_wavelet_b200 import _cabi

    with _cabi.nvtx_range("b200/test/outer"):
        with _cabi.nvtx_range("b200/test/inner") as r:
            assert r.name == "b200/test/inner"
    try:
        with _cabi.nvtx_range("b200/test/raises"):
            raise KeyError("x")
    except KeyError:
        pass
    else:
        raise AssertionError("the exception was swallowed")
    monkeypatch.setattr(_cabi.nvtx_range, "_on", False)
    with _cabi.nvtx_range("b200/test/off") as r:
        assert r.pushed is False
