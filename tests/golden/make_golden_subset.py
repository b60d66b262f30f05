#!/usr/bin/env python
"""Generate ``tests/golden/subset_golden.npz``: the image indices ``build_fast_eval_subset`` (the reference's
``main/engine/batch_map.py:39-91``) selects from the seeded fake dataset of ``tests/test_host_logic.py``.

The reference's own function is recorded when its tree is readable (``REFERENCE_ROOT``, see ``oracle/ref_loader.py``);
otherwise the package's mirror is, which ``test_build_fast_eval_subset_mirror`` has checked against the reference's
function whenever that tree was readable.  The file's ``source`` entry says which one produced it.

    python tests/golden/make_golden_subset.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "subset_golden.npz")
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

CASES = ((64, 3), (17, 0), (10 ** 6, 9))            # (size, seed)


def subset_fn():
    from oracle import ref_loader

    if ref_loader.available():
        import importlib.util

        ref_loader.load_reference()
        for mod in ("make_subset", "batch_map"):
            spec = importlib.util.spec_from_file_location(f"main.engine.{mod}", os.path.join(ref_loader.REF, f"main/engine/{mod}.py"))
            m = importlib.util.module_from_spec(spec)
            sys.modules[f"main.engine.{mod}"] = m
            spec.loader.exec_module(m)
        return m.build_fast_eval_subset, "reference main/engine/batch_map.py"
    from image_retrieval_wavelet_b200.engine import build_fast_eval_subset

    return build_fast_eval_subset, "image_retrieval_wavelet_b200.engine.build_fast_eval_subset"


def main():
    from test_host_logic import _FakeDataset

    fn, source = subset_fn()
    ds = _FakeDataset(300, 12, 1)
    ds.instance_dict[99] = [5]
    out = {"source": np.array(source)}
    for size, seed in CASES:
        paths = fn(ds, size, seed=seed).paths
        out[f"size{size}_seed{seed}"] = np.array([ds.paths.index(p) for p in paths], dtype=np.int32)
    np.savez_compressed(OUT, **out)
    print(f"wrote {OUT} ({os.path.getsize(OUT)} bytes) from {source}")


if __name__ == "__main__":
    main()
