"""SWT C1 / C4 grid (bench.py's cases): time and fraction of the HBM roofline per case.  A/B of two builds: run it once
per library with B200RET_LIB=<path to libb200ret.so>.  python tools/swt_probe.py [steps] [filter substring]"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
only = sys.argv[2] if len(sys.argv) > 2 else ""
args = argparse.Namespace(steps=steps, warmup=3)
dev = torch.device("cuda")
cases = [((64, 3, 224, 224), "haar", 1, "u8"), ((64, 3, 224, 224), "haar", 1, "f32")]
for lv in (1, 2, 3):
    for wv in ("haar", "db2", "db4", "sym4"):
        cases.append(((256, 3, 518, 518) if lv == 1 else (256, 3, 520, 520), wv, lv, "u8"))
cases.append(((256, 3, 518, 518), "bior4.4", 1, "u8"))
for shape, wv, lv, dt in cases:
    tag = f"{wv} L{lv} {shape[2]} {dt}"
    if only and only not in tag:
        continue
    r = bench.bench_swt(shape, wv, lv, dt, args, dev)
    print(f"{tag:24s} {r['ms']*1e3:9.1f} us  frac {r['roofline']['frac']:.3f}", flush=True)
