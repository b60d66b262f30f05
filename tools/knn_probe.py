"""Times b200_knn_topk on the BASELINE configs[2] cosine shape at k = 2048 (fused path) and k = 5000 (score matrix, two
select passes) and prints a hash of the index and score bytes.  A/B of two builds: run it once per library with
B200RET_LIB=<path to libb200ret.so>.  python tools/knn_probe.py [reps]"""
import hashlib
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from image_retrieval_wavelet_b200.engine.get_knn import knn_topk

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
g = torch.Generator().manual_seed(0)
refs = torch.nn.functional.normalize(torch.randn(117000, 768, generator=g), dim=1).cuda()
qs = torch.nn.functional.normalize(torch.randn(5000, 768, generator=g), dim=1).cuda()
flush = bench.l2_flusher(torch.device("cuda"))
for k in (2048, 5000):
    knn_topk(refs, qs, k, "cosine")
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        sc, idx = knn_topk(refs, qs, k, "cosine")
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    h = hashlib.sha256(idx.cpu().numpy().tobytes() + sc.cpu().numpy().tobytes()).hexdigest()[:16]
    print(f"knn 5000x117000x768 k={k}: min {min(ts):.3f} ms mean {sum(ts)/len(ts):.3f} ms  hash {h}", flush=True)
