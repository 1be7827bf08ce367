"""Times dz_pdist + dz_linkage_centroid on clustered unit-norm rows (the shape of the AHC input in the pipeline bench).
usage: python scripts/linkage_time.py N [check]   (env LINK_VARIANT is the variant argument of dz_linkage_centroid_variant:
0 default, 1 first-generation loop, 2 lazy loop with its state in global memory)"""
import ctypes as C
import sys
import time

import os
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

from diarizen_b200 import _lib

N = int(sys.argv[1]) if len(sys.argv) > 1 else 8964
check = len(sys.argv) > 2
L = _lib.lib()
g = np.random.default_rng(5)
kind = os.environ.get("LINK_DATA", "hard")
variant = int(os.environ.get("LINK_VARIANT", "0"))
cent = g.standard_normal((6, 256))
noise = {"hard": 0.35, "easy": 0.05, "uniform": 10.0}[kind]
x = cent[g.integers(0, 6, N)] + noise * g.standard_normal((N, 256))
x = (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)
dev = torch.device("cuda:0")
xd = torch.from_numpy(x).to(dev)
dist = torch.empty((N, N), dtype=torch.float64, device=dev)
Z = torch.empty((N - 1, 4), dtype=torch.float64, device=dev)
ws = torch.empty(int(L.dz_linkage_workspace_bytes(N)), dtype=torch.uint8, device=dev)
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
res = []
for it in range(4):
    ev[0].record()
    _lib.check(L.dz_pdist(C.c_void_p(xd.data_ptr()), N, 256, C.c_void_p(dist.data_ptr()), st))
    ev[1].record()
    _lib.check(L.dz_linkage_centroid_variant(C.c_void_p(dist.data_ptr()), N, C.c_void_p(Z.data_ptr()), C.c_void_p(ws.data_ptr()), st,
                                             variant))
    ev[2].record()
    torch.cuda.synchronize()
    res.append((ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])))
print(kind, "N", N, "pdist ms", [round(a, 2) for a, _ in res], "linkage ms", [round(b, 2) for _, b in res],
      "us/merge", round(1e3 * min(b for _, b in res) / (N - 1), 3),
      "rescans", int(ws[24 * N:24 * N + 8].view(torch.int64).item()))
if check:
    from scipy.cluster.hierarchy import linkage
    t = time.time()
    Zr = linkage(x.astype(np.float64), method="centroid", metric="euclidean")
    print("scipy s", round(time.time() - t, 1), "bit-identical", bool((Z.cpu().numpy() == Zr).all()))
