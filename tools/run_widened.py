"""One pass over the widened rows (SURVEY 8f) for profiling: batch codecs on 2^20 points, per-signature verification on
2^20 signatures, precomputed MSM over 2^20 resident points."""
import os, sys, ctypes as C
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import curve25519_dalek_b200 as pkg
import bench
eng = pkg.Engine(0)
wl = bench.MsmWorkload(eng, 1 << 20, 1 << 20, 0, torch)
print(bench.run_codecs(eng, wl, steps=2))
print(bench.run_precomputed(eng, wl, steps=2))
n = 1 << 20
flat, offs, sigs, pks = bench.build_verify_inputs(eng, n)
dev = torch.device("cuda", 0)
d = [torch.from_numpy(x if x.dtype == np.uint8 else x.view(np.int64)).to(dev) for x in (flat, offs, sigs, pks)]
res = np.zeros(n, dtype=np.uint8)
for _ in range(2):
    assert eng.lib.ed25519_b200_verify_each_flat_dev(eng.h, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), n, 0, res.ctypes.data) == 0
print("verify_each device ms", eng.last_call_ms())
