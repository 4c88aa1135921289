"""Precomputed MSM over 2^20 resident points: window tables on/off x scalar chunks, wall / device / accumulate ms."""
import os, sys, time, ctypes as C
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import curve25519_dalek_b200 as pkg
import bench
eng = pkg.Engine(0)
wl = bench.MsmWorkload(eng, 1 << 20, 1 << 20, 0, torch)
out = (C.c_uint8 * 32)()
for tables in (1, 0):
    eng.set_option("precomp_tables", tables)
    pre = C.c_void_p()
    t0 = time.perf_counter()
    assert eng.lib.dalek_b200_precomp_new(eng.h, wl.h_points.data_ptr(), 1, wl.n, C.byref(pre)) == 0
    print("tables=%d construction %.1f ms" % (tables, (time.perf_counter() - t0) * 1e3), flush=True)
    for chunks in (1, 2, 4):
        eng.set_option("host_chunks", chunks)
        for _ in range(3):
            assert eng.lib.dalek_b200_precomp_mixed_msm(eng.h, pre, wl.h_scalars.data_ptr(), wl.n, None, None, 1, 0, C.addressof(out), None) == 0
        t0 = time.perf_counter(); dev = []; acc = []
        for _ in range(10):
            eng.lib.dalek_b200_precomp_mixed_msm(eng.h, pre, wl.h_scalars.data_ptr(), wl.n, None, None, 1, 0, C.addressof(out), None)
            dev.append(eng.last_call_ms()); acc.append(eng.last_kernel_ms()[0])
        print("tables=%d chunks=%d wall %.3f ms  device %.3f ms  accumulate span %.3f ms" %
              (tables, chunks, (time.perf_counter() - t0) / 10 * 1e3, sum(dev) / 10, sum(acc) / 10), flush=True)
    eng.lib.dalek_b200_precomp_destroy(pre)
