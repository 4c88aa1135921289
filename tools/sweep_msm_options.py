import os, sys, time, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import curve25519_dalek_b200 as pkg
import bench
eng = pkg.Engine(0)
wl = bench.MsmWorkload(eng, 1 << 20, 1 << 20, 0, torch)
def run(tag, steps=20):
    for _ in range(3): wl.step_device_single()
    torch.cuda.synchronize(); t0 = time.perf_counter(); km = []
    for _ in range(steps):
        wl.step_device_single(); km.append(eng.last_kernel_ms()[0])
    torch.cuda.synchronize(); dt = (time.perf_counter() - t0) / steps
    print(tag, "ms/step %.3f" % (dt * 1e3), "acc_ms %.3f" % (sum(km) / len(km)), flush=True)
def run_host(tag, steps=10):
    for _ in range(2): wl.step_host_single()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(steps): wl.step_host_single()
    torch.cuda.synchronize(); print(tag, "e2e ms/step %.3f" % ((time.perf_counter() - t0) / steps * 1e3), flush=True)
for f in (1, 0):
    eng.set_option("field_f64", f)
    run("f64=%d" % f)
eng.set_option("field_f64", 1)
for k in (1, 2, 4, 8):
    eng.set_option("host_chunks", k)
    run_host("host_chunks=%d" % k)
