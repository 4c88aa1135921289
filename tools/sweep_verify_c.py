import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import curve25519_dalek_b200 as pkg
import bench
eng = pkg.Engine(0)
n = 1 << 22
flat, offs, sigs, pks = bench.build_verify_inputs(eng, n)
dev = torch.device("cuda", 0)
d = [torch.from_numpy(x if x.dtype == np.uint8 else x.view(np.int64)).to(dev) for x in (flat, offs, sigs, pks)]
for c in (0, 16, 17, 18, 19, 20, 0, 17):
    eng.set_option("window_bits", c)
    for _ in range(2):
        assert eng.verify_batch_flat(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), n, device_ptrs=True) == 0
    torch.cuda.synchronize(); t0 = time.perf_counter()
    acc = []
    for _ in range(5):
        eng.verify_batch_flat(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), n, device_ptrs=True)
        acc.append(eng.last_kernel_ms()[0])
    torch.cuda.synchronize()
    print("window_bits=%d verify ms/step %.2f acc_ms %s" % (c, (time.perf_counter() - t0) / 5 * 1e3, " ".join("%.2f" % a for a in acc)), flush=True)
eng.set_option("window_bits", 0)
wl = bench.MsmWorkload(eng, 1 << 20, 1 << 20, 0, torch)
for c in (14, 15, 16, 17):
    eng.set_option("window_bits", c)
    for _ in range(3): wl.step_device_single()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(20): wl.step_device_single()
    torch.cuda.synchronize()
    print("window_bits=%d msm ms/step %.3f acc_ms %.3f" % (c, (time.perf_counter() - t0) / 20 * 1e3, eng.last_kernel_ms()[0]), flush=True)
