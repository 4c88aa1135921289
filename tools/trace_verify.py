"""Per-stage device timeline (option "trace") of verify calls over 2^22 signatures: independent batches of 256, device-resident
and from pinned host buffers (pieces streamed over PCIe), for 1..8 pieces.  Run on the B200; the timeline goes to stderr."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
torch.set_num_threads(1)            # pinned buffers first-touched by one thread (NUMA-local): 55 instead of 35 GB/s over PCIe
import curve25519_dalek_b200 as pkg
import bench
eng = pkg.Engine(0)
n = 1 << 22
flat, offs, sigs, pks = bench.build_verify_inputs(eng, n)
dev = torch.device("cuda", 0)
h = [torch.from_numpy(x if x.dtype == np.uint8 else x.view(np.int64)).pin_memory() for x in (flat, offs, sigs, pks)]
d = [x.to(dev) for x in h]


def call(bufs, host):
    rc, v = eng.verify_batches_flat(bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr(), bufs[3].data_ptr(), n, 256, device_ptrs=not host)
    assert rc == 0


for _ in range(3):
    call(d, False)
print("== device-resident, batches of 256", file=sys.stderr, flush=True)
eng.set_option("trace", 1); call(d, False); eng.set_option("trace", 0)
for pieces in (1, 2, 4, 8):
    eng.set_option("verify_pieces", pieces)
    for _ in range(2):
        call(h, True)
    import time
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(5):
        call(h, True)
    torch.cuda.synchronize()
    print("== host buffers, verify_pieces = %d: %.2f ms per call" % (pieces, (time.perf_counter() - t0) / 5 * 1e3), file=sys.stderr, flush=True)
    eng.set_option("trace", 1); call(h, True); eng.set_option("trace", 0)
eng.set_option("verify_pieces", 4)
