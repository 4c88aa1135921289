"""verify_batch 2^22: device-resident and host-streamed ms/step for several transcript chunk sizes / piece counts."""
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
h = [torch.from_numpy(x if x.dtype == np.uint8 else x.view(np.int64)).pin_memory() for x in (flat, offs, sigs, pks)]
d = [x.to(dev) for x in h]

def run(bufs, device):
    for _ in range(2):
        assert eng.verify_batch_flat(bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr(), bufs[3].data_ptr(), n, device_ptrs=device) == 0
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(6):
        eng.verify_batch_flat(bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr(), bufs[3].data_ptr(), n, device_ptrs=device)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / 6 * 1e3

for chunk in (64,):
    eng.set_option("verify_chunk", chunk)
    print("verify_chunk=%d device %.2f ms  host(4 pieces) %.2f ms" % (chunk, run(d, True), run(h, False)), flush=True)
eng.set_option("verify_chunk", 64)
for pieces in (4, 6, 8):
    eng.set_option("verify_pieces", pieces)
    print("verify_pieces=%d host %.2f ms" % (pieces, run(h, False)), flush=True)
