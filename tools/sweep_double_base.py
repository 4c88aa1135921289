"""Time the Ristretto double-base batch (BASELINE configs[4]) through the per-pair Straus kernel (0) and the
fixed-base comb kernel (1); checksums must agree."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import curve25519_dalek_b200 as pkg
import bench
eng = pkg.Engine(0)
for variant in (0, 1, 1):
    eng.set_option("double_base_comb", variant)
    r = bench.run_double_base(eng, steps=5)
    print("variant %d: %.2f M pairs/s  call %.2f ms  kernel %.2f ms  checksum %s" %
          (variant, r["value"] / 1e6, r["ms_per_step"], r["device_span_ms"], r["checksum"]), flush=True)
