"""Batched vartime MSM (dalek_b200_edwards_vartime_msm_batch) against the loop of single calls and the CPU oracle pool.

Workloads (m MSMs of n pairs) sit on both sides of the bucket threshold: (2^14, 16), (2^12, 64), (2^12, 256), (2^10, 1024),
(64, 2^14), (8, 2^18), and a mixed set of log-uniform lengths in 1 .. 2^16.  Points are extended limbs (t_i B from the
engine's fixed-base batch), scalars uniform below 2^253.  Each workload is timed from device-resident and from pinned
host buffers; every timed batch result is compared byte for byte with the single call on the same slice (the singles
loop runs a stated subset of the MSMs and is scaled to m).  A sweep of the option batch_bucket_min picks the default.
The GPU's name and power limit are read in the same run.

    python tools/msm_batch_bench.py --out profiles/msm_batch_r1.json
"""
import argparse
import json
import math
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SWEEP = [256, 1024, 4096, 16384, 65536, 262144, 2**31 - 1]


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip()
    except Exception as exc:                      # reported, not guessed
        info["power_limit_and_max_sm_clock"] = "unavailable: %s" % exc
    return info


def workloads(quick):
    rnd = random.Random(2026)
    mixed = [max(1, int(2 ** rnd.uniform(0, 16))) for _ in range(200)]
    w = [("m16384_n16", [16] * 16384), ("m4096_n64", [64] * 4096), ("m4096_n256", [256] * 4096), ("m1024_n1024", [1024] * 1024),
         ("m64_n16384", [16384] * 64), ("m8_n262144", [262144] * 8), ("mixed_m200_loguniform", mixed)]
    if quick:
        w = [(name, ls[:max(2, len(ls) // 64)]) for name, ls in w]
    return w


def make_inputs(eng, n, seed):
    import numpy as np
    import torch
    rng = np.random.default_rng(seed)
    sc = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    sc[:, 31] &= 0x1f                                             # below 2^253
    t = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    t[:, 31] &= 0x0f
    limbs, _ = eng.mul_base_batch(t.tobytes(), n, want_compressed=False)
    pts = np.frombuffer(limbs, dtype=np.uint64, count=20 * n).reshape(n, 20).copy()
    h_sc = torch.from_numpy(sc.reshape(-1)).pin_memory()
    h_pt = torch.from_numpy(pts.view(np.uint8).reshape(-1)).pin_memory()
    return sc, pts, h_sc, h_pt, h_sc.cuda(), h_pt.cuda()


def timed(fn, reps):
    """Median host wall time (ms) of a blocking call: it ends in a stream synchronise."""
    fn()                                                          # warm-up: same shapes, workspaces grown
    walls = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        walls.append(time.perf_counter() - t0)
    return statistics.median(walls) * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--singles", type=int, default=512, help="single calls timed per workload (scaled to m)")
    ap.add_argument("--quick", action="store_true")
    args = ap.parse_args()
    import torch
    import curve25519_dalek_b200 as pkg
    if not torch.cuda.is_available():
        raise SystemExit("needs the B200")
    eng = pkg.Engine(0)                                            # default options
    eng_s = pkg.Engine(0)                                          # the sweep of batch_bucket_min
    import bench
    pool = bench.CpuPool(len(os.sched_getaffinity(0)))
    report = {"gpu": gpu_info(), "cpu_threads": pool.threads, "reps": args.reps, "timing": "median host wall time of the blocking call, ms",
              "points": "extended limbs", "workloads": []}
    for wi, (name, lengths) in enumerate(workloads(args.quick)):
        m, n = len(lengths), sum(lengths)
        offs = [0]
        for ln in lengths:
            offs.append(offs[-1] + ln)
        sc, pts, h_sc, h_pt, d_sc, d_pt = make_inputs(eng, n, 100 + wi)
        row = {"name": name, "m": m, "pairs": n}

        def batch_host():
            return eng.edwards_vartime_msm_batch(h_sc.data_ptr(), h_pt.data_ptr(), offs, point_fmt=1)

        def batch_dev():
            return eng.edwards_vartime_msm_batch(d_sc.data_ptr(), d_pt.data_ptr(), offs, point_fmt=1, device_ptrs=True)

        ms, (rc, res_host, _) = timed(batch_host, args.reps)
        row["batch_host_ms"] = ms; row["batch_host_call_ms"] = eng.last_call_ms()
        ms, (rc2, res_dev, _) = timed(batch_dev, args.reps)
        row["batch_dev_ms"] = ms; row["batch_dev_call_ms"] = eng.last_call_ms()
        assert rc == rc2 == 0 and res_host == res_dev, name
        # the loop of single calls over a subset of the MSMs, from the same pinned host buffers; results compared
        S = min(m, args.singles)
        idx = sorted(random.Random(wi).sample(range(m), S))
        eng.edwards_vartime_msm(h_sc.data_ptr() + 32 * offs[idx[0]], h_pt.data_ptr() + 160 * offs[idx[0]], lengths[idx[0]], point_fmt=1)
        t0 = time.perf_counter()
        singles = []
        for k in idx:
            singles.append(eng.edwards_vartime_msm(h_sc.data_ptr() + 32 * offs[k], h_pt.data_ptr() + 160 * offs[k], lengths[k], point_fmt=1))
        dt = (time.perf_counter() - t0) * 1e3
        for k, (src, got, _) in zip(idx, singles):
            assert src == 0 and got == res_host[k], (name, k)
        row["singles_timed"] = S
        row["singles_loop_ms_scaled_to_m"] = dt * m / S
        row["speedup_host_vs_singles"] = row["singles_loop_ms_scaled_to_m"] / row["batch_host_ms"]
        if len(set(lengths)) == 1:
            secs, _ = pool.msm(sc, pts, n, slice_pairs=lengths[0])
            row["cpu_pool_ms"] = secs * 1e3
        # bucket threshold sweep (device-resident inputs); the results must not move
        sweep = {}
        for T in SWEEP:
            eng_s.set_option("batch_bucket_min", T)
            ms, (rc3, res_t, _) = timed(lambda: eng_s.edwards_vartime_msm_batch(d_sc.data_ptr(), d_pt.data_ptr(), offs, point_fmt=1,
                                                                                device_ptrs=True), max(2, args.reps // 2))
            assert rc3 == 0 and res_t == res_host, (name, T)
            sweep[str(T)] = ms
        row["sweep_bucket_min_dev_ms"] = sweep
        report["workloads"].append(row)
        print(json.dumps(row), flush=True)
        del h_sc, h_pt, d_sc, d_pt
        torch.cuda.empty_cache()
    # default: the threshold with the least geometric mean of (time / best time over the sweep) across the workloads
    score = {}
    for T in SWEEP:
        rel = [w["sweep_bucket_min_dev_ms"][str(T)] / min(w["sweep_bucket_min_dev_ms"].values()) for w in report["workloads"]]
        score[str(T)] = math.exp(sum(math.log(r) for r in rel) / len(rel))
    report["sweep_geomean_relative"] = score
    report["best_bucket_min"] = int(min(score, key=score.get))
    pool.close()
    eng.close()
    eng_s.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps({"best_bucket_min": report["best_bucket_min"], "geomean": score, "gpu": report["gpu"]}))


if __name__ == "__main__":
    main()
