#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 MSM / batch-verify engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload msm|verify] [--impl reference] [--dump-outputs DIR]

Metric (BASELINE.json): Pippenger MSM points/sec (default workload) and Ed25519 verify_batch
signatures/sec (reported in the same line under "verify_batch", or as the main metric with
--workload verify).  One "step" = one pass of the hot path over one batch of synthetic input.

  N = 1 : BASELINE configs[1] -- one MSM over 2^20 (scalar, EdwardsPoint) pairs, 192 B per pair
          (32 B scalar + 160 B radix-2^51 extended point), inputs resident in HBM when timing starts.
  N > 1 : BASELINE configs[3] layout -- 2^21 pairs per GPU (2^24 at N = 8), contiguous shards, each
          rank reduces its shard to window accumulators, one NCCL all-gather of the accumulators,
          every rank combines (SURVEY 8e).  Weak scaling.

`value` is device-resident throughput; `e2e` is the same call made through the C ABI with HOST
buffers (pinned), host->device copies and the result read-back inside the timed region.
`--impl reference` times the CPU oracle (the Rust reference cannot be built in this image) on all
host cores with the same metric.  Only the cpu_baseline / reference legs touch oracle/.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

L_ORDER = 2**252 + 27742317777372353535851937790883648493
SEED = 0xDA1EC00000000001
IMAD_WIDE_PEAK_PER_S = 8.96e12      # measured on this pool's B200, profiles/microbench_r1.json
FIELD_MUL_PEAK_PER_S = 119e9        # field multiplications/s of the FP64-pipe field in isolation, profiles/microbench_f64_r1.json
FIELD_SQ_PEAK_PER_S = 142e9          # field squarings/s of the FP64-pipe field in isolation (fe64_sq), profiles/microbench_f64_r1.json
FIELD_MUL_PEAK_INT_PER_S = 71e9     # same for the IMAD.WIDE field (fe.cuh), profiles/microbench_r1.json


# ------------------------------------------------------------------------------------------ utils
def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


DUMP_MAX_VALUES = 1 << 21           # per array: 16 MB of float64; larger outputs are sampled at fixed, seeded indices


def dump_outputs(path, outputs):
    """Write each output (bytes: one value per byte; a verdict list or array: one value per entry) as
    path/<name>.npy in float64, so that two builds run with the same arguments can be compared value for value."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, v in outputs.items():
        a = np.frombuffer(v, dtype=np.uint8) if isinstance(v, bytes) else np.atleast_1d(np.asarray(v))
        if a.size > DUMP_MAX_VALUES:
            a = a[np.sort(np.random.Generator(np.random.PCG64(SEED)).choice(a.size, DUMP_MAX_VALUES, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def labelled_scalars(label, n, seed=SEED):
    """n x 32 B: from_bytes_mod_order_wide(SHA-512(label || seed || i)) (SURVEY 8d generators).  Uses
    SHAKE-free bulk hashing through hashlib; 2^21 scalars take ~2 s."""
    import numpy as np
    out = np.empty((n, 32), dtype=np.uint8)
    pre = label + seed.to_bytes(8, "little")
    for i in range(n):
        h = hashlib.sha512(pre + i.to_bytes(8, "little")).digest()
        out[i] = np.frombuffer((int.from_bytes(h, "little") % L_ORDER).to_bytes(32, "little"), dtype=np.uint8)
    return out


def fast_scalars(n, seed):
    """Cheaper bulk generator for 2^20+ scalars: numpy PCG64 bytes reduced below 2^252 (uniform 252-bit
    values, all < l).  Used for the timed workloads; the labelled generator is used in the parity tests."""
    import numpy as np
    rng = np.random.Generator(np.random.PCG64(seed))
    a = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    a[:, 31] &= 0x0F
    return a


# ------------------------------------------------------------------------------------------ MSM workload
class MsmWorkload:
    def __init__(self, eng, n_local, n_total, rank, torch):
        import numpy as np
        self.eng, self.n, self.n_total, self.torch = eng, n_local, n_total, torch
        self.np = np
        # points P_i = t_i * B generated on the GPU (fixed-base kernel), extended limbs (Z != 1 is
        # produced by the additions inside the kernel); scalars uniform 252-bit.
        self.t = fast_scalars(n_local, seed=1000 + rank)
        self.s = fast_scalars(n_local, seed=2000 + rank)
        limbs, _ = eng.mul_base_batch(self.t, n_local, want_compressed=False)
        pts = np.frombuffer(limbs, dtype=np.uint64).reshape(n_local, 20).copy()
        self.h_scalars = torch.from_numpy(self.s).pin_memory()
        self.h_points = torch.from_numpy(pts.view(np.int64)).pin_memory()
        dev = torch.device("cuda", torch.cuda.current_device())
        self.d_scalars = self.h_scalars.to(dev)
        self.d_points = self.h_points.to(dev)
        torch.cuda.synchronize()
        self.bytes_per_step = n_local * 192

    def expected_local_scalar(self):
        """sum s_i t_i mod l (C/edwards.rs:2281-2295 identity), vectorised big-int arithmetic."""
        s = [int.from_bytes(r.tobytes(), "little") for r in self.s]
        t = [int.from_bytes(r.tobytes(), "little") for r in self.t]
        return sum(a * b for a, b in zip(s, t)) % L_ORDER

    def step_device_single(self):
        rc, comp, _ = self.eng.edwards_vartime_msm(self.d_scalars.data_ptr(), self.d_points.data_ptr(), self.n,
                                                   point_fmt=1, device_ptrs=True)
        assert rc == 0
        return comp

    def step_host_single(self):
        rc, comp, _ = self.eng.edwards_vartime_msm(self.h_scalars.data_ptr(), self.h_points.data_ptr(), self.n,
                                                   point_fmt=1, device_ptrs=False)
        assert rc == 0
        return comp


def run_msm(args, rank, world, local, outputs=None):
    import numpy as np
    import torch
    import torch.distributed as dist
    import curve25519_dalek_b200 as pkg

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))      # NCCL_DEBUG is left to the caller
    eng = pkg.Engine(local)
    n_local = args.pairs_per_gpu or ((1 << 20) if world == 1 else (1 << 21))
    n_total = n_local * world
    wl = MsmWorkload(eng, n_local, n_total, rank, torch)
    dev = torch.device("cuda", local)
    # N > 1: the shard's MSM, the NCCL all-gather of the window-accumulator records and the combine are all enqueued
    # on the engine's stream (curve25519_dalek_b200/sharding.py); the window width comes from the shard size
    from curve25519_dalek_b200.sharding import ShardedMsm
    sharded = ShardedMsm(eng, world, n_local, dev) if world > 1 else None
    nwin = eng.msm_window_count(n_local)

    def step(host=False):
        if world == 1:
            return wl.step_host_single() if host else wl.step_device_single()
        s = wl.h_scalars if host else wl.d_scalars
        p = wl.h_points if host else wl.d_points
        rc, comp = sharded.run(s.data_ptr(), p.data_ptr(), n_local, 1, not host)
        assert rc == 0
        return comp

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # --- correctness at full size: sum s_i (t_i B) == (sum s_i t_i mod l) B  (C/edwards.rs:2281-2295)
    got = step()
    k_local = wl.expected_local_scalar()
    if world > 1:
        ks = [None] * world
        dist.all_gather_object(ks, k_local)
        k = sum(ks) % L_ORDER
    else:
        k = k_local
    _, want = eng.mul_base_batch(np.frombuffer(k.to_bytes(32, "little"), dtype=np.uint8).copy(), 1)
    parity = (got == want)
    if not parity:
        raise SystemExit("bench: MSM result does not satisfy the algebraic identity")

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    kernel_ms = []
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = eng.launch_count()
    t0 = time.perf_counter()
    call_ms = []
    for _ in range(args.steps):
        comp = step()
        kernel_ms.append(eng.last_kernel_ms()[0])
        call_ms.append(eng.last_call_ms())           # CUDA events on the engine's stream around the MSM call
    barrier()
    t1 = time.perf_counter()
    launches = eng.launch_count() - launches0
    elapsed = torch.tensor([t1 - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(elapsed, op=dist.ReduceOp.MAX)
    elapsed = float(elapsed.item())

    # --- end to end: host (pinned) buffers through the same C-ABI call
    for _ in range(min(2, args.warmup)):
        step(host=True)
    barrier()
    e0 = time.perf_counter()
    e2e_call_ms = []
    for _ in range(args.steps):
        comp_e2e = step(host=True)
        e2e_call_ms.append(eng.last_call_ms())
    barrier()
    e1 = time.perf_counter()
    if outputs is not None:
        outputs.update(msm_point=comp, msm_point_e2e=comp_e2e)
    clocks = sampler.stop() if rank == 0 else None        # sampled over both timed regions
    e2e_t = torch.tensor([e1 - e0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_t = float(e2e_t.item())

    line = None
    if rank == 0:
        peaks, how = measured_peaks()
        kms = statistics.mean(kernel_ms)
        algo_bytes = n_local * 192
        achieved = algo_bytes / (kms * 1e-3) / 1e9
        c = eng_window_bits(n_local)          # chosen from the shard size (the work one GPU does)
        adds = n_local * ((253 + c - 1) // c)
        field_muls = adds * 8                # 8M per projective-Niels addition (curve_models.rs:411-430 + :365-372)
        traffic = None
        tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                traffic = json.load(f).get("k_bucket_accumulate_msm_2p20_bytes")
        line = {
            "metric": "Pippenger MSM points/sec", "value": n_total * args.steps / elapsed, "unit": "points/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "exact integers: f64 limbs (radix 2^51, FP64 pipe) in the bucket kernel, u32 limbs (radix 2^25.5) elsewhere",
            "data": "synthetic: uniform 252-bit scalars, points t_i*B from the on-GPU fixed-base kernel",
            "config": {"workload": "pippenger_msm", "pairs_total": n_total, "pairs_per_gpu": n_local,
                       "point_format": "extended radix-2^51 limbs (160 B)", "window_bits": c,
                       "l2": "inputs (%.0f MB per GPU) exceed the 126 MB L2" % (algo_bytes / 1e6),
                       "host_buffers": "pinned, filled by one thread (NUMA-local first touch)",
                   "timing": "value / ms_per_step: K blocking C-ABI calls bracketed by barrier + device sync, max over ranks; "
                                 "device_ms_per_step: CUDA events on the engine's stream around each call (rank 0)",
                       "device_ms_per_step": statistics.mean(call_ms), "e2e_device_ms_per_step": statistics.mean(e2e_call_ms),
                       "parity": "algebraic identity sum s_i(t_i B) == (sum s_i t_i)B checked at full size",
                       "exchange": None if world == 1 else "one NCCL all-gather of %d-byte records (window accumulators) per rank, enqueued on "
                                   "the engine's stream between the shard MSM and the combine; no host bounce" % sharded.rec_bytes},
            "e2e": {"value": n_total * args.steps / e2e_t, "unit": "points/s",
                    "h2d_bytes_per_step": n_local * 192, "d2h_bytes_per_step": 192},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "k_bucket_accumulate", "achieved": achieved, "peak": peaks["hbm_gbs"],
                         "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "traffic": traffic,
                         "peak_source": how + " (MEASURED_PEAKS.json hbm_gbs)", "kernel_ms": kms,
                         "algorithmic_bytes_per_launch": algo_bytes,
                         "note": "arithmetic-bound, not HBM-bound: see roofline_fieldmul"},
            "roofline_fieldmul": {"bound": "exact GF(2^255-19) multiplications (FP64 DFMA + integer pipes)",
                                  "achieved": field_muls / (kms * 1e-3) / 1e9, "peak": FIELD_MUL_PEAK_PER_S / 1e9,
                                  "unit": "G field mul/s", "frac": field_muls / (kms * 1e-3) / FIELD_MUL_PEAK_PER_S,
                                  "peak_source": "register-resident multiplication chain of the same field code, measured "
                                                 "(profiles/microbench_f64_r1.json; the IMAD.WIDE form peaks at %.0f G/s, "
                                                 "IMAD.WIDE.U32 itself at %.2f T/s)" % (FIELD_MUL_PEAK_INT_PER_S / 1e9, IMAD_WIDE_PEAK_PER_S / 1e12),
                                  "algorithmic_field_muls_per_launch": field_muls},
            "clocks": clocks,
        }
    return line, eng, wl


def run_msm_two_callers(eng, wl, local, steps=40):
    """Throughput of a SERVICE rather than the latency of one call: two host threads, each with its own engine context on the
    same GPU, issue blocking 2^20-pair MSM calls on the same resident inputs.  The latency-bound tail of one call (bucket
    reduction trees, the 240 sequential doublings of the final Horner: ~0.6 ms on a handful of warps) then overlaps the other
    call's arithmetic.  Same C-ABI entry point, same results; nothing is shared between the two contexts."""
    import threading
    import torch
    import curve25519_dalek_b200 as pkg
    eng2 = pkg.Engine(local)
    want = wl.step_device_single()
    engines = [eng, eng2]

    def call(e):
        rc, comp, _ = e.edwards_vartime_msm(wl.d_scalars.data_ptr(), wl.d_points.data_ptr(), wl.n, point_fmt=1, device_ptrs=True)
        if rc != 0 or comp != want:
            raise SystemExit("bench: two-caller MSM result differs")

    for e in engines:
        for _ in range(3):
            call(e)
    per = steps // 2
    errs = []

    def worker(e):
        try:
            torch.cuda.set_device(local)
            for _ in range(per):
                call(e)
        except BaseException as ex:      # surfaced after the join
            errs.append(ex)

    torch.cuda.synchronize()
    ts = [threading.Thread(target=worker, args=(e,)) for e in engines]
    t0 = time.perf_counter()
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    eng2.close() if hasattr(eng2, "close") else None
    if errs:
        raise errs[0]
    return {"metric": "Pippenger MSM points/sec, two concurrent callers (one engine context each) on one GPU", "value": wl.n * 2 * per / dt,
            "unit": "points/s", "calls": 2 * per, "ms_per_call_amortised": dt / (2 * per) * 1e3, "pairs_per_call": wl.n,
            "note": "value / ms_per_step of the main line are ONE caller's blocking calls; this leg shows what overlapping the tail of one call with the next call's arithmetic yields"}


def run_msm_like_for_like(eng, n, steps):
    """The N = 1 rate at the per-GPU size of the N > 1 runs (2^21 pairs): the like-for-like denominator of the scaling
    efficiency.  Device-resident, same call as the headline."""
    import torch
    wl = MsmWorkload(eng, n, n, 7, torch)
    for _ in range(3):
        wl.step_device_single()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    kms = []
    for _ in range(steps):
        wl.step_device_single()
        kms.append(eng.last_kernel_ms()[0])
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    return {"metric": "Pippenger MSM points/sec, 2^21 pairs on one GPU (the shard size of the N > 1 runs)", "value": n / dt,
            "unit": "points/s", "ms_per_step": dt * 1e3, "pairs": n, "window_bits": eng_window_bits(n),
            "bucket_kernel_ms": statistics.mean(kms)}


def eng_window_bits(n):
    best, best_cost = 4, 1e300
    for c in range(4, 21):
        W = (253 + c - 1) // c
        cost = W * (n + 4.0 * (1 << (c - 1)))
        if cost < best_cost:
            best, best_cost = c, cost
    return best


# ------------------------------------------------------------------------------------------ verify workload
def build_verify_inputs(eng, n, nkeys=1024):
    """BASELINE configs[2]: n signatures over 59-byte messages (51 x 'a' || i_le64) by `nkeys` keys,
    signed on the GPU (byte-identical to RFC 8032 signing, spot-checked in tests)."""
    import numpy as np
    if nkeys <= 65536:
        seeds_k = np.stack([np.frombuffer(hashlib.sha512(b"dalek-b200/sk" + SEED.to_bytes(8, "little") + k.to_bytes(8, "little")).digest()[:32], dtype=np.uint8)
                            for k in range(nkeys)])
    else:
        seeds_k = np.random.Generator(np.random.PCG64(SEED & 0xffffffff)).integers(0, 256, size=(nkeys, 32), dtype=np.uint8)
    idx = np.arange(n) % nkeys
    seeds = np.ascontiguousarray(seeds_k[idx])
    msgs = np.full((n, 59), ord("a"), dtype=np.uint8)
    msgs[:, 51:] = np.arange(n, dtype="<u8").view(np.uint8).reshape(n, 8)
    flat = np.ascontiguousarray(msgs.reshape(-1))
    offs = (np.arange(n + 1, dtype=np.uint64) * 59)
    pks, sigs = eng.sign_batch_flat(seeds, flat, offs, n)
    return flat, offs, np.frombuffer(sigs, dtype=np.uint8).copy(), np.frombuffer(pks, dtype=np.uint8).copy()


def run_verify(args, rank, world, local, eng=None, steps=None, warmup=None, nkeys=1024, batch_size=None, each=False, key_points=False,
               outputs=None):
    import numpy as np
    import torch
    import torch.distributed as dist
    import curve25519_dalek_b200 as pkg
    steps = steps or args.steps
    warmup = args.warmup if warmup is None else warmup
    torch.cuda.set_device(local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    eng = eng or pkg.Engine(local)
    n = args.sigs_per_gpu or (1 << 22)
    # the primary leg: the 2^22 signatures as independent verify_batch calls of `verify_batch_size` (256: the reference's
    # largest published batch size, BASELINE.md section 2 config 3), every batch with exactly the reference's transcript and
    # verdict; batch_size = 0: ONE verdict over all signatures
    if batch_size is None:
        batch_size = 0 if each else args.verify_batch_size
    flat, offs, sigs, pks = build_verify_inputs(eng, n, nkeys=min(nkeys, n))
    dev = torch.device("cuda", local)
    h = [torch.from_numpy(x if x.dtype == np.uint8 else x.view(np.int64)).pin_memory() for x in (flat, offs, sigs, pks)]
    d = [x.to(dev) for x in h]
    torch.cuda.synchronize()
    if key_points:
        # what a Rust caller holds: the VerifyingKeys' decompressed points (E/verifying.rs:65-71), made here once with the
        # batch codec, outside the timed region -- as VerifyingKey::from_bytes is outside verify_batch in the reference
        rc_k, limbs, okk = eng.decompress_batch(pks.tobytes(), n)
        if rc_k != 0 or not all(okk):
            raise SystemExit("bench: key decompression failed")
        hk = torch.from_numpy(np.frombuffer(limbs, dtype=np.uint64).copy().view(np.int64)).pin_memory()
        dk = hk.to(dev)
        torch.cuda.synchronize()

    each_res = np.zeros(n, dtype=np.uint8) if each else None
    # One call over n = 2^22 signatures: the reference's single Merlin transcript is a strictly sequential sponge of
    # 1.73 Keccak permutations per signature (seconds for 2^22, on any hardware), so this leg opts into one transcript per
    # `transcript_chunk` signatures (verdict-equivalent on inputs without small-order components; INTEGRATION.md).  The
    # batches_of_256 leg and every call with the default options use exactly the reference's transcripts.
    transcript_chunk = 0 if (each or batch_size) else args.transcript_chunk
    eng.set_option("verify_chunk", transcript_chunk)

    def step(host=False):
        b = h if host else d
        if each:            # SURVEY 8f rank 3: one verdict per signature (VerifyingKey::verify semantics)
            fn = eng.lib.ed25519_b200_verify_each_flat if host else eng.lib.ed25519_b200_verify_each_flat_dev
            rc = fn(eng.h, b[0].data_ptr(), b[1].data_ptr(), b[2].data_ptr(), b[3].data_ptr(), n, 0, each_res.ctypes.data)
            if rc != 0:
                raise SystemExit("bench: verify_each rejected valid signatures (rc=%d)" % rc)
            return each_res
        if batch_size and key_points:
            rc, verdicts = eng.verify_batches_flat_points(b[0].data_ptr(), b[1].data_ptr(), b[2].data_ptr(), b[3].data_ptr(),
                                                          (hk if host else dk).data_ptr(), n, batch_size, device_ptrs=not host)
            if rc != 0 or any(verdicts):
                raise SystemExit("bench: verify_batches (key points) rejected valid signatures")
            return verdicts
        if batch_size:      # SURVEY 8d config 3B: independent batches of `batch_size`, one verdict each
            rc, verdicts = eng.verify_batches_flat(b[0].data_ptr(), b[1].data_ptr(), b[2].data_ptr(), b[3].data_ptr(), n, batch_size,
                                                   device_ptrs=not host)
            if rc != 0 or any(verdicts):
                raise SystemExit("bench: verify_batches rejected valid signatures")
            return verdicts
        rc = eng.verify_batch_flat(b[0].data_ptr(), b[1].data_ptr(), b[2].data_ptr(), b[3].data_ptr(), n,
                                   device_ptrs=not host, msgs_bytes=n * 59)
        if rc != 0:
            raise SystemExit("bench: verify_batch returned %d on valid signatures" % rc)
        return rc

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # negative control: one flipped message bit must give Verify (1)
    d[0][59 * 777 + 3] ^= 1
    if each:
        rc_e, res_e = eng.verify_each_flat(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), 1024, device_ptrs=True)
        if rc_e != 1 or [i for i, r in enumerate(res_e) if r] != [777]:
            raise SystemExit("bench: verify_each did not single out the corrupted signature")
        rc = 1
    elif batch_size:
        rc, verd = eng.verify_batches_flat(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), n, batch_size, device_ptrs=True)
        if [k for k, v in enumerate(verd) if v] != [777 // batch_size]:
            raise SystemExit("bench: verify_batches did not single out the corrupted batch")
    else:
        rc = eng.verify_batch_flat(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), n, device_ptrs=True)
    d[0][59 * 777 + 3] ^= 1
    if rc != 1:
        raise SystemExit("bench: corrupted batch was not rejected (rc=%d)" % rc)
    for _ in range(warmup):
        step()
    sampler = ClockSampler(local)
    kernel_ms = []
    barrier()
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count()
    t0 = time.perf_counter()
    call_ms, e2e_call_ms, prep_ms = [], [], []
    for _ in range(steps):
        res = step()
        kernel_ms.append(eng.last_kernel_ms()[0])
        call_ms.append(eng.last_call_ms())
        if not each:
            prep_ms.append(eng.last_stage_ms("decompress_R"))
    barrier()
    t1 = time.perf_counter()
    if outputs is not None:
        outputs["verify_result"] = np.array(res)          # a copy: verify_each reuses its result buffer in the next loop
    launches = eng.launch_count() - l0
    el = torch.tensor([t1 - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    el = float(el.item())
    step(host=True)
    barrier()
    e0 = time.perf_counter()
    for _ in range(steps):
        res = step(host=True)
        e2e_call_ms.append(eng.last_call_ms())
    barrier()
    e1 = time.perf_counter()
    if outputs is not None:
        outputs["verify_result_e2e"] = np.array(res)
    clocks = sampler.stop() if rank == 0 else None
    et = torch.tensor([e1 - e0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(et, op=dist.ReduceOp.MAX)
    et = float(et.item())
    eng.set_option("verify_chunk", 0)
    if rank != 0:
        return None
    peaks, how = measured_peaks()
    kms = statistics.mean(kernel_ms)
    achieved = n * 155 / (el / steps) / 1e9
    # dominant kernel of verify_batch: the decompression of the n R points (252 squarings + 13 multiplications each, on the
    # FP64-pipe field), timed with CUDA events on its stream while the hashing / transcript kernels share the SMs
    pms = statistics.mean(prep_ms) if prep_ms and min(prep_ms) > 0 else None
    traffic = None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            traffic = json.load(f).get("k_prep_R_verify_2p22_bytes")
    dominant = None
    if pms:
        sq = n * 265.0
        dominant = {"bound": "hbm", "kernel": "k_prep_R (R decompression)", "kernel_ms": pms,
                    "achieved": n * 155 / (pms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": n * 155 / (pms * 1e-3) / 1e9 / peaks["hbm_gbs"], "traffic": traffic,
                    "algorithmic_bytes_per_launch": n * 155, "peak_source": how + " (MEASURED_PEAKS.json hbm_gbs)",
                    "note": "arithmetic-bound: see field_ops",
                    "field_ops": {"achieved": sq / (pms * 1e-3) / 1e9, "peak": FIELD_SQ_PEAK_PER_S / 1e9, "unit": "G field squarings/s",
                                  "frac": sq / (pms * 1e-3) / FIELD_SQ_PEAK_PER_S,
                                  "algorithmic_field_ops_per_launch": sq,
                                  "peak_source": "register-resident squaring chain of the same FP64-pipe field code (profiles/microbench_f64_r1.json); "
                                                 "252 squarings + 13 multiplications per point (field.rs:297-306, :320-366), the kernel runs "
                                                 "concurrently with the SHA-512 and Merlin kernels of the same call"}}
    return {
        "metric": "Ed25519 verify_batch signatures/sec", "value": n * world * steps / el, "unit": "sigs/s",
        "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": el / steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "exact integers: f64 limbs (radix 2^51, FP64 pipe) in the bucket kernel, u32 limbs (radix 2^25.5) elsewhere", "data": "synthetic: 59-byte messages, %d distinct keys, signatures made on the GPU (RFC 8032)" % min(nkeys, n),
        "config": {"workload": "ed25519_verify_batch", "signatures_per_gpu": n, "message_bytes": 59, "distinct_keys": min(nkeys, n),
                   "transcript": ("one Merlin transcript per %d signatures (option verify_chunk, opt-in; default = the reference's single transcript)" % transcript_chunk)
                                 if transcript_chunk else "the reference's transcripts (one per batch)",
                   "keys": "the callers' decompressed points (VerifyingKey, 160 B each) beside the 32-byte encodings" if key_points
                           else "32-byte encodings, decompressed inside the call",
                   "batch_size": batch_size or None,
                   "host_buffers": "pinned, filled by one thread (NUMA-local first touch)",
                   "timing": "value / ms_per_step: K blocking C-ABI calls bracketed by barrier + device sync, max over ranks; "
                             "device_ms_per_step: CUDA events on the engine's stream around each call (rank 0)",
                   "device_ms_per_step": statistics.mean(call_ms), "e2e_device_ms_per_step": statistics.mean(e2e_call_ms),
                   "l2": "inputs (%.0f MB) exceed the 126 MB L2" % (n * 155 / 1e6),
                   "replicas": "independent batches per GPU, no collective" if world > 1 else "single batch"},
        "e2e": {"value": n * world * steps / et, "unit": "sigs/s", "h2d_bytes_per_step": n * 155 + (n + 1) * 8 + (n * 160 if key_points else 0),
                "d2h_bytes_per_step": n if each else (4 * ((n + batch_size - 1) // batch_size) if batch_size else 192)},
        "gpu_launches": int(launches),
        "roofline": dominant or {"bound": "hbm", "kernel": "whole call (155 B per signature)", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                 "frac": achieved / peaks["hbm_gbs"], "traffic": None, "peak_source": how,
                                 "note": "integer-multiply bound (decompression + MSM)"},
        "roofline_whole_call": {"achieved": achieved, "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "bucket_kernel_ms": kms},
        "clocks": clocks,
    }


def run_verify_exact_once(eng, args, n=1 << 18):
    """One verify_batch call over n signatures with the DEFAULT options: the reference's single Merlin transcript
    (batch.rs:168-222), a sequential sponge of 1.73 Keccak-f[1600] permutations per signature on one GPU thread."""
    import numpy as np
    import torch
    flat, offs, sigs, pks = build_verify_inputs(eng, n, nkeys=1024)
    dev = torch.device("cuda", torch.cuda.current_device())
    d = [torch.from_numpy(x if x.dtype == np.uint8 else x.view(np.int64)).to(dev) for x in (flat, offs, sigs, pks)]
    eng.set_option("verify_chunk", 0)
    t0 = time.perf_counter()
    rc = eng.verify_batch_flat(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), n, device_ptrs=True, msgs_bytes=n * 59)
    dt = time.perf_counter() - t0
    if rc != 0:
        raise SystemExit("bench: verify_batch (single transcript) returned %d on valid signatures" % rc)
    return {"signatures": n, "seconds": dt, "value": n / dt, "unit": "sigs/s",
            "note": "ONE call, ONE transcript over all signatures (exactly the reference's z_i): bound by the sequential sponge, "
                    "not by the GPU's arithmetic; callers with large inputs use verify_batches (one reference transcript per batch) "
                    "or opt into verify_chunk"}


def run_precomputed(eng, wl, steps=10):
    """SURVEY 8f rank 1: VartimePrecomputedMultiscalarMul with the 2^20 points of the MSM workload as static points,
    resident on the GPU; a call sends the scalars only (32 B per term, pinned host memory) and must give the same
    encoding as the plain MSM."""
    import ctypes as C
    pre = C.c_void_p()
    rc = eng.lib.dalek_b200_precomp_new(eng.h, wl.h_points.data_ptr(), 1, wl.n, C.byref(pre))
    assert rc == 0
    out = (C.c_uint8 * 32)()

    def step():
        rc = eng.lib.dalek_b200_precomp_mixed_msm(eng.h, pre, wl.h_scalars.data_ptr(), wl.n, None, None, 1, 0, C.addressof(out), None)
        assert rc == 0
    for _ in range(3):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    same = bytes(out) == wl.step_device_single()
    eng.lib.dalek_b200_precomp_destroy(pre)
    return {"metric": "precomputed-static-points MSM points/sec, scalars from pinned host memory", "value": wl.n / dt, "unit": "points/s",
            "ms_per_step": dt * 1e3, "static_points": wl.n, "h2d_bytes_per_step": 32 * wl.n, "d2h_bytes_per_step": 192,
            "matches_plain_msm": bool(same)}


def run_codecs(eng, wl, steps=5):
    """SURVEY 8f rank 2: batch codecs on the 2^20 points of the MSM workload, pinned host buffers in and out."""
    import torch
    n = wl.n
    enc = torch.empty(32 * n, dtype=torch.uint8).pin_memory()
    enc2 = torch.empty(32 * n, dtype=torch.uint8).pin_memory()
    limbs = torch.empty(20 * n, dtype=torch.int64).pin_memory()
    ok = torch.empty(n, dtype=torch.uint8).pin_memory()
    lib, h = eng.lib, eng.h

    def timed(fn):
        fn(); fn()
        t0 = time.perf_counter()
        for _ in range(steps):
            rc = fn()
        dt = (time.perf_counter() - t0) / steps
        assert rc == 0
        return {"value": n / dt, "unit": "points/s", "ms_per_step": dt * 1e3, "device_span_ms": eng.last_kernel_ms()[0]}
    out = {"points": n}
    out["compress_batch"] = timed(lambda: lib.dalek_b200_edwards_compress_batch(h, wl.h_points.data_ptr(), n, enc.data_ptr()))
    out["decompress_batch"] = timed(lambda: lib.dalek_b200_edwards_decompress_batch(h, enc.data_ptr(), n, limbs.data_ptr(), ok.data_ptr()))
    out["ristretto_double_and_compress_batch"] = timed(
        lambda: lib.dalek_b200_ristretto_double_and_compress_batch(h, wl.h_points.data_ptr(), n, enc2.data_ptr()))
    assert lib.dalek_b200_edwards_compress_batch(h, limbs.data_ptr(), n, enc2.data_ptr()) == 0
    out["round_trip_ok"] = bool(torch.equal(enc, enc2)) and bool(ok.all())
    return out


def run_double_base(eng, n=1 << 20, steps=3, cpu_threads=1):
    """BASELINE configs[4]: RistrettoPoint::multiscalar_mul([a_i, b_i], [G, H]) for 2^20 pairs (constant-time
    contract), host buffers in, compressed points out (64 B in + 32 B out per pair).  A 4096-pair sample of the output is
    compared with the oracle's constant-time Straus (straus.rs:103-144 -> ristretto.rs:500-533); the same oracle run on
    one host thread is the cpu_baseline."""
    import numpy as np
    a, b = fast_scalars(n, seed=31), fast_scalars(n, seed=32)
    # Ristretto basepoint encoding (curve25519-dalek/src/constants.rs:57-60) and H = h*G via the engine itself
    G = bytes.fromhex("e2f2ae0a6abc4e71a884a961c500515f58e30b6aa582dd8db6a65945e08d2d76")
    h = np.frombuffer(hashlib.sha512(b"dalek-b200/H").digest()[:32], dtype=np.uint8).copy(); h[31] &= 0x0F
    rc, H = eng.ristretto_double_base_batch(np.zeros(32, dtype=np.uint8), h, G, G, 1)
    assert rc == 0
    import torch
    ha, hb = torch.from_numpy(a).pin_memory(), torch.from_numpy(b).pin_memory()
    hout = torch.empty(32 * n, dtype=torch.uint8).pin_memory()
    eng.ristretto_double_base_batch(ha, hb, G, H, n, out=hout)
    t0 = time.perf_counter()
    for _ in range(steps):
        rc, _ = eng.ristretto_double_base_batch(ha, hb, G, H, n, out=hout)
    dt = (time.perf_counter() - t0) / steps
    assert rc == 0
    out = hout.numpy().reshape(n, 32)
    # oracle parity on a sample spread over the batch (first, last and strided pairs), timed as the CPU baseline
    ns = 4096
    idx = np.unique(np.concatenate([np.arange(0, 1024), np.arange(n - 1024, n), np.linspace(1024, n - 1025, 2048).astype(np.int64)]))[:ns]
    pool = CpuPool(cpu_threads)
    cdt, want = pool.double_base(np.ascontiguousarray(a[idx]), np.ascontiguousarray(b[idx]), G, H, len(idx))
    pool.close()
    if not np.array_equal(want, out[idx]):
        raise SystemExit("bench: double-base batch differs from the oracle on the %d-pair sample" % len(idx))
    return {"metric": "Ristretto double-base (aG+bH) pairs/sec, pinned host buffers in and out", "value": n / dt, "unit": "pairs/s",
            "ms_per_step": dt * 1e3, "device_span_ms": eng.last_kernel_ms()[0], "pairs": n,
            "h2d_bytes_per_step": 64 * n, "d2h_bytes_per_step": 32 * n,
            "parity": "%d-pair sample (first 1024, last 1024, 2048 strided) byte-equal to the oracle's constant-time Straus + Ristretto encoding" % len(idx),
            "checksum": hashlib.sha256(hout.numpy().tobytes()).hexdigest()[:16],
            "cpu_baseline": {"value": len(idx) / cdt, "unit": "pairs/s", "cores": cpu_threads, "kind": "port",
                             "sample": "oracle RistrettoPoint::multiscalar_mul([a,b],[G,H]) + compress on the %d-pair parity sample (%.1f s)" % (len(idx), cdt)}}


def run_msm_compressed(eng, wl, steps=10):
    """SURVEY 8d: the compressed-input variant of config 2 -- 64 B per pair (32 B scalar + 32 B CompressedEdwardsY), the
    points are decompressed inside the call (edwards.rs:211-257).  Device-resident and end to end from pinned host memory."""
    import torch
    n = wl.n
    enc = torch.empty(32 * n, dtype=torch.uint8).pin_memory()
    assert eng.lib.dalek_b200_edwards_compress_batch(eng.h, wl.h_points.data_ptr(), n, enc.data_ptr()) == 0
    d_enc = enc.cuda()
    want = wl.step_device_single()
    res = {}
    for name, sp, pp, dev_ptrs in (("device_resident", wl.d_scalars, d_enc, True), ("e2e", wl.h_scalars, enc, False)):
        for _ in range(3):
            rc, got, _ = eng.edwards_vartime_msm(sp.data_ptr(), pp.data_ptr(), n, point_fmt=0, device_ptrs=dev_ptrs)
        assert rc == 0 and got == want, "compressed-input MSM differs from the extended-input result"
        torch.cuda.synchronize(); t0 = time.perf_counter()
        for _ in range(steps):
            eng.edwards_vartime_msm(sp.data_ptr(), pp.data_ptr(), n, point_fmt=0, device_ptrs=dev_ptrs)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        res[name] = {"value": n / dt, "unit": "points/s", "ms_per_step": dt * 1e3}
    res["e2e"].update({"h2d_bytes_per_step": 64 * n, "d2h_bytes_per_step": 192})
    res.update({"metric": "Pippenger MSM points/sec, compressed points (64 B per pair), decompression inside the call", "pairs": n,
                "matches_extended_input_result": True})
    return res


def run_small_latency(eng, sizes=(1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024), reps=30):
    """BASELINE configs[0] and the reference's own bench sizes (dalek_benchmarks.rs:16, :145-189): latency of ONE
    vartime_multiscalar_mul call on host buffers (in-memory EdwardsPoints, 160 B each), GPU engine against the oracle on one
    host thread, results compared byte for byte.  Below 190 points both GPU paths are timed (vartime Straus / bucket pipeline)."""
    import numpy as np
    nmax = max(sizes)
    t = fast_scalars(nmax, seed=501)
    sc = fast_scalars(nmax, seed=502)
    limbs, _ = eng.mul_base_batch(t, nmax, want_compressed=False)
    pts = np.frombuffer(limbs, dtype=np.uint64).reshape(nmax, 20).copy()
    pool = CpuPool(1)
    rows = []

    def gpu_us(n):
        for _ in range(3):
            rc, got, _ = eng.edwards_vartime_msm(sc, pts, n, point_fmt=1)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            eng.edwards_vartime_msm(sc, pts, n, point_fmt=1)
            ts.append(time.perf_counter() - t0)
        return statistics.median(ts) * 1e6, got

    for n in sizes:
        cpu = []
        for _ in range(3):
            dt, want = pool.msm(sc, pts, n, slice_pairs=n)
            cpu.append(dt)
        row = {"n": n, "cpu_us": statistics.median(cpu) * 1e6}
        us, got = gpu_us(n)
        if got != want:
            raise SystemExit("bench: small MSM (n=%d) differs from the oracle" % n)
        row["gpu_us"] = us
        if n < 190:
            eng.set_option("small_straus", 0)
            row["gpu_bucket_pipeline_us"], got2 = gpu_us(n)
            eng.set_option("small_straus", 1)
            if got2 != want:
                raise SystemExit("bench: small MSM through the bucket pipeline (n=%d) differs from the oracle" % n)
        rows.append(row)
    pool.close()
    faster = [r["n"] for r in rows if r["gpu_us"] < r["cpu_us"]]
    return {"metric": "latency of one EdwardsPoint::vartime_multiscalar_mul call, host buffers (160-byte points), microseconds",
            "sizes": rows, "gpu_faster_from_n": min(faster) if faster else None,
            "cpu": "oracle (reference algorithm: Straus below 190 points, Pippenger above), 1 host thread, median of 3",
            "gpu": "blocking C-ABI call incl. copies, median of %d; n < 190: vartime Straus kernels (4 launches), else the bucket pipeline" % reps,
            "config1_n256": next((r for r in rows if r["n"] == 256), None)}


# ------------------------------------------------------------------------------------------ CPU baseline (oracle)
def physical_cores():
    """Distinct (package, core) pairs of /proc/cpuinfo; None if it cannot be read."""
    try:
        seen, phys, core = set(), None, None
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("physical id"):
                phys = ln.split(":")[1].strip()
            elif ln.startswith("core id"):
                core = ln.split(":")[1].strip()
            elif not ln.strip():
                if phys is not None and core is not None:
                    seen.add((phys, core))
                phys = core = None
        return len(seen) or None
    except OSError:
        return None


def effective_cpus():
    """CPUs this process may actually use: the affinity mask, capped by the cgroup CPU quota (the GPU boxes expose 128
    logical CPUs behind a 16-CPU quota: more threads than that only add context switches -- tools/cpu_pool_scaling.py,
    profiles/cpu_pool_scaling_r2.json)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = int(q) / int(per)
    except (OSError, ValueError):
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except (OSError, ValueError):
            pass
    if quota:
        n = max(1, min(n, int(quota + 0.5)))
    return n, quota


class CpuPool:
    """Persistent worker threads of the oracle (oracle/parallel.c): every thread runs the unmodified, single-threaded
    reference restatement on an independent slice.  Checker / baseline infrastructure only."""

    def __init__(self, threads):
        import oracle_lib
        self.orc = oracle_lib.load()
        lib = self.lib = self.orc.lib
        vp, sz, dbl = C.c_void_p, C.c_size_t, C.c_double
        lib.oracle_pool_create.restype = vp; lib.oracle_pool_create.argtypes = [C.c_int]
        lib.oracle_pool_destroy.argtypes = [vp]
        lib.oracle_pool_msm.restype = dbl; lib.oracle_pool_msm.argtypes = [vp, vp, vp, vp, sz, sz]
        lib.oracle_pool_verify_batches.restype = dbl; lib.oracle_pool_verify_batches.argtypes = [vp, vp, sz, vp, vp, sz, sz, vp]
        lib.oracle_pool_verify_each.restype = dbl; lib.oracle_pool_verify_each.argtypes = [vp, vp, sz, vp, vp, sz, C.c_int, vp]
        lib.oracle_pool_double_base.restype = dbl; lib.oracle_pool_double_base.argtypes = [vp, vp, vp, vp, vp, vp, sz, vp]
        self.threads = threads
        self.h = lib.oracle_pool_create(threads)

    def close(self):
        if self.h:
            self.lib.oracle_pool_destroy(self.h)
            self.h = None

    def msm_inputs(self, n):
        import numpy as np
        pts = np.empty((n, 20), dtype=np.uint64)
        t0b = (0x1234567 + SEED).to_bytes(32, "little")
        qb = (0x9e3779b97f4a7c15f39cc0605cedc834 % L_ORDER).to_bytes(32, "little")
        self.lib.oracle_points_progression(pts.ctypes.data_as(C.c_void_p), C.c_size_t(n), t0b, qb)
        return fast_scalars(n, seed=77), pts

    def msm(self, sc, pts, n, slice_pairs=8192):
        """One n-pair MSM as independent reference Pippenger sub-MSMs (w = 8, pippenger.rs:81-87) of `slice_pairs` pairs
        pulled by the pool's threads; partial sums added.  Returns seconds."""
        out = (C.c_uint8 * 32)()
        return self.lib.oracle_pool_msm(self.h, C.addressof(out), sc.ctypes.data, pts.ctypes.data, n, slice_pairs), bytes(out)

    def verify_inputs(self, nsigs, nkeys=64):
        import numpy as np
        orc = self.orc
        seeds = [hashlib.sha512(b"dalek-b200/sk" + k.to_bytes(8, "little")).digest()[:32] for k in range(nkeys)]
        pk = [orc.public_key(s) for s in seeds]
        base = 256                                          # sign 256 distinct messages, tile them (the CPU cost does not depend on repeats)
        msgs = [b"a" * 51 + i.to_bytes(8, "little") for i in range(base)]
        sigs = [orc.sign(m, seeds[i % nkeys]) for i, m in enumerate(msgs)]
        reps = (nsigs + base - 1) // base
        m = np.frombuffer(b"".join(msgs) * reps, dtype=np.uint8)[:59 * nsigs].copy()
        s = np.frombuffer(b"".join(sigs) * reps, dtype=np.uint8)[:64 * nsigs].copy()
        k = np.frombuffer(b"".join(pk[i % nkeys] for i in range(base)) * reps, dtype=np.uint8)[:32 * nsigs].copy()
        return m, s, k

    def verify_batches(self, m, s, k, nsigs, batch=256):
        import numpy as np
        verd = np.zeros((nsigs + batch - 1) // batch, dtype=np.int32)
        dt = self.lib.oracle_pool_verify_batches(self.h, m.ctypes.data, 59, s.ctypes.data, k.ctypes.data, nsigs, batch, verd.ctypes.data)
        assert not verd.any(), "oracle rejected valid signatures"
        return dt

    def verify_each(self, m, s, k, nsigs):
        import numpy as np
        res = np.zeros(nsigs, dtype=np.uint8)
        dt = self.lib.oracle_pool_verify_each(self.h, m.ctypes.data, 59, s.ctypes.data, k.ctypes.data, nsigs, 0, res.ctypes.data)
        assert not res.any(), "oracle rejected valid signatures"
        return dt

    def double_base(self, a, b, G, H, n):
        import numpy as np
        out = np.zeros((n, 32), dtype=np.uint8)
        ok = C.c_int(0)
        dt = self.lib.oracle_pool_double_base(self.h, out.ctypes.data, a.ctypes.data, b.ctypes.data, G, H, n, C.byref(ok))
        assert ok.value == 1
        return dt, out


def cpu_msm_baseline(n, threads):
    """Oracle Pippenger (reference algorithm) on `n` pairs over `threads` persistent host threads: (points/s, seconds)."""
    pool = CpuPool(threads)
    sc, pts = pool.msm_inputs(n)
    dt, _ = pool.msm(sc, pts, n, slice_pairs=n if threads == 1 else 8192)
    pool.close()
    return n / dt, dt


def cpu_verify_baseline(nsigs, threads, batch=256):
    pool = CpuPool(threads)
    m, s, k = pool.verify_inputs(nsigs)
    dt = pool.verify_batches(m, s, k, nsigs, batch)
    pool.close()
    return nsigs / dt, dt


def run_reference(args, rank, world):
    """The reference arm: the CPU oracle (C restatement of the reference's serial u64 backend; the Rust reference cannot
    be built in this image) on ALL host threads, same metric and -- for the MSM -- the same configuration as the GPU arm
    at N = 1 (2^20 pairs per step), persistent worker threads, sub-MSMs of 2^13 pairs."""
    if rank != 0:
        return None
    threads, quota = effective_cpus()
    steps = max(1, args.steps)
    pool = CpuPool(threads)
    vals = []
    if args.workload == "verify":
        nsigs = 256 * threads * 4
        m, s, k = pool.verify_inputs(nsigs)
        for _ in range(min(args.warmup, 1)):
            pool.verify_batches(m, s, k, nsigs)
        t0 = time.perf_counter()
        for _ in range(steps):
            vals.append(nsigs / pool.verify_batches(m, s, k, nsigs))
        el = time.perf_counter() - t0
        metric, unit = "Ed25519 verify_batch signatures/sec", "sigs/s"
        sample = "each step: %d independent verify_batch calls of 256 signatures (the reference's largest published batch size) pulled by %d persistent threads" % (nsigs // 256, threads)
        config = {"workload": "ed25519_verify_batch", "batch": 256, "signatures_per_step": nsigs}
        same = False
    else:
        n_total = (args.pairs_per_gpu or ((1 << 20) if world == 1 else (1 << 21))) * world      # the GPU arm's configuration
        n = min(n_total, 1 << 22)                           # bounded sample per step (the rate does not depend on n beyond 2^13-pair slices)
        sc, pts = pool.msm_inputs(n)
        for _ in range(min(args.warmup, 1)):
            pool.msm(sc, pts, n)
        t0 = time.perf_counter()
        for _ in range(steps):
            vals.append(n / pool.msm(sc, pts, n)[0])
        el = time.perf_counter() - t0
        metric, unit = "Pippenger MSM points/sec", "points/s"
        sample = ("each step: one 2^%d-pair MSM (the GPU arm's configuration%s) as %d independent reference Pippenger sub-MSMs of 8192 pairs "
                  "(w = 8) pulled by %d persistent threads, partial sums added" % (n.bit_length() - 1, "" if n == n_total else ", capped at 2^22 pairs per step", (n + 8191) // 8192, threads))
        config = {"workload": "pippenger_msm", "pairs_total": n_total, "pairs_per_gpu": n_total // world, "pairs_per_step_sampled": n,
                  "point_format": "extended radix-2^51 limbs (160 B)"}
        same = n == n_total
    pool.close()
    val = statistics.mean(vals)
    return {"impl": "reference", "metric": metric, "value": val, "unit": unit, "n_gpus": world, "steps": steps,
            "warmup": args.warmup, "ms_per_step": el / steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64 limbs (radix 2^51), exact", "data": "synthetic", "config": config,
            "same_config_as_gpu_arm": same,
            "cpu_baseline": {"value": val, "unit": unit, "cores": threads, "logical_cpus": os.cpu_count(), "physical_cores": physical_cores(),
                             "cgroup_cpu_quota": quota, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "CPU oracle = C restatement of the reference's serial u64 backend (Rust toolchain absent: oracle/_ref cannot be built)"}


# ------------------------------------------------------------------------------------------ main
def main():
    # Pinned host buffers are filled by ONE thread, so that their pages sit on one NUMA node (first touch): a buffer filled
    # by torch's CPU thread pool is spread over both sockets and crosses PCIe at 34.5 GB/s instead of 55.5 GB/s on these boxes
    # (tools/pcie_probe.py, profiles/pcie_probe_r2.json).  Nothing else in this process uses torch's CPU threads.
    try:
        import torch
        torch.set_num_threads(1)
    except ImportError:
        pass
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="msm", choices=["msm", "verify"])
    ap.add_argument("--pairs-per-gpu", type=int, default=0)
    ap.add_argument("--sigs-per-gpu", type=int, default=0)
    ap.add_argument("--verify-batch-size", type=int, default=256,
                    help="verify workload: signatures per independent verify_batch (reference-exact transcripts and verdicts, one per batch); "
                         "0 = ONE verdict over all signatures with --transcript-chunk")
    ap.add_argument("--transcript-chunk", type=int, default=64, help="signatures per Merlin transcript in the single-call verify_batch leg (0 = the reference's single transcript)")
    ap.add_argument("--exact-transcript-leg", type=int, default=1, help="also time ONE 2^18-signature verify_batch call with the reference's single transcript")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary verify_batch / cpu_baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed calls returned in their last step (device-resident and from host buffers) "
                         "as DIR/<name>.npy, float64")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank, world, local = dist_env()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the engine's results: it needs --impl b200")
    if args.impl == "reference":
        line = run_reference(args, rank, world)
        if line is not None:
            print(json.dumps(line), flush=True)
        return
    if world != args.gpus and rank == 0:
        print("bench: --gpus %d but WORLD_SIZE=%d (launch with torch.distributed.run)" % (args.gpus, world), file=sys.stderr)
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench: no CUDA device; the engine has no CPU fallback")
    outputs = {}
    if args.workload == "verify":
        line = run_verify(args, rank, world, local, outputs=outputs)
    else:
        line, eng, wl = run_msm(args, rank, world, local, outputs=outputs)
        if not args.no_extras and world > 1:
            # BASELINE.json's metric names verify_batch at 1/2/4/8 GPUs too: independent replicas, one batch per GPU
            v = run_verify(args, rank, world, local, eng=eng, steps=min(args.steps, 5), warmup=3)
            if rank == 0:
                line["verify_batch"] = {k: v[k] for k in ("metric", "value", "unit", "n_gpus", "ms_per_step", "scaling", "e2e", "config", "gpu_launches", "roofline")}
        if not args.no_extras and world == 1:
            line["msm_2p21_pairs"] = run_msm_like_for_like(eng, 1 << 21, min(args.steps, 20))
            line["msm_two_callers"] = run_msm_two_callers(eng, wl, local, min(2 * args.steps, 60))
            line["msm_compressed_input"] = run_msm_compressed(eng, wl)
            line["small_msm_latency"] = run_small_latency(eng)
            line["msm_precomputed"] = run_precomputed(eng, wl)
            line["codecs"] = run_codecs(eng, wl)
            # primary: 2^14 independent batches of 256 (per-batch verdicts, the reference's transcript for every batch)
            v = run_verify(args, rank, world, local, eng=eng, steps=min(args.steps, 5), warmup=3)
            line["verify_batch"] = {k: v[k] for k in ("metric", "value", "unit", "ms_per_step", "e2e", "config", "gpu_launches", "roofline")}
            # the same with every public key different (no key de-duplication possible)
            v2 = run_verify(args, rank, world, local, eng=eng, steps=3, warmup=3, nkeys=1 << 30)
            line["verify_batch"]["all_distinct_keys"] = {k: v2[k] for k in ("value", "unit", "ms_per_step", "e2e")}
            # ... and with the VerifyingKeys' points passed in, as the reference's verify_batch receives them (batch.rs:236-238)
            v2p = run_verify(args, rank, world, local, eng=eng, steps=3, warmup=3, nkeys=1 << 30, key_points=True)
            line["verify_batch"]["all_distinct_keys_with_key_points"] = {k: v2p[k] for k in ("value", "unit", "ms_per_step", "e2e")}
            # ONE verdict over all 2^22 signatures with the opt-in chunked transcript (NOT reference-equivalent on inputs
            # with small-order components: include/dalek_b200.h)
            v3 = run_verify(args, rank, world, local, eng=eng, steps=3, warmup=3, batch_size=0)
            line["verify_batch"]["one_verdict_chunked_transcript"] = dict({k: v3[k] for k in ("value", "unit", "ms_per_step", "e2e")},
                                                                          transcript=v3["config"]["transcript"])
            # the single-call leg again with the reference's ONE transcript over all 2^22 signatures (the default of the API):
            # a strictly sequential sponge, one GPU thread -- timed once
            if args.exact_transcript_leg:
                line["verify_batch"]["single_reference_transcript"] = run_verify_exact_once(eng, args)
            # one verdict per signature (VerifyingKey::verify semantics: R' recomputed and compared as bytes)
            v4 = run_verify(args, rank, world, local, eng=eng, steps=2, warmup=1, each=True)
            line["verify_each"] = {k: v4[k] for k in ("value", "unit", "ms_per_step", "e2e")}
            line["verify_each"]["path"] = ("1024 distinct keys: per-key comb tables (64 x 8 multiples of every key resident in L2), "
                                           "128 mixed additions and no doubling per signature")
            # every key different: nothing to tabulate, the 252-doubling double-scalar multiplication per signature
            v5 = run_verify(args, rank, world, local, eng=eng, steps=1, warmup=1, each=True, nkeys=1 << 30)
            line["verify_each"]["all_distinct_keys"] = {k: v5[k] for k in ("value", "unit", "ms_per_step", "e2e")}
            pool = CpuPool(1)
            m_, s_, k_ = pool.verify_inputs(2048)
            cdt = pool.verify_each(m_, s_, k_, 2048)
            pool.close()
            line["verify_each"]["cpu_baseline"] = {"value": 2048 / cdt, "unit": "sigs/s", "cores": 1, "kind": "port",
                                                   "sample": "2048 oracle VerifyingKey::verify calls, 1 thread (%.1f s)" % cdt}
            line["ristretto_double_base"] = run_double_base(eng)
    if rank == 0 and world == 1 and not args.no_extras:
        threads = 1
        if args.workload == "verify":
            val, dt = cpu_verify_baseline(4096, 1)
            line["cpu_baseline"] = {"value": val, "unit": "sigs/s", "cores": 1, "kind": "port",
                                    "sample": "16 oracle verify_batch calls of 256 signatures, 1 thread (%.1f s)" % dt}
        else:
            val, dt = cpu_msm_baseline(1 << 19, threads)
            line["cpu_baseline"] = {"value": val, "unit": "points/s", "cores": 1, "kind": "port",
                                    "sample": "one 2^19-pair oracle Pippenger MSM (w=8), 1 thread (%.1f s)" % dt}
            if "verify_batch" in line:
                v2, dt2 = cpu_verify_baseline(4096, 1)
                line["verify_batch"]["cpu_baseline"] = {"value": v2, "unit": "sigs/s", "cores": 1, "kind": "port",
                                                        "sample": "16 oracle verify_batch calls of 256 signatures, 1 thread (%.1f s)" % dt2}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1 and dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
