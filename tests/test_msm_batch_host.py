"""The batched vartime MSM's host planner and its segmented Straus group routine (csrc/msm_batch.cuh), executed on the
CPU (tests/host/msm_batch_host_check.cpp: the emulated warp of w4_host_check.cpp, operand-rule assertions on) against
the oracle.  CPU only: the emulation is test infrastructure, not a fallback of the product."""
import ctypes as C
import os
import random
import subprocess

import pytest

import pyref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def mb():
    host = os.path.join(ROOT, "tests", "host")
    src = os.path.join(host, "msm_batch_host_check.cpp")
    so = os.path.join(host, "libmsmbatchhost.so")
    csrc = os.path.join(ROOT, "curve25519_dalek_b200", "csrc")
    deps = [src, os.path.join(host, "w4_host_check.cpp")] + [os.path.join(csrc, f) for f in (
        "fe.cuh", "fe64.cuh", "ge.cuh", "ge64.cuh", "warp4_f64.cuh", "straus_vt.cuh", "msm_batch.cuh", "transcript_warp.cuh",
        "constants.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", so, src, "-lpthread"])
    lib = C.CDLL(so)
    lib.h_plan.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64, C.c_int, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.h_straus_segmented.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_void_p, C.c_size_t, C.c_uint32]
    return lib


def _offsets(lengths):
    offs = (C.c_uint64 * (len(lengths) + 1))()
    for k, n in enumerate(lengths):
        offs[k + 1] = offs[k] + n
    return offs


def plan(mb, lengths, bucket_min, sm=148, cap=1 << 20):
    offs = _offsets(lengths)
    path = (C.c_uint8 * max(1, len(lengths)))()
    npieces, p = C.c_uint64(), C.c_uint32()
    rc = mb.h_plan(offs, len(lengths), bucket_min, sm, cap, path, C.byref(npieces), C.byref(p))
    assert rc == 1, rc
    return list(path)[:len(lengths)], npieces.value, p.value


def test_plan_threshold_sides(mb):
    """Lengths T-1, T and T+1 take Straus, bucket, bucket; empty segments are Straus segments of zero tasks."""
    for T in (1, 2, 190, 4096, 1 << 16):
        lengths = [0, T - 1, T, T + 1, 0, T - 1, 0]
        path, _, _ = plan(mb, lengths, T)
        assert path == [0, 0, 1, 1, 0, 0, 0]


def test_plan_invariants(mb):
    """Every pair is covered exactly once, pieces end at segment boundaries, Straus pieces stay within the piece size
    (a longer segment takes the bucket pipeline whatever the threshold), empty segments are planned, and the pairs per
    task follow the total."""
    rnd = random.Random(7)
    for trial in range(60):
        m = rnd.choice((1, 2, 5, 40, 300))
        lengths = [rnd.choice((0, 0, 1, 2, 3, 7, 64, 189, 190, 1000, rnd.randrange(1, 5000))) for _ in range(m)]
        T = rnd.choice((1, 100, 190, 2000, 2**31 - 1))
        cap = rnd.choice((1, 50, 1000, 1 << 20))
        plan(mb, lengths, T, sm=rnd.choice((1, 148)), cap=cap)
    assert plan(mb, [], 190)[1] == 0
    assert plan(mb, [0, 0, 0], 190)[1] == 1
    assert plan(mb, [10] * 100, 190, cap=100)[1] == 10          # pieces of ten segments
    path, npieces, _ = plan(mb, [500, 10, 10], 2**31 - 1, cap=100)
    assert path == [1, 0, 0] and npieces == 2                      # longer than a piece: the bucket pipeline
    assert plan(mb, [64] * 4096, 1 << 16)[2] == 16                 # 2^18 pairs on 148 SMs: 16 pairs per task
    assert plan(mb, [64] * 4, 1 << 16)[2] == 1                     # few pairs: one per task, every SM busy


def _points(oracle, rnd, n):
    B = oracle.basepoint()
    pts = [oracle.scalarmul(rnd.randrange(pyref.L).to_bytes(32, "little"), B) for _ in range(n)]
    special = [oracle.identity(), oracle.decompress((pyref.p - 1).to_bytes(32, "little")),    # identity, order 2
               oracle.decompress((0).to_bytes(32, "little"))]                                 # order 4
    for k, q in enumerate(special):
        if 3 * k + 1 < n:
            pts[3 * k + 1] = q
    return pts


def _want(oracle, scalars, points):
    """sum s_i P_i by exact integer arithmetic (scalars up to 2^256 - 1: v = lo + 2^252 hi)."""
    acc = oracle.identity()
    for sc, pt in zip(scalars, points):
        v = int.from_bytes(sc, "little")
        lo = oracle.scalarmul((v % 2**252).to_bytes(32, "little"), pt)
        hi = oracle.mul_by_pow_2(oracle.scalarmul((v >> 252).to_bytes(32, "little"), pt), 252)
        acc = oracle.add(acc, oracle.add(lo, hi))
    return oracle.compress(acc)


@pytest.mark.parametrize("p", [1, 2, 3, 5, 16, 33])
def test_segmented_straus_matches_oracle(mb, oracle, p):
    """straus_task_group: one accumulator per task of <= p pairs, uniform op stream; warps span several segments and the
    last warp is partly filled.  Edge scalars 0, l-1, 2^255-1, 2^256-1; identity and small-order points."""
    rnd = random.Random(100 + p)
    lengths = [0, 1, p + 1, 2, 0, p, 3] if p > 1 else [0, 1, 2, 2, 0, 1, 3]
    n = sum(lengths)
    pts = _points(oracle, rnd, n)
    edge = [0, pyref.L - 1, 2**255 - 1, 2**256 - 1]
    scalars = [(edge[i] if i < 4 else rnd.randrange(2**256 if i % 5 == 0 else pyref.L)).to_bytes(32, "little")
               for i in range(n)]
    rnd.shuffle(scalars)
    offs = _offsets(lengths)
    out = (C.c_uint8 * (32 * len(lengths)))()
    assert mb.h_straus_segmented(out, b"".join(scalars), b"".join(oracle.compress(q) for q in pts), offs, len(lengths), p) == 1
    got = bytes(out)
    for k in range(len(lengths)):
        a, b = offs[k], offs[k + 1]
        assert got[32 * k:32 * k + 32] == _want(oracle, scalars[a:b], pts[a:b]), (p, k)


@pytest.mark.parametrize("n", [10, 16])
def test_vartime_straus_with_even_scalars(mb, oracle, n):
    """straus_vt.cuh when no group of a warp adds at bit 0 (every scalar even): the last doubling must still refresh T,
    which the sum of the warp's accumulators reads.  The single-call Straus path and the batch must agree with the oracle."""
    rnd = random.Random(n)
    pts = _points(oracle, rnd, n)
    scalars = [(2 * rnd.randrange(pyref.L // 2)).to_bytes(32, "little") for _ in range(n)]
    want = _want(oracle, scalars, pts)
    enc = b"".join(oracle.compress(q) for q in pts)
    out = (C.c_uint8 * 32)()
    mb.h_straus_vartime.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_int]
    assert mb.h_straus_vartime(out, b"".join(scalars), enc, n) == 1
    assert bytes(out) == want
    assert mb.h_straus_segmented(out, b"".join(scalars), enc, _offsets([n]), 1, 16) == 1
    assert bytes(out) == want
