"""GPU tests of the batched vartime MSM (csrc/msm_batch.cu): m independent optional_multiscalar_mul calls in one call,
each result byte for byte the single call's on its slice, against the oracle."""
import ctypes as C
import random

import pytest

import pyref
from test_gpu_msm import gen_case

pytestmark = pytest.mark.gpu

LENGTHS = [0, 1, 2, 3, 7, 8, 9, 64, 189, 190, 191, 256, 500, 1000]


@pytest.fixture(scope="module")
def eng():
    import curve25519_dalek_b200 as pkg
    e = pkg.Engine(0)
    yield e
    e.close()


def _offsets(lengths):
    offs = [0]
    for n in lengths:
        offs.append(offs[-1] + n)
    return offs


def _ext(oracle, points):
    ext = (C.c_uint64 * (20 * max(1, len(points))))()
    for i, p in enumerate(points):
        q = oracle.sub(oracle.add(oracle.double(p), p), oracle.double(p))      # Z != 1
        for k, v in enumerate(oracle.p3_limbs(q)):
            ext[20 * i + k] = v
    return ext


@pytest.fixture(scope="module")
def case(oracle):
    scalars, points, wants = [], [], []
    for k, n in enumerate(LENGTHS):
        s, p = gen_case(oracle, n, seed=1000 + k)
        scalars += s; points += p
        wants.append(oracle.compress(oracle.msm("optional", s, p)) if n else oracle.compress(oracle.identity()))
    return scalars, points, wants


@pytest.mark.parametrize("fmt", [0, 1])
def test_batch_parity_with_oracle_and_single_calls(eng, oracle, case, fmt):
    scalars, points, wants = case
    offs = _offsets(LENGTHS)
    sb = b"".join(scalars)
    pb = b"".join(oracle.compress(p) for p in points) if fmt == 0 else _ext(oracle, points)
    for T in (1, 190, 2**31 - 1, None):                  # everything bucket, split at the reference's 190, all Straus, default
        if T is not None:
            eng.set_option("batch_bucket_min", T)
        try:
            rc, res, limbs = eng.edwards_vartime_msm_batch(sb, pb, offs, point_fmt=fmt, want_limbs=True)
        finally:
            eng.set_option("batch_bucket_min", 65536)
        assert rc == 0 and res == wants, T
        for k, w in enumerate(wants):
            assert oracle.compress(oracle.p3_from_limbs(limbs[k])) == w                        # projectively equal
    for k in range(len(LENGTHS)):
        a, b = offs[k], offs[k + 1]
        one = b"".join(oracle.compress(p) for p in points[a:b]) if fmt == 0 else _ext(oracle, points[a:b])
        rc, got, _ = eng.edwards_vartime_msm(b"".join(scalars[a:b]), one, b - a, point_fmt=fmt)
        assert rc == 0 and got == wants[k]


@pytest.mark.parametrize("T", [200, 65536])
def test_batch_none_isolation(eng, oracle, case, T):
    """A bad point marks its own segment only: first, a middle one, the last, and (T = 200) bucket-path segments."""
    scalars, points, wants = case
    offs = _offsets(LENGTHS)
    comp = [oracle.compress(p) for p in points]
    bad_segs = [1, 7, 11, len(LENGTHS) - 1]                 # lengths 1, 64, 256 (bucket path at T = 200), 1000
    for k in bad_segs:
        comp[offs[k + 1] - 1] = (2).to_bytes(32, "little")  # y = 2 is not on the curve
    eng.set_option("batch_bucket_min", T)
    try:
        rc, res, limbs = eng.edwards_vartime_msm_batch(b"".join(scalars), b"".join(comp), offs, want_limbs=True)
    finally:
        eng.set_option("batch_bucket_min", 65536)
    assert rc == 1
    for k, w in enumerate(wants):
        if k in bad_segs:
            assert res[k] is None and limbs[k] == [0] * 20
        else:
            assert res[k] == w, k


def _pool_case(oracle, rnd, lengths, pool=64):
    """Points from a pool of t_j B, so that sum s_i (t_i B) = (sum s_i t_i) B gives every segment's result cheaply."""
    B = oracle.basepoint()
    pool_t = [rnd.randrange(pyref.L) for _ in range(pool)]
    pool_p = [oracle.compress(oracle.scalarmul(t.to_bytes(32, "little"), B)) for t in pool_t]
    n = sum(lengths)
    idx = [rnd.randrange(pool) for _ in range(n)]
    ss = [rnd.randrange(pyref.L) for _ in range(n)]
    wants, a = [], 0
    for ln in lengths:
        k = sum(ss[i] * pool_t[idx[i]] for i in range(a, a + ln)) % pyref.L
        wants.append(oracle.compress(oracle.scalarmul(k.to_bytes(32, "little"), B)))
        a += ln
    import numpy as np
    sb = np.frombuffer(b"".join(s.to_bytes(32, "little") for s in ss), dtype=np.uint8).copy()
    pb = np.frombuffer(b"".join(pool_p[j] for j in idx), dtype=np.uint8).copy()
    return sb, pb, wants


def test_batch_4096_msms_of_64_identity_and_launches(eng, oracle):
    """4096 x 64 pairs: every segment checked by sum s_i (t_i B) == (sum s_i t_i) B; the call takes a bounded number of
    kernel launches whatever m is; the _dev form equals the host form."""
    import torch
    rnd = random.Random(4096)
    lengths = [64] * 4096
    sb, pb, wants = _pool_case(oracle, rnd, lengths)
    offs = _offsets(lengths)
    l0 = eng.launch_count()
    rc, res, _ = eng.edwards_vartime_msm_batch(sb, pb, offs)
    launches = eng.launch_count() - l0
    assert launches <= 8
    assert rc == 0 and res == wants
    # the same 2^18 pairs as 16 MSMs of 2^14: the same number of launches
    few = [1 << 14] * 16
    sb16, pb16, wants16 = _pool_case(oracle, rnd, few)
    l0 = eng.launch_count()
    rc, res16, _ = eng.edwards_vartime_msm_batch(sb16, pb16, _offsets(few))
    assert eng.launch_count() - l0 == launches
    assert rc == 0 and res16 == wants16
    ds, dp = torch.from_numpy(sb).cuda(), torch.from_numpy(pb).cuda()
    rc, res2, _ = eng.edwards_vartime_msm_batch(ds.data_ptr(), dp.data_ptr(), offs, device_ptrs=True)
    torch.cuda.synchronize()
    assert rc == 0 and res2 == wants
    assert eng.last_call_ms() > 0


def test_batch_mixed_sizes_host_pieces(eng, oracle):
    """One 2^17 segment (bucket path), one 2^15 and 1000 small ones, over 2^18 pairs in all, from host buffers."""
    rnd = random.Random(17)
    lengths = [rnd.randrange(0, 200) for _ in range(500)] + [1 << 17] + [rnd.randrange(0, 200) for _ in range(300)] + \
        [1 << 15] + [rnd.randrange(0, 200) for _ in range(200)]
    assert sum(lengths) > 1 << 18
    sb, pb, wants = _pool_case(oracle, rnd, lengths)
    rc, res, _ = eng.edwards_vartime_msm_batch(sb, pb, _offsets(lengths))
    assert rc == 0 and res == wants


def test_ristretto_batch(eng, oracle):
    rnd = random.Random(5)
    B = oracle.basepoint()
    lengths = [0, 1, 5, 64, 189, 190, 300]
    n = sum(lengths)
    pts = [oracle.ristretto_compress(oracle.scalarmul(rnd.randrange(pyref.L).to_bytes(32, "little"), B)) for _ in range(n)]
    sc = [rnd.randrange(pyref.L).to_bytes(32, "little") for _ in range(n)]
    offs = _offsets(lengths)
    wants = []
    for k in range(len(lengths)):
        a, b = offs[k], offs[k + 1]
        w = oracle.ristretto_compress(oracle.msm("optional", sc[a:b], [oracle.ristretto_decompress(p) for p in pts[a:b]])) if b > a \
            else oracle.ristretto_compress(oracle.identity())
        rc, single = eng.ristretto_vartime_msm(b"".join(sc[a:b]), b"".join(pts[a:b]), b - a)
        assert rc == 0 and single == w
        wants.append(w)
    rc, res = eng.ristretto_vartime_msm_batch(b"".join(sc), b"".join(pts), offs)
    assert rc == 0 and res == wants
    bad = list(pts); bad[offs[3]] = (1).to_bytes(32, "little")          # negative s: does not decode
    rc, res = eng.ristretto_vartime_msm_batch(b"".join(sc), b"".join(bad), offs)
    assert rc == 1 and res[3] is None and res[:3] == wants[:3] and res[4:] == wants[4:]


def test_invalid_offsets_then_valid_call(eng, oracle, case):
    from curve25519_dalek_b200 import EngineError
    scalars, points, wants = case
    sb, pb = b"".join(scalars), b"".join(oracle.compress(p) for p in points)
    for offs in ([1, 5], [0, 5, 3], [0, 2**31]):
        with pytest.raises(EngineError):
            eng.edwards_vartime_msm_batch(sb, pb, offs)
    with pytest.raises(EngineError):
        eng.edwards_vartime_msm_batch(sb, pb, [0, 1], point_fmt=7)
    assert eng.edwards_vartime_msm_batch(sb, pb, [0]) == (0, [], None)              # m = 0
    with pytest.raises(ValueError):
        eng.edwards_vartime_msm_batch(sb, pb, [])                                    # no m + 1 offsets
    with pytest.raises(EngineError, match="Ristretto"):
        eng.edwards_vartime_msm_batch(sb, pb, [0, 1], point_fmt=2)
    rc, res, _ = eng.edwards_vartime_msm_batch(sb, pb, _offsets(LENGTHS))
    assert rc == 0 and res == wants


def test_python_wrappers(eng, oracle, case):
    import curve25519_dalek_b200 as pkg
    scalars, points, wants = case
    offs = _offsets(LENGTHS)
    comp = [oracle.compress(p) for p in points]
    msms = [(scalars[offs[k]:offs[k + 1]], comp[offs[k]:offs[k + 1]]) for k in range(len(LENGTHS))]
    assert pkg.EdwardsPoint.optional_multiscalar_mul_batch(msms, engine=eng) == wants
    msms[2] = (msms[2][0], [None] + msms[2][1][1:])
    got = pkg.EdwardsPoint.optional_multiscalar_mul_batch(msms, engine=eng)
    assert got[2] is None and got[:2] == wants[:2] and got[3:] == wants[3:]
    with pytest.raises(AssertionError):
        pkg.EdwardsPoint.optional_multiscalar_mul_batch([(scalars[:2], comp[:3])], engine=eng)
    B = oracle.basepoint()
    rp = [oracle.ristretto_compress(oracle.scalarmul((i + 2).to_bytes(32, "little"), B)) for i in range(6)]
    rs = [(i + 1).to_bytes(32, "little") for i in range(6)]
    want = pkg.RistrettoPoint.vartime_multiscalar_mul(rs, rp, engine=eng)
    assert pkg.RistrettoPoint.optional_multiscalar_mul_batch([(rs, rp), (rs[:1], [None])], engine=eng) == [want, None]


@pytest.mark.parametrize("n", [10, 16, 100])
def test_single_straus_call_with_even_scalars(eng, oracle, n):
    """Every scalar even: no warp of the single call's Straus path adds at bit 0.  Its result, and the batch's, must
    still be the oracle's (the last doubling refreshes T, which the sum of the warp accumulators reads)."""
    rnd = random.Random(n)
    scalars, points = gen_case(oracle, n, seed=77 + n, special=False)
    scalars = [(2 * rnd.randrange(pyref.L // 2)).to_bytes(32, "little") for _ in range(n)]
    want = oracle.compress(oracle.msm("optional", scalars, points))
    comp = b"".join(oracle.compress(p) for p in points)
    rc, got, _ = eng.edwards_vartime_msm(b"".join(scalars), comp, n)
    assert rc == 0 and got == want
    rc, res, _ = eng.edwards_vartime_msm_batch(b"".join(scalars), comp, [0, n])
    assert rc == 0 and res == [want]
