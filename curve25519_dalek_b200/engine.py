"""ctypes binding of libdalek_b200.so plus thin classes mirroring the reference's trait surface."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
POINTS_RISTRETTO = 2
POINTS_COMPRESSED = 0
POINTS_EXTENDED = 1

_lib = None


def library_path():
    # DALEK_B200_LIB selects an alternative build of the same engine (tuning experiments only)
    return os.environ.get("DALEK_B200_LIB") or os.path.join(HERE, "libdalek_b200.so")


def load_library():
    """Load the CUDA engine.  Fails loudly if the extension has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError("libdalek_b200.so is missing: run `python -m curve25519_dalek_b200.build` "
                           "(or __graft_entry__.build()); there is no CPU fallback")
    lib = C.CDLL(path)
    vp, sz, u8p, u64p = C.c_void_p, C.c_size_t, C.c_char_p, C.c_void_p
    lib.dalek_b200_init.argtypes = [C.c_int, C.POINTER(vp)]
    lib.dalek_b200_destroy.argtypes = [vp]
    lib.dalek_b200_destroy.restype = None
    lib.dalek_b200_last_error.argtypes = [vp]
    lib.dalek_b200_last_error.restype = C.c_char_p
    lib.dalek_b200_set_option.argtypes = [vp, C.c_char_p, C.c_long]
    lib.dalek_b200_launch_count.argtypes = [vp]
    lib.dalek_b200_launch_count.restype = C.c_uint64
    lib.dalek_b200_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_int)]
    lib.dalek_b200_last_call_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.dalek_b200_last_stage_ms.argtypes = [vp, C.c_char_p, C.POINTER(C.c_float)]
    for name in ("dalek_b200_edwards_vartime_msm", "dalek_b200_edwards_ct_msm", "dalek_b200_edwards_vartime_msm_dev"):
        getattr(lib, name).argtypes = [vp, vp, vp, C.c_int, sz, vp, vp]
    lib.dalek_b200_edwards_vartime_msm_batch.argtypes = [vp, vp, vp, C.c_int, vp, sz, vp, vp, vp]
    lib.dalek_b200_edwards_vartime_msm_batch_dev.argtypes = [vp, vp, vp, C.c_int, vp, sz, vp, vp, vp]
    lib.dalek_b200_ristretto_vartime_msm_batch.argtypes = [vp, vp, vp, vp, sz, vp, vp]
    lib.dalek_b200_msm_window_count.argtypes = [vp, sz]
    lib.dalek_b200_edwards_msm_partial.argtypes = [vp, vp, vp, C.c_int, sz, sz, vp]
    lib.dalek_b200_edwards_msm_partial_dev.argtypes = [vp, vp, vp, C.c_int, sz, sz, vp]
    lib.dalek_b200_edwards_msm_combine.argtypes = [vp, vp, C.c_int, sz, vp, vp]
    lib.dalek_b200_edwards_msm_combine_dev.argtypes = [vp, vp, C.c_int, sz, vp, vp]
    lib.dalek_b200_edwards_msm_partial_async.argtypes = [vp, vp, vp, C.c_int, sz, sz, vp]
    lib.dalek_b200_edwards_msm_partial_dev_async.argtypes = [vp, vp, vp, C.c_int, sz, sz, vp]
    lib.dalek_b200_msm_partial_bytes.argtypes = [vp, sz]
    lib.dalek_b200_msm_partial_bytes.restype = sz
    lib.dalek_b200_stream.argtypes = [vp]
    lib.dalek_b200_stream.restype = vp
    lib.dalek_b200_init_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    lib.dalek_b200_destroy_multi.argtypes = [vp]
    lib.dalek_b200_destroy_multi.restype = None
    lib.dalek_b200_multi_device_count.argtypes = [vp]
    lib.dalek_b200_multi_ctx.argtypes = [vp, C.c_int]
    lib.dalek_b200_multi_ctx.restype = vp
    lib.dalek_b200_multi_last_error.argtypes = [vp]
    lib.dalek_b200_multi_last_error.restype = C.c_char_p
    lib.dalek_b200_edwards_vartime_msm_multi.argtypes = [vp, vp, vp, C.c_int, sz, vp, vp]
    lib.dalek_b200_ristretto_double_base_batch.argtypes = [vp, vp, vp, vp, vp, sz, vp]
    lib.dalek_b200_ristretto_vartime_msm.argtypes = [vp, vp, vp, sz, vp]
    lib.ed25519_b200_verify_batch.argtypes = [vp, vp, vp, vp, vp, sz]
    lib.ed25519_b200_verify_batch_flat.argtypes = [vp, vp, vp, vp, vp, sz]
    lib.ed25519_b200_verify_batch_flat_dev.argtypes = [vp, vp, vp, vp, vp, sz, sz]
    lib.ed25519_b200_verify_batches_flat.argtypes = [vp, vp, vp, vp, vp, sz, sz, vp]
    lib.ed25519_b200_verify_batch_flat_points.argtypes = [vp, vp, vp, vp, vp, vp, sz]
    lib.ed25519_b200_verify_batch_flat_points_dev.argtypes = [vp, vp, vp, vp, vp, vp, sz]
    lib.ed25519_b200_verify_batches_flat_points.argtypes = [vp, vp, vp, vp, vp, vp, sz, sz, vp]
    lib.ed25519_b200_verify_batches_flat_points_dev.argtypes = [vp, vp, vp, vp, vp, vp, sz, sz, vp]
    lib.ed25519_b200_verify_batches_flat_dev.argtypes = [vp, vp, vp, vp, vp, sz, sz, vp]
    lib.dalek_b200_precomp_new.argtypes = [vp, vp, C.c_int, sz, C.POINTER(vp)]
    lib.dalek_b200_precomp_len.argtypes = [vp]
    lib.dalek_b200_precomp_len.restype = sz
    lib.dalek_b200_precomp_destroy.argtypes = [vp]
    lib.dalek_b200_precomp_destroy.restype = None
    lib.dalek_b200_precomp_mixed_msm.argtypes = [vp, vp, vp, sz, vp, vp, C.c_int, sz, vp, vp]
    lib.dalek_b200_edwards_decompress_batch.argtypes = [vp, vp, sz, vp, vp]
    lib.dalek_b200_ristretto_decompress_batch.argtypes = [vp, vp, sz, vp, vp]
    lib.dalek_b200_edwards_compress_batch.argtypes = [vp, vp, sz, vp]
    lib.dalek_b200_ristretto_double_and_compress_batch.argtypes = [vp, vp, sz, vp]
    lib.ed25519_b200_verify_each_flat.argtypes = [vp, vp, vp, vp, vp, sz, C.c_int, vp]
    lib.ed25519_b200_verify_each_flat_dev.argtypes = [vp, vp, vp, vp, vp, sz, C.c_int, vp]
    lib.dalek_b200_scalar_from_wide_batch.argtypes = [vp, vp, sz, vp]
    lib.dalek_b200_scalar_invert_batch.argtypes = [vp, vp, sz, vp, vp]
    lib.ed25519_b200_last_zs.argtypes = [vp, vp, sz]
    lib.dalek_b200_edwards_mul_base_batch.argtypes = [vp, vp, sz, vp, vp]
    lib.ed25519_b200_sign_batch_flat.argtypes = [vp, vp, vp, vp, sz, vp, vp]
    _lib = lib
    return lib


class EngineError(RuntimeError):
    pass


class SignatureError(Exception):
    """ed25519_dalek::SignatureError (ed25519-dalek/src/errors.rs:23-53): `.kind` is one of
    'Verify', 'ArrayLength', 'ScalarFormat', 'PointDecompression'."""
    KINDS = {1: "Verify", 2: "ArrayLength", 3: "ScalarFormat", 4: "PointDecompression"}

    def __init__(self, code):
        self.code = code
        self.kind = self.KINDS.get(code, "Unknown")
        super().__init__(self.kind)


def _ptr(obj):
    """Host pointer of bytes / bytearray / numpy array / torch CPU tensor / int address."""
    if obj is None:
        return None
    if isinstance(obj, int):
        return obj
    if isinstance(obj, bytes):
        return C.cast(C.c_char_p(obj), C.c_void_p).value      # caller keeps `obj` alive across the call
    if isinstance(obj, bytearray):
        return C.addressof((C.c_char * len(obj)).from_buffer(obj)) if len(obj) else None
    if isinstance(obj, C.Array):
        return C.addressof(obj)
    if hasattr(obj, "data_ptr"):
        return obj.data_ptr()
    if hasattr(obj, "ctypes"):
        return obj.ctypes.data
    raise TypeError("unsupported buffer type %r" % type(obj))


class Engine:
    """One engine context bound to one CUDA device (dalek_b200_init)."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.dalek_b200_init(device, C.byref(h))
        if rc != 0:
            raise EngineError("dalek_b200_init(device=%d) failed with %d: no usable sm_100 CUDA device "
                              "(the engine has no CPU fallback)" % (device, rc))
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.dalek_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc < 0:
            raise EngineError("engine error %d: %s" % (rc, self.lib.dalek_b200_last_error(self.h).decode()))
        return rc

    def set_option(self, name, value):
        self._check(self.lib.dalek_b200_set_option(self.h, name.encode(), int(value)))

    def launch_count(self):
        return int(self.lib.dalek_b200_launch_count(self.h))

    def last_call_ms(self):
        """Device time (CUDA events on the engine's stream) of the last MSM / verify_batch call, in ms."""
        ms = C.c_float()
        self.lib.dalek_b200_last_call_ms(self.h, C.byref(ms))
        return float(ms.value)

    def last_stage_ms(self, stage):
        """Device time of a named stage of the last call: 'bucket_accumulate' or 'decompress_R'."""
        ms = C.c_float()
        self._check(self.lib.dalek_b200_last_stage_ms(self.h, stage.encode(), C.byref(ms)))
        return float(ms.value)

    def last_kernel_ms(self):
        ms, n = C.c_float(), C.c_int()
        self.lib.dalek_b200_last_kernel_ms(self.h, C.byref(ms), C.byref(n))
        return ms.value, n.value

    # ---- MSM ----
    def edwards_vartime_msm(self, scalars, points, n, point_fmt=POINTS_COMPRESSED, device_ptrs=False, want_limbs=False):
        """Returns (rc, compressed32, limbs20 or None); rc 1 == None (a point did not decompress)."""
        out = (C.c_uint8 * 32)()
        limbs = (C.c_uint64 * 20)() if want_limbs else None
        fn = self.lib.dalek_b200_edwards_vartime_msm_dev if device_ptrs else self.lib.dalek_b200_edwards_vartime_msm
        keep = (scalars, points)
        rc = self._check(fn(self.h, _ptr(scalars), _ptr(points), point_fmt, n, C.addressof(out),
                            C.addressof(limbs) if want_limbs else None))
        del keep
        return rc, bytes(out), (list(limbs) if want_limbs else None)

    @staticmethod
    def _offsets(offsets):
        if len(offsets) < 1:
            raise ValueError("offsets holds m + 1 entries (at least [0])")
        offs = offsets if isinstance(offsets, C.Array) else (C.c_uint64 * len(offsets))(*[int(o) for o in offsets])
        return offs, len(offs) - 1

    def edwards_vartime_msm_batch(self, scalars, points, offsets, point_fmt=POINTS_COMPRESSED, device_ptrs=False, want_limbs=False):
        """m = len(offsets) - 1 independent MSMs in one call: MSM k takes the pairs [offsets[k], offsets[k+1]) of the flat
        scalars / points buffers (offsets: host, offsets[0] = 0, non-decreasing).  Returns (rc, results, limbs): results[k] is
        the 32-byte compressed result or None (a point of segment k did not decode), limbs (want_limbs) m lists of 20 u64
        (canonical limbs of an equal point; zeros for None); rc 1 if any result is None."""
        offs, m = self._offsets(offsets)
        out = (C.c_uint8 * (32 * max(m, 1)))()
        st = (C.c_uint8 * max(m, 1))()
        limbs = (C.c_uint64 * (20 * max(m, 1)))() if want_limbs else None
        fn = self.lib.dalek_b200_edwards_vartime_msm_batch_dev if device_ptrs else self.lib.dalek_b200_edwards_vartime_msm_batch
        keep = (scalars, points)
        rc = self._check(fn(self.h, _ptr(scalars), _ptr(points), point_fmt, C.addressof(offs), m, C.addressof(out),
                            C.addressof(limbs) if want_limbs else None, C.addressof(st)))
        del keep
        raw = bytes(out)
        res = [None if st[k] else raw[32 * k:32 * k + 32] for k in range(m)]
        return rc, res, ([list(limbs[20 * k:20 * k + 20]) for k in range(m)] if want_limbs else None)

    def ristretto_vartime_msm_batch(self, scalars, points, offsets):
        """The Ristretto form of edwards_vartime_msm_batch (CompressedRistretto points and results): (rc, results)."""
        offs, m = self._offsets(offsets)
        out = (C.c_uint8 * (32 * max(m, 1)))()
        st = (C.c_uint8 * max(m, 1))()
        keep = (scalars, points)
        rc = self._check(self.lib.dalek_b200_ristretto_vartime_msm_batch(self.h, _ptr(scalars), _ptr(points), C.addressof(offs), m,
                                                                         C.addressof(out), C.addressof(st)))
        del keep
        raw = bytes(out)
        return rc, [None if st[k] else raw[32 * k:32 * k + 32] for k in range(m)]

    def edwards_ct_msm(self, scalars, points, n, point_fmt=POINTS_COMPRESSED, want_limbs=False):
        out = (C.c_uint8 * 32)()
        limbs = (C.c_uint64 * 20)() if want_limbs else None
        rc = self._check(self.lib.dalek_b200_edwards_ct_msm(self.h, _ptr(scalars), _ptr(points), point_fmt, n,
                                                            C.addressof(out), C.addressof(limbs) if want_limbs else None))
        return rc, bytes(out), (list(limbs) if want_limbs else None)

    # ---- sharded MSM: n_shard = size of the largest shard, the same on every rank (it selects the window width) ----
    def msm_window_count(self, n_shard):
        return self._check(self.lib.dalek_b200_msm_window_count(self.h, n_shard))

    def msm_partial_bytes(self, n_shard):
        """Bytes of a shard's device record (window accumulators + status word)."""
        return int(self.lib.dalek_b200_msm_partial_bytes(self.h, n_shard))

    def stream_ptr(self):
        """The context's main cudaStream_t as an integer (torch.cuda.ExternalStream(ptr))."""
        return int(self.lib.dalek_b200_stream(self.h) or 0)

    def edwards_msm_partial(self, scalars, points, n_local, n_shard, point_fmt=POINTS_COMPRESSED, device_ptrs=False):
        nwin = self.msm_window_count(n_shard)
        out = (C.c_uint64 * (20 * nwin))()
        fn = self.lib.dalek_b200_edwards_msm_partial_dev if device_ptrs else self.lib.dalek_b200_edwards_msm_partial
        rc = self._check(fn(self.h, _ptr(scalars), _ptr(points), point_fmt, n_local, n_shard, C.addressof(out)))
        return rc, out

    def edwards_msm_combine(self, windows, ranks, n_shard, want_limbs=False):
        out = (C.c_uint8 * 32)()
        limbs = (C.c_uint64 * 20)() if want_limbs else None
        self._check(self.lib.dalek_b200_edwards_msm_combine(self.h, _ptr(windows) if not isinstance(windows, C.Array) else C.addressof(windows),
                                                            ranks, n_shard, C.addressof(out),
                                                            C.addressof(limbs) if want_limbs else None))
        return bytes(out), (list(limbs) if want_limbs else None)

    def edwards_msm_partial_async(self, scalars, points, n_local, n_shard, d_out_record, point_fmt=POINTS_COMPRESSED,
                                  device_ptrs=False):
        """Enqueue the shard's MSM on the context's stream; its record lands in the device buffer d_out_record."""
        fn = self.lib.dalek_b200_edwards_msm_partial_dev_async if device_ptrs else self.lib.dalek_b200_edwards_msm_partial_async
        return self._check(fn(self.h, _ptr(scalars), _ptr(points), point_fmt, n_local, n_shard, _ptr(d_out_record)))

    def edwards_msm_combine_dev(self, d_records, ranks, n_shard, want_limbs=False):
        """(rc, compressed, limbs) from `ranks` gathered device records; rc 1 == None."""
        out = (C.c_uint8 * 32)()
        limbs = (C.c_uint64 * 20)() if want_limbs else None
        rc = self._check(self.lib.dalek_b200_edwards_msm_combine_dev(self.h, _ptr(d_records), ranks, n_shard, C.addressof(out),
                                                                     C.addressof(limbs) if want_limbs else None))
        return rc, bytes(out), (list(limbs) if want_limbs else None)

    # ---- Ristretto ----
    def ristretto_double_base_batch(self, a, b, G, H, n, out=None):
        """a_i*G + b_i*H for n pairs (host buffers).  With `out` (a writable 32*n-byte host buffer, e.g. a pinned
        tensor) the encodings are written there and `out` is returned instead of a bytes copy."""
        if out is not None:
            rc = self._check(self.lib.dalek_b200_ristretto_double_base_batch(self.h, _ptr(a), _ptr(b), _ptr(G), _ptr(H), n, _ptr(out)))
            return rc, out
        buf = (C.c_uint8 * (32 * max(n, 1)))()
        rc = self._check(self.lib.dalek_b200_ristretto_double_base_batch(self.h, _ptr(a), _ptr(b), _ptr(G), _ptr(H), n,
                                                                         C.addressof(buf)))
        return rc, bytes(buf)[:32 * n]

    def ristretto_vartime_msm(self, scalars, points, n):
        out = (C.c_uint8 * 32)()
        rc = self._check(self.lib.dalek_b200_ristretto_vartime_msm(self.h, _ptr(scalars), _ptr(points), n, C.addressof(out)))
        return rc, bytes(out)

    # ---- scalar batches ----
    def scalar_from_wide_batch(self, wide, n):
        """Scalar::from_bytes_mod_order_wide for n x 64 B -> n x 32 B."""
        out = (C.c_uint8 * (32 * max(n, 1)))()
        self._check(self.lib.dalek_b200_scalar_from_wide_batch(self.h, _ptr(wide), n, C.addressof(out)))
        return bytes(out)[:32 * n]

    def scalar_invert_batch(self, scalars, n):
        """Scalar::invert_batch: (inverses n x 32 B, product of all inverses)."""
        out = (C.c_uint8 * (32 * max(n, 1)))()
        prod = (C.c_uint8 * 32)()
        self._check(self.lib.dalek_b200_scalar_invert_batch(self.h, _ptr(scalars), n, C.addressof(out), C.addressof(prod)))
        return bytes(out)[:32 * n], bytes(prod)

    # ---- batch codecs ----
    def decompress_batch(self, encodings, n, ristretto=False):
        """CompressedEdwardsY / CompressedRistretto decompress for n x 32 B: (rc, limbs [n x 20 u64], ok bytes)."""
        limbs = (C.c_uint64 * (20 * max(n, 1)))()
        ok = (C.c_uint8 * max(n, 1))()
        fn = self.lib.dalek_b200_ristretto_decompress_batch if ristretto else self.lib.dalek_b200_edwards_decompress_batch
        rc = self._check(fn(self.h, _ptr(encodings), n, C.addressof(limbs), C.addressof(ok)))
        return rc, limbs, bytes(ok)[:n]

    def compress_batch(self, limbs, n):
        """EdwardsPoint::compress_batch for n points given as 20 u64 limbs each -> n x 32 B."""
        out = (C.c_uint8 * (32 * max(n, 1)))()
        self._check(self.lib.dalek_b200_edwards_compress_batch(self.h, _ptr(limbs), n, C.addressof(out)))
        return bytes(out)[:32 * n]

    def ristretto_double_and_compress_batch(self, limbs, n):
        out = (C.c_uint8 * (32 * max(n, 1)))()
        self._check(self.lib.dalek_b200_ristretto_double_and_compress_batch(self.h, _ptr(limbs), n, C.addressof(out)))
        return bytes(out)[:32 * n]

    # ---- ed25519 ----
    def verify_batch_raw(self, messages, sigs, pubkeys):
        """messages: list of bytes; sigs: n*64 bytes; pubkeys: n*32 bytes.  Returns the C return code."""
        n = len(messages)
        bufs = [C.create_string_buffer(m, max(len(m), 1)) for m in messages]
        ptrs = (C.c_void_p * max(n, 1))(*[C.addressof(b) for b in bufs])
        lens = (C.c_size_t * max(n, 1))(*[len(m) for m in messages])
        return self._check(self.lib.ed25519_b200_verify_batch(self.h, C.addressof(ptrs), C.addressof(lens),
                                                              _ptr(sigs), _ptr(pubkeys), n))

    def verify_batch_flat(self, msgs_flat, offsets, sigs, pubkeys, n, device_ptrs=False, msgs_bytes=0):
        if device_ptrs:
            return self._check(self.lib.ed25519_b200_verify_batch_flat_dev(self.h, _ptr(msgs_flat), _ptr(offsets), _ptr(sigs),
                                                                           _ptr(pubkeys), n, msgs_bytes))
        return self._check(self.lib.ed25519_b200_verify_batch_flat(self.h, _ptr(msgs_flat), _ptr(offsets), _ptr(sigs),
                                                                   _ptr(pubkeys), n))

    def verify_batch_flat_points(self, msgs_flat, offsets, sigs, pubkeys, key_points, n, device_ptrs=False):
        """verify_batch for callers holding VerifyingKeys: key_points = n x 20 u64 limbs, the decompressed point of each key
        (E/verifying.rs:65-71); no key is decompressed inside the call."""
        fn = self.lib.ed25519_b200_verify_batch_flat_points_dev if device_ptrs else self.lib.ed25519_b200_verify_batch_flat_points
        return self._check(fn(self.h, _ptr(msgs_flat), _ptr(offsets), _ptr(sigs), _ptr(pubkeys), _ptr(key_points), n))

    def verify_batches_flat(self, msgs_flat, offsets, sigs, pubkeys, n, batch_size, device_ptrs=False):
        """Independent batches of `batch_size` signatures in one call: (rc, verdicts) with verdicts[k] the result of
        verify_batch on batch k (0 Ok, 1 Verify, 3 ScalarFormat, 4 PointDecompression); rc = 0 iff all are 0."""
        nb = (n + batch_size - 1) // batch_size
        verdicts = (C.c_int32 * max(nb, 1))()
        fn = self.lib.ed25519_b200_verify_batches_flat_dev if device_ptrs else self.lib.ed25519_b200_verify_batches_flat
        rc = self._check(fn(self.h, _ptr(msgs_flat), _ptr(offsets), _ptr(sigs), _ptr(pubkeys), n, batch_size, C.addressof(verdicts)))
        return rc, list(verdicts)[:nb]

    def verify_batches_flat_points(self, msgs_flat, offsets, sigs, pubkeys, key_points, n, batch_size, device_ptrs=False):
        """verify_batches_flat for callers holding VerifyingKeys (key_points = n x 20 u64 limbs): no key decompression."""
        nb = (n + batch_size - 1) // batch_size
        verdicts = (C.c_int32 * max(nb, 1))()
        fn = self.lib.ed25519_b200_verify_batches_flat_points_dev if device_ptrs else self.lib.ed25519_b200_verify_batches_flat_points
        rc = self._check(fn(self.h, _ptr(msgs_flat), _ptr(offsets), _ptr(sigs), _ptr(pubkeys), _ptr(key_points), n, batch_size, C.addressof(verdicts)))
        return rc, list(verdicts)[:nb]

    def verify_each_flat(self, msgs_flat, offsets, sigs, pubkeys, n, strict=False, device_ptrs=False):
        """n independent verifications: (rc, results) with results[i] the code of VerifyingKey::verify (or verify_strict)
        for signature i alone; rc = 0 iff all are 0."""
        res = (C.c_uint8 * max(n, 1))()
        fn = self.lib.ed25519_b200_verify_each_flat_dev if device_ptrs else self.lib.ed25519_b200_verify_each_flat
        rc = self._check(fn(self.h, _ptr(msgs_flat), _ptr(offsets), _ptr(sigs), _ptr(pubkeys), n, 1 if strict else 0, C.addressof(res)))
        return rc, list(res)[:n]

    def last_zs(self, n):
        out = (C.c_uint8 * (16 * max(n, 1)))()
        self._check(self.lib.ed25519_b200_last_zs(self.h, C.addressof(out), n))
        return bytes(out)[:16 * n]

    # ---- synthesis ----
    def mul_base_batch(self, scalars, n, want_compressed=True):
        limbs = (C.c_uint64 * (20 * max(n, 1)))()
        comp = (C.c_uint8 * (32 * max(n, 1)))() if want_compressed else None
        self._check(self.lib.dalek_b200_edwards_mul_base_batch(self.h, _ptr(scalars), n, C.addressof(limbs),
                                                               C.addressof(comp) if want_compressed else None))
        return limbs, (bytes(comp)[:32 * n] if want_compressed else None)

    def sign_batch_flat(self, seeds, msgs_flat, offsets, n):
        pks = (C.c_uint8 * (32 * max(n, 1)))()
        sigs = (C.c_uint8 * (64 * max(n, 1)))()
        self._check(self.lib.ed25519_b200_sign_batch_flat(self.h, _ptr(seeds), _ptr(msgs_flat), _ptr(offsets), n,
                                                          C.addressof(pks), C.addressof(sigs)))
        return bytes(pks)[:32 * n], bytes(sigs)[:64 * n]


class MultiEngine:
    """One MSM over several GPUs of this node from a single process (dalek_b200_init_multi): contiguous shards, peer
    copies of the window-accumulator records to the first device, combine there."""

    def __init__(self, devices):
        self.lib = load_library()
        devs = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        rc = self.lib.dalek_b200_init_multi(devs, len(devices), C.byref(h))
        if rc != 0:
            raise EngineError("dalek_b200_init_multi(%r) failed with %d (the engine has no CPU fallback)" % (list(devices), rc))
        self.h = h
        self.devices = list(devices)

    def close(self):
        if getattr(self, "h", None):
            self.lib.dalek_b200_destroy_multi(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name, value):
        for i in range(len(self.devices)):
            rc = self.lib.dalek_b200_set_option(self.lib.dalek_b200_multi_ctx(self.h, i), name.encode(), int(value))
            if rc:
                raise EngineError("set_option(%s) failed" % name)

    def last_call_ms(self):
        ms = C.c_float()
        self.lib.dalek_b200_last_call_ms(self.lib.dalek_b200_multi_ctx(self.h, 0), C.byref(ms))
        return float(ms.value)

    def edwards_vartime_msm(self, scalars, points, n, point_fmt=POINTS_COMPRESSED, want_limbs=False):
        """(rc, compressed32, limbs20 or None) like Engine.edwards_vartime_msm, host buffers."""
        out = (C.c_uint8 * 32)()
        limbs = (C.c_uint64 * 20)() if want_limbs else None
        keep = (scalars, points)
        rc = self.lib.dalek_b200_edwards_vartime_msm_multi(self.h, _ptr(scalars), _ptr(points), point_fmt, n, C.addressof(out),
                                                           C.addressof(limbs) if want_limbs else None)
        del keep
        if rc < 0:
            raise EngineError("engine error %d: %s" % (rc, self.lib.dalek_b200_multi_last_error(self.h).decode()))
        return rc, bytes(out), (list(limbs) if want_limbs else None)


_default = None


def default_engine():
    global _default
    if _default is None:
        _default = Engine(int(os.environ.get("LOCAL_RANK", "0")))
    return _default


class EdwardsPoint:
    """Mirror of the trait impls on curve25519_dalek::edwards::EdwardsPoint.  Points are handled in
    their 32-byte CompressedEdwardsY encoding; results are returned compressed."""

    @staticmethod
    def optional_multiscalar_mul(scalars, points, engine=None):
        """VartimeMultiscalarMul::optional_multiscalar_mul (traits.rs:196-200): `points` holds 32-byte
        encodings; an entry that is None or fails to decompress makes the result None."""
        scalars, points = list(scalars), list(points)
        # both iterators must have equal, exact sizes (edwards.rs:1013-1019 asserts)
        assert len(scalars) == len(points), "scalars and points must have the same length"
        if any(p is None for p in points):
            return None
        eng = engine or default_engine()
        rc, comp, _ = eng.edwards_vartime_msm(b"".join(scalars), b"".join(points), len(scalars))
        return None if rc == 1 else comp

    @staticmethod
    def optional_multiscalar_mul_batch(msms, engine=None):
        """optional_multiscalar_mul for every (scalars, points) of `msms` in one engine call: a list of Optional[bytes].
        A point that is None or does not decompress makes that MSM's result None, and only that one."""
        return _msm_batch(msms, engine, ristretto=False)

    @staticmethod
    def vartime_multiscalar_mul(scalars, points, engine=None):
        """traits.rs:249-262: .expect() on the optional form."""
        r = EdwardsPoint.optional_multiscalar_mul(scalars, points, engine)
        if r is None:
            raise ValueError("should return some point")
        return r

    @staticmethod
    def multiscalar_mul(scalars, points, engine=None):
        """MultiscalarMul::multiscalar_mul (traits.rs:128-133, edwards.rs:970-995), constant-time contract."""
        scalars, points = list(scalars), list(points)
        assert len(scalars) == len(points), "scalars and points must have the same length"
        eng = engine or default_engine()
        rc, comp, _ = eng.edwards_ct_msm(b"".join(scalars), b"".join(points), len(scalars))
        return comp


# encodings that never decode, standing in for None points: y = 2 is not on the curve; s = 1 is a negative field element,
# which CompressedRistretto::decompress rejects (ristretto.rs:266-345)
_BAD_EDWARDS = (2).to_bytes(32, "little")
_BAD_RISTRETTO = (1).to_bytes(32, "little")


def _msm_batch(msms, engine, ristretto):
    sc, pt, offsets = [], [], [0]
    bad = _BAD_RISTRETTO if ristretto else _BAD_EDWARDS
    for scalars, points in msms:
        scalars, points = list(scalars), list(points)
        assert len(scalars) == len(points), "scalars and points must have the same length"
        sc += scalars
        pt += [bad if p is None else p for p in points]
        offsets.append(len(sc))
    eng = engine or default_engine()
    sb, pb = b"".join(sc), b"".join(pt)
    if ristretto:
        _, res = eng.ristretto_vartime_msm_batch(sb, pb, offsets)
    else:
        _, res, _ = eng.edwards_vartime_msm_batch(sb, pb, offsets)
    return res


class _Precomputation:
    """VartimePrecomputedMultiscalarMul (traits.rs:290-406): static points converted once, resident on the GPU."""
    _FMT = POINTS_COMPRESSED

    def __init__(self, static_points, engine=None, fmt=None):
        """`new` (traits.rs:297-300): static_points = iterable of 32-byte encodings (or, with fmt=POINTS_EXTENDED, a
        buffer of n x 20 u64 limbs passed as (buffer, n))."""
        self.eng = engine or default_engine()
        fmt = self._FMT if fmt is None else fmt
        if fmt == POINTS_EXTENDED:
            buf, n = static_points
        else:
            pts = list(static_points)
            buf, n = b"".join(pts), len(pts)
        h = C.c_void_p()
        rc = self.eng._check(self.eng.lib.dalek_b200_precomp_new(self.eng.h, _ptr(buf) if n else None, fmt, n, C.byref(h)))
        if rc == 1:
            raise ValueError("a static point does not decode")
        self.h = h

    def __len__(self):                                   # traits.rs:303
        return int(self.eng.lib.dalek_b200_precomp_len(self.h))

    def is_empty(self):                                  # traits.rs:306
        return len(self) == 0

    def close(self):
        if getattr(self, "h", None):
            self.eng.lib.dalek_b200_precomp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def optional_mixed_multiscalar_mul(self, static_scalars, dynamic_scalars, dynamic_points, dynamic_fmt=None):
        """traits.rs:402-413.  A dynamic point that is None or undecodable gives None."""
        ss, ds, dp = list(static_scalars), list(dynamic_scalars), list(dynamic_points)
        assert len(ss) <= len(self), "more static scalars than static points"
        assert len(ds) == len(dp), "dynamic scalars and points must have the same length"
        if any(p is None for p in dp):
            return None
        out = (C.c_uint8 * 32)()
        sb, db, pb = b"".join(ss), b"".join(ds), b"".join(dp)      # kept alive across the call
        rc = self.eng._check(self.eng.lib.dalek_b200_precomp_mixed_msm(
            self.eng.h, self.h, _ptr(sb) if ss else None, len(ss), _ptr(db) if ds else None, _ptr(pb) if dp else None,
            self._FMT if dynamic_fmt is None else dynamic_fmt, len(ds), C.addressof(out), None))
        return None if rc == 1 else bytes(out)

    def vartime_mixed_multiscalar_mul(self, static_scalars, dynamic_scalars, dynamic_points):
        """traits.rs:357-383: .expect() on the optional form."""
        r = self.optional_mixed_multiscalar_mul(static_scalars, dynamic_scalars, dynamic_points)
        if r is None:
            raise ValueError("should return some point")
        return r

    def vartime_multiscalar_mul(self, static_scalars):
        """traits.rs:324-338."""
        return self.vartime_mixed_multiscalar_mul(static_scalars, [], [])


class VartimeEdwardsPrecomputation(_Precomputation):
    """curve25519-dalek/src/edwards.rs:1038-1076 (CompressedEdwardsY encodings in and out)."""
    _FMT = POINTS_COMPRESSED


class VartimeRistrettoPrecomputation(_Precomputation):
    """curve25519-dalek/src/ristretto.rs:1004-1049 (CompressedRistretto encodings in and out)."""
    _FMT = POINTS_RISTRETTO


class RistrettoPoint:
    """Mirror of the forwarding impls in curve25519-dalek/src/ristretto.rs:964-994 (CompressedRistretto I/O)."""

    @staticmethod
    def vartime_multiscalar_mul(scalars, points, engine=None):
        scalars, points = list(scalars), list(points)
        assert len(scalars) == len(points)
        eng = engine or default_engine()
        rc, comp = eng.ristretto_vartime_msm(b"".join(scalars), b"".join(points), len(scalars))
        if rc == 1:
            raise ValueError("should return some point")
        return comp

    @staticmethod
    def optional_multiscalar_mul_batch(msms, engine=None):
        """Independent Ristretto MSMs in one engine call (CompressedRistretto points and results): a list of
        Optional[bytes]; a None or undecodable point makes that MSM's result None, and only that one."""
        return _msm_batch(msms, engine, ristretto=True)

    @staticmethod
    def double_base_batch(a, b, G, H, engine=None):
        eng = engine or default_engine()
        n = len(a) // 32
        rc, out = eng.ristretto_double_base_batch(a, b, G, H, n)
        if rc == 1:
            raise ValueError("G or H is not a valid Ristretto encoding")
        return out


def verify_batch(messages, signatures, verifying_keys, engine=None):
    """ed25519_dalek::verify_batch (batch.rs:146-251): returns None on Ok, raises SignatureError otherwise."""
    messages, signatures, verifying_keys = list(messages), list(signatures), list(verifying_keys)
    if not (len(messages) == len(signatures) == len(verifying_keys)):
        raise SignatureError(2)                      # batch.rs:152-165 ArrayLength
    eng = engine or default_engine()
    rc = eng.verify_batch_raw(messages, b"".join(signatures), b"".join(verifying_keys))
    if rc != 0:
        raise SignatureError(rc)
    return None
