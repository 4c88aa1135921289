/*
 * dalek_b200.h -- C ABI of the B200 multiscalar-multiplication / batch-verification engine.
 *
 * The reference (curve25519-dalek / ed25519-dalek, 100 % Rust) has no FFI for this path: the
 * hot path sits behind Rust traits.  Each entry point below replaces one of those trait
 * methods / functions and names it (paths relative to the reference tree):
 *
 *   C/ = curve25519-dalek/src/   E/ = ed25519-dalek/src/
 *
 * A thin Rust shim (shown in INTEGRATION.md) collects the trait iterators into the flat
 * buffers used here.  All buffers are caller-owned; unless a `_dev` variant is named, pointers
 * are HOST pointers and the call copies them to the device, runs, copies the result back and
 * returns (blocking).  A context may be used by one thread at a time; different contexts may
 * be used concurrently.
 *
 * Data formats
 *   scalar            32 bytes little-endian, any value < 2^256 (the reference's Scalar
 *                     invariant is bit 255 clear, C/scalar.rs:193-230; not required here)
 *   compressed point  32 bytes CompressedEdwardsY (C/edwards.rs:175) or CompressedRistretto
 *   extended point    20 x uint64_t: X, Y, Z, T as FieldElement51 radix-2^51 limbs
 *                     (C/edwards.rs:390-395, C/backend/serial/u64/field.rs:43); limbs < 2^54
 *
 * Return codes: 0 = success / Ok; positive = the reference's own error values (see the
 * DALEK_* constants); negative = engine errors (bad argument, CUDA failure).  There is no CPU
 * fallback: without a usable CUDA device dalek_b200_init fails with DALEK_E_NO_DEVICE.
 */
#ifndef DALEK_B200_H
#define DALEK_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dalek_b200_ctx dalek_b200_ctx;

/* reference-level outcomes */
#define DALEK_OK 0
#define DALEK_NONE 1                      /* Option::None: a point failed to decompress (C/traits.rs:196) */
#define ED25519_ERR_VERIFY 1              /* InternalError::Verify             (E/errors.rs:38) */
#define ED25519_ERR_ARRAY_LENGTH 2        /* InternalError::ArrayLength        (E/errors.rs:41-49) */
#define ED25519_ERR_SCALAR_FORMAT 3       /* InternalError::ScalarFormat       (E/errors.rs:27) */
#define ED25519_ERR_POINT_DECOMPRESSION 4 /* InternalError::PointDecompression (E/errors.rs:26) */
/* engine errors */
#define DALEK_E_INVALID_ARG (-1)
#define DALEK_E_NO_DEVICE (-2)
#define DALEK_E_CUDA (-3)
#define DALEK_E_NOMEM (-4)

#define DALEK_POINTS_COMPRESSED 0         /* n x 32 B CompressedEdwardsY */
#define DALEK_POINTS_EXTENDED 1           /* n x 20 x u64 radix-2^51 limbs */
#define DALEK_POINTS_RISTRETTO 2          /* n x 32 B CompressedRistretto (precomputation API only) */

/* -------- context ---------------------------------------------------------------------- */
/* Create an engine context on CUDA device `device`.  Fails (no CPU fallback) if the device
 * is missing or is not an sm_100 part. */
int dalek_b200_init(int device, dalek_b200_ctx **out);
void dalek_b200_destroy(dalek_b200_ctx *ctx);
const char *dalek_b200_last_error(const dalek_b200_ctx *ctx);
/* Tunables.  None changes a result except "verify_chunk" (see verify_batch): "window_bits" (4..20, 0 = choose from n),
 * "verify_chunk" (0, default: the reference's single transcript per batch; k > 0: opt-in, one transcript per k signatures --
 * NOT reference-equivalent on inputs with small-order components), "field_f64" (1 = bucket kernel on the FP64-pipe field,
 * default; 0 = IMAD.WIDE field), "acc_tma" (1 = the bucket kernel gathers points with TMA bulk copies, default 0: cp.async),
 * "small_straus" (1 = fewer than 190 pairs run vartime Straus like the reference, default; 0 = bucket pipeline),
 * "host_chunks" (1..8, host-buffer MSM calls stream their input in this many chunks, default 8), "verify_pieces" (1..8, same
 * for verify_batch, default 4), "decompress_f64" (1 = square-root exponentiation of decompression on the FP64 field, default),
 * "dedupe_keys" (1 = decompress every distinct public key once and give it one MSM term, default), "double_base_comb" (1 =
 * fixed-base comb for double-base batches of >= 4096 pairs, default), "precomp_tables" (1 = precomputations of >= 4096 points
 * also keep the 2^(cw) P window tables; default 0: measured, the 1.7 GB of randomly gathered table entries cost the bucket
 * kernel what the shorter tail saves), "transcript_warp" (1 = launches of up to 2048 Merlin transcripts run one warp each,
 * default), "transcript_blocks" (1 = larger launches run one thread per transcript with the rate block staged in shared
 * memory, default; 0 = byte-wise sponge), "each_comb" (per-signature verification: 1 = per-key comb tables when
 * every distinct key signs at least eight signatures on average, default; 2 = always; 0 = never), "batch_bucket_min"
 * (1..2^31-1: segments of a batched MSM with at least this many pairs run the bucket pipeline, shorter ones the
 * segmented Straus; default 65536), "trace" (1 = per-stage device timeline of verify_batch on stderr).
 * Returns 0 or DALEK_E_INVALID_ARG. */
int dalek_b200_set_option(dalek_b200_ctx *ctx, const char *name, long value);
/* Number of kernels launched by this context since creation (bench.py's gpu_launches). */
uint64_t dalek_b200_launch_count(const dalek_b200_ctx *ctx);
/* Milliseconds (CUDA events on the context's stream) spent in the dominant kernel of the last
 * call (bucket accumulation for MSM calls), and that kernel's launch count in the last call. */
int dalek_b200_last_kernel_ms(const dalek_b200_ctx *ctx, float *ms, int *launches);
/* Same by name: "bucket_accumulate" (the figure above) or "decompress_R" (the R-decompression kernel of the last
 * verify_batch call, the largest kernel of that path; summed over the pieces of a host-streamed call). */
int dalek_b200_last_stage_ms(const dalek_b200_ctx *ctx, const char *stage, float *ms);
/* Milliseconds between CUDA events recorded on the context's stream at entry of the last MSM / verify_batch /
 * precomputed-MSM call and after the last work it enqueued (all of the call's streams joined): the device time
 * of that call, copies of host-buffer calls included. */
int dalek_b200_last_call_ms(const dalek_b200_ctx *ctx, float *ms);

/* -------- EdwardsPoint multiscalar multiplication --------------------------------------- */
/*
 * VartimeMultiscalarMul::optional_multiscalar_mul / vartime_multiscalar_mul for EdwardsPoint
 * (C/traits.rs:196-262, C/edwards.rs:1002-1030; algorithms C/backend/serial/scalar_mul/
 * pippenger.rs:67-160 and straus.rs:159-200).  Computes sum scalars[i] * points[i].
 * Returns DALEK_NONE when point_fmt is COMPRESSED and any point fails to decompress
 * (the reference returns None when any Option<Point> is None).  n = 0 yields the identity.
 * out_compressed receives the 32-byte CompressedEdwardsY of the result (EdwardsPoint::compress,
 * C/edwards.rs:564-617); out_limbs (nullable) receives canonical radix-2^51 X,Y,Z,T limbs of an
 * equal point (projectively equal to the reference's result; limb values themselves differ
 * between the reference's own backends).
 */
int dalek_b200_edwards_vartime_msm(dalek_b200_ctx *ctx, const uint8_t *scalars, const void *points,
                                   int point_fmt, size_t n, uint8_t out_compressed[32],
                                   uint64_t out_limbs[20]);
/*
 * MultiscalarMul::multiscalar_mul for EdwardsPoint (constant-time contract, C/traits.rs:78-134,
 * C/edwards.rs:970-995, straus.rs:103-144): uniform control flow and table scans that do not
 * depend on the scalars.  Points must all be valid (the trait takes points, not Options):
 * an undecodable compressed point is DALEK_E_INVALID_ARG.
 */
int dalek_b200_edwards_ct_msm(dalek_b200_ctx *ctx, const uint8_t *scalars, const void *points,
                              int point_fmt, size_t n, uint8_t out_compressed[32],
                              uint64_t out_limbs[20]);
/* Same two calls with device-resident inputs (scalars: n x 32 B; points as point_fmt says);
 * outputs are still written to host memory. */
int dalek_b200_edwards_vartime_msm_dev(dalek_b200_ctx *ctx, const void *d_scalars, const void *d_points,
                                       int point_fmt, size_t n, uint8_t out_compressed[32],
                                       uint64_t out_limbs[20]);

/* -------- many independent MSMs in one call ------------------------------------------------
 * m independent VartimeMultiscalarMul::optional_multiscalar_mul calls (C/traits.rs:196-262) in one call.
 * MSM k takes the pairs [offsets[k], offsets[k+1]) of the flat scalars / points arrays (offsets: m + 1 u64, HOST memory
 * in both forms, offsets[0] = 0, non-decreasing, offsets[m] < 2^31).  Result k is byte for byte what
 * dalek_b200_edwards_vartime_msm returns on slice k: out_compressed[32 k ..] the CompressedEdwardsY, out_limbs[20 k ..]
 * (nullable) canonical limbs of an equal point, status[k] = 1 (None) when a point of segment k does not decode -- its 32
 * output bytes (and limbs) are then zero; a bad point affects only its own segment.  point_fmt: COMPRESSED or EXTENDED;
 * scalars may be any 256-bit value; an empty segment gives the identity with status 0.
 * Returns 0 if every status is 0, DALEK_NONE if any is 1, DALEK_E_INVALID_ARG for malformed offsets, null buffers or a bad
 * point_fmt, or m >= 2^31, other negative codes for engine errors; m = 0 succeeds and writes nothing.  dalek_b200_last_call_ms covers
 * the whole call.  Segments shorter than the option "batch_bucket_min" (default 65536 pairs) run as a segmented Straus
 * (one accumulator per task of up to 64 pairs of one segment), all of them in a few launches per ~2^20 pairs; longer
 * segments, and any longer than 2^20 pairs, run the bucket pipeline one after another.  The results do not depend on the
 * option. */
int dalek_b200_edwards_vartime_msm_batch(dalek_b200_ctx *ctx, const uint8_t *scalars, const void *points, int point_fmt,
                                         const uint64_t *offsets, size_t m, uint8_t *out_compressed /* m x 32 */,
                                         uint64_t *out_limbs /* nullable, m x 20 */, uint8_t *status /* m */);
/* The same with device-resident scalars and points; offsets and outputs are host memory. */
int dalek_b200_edwards_vartime_msm_batch_dev(dalek_b200_ctx *ctx, const void *d_scalars, const void *d_points, int point_fmt,
                                             const uint64_t *offsets, size_t m, uint8_t *out_compressed,
                                             uint64_t *out_limbs, uint8_t *status);
/* RistrettoPoint form over CompressedRistretto points; result k as dalek_b200_ristretto_vartime_msm returns it on slice k. */
int dalek_b200_ristretto_vartime_msm_batch(dalek_b200_ctx *ctx, const uint8_t *scalars, const uint8_t *points,
                                           const uint64_t *offsets, size_t m, uint8_t *out_compressed, uint8_t *status);

/* -------- sharded MSM (one call per GPU / rank, SURVEY 8e) --------------------------------
 * MSM is linear: every rank reduces a contiguous shard of the pairs to one accumulator per bucket window
 * (pippenger.rs:146-151 for its shard), the accumulators are exchanged once (all-gather: point addition is
 * not an NCCL reduction operator), and every rank adds them per window and runs the Horner pass of
 * pippenger.rs:159.  `n_shard` is the size of the LARGEST shard (ceil(n_total / ranks) for an even split)
 * and must be the same on every rank: the window width is chosen from it, i.e. for the work one GPU does.
 *
 * Number of window accumulators of a partial MSM for that shard size. */
int dalek_b200_msm_window_count(dalek_b200_ctx *ctx, size_t n_shard);
/* Size in bytes of a shard's device RECORD: window_count x 20 u64 limbs, then one u64 status word
 * (non-zero: a compressed point of the shard did not decode -> the combined result is None). */
size_t dalek_b200_msm_partial_bytes(dalek_b200_ctx *ctx, size_t n_shard);
/* Partial MSM over this rank's shard, blocking: writes `window_count` window accumulators
 * (each 20 x u64 extended limbs, window 0 = least significant) to out_windows (host).
 * DALEK_NONE if a compressed point did not decode. */
int dalek_b200_edwards_msm_partial(dalek_b200_ctx *ctx, const uint8_t *scalars, const void *points,
                                   int point_fmt, size_t n_local, size_t n_shard,
                                   uint64_t *out_windows);
int dalek_b200_edwards_msm_partial_dev(dalek_b200_ctx *ctx, const void *d_scalars, const void *d_points,
                                       int point_fmt, size_t n_local, size_t n_shard,
                                       uint64_t *out_windows);
/* Combine the gathered accumulators of `ranks` shards (host, rank-major: ranks x window_count x 20 u64)
 * into the final point: per-window sum over ranks, then total = total * 2^w + window
 * (pippenger.rs:159). */
int dalek_b200_edwards_msm_combine(dalek_b200_ctx *ctx, const uint64_t *windows, int ranks,
                                   size_t n_shard, uint8_t out_compressed[32], uint64_t out_limbs[20]);
/* The same exchange without leaving the device: ..._partial[_dev]_async ENQUEUES the shard's MSM on the
 * context's stream and writes its record (dalek_b200_msm_partial_bytes) to the device buffer d_out_record;
 * it returns without synchronising.  The caller enqueues the all-gather of the records behind it ON THAT
 * STREAM (dalek_b200_stream: e.g. torch.cuda.ExternalStream + torch.distributed.all_gather_into_tensor, or
 * ncclAllGather(..., stream)), then ..._combine_dev takes the gathered device buffer (ranks records,
 * rank-major), runs the Horner pass and blocks only for the 192-byte result.  DALEK_NONE if any shard's
 * status word is set.  dalek_b200_last_call_ms then spans partial + exchange + combine on the device. */
int dalek_b200_edwards_msm_partial_async(dalek_b200_ctx *ctx, const uint8_t *scalars, const void *points,
                                         int point_fmt, size_t n_local, size_t n_shard, void *d_out_record);
int dalek_b200_edwards_msm_partial_dev_async(dalek_b200_ctx *ctx, const void *d_scalars, const void *d_points,
                                             int point_fmt, size_t n_local, size_t n_shard, void *d_out_record);
int dalek_b200_edwards_msm_combine_dev(dalek_b200_ctx *ctx, const void *d_records, int ranks, size_t n_shard,
                                       uint8_t out_compressed[32], uint64_t out_limbs[20]);
/* The context's main CUDA stream (a cudaStream_t) for callers that order their own work with the engine's. */
void *dalek_b200_stream(dalek_b200_ctx *ctx);

/* -------- one MSM over several GPUs from a single process (SURVEY 8b / 8e) ---------------------
 * dalek_b200_init_multi creates one engine context per listed CUDA device (distinct sm_100 devices of one node)
 * and enables peer access to the first one.  ..._vartime_msm_multi is VartimeMultiscalarMul::optional_multiscalar_mul
 * (C/traits.rs:196-262, same conventions as dalek_b200_edwards_vartime_msm, host buffers) with the pair range cut
 * into contiguous shards, one per device: every device reduces its shard to window accumulators, the ~2.7 KB records
 * are written into the first device's memory by peer copies over NVLink, and the first device combines them
 * (pippenger.rs:146-159).  Inputs of fewer than 2^14 pairs per device run on the first device alone. */
typedef struct dalek_b200_multi dalek_b200_multi;
int dalek_b200_init_multi(const int *devices, int ndev, dalek_b200_multi **out);
void dalek_b200_destroy_multi(dalek_b200_multi *m);
int dalek_b200_multi_device_count(const dalek_b200_multi *m);
/* The context of device i (e.g. to set options, or to run replicas of verify_batch on every GPU). */
dalek_b200_ctx *dalek_b200_multi_ctx(dalek_b200_multi *m, int i);
const char *dalek_b200_multi_last_error(const dalek_b200_multi *m);
int dalek_b200_edwards_vartime_msm_multi(dalek_b200_multi *m, const uint8_t *scalars, const void *points,
                                         int point_fmt, size_t n, uint8_t out_compressed[32],
                                         uint64_t out_limbs[20]);

/* -------- VartimePrecomputedMultiscalarMul (SURVEY 8f rank 1) ---------------------------------
 * C/traits.rs:290-406; VartimeEdwardsPrecomputation C/edwards.rs:1038-1076, VartimeRistrettoPrecomputation
 * C/ristretto.rs:1004-1049 (serial backend: precomputed_straus.rs:33-127).  The static points are decoded
 * and converted once and stay resident in device memory; later calls send scalars only.  With the option
 * "precomp_tables" the tables 2^(c w) P_i of every window are kept too (96 B x windows per point, e.g. 1.7 GB for
 * 2^20 points), so that all windows share one bucket set and the final doublings disappear.
 *
 * new (traits.rs:297-300): static_points in format DALEK_POINTS_* (RISTRETTO makes a Ristretto
 * precomputation: Ristretto encodings in and out).  DALEK_NONE if an encoded static point does not decode. */
typedef struct dalek_b200_precomp dalek_b200_precomp;
int dalek_b200_precomp_new(dalek_b200_ctx *ctx, const void *static_points, int point_fmt, size_t n,
                           dalek_b200_precomp **out);
size_t dalek_b200_precomp_len(const dalek_b200_precomp *pre);     /* traits.rs:303 */
void dalek_b200_precomp_destroy(dalek_b200_precomp *pre);
/* optional_mixed_multiscalar_mul (traits.rs:402-413):  Q = sum a_i A_i + sum b_j B_j  with B_j the static
 * points.  n_static may be smaller than len() (unused points are ignored, traits.rs:314-316); larger is
 * DALEK_E_INVALID_ARG (the reference asserts).  n_dynamic = 0 gives vartime_multiscalar_mul
 * (traits.rs:324-338).  DALEK_NONE if a dynamic point does not decode.  dynamic_fmt: EXTENDED, or the
 * encoding matching the precomputation (COMPRESSED for Edwards, RISTRETTO for Ristretto).
 * out_compressed: CompressedEdwardsY, or CompressedRistretto for a Ristretto precomputation. */
int dalek_b200_precomp_mixed_msm(dalek_b200_ctx *ctx, const dalek_b200_precomp *pre,
                                 const uint8_t *static_scalars, size_t n_static,
                                 const uint8_t *dynamic_scalars, const void *dynamic_points,
                                 int dynamic_fmt, size_t n_dynamic, uint8_t out_compressed[32],
                                 uint64_t out_limbs[20]);

/* -------- batch wire-format codecs (SURVEY 8f rank 2) -----------------------------------------
 * Points are the reference's in-memory EdwardsPoint / RistrettoPoint: 20 u64 limbs X | Y | Z | T, radix 2^51.
 * Host buffers; the batch is streamed in pieces so that the copies overlap the arithmetic.
 *
 * CompressedEdwardsY::decompress (C/edwards.rs:211-257) for n encodings: ok[i] = 1 and out_limbs[20 i ..] =
 * the point (Z = 1), or ok[i] = 0 (None; the slot holds the identity).  Returns DALEK_NONE if any ok[i] = 0. */
int dalek_b200_edwards_decompress_batch(dalek_b200_ctx *ctx, const uint8_t *in, size_t n,
                                        uint64_t *out_limbs, uint8_t *ok);
/* EdwardsPoint::compress_batch (C/edwards.rs:619-647): n points -> n x 32 B, one shared inversion per 8
 * points (FieldElement::invert_batch, C/field.rs:239-274). */
int dalek_b200_edwards_compress_batch(dalek_b200_ctx *ctx, const uint64_t *limbs, size_t n, uint8_t *out);
/* CompressedRistretto::decompress (C/ristretto.rs:266-345), same conventions as the Edwards form. */
int dalek_b200_ristretto_decompress_batch(dalek_b200_ctx *ctx, const uint8_t *in, size_t n,
                                          uint64_t *out_limbs, uint8_t *ok);
/* RistrettoPoint::double_and_compress_batch (C/ristretto.rs:564-646): out[i] = compress(2 P_i). */
int dalek_b200_ristretto_double_and_compress_batch(dalek_b200_ctx *ctx, const uint64_t *limbs, size_t n,
                                                   uint8_t *out);

/* -------- scalar batch helpers (SURVEY 8f rank 4) ---------------------------------------------
 * Scalar::from_bytes_mod_order_wide (C/scalar.rs:248-250) for n 64-byte strings -> n canonical 32-byte scalars. */
int dalek_b200_scalar_from_wide_batch(dalek_b200_ctx *ctx, const uint8_t *in, size_t n, uint8_t *out);
/* Scalar::invert_batch / invert_batch_alloc (C/scalar.rs:779-853): out[i] = in[i]^-1 mod l (inputs are taken mod l),
 * out_product = the product of all inverses (the reference's return value; 1 for n = 0).  The reference requires
 * nonzero inputs (scalar.rs:796-799): a zero input is DALEK_E_INVALID_ARG here. */
int dalek_b200_scalar_invert_batch(dalek_b200_ctx *ctx, const uint8_t *in, size_t n, uint8_t *out,
                                   uint8_t out_product[32]);

/* -------- RistrettoPoint ----------------------------------------------------------------- */
/* n independent RistrettoPoint::multiscalar_mul([a_i, b_i], [G, H]) (constant-time Straus,
 * C/ristretto.rs:964-977 -> C/edwards.rs:970-995 -> straus.rs:103-144), each result compressed
 * (RistrettoPoint::compress, C/ristretto.rs:500-533).  G, H: CompressedRistretto; a, b: n x 32 B.
 * out: n x 32 B.  Returns DALEK_NONE if G or H does not decode (C/ristretto.rs:266-345; `out` is then
 * unspecified), DALEK_E_INVALID_ARG for a scalar with bit 255 set.  The results are those of the
 * reference's Straus; batches of >= 4096 pairs are computed with a fixed-base comb over tables of G
 * and H (same constant-time discipline: masked full-row scans, uniform control flow).  Pinned host
 * buffers let the copies overlap the arithmetic. */
int dalek_b200_ristretto_double_base_batch(dalek_b200_ctx *ctx, const uint8_t *a, const uint8_t *b,
                                           const uint8_t G[32], const uint8_t H[32], size_t n,
                                           uint8_t *out);
/* RistrettoPoint::vartime_multiscalar_mul over compressed Ristretto points
 * (C/ristretto.rs:980-994); result as CompressedRistretto. */
int dalek_b200_ristretto_vartime_msm(dalek_b200_ctx *ctx, const uint8_t *scalars,
                                     const uint8_t *points, size_t n, uint8_t out_compressed[32]);

/* -------- ed25519 --------------------------------------------------------------------------- */
/*
 * ed25519_dalek::verify_batch (E/batch.rs:146-251).
 *   msgs / msg_lens   n message pointers and lengths          (messages: &[&[u8]])
 *   sigs              n x 64 B R || s                          (signatures: &[Signature])
 *   pubkeys           n x 32 B compressed keys                 (verifying_keys: &[VerifyingKey])
 * In Rust a VerifyingKey already holds its decompressed point (E/verifying.rs:65-71); here keys
 * arrive as bytes and VerifyingKey::from_bytes (E/verifying.rs:167-175) runs inside the call (once
 * per DISTINCT key: repeated keys are de-duplicated on the device): an undecodable key is
 * ED25519_ERR_POINT_DECOMPRESSION.  Then, in the reference's order
 * (E/batch.rs:208-250): non-canonical s -> ED25519_ERR_SCALAR_FORMAT; undecodable R or a
 * non-identity result -> ED25519_ERR_VERIFY; else 0.  No cofactor multiplication.
 * Coefficients z_i: exactly the reference's -- ONE Merlin transcript over the whole batch (batch.rs:168-222), whatever n
 * is.  That transcript is a strictly sequential sponge (1.73 Keccak-f[1600] permutations per signature, one GPU warp:
 * about 12 us per signature), so callers with very large inputs either use ed25519_b200_verify_batches_flat (independent
 * batches, each with the reference's transcript, hashed in parallel) or OPT INTO the option "verify_chunk" = k > 0: one
 * transcript per k consecutive signatures and one combined equation.  The chunked mode is NOT reference-equivalent: its z_i
 * differ from the reference's for n > k, and while the verdict is the same for every batch without small-order components
 * (valid batches pass, invalid ones fail except with probability ~2^-128), for signatures or keys carrying small-order
 * components the un-cofactored equation's verdict depends on the z_i modulo 8 and can differ from the reference's.
 */
int ed25519_b200_verify_batch(dalek_b200_ctx *ctx, const uint8_t *const *msgs, const size_t *msg_lens,
                              const uint8_t *sigs, const uint8_t *pubkeys, size_t n);
/* Same with the messages laid out back to back: message i = msgs_flat[msg_offsets[i] ..
 * msg_offsets[i+1]) (n+1 offsets).  Avoids the host-side gather of the pointer form. */
int ed25519_b200_verify_batch_flat(dalek_b200_ctx *ctx, const uint8_t *msgs_flat,
                                   const uint64_t *msg_offsets, const uint8_t *sigs,
                                   const uint8_t *pubkeys, size_t n);
/* Device-resident variant of the flat form (all four buffers are device pointers). */
int ed25519_b200_verify_batch_flat_dev(dalek_b200_ctx *ctx, const void *d_msgs_flat,
                                       const void *d_msg_offsets, const void *d_sigs,
                                       const void *d_pubkeys, size_t n, size_t msgs_bytes);
/* verify_batch for callers that hold VerifyingKeys: key_points[20 i ..] is the decompressed point of key i (X | Y | Z | T,
 * radix-2^51 limbs, the reference's in-memory EdwardsPoint; what VerifyingKey::from_bytes computed once, E/verifying.rs:
 * 65-71, :167-175) and pubkeys[32 i ..] its encoding (hashed as in batch.rs:179-191).  No key is decompressed inside the
 * call -- the reference's verify_batch does not either (batch.rs:236-238) -- so a batch whose keys are all different costs
 * what a batch with few keys costs.  The points are trusted to be the decodings of the encodings (as a VerifyingKey
 * guarantees); Z = 1 is free, another Z costs one inversion per distinct key.  Never returns POINT_DECOMPRESSION. */
int ed25519_b200_verify_batch_flat_points(dalek_b200_ctx *ctx, const uint8_t *msgs_flat, const uint64_t *msg_offsets,
                                          const uint8_t *sigs, const uint8_t *pubkeys, const uint64_t *key_points, size_t n);
int ed25519_b200_verify_batch_flat_points_dev(dalek_b200_ctx *ctx, const void *d_msgs_flat, const void *d_msg_offsets,
                                              const void *d_sigs, const void *d_pubkeys, const void *d_key_points, size_t n);
/* Many independent batches in one call (SURVEY 8d config 3B: 2^14 batches of 256): signatures
 * [k * batch_size, min(n, (k+1) * batch_size)) form batch k and verdicts[k] receives what
 * ed25519_dalek::verify_batch (batch.rs:146-251) returns for that batch alone (0 / 1 / 3 / 4); each batch
 * uses exactly the reference's transcript (whatever "verify_chunk" is).  A batch passes iff the value E_k of its equation
 * (batch.rs:240-250) is the identity.  The small-order part of every E_k is tested exactly, per batch (it only depends on the
 * scalars modulo 8: S_k = sum (z_i mod 8) R_i + sum ((z_i h_i mod l) mod 8) A_i, [l] S_k == identity) -- sums of batch
 * equations would let the small-order defects of different batches cancel, one input in eight.  For the prime-order parts the
 * combined equation over all undecided batches is tested first (independent transcripts: a non-zero prime-order part
 * leaves it non-zero except with the probability a forgery passes batch.rs itself, ~2^-125); only when it fails are halves
 * re-tested down to single batches, so a clean call costs little more than one large verify_batch, and k failing batches
 * add about k * log2(n / batch_size) partial re-tests.
 * Returns 0 if every verdict is 0, 1 otherwise, negative on engine errors.  verdicts: ceil(n / batch_size) ints (host). */
int ed25519_b200_verify_batches_flat(dalek_b200_ctx *ctx, const uint8_t *msgs_flat,
                                     const uint64_t *msg_offsets, const uint8_t *sigs,
                                     const uint8_t *pubkeys, size_t n, size_t batch_size, int32_t *verdicts);
int ed25519_b200_verify_batches_flat_dev(dalek_b200_ctx *ctx, const void *d_msgs_flat,
                                         const void *d_msg_offsets, const void *d_sigs,
                                         const void *d_pubkeys, size_t n, size_t batch_size, int32_t *verdicts);
/* The same for callers that hold VerifyingKeys (the reference's bench shape, E/benches/ed25519_benchmarks.rs:56-73: every key
 * different): key_points as in ed25519_b200_verify_batch_flat_points -- no key is decompressed inside the call (batch.rs:236-238). */
int ed25519_b200_verify_batches_flat_points(dalek_b200_ctx *ctx, const uint8_t *msgs_flat, const uint64_t *msg_offsets,
                                            const uint8_t *sigs, const uint8_t *pubkeys, const uint64_t *key_points, size_t n,
                                            size_t batch_size, int32_t *verdicts);
int ed25519_b200_verify_batches_flat_points_dev(dalek_b200_ctx *ctx, const void *d_msgs_flat, const void *d_msg_offsets,
                                                const void *d_sigs, const void *d_pubkeys, const void *d_key_points, size_t n,
                                                size_t batch_size, int32_t *verdicts);
/* Many independent single verifications (SURVEY 8f rank 3): results[i] = what VerifyingKey::from_bytes followed by
 * verify (strict = 0, E/verifying.rs:167-175, :203-219) or verify_strict (strict = 1, E/verifying.rs:359-382)
 * returns for signature i alone: 0 Ok, 1 Verify, 3 ScalarFormat, 4 PointDecompression.  R' = [s]B - [k]A is
 * recomputed (RCompute, E/verifying.rs:496-557) and its ENCODING compared with the signature's R bytes, so --
 * unlike verify_batch -- a non-canonical R is rejected; verify_strict also rejects small-order R or A.
 * When the batch holds few distinct keys (every key signing at least eight signatures on average; option "each_comb") the
 * 64 x 8 multiples (j+1) 16^i A of every distinct key are tabulated once per call and each signature costs 128 mixed
 * additions and no doubling; otherwise every signature pays its own 252 doublings.  Same results either way.
 * Returns 0 if every result is 0, 1 otherwise; negative on engine errors.  results: n bytes (host). */
int ed25519_b200_verify_each_flat(dalek_b200_ctx *ctx, const uint8_t *msgs_flat, const uint64_t *msg_offsets,
                                  const uint8_t *sigs, const uint8_t *pubkeys, size_t n, int strict,
                                  uint8_t *results);
int ed25519_b200_verify_each_flat_dev(dalek_b200_ctx *ctx, const void *d_msgs_flat, const void *d_msg_offsets,
                                      const void *d_sigs, const void *d_pubkeys, size_t n, int strict,
                                      uint8_t *results);
/* Debug/parity aid: the 16-byte z_i coefficients drawn in the last verify_batch call. */
int ed25519_b200_last_zs(dalek_b200_ctx *ctx, uint8_t *zs_out, size_t n);

/* -------- input synthesis (benchmarks / tests): fixed-base multiples and RFC 8032 signing ---- */
/* out[i] = scalars[i] * B as extended limbs (EdwardsPoint::mul_base, C/edwards.rs:918-928). */
int dalek_b200_edwards_mul_base_batch(dalek_b200_ctx *ctx, const uint8_t *scalars, size_t n,
                                      uint64_t *out_limbs /* n x 20 */, uint8_t *out_compressed /* n x 32, nullable */);
/* Deterministic Ed25519 keygen + sign on the GPU: seeds n x 32 B -> pubkeys n x 32 B, sigs n x 64 B
 * (E/signing.rs, hazmat.rs:40-99); message layout as in verify_batch_flat. */
int ed25519_b200_sign_batch_flat(dalek_b200_ctx *ctx, const uint8_t *seeds, const uint8_t *msgs_flat,
                                 const uint64_t *msg_offsets, size_t n, uint8_t *pubkeys_out,
                                 uint8_t *sigs_out);

#ifdef __cplusplus
}
#endif
#endif
