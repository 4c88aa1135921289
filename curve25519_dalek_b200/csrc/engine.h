// engine.h -- internal (C++) interface between the translation units of libdalek_b200.so.
// The public boundary is include/dalek_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <cstdio>
#include <string>
#include <utility>
#include <vector>

#include "ge.cuh"

// Batched MSM: default of the option "batch_bucket_min" (msm_batch.cu): the best value of the sweep in
// tools/msm_batch_bench.py on a B200 (profiles/msm_batch_r1.json)
#define BATCH_BUCKET_MIN_DEFAULT 65536

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct dalek_b200_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;
    cudaStream_t stream_copy = nullptr;
    cudaStream_t stream3 = nullptr;      // second transcript chain (odd verify pieces)
    cudaStream_t stream_hash = nullptr;  // SHA-512 of every verify piece: never queued behind a transcript (a long dependent chain)
    cudaEvent_t ev_hram[8] = {};         // "hram of piece k done" (stream_hash)
    cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_fork = nullptr, ev_join = nullptr, ev_join2 = nullptr;
    cudaEvent_t ev_call0 = nullptr, ev_call1 = nullptr;   // device span of the last hot-path call (CallTimer)
    cudaEvent_t ev_prep[8][2] = {};      // around the R-decompression kernel of each verify_batch piece (stream2)
    int prep_pieces = 0;
    float last_prep_ms = 0.f;            // their sum in the last verify_batch call
    cudaEvent_t ev_grp[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // one per input piece
    std::string last_error;
    uint64_t launches = 0;
    // options
    long opt_window_bits = 0;
    long opt_verify_chunk = 0;     // 0: the reference's single transcript over the whole batch; k > 0: opt-in, one transcript per k signatures
    long opt_host_chunks = 8;   // host-buffer MSM calls stream the pairs in this many chunks (copy/compute overlap)
    long opt_trace = 0;            // 1: print a per-stage device timeline of verify_batch calls to stderr (diagnostics)
    long opt_precomp_tables = 0;   // 1: precomputations of >= 4096 points also keep 2^(cw) P tables (one bucket window, no doublings)
    long opt_double_base_comb = 1; // double-base batch through the shared-memory fixed-base comb (0 = per-pair Straus)
    long opt_dedupe_keys = 1;   // verify_batch decompresses every distinct public key once
    long opt_verify_pieces = 4; // host-buffer verify_batch calls stream the signatures in this many pieces
    long opt_decompress_f64 = 1; // square-root exponentiation of point decompression on the FP64-pipe field
    long opt_acc_tma = 0;       // bucket kernel gathers points with TMA bulk copies + mbarriers instead of cp.async (A/B option)
    long opt_transcript_warp = 1; // up to 2048 Merlin transcripts per launch run one WARP each (25-lane Keccak); 0 = one thread each
    long opt_transcript_blocks = 1; // more transcripts than that: one THREAD each with the rate block staged in shared memory (0 = byte-wise sponge)
    long opt_each_comb = 1;     // verify_each: 1 = per-key comb tables when every key signs >= 8 signatures on average, 2 = always, 0 = never
    long opt_small_straus = 1;  // fewer than 190 pairs: vartime Straus (3 launches) instead of the bucket pipeline
    long opt_field_f64 = 1;     // bucket kernel on the FP64 pipe (fe64.cuh) instead of IMAD.WIDE (fe.cuh)
    long opt_batch_bucket_min = BATCH_BUCKET_MIN_DEFAULT;   // batched MSM: segments of at least this many pairs take the bucket pipeline
    // timing of the dominant kernel in the last call
    float last_kernel_ms = 0.f;
    float last_call_ms = 0.f;
    int last_kernel_launches = 0;
    bool async_open = false;       // a ..._partial_async call is in flight: its device span ends in ..._combine_dev
    // device workspaces (grown on demand, reused across calls)
    DevBuf scalars, points_in, points, digits, counts, offsets, sorted, buckets, red_a, red_b, red_c,
        red_d, key_pts, result, flags, misc0, misc1, misc2, misc3, misc4, misc5, zs, base_table, ntasks, task_off, tasks, task_sums, msg_offs, sum_desc, sum_part, key_table, key_acc, task_order, sig_status, misc6, each_pow, each_tab, each_kstat,
        bt_meta, bt_status, bt_res, bt_nafs, bt_tables, bt_part;   // batched MSM (msm_batch.cu)
    const uint64_t *key_points = nullptr;   // device: callers' decompressed key points for the current verify_batch call (or null)
    uint32_t hash_seed[4] = {0x243F6A88u, 0x85A308D3u, 0x13198A2Eu, 0x03707344u};   // key of the public-key de-duplication hash, redrawn per context
    int sum_desc_c = -1;
    bool base_table_ready = false;
    bool each_attr_set = false;     // the same for k_verify_each_comb
    bool comb_attr_set = false;     // cudaFuncAttributeMaxDynamicSharedMemorySize set for the comb kernel on this device
    // pinned host staging
    void *h_pinned = nullptr;
    size_t h_pinned_cap = 0;
    size_t last_zs_n = 0;
    std::vector<std::pair<const char *, cudaEvent_t>> trace;   // stage marks of the current call (opt_trace)
};

#define CUDA_TRY(ctx, expr)                                                                      \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            (ctx)->last_error = std::string(#expr) + ": " + cudaGetErrorString(_e);              \
            return -3;                                                                           \
        }                                                                                        \
    } while (0)

// Milliseconds between two events, or a negative value if either was never recorded / has not completed; a failure does
// not stay behind as the context's "last CUDA error" (a later cudaGetLastError() would report it for an innocent call).
inline float elapsed_ms(cudaEvent_t a, cudaEvent_t b)
{
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, a, b) == cudaSuccess) return ms;
    cudaGetLastError();
    return -1.f;
}

// Device time of one blocking call: an event on the main stream at entry, one after everything the call enqueued
// (the other streams are joined into the main one before a call returns); read with dalek_b200_last_call_ms.
struct CallTimer {
    dalek_b200_ctx *ctx;
    explicit CallTimer(dalek_b200_ctx *c) : ctx(c) { if (ctx) cudaEventRecord(ctx->ev_call0, ctx->stream); }
    ~CallTimer()
    {
        if (!ctx) return;
        float ms = 0.f;
        if (cudaEventRecord(ctx->ev_call1, ctx->stream) == cudaSuccess && cudaEventSynchronize(ctx->ev_call1) == cudaSuccess &&
            (ms = elapsed_ms(ctx->ev_call0, ctx->ev_call1)) >= 0.f)
            ctx->last_call_ms = ms;
    }
};

// diagnostics: timestamp `name` on `st` (relative to the CallTimer start), printed by trace_dump
inline void trace_mark(dalek_b200_ctx *ctx, const char *name, cudaStream_t st)
{
    if (!ctx->opt_trace) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, st);
    ctx->trace.push_back({name, e});
}
inline void trace_dump(dalek_b200_ctx *ctx)
{
    if (!ctx->opt_trace) return;
    cudaDeviceSynchronize();
    for (auto &m : ctx->trace) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ctx->ev_call0, m.second);
        fprintf(stderr, "[trace] %8.3f ms  %s\n", ms, m.first);
        cudaEventDestroy(m.second);
    }
    ctx->trace.clear();
}

int ws_reserve(dalek_b200_ctx *ctx, DevBuf &b, size_t bytes);
int pinned_reserve(dalek_b200_ctx *ctx, size_t bytes);

// ---- point preparation (msm.cu) ----
// kinds of device point arrays fed to the bucket kernels
enum { PK_NIELS = 0 /* ge_niels_packed, 96 B */, PK_PNIELS = 1 /* ge_pniels_packed, 128 B */ };

// Convert n input points (device memory, format DALEK_POINTS_*) into packed Niels form.
// Compressed inputs give PK_NIELS and set *d_bad (device int) nonzero if any fails to decode;
// extended inputs give PK_PNIELS.
int msm_prepare_points(dalek_b200_ctx *ctx, const void *d_in, int point_fmt, size_t n, void *d_out,
                       int *d_bad);

// Window width (bits) the engine uses for an MSM over n pairs.
int msm_choose_window_bits(const dalek_b200_ctx *ctx, size_t n);
int msm_window_count_for_bits(int c);

// Bucket MSM over device inputs: writes `nwin` window accumulators (raw p3) to d_windows.
int msm_window_sums(dalek_b200_ctx *ctx, const uint32_t *d_scalars /* n x 8 words */, const void *d_points,
                    int point_kind, size_t n, int c, ge_p3_raw *d_windows);
// total = sum over ranks of windows, Horner-combined; writes compressed (8 words) + canonical
// limbs51 (20 u64) + identity flag to d_result (layout: 8 u32 | pad | 20 u64 | u32 flag).
struct MsmResult { uint32_t compressed[8]; uint64_t limbs[20]; uint32_t is_identity; uint32_t pad; };
// building blocks: one chunk of pairs into the buckets; then reduction (+ Horner + encode if d_result)
// points_ready (optional): an event after which d_points may be read -- the digit and sort passes do not wait for it
int msm_accumulate_chunk(dalek_b200_ctx *ctx, const uint32_t *d_scalars, const void *d_points, int point_kind, size_t n,
                         int c, bool first, int active_windows = 0, size_t flat = 0, cudaEvent_t points_ready = nullptr);
int msm_prepare_points_on(dalek_b200_ctx *ctx, cudaStream_t st, const void *d_in, int point_fmt, size_t n, void *d_out, int *d_bad);
// window width for `n_short` scalars of `short_bits` bits plus `n_long` full-width scalars (verify_batch)
int msm_choose_window_bits_mixed(const dalek_b200_ctx *ctx, size_t n_short, int short_bits, size_t n_long);
int msm_reduce_finish(dalek_b200_ctx *ctx, int c, ge_p3_raw *d_windows, MsmResult *d_result, bool flat = false);
int msm_fill_identity(dalek_b200_ctx *ctx, ge_p3_raw *d_out, uint32_t count);
// window sums + Horner + encode in one go (single-shard case)
int msm_full(dalek_b200_ctx *ctx, const uint32_t *d_scalars, const void *d_points, int point_kind, size_t n, int c,
             ge_p3_raw *d_windows, MsmResult *d_result);
int msm_combine_windows(dalek_b200_ctx *ctx, const ge_p3_raw *d_windows, int ranks, int nwin, int c,
                        MsmResult *d_result);

// ---- sharded MSM building blocks (api.cu), shared with the single-process multi-GPU entry points (multi.cu) ----
// Enqueue the MSM of one shard on ctx's stream; its record (window accumulators + status word) is copied to
// d_out_record (on device dst_device if >= 0 and different from ctx's: a peer copy).  Nothing is synchronised.
int msm_partial_enqueue_record(dalek_b200_ctx *ctx, const void *scalars, const void *points, bool on_device, int point_fmt,
                               size_t n_local, size_t n_shard, void *d_out_record, int dst_device);
// `ranks` records (host or device, rec_bytes apart) -> per-window sums, Horner, encode; blocks for the result.
int msm_combine_records(dalek_b200_ctx *ctx, const void *records, bool on_device, size_t rec_bytes, int ranks, size_t n_shard,
                        uint8_t out_compressed[32], uint64_t out_limbs[20]);

// ---- front end of verify_batch reused by the per-signature verifier (batch.cu -> single.cu) ----
struct EachFront { const uint32_t *hs; const uint8_t *bad_s; const uint32_t *rep, *dense, *uniq; size_t nkeys; };
int verify_each_front(dalek_b200_ctx *ctx, const uint8_t *d_msgs, const uint64_t *d_offs, const uint32_t *d_sigs, const uint32_t *d_keys,
                      size_t n, EachFront *out);

// ---- variable-time Straus for small inputs (straus_vt.cu): the reference's path below 190 points ----
#define STRAUS_VT_THRESHOLD 190            // edwards.rs:1025-1029
int straus_vartime_msm(dalek_b200_ctx *ctx, const uint32_t *d_scalars, const void *d_points, int point_kind, size_t n,
                       MsmResult *d_result);

// ---- constant-time Straus (straus.cu) ----
int straus_ct_msm(dalek_b200_ctx *ctx, const uint32_t *d_scalars, const void *d_points_pniels, size_t n,
                  MsmResult *d_result);
// ---- fixed-base table (base.cu): 64 x 8 affine Niels entries (j+1) 16^i B, built once per context ----
int base_table_ensure(dalek_b200_ctx *ctx);

int ristretto_prepare_points(dalek_b200_ctx *ctx, const void *d_in, size_t n, void *d_out, int *d_bad);

// ---- batched MSM (msm_batch.cu): building blocks in msm.cu / straus.cu / straus_vt.cu ----
// A point that does not decode marks its SEGMENT: bad[k] = 1 for the k with offs[k] <= base + i < offs[k + 1]
// (offs: m + 1 non-decreasing device u64), instead of the call-wide flag.
struct SegStatus { const uint64_t *offs; size_t m; uint64_t base; uint32_t *bad; };
#ifdef __CUDACC__
__device__ __forceinline__ void seg_mark_bad(const SegStatus &s, size_t i)
{
    const uint64_t g = s.base + i;
    size_t lo = 0, hi = s.m;                       // last k with offs[k] <= g (empty segments are skipped)
    while (hi - lo > 1) { const size_t mid = (lo + hi) / 2; if (s.offs[mid] <= g) lo = mid; else hi = mid; }
    s.bad[lo] = 1;
}
#endif
// point_fmt: DALEK_POINTS_COMPRESSED (-> PK_NIELS), _EXTENDED or _RISTRETTO (-> PK_PNIELS)
int msm_prepare_points_seg(dalek_b200_ctx *ctx, cudaStream_t st, const void *d_in, int point_fmt, size_t n, void *d_out,
                           const SegStatus &seg);
int ristretto_prepare_points_seg(dalek_b200_ctx *ctx, cudaStream_t st, const void *d_in, size_t n, void *d_out, const SegStatus &seg);
// width-5 NAF (NAF_LEN bytes) and the table of odd multiples (8 projective Niels) of n pairs (k_straus_prepare)
int straus_prepare(dalek_b200_ctx *ctx, cudaStream_t st, const uint32_t *d_scalars, const void *d_points, int point_kind, size_t n,
                   int8_t *d_nafs, ge_pniels_packed *d_tables);
// out[k] = sum of pool[d.x .. d.x + d.y) for the count descriptors d = desc[k] (uint2, device)
int msm_plain_sums(dalek_b200_ctx *ctx, cudaStream_t st, const ge_p3_raw *pool, const void *d_desc, uint32_t count, ge_p3_raw *out);
int ristretto_encode_result(dalek_b200_ctx *ctx, const MsmResult *d_res, uint32_t *d_enc);
int ristretto_double_base(dalek_b200_ctx *ctx, const uint8_t *d_a, const uint8_t *d_b, const uint8_t G[32],
                          const uint8_t H[32], size_t n, uint8_t *d_out, int *h_status);
