// api.cu -- the extern "C" boundary of libdalek_b200.so (include/dalek_b200.h): context handling,
// host<->device staging and the MSM entry points.  verify_batch lives in batch.cu, the
// constant-time / Ristretto entry points in straus.cu.
#include <cstring>
#include <new>
#include <random>

#include "../../include/dalek_b200.h"
#include "engine.h"

extern "C" {

int dalek_b200_init(int device, dalek_b200_ctx **out)
{
    if (!out) return DALEK_E_INVALID_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) return DALEK_E_NO_DEVICE;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return DALEK_E_NO_DEVICE;
    if (prop.major != 10) return DALEK_E_NO_DEVICE;   // built for sm_100a only; no fallback path
    if (cudaSetDevice(device) != cudaSuccess) return DALEK_E_CUDA;
    dalek_b200_ctx *ctx = new (std::nothrow) dalek_b200_ctx();
    if (!ctx) return DALEK_E_NOMEM;
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    try { std::random_device rd; for (int i = 0; i < 4; i++) ctx->hash_seed[i] ^= rd(); } catch (...) { }   // results never depend on it
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);       // (greatest priority is the lower number)
    if (cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
        cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, prio_lo) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->stream_copy, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithPriority(&ctx->stream3, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
        cudaStreamCreateWithPriority(&ctx->stream_hash, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
        cudaEventCreate(&ctx->ev_a) != cudaSuccess || cudaEventCreate(&ctx->ev_b) != cudaSuccess ||
        cudaEventCreate(&ctx->ev_call0) != cudaSuccess || cudaEventCreate(&ctx->ev_call1) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_join2, cudaEventDisableTiming) != cudaSuccess) {
        delete ctx;
        return DALEK_E_CUDA;
    }
    for (int i = 0; i < 8; i++)
        if (cudaEventCreateWithFlags(&ctx->ev_grp[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_hram[i], cudaEventDisableTiming) != cudaSuccess || cudaEventCreate(&ctx->ev_prep[i][0]) != cudaSuccess ||
            cudaEventCreate(&ctx->ev_prep[i][1]) != cudaSuccess) { delete ctx; return DALEK_E_CUDA; }
    *out = ctx;
    return DALEK_OK;
}

void dalek_b200_destroy(dalek_b200_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->stream2);
    cudaStreamSynchronize(ctx->stream3);
    cudaStreamSynchronize(ctx->stream_hash);
    DevBuf *bufs[] = {&ctx->scalars, &ctx->points_in, &ctx->points, &ctx->digits, &ctx->counts, &ctx->offsets,
                      &ctx->sorted, &ctx->buckets, &ctx->red_a, &ctx->red_b, &ctx->red_c, &ctx->red_d, &ctx->key_pts,
                      &ctx->result, &ctx->flags, &ctx->misc0, &ctx->misc1, &ctx->misc2, &ctx->misc3,
                      &ctx->misc4, &ctx->misc5, &ctx->zs, &ctx->base_table, &ctx->ntasks, &ctx->task_off, &ctx->tasks, &ctx->task_sums, &ctx->msg_offs, &ctx->sum_desc, &ctx->sum_part, &ctx->key_table, &ctx->key_acc, &ctx->task_order, &ctx->sig_status, &ctx->misc6, &ctx->each_pow, &ctx->each_tab, &ctx->each_kstat,
                      &ctx->bt_meta, &ctx->bt_status, &ctx->bt_res, &ctx->bt_nafs, &ctx->bt_tables, &ctx->bt_part};
    for (DevBuf *b : bufs) if (b->p) cudaFree(b->p);
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    cudaEventDestroy(ctx->ev_a); cudaEventDestroy(ctx->ev_b); cudaEventDestroy(ctx->ev_fork); cudaEventDestroy(ctx->ev_join);
    cudaEventDestroy(ctx->ev_join2); cudaEventDestroy(ctx->ev_call0); cudaEventDestroy(ctx->ev_call1);
    for (int i = 0; i < 8; i++) { cudaEventDestroy(ctx->ev_grp[i]); cudaEventDestroy(ctx->ev_hram[i]); cudaEventDestroy(ctx->ev_prep[i][0]); cudaEventDestroy(ctx->ev_prep[i][1]); }
    cudaStreamDestroy(ctx->stream_hash);
    cudaStreamDestroy(ctx->stream); cudaStreamDestroy(ctx->stream2); cudaStreamDestroy(ctx->stream_copy); cudaStreamDestroy(ctx->stream3);
    delete ctx;
}

const char *dalek_b200_last_error(const dalek_b200_ctx *ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }

int dalek_b200_set_option(dalek_b200_ctx *ctx, const char *name, long value)
{
    if (!ctx || !name) return DALEK_E_INVALID_ARG;
    if (!strcmp(name, "window_bits")) { if (value != 0 && (value < 4 || value > 20)) return DALEK_E_INVALID_ARG; ctx->opt_window_bits = value; return 0; }
    if (!strcmp(name, "host_chunks")) { if (value < 1 || value > 8) return DALEK_E_INVALID_ARG; ctx->opt_host_chunks = value; return 0; }
    if (!strcmp(name, "decompress_f64")) { ctx->opt_decompress_f64 = value ? 1 : 0; return 0; }
    if (!strcmp(name, "trace")) { ctx->opt_trace = value ? 1 : 0; return 0; }
    if (!strcmp(name, "precomp_tables")) { ctx->opt_precomp_tables = value ? 1 : 0; return 0; }
    if (!strcmp(name, "double_base_comb")) { ctx->opt_double_base_comb = value ? 1 : 0; return 0; }
    if (!strcmp(name, "dedupe_keys")) { ctx->opt_dedupe_keys = value ? 1 : 0; return 0; }
    if (!strcmp(name, "verify_pieces")) { if (value < 1 || value > 8) return DALEK_E_INVALID_ARG; ctx->opt_verify_pieces = value; return 0; }
    if (!strcmp(name, "transcript_warp")) { ctx->opt_transcript_warp = value ? 1 : 0; return 0; }
    if (!strcmp(name, "transcript_blocks")) { ctx->opt_transcript_blocks = value ? 1 : 0; return 0; }
    if (!strcmp(name, "each_comb")) { if (value < 0 || value > 2) return DALEK_E_INVALID_ARG; ctx->opt_each_comb = value; return 0; }
    if (!strcmp(name, "small_straus")) { ctx->opt_small_straus = value ? 1 : 0; return 0; }
    if (!strcmp(name, "acc_tma")) { ctx->opt_acc_tma = value ? 1 : 0; return 0; }
    if (!strcmp(name, "batch_bucket_min")) { if (value < 1 || value > 0x7fffffffL) return DALEK_E_INVALID_ARG; ctx->opt_batch_bucket_min = value; return 0; }
    if (!strcmp(name, "field_f64")) { ctx->opt_field_f64 = value ? 1 : 0; return 0; }
    if (!strcmp(name, "verify_chunk")) { if (value < 0 || value > (1 << 20)) return DALEK_E_INVALID_ARG; ctx->opt_verify_chunk = value; return 0; }
    return DALEK_E_INVALID_ARG;
}

uint64_t dalek_b200_launch_count(const dalek_b200_ctx *ctx) { return ctx ? ctx->launches : 0; }

int dalek_b200_last_kernel_ms(const dalek_b200_ctx *ctx, float *ms, int *launches)
{
    if (!ctx) return DALEK_E_INVALID_ARG;
    if (ms) *ms = ctx->last_kernel_ms;
    if (launches) *launches = ctx->last_kernel_launches;
    return 0;
}

int dalek_b200_last_stage_ms(const dalek_b200_ctx *ctx, const char *stage, float *ms)
{
    if (!ctx || !stage || !ms) return DALEK_E_INVALID_ARG;
    if (!strcmp(stage, "bucket_accumulate")) { *ms = ctx->last_kernel_ms; return 0; }
    if (!strcmp(stage, "decompress_R")) { *ms = ctx->last_prep_ms; return 0; }
    return DALEK_E_INVALID_ARG;
}

int dalek_b200_last_call_ms(const dalek_b200_ctx *ctx, float *ms)
{
    if (!ctx || !ms) return DALEK_E_INVALID_ARG;
    *ms = ctx->last_call_ms;
    return 0;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
static size_t point_in_bytes(int fmt) { return fmt == DALEK_POINTS_COMPRESSED ? 32 : 160; }

// device scalars/points -> window sums in ctx->red? -> result.  Returns reference-level code.
// Inputs (host or device) -> bucket sums -> window accumulators (-> result if d_result).
// Host inputs are streamed in chunks on a dedicated copy stream: while chunk k+1 crosses PCIe,
// chunk k is converted, sorted and added into the (persistent) bucket sums.
static int run_msm(dalek_b200_ctx *ctx, const void *scalars, const void *points_in, bool on_device, int point_fmt, size_t n,
                   size_t n_window /* the size the window width is chosen from: n, or the shard size of a sharded MSM */,
                   ge_p3_raw *d_windows, int *bad_out, MsmResult *d_result)
{
    int rc;
    const int kind = point_fmt == DALEK_POINTS_COMPRESSED ? PK_NIELS : PK_PNIELS;
    const size_t psz = kind == PK_NIELS ? sizeof(ge_niels_packed) : sizeof(ge_pniels_packed);
    const size_t pin = point_in_bytes(point_fmt);
    cudaStream_t st = ctx->stream;
    if ((rc = ws_reserve(ctx, ctx->points, std::max<size_t>(1, n) * psz))) return rc;
    if ((rc = ws_reserve(ctx, ctx->flags, 64))) return rc;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->flags.p, 0, 64, st));
    const int c = msm_choose_window_bits(ctx, n_window);
    // the reference's dispatch (edwards.rs:1025-1029): below 190 points vartime Straus -- here three launches
    // (straus_vt.cu) instead of the ~27 of the bucket pipeline; only for whole MSMs (a shard must yield window sums)
    const bool straus = d_result && n == n_window && n < STRAUS_VT_THRESHOLD && ctx->opt_small_straus && ctx->opt_field_f64;
    if (on_device) {
        if (straus) {
            if ((rc = msm_prepare_points(ctx, points_in, point_fmt, n, ctx->points.p, (int *)ctx->flags.p))) return rc;
            if ((rc = straus_vartime_msm(ctx, (const uint32_t *)scalars, ctx->points.p, kind, n, d_result))) return rc;
        } else {
            // the point conversion (or decompression) runs on the second stream under the digit / sort passes of the main one
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_fork, st));
            CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
            if ((rc = msm_prepare_points_on(ctx, ctx->stream2, points_in, point_fmt, n, ctx->points.p, (int *)ctx->flags.p))) return rc;
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_join, ctx->stream2));
            if ((rc = msm_accumulate_chunk(ctx, (const uint32_t *)scalars, ctx->points.p, kind, n, c, true, 0, 0, ctx->ev_join))) return rc;
        }
    } else {
        if ((rc = ws_reserve(ctx, ctx->scalars, std::max<size_t>(1, n) * 32))) return rc;
        if ((rc = ws_reserve(ctx, ctx->points_in, std::max<size_t>(1, n) * pin))) return rc;
        int K = n >= (1u << 18) ? (int)std::min<long>(8, std::max<long>(1, ctx->opt_host_chunks)) : 1;
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_fork, st));
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream_copy, ctx->ev_fork, 0));
        // equal pieces; more than two pieces do not pay: every piece re-runs the per-bucket passes
        // (scans, task lists) and revisits all bucket sums (profiles/sweep_r1.txt)
        for (int k = 0; k < K; k++) {
            const size_t i0 = n * k / K, i1 = n * (k + 1) / K, cnt = i1 - i0;
            char *ds = (char *)ctx->scalars.p + i0 * 32, *dp = (char *)ctx->points_in.p + i0 * pin;
            if (cnt) {
                CUDA_TRY(ctx, cudaMemcpyAsync(ds, (const char *)scalars + i0 * 32, cnt * 32, cudaMemcpyHostToDevice, ctx->stream_copy));
                CUDA_TRY(ctx, cudaMemcpyAsync(dp, (const char *)points_in + i0 * pin, cnt * pin, cudaMemcpyHostToDevice, ctx->stream_copy));
            }
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_grp[k], ctx->stream_copy));
            CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_grp[k], 0));
            char *dq = (char *)ctx->points.p + i0 * psz;
            if ((rc = msm_prepare_points(ctx, dp, point_fmt, cnt, dq, (int *)ctx->flags.p))) return rc;
            if (straus) {                                            // K = 1 for small inputs
                if ((rc = straus_vartime_msm(ctx, (const uint32_t *)ds, dq, kind, cnt, d_result))) return rc;
            } else if ((rc = msm_accumulate_chunk(ctx, (const uint32_t *)ds, dq, kind, cnt, c, k == 0))) return rc;
        }
    }
    if (!straus && (rc = msm_reduce_finish(ctx, c, d_windows, d_result))) return rc;
    if (bad_out) CUDA_TRY(ctx, cudaMemcpyAsync(bad_out, ctx->flags.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    return 0;
}

static int finish_msm(dalek_b200_ctx *ctx, const ge_p3_raw *d_windows, int ranks, size_t n_total,
                      uint8_t out_compressed[32], uint64_t out_limbs[20], uint32_t *is_identity, bool already_combined = false)
{
    int rc;
    int c = msm_choose_window_bits(ctx, n_total);
    int nwin = msm_window_count_for_bits(c);
    if ((rc = ws_reserve(ctx, ctx->result, sizeof(MsmResult)))) return rc;
    if (!already_combined && (rc = msm_combine_windows(ctx, d_windows, ranks, nwin, c, (MsmResult *)ctx->result.p))) return rc;
    if ((rc = pinned_reserve(ctx, sizeof(MsmResult) + 64))) return rc;
    MsmResult *h = (MsmResult *)ctx->h_pinned;
    CUDA_TRY(ctx, cudaMemcpyAsync(h, ctx->result.p, sizeof(MsmResult), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    if ((ms = elapsed_ms(ctx->ev_a, ctx->ev_b)) >= 0.f) ctx->last_kernel_ms = ms;
    if (out_compressed) memcpy(out_compressed, h->compressed, 32);
    if (out_limbs) memcpy(out_limbs, h->limbs, 160);
    if (is_identity) *is_identity = h->is_identity;
    return 0;
}

static int msm_common(dalek_b200_ctx *ctx, const void *scalars, const void *points, bool on_device, int point_fmt,
                      size_t n, uint8_t out_compressed[32], uint64_t out_limbs[20])
{
    if (!ctx || (n && (!scalars || !points)) || (point_fmt != DALEK_POINTS_COMPRESSED && point_fmt != DALEK_POINTS_EXTENDED))
        return DALEK_E_INVALID_ARG;
    if (n >= (1ull << 31)) return DALEK_E_INVALID_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CallTimer timer(ctx);
    int rc;
    int c = msm_choose_window_bits(ctx, n);
    int nwin = msm_window_count_for_bits(c);
    if ((rc = ws_reserve(ctx, ctx->misc0, (size_t)nwin * sizeof(ge_p3_raw)))) return rc;
    if ((rc = pinned_reserve(ctx, sizeof(MsmResult) + 64))) return rc;
    int *h_bad = (int *)((char *)ctx->h_pinned + sizeof(MsmResult));
    *h_bad = 0;
    if ((rc = ws_reserve(ctx, ctx->result, sizeof(MsmResult)))) return rc;
    if ((rc = run_msm(ctx, scalars, points, on_device, point_fmt, n, n, (ge_p3_raw *)ctx->misc0.p, h_bad, (MsmResult *)ctx->result.p))) return rc;
    if ((rc = finish_msm(ctx, (const ge_p3_raw *)ctx->misc0.p, 1, n, out_compressed, out_limbs, nullptr, true))) return rc;
    return *h_bad ? DALEK_NONE : DALEK_OK;
}

extern "C" {

int dalek_b200_edwards_vartime_msm(dalek_b200_ctx *ctx, const uint8_t *scalars, const void *points, int point_fmt,
                                   size_t n, uint8_t out_compressed[32], uint64_t out_limbs[20])
{
    return msm_common(ctx, scalars, points, false, point_fmt, n, out_compressed, out_limbs);
}

int dalek_b200_edwards_vartime_msm_dev(dalek_b200_ctx *ctx, const void *d_scalars, const void *d_points, int point_fmt,
                                       size_t n, uint8_t out_compressed[32], uint64_t out_limbs[20])
{
    return msm_common(ctx, d_scalars, d_points, true, point_fmt, n, out_compressed, out_limbs);
}

int dalek_b200_msm_window_count(dalek_b200_ctx *ctx, size_t n_shard)
{
    if (!ctx) return DALEK_E_INVALID_ARG;
    return msm_window_count_for_bits(msm_choose_window_bits(ctx, n_shard));
}

size_t dalek_b200_msm_partial_bytes(dalek_b200_ctx *ctx, size_t n_shard)
{
    if (!ctx) return 0;
    return (size_t)msm_window_count_for_bits(msm_choose_window_bits(ctx, n_shard)) * 160 + 8;
}

void *dalek_b200_stream(dalek_b200_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

}  // extern "C"

// A shard's record as it crosses the boundary (and the exchange between ranks): the window accumulators as
// canonical radix-2^51 limbs (20 u64 each, window 0 = least significant) followed by one u64 status word
// (non-zero: a compressed point of the shard did not decode).
__global__ void k_windows_to_record(const ge_p3_raw *__restrict__ win, int nwin, const int *__restrict__ bad, uint64_t *__restrict__ out)
{
    int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w == nwin) out[20 * (size_t)nwin] = (uint64_t)(*bad != 0);
    if (w >= nwin) return;
    ge_p3 p; ge_p3_raw r = win[w]; ge_p3_load_raw(p, r);
    fe_to_limbs51(out + 20 * w, p.X); fe_to_limbs51(out + 20 * w + 5, p.Y);
    fe_to_limbs51(out + 20 * w + 10, p.Z); fe_to_limbs51(out + 20 * w + 15, p.T);
}
// `ranks` records of `rec_words` u64 each -> ranks x nwin raw accumulators; *any_bad |= status words
__global__ void k_records_to_windows(const uint64_t *__restrict__ in, int ranks, int nwin, size_t rec_words,
                                     ge_p3_raw *__restrict__ win, int *__restrict__ any_bad)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ranks * nwin) return;
    const int r = t / nwin, w = t % nwin;
    const uint64_t *src = in + (size_t)r * rec_words + 20 * (size_t)w;
    ge_p3 p;
    fe_from_limbs51(p.X, src); fe_from_limbs51(p.Y, src + 5); fe_from_limbs51(p.Z, src + 10); fe_from_limbs51(p.T, src + 15);
    ge_p3_raw o; ge_p3_store_raw(o, p); win[t] = o;
    if (w == 0 && rec_words > 20 * (size_t)nwin && in[(size_t)r * rec_words + 20 * (size_t)nwin]) atomicOr(any_bad, 1);
}

// Enqueue the partial MSM of one shard on the context's stream and leave its record (window accumulators +
// status word) in ctx->misc1; nothing is synchronised.  ev_a .. ev_b bracket the bucket accumulation.
static int partial_enqueue(dalek_b200_ctx *ctx, const void *scalars, const void *points, bool on_device, int point_fmt,
                           size_t n_local, size_t n_shard, int *nwin_out)
{
    if (!ctx || (n_local && (!scalars || !points)) || n_local > n_shard ||
        (point_fmt != DALEK_POINTS_COMPRESSED && point_fmt != DALEK_POINTS_EXTENDED) || n_local >= (1ull << 31))
        return DALEK_E_INVALID_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    int rc;
    const int c = msm_choose_window_bits(ctx, n_shard);
    const int nwin = msm_window_count_for_bits(c);
    if ((rc = ws_reserve(ctx, ctx->misc0, (size_t)nwin * sizeof(ge_p3_raw)))) return rc;
    if ((rc = ws_reserve(ctx, ctx->misc1, (size_t)nwin * 160 + 8))) return rc;
    if ((rc = run_msm(ctx, scalars, points, on_device, point_fmt, n_local, n_shard, (ge_p3_raw *)ctx->misc0.p, nullptr, nullptr))) return rc;
    k_windows_to_record<<<(nwin + 1 + 63) / 64, 64, 0, ctx->stream>>>((const ge_p3_raw *)ctx->misc0.p, nwin, (const int *)ctx->flags.p,
                                                                     (uint64_t *)ctx->misc1.p);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    *nwin_out = nwin;
    return 0;
}

static void read_kernel_ms(dalek_b200_ctx *ctx)
{
    float ms = 0.f;
    if ((ms = elapsed_ms(ctx->ev_a, ctx->ev_b)) >= 0.f) ctx->last_kernel_ms = ms;
}

static int partial_common(dalek_b200_ctx *ctx, const void *scalars, const void *points, bool on_device, int point_fmt,
                          size_t n_local, size_t n_shard, uint64_t *out_windows)
{
    if (!ctx || !out_windows) return DALEK_E_INVALID_ARG;
    CallTimer timer(ctx);
    int rc, nwin = 0;
    if ((rc = partial_enqueue(ctx, scalars, points, on_device, point_fmt, n_local, n_shard, &nwin))) return rc;
    const size_t bytes = (size_t)nwin * 160 + 8;
    if ((rc = pinned_reserve(ctx, bytes))) return rc;
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_pinned, ctx->misc1.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    read_kernel_ms(ctx);
    memcpy(out_windows, ctx->h_pinned, (size_t)nwin * 160);
    uint64_t status; memcpy(&status, (const char *)ctx->h_pinned + (size_t)nwin * 160, 8);
    return status ? DALEK_NONE : DALEK_OK;
}

// dst_device >= 0: d_out_record lives on that (other) device -- the record crosses NVLink as a peer copy
int msm_partial_enqueue_record(dalek_b200_ctx *ctx, const void *scalars, const void *points, bool on_device, int point_fmt,
                               size_t n_local, size_t n_shard, void *d_out_record, int dst_device)
{
    if (!ctx || !d_out_record) return DALEK_E_INVALID_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_call0, ctx->stream));     // the device span ends in ..._combine_dev
    ctx->async_open = true;
    int rc, nwin = 0;
    if ((rc = partial_enqueue(ctx, scalars, points, on_device, point_fmt, n_local, n_shard, &nwin))) return rc;
    if (dst_device >= 0 && dst_device != ctx->device)
        CUDA_TRY(ctx, cudaMemcpyPeerAsync(d_out_record, dst_device, ctx->misc1.p, ctx->device, (size_t)nwin * 160 + 8, ctx->stream));
    else
        CUDA_TRY(ctx, cudaMemcpyAsync(d_out_record, ctx->misc1.p, (size_t)nwin * 160 + 8, cudaMemcpyDeviceToDevice, ctx->stream));
    return DALEK_OK;
}

// records (host or device) -> Horner over windows -> result read-back
int msm_combine_records(dalek_b200_ctx *ctx, const void *records, bool on_device, size_t rec_bytes, int ranks, size_t n_shard,
                        uint8_t out_compressed[32], uint64_t out_limbs[20])
{
    if (!ctx || !records || ranks < 1 || ranks > 1024) return DALEK_E_INVALID_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    int rc;
    const int c = msm_choose_window_bits(ctx, n_shard);
    const int nwin = msm_window_count_for_bits(c);
    const size_t cnt = (size_t)ranks * nwin;
    if ((rc = ws_reserve(ctx, ctx->red_c, cnt * sizeof(ge_p3_raw)))) return rc;
    if ((rc = ws_reserve(ctx, ctx->flags, 64))) return rc;
    if ((rc = ws_reserve(ctx, ctx->result, sizeof(MsmResult)))) return rc;
    if ((rc = pinned_reserve(ctx, sizeof(MsmResult) + 64))) return rc;
    cudaStream_t st = ctx->stream;
    const void *d_rec = records;
    if (!on_device) {
        if ((rc = ws_reserve(ctx, ctx->red_d, (size_t)ranks * rec_bytes))) return rc;
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->red_d.p, records, (size_t)ranks * rec_bytes, cudaMemcpyHostToDevice, st));
        d_rec = ctx->red_d.p;
    }
    int *d_bad = (int *)ctx->flags.p + 8;                       // flags[0] belongs to a partial call still in flight
    CUDA_TRY(ctx, cudaMemsetAsync(d_bad, 0, 4, st));
    k_records_to_windows<<<(unsigned)((cnt + 63) / 64), 64, 0, st>>>((const uint64_t *)d_rec, ranks, nwin, rec_bytes / 8,
                                                                      (ge_p3_raw *)ctx->red_c.p, d_bad);
    ctx->launches++;
    if ((rc = msm_combine_windows(ctx, (const ge_p3_raw *)ctx->red_c.p, ranks, nwin, c, (MsmResult *)ctx->result.p))) return rc;
    MsmResult *h = (MsmResult *)ctx->h_pinned;
    int *h_bad = (int *)((char *)ctx->h_pinned + sizeof(MsmResult));
    CUDA_TRY(ctx, cudaMemcpyAsync(h, ctx->result.p, sizeof(MsmResult), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(h_bad, d_bad, 4, cudaMemcpyDeviceToHost, st));
    if (ctx->async_open) CUDA_TRY(ctx, cudaEventRecord(ctx->ev_call1, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (ctx->async_open) {
        float ms = 0.f;
        if ((ms = elapsed_ms(ctx->ev_call0, ctx->ev_call1)) >= 0.f) ctx->last_call_ms = ms;
        read_kernel_ms(ctx);                                     // the bucket kernels of the partial call
        ctx->async_open = false;
    }
    if (out_compressed) memcpy(out_compressed, h->compressed, 32);
    if (out_limbs) memcpy(out_limbs, h->limbs, 160);
    return *h_bad ? DALEK_NONE : DALEK_OK;
}

extern "C" {

int dalek_b200_edwards_msm_partial(dalek_b200_ctx *ctx, const uint8_t *scalars, const void *points, int point_fmt,
                                   size_t n_local, size_t n_shard, uint64_t *out_windows)
{
    return partial_common(ctx, scalars, points, false, point_fmt, n_local, n_shard, out_windows);
}

int dalek_b200_edwards_msm_partial_dev(dalek_b200_ctx *ctx, const void *d_scalars, const void *d_points, int point_fmt,
                                       size_t n_local, size_t n_shard, uint64_t *out_windows)
{
    return partial_common(ctx, d_scalars, d_points, true, point_fmt, n_local, n_shard, out_windows);
}

int dalek_b200_edwards_msm_partial_async(dalek_b200_ctx *ctx, const uint8_t *scalars, const void *points, int point_fmt,
                                         size_t n_local, size_t n_shard, void *d_out_record)
{
    return msm_partial_enqueue_record(ctx, scalars, points, false, point_fmt, n_local, n_shard, d_out_record, -1);
}

int dalek_b200_edwards_msm_partial_dev_async(dalek_b200_ctx *ctx, const void *d_scalars, const void *d_points, int point_fmt,
                                             size_t n_local, size_t n_shard, void *d_out_record)
{
    return msm_partial_enqueue_record(ctx, d_scalars, d_points, true, point_fmt, n_local, n_shard, d_out_record, -1);
}

int dalek_b200_edwards_msm_combine(dalek_b200_ctx *ctx, const uint64_t *windows, int ranks, size_t n_shard,
                                   uint8_t out_compressed[32], uint64_t out_limbs[20])
{
    if (!ctx) return DALEK_E_INVALID_ARG;
    const size_t rec = (size_t)msm_window_count_for_bits(msm_choose_window_bits(ctx, n_shard)) * 160;   // no status words
    return msm_combine_records(ctx, windows, false, rec, ranks, n_shard, out_compressed, out_limbs);
}

int dalek_b200_edwards_msm_combine_dev(dalek_b200_ctx *ctx, const void *d_records, int ranks, size_t n_shard,
                                       uint8_t out_compressed[32], uint64_t out_limbs[20])
{
    if (!ctx) return DALEK_E_INVALID_ARG;
    return msm_combine_records(ctx, d_records, true, dalek_b200_msm_partial_bytes(ctx, n_shard), ranks, n_shard, out_compressed, out_limbs);
}

}  // extern "C"
