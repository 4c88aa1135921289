// msm_batch.cu -- m independent vartime multiscalar multiplications in one call (VartimeMultiscalarMul::
// optional_multiscalar_mul, traits.rs:196-262, once per segment of the flat pair arrays), Edwards and Ristretto.
//
// A single MSM call has a fixed floor of a few hundred microseconds (dependent launches, read-back); callers with many
// small MSMs (vector-commitment provers, per-proof verification) would pay it once per MSM.  Here the whole batch is a
// handful of launches per piece of ~2^20 pairs, whatever m is.  The host plan (msm_batch.cuh) sends
//   * segments of >= batch_bucket_min pairs to the bucket pipeline (msm.cu), one segment after another, each writing
//     its slot of a device result array (no read-back per segment);
//   * all shorter segments (and at most BATCH_PIECE_PAIRS long) to a segmented vartime Straus, in pieces of at most
//     BATCH_PIECE_PAIRS pairs cut at segment boundaries:
//       k_prep_* (msm.cu / straus.cu)   decode / convert the points; a bad point marks its segment only
//       k_straus_prepare (straus_vt.cu) per pair: width-5 NAF and the table of odd multiples
//       k_straus_tasks                  one 4-lane group per task (<= p consecutive pairs of one segment), one
//                                       accumulator per task, uniform op stream (msm_batch.cuh)
//       k_plain_sum (msm.cu)            per segment: sum of its task accumulators
//       k_batch_encode                  per segment: EdwardsPoint::compress + limbs (as k_combine writes them)
// Ristretto results are then encoded with RistrettoPoint::compress (k_batch_ristretto_encode), one thread per result.
// Host-buffer calls copy piece k + 1 in on the copy stream while piece k computes.
#include <algorithm>
#include <cstring>

#include "../../include/dalek_b200.h"
#include "engine.h"
#include "warp4.cuh"
#include "msm_batch.cuh"

static inline unsigned cdiv(size_t a, unsigned b) { return (unsigned)((a + b - 1) / b); }

__global__ void __launch_bounds__(128)
k_straus_tasks(const int8_t *__restrict__ nafs, const ge_pniels_packed *__restrict__ tables, const BatchTask *__restrict__ tasks,
               uint32_t ntasks, ge_p3_raw *__restrict__ partial)
{
    const uint32_t role = threadIdx.x & 3;
    const uint32_t t = (blockIdx.x * blockDim.x + threadIdx.x) >> 2;
    if (((blockIdx.x * blockDim.x + (threadIdx.x & ~31u)) >> 2) >= ntasks) return;    // whole warp out of range
    const bool live = t < ntasks;
    const BatchTask tk = tasks[live ? t : 0];
    w4f_point Q;
    straus_task_group(Q, nafs, tables, tk.pair, tk.len, live, role);
    if (live) {
        ge_p3 o; w4f_to_p3(o, Q);
        fe mine; fe_sel4(mine, o.X, o.Y, o.Z, o.T, role);
        uint32_t *dst = partial[t].w + 10 * role;
#pragma unroll
        for (int i = 0; i < 10; i += 2) *reinterpret_cast<uint2 *>(dst + i) = make_uint2(mine.v[i], mine.v[i + 1]);
    }
}

// one thread per segment: the result record of k_combine (compressed, canonical limbs, identity flag)
__global__ void k_batch_encode(const ge_p3_raw *__restrict__ sums, uint32_t count, MsmResult *__restrict__ res)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    ge_p3 p; ge_p3_raw r = sums[i]; ge_p3_load_raw(p, r);
    uint32_t s[8];
    ge_compress(s, p);
    MsmResult &o = res[i];
#pragma unroll
    for (int k = 0; k < 8; k++) o.compressed[k] = s[k];
    fe_to_limbs51(o.limbs, p.X); fe_to_limbs51(o.limbs + 5, p.Y); fe_to_limbs51(o.limbs + 10, p.Z); fe_to_limbs51(o.limbs + 15, p.T);
    o.is_identity = ge_is_identity(p);
    o.pad = 0;
}

// one thread per result: RistrettoPoint::compress (ristretto.rs:980-994), the batched k_ristretto_encode_result
__global__ void k_batch_ristretto_encode(const MsmResult *__restrict__ res, size_t m, uint32_t *__restrict__ out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    ge_p3 p;
    fe_from_limbs51(p.X, res[i].limbs); fe_from_limbs51(p.Y, res[i].limbs + 5);
    fe_from_limbs51(p.Z, res[i].limbs + 10); fe_from_limbs51(p.T, res[i].limbs + 15);
    uint32_t enc[8];
    ristretto_compress(enc, p);
#pragma unroll
    for (int k = 0; k < 8; k++) out[8 * i + k] = enc[k];
}

// point_fmt: DALEK_POINTS_COMPRESSED / _EXTENDED (Edwards) or DALEK_POINTS_RISTRETTO
static int msm_batch(dalek_b200_ctx *ctx, const uint8_t *scalars, const void *points, bool on_device, int point_fmt,
                     const uint64_t *offsets, size_t m, uint8_t *out_compressed, uint64_t *out_limbs, uint8_t *status)
{
    if (!ctx) return DALEK_E_INVALID_ARG;
    if (point_fmt != DALEK_POINTS_COMPRESSED && point_fmt != DALEK_POINTS_EXTENDED && point_fmt != DALEK_POINTS_RISTRETTO) {
        ctx->last_error = "point_fmt"; return DALEK_E_INVALID_ARG;
    }
    if (m == 0) return DALEK_OK;
    if (m >= (1ull << 31)) { ctx->last_error = "m must be below 2^31"; return DALEK_E_INVALID_ARG; }
    if (!offsets || !out_compressed || !status) { ctx->last_error = "null buffer"; return DALEK_E_INVALID_ARG; }
    if (offsets[0] != 0) { ctx->last_error = "offsets[0] must be 0"; return DALEK_E_INVALID_ARG; }
    for (size_t k = 0; k < m; k++)
        if (offsets[k + 1] < offsets[k]) { ctx->last_error = "offsets must not decrease"; return DALEK_E_INVALID_ARG; }
    const uint64_t n = offsets[m];
    if (n >= (1ull << 31)) { ctx->last_error = "offsets[m] must be below 2^31"; return DALEK_E_INVALID_ARG; }
    if (n && (!scalars || !points)) { ctx->last_error = "null buffer"; return DALEK_E_INVALID_ARG; }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CallTimer timer(ctx);
    int rc;
    cudaStream_t st = ctx->stream;

    BatchPlan plan;
    batch_plan(plan, offsets, m, (uint64_t)ctx->opt_batch_bucket_min, ctx->sm_count, BATCH_PIECE_PAIRS);
    size_t max_pairs = 1, max_tasks = 1, max_segs = 1, ntask_all = 0, nsum_all = 0;
    for (const BatchPiece &pc : plan.pieces) {
        if (pc.bucket) continue;
        max_pairs = std::max<size_t>(max_pairs, pc.pair1 - pc.pair0);
        max_tasks = std::max(max_tasks, pc.tasks.size());
        max_segs = std::max(max_segs, pc.sums.size());
        ntask_all += pc.tasks.size(); nsum_all += pc.sums.size();
    }
    // device metadata: offsets (m + 1 u64) | tasks of every Straus piece | their sum descriptors
    std::vector<uint64_t> meta(m + 1 + ntask_all + nsum_all);
    memcpy(meta.data(), offsets, (m + 1) * 8);
    std::vector<size_t> task_base(plan.pieces.size()), sum_base(plan.pieces.size());
    {
        size_t t = m + 1, s = m + 1 + ntask_all;
        for (size_t q = 0; q < plan.pieces.size(); q++) {
            const BatchPiece &pc = plan.pieces[q];
            task_base[q] = t; sum_base[q] = s;
            if (!pc.tasks.empty()) memcpy(&meta[t], pc.tasks.data(), pc.tasks.size() * 8);
            if (!pc.sums.empty()) memcpy(&meta[s], pc.sums.data(), pc.sums.size() * 8);
            t += pc.tasks.size(); s += pc.sums.size();
        }
    }
    const bool ristretto = point_fmt == DALEK_POINTS_RISTRETTO;
    const int kind = point_fmt == DALEK_POINTS_COMPRESSED ? PK_NIELS : PK_PNIELS;
    const size_t psz = kind == PK_NIELS ? sizeof(ge_niels_packed) : sizeof(ge_pniels_packed);
    const size_t pin = point_fmt == DALEK_POINTS_EXTENDED ? 160 : 32;
    const size_t n1 = std::max<uint64_t>(1, n);
    const size_t res_bytes = m * sizeof(MsmResult), enc_bytes = ristretto ? m * 32 : 0;
    if ((rc = ws_reserve(ctx, ctx->bt_meta, meta.size() * 8))) return rc;
    if ((rc = ws_reserve(ctx, ctx->bt_status, m * 4))) return rc;
    if ((rc = ws_reserve(ctx, ctx->bt_res, res_bytes + enc_bytes))) return rc;
    if ((rc = ws_reserve(ctx, ctx->points, n1 * psz))) return rc;
    if ((rc = ws_reserve(ctx, ctx->bt_nafs, max_pairs * NAF_LEN))) return rc;
    if ((rc = ws_reserve(ctx, ctx->bt_tables, max_pairs * 8 * sizeof(ge_pniels_packed)))) return rc;
    if ((rc = ws_reserve(ctx, ctx->bt_part, (max_tasks + max_segs) * sizeof(ge_p3_raw)))) return rc;
    if (!on_device) {
        if ((rc = ws_reserve(ctx, ctx->scalars, n1 * 32))) return rc;
        if ((rc = ws_reserve(ctx, ctx->points_in, n1 * pin))) return rc;
    }
    if ((rc = pinned_reserve(ctx, (ristretto ? enc_bytes : res_bytes) + m * 4))) return rc;
    const uint64_t *d_offs = (const uint64_t *)ctx->bt_meta.p;
    uint32_t *d_status = (uint32_t *)ctx->bt_status.p;
    MsmResult *d_res = (MsmResult *)ctx->bt_res.p;
    ge_p3_raw *d_part = (ge_p3_raw *)ctx->bt_part.p, *d_sums = d_part + max_tasks;
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->bt_meta.p, meta.data(), meta.size() * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemsetAsync(d_status, 0, m * 4, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));                  // `meta` is a host temporary
    const uint8_t *d_scalars = on_device ? scalars : (const uint8_t *)ctx->scalars.p;
    const uint8_t *d_points_in = on_device ? (const uint8_t *)points : (const uint8_t *)ctx->points_in.p;
    uint8_t *d_points = (uint8_t *)ctx->points.p;
    if (!on_device) {
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_fork, st));
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream_copy, ctx->ev_fork, 0));
    }
    for (size_t q = 0; q < plan.pieces.size(); q++) {
        const BatchPiece &pc = plan.pieces[q];
        const uint64_t p0 = pc.pair0, cnt = pc.pair1 - pc.pair0;
        if (!on_device && cnt) {                                  // copy-in of this piece overlaps the kernels of the previous ones
            CUDA_TRY(ctx, cudaMemcpyAsync((char *)ctx->scalars.p + p0 * 32, scalars + p0 * 32, cnt * 32, cudaMemcpyHostToDevice,
                                          ctx->stream_copy));
            CUDA_TRY(ctx, cudaMemcpyAsync((char *)ctx->points_in.p + p0 * pin, (const char *)points + p0 * pin, cnt * pin,
                                          cudaMemcpyHostToDevice, ctx->stream_copy));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_grp[q & 7], ctx->stream_copy));
            CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_grp[q & 7], 0));
        }
        const SegStatus seg{d_offs, m, p0, d_status};
        if ((rc = msm_prepare_points_seg(ctx, st, d_points_in + p0 * pin, point_fmt, cnt, d_points + p0 * psz, seg))) return rc;
        const uint32_t *sc = (const uint32_t *)(d_scalars + p0 * 32);
        if (pc.bucket) {
            const int c = msm_choose_window_bits(ctx, cnt);
            if ((rc = ws_reserve(ctx, ctx->misc0, (size_t)msm_window_count_for_bits(c) * sizeof(ge_p3_raw)))) return rc;
            if ((rc = msm_accumulate_chunk(ctx, sc, d_points + p0 * psz, kind, cnt, c, true))) return rc;
            if ((rc = msm_reduce_finish(ctx, c, (ge_p3_raw *)ctx->misc0.p, d_res + pc.seg0))) return rc;
            continue;
        }
        const uint32_t ntasks = (uint32_t)pc.tasks.size(), nseg = (uint32_t)pc.sums.size();
        if (ntasks) {
            if ((rc = straus_prepare(ctx, st, sc, d_points + p0 * psz, kind, cnt, (int8_t *)ctx->bt_nafs.p, (ge_pniels_packed *)ctx->bt_tables.p))) return rc;
            k_straus_tasks<<<cdiv((size_t)ntasks * 4, 128), 128, 0, st>>>((const int8_t *)ctx->bt_nafs.p, (const ge_pniels_packed *)ctx->bt_tables.p,
                                                                          (const BatchTask *)(d_offs + task_base[q]), ntasks, d_part);
            ctx->launches++;
        }
        if ((rc = msm_plain_sums(ctx, st, d_part, d_offs + sum_base[q], nseg, d_sums))) return rc;
        k_batch_encode<<<cdiv(nseg, 128), 128, 0, st>>>(d_sums, nseg, d_res + pc.seg0);
        ctx->launches++;
        CUDA_TRY(ctx, cudaGetLastError());
    }
    uint8_t *h = (uint8_t *)ctx->h_pinned;
    const size_t out_bytes = ristretto ? enc_bytes : res_bytes;
    if (ristretto) {
        uint32_t *d_enc = (uint32_t *)((char *)ctx->bt_res.p + res_bytes);
        k_batch_ristretto_encode<<<cdiv(m, 128), 128, 0, st>>>(d_res, m, d_enc);
        ctx->launches++;
        CUDA_TRY(ctx, cudaMemcpyAsync(h, d_enc, enc_bytes, cudaMemcpyDeviceToHost, st));
    } else {
        CUDA_TRY(ctx, cudaMemcpyAsync(h, d_res, res_bytes, cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(ctx, cudaMemcpyAsync(h + out_bytes, d_status, m * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    const uint32_t *hs = (const uint32_t *)(h + out_bytes);
    bool any = false;
    for (size_t k = 0; k < m; k++) {
        const bool bad = hs[k] != 0;
        any |= bad;
        status[k] = bad ? 1 : 0;
        const void *src = ristretto ? (const void *)(h + 32 * k) : (const void *)((const MsmResult *)h)[k].compressed;
        if (bad) memset(out_compressed + 32 * k, 0, 32); else memcpy(out_compressed + 32 * k, src, 32);
        if (out_limbs) {
            if (bad) memset(out_limbs + 20 * k, 0, 160); else memcpy(out_limbs + 20 * k, ((const MsmResult *)h)[k].limbs, 160);
        }
    }
    return any ? DALEK_NONE : DALEK_OK;
}

extern "C" {

int dalek_b200_edwards_vartime_msm_batch(dalek_b200_ctx *ctx, const uint8_t *scalars, const void *points, int point_fmt,
                                         const uint64_t *offsets, size_t m, uint8_t *out_compressed, uint64_t *out_limbs,
                                         uint8_t *status)
{
    if (ctx && point_fmt == DALEK_POINTS_RISTRETTO) ctx->last_error = "point_fmt: the Ristretto form is dalek_b200_ristretto_vartime_msm_batch";
    if (point_fmt == DALEK_POINTS_RISTRETTO) return DALEK_E_INVALID_ARG;
    return msm_batch(ctx, scalars, points, false, point_fmt, offsets, m, out_compressed, out_limbs, status);
}

int dalek_b200_edwards_vartime_msm_batch_dev(dalek_b200_ctx *ctx, const void *d_scalars, const void *d_points, int point_fmt,
                                             const uint64_t *offsets, size_t m, uint8_t *out_compressed, uint64_t *out_limbs,
                                             uint8_t *status)
{
    if (ctx && point_fmt == DALEK_POINTS_RISTRETTO) ctx->last_error = "point_fmt: the Ristretto form is dalek_b200_ristretto_vartime_msm_batch";
    if (point_fmt == DALEK_POINTS_RISTRETTO) return DALEK_E_INVALID_ARG;
    return msm_batch(ctx, (const uint8_t *)d_scalars, d_points, true, point_fmt, offsets, m, out_compressed, out_limbs, status);
}

int dalek_b200_ristretto_vartime_msm_batch(dalek_b200_ctx *ctx, const uint8_t *scalars, const uint8_t *points,
                                           const uint64_t *offsets, size_t m, uint8_t *out_compressed, uint8_t *status)
{
    return msm_batch(ctx, scalars, points, false, DALEK_POINTS_RISTRETTO, offsets, m, out_compressed, nullptr, status);
}

}  // extern "C"
