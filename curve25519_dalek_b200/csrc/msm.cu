// msm.cu -- bucket-method (Pippenger) multiscalar multiplication on one B200.
//
// Replaces curve25519-dalek/src/backend/serial/scalar_mul/pippenger.rs:67-160 (and, being
// size-agnostic, the vartime Straus path straus.rs:159-200 the reference dispatches to below 190
// points, src/edwards.rs:1025-1029).  The reference walks 33-43 windows of 6-8 bits serially;
// here all windows run at once with c = 4..20-bit signed digits:
//
//   k_digits            one thread per scalar: signed radix-2^c digits (scalar.rs:1093-1150
//                       generalised to c > 8), histogram of bucket sizes, rank inside the bucket
//   k_scan_*            exclusive scan of the bucket sizes per window (multi-block)
//   k_scatter           counting-sort scatter: point indices grouped by (window, bucket)
//   k_task_count/fill   buckets cut into tasks of <= task_len entries (skewed / adversarial inputs)
//   k_task_hist/scan/scatter
//                       counting sort of the tasks by length: warps run equal trip counts and the
//                       grid drains longest-first
//   k_bucket_accumulate one thread per task: sum of its points with the complete unified mixed
//                       addition (curve_models.rs:411-494), 7M (affine Niels) or 8M, on the
//                       FP64-pipe field (fe64.cuh) with cp.async point prefetch
//   k_heavy_fixup       sums the task sums of buckets that were cut
//   k_chunk_reduce, k_plain_sum, k_finish_windows
//                       sum_k k*B_k per window (pippenger.rs:146-151) in log depth on 4-lane groups
//   k_combine           total = total*2^c + window (pippenger.rs:159), compress
//
// Data layout in HBM: scalars n x 32 B; points packed Niels (96 B) or projective Niels (128 B),
// canonical 32-byte coordinates, 16-byte aligned for 128-bit loads; digit/rank entries 8 B per
// (window, scalar); sorted indices 4 B per entry; bucket sums 160 B (10 x u32 limbs x 4).
#include <algorithm>
#include <cstdio>
#include <utility>
#include <vector>

#include "../../include/dalek_b200.h"
#include "engine.h"
#include "ge64.cuh"
#include "warp4.cuh"
#include "warp4_f64.cuh"

// ------------------------------------------------------------------------------------------
static inline unsigned cdiv(size_t a, unsigned b) { return (unsigned)((a + b - 1) / b); }

int ws_reserve(dalek_b200_ctx *ctx, DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap) return 0;
    if (b.p) { cudaFree(b.p); b.p = nullptr; b.cap = 0; }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) { ctx->last_error = std::string("cudaMalloc: ") + cudaGetErrorString(e); return DALEK_E_NOMEM; }
    b.cap = want;
    return 0;
}

int pinned_reserve(dalek_b200_ctx *ctx, size_t bytes)
{
    if (bytes <= ctx->h_pinned_cap) return 0;
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    ctx->h_pinned = nullptr; ctx->h_pinned_cap = 0;
    cudaError_t e = cudaMallocHost(&ctx->h_pinned, bytes + 4096);
    if (e != cudaSuccess) { ctx->last_error = std::string("cudaMallocHost: ") + cudaGetErrorString(e); return DALEK_E_NOMEM; }
    ctx->h_pinned_cap = bytes + 4096;
    return 0;
}

// ------------------------------------------------------------------------------------------
// point preparation
// SEG = 1: a point that does not decode marks its segment (batched MSM) instead of the call-wide flag
template <int F64, int SEG>
__global__ void __launch_bounds__(128, 3) k_prep_compressed(const uint4 *__restrict__ in, ge_niels_packed *__restrict__ out, size_t n,
                                  int *__restrict__ bad, SegStatus seg)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4 a = in[2 * i], b = in[2 * i + 1];
    uint32_t s[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    fe x, y;
    uint32_t ok = ge_decompress_affine<F64>(x, y, s);
    if (!ok) {                                          // identity placeholder keeps the kernels total
        if (SEG) seg_mark_bad(seg, i); else atomicOr(bad, 1);
        fe_0(x); fe_1(y);
    }
    ge_niels nl; ge_affine_to_niels(nl, x, y);
    ge_niels_packed p; ge_niels_pack(p, nl);
    uint4 *o = reinterpret_cast<uint4 *>(out + i);
#pragma unroll
    for (int k = 0; k < 6; k++) o[k] = make_uint4(p.w[4 * k], p.w[4 * k + 1], p.w[4 * k + 2], p.w[4 * k + 3]);
}

__global__ void k_prep_extended(const uint64_t *__restrict__ in, ge_pniels_packed *__restrict__ out, size_t n)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const ulonglong2 *src = reinterpret_cast<const ulonglong2 *>(in + 20 * i);
    uint64_t l[20];
#pragma unroll
    for (int k = 0; k < 10; k++) { ulonglong2 v = src[k]; l[2 * k] = v.x; l[2 * k + 1] = v.y; }
    ge_p3 p;
    fe_from_limbs51(p.X, l); fe_from_limbs51(p.Y, l + 5); fe_from_limbs51(p.Z, l + 10); fe_from_limbs51(p.T, l + 15);
    ge_pniels pn; ge_p3_to_pniels(pn, p);
    ge_pniels_packed pk; ge_pniels_pack(pk, pn);
    uint4 *o = reinterpret_cast<uint4 *>(out + i);
#pragma unroll
    for (int k = 0; k < 8; k++) o[k] = make_uint4(pk.w[4 * k], pk.w[4 * k + 1], pk.w[4 * k + 2], pk.w[4 * k + 3]);
}

int msm_prepare_points_on(dalek_b200_ctx *ctx, cudaStream_t st, const void *d_in, int point_fmt, size_t n, void *d_out, int *d_bad)
{
    if (n == 0) return 0;
    if (point_fmt == DALEK_POINTS_COMPRESSED) {
        if (ctx->opt_decompress_f64) k_prep_compressed<1, 0><<<cdiv(n, 128), 128, 0, st>>>((const uint4 *)d_in, (ge_niels_packed *)d_out, n, d_bad, SegStatus{});
        else k_prep_compressed<0, 0><<<cdiv(n, 128), 128, 0, st>>>((const uint4 *)d_in, (ge_niels_packed *)d_out, n, d_bad, SegStatus{});
    } else {
        k_prep_extended<<<cdiv(n, 128), 128, 0, st>>>((const uint64_t *)d_in, (ge_pniels_packed *)d_out, n);
    }
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

int msm_prepare_points(dalek_b200_ctx *ctx, const void *d_in, int point_fmt, size_t n, void *d_out, int *d_bad)
{
    return msm_prepare_points_on(ctx, ctx->stream, d_in, point_fmt, n, d_out, d_bad);
}

int msm_prepare_points_seg(dalek_b200_ctx *ctx, cudaStream_t st, const void *d_in, int point_fmt, size_t n, void *d_out,
                           const SegStatus &seg)
{
    if (n == 0) return 0;
    if (point_fmt == DALEK_POINTS_RISTRETTO) return ristretto_prepare_points_seg(ctx, st, d_in, n, d_out, seg);
    if (point_fmt == DALEK_POINTS_COMPRESSED) {
        if (ctx->opt_decompress_f64) k_prep_compressed<1, 1><<<cdiv(n, 128), 128, 0, st>>>((const uint4 *)d_in, (ge_niels_packed *)d_out, n, nullptr, seg);
        else k_prep_compressed<0, 1><<<cdiv(n, 128), 128, 0, st>>>((const uint4 *)d_in, (ge_niels_packed *)d_out, n, nullptr, seg);
    } else {
        k_prep_extended<<<cdiv(n, 128), 128, 0, st>>>((const uint64_t *)d_in, (ge_pniels_packed *)d_out, n);
    }
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------
// window selection: minimise windows * (n + ~2.5 * buckets) (bucket adds + reduction adds)
int msm_window_count_for_bits(int c) { return 256 / c + 1; }

int msm_choose_window_bits(const dalek_b200_ctx *ctx, size_t n)
{
    if (ctx->opt_window_bits >= 4 && ctx->opt_window_bits <= 20) return (int)ctx->opt_window_bits;
    int best = 4; double best_cost = 1e300;
    for (int c = 4; c <= 20; c++) {
        double W = (double)((253 + c - 1) / c);
        double cost = W * ((double)n + 4.0 * (double)(1u << (c - 1)));
        if (cost < best_cost) { best_cost = cost; best = c; }
    }
    return best;
}

// The same cost model when `n_short` scalars have only `short_bits` bits: they contribute ceil((bits+1)/c)
// bucket additions each (one spare bit for the signed-digit carry).
int msm_choose_window_bits_mixed(const dalek_b200_ctx *ctx, size_t n_short, int short_bits, size_t n_long)
{
    if (ctx->opt_window_bits >= 4 && ctx->opt_window_bits <= 20) return (int)ctx->opt_window_bits;
    int best = 4; double best_cost = 1e300;
    for (int c = 4; c <= 20; c++) {
        double W = (double)((253 + c - 1) / c), Ws = (double)((short_bits + 1 + c - 1) / c);
        double cost = Ws * (double)n_short + W * ((double)n_long + 4.0 * (double)(1u << (c - 1)));
        if (cost < best_cost) { best_cost = cost; best = c; }
    }
    return best;
}

// ------------------------------------------------------------------------------------------
// digits + histogram.  entry = (int32 digit << 32) | rank
// flat = 1: the digits of every window count into the buckets of window 0 (precomputed 2^(cw) P tables)
__global__ void k_digits(const uint4 *__restrict__ scalars, size_t n, int c, int nwin, uint32_t nbuckets,
                         uint32_t *__restrict__ counts, uint64_t *__restrict__ entries, int flat)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4 a = scalars[2 * i], b = scalars[2 * i + 1];
    uint32_t s[9] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, 0};
    const uint32_t mask = (1u << c) - 1, half = 1u << (c - 1);
    uint32_t carry = 0;
    for (int w = 0; w < nwin; w++) {
        int o = w * c;
        uint32_t raw = 0;
        if (o < 256) {
            int wi = o >> 5, bi = o & 31;
            uint64_t two = (uint64_t)s[wi] | ((uint64_t)s[wi + 1] << 32);
            raw = (uint32_t)(two >> bi) & mask;
            if (o + c > 256) raw &= (1u << (256 - o)) - 1;
        }
        uint32_t v = raw + carry;
        int32_t d;
        if (v > half) { d = (int32_t)v - (int32_t)(1u << c); carry = 1; } else { d = (int32_t)v; carry = 0; }
        uint32_t rank = 0;
        if (d != 0) {
            uint32_t bkt = (uint32_t)(d < 0 ? -d : d) - 1;
            rank = atomicAdd(&counts[(flat ? (size_t)0 : (size_t)w * nbuckets) + bkt], 1u);
        }
        entries[(size_t)w * n + i] = ((uint64_t)(uint32_t)d << 32) | rank;
    }
}

// per-window exclusive scan of counts -> offsets (relative to the window's segment), multi-block:
// k_scan_partial (sum of each 4096-entry part), k_scan_bases (exclusive scan of the part sums of a
// window, one CTA per window), k_scan_apply (local scan + part base).
#define SCAN_PART 4096u
__global__ void __launch_bounds__(1024) k_scan_partial(const uint32_t *__restrict__ in, uint32_t nbuckets, uint32_t parts,
                                                       uint32_t *__restrict__ part_sums)
{
    __shared__ uint32_t sh[32];
    uint32_t w = blockIdx.x / parts, part = blockIdx.x % parts;
    const uint32_t *src = in + (size_t)w * nbuckets;
    uint32_t base = part * SCAN_PART + threadIdx.x * 4, sum = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) if (base + k < nbuckets) sum += src[base + k];
    for (int d = 16; d > 0; d >>= 1) sum += __shfl_down_sync(0xffffffffu, sum, d);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t v = sh[threadIdx.x];
        for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
        if (threadIdx.x == 0) part_sums[blockIdx.x] = v;
    }
}
__global__ void k_scan_bases(uint32_t *__restrict__ part_sums, uint32_t parts)
{
    // one CTA (one thread is enough: parts <= 128) per window: in-place exclusive scan
    if (threadIdx.x) return;
    uint32_t *p = part_sums + (size_t)blockIdx.x * parts, run = 0;
    for (uint32_t k = 0; k < parts; k++) { uint32_t v = p[k]; p[k] = run; run += v; }
}
__global__ void __launch_bounds__(1024) k_scan_apply(const uint32_t *__restrict__ in, const uint32_t *__restrict__ part_base,
                                                     uint32_t nbuckets, uint32_t parts, uint32_t *__restrict__ out)
{
    __shared__ uint32_t sh[32];
    uint32_t w = blockIdx.x / parts, part = blockIdx.x % parts;
    const uint32_t *src = in + (size_t)w * nbuckets;
    uint32_t *dst = out + (size_t)w * nbuckets;
    uint32_t base = part * SCAN_PART + threadIdx.x * 4;
    uint32_t v[4], sum = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) { v[k] = base + k < nbuckets ? src[base + k] : 0; sum += v[k]; }
    uint32_t incl = sum;                                   // inclusive scan of thread sums inside the warp
    for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, d); if ((threadIdx.x & 31) >= d) incl += t; }
    if ((threadIdx.x & 31) == 31) sh[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t x = sh[threadIdx.x], inc2 = x;
        for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc2, d); if (threadIdx.x >= d) inc2 += t; }
        sh[threadIdx.x] = inc2 - x;                        // exclusive warp bases
    }
    __syncthreads();
    uint32_t run = part_base[blockIdx.x] + sh[threadIdx.x >> 5] + incl - sum;
#pragma unroll
    for (int k = 0; k < 4; k++) { if (base + k < nbuckets) dst[base + k] = run; run += v[k]; }
}

// Launched per group of windows [w0, w1) sized so that the group's slice of `sorted` stays in L2: the
// 4-byte scattered writes of one 32-byte sector then merge in L2 instead of each costing a DRAM
// read-modify-write.
// flat != 0: one bucket window; the stored index is w * flat + i, the position of 2^(cw) P_i in the point table
__global__ void k_scatter(const uint64_t *__restrict__ entries, const uint32_t *__restrict__ offsets, size_t n,
                          int w0, int w1, uint32_t nbuckets, uint32_t *__restrict__ sorted, size_t flat /* table stride, 0 = off */)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int w = w0; w < w1; w++) {
        uint64_t e = entries[(size_t)w * n + i];
        int32_t d = (int32_t)(e >> 32);
        if (d == 0) continue;
        uint32_t neg = d < 0, bkt = (uint32_t)(neg ? -d : d) - 1;
        if (flat) {
            uint32_t pos = offsets[bkt] + (uint32_t)e;
            sorted[pos] = (uint32_t)((size_t)w * flat + i) | (neg << 31);
        } else {
            uint32_t pos = offsets[(size_t)w * nbuckets + bkt] + (uint32_t)e;
            sorted[(size_t)w * n + pos] = (uint32_t)i | (neg << 31);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Bucket accumulation as a list of tasks.  A task is at most task_len consecutive entries of one
// bucket; a bucket with more entries (skewed inputs: the 128-bit z_i of verify_batch put n/256
// points into each of 256 buckets of one window; adversarial inputs can put everything into one)
// is cut into several tasks whose partial sums are added afterwards by k_heavy_fixup.
// task_len (msm_task_len) is twice the mean bucket size when the buckets alone give enough parallelism,
// so that only genuinely skewed buckets are cut; with few buckets it is what yields >= 2^18 tasks.
#define TASK_LEN_MIN 64u
static uint32_t msm_task_len(size_t n, int nwin, uint32_t nb)
{
    const size_t total_buckets = (size_t)nwin * nb;
    const size_t want = total_buckets >= ((size_t)1 << 18) ? 2 * (n / nb) : (n * (size_t)nwin) >> 18;
    uint32_t len = TASK_LEN_MIN;
    while (len < want && len < (1u << 22)) len <<= 1;
    return len;
}
#ifndef ACC_MIN_BLOCKS
#define ACC_MIN_BLOCKS 4
#endif

// also appends every bucket that needs more than one task to the heavy list (heavy[0] = count)
__global__ void k_task_count(const uint32_t *__restrict__ counts, uint32_t total_buckets, uint32_t task_len,
                             uint32_t *__restrict__ ntasks, uint32_t *__restrict__ heavy)
{
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total_buckets) return;
    uint32_t c = counts[t];
    uint32_t k = c <= task_len ? 1u : (c + task_len - 1) / task_len;
    ntasks[t] = k;
    if (k > 1) heavy[1 + atomicAdd(&heavy[0], 1u)] = t;
}

// per-window bases of the task lists (exclusive prefix over windows) and the grand total
__global__ void k_task_bases(const uint32_t *__restrict__ ntasks, const uint32_t *__restrict__ task_off, uint32_t nbuckets,
                             int nwin, uint32_t *__restrict__ win_base /* nwin + 1 */)
{
    if (blockIdx.x || threadIdx.x) return;
    uint32_t run = 0;
    for (int w = 0; w < nwin; w++) {
        win_base[w] = run;
        size_t last = (size_t)w * nbuckets + nbuckets - 1;
        run += task_off[last] + ntasks[last];
    }
    win_base[nwin] = run;
}

// task p = (bucket t, piece j) stored as two u32
__global__ void k_task_fill(const uint32_t *__restrict__ ntasks, const uint32_t *__restrict__ task_off,
                            const uint32_t *__restrict__ win_base, uint32_t nbuckets, uint32_t total_buckets,
                            uint2 *__restrict__ tasks)
{
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total_buckets) return;
    uint32_t w = t / nbuckets;
    uint32_t base = win_base[w] + task_off[t], k = ntasks[t];
    for (uint32_t j = 0; j < k; j++) tasks[base + j] = make_uint2(t, j);
}

// Tasks are processed in order of decreasing length (counting sort on the quantised length, TASK_BINS bins):
// the lanes of a warp then run the same trip count, and the grid drains longest-first, so the kernel does not
// end on a few long tasks.  order[q] = task index; hist | cursor | start are TASK_BINS words each.
#define TASK_BINS 256u
__device__ __forceinline__ uint32_t task_key(uint32_t len, uint32_t task_len)
{
    return (uint32_t)(((uint64_t)len * (TASK_BINS - 1) + task_len - 1) / task_len);     // 0 only for an empty task
}
__device__ __forceinline__ uint32_t task_length(const uint2 tk, const uint32_t *__restrict__ counts, uint32_t task_len)
{
    return min(task_len, counts[tk.x] - tk.y * task_len);
}

__global__ void __launch_bounds__(256)
k_task_hist(const uint2 *__restrict__ tasks, const uint32_t *__restrict__ counts, const uint32_t *__restrict__ total_ptr,
            uint32_t task_len, uint32_t *__restrict__ hist)
{
    __shared__ uint32_t sh[TASK_BINS];
    sh[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < *total_ptr) atomicAdd(&sh[task_key(task_length(tasks[p], counts, task_len), task_len)], 1u);
    __syncthreads();
    if (sh[threadIdx.x]) atomicAdd(&hist[threadIdx.x], sh[threadIdx.x]);
}

// start[k] = number of tasks with a larger key
__global__ void __launch_bounds__(256) k_task_scan(const uint32_t *__restrict__ hist, uint32_t *__restrict__ start)
{
    __shared__ uint32_t sh[TASK_BINS];
    const uint32_t k = TASK_BINS - 1 - threadIdx.x;              // thread 0 holds the largest key
    sh[threadIdx.x] = hist[k];
    __syncthreads();
    for (uint32_t d = 1; d < TASK_BINS; d <<= 1) {
        uint32_t v = threadIdx.x >= d ? sh[threadIdx.x - d] : 0;
        __syncthreads();
        sh[threadIdx.x] += v;
        __syncthreads();
    }
    start[k] = sh[threadIdx.x] - hist[k];
}

__global__ void __launch_bounds__(256)
k_task_scatter(const uint2 *__restrict__ tasks, const uint32_t *__restrict__ counts, const uint32_t *__restrict__ total_ptr,
               uint32_t task_len, const uint32_t *__restrict__ start, uint32_t *__restrict__ cursor, uint32_t *__restrict__ order)
{
    __shared__ uint32_t cnt[TASK_BINS], base[TASK_BINS];
    cnt[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = p < *total_ptr;
    uint32_t key = 0, rank = 0;
    if (live) { key = task_key(task_length(tasks[p], counts, task_len), task_len); rank = atomicAdd(&cnt[key], 1u); }
    __syncthreads();
    if (cnt[threadIdx.x]) base[threadIdx.x] = start[threadIdx.x] + atomicAdd(&cursor[threadIdx.x], cnt[threadIdx.x]);
    __syncthreads();
    if (live) order[base[key] + rank] = p;
}

__device__ __forceinline__ void load_p3(ge_p3 &p, const ge_p3_raw *src)
{
    const uint4 *s = reinterpret_cast<const uint4 *>(src);
    ge_p3_raw r;
#pragma unroll
    for (int q = 0; q < 10; q++) { uint4 v = s[q]; r.w[4 * q] = v.x; r.w[4 * q + 1] = v.y; r.w[4 * q + 2] = v.z; r.w[4 * q + 3] = v.w; }
    ge_p3_load_raw(p, r);
}

// TMA = 1: the gather of the next point is ONE bulk copy of the TMA unit (cp.async.bulk.shared.global, completion
// on a per-thread mbarrier) instead of 6-8 16-byte cp.async (LDGSTS); see profiles/ for the A/B measurement.
template <int KIND, int F64, int TMA>
__global__ void __launch_bounds__(128, ACC_MIN_BLOCKS)
k_bucket_accumulate(const void *__restrict__ points, const uint32_t *__restrict__ sorted,
                    const uint32_t *__restrict__ counts, const uint32_t *__restrict__ offsets,
                    const uint32_t *__restrict__ ntasks, const uint2 *__restrict__ tasks, const uint32_t *__restrict__ order,
                    const uint32_t *__restrict__ win_base, int w0, int w1, size_t n, uint32_t nbuckets, uint32_t task_len,
                    ge_p3_raw *__restrict__ buckets, ge_p3_raw *__restrict__ task_sums, int first)
{
    constexpr int NQ = KIND == PK_NIELS ? 6 : 8;              // 16-byte pieces per point
    constexpr int TSTRIDE = NQ * 16 + 16;                     // bulk copies land contiguously: pad the per-thread slot so
                                                              // that the 16-byte reads of 8 consecutive threads hit 8 different bank groups
    __shared__ uint4 s_pts[(F64 && !TMA) ? 2 : 1][(F64 && !TMA) ? 8 : 1][(F64 && !TMA) ? 128 : 1];   // cp.async slots, [buffer][piece][thread]: conflict-free
    __shared__ __align__(16) unsigned char s_bulk[(F64 && TMA) ? 2 : 1][(F64 && TMA) ? 128 : 1][(F64 && TMA) ? TSTRIDE : 16];
    __shared__ __align__(8) unsigned long long s_bar[(F64 && TMA) ? 2 : 1][(F64 && TMA) ? 128 : 1];
    const uint32_t total_tasks = win_base[w1];            // this launch covers the tasks of windows [w0, w1)
    const uint32_t slot = blockIdx.x * 128u + threadIdx.x;
    if (slot >= total_tasks) return;
    const uint32_t p = order[slot];                        // tasks in order of decreasing length
    const uint2 tk = tasks[p];
    const uint32_t t = tk.x, w = t / nbuckets;
    const uint32_t cnt = counts[t], start = tk.y * task_len;
    const uint32_t len = min(task_len, cnt - start);
    // `first` = first chunk of points: buckets start at the identity.  Later chunks (host inputs are
    // streamed in chunks so that the copies overlap the arithmetic) add onto the stored bucket sums;
    // the stored sum is folded in by piece 0 of the bucket (or by k_heavy_fixup for split buckets).
    const bool split = ntasks[t] != 1;
    if (!first && len == 0) return;                        // nothing new for this bucket
    const bool fold_old = !first && !split;
    const uint32_t *idx = sorted + (size_t)w * n + offsets[t] + start;
    ge_p3 acc;
    if (F64) {
        // FP64-pipe field (fe64.cuh): 1.65x the multiplication rate of the IMAD.WIDE form
        // The gather of the NEXT point (into this thread's shared-memory slot, two slots per thread) is in flight
        // while the current addition runs, so the HBM/L2 latency of the random gathers is off the dependent path.
        ge64_p3 acc64;
        if (fold_old) {
            ge_p3 old; load_p3(old, buckets + t);
            fe64_from_fe(acc64.X, old.X); fe64_from_fe(acc64.Y, old.Y); fe64_from_fe(acc64.Z, old.Z); fe64_from_fe(acc64.T, old.T);
        } else {
            ge64_identity(acc64);
        }
        uint32_t e_next = len ? idx[0] : 0;
        if (TMA) {
            const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(&s_bar[0][threadIdx.x]);
            const uint32_t bar1 = (uint32_t)__cvta_generic_to_shared(&s_bar[1][threadIdx.x]);
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar1) : "memory");
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        }
        auto prefetch = [&](uint32_t e, int buf) {
            const uint32_t pi = e & 0x7fffffffu;
            const char *src = reinterpret_cast<const char *>(points) + (size_t)pi * (NQ * 16);
            if (TMA) {
                const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_bar[buf][threadIdx.x]);
                const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&s_bulk[buf][threadIdx.x][0]);
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(NQ * 16) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(dst), "l"(src), "r"(NQ * 16), "r"(bar) : "memory");
            } else {
#pragma unroll
                for (int q = 0; q < NQ; q++) {
                    uint32_t dst = (uint32_t)__cvta_generic_to_shared(&s_pts[buf][q][threadIdx.x]);
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src + 16 * q) : "memory");
                }
            }
        };
        if (len) prefetch(e_next, 0);
        if (!TMA) asm volatile("cp.async.commit_group;" ::: "memory");
        for (uint32_t k = 0; k < len; k++) {
            const uint32_t e = e_next, neg = e >> 31;
            const int buf = k & 1;
            if (k + 1 < len) { e_next = idx[k + 1]; prefetch(e_next, buf ^ 1); }
            uint32_t words[NQ * 4];
            if (TMA) {
                const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_bar[buf][threadIdx.x]);
                const uint32_t parity = (k >> 1) & 1u;
                uint32_t done;
                do {
                    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
                } while (!done);
                const uint4 *sp = reinterpret_cast<const uint4 *>(&s_bulk[buf][threadIdx.x][0]);
#pragma unroll
                for (int q = 0; q < NQ; q++) { uint4 v = sp[q]; words[4 * q] = v.x; words[4 * q + 1] = v.y; words[4 * q + 2] = v.z; words[4 * q + 3] = v.w; }
            } else {
                asm volatile("cp.async.commit_group;" ::: "memory");
                asm volatile("cp.async.wait_group 1;" ::: "memory");
#pragma unroll
                for (int q = 0; q < NQ; q++) { uint4 v = s_pts[buf][q][threadIdx.x]; words[4 * q] = v.x; words[4 * q + 1] = v.y; words[4 * q + 2] = v.z; words[4 * q + 3] = v.w; }
            }
            if constexpr (KIND == PK_NIELS) {
                ge_niels_packed pk;
#pragma unroll
                for (int q = 0; q < 24; q++) pk.w[q] = words[q];
                ge64_niels nl; ge64_niels_unpack(nl, pk);
                ge64_madd(acc64, acc64, nl, neg);
            } else {
                ge_pniels_packed pk;
#pragma unroll
                for (int q = 0; q < 32; q++) pk.w[q] = words[q];
                ge64_pniels pn; ge64_pniels_unpack(pn, pk);
                ge64_padd(acc64, acc64, pn, neg);
            }
        }
        ge64_to_p3(acc, acc64);
    } else {
    if (fold_old) load_p3(acc, buckets + t); else ge_p3_identity(acc);
    for (uint32_t k = 0; k < len; k++) {
        uint32_t e = idx[k];
        uint32_t neg = e >> 31, pi = e & 0x7fffffffu;
        if (KIND == PK_NIELS) {
            const uint4 *src = reinterpret_cast<const uint4 *>(reinterpret_cast<const ge_niels_packed *>(points) + pi);
            ge_niels_packed pk;
#pragma unroll
            for (int q = 0; q < 6; q++) { uint4 v = __ldg(src + q); pk.w[4 * q] = v.x; pk.w[4 * q + 1] = v.y; pk.w[4 * q + 2] = v.z; pk.w[4 * q + 3] = v.w; }
            ge_niels nl; ge_niels_unpack(nl, pk);
            ge_madd(acc, acc, nl, neg);
        } else {
            const uint4 *src = reinterpret_cast<const uint4 *>(reinterpret_cast<const ge_pniels_packed *>(points) + pi);
            ge_pniels_packed pk;
#pragma unroll
            for (int q = 0; q < 8; q++) { uint4 v = __ldg(src + q); pk.w[4 * q] = v.x; pk.w[4 * q + 1] = v.y; pk.w[4 * q + 2] = v.z; pk.w[4 * q + 3] = v.w; }
            ge_pniels pn; ge_pniels_unpack(pn, pk);
            ge_padd(acc, acc, pn, neg);
        }
    }
    }
    ge_p3_raw r; ge_p3_store_raw(r, acc);
    uint4 *o = reinterpret_cast<uint4 *>(!split ? buckets + t : task_sums + p);
#pragma unroll
    for (int q = 0; q < 10; q++) o[q] = make_uint4(r.w[4 * q], r.w[4 * q + 1], r.w[4 * q + 2], r.w[4 * q + 3]);
}

// Everything below is latency-bound tree work on few points: it runs on groups of four lanes
// (warp4.cuh), one point operation per group at a time.

// One warp per heavy bucket (grid-stride over the heavy list): the 8 groups of the warp take
// strided task sums, then a 3-level shuffle tree across groups.
__global__ void __launch_bounds__(128)
k_heavy_fixup(const uint32_t *__restrict__ heavy, const uint32_t *__restrict__ ntasks, const uint32_t *__restrict__ task_off,
              const uint32_t *__restrict__ win_base, uint32_t nbuckets, uint32_t w0, uint32_t w1,
              const ge_p3_raw *__restrict__ task_sums, ge_p3_raw *__restrict__ buckets, int first)
{
    const uint32_t lane = threadIdx.x & 31, role = lane & 3, grp = lane >> 2;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t nheavy = heavy[0];
    for (uint32_t h = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; h < nheavy; h += nwarps) {
        uint32_t tb = heavy[1 + h];
        if (tb / nbuckets < w0 || tb / nbuckets >= w1) continue;      // another window group's bucket
        uint32_t kk = ntasks[tb];
        uint32_t base = win_base[tb / nbuckets] + task_off[tb];
        w4_point acc, x;
        if (first || grp != 0) w4_identity(acc); else w4_load(acc, buckets + tb);   // later chunks: keep the old sum
        for (uint32_t j0 = 0; j0 < kk; j0 += 8) {          // uniform trip count across the warp
            uint32_t j = j0 + grp;
            if (j < kk) w4_load(x, task_sums + base + j); else w4_identity(x);
            w4_add(acc, x, role);
        }
        for (int d = 16; d >= 4; d >>= 1) { w4_shfl_down(x, acc, d); w4_add(acc, x, role); }
        if (grp == 0) w4_store(buckets + tb, acc, role);
    }
}

__device__ __forceinline__ void load_p3_f64(ge64_p3 &o, const ge_p3_raw *src)
{
    ge_p3 q; load_p3(q, src);
    fe64_from_fe_limbs(o.X, q.X); fe64_from_fe_limbs(o.Y, q.Y); fe64_from_fe_limbs(o.Z, q.Z); fe64_from_fe_limbs(o.T, q.T);
}

// Level 1 of the bucket reduction (see k_chunk_reduce below) with ONE THREAD per chunk of m buckets on the
// FP64-pipe field: 2^(c-1) W / m chunks (32768 for 2^20 pairs) are enough threads for the throughput field, and
// a thread's 2(m-1) additions need no shuffles.  S_q = sum_r B_{qm+r},  W_q = sum_r (r+1) B_{qm+r}.
__global__ void __launch_bounds__(32)
k_chunk_reduce_f64(const ge_p3_raw *__restrict__ S_in, uint32_t n_in, uint32_t m, uint32_t n_out, uint32_t nwin,
                   ge_p3_raw *__restrict__ S_out, ge_p3_raw *__restrict__ W_out)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_out * nwin) return;
    const uint32_t w = t / n_out, q = t % n_out;
    const ge_p3_raw *S = S_in + (size_t)w * n_in + (size_t)q * m;
    fe64 d2; fe64_const_2d(d2);
    ge64_p3 run, acc, x;
    load_p3_f64(run, S + (m - 1));
    acc = run;
    ge_p3 nxt;                                              // the next bucket is loaded one iteration ahead
    if (m > 1) load_p3(nxt, S + (m - 2));
#pragma unroll 1
    for (uint32_t r = m - 1; r-- > 0;) {
        fe64_from_fe_limbs(x.X, nxt.X); fe64_from_fe_limbs(x.Y, nxt.Y); fe64_from_fe_limbs(x.Z, nxt.Z); fe64_from_fe_limbs(x.T, nxt.T);
        if (r > 0) load_p3(nxt, S + (r - 1));
        ge64_add_p3(run, run, x, d2);
        ge64_add_p3(acc, acc, run, d2);
    }
    ge_p3 o; ge_p3_raw raw;
    ge64_to_p3(o, run); ge_p3_store_raw(raw, o);
    uint4 *d = reinterpret_cast<uint4 *>(S_out + t);
#pragma unroll
    for (int k = 0; k < 10; k++) d[k] = make_uint4(raw.w[4 * k], raw.w[4 * k + 1], raw.w[4 * k + 2], raw.w[4 * k + 3]);
    ge64_to_p3(o, acc); ge_p3_store_raw(raw, o);
    d = reinterpret_cast<uint4 *>(W_out + t);
#pragma unroll
    for (int k = 0; k < 10; k++) d[k] = make_uint4(raw.w[4 * k], raw.w[4 * k + 1], raw.w[4 * k + 2], raw.w[4 * k + 3]);
}

// Bucket reduction  sum_b (b+1) B_b  per window (pippenger.rs:146-151), in log depth:
//   level 1   chunks of m buckets: S_q = sum_r B_{qm+r},  W_q = sum_r (r+1) B_{qm+r}   (running sums)
//   level l   chunks of m items of S^{l-1}: S^l_q, W^l_q = sum_r r S^{l-1}_{qm+r}      (0-based weights)
//   then      target = A_1 + m_1 (A_2 + m_2 (A_3 + ...)),  A_l = plain sum of the W^l array
// Doublings happen once per level in the final per-window Horner, not inside every level.
// One 4-lane group per chunk; n_in is a power of two and m divides it, so every chunk has m items.
__global__ void __launch_bounds__(128)
k_chunk_reduce(const ge_p3_raw *__restrict__ S_in, uint32_t n_in, uint32_t m, uint32_t one_based, uint32_t n_out,
               uint32_t nwin, ge_p3_raw *__restrict__ S_out, ge_p3_raw *__restrict__ W_out)
{
    const uint32_t role = threadIdx.x & 3;
    const uint32_t total = n_out * nwin;
    uint32_t t = (blockIdx.x * blockDim.x + threadIdx.x) >> 2;
    if (((blockIdx.x * blockDim.x + (threadIdx.x & ~31u)) >> 2) >= total) return;    // whole warp out of range
    const bool live = t < total;
    if (!live) t = total - 1;                                                       // keep the warp converged
    const uint32_t w = t / n_out, q = t % n_out;
    const ge_p3_raw *S = S_in + (size_t)w * n_in + (size_t)q * m;
    w4_point run, acc, x;
    w4_load(run, S + (m - 1));
    acc = run;
    for (uint32_t r = m - 1; r-- > 1;) {
        w4_load(x, S + r);
        w4_add(run, x, role);
        w4_add(acc, run, role);
    }
    if (m > 1) {
        w4_load(x, S);
        w4_add(run, x, role);
        if (one_based) w4_add(acc, run, role);
    } else if (!one_based) {
        w4_identity(acc);
    }
    if (live) { w4_store(S_out + t, run, role); w4_store(W_out + t, acc, role); }
}

// plain sum of one array per CTA (blockIdx.x = array id): 32 groups take strided items, then a
// shared-memory tree over the 32 partial sums
// Arrays are described by (offset, length) pairs in device memory (fixed per window width, cached in the
// context).  Two stages: pieces of at most SUM_PIECE items, then the per-array sum of the piece sums.
#define SUM_PIECE 256u
__global__ void __launch_bounds__(128)
k_plain_sum(const ge_p3_raw *__restrict__ pool, const uint2 *__restrict__ desc, ge_p3_raw *__restrict__ out)
{
    __shared__ ge_p3_raw sh[32];
    const uint32_t role = threadIdx.x & 3, grp = threadIdx.x >> 2;
    const uint2 d = desc[blockIdx.x];
    const ge_p3_raw *a = pool + d.x;
    const uint32_t len = d.y;
    w4_point acc, x;
    w4_identity(acc);
    for (uint32_t i0 = 0; i0 < len; i0 += 32) {
        uint32_t i = i0 + grp;
        if (i < len) w4_load(x, a + i); else w4_identity(x);
        w4_add(acc, x, role);
    }
    w4_store(&sh[grp], acc, role);
    __syncthreads();
    for (uint32_t d = 16; d > 0; d >>= 1) {
        if (threadIdx.x < 32 * ((d + 7) / 8)) {            // whole warps only
            uint32_t g2 = grp < d ? grp + d : grp;        // idle groups add their own value (discarded)
            w4_load(acc, &sh[grp]); w4_load(x, &sh[g2]);
            w4_add(acc, x, role);
        }
        __syncthreads();
        if (grp < d) w4_store(&sh[grp], acc, role);
        __syncthreads();
    }
    if (grp == 0) { w4_load(acc, &sh[0]); w4_store(out + blockIdx.x, acc, role); }
}

int msm_plain_sums(dalek_b200_ctx *ctx, cudaStream_t st, const ge_p3_raw *pool, const void *d_desc, uint32_t count, ge_p3_raw *out)
{
    if (!count) return 0;
    k_plain_sum<<<count, 128, 0, st>>>(pool, (const uint2 *)d_desc, out);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

// per window: target = A_1 + m_1 (A_2 + m_2 (...)); A sums are laid out [level][window]
struct LevelInfo { int nlevels; int log2m[16]; };
__global__ void __launch_bounds__(128)
k_finish_windows(const ge_p3_raw *__restrict__ S_top, const ge_p3_raw *__restrict__ A, LevelInfo li, uint32_t nwin,
                 ge_p3_raw *__restrict__ out)
{
    const uint32_t role = threadIdx.x & 3;
    uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 2;
    if (((blockIdx.x * blockDim.x + (threadIdx.x & ~31u)) >> 2) >= nwin) return;
    const bool live = w < nwin;
    if (!live) w = nwin - 1;
    w4_point t, x;
    if (li.nlevels > 0) {
        w4_load(t, A + (size_t)(li.nlevels - 1) * nwin + w);
        for (int l = li.nlevels - 2; l >= 0; l--) {
            for (int k = 0; k < li.log2m[l]; k++) w4_dbl(t, role, k == li.log2m[l] - 1);
            w4_load(x, A + (size_t)l * nwin + w);
            w4_add(t, x, role);
        }
    } else {
        w4_load(t, S_top + w);            // a single bucket of weight 1
    }
    if (live) w4_store(out + w, t, role);
}

// Final Horner over windows (pippenger.rs:159): total = total * 2^c + window, ~250 sequential
// doublings on one 4-lane group over the FP64 field (warp4_f64.cuh), then encode.
__global__ void __launch_bounds__(32)
k_combine(const ge_p3_raw *__restrict__ windows, int ranks, int nwin, int c, MsmResult *__restrict__ res)
{
    const uint32_t role = threadIdx.x & 3;
    w4f_point tot;
    w4f_horner(tot, windows, ranks, nwin, c, role);
    if (threadIdx.x != 0) return;
    ge_p3 total; w4f_to_p3(total, tot);
    uint32_t s[8];
    ge_compress(s, total);
#pragma unroll
    for (int i = 0; i < 8; i++) res->compressed[i] = s[i];
    fe_to_limbs51(res->limbs, total.X); fe_to_limbs51(res->limbs + 5, total.Y);
    fe_to_limbs51(res->limbs + 10, total.Z); fe_to_limbs51(res->limbs + 15, total.T);
    res->is_identity = ge_is_identity(total);
    res->pad = 0;
}

// ------------------------------------------------------------------------------------------
// One chunk of (scalar, point) pairs: digits, counting sort, task lists and bucket accumulation.
// `first` chunks start the buckets at the identity; later chunks add onto them.  All chunks of one
// MSM must use the same window width c.
// `active_windows` > 0 promises that every scalar of this chunk is below 2^(c * active_windows - 1): digits are
// extracted, sorted and accumulated for the low `active_windows` windows only (verify_batch: the 128-bit z_i).
// `flat` (a table stride): d_points holds nwin tables of `flat` points, table w = 2^(cw) P_i (precomp.cu); every digit then goes into ONE
// bucket window, so the reduction handles 2^(c-1) buckets instead of nwin times as many and no doubling is left
// (pair with msm_reduce_finish(..., flat = true)).
int msm_accumulate_chunk(dalek_b200_ctx *ctx, const uint32_t *d_scalars, const void *d_points, int point_kind, size_t n,
                         int c, bool first, int active_windows, size_t flat, cudaEvent_t points_ready)
{
    const int nwin_d = msm_window_count_for_bits(c);               // digit windows
    const int nact = active_windows > 0 && active_windows < nwin_d ? active_windows : nwin_d;
    const int nwin = flat ? 1 : nwin_d;                            // bucket windows
    const uint32_t nb = 1u << (c - 1);
    const size_t total_buckets = (size_t)nwin * nb;
    const uint32_t task_len = flat ? msm_task_len(n * (size_t)nact, 1, nb) : msm_task_len(n, nact, nb);
    const size_t max_tasks = total_buckets + (std::max<size_t>(1, n) * nact) / task_len + 1;
    const size_t max_heavy = (std::max<size_t>(1, n) * nact) / task_len + 1;
    const uint32_t parts = (nb + SCAN_PART - 1) / SCAN_PART;
    cudaStream_t st = ctx->stream;
    int rc;
    // counts | heavy list (count + entries): one memset clears both
    if ((rc = ws_reserve(ctx, ctx->counts, total_buckets * 4 + (1 + max_heavy) * 4))) return rc;
    if ((rc = ws_reserve(ctx, ctx->offsets, total_buckets * 4 + (size_t)nwin * parts * 4))) return rc;
    if ((rc = ws_reserve(ctx, ctx->ntasks, total_buckets * 4))) return rc;
    if ((rc = ws_reserve(ctx, ctx->task_off, total_buckets * 4 + (nwin + 1) * 4))) return rc;
    if ((rc = ws_reserve(ctx, ctx->tasks, max_tasks * 8))) return rc;
    if ((rc = ws_reserve(ctx, ctx->task_sums, max_tasks * sizeof(ge_p3_raw)))) return rc;
    if ((rc = ws_reserve(ctx, ctx->task_order, (3 * TASK_BINS + max_tasks) * 4))) return rc;   // hist | cursor | start | order
    if ((rc = ws_reserve(ctx, ctx->digits, std::max<size_t>(1, n) * nact * 8))) return rc;
    if ((rc = ws_reserve(ctx, ctx->sorted, std::max<size_t>(1, n) * nact * 4))) return rc;
    if ((rc = ws_reserve(ctx, ctx->buckets, total_buckets * sizeof(ge_p3_raw)))) return rc;
    uint32_t *counts = (uint32_t *)ctx->counts.p, *offsets = (uint32_t *)ctx->offsets.p;
    uint32_t *ntasks = (uint32_t *)ctx->ntasks.p, *task_off = (uint32_t *)ctx->task_off.p;
    uint32_t *win_base = task_off + total_buckets;
    uint32_t *heavy = counts + total_buckets;
    uint32_t *part_sums = offsets + total_buckets;
    uint2 *tasks = (uint2 *)ctx->tasks.p;
    uint32_t *t_hist = (uint32_t *)ctx->task_order.p, *t_cursor = t_hist + TASK_BINS, *t_start = t_cursor + TASK_BINS;
    uint32_t *order = t_start + TASK_BINS;
    ge_p3_raw *task_sums = (ge_p3_raw *)ctx->task_sums.p;
    uint64_t *entries = (uint64_t *)ctx->digits.p;
    uint32_t *sorted = (uint32_t *)ctx->sorted.p;
    ge_p3_raw *buckets = (ge_p3_raw *)ctx->buckets.p;

    CUDA_TRY(ctx, cudaMemsetAsync(counts, 0, (total_buckets + 1) * 4, st));
    CUDA_TRY(ctx, cudaMemsetAsync(t_hist, 0, 2 * TASK_BINS * 4, st));
    if (n) {
        k_digits<<<cdiv(n, 256), 256, 0, st>>>((const uint4 *)d_scalars, n, c, nact, nb, counts, entries, flat ? 1 : 0);
        ctx->launches++;
    }
    k_scan_partial<<<nwin * parts, 1024, 0, st>>>(counts, nb, parts, part_sums);
    k_scan_bases<<<nwin, 32, 0, st>>>(part_sums, parts);
    k_scan_apply<<<nwin * parts, 1024, 0, st>>>(counts, part_sums, nb, parts, offsets);
    k_task_count<<<cdiv(total_buckets, 256), 256, 0, st>>>(counts, (uint32_t)total_buckets, task_len, ntasks, heavy);
    k_scan_partial<<<nwin * parts, 1024, 0, st>>>(ntasks, nb, parts, part_sums);
    k_scan_bases<<<nwin, 32, 0, st>>>(part_sums, parts);
    k_scan_apply<<<nwin * parts, 1024, 0, st>>>(ntasks, part_sums, nb, parts, task_off);
    k_task_bases<<<1, 32, 0, st>>>(ntasks, task_off, nb, nwin, win_base);
    k_task_fill<<<cdiv(total_buckets, 256), 256, 0, st>>>(ntasks, task_off, win_base, nb, (uint32_t)total_buckets, tasks);
    k_task_hist<<<cdiv(max_tasks, 256), 256, 0, st>>>(tasks, counts, win_base + nwin, task_len, t_hist);
    k_task_scan<<<1, 256, 0, st>>>(t_hist, t_start);
    k_task_scatter<<<cdiv(max_tasks, 256), 256, 0, st>>>(tasks, counts, win_base + nwin, task_len, t_start, t_cursor, order);
    ctx->launches += 12;
    if (n) {
        const int wg = (int)std::max<size_t>(1, std::min<size_t>((size_t)nact, ((size_t)64 << 20) / (n * 4)));
        for (int w0 = 0; w0 < nact; w0 += wg) {
            k_scatter<<<cdiv(n, 256), 256, 0, st>>>(entries, offsets, n, w0, std::min(nact, w0 + wg), nb, sorted, flat);
            ctx->launches++;
        }
    }
    // the digit / sort passes above only read the scalars: the conversion of the points may still be running on another stream
    if (points_ready) CUDA_TRY(ctx, cudaStreamWaitEvent(st, points_ready, 0));
    if (first) CUDA_TRY(ctx, cudaEventRecord(ctx->ev_a, st));
    {
        const unsigned grid = cdiv(max_tasks, 128);
        const int f = first ? 1 : 0;
#define LAUNCH_ACC(KIND_, F64_, TMA_) k_bucket_accumulate<KIND_, F64_, TMA_><<<grid, 128, 0, st>>>(d_points, sorted, counts, offsets, ntasks, tasks, order, win_base, 0, nwin, n, nb, task_len, buckets, task_sums, f)
        const bool tma = ctx->opt_field_f64 && ctx->opt_acc_tma;
        if (point_kind == PK_NIELS) { if (tma) LAUNCH_ACC(PK_NIELS, 1, 1); else if (ctx->opt_field_f64) LAUNCH_ACC(PK_NIELS, 1, 0); else LAUNCH_ACC(PK_NIELS, 0, 0); }
        else { if (tma) LAUNCH_ACC(PK_PNIELS, 1, 1); else if (ctx->opt_field_f64) LAUNCH_ACC(PK_PNIELS, 1, 0); else LAUNCH_ACC(PK_PNIELS, 0, 0); }
#undef LAUNCH_ACC
        k_heavy_fixup<<<ctx->sm_count * 4, 128, 0, st>>>(heavy, ntasks, task_off, win_base, nb, 0u, (uint32_t)nwin, task_sums, buckets, f);
        ctx->launches += 2;
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_b, st));          // ev_a .. ev_b brackets the accumulation kernels
    ctx->last_kernel_launches = first ? 1 : ctx->last_kernel_launches + 1;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

// Bucket reduction of all windows, and (if d_result) the Horner over windows + encoding.
// flat: the buckets are the single window filled by msm_accumulate_chunk(..., flat = true): d_windows[0] is already
// the whole sum and d_result (if given) needs no doubling.
int msm_reduce_finish(dalek_b200_ctx *ctx, int c, ge_p3_raw *d_windows, MsmResult *d_result, bool flat)
{
    const int nwin = flat ? 1 : msm_window_count_for_bits(c);
    const int desc_key = c + (flat ? 64 : 0);
    const uint32_t nb = 1u << (c - 1);
    cudaStream_t st = ctx->stream;
    int rc;
    ge_p3_raw *buckets = (ge_p3_raw *)ctx->buckets.p;
    LevelInfo li; li.nlevels = 0;
    std::vector<uint32_t> lvl_m, lvl_nout;
    size_t pool_pts = 0;
    {
        uint32_t n_in = nb; bool first = true;
        while (n_in > 1) {
            uint32_t m = first ? std::min<uint32_t>(n_in, 16) : std::min<uint32_t>(n_in, 8);
            uint32_t n_out = (n_in + m - 1) / m;
            lvl_m.push_back(m); lvl_nout.push_back(n_out);
            int lg = 0; while ((1u << lg) < m) lg++;
            li.log2m[li.nlevels++] = lg;
            pool_pts += 2 * (size_t)n_out * nwin;
            n_in = n_out; first = false;
        }
    }
    if ((rc = ws_reserve(ctx, ctx->red_a, std::max<size_t>(1, pool_pts) * sizeof(ge_p3_raw)))) return rc;
    if ((rc = ws_reserve(ctx, ctx->red_b, (size_t)16 * nwin * sizeof(ge_p3_raw)))) return rc;
    ge_p3_raw *pool = (ge_p3_raw *)ctx->red_a.p, *A = (ge_p3_raw *)ctx->red_b.p;
    const ge_p3_raw *S_in = buckets;
    uint32_t n_in = nb;
    size_t pos = 0;
    std::vector<std::pair<size_t, uint32_t>> w_arrays;        // (offset of W array, n_out) per level
    for (int l = 0; l < li.nlevels; l++) {
        uint32_t m = lvl_m[l], n_out = lvl_nout[l];
        ge_p3_raw *S_out = pool + pos, *W_out = pool + pos + (size_t)n_out * nwin;
        if (l == 0 && ctx->opt_field_f64 && n_in % m == 0)
            k_chunk_reduce_f64<<<cdiv((size_t)n_out * nwin, 32), 32, 0, st>>>(S_in, n_in, m, n_out, nwin, S_out, W_out);   // small CTAs: 1024 warps spread evenly over the SMs
        else
            k_chunk_reduce<<<cdiv((size_t)n_out * nwin * 4, 128), 128, 0, st>>>(S_in, n_in, m, l == 0 ? 1u : 0u, n_out, nwin, S_out, W_out);
        ctx->launches++;
        w_arrays.push_back({pos + (size_t)n_out * nwin, n_out});
        S_in = S_out; n_in = n_out; pos += 2 * (size_t)n_out * nwin;
    }
    {   // plain sums of every (level, window) W array, two stages; descriptors depend only on c
        std::vector<uint2> d1, d2;
        for (int l = 0; l < li.nlevels; l++)
            for (int w = 0; w < nwin; w++) {
                uint32_t off = (uint32_t)(w_arrays[l].first + (size_t)w * w_arrays[l].second), len = w_arrays[l].second;
                uint32_t first_piece = (uint32_t)d1.size();
                for (uint32_t o = 0; o < len; o += SUM_PIECE) d1.push_back(make_uint2(off + o, std::min(SUM_PIECE, len - o)));
                d2.push_back(make_uint2(first_piece, (uint32_t)d1.size() - first_piece));
            }
        const size_t n1 = d1.size(), n2 = d2.size();
        if ((rc = ws_reserve(ctx, ctx->sum_desc, (n1 + n2) * sizeof(uint2)))) return rc;
        if ((rc = ws_reserve(ctx, ctx->sum_part, n1 * sizeof(ge_p3_raw)))) return rc;
        uint2 *dd1 = (uint2 *)ctx->sum_desc.p, *dd2 = dd1 + n1;
        if (ctx->sum_desc_c != desc_key) {
            CUDA_TRY(ctx, cudaMemcpyAsync(dd1, d1.data(), n1 * sizeof(uint2), cudaMemcpyHostToDevice, st));
            CUDA_TRY(ctx, cudaMemcpyAsync(dd2, d2.data(), n2 * sizeof(uint2), cudaMemcpyHostToDevice, st));
            CUDA_TRY(ctx, cudaStreamSynchronize(st));       // d1/d2 are host temporaries (rare: once per width)
            ctx->sum_desc_c = desc_key;
        }
        ge_p3_raw *parts = (ge_p3_raw *)ctx->sum_part.p;
        k_plain_sum<<<(unsigned)n1, 128, 0, st>>>(pool, dd1, parts);
        k_plain_sum<<<(unsigned)n2, 128, 0, st>>>(parts, dd2, A);
        ctx->launches += 2;
    }
    k_finish_windows<<<cdiv((size_t)nwin * 4, 128), 128, 0, st>>>(S_in, A, li, nwin, d_windows);
    ctx->launches++;
    if (d_result) {
        k_combine<<<1, 32, 0, st>>>(d_windows, 1, nwin, c, d_result);
        ctx->launches++;
    }
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

__global__ void k_fill_identity(ge_p3_raw *__restrict__ out, uint32_t count)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    ge_p3 id; ge_p3_identity(id);
    ge_p3_raw r; ge_p3_store_raw(r, id);
    out[i] = r;
}

int msm_fill_identity(dalek_b200_ctx *ctx, ge_p3_raw *d_out, uint32_t count)
{
    if (!count) return 0;
    k_fill_identity<<<cdiv(count, 128), 128, 0, ctx->stream>>>(d_out, count);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

int msm_window_sums(dalek_b200_ctx *ctx, const uint32_t *d_scalars, const void *d_points, int point_kind, size_t n,
                    int c, ge_p3_raw *d_windows)
{
    int rc;
    if ((rc = msm_accumulate_chunk(ctx, d_scalars, d_points, point_kind, n, c, true))) return rc;
    return msm_reduce_finish(ctx, c, d_windows, nullptr);
}

int msm_full(dalek_b200_ctx *ctx, const uint32_t *d_scalars, const void *d_points, int point_kind, size_t n, int c,
             ge_p3_raw *d_windows, MsmResult *d_result)
{
    int rc;
    if ((rc = msm_accumulate_chunk(ctx, d_scalars, d_points, point_kind, n, c, true))) return rc;
    return msm_reduce_finish(ctx, c, d_windows, d_result);
}

int msm_combine_windows(dalek_b200_ctx *ctx, const ge_p3_raw *d_windows, int ranks, int nwin, int c, MsmResult *d_result)
{
    k_combine<<<1, 32, 0, ctx->stream>>>(d_windows, ranks, nwin, c, d_result);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}
