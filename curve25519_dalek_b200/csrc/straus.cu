// straus.cu -- constant-time multiscalar multiplication (the MultiscalarMul contract,
// curve25519-dalek/src/traits.rs:78-134) and the Ristretto forwarders.
//
// Reference algorithm: Straus with radix-16 signed digits and a constant-time 8-entry table scan
// per point (src/backend/serial/scalar_mul/straus.rs:103-144, src/window.rs:54-76, :97-105,
// src/scalar.rs:1019-1051).  On the GPU:
//   * k_ct_scalar_mul    one thread per (scalar, point): its own [P..8P] table in local memory,
//                        64 x (4 doublings + masked table scan + add); control flow and addresses are
//                        independent of the scalar.  The n products are then summed by a tree.
//   * k_double_base      one thread per (a_i, b_i): Straus over the two shared bases G, H whose
//                        tables sit in shared memory (uniform-address broadcast reads), output
//                        Ristretto-compressed (src/ristretto.rs:500-533, :964-977).
#include <algorithm>
#include <cstring>

#include "../../include/dalek_b200.h"
#include "engine.h"
#include "ge64.cuh"

static inline unsigned cdiv(size_t a, unsigned b) { return (unsigned)((a + b - 1) / b); }
void launch_niels_to_pniels(dalek_b200_ctx *ctx, const void *in, void *out, size_t n);

// Scalar::as_radix_16 (scalar.rs:1019-1051): 64 digits in [-8, 8), top digit in [-8, 8]; packed one per
// byte.  Requires the scalar < 2^255 (Scalar invariant #1).
__device__ __forceinline__ void radix16_digits(int8_t d[64], const uint32_t s[8])
{
#pragma unroll
    for (int i = 0; i < 64; i++) d[i] = (int8_t)((s[i >> 3] >> (4 * (i & 7))) & 15);
    int8_t carry = 0;
#pragma unroll
    for (int i = 0; i < 63; i++) {
        d[i] = (int8_t)(d[i] + carry);
        carry = (int8_t)((d[i] + 8) >> 4);
        d[i] = (int8_t)(d[i] - (carry << 4));
    }
    d[63] = (int8_t)(d[63] + carry);
}

// LookupTable::select (window.rs:54-76) over 8 projective Niels entries stored as raw limbs
// (40 words each): masked OR over all entries, then conditional negation.
__device__ __forceinline__ void ct_select_pniels(ge_pniels &r, const uint32_t *table /* 8 x 40 words */, int digit)
{
    int32_t xmask = digit >> 31;
    uint32_t xabs = (uint32_t)((digit + xmask) ^ xmask);
    uint32_t w[40];
#pragma unroll
    for (int k = 0; k < 40; k++) w[k] = 0;
#pragma unroll 1
    for (uint32_t j = 1; j <= 8; j++) {
        uint32_t m = 0u - (uint32_t)(xabs == j);
#pragma unroll
        for (int k = 0; k < 40; k++) w[k] |= table[(j - 1) * 40 + k] & m;
    }
    // digit 0 selects the identity (1, 1, 1, 0)
    uint32_t z = (uint32_t)(xabs == 0);
    w[0] |= z; w[10] |= z; w[20] |= z;
#pragma unroll
    for (int k = 0; k < 10; k++) { r.YpX.v[k] = w[k]; r.YmX.v[k] = w[10 + k]; r.Z.v[k] = w[20 + k]; r.T2d.v[k] = w[30 + k]; }
}

__device__ __forceinline__ void store_pniels_raw(uint32_t *dst, const ge_pniels &n)
{
#pragma unroll
    for (int k = 0; k < 10; k++) { dst[k] = n.YpX.v[k]; dst[10 + k] = n.YmX.v[k]; dst[20 + k] = n.Z.v[k]; dst[30 + k] = n.T2d.v[k]; }
}

// LookupTable::from (window.rs:97-105): [P, 2P, ..., 8P] as projective Niels
__device__ __forceinline__ void build_table(uint32_t *table, const ge_p3 &P)
{
    ge_pniels n; ge_p3_to_pniels(n, P);
    store_pniels_raw(table, n);
    ge_p3 acc = P;
#pragma unroll 1
    for (int j = 1; j < 8; j++) {
        ge_pniels prev;
#pragma unroll
        for (int k = 0; k < 10; k++) { prev.YpX.v[k] = table[(j - 1) * 40 + k]; prev.YmX.v[k] = table[(j - 1) * 40 + 10 + k];
                                        prev.Z.v[k] = table[(j - 1) * 40 + 20 + k]; prev.T2d.v[k] = table[(j - 1) * 40 + 30 + k]; }
        ge_padd(acc, P, prev, 0);                    // (j+1) P = P + j P
        ge_p3_to_pniels(n, acc);
        store_pniels_raw(table + j * 40, n);
    }
}

// one thread: Q = s * P, constant-time (variable_base.rs:11-48 structure)
__global__ void __launch_bounds__(64)
k_ct_scalar_mul(const uint32_t *__restrict__ scalars, const ge_pniels_packed *__restrict__ points, size_t n,
                ge_p3_raw *__restrict__ out)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t s[8];
#pragma unroll
    for (int k = 0; k < 8; k++) s[k] = scalars[8 * i + k];
    // recover the extended point from its projective Niels form: X = (YpX - YmX)/2 ... avoid halving by
    // working with 2P' = (YpX - YmX, YpX + YmX, 2Z, .) which is the same projective point.
    ge_pniels_packed pk = points[i];
    ge_pniels pn; ge_pniels_unpack(pn, pk);
    ge_p3 P;
    {
        fe twoX, twoY, twoZ;
        fe_sub(twoX, pn.YpX, pn.YmX); fe_carry(twoX, twoX);
        fe_add(twoY, pn.YpX, pn.YmX); fe_carry(twoY, twoY);
        fe_add(twoZ, pn.Z, pn.Z); fe_carry(twoZ, twoZ);
        // extended coordinates of the same point with Z' = 2Z * 2Z ... : (X'Z', Y'Z', Z'^2, X'Y')
        fe_mul(P.X, twoX, twoZ); fe_mul(P.Y, twoY, twoZ); fe_sq(P.Z, twoZ); fe_mul(P.T, twoX, twoY);
    }
    uint32_t table[8 * 40];
    build_table(table, P);
    int8_t d[64];
    radix16_digits(d, s);
    ge_p3 Q; ge_p3_identity(Q);
#pragma unroll 1
    for (int j = 63; j >= 0; j--) {
        if (j != 63) ge_mul_by_pow_2(Q, Q, 4);
        ge_pniels sel; ct_select_pniels(sel, table, d[j]);
        uint32_t neg = (uint32_t)(d[j] < 0);
        ge_padd(Q, Q, sel, neg);
    }
    ge_p3_raw r; ge_p3_store_raw(r, Q);
    out[i] = r;
}

// plain tree sum: out[q] = sum of in[8q .. 8q+8)
__global__ void __launch_bounds__(64)
k_sum_level(const ge_p3_raw *__restrict__ in, size_t n_in, ge_p3_raw *__restrict__ out, size_t n_out)
{
    size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_out) return;
    size_t lo = q * 8, hi = min(lo + 8, n_in);
    ge_p3 acc, x;
    ge_p3_raw r = in[lo]; ge_p3_load_raw(acc, r);
    for (size_t k = lo + 1; k < hi; k++) { r = in[k]; ge_p3_load_raw(x, r); ge_add(acc, acc, x); }
    ge_p3_store_raw(r, acc);
    out[q] = r;
}

__global__ void k_store_identity(ge_p3_raw *out)
{
    ge_p3 p; ge_p3_identity(p); ge_p3_raw r; ge_p3_store_raw(r, p); out[0] = r;
}

int straus_ct_msm(dalek_b200_ctx *ctx, const uint32_t *d_scalars, const void *d_points_pniels, size_t n, MsmResult *d_result)
{
    int rc;
    cudaStream_t st = ctx->stream;
    if ((rc = ws_reserve(ctx, ctx->buckets, std::max<size_t>(1, n) * sizeof(ge_p3_raw)))) return rc;
    if ((rc = ws_reserve(ctx, ctx->red_a, std::max<size_t>(1, (n + 7) / 8) * sizeof(ge_p3_raw)))) return rc;
    ge_p3_raw *a = (ge_p3_raw *)ctx->buckets.p, *b = (ge_p3_raw *)ctx->red_a.p;
    if (n == 0) {
        k_store_identity<<<1, 1, 0, st>>>(a);
        ctx->launches++;
    } else {
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_a, st));
        k_ct_scalar_mul<<<cdiv(n, 64), 64, 0, st>>>(d_scalars, (const ge_pniels_packed *)d_points_pniels, n, a);
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_b, st));
        ctx->launches++;
        ctx->last_kernel_launches = 1;
        size_t cur = n;
        while (cur > 1) {
            size_t nxt = (cur + 7) / 8;
            k_sum_level<<<cdiv(nxt, 64), 64, 0, st>>>(a, cur, b, nxt);
            ctx->launches++;
            std::swap(a, b);
            cur = nxt;
        }
    }
    return msm_combine_windows(ctx, a, 1, 1, 4, d_result);
}

// ------------------------------------------------------------------------------------------
// Ristretto double-base batch
__global__ void k_double_base_tables(const uint32_t *__restrict__ GH /* 16 words: G | H compressed */,
                                     uint32_t *__restrict__ tables /* 2 x 8 x 40 words */, int *__restrict__ status)
{
    int t = threadIdx.x;
    if (t >= 2) return;
    uint32_t enc[8];
#pragma unroll
    for (int k = 0; k < 8; k++) enc[k] = GH[8 * t + k];
    ge_p3 P;
    if (!ristretto_decompress(P, enc)) { atomicOr(status, 1); ge_p3_identity(P); }
    uint32_t tab[8 * 40];
    build_table(tab, P);
    for (int k = 0; k < 8 * 40; k++) tables[t * 320 + k] = tab[k];
}

__global__ void __launch_bounds__(128)
k_double_base(const uint32_t *__restrict__ a, const uint32_t *__restrict__ b, const uint32_t *__restrict__ tables, size_t n,
              uint32_t *__restrict__ out)
{
    __shared__ uint32_t sh[2 * 8 * 40];
    for (int k = threadIdx.x; k < 640; k += blockDim.x) sh[k] = tables[k];
    __syncthreads();
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t sa[8], sb[8];
#pragma unroll
    for (int k = 0; k < 8; k++) { sa[k] = a[8 * i + k]; sb[k] = b[8 * i + k]; }
    int8_t da[64], db[64];
    radix16_digits(da, sa);
    radix16_digits(db, sb);
    ge_p3 Q; ge_p3_identity(Q);
#pragma unroll 1
    for (int j = 63; j >= 0; j--) {                          // straus.rs:129-138
        if (j != 63) ge_mul_by_pow_2(Q, Q, 4);
        ge_pniels sel;
        ct_select_pniels(sel, sh, da[j]);
        ge_padd(Q, Q, sel, (uint32_t)(da[j] < 0));
        ct_select_pniels(sel, sh + 320, db[j]);
        ge_padd(Q, Q, sel, (uint32_t)(db[j] < 0));
    }
    uint32_t enc[8];
    ristretto_compress<1>(enc, Q);
#pragma unroll
    for (int k = 0; k < 8; k++) out[8 * i + k] = enc[k];
}

// ---- fixed-base comb for the double-base batch ------------------------------------------------
// With G and H shared by the whole batch, a*G + b*H = sum_i a_i (16^i G) + b_i (16^i H) over the radix-16
// signed digits (scalar.rs:1019-1051): 128 mixed additions per pair and NO doublings, against 256
// doublings + 128 additions for Straus.  The contract of MultiscalarMul is kept: the 2 x 64 x 8 table
// entries (j+1) 16^i {G,H} sit in shared memory as balanced FP64 limbs (15 doubles each, 120 KiB), every
// lookup scans all 8 entries of a row at warp-uniform addresses with arithmetic masks (window.rs:54-76),
// and the digit's sign is applied by masked swap / negate inside the addition.
#define COMB_ROWS 128          // 2 bases x 64 digit positions
#define COMB_ENTRY 15          // doubles per affine Niels entry

__global__ void __launch_bounds__(128)
k_comb_tables(const uint32_t *__restrict__ GH, double *__restrict__ table, int *__restrict__ status)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= COMB_ROWS * 8) return;
    int b = t >> 9, i = (t >> 3) & 63, j = t & 7;
    uint32_t enc[8];
#pragma unroll
    for (int k = 0; k < 8; k++) enc[k] = GH[8 * b + k];
    ge_p3 base, P;
    if (!ristretto_decompress(base, enc)) { atomicOr(status, 1); ge_p3_identity(base); }
    ge_pniels nb; ge_p3_to_pniels(nb, base);
    P = base;
    for (int k = 0; k < j; k++) ge_padd(P, P, nb, 0);            // (j+1) * base
    if (i) ge_mul_by_pow_2(P, P, 4 * i);                         // * 16^i
    fe zi, x, y;
    fe_invert(zi, P.Z);
    fe_mul(x, P.X, zi); fe_mul(y, P.Y, zi);
    ge_niels n; ge_affine_to_niels(n, x, y);
    fe64 e[3];
    fe64_from_fe(e[0], n.ypx); fe64_from_fe(e[1], n.ymx); fe64_from_fe(e[2], n.xy2d);
    double *dst = table + (size_t)t * COMB_ENTRY;
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
        for (int k = 0; k < 5; k++) dst[5 * c + k] = e[c].v[k];
}

// constant-time: select |digit| * 16^i * base from the 8 entries of one table row (digit 0 -> identity)
__device__ __forceinline__ void comb_select(ge64_niels &q, const double *__restrict__ row, uint32_t xabs)
{
    long long w[COMB_ENTRY];
#pragma unroll
    for (int k = 0; k < COMB_ENTRY; k++) w[k] = 0;
#pragma unroll 1
    for (uint32_t j = 1; j <= 8; j++) {
        const long long m = 0LL - (long long)(xabs == j);
#pragma unroll
        for (int k = 0; k < COMB_ENTRY; k++) w[k] |= __double_as_longlong(row[(j - 1) * COMB_ENTRY + k]) & m;
    }
    const long long one = 0x3ff0000000000000LL & (0LL - (long long)(xabs == 0));      // 1.0 for the identity (1, 1, 0)
    w[0] |= one; w[5] |= one;
#pragma unroll
    for (int k = 0; k < 5; k++) {
        q.ypx.v[k] = __longlong_as_double(w[k]); q.ymx.v[k] = __longlong_as_double(w[5 + k]); q.xy2d.v[k] = __longlong_as_double(w[10 + k]);
    }
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
k_double_base_comb(const uint32_t *__restrict__ a, const uint32_t *__restrict__ b, const double *__restrict__ table, size_t n,
                   uint32_t *__restrict__ out)
{
    extern __shared__ double s_tab[];                             // COMB_ROWS * 8 * COMB_ENTRY doubles
    for (int k = threadIdx.x; k < COMB_ROWS * 8 * COMB_ENTRY; k += blockDim.x) s_tab[k] = table[k];
    __syncthreads();
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ge64_p3 acc; ge64_identity(acc);
    int ca = 0, cb = 0;                                           // radix-16 recoding carries (scalar.rs:1040-1046)
    uint32_t wa = 0, wb = 0;
#pragma unroll 1
    for (int pos = 0; pos < 64; pos++) {
        if ((pos & 7) == 0) { wa = a[8 * i + (pos >> 3)]; wb = b[8 * i + (pos >> 3)]; }   // one scalar word per 8 digits
        int da = (int)(wa & 15) + ca; wa >>= 4;
        int db = (int)(wb & 15) + cb; wb >>= 4;
        if (pos < 63) { ca = (da + 8) >> 4; da -= ca << 4; cb = (db + 8) >> 4; db -= cb << 4; }
        ge64_niels q;
        int m = da >> 31;
        comb_select(q, s_tab + (size_t)pos * 8 * COMB_ENTRY, (uint32_t)((da + m) ^ m));
        ge64_madd(acc, acc, q, (uint32_t)(da < 0));
        m = db >> 31;
        comb_select(q, s_tab + (size_t)(64 + pos) * 8 * COMB_ENTRY, (uint32_t)((db + m) ^ m));
        ge64_madd(acc, acc, q, (uint32_t)(db < 0));
    }
    ge_p3 Q; ge64_to_p3(Q, acc);
    uint32_t enc[8];
    ristretto_compress<1>(enc, Q);                                 // inverse square root on the FP64 field too
#pragma unroll
    for (int k = 0; k < 8; k++) out[8 * i + k] = enc[k];
}

// Table build for one (G, H) pair on ctx->stream; returns the device table and which kernel reads it.
struct DoubleBasePlan { const void *table; int *d_status; int variant; size_t smem; };

static int double_base_setup(dalek_b200_ctx *ctx, const uint8_t G[32], const uint8_t H[32], size_t n, DoubleBasePlan &plan)
{
    int rc;
    cudaStream_t st = ctx->stream;
    const size_t comb_bytes = (size_t)COMB_ROWS * 8 * COMB_ENTRY * sizeof(double);
    const size_t head = 64 + 2 * 8 * 40 * 4 + 64;
    if ((rc = ws_reserve(ctx, ctx->misc0, head + comb_bytes))) return rc;
    uint32_t *d_gh = (uint32_t *)ctx->misc0.p;
    uint32_t *d_tables = d_gh + 16;
    plan.d_status = (int *)(d_tables + 640);
    double *d_comb = (double *)((char *)ctx->misc0.p + head);
    if ((rc = pinned_reserve(ctx, 256))) return rc;
    memcpy(ctx->h_pinned, G, 32); memcpy((char *)ctx->h_pinned + 32, H, 32);
    CUDA_TRY(ctx, cudaMemcpyAsync(d_gh, ctx->h_pinned, 64, cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemsetAsync(plan.d_status, 0, 4, st));
    const bool comb = ctx->opt_double_base_comb && n >= 4096;     // the table build only pays off for a real batch
    if (comb) {
        if (!ctx->comb_attr_set) {                               // per context: the attribute is per device
            CUDA_TRY(ctx, cudaFuncSetAttribute(k_double_base_comb<384>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)comb_bytes));
            ctx->comb_attr_set = true;
        }
        k_comb_tables<<<8, 128, 0, st>>>(d_gh, d_comb, plan.d_status);
        plan.table = d_comb; plan.variant = 1; plan.smem = comb_bytes;
    } else {
        k_double_base_tables<<<1, 32, 0, st>>>(d_gh, d_tables, plan.d_status);
        plan.table = d_tables; plan.variant = 0; plan.smem = 0;
    }
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

static int double_base_launch(dalek_b200_ctx *ctx, const DoubleBasePlan &plan, const uint8_t *d_a, const uint8_t *d_b, size_t n,
                              uint8_t *d_out, cudaStream_t st)
{
    if (!n) return 0;
    const uint32_t *a = (const uint32_t *)d_a, *b = (const uint32_t *)d_b;
    // 384 threads x 168 registers fill the register file with the 120 KiB table resident (512 x 128 spills; measured slower)
    if (plan.variant == 1) k_double_base_comb<384><<<cdiv(n, 384), 384, plan.smem, st>>>(a, b, (const double *)plan.table, n, (uint32_t *)d_out);
    else k_double_base<<<cdiv(n, 128), 128, 0, st>>>(a, b, (const uint32_t *)plan.table, n, (uint32_t *)d_out);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

static int double_base_status(dalek_b200_ctx *ctx, const DoubleBasePlan &plan, int *h_status)
{
    cudaStream_t st = ctx->stream;
    int *hs = (int *)((char *)ctx->h_pinned + 128);
    CUDA_TRY(ctx, cudaMemcpyAsync(hs, plan.d_status, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    float ms = 0.f;
    if ((ms = elapsed_ms(ctx->ev_a, ctx->ev_b)) >= 0.f) ctx->last_kernel_ms = ms;
    ctx->last_kernel_launches = 1;
    *h_status = *hs;
    return 0;
}

// device-resident scalars in, device-resident encodings out
int ristretto_double_base(dalek_b200_ctx *ctx, const uint8_t *d_a, const uint8_t *d_b, const uint8_t G[32], const uint8_t H[32],
                          size_t n, uint8_t *d_out, int *h_status)
{
    int rc;
    DoubleBasePlan plan;
    if ((rc = double_base_setup(ctx, G, H, n, plan))) return rc;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_a, ctx->stream));
    if ((rc = double_base_launch(ctx, plan, d_a, d_b, n, d_out, ctx->stream))) return rc;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_b, ctx->stream));
    return double_base_status(ctx, plan, h_status);
}

// ------------------------------------------------------------------------------------------
// Ristretto vartime MSM: decode with the Ristretto rules, then the Edwards bucket MSM; encode the
// result with RistrettoPoint::compress (ristretto.rs:980-994).
// SEG = 1: a point that does not decode marks its segment (batched MSM) instead of the call-wide flag
template <int F64, int SEG>
__global__ void k_prep_ristretto(const uint32_t *__restrict__ in, ge_pniels_packed *__restrict__ out, size_t n, int *__restrict__ bad,
                                 SegStatus seg)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t enc[8];
#pragma unroll
    for (int k = 0; k < 8; k++) enc[k] = in[8 * i + k];
    ge_p3 P;
    if (!ristretto_decompress<F64>(P, enc)) {
        if (SEG) seg_mark_bad(seg, i); else atomicOr(bad, 1);
        ge_p3_identity(P);
    }
    ge_pniels pn; ge_p3_to_pniels(pn, P);
    ge_pniels_packed pk; ge_pniels_pack(pk, pn);
    out[i] = pk;
}

__global__ void k_ristretto_encode_result(const MsmResult *__restrict__ res, uint32_t *__restrict__ out)
{
    ge_p3 p;
    fe_from_limbs51(p.X, res->limbs); fe_from_limbs51(p.Y, res->limbs + 5);
    fe_from_limbs51(p.Z, res->limbs + 10); fe_from_limbs51(p.T, res->limbs + 15);
    uint32_t enc[8];
    ristretto_compress(enc, p);
    for (int k = 0; k < 8; k++) out[k] = enc[k];
}

// CompressedRistretto (device, n x 32 B) -> packed projective Niels; *d_bad set if one does not decode
int ristretto_prepare_points(dalek_b200_ctx *ctx, const void *d_in, size_t n, void *d_out, int *d_bad)
{
    if (!n) return 0;
    if (ctx->opt_decompress_f64) k_prep_ristretto<1, 0><<<cdiv(n, 128), 128, 0, ctx->stream>>>((const uint32_t *)d_in, (ge_pniels_packed *)d_out, n, d_bad, SegStatus{});
    else k_prep_ristretto<0, 0><<<cdiv(n, 128), 128, 0, ctx->stream>>>((const uint32_t *)d_in, (ge_pniels_packed *)d_out, n, d_bad, SegStatus{});
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

int ristretto_prepare_points_seg(dalek_b200_ctx *ctx, cudaStream_t st, const void *d_in, size_t n, void *d_out, const SegStatus &seg)
{
    if (!n) return 0;
    if (ctx->opt_decompress_f64) k_prep_ristretto<1, 1><<<cdiv(n, 128), 128, 0, st>>>((const uint32_t *)d_in, (ge_pniels_packed *)d_out, n, nullptr, seg);
    else k_prep_ristretto<0, 1><<<cdiv(n, 128), 128, 0, st>>>((const uint32_t *)d_in, (ge_pniels_packed *)d_out, n, nullptr, seg);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

// RistrettoPoint::compress of an MSM result (device): 8 words at d_enc
int ristretto_encode_result(dalek_b200_ctx *ctx, const MsmResult *d_res, uint32_t *d_enc)
{
    k_ristretto_encode_result<<<1, 1, 0, ctx->stream>>>(d_res, d_enc);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

extern "C" {

int dalek_b200_edwards_ct_msm(dalek_b200_ctx *ctx, const uint8_t *scalars, const void *points, int point_fmt, size_t n,
                              uint8_t out_compressed[32], uint64_t out_limbs[20])
{
    if (!ctx || (n && (!scalars || !points)) || (point_fmt != DALEK_POINTS_COMPRESSED && point_fmt != DALEK_POINTS_EXTENDED))
        return DALEK_E_INVALID_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    int rc;
    cudaStream_t st = ctx->stream;
    for (size_t i = 0; i < n; i++)
        if (scalars[32 * i + 31] & 0x80) { ctx->last_error = "scalar with bit 255 set (Scalar invariant #1)"; return DALEK_E_INVALID_ARG; }
    size_t pin = point_fmt == DALEK_POINTS_COMPRESSED ? 32 : 160;
    if ((rc = ws_reserve(ctx, ctx->scalars, std::max<size_t>(1, n) * 32))) return rc;
    if ((rc = ws_reserve(ctx, ctx->points_in, std::max<size_t>(1, n) * pin))) return rc;
    if ((rc = ws_reserve(ctx, ctx->points, std::max<size_t>(1, n) * sizeof(ge_pniels_packed)))) return rc;
    if ((rc = ws_reserve(ctx, ctx->flags, 64))) return rc;
    if ((rc = ws_reserve(ctx, ctx->result, sizeof(MsmResult)))) return rc;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->flags.p, 0, 64, st));
    if (n) {
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->scalars.p, scalars, n * 32, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->points_in.p, points, n * pin, cudaMemcpyHostToDevice, st));
    }
    const void *d_pn = ctx->points.p;
    if (point_fmt == DALEK_POINTS_COMPRESSED) {
        // decompress to Niels (Z = 1), then widen to the projective-Niels layout the kernel reads
        if ((rc = ws_reserve(ctx, ctx->misc1, std::max<size_t>(1, n) * sizeof(ge_niels_packed)))) return rc;
        if ((rc = msm_prepare_points(ctx, ctx->points_in.p, point_fmt, n, ctx->misc1.p, (int *)ctx->flags.p))) return rc;
        launch_niels_to_pniels(ctx, ctx->misc1.p, ctx->points.p, n);
    } else {
        if ((rc = msm_prepare_points(ctx, ctx->points_in.p, point_fmt, n, ctx->points.p, (int *)ctx->flags.p))) return rc;
    }
    if ((rc = straus_ct_msm(ctx, (const uint32_t *)ctx->scalars.p, d_pn, n, (MsmResult *)ctx->result.p))) return rc;
    if ((rc = pinned_reserve(ctx, sizeof(MsmResult) + 64))) return rc;
    MsmResult *h = (MsmResult *)ctx->h_pinned;
    int *h_bad = (int *)((char *)ctx->h_pinned + sizeof(MsmResult));
    CUDA_TRY(ctx, cudaMemcpyAsync(h, ctx->result.p, sizeof(MsmResult), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(h_bad, ctx->flags.p, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    float ms = 0.f;
    if (n && (ms = elapsed_ms(ctx->ev_a, ctx->ev_b)) >= 0.f) ctx->last_kernel_ms = ms;
    if (*h_bad) { ctx->last_error = "a compressed point does not decode (multiscalar_mul takes points, not Options)"; return DALEK_E_INVALID_ARG; }
    if (out_compressed) memcpy(out_compressed, h->compressed, 32);
    if (out_limbs) memcpy(out_limbs, h->limbs, 160);
    return DALEK_OK;
}

int dalek_b200_ristretto_double_base_batch(dalek_b200_ctx *ctx, const uint8_t *a, const uint8_t *b, const uint8_t G[32],
                                           const uint8_t H[32], size_t n, uint8_t *out)
{
    if (!ctx || !G || !H || (n && (!a || !b || !out))) return DALEK_E_INVALID_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    {   // Scalar invariant #1 (scalar.rs:214-230): bit 255 clear
        uint8_t top = 0;
        for (size_t i = 0; i < n; i++) top |= a[32 * i + 31] | b[32 * i + 31];
        if (top & 0x80) { ctx->last_error = "scalar with bit 255 set (Scalar invariant #1)"; return DALEK_E_INVALID_ARG; }
    }
    int rc;
    if ((rc = ws_reserve(ctx, ctx->scalars, std::max<size_t>(1, n) * 64))) return rc;
    if ((rc = ws_reserve(ctx, ctx->points_in, std::max<size_t>(1, n) * 32))) return rc;
    uint8_t *d_a = (uint8_t *)ctx->scalars.p, *d_b = d_a + n * 32, *d_out = (uint8_t *)ctx->points_in.p;
    DoubleBasePlan plan;
    if ((rc = double_base_setup(ctx, G, H, n, plan))) return rc;
    // The batch is independent per pair: pieces alternate between two streams, each doing copy-in -> kernel ->
    // copy-out, so that the PCIe traffic of one piece (both directions) hides under the arithmetic of its
    // neighbours.  (With pageable caller memory the copies are staged by the driver and overlap less.)
    cudaStream_t ss[2] = {ctx->stream, ctx->stream2};
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));
    CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_a, ctx->stream));
    // piece size: two full waves of the comb kernel (one 384-thread CTA per SM), so that no piece ends in a
    // partly filled wave; the per-pair Straus kernel has small CTAs and simply gets 8 pieces
    size_t piece = n;
    if (n >= (1u << 16)) piece = plan.variant == 1 ? (size_t)2 * ctx->sm_count * 384 : (n + 7) / 8;
    size_t k = 0;
    for (size_t lo = 0; lo < n; lo += piece, k++) {
        const size_t m = std::min(piece, n - lo);
        cudaStream_t st = ss[k & 1];
        CUDA_TRY(ctx, cudaMemcpyAsync(d_a + 32 * lo, a + 32 * lo, 32 * m, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(d_b + 32 * lo, b + 32 * lo, 32 * m, cudaMemcpyHostToDevice, st));
        if ((rc = double_base_launch(ctx, plan, d_a + 32 * lo, d_b + 32 * lo, m, d_out + 32 * lo, st))) return rc;
        CUDA_TRY(ctx, cudaMemcpyAsync(out + 32 * lo, d_out + 32 * lo, 32 * m, cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_join, ctx->stream2));
    CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_b, ctx->stream));          // ev_a .. ev_b: device span of the whole batch, copies included
    int status = 0;
    if ((rc = double_base_status(ctx, plan, &status))) return rc;
    if (status) return DALEK_NONE;                                   // G or H does not decode; `out` is unspecified
    return DALEK_OK;
}

int dalek_b200_ristretto_vartime_msm(dalek_b200_ctx *ctx, const uint8_t *scalars, const uint8_t *points, size_t n,
                                     uint8_t out_compressed[32])
{
    if (!ctx || !out_compressed || (n && (!scalars || !points)) || n >= (1ull << 31)) return DALEK_E_INVALID_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    int rc;
    cudaStream_t st = ctx->stream;
    if ((rc = ws_reserve(ctx, ctx->scalars, std::max<size_t>(1, n) * 32))) return rc;
    if ((rc = ws_reserve(ctx, ctx->points_in, std::max<size_t>(1, n) * 32))) return rc;
    if ((rc = ws_reserve(ctx, ctx->points, std::max<size_t>(1, n) * sizeof(ge_pniels_packed)))) return rc;
    if ((rc = ws_reserve(ctx, ctx->flags, 64))) return rc;
    if ((rc = ws_reserve(ctx, ctx->result, sizeof(MsmResult) + 64))) return rc;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->flags.p, 0, 64, st));
    if (n) {
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->scalars.p, scalars, n * 32, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->points_in.p, points, n * 32, cudaMemcpyHostToDevice, st));
        if (ctx->opt_decompress_f64) k_prep_ristretto<1, 0><<<cdiv(n, 128), 128, 0, st>>>((const uint32_t *)ctx->points_in.p, (ge_pniels_packed *)ctx->points.p, n, (int *)ctx->flags.p, SegStatus{});
        else k_prep_ristretto<0, 0><<<cdiv(n, 128), 128, 0, st>>>((const uint32_t *)ctx->points_in.p, (ge_pniels_packed *)ctx->points.p, n, (int *)ctx->flags.p, SegStatus{});
        ctx->launches++;
    }
    int c = msm_choose_window_bits(ctx, n);
    int nwin = msm_window_count_for_bits(c);
    if ((rc = ws_reserve(ctx, ctx->misc0, (size_t)nwin * sizeof(ge_p3_raw)))) return rc;
    if ((rc = msm_full(ctx, (const uint32_t *)ctx->scalars.p, ctx->points.p, PK_PNIELS, n, c, (ge_p3_raw *)ctx->misc0.p, (MsmResult *)ctx->result.p))) return rc;
    uint32_t *d_enc = (uint32_t *)((char *)ctx->result.p + sizeof(MsmResult));
    k_ristretto_encode_result<<<1, 1, 0, st>>>((const MsmResult *)ctx->result.p, d_enc);
    ctx->launches++;
    if ((rc = pinned_reserve(ctx, 128))) return rc;
    int *h_bad = (int *)((char *)ctx->h_pinned + 64);
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_pinned, d_enc, 32, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(h_bad, ctx->flags.p, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    memcpy(out_compressed, ctx->h_pinned, 32);
    return *h_bad ? DALEK_NONE : DALEK_OK;
}

}  // extern "C"

// Niels (Z = 1) -> projective Niels layout
__global__ void k_niels_to_pniels(const ge_niels_packed *__restrict__ in, ge_pniels_packed *__restrict__ out, size_t n)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ge_niels_packed a = in[i];
    ge_pniels_packed o;
#pragma unroll
    for (int k = 0; k < 8; k++) { o.w[k] = a.w[k]; o.w[8 + k] = a.w[8 + k]; o.w[16 + k] = k == 0 ? 1u : 0u; o.w[24 + k] = a.w[16 + k]; }
    out[i] = o;
}
void launch_niels_to_pniels(dalek_b200_ctx *ctx, const void *in, void *out, size_t n)
{
    if (!n) return;
    k_niels_to_pniels<<<cdiv(n, 128), 128, 0, ctx->stream>>>((const ge_niels_packed *)in, (ge_pniels_packed *)out, n);
    ctx->launches++;
}
