// straus_vt.cu -- variable-time Straus for SMALL inputs: what EdwardsPoint::optional_multiscalar_mul dispatches to
// below 190 points (curve25519-dalek/src/edwards.rs:1025-1029 -> backend/serial/scalar_mul/straus.rs:159-200).
//
// The bucket pipeline (msm.cu) costs ~27 dependent kernel launches whatever n is; for a few dozen points the call is
// then launch- and latency-bound.  This path is three launches:
//
//   k_straus_prepare   one thread per (scalar, point): width-5 non-adjacent form of the scalar
//                      (Scalar::non_adjacent_form, scalar.rs:955-1007) and the table [A, 3A, ..., 15A] of projective
//                      Niels points (NafLookupTable5::from, window.rs:201-211)
//   k_straus_vartime   one warp per 8 points, one 4-lane group per point (warp4_f64.cuh): for i = 255..0
//                      Q <- 2Q; Q <- Q +/- table[|naf_i| / 2] when naf_i != 0 (straus.rs:181-197, window.rs:187-192);
//                      the reference shares ONE accumulator between the points of a call, here every group keeps its
//                      own (the doublings of different groups run in parallel lanes) and the warp adds its eight
//                      accumulators at the end -- the same group element
//   k_combine (msm.cu) sum of the per-warp results, encoding
//
// Variable time by contract (VartimeMultiscalarMul): digits select table entries by address and skip additions.
#include "../../include/dalek_b200.h"
#include "engine.h"
#include "warp4.cuh"
#include "straus_vt.cuh"

template <int KIND>
__global__ void __launch_bounds__(64)
k_straus_prepare(const uint32_t *__restrict__ scalars, const void *__restrict__ points, size_t n, int8_t *__restrict__ nafs,
                 ge_pniels_packed *__restrict__ tables)
{
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    uint32_t s[8];
#pragma unroll
    for (int k = 0; k < 8; k++) s[k] = scalars[8 * j + k];
    naf5(nafs + NAF_LEN * j, s);
    // A as an extended point: identity + the prepared (Niels / projective Niels) form of the input
    ge64_p3 A;
    ge64_identity(A);
    if (KIND == PK_NIELS) {
        ge_niels_packed pk = reinterpret_cast<const ge_niels_packed *>(points)[j];
        ge64_niels nl; ge64_niels_unpack(nl, pk);
        ge64_madd(A, A, nl, 0u);
    } else {
        ge_pniels_packed pk = reinterpret_cast<const ge_pniels_packed *>(points)[j];
        ge64_pniels pn; ge64_pniels_unpack(pn, pk);
        ge64_padd(A, A, pn, 0u);
    }
    ge_pniels_packed tab[8];
    straus_table5(tab, A);
#pragma unroll 1
    for (int i = 0; i < 8; i++) {
        uint4 *o = reinterpret_cast<uint4 *>(tables + 8 * j + i);
#pragma unroll
        for (int k = 0; k < 8; k++) o[k] = make_uint4(tab[i].w[4 * k], tab[i].w[4 * k + 1], tab[i].w[4 * k + 2], tab[i].w[4 * k + 3]);
    }
}

__global__ void __launch_bounds__(32)
k_straus_vartime(const int8_t *__restrict__ nafs, const ge_pniels_packed *__restrict__ tables, size_t n, ge_p3_raw *__restrict__ partial)
{
    const uint32_t lane = threadIdx.x, role = lane & 3, grp = lane >> 2;
    w4f_point Q;
    straus_warp(Q, nafs, tables, n, blockIdx.x, role, grp);
    if (grp == 0) {
        ge_p3 o; w4f_to_p3(o, Q);
        fe mine; fe_sel4(mine, o.X, o.Y, o.Z, o.T, role);
        uint32_t *dst = partial[blockIdx.x].w + 10 * role;
#pragma unroll
        for (int i = 0; i < 10; i += 2) *reinterpret_cast<uint2 *>(dst + i) = make_uint2(mine.v[i], mine.v[i + 1]);
    }
}

int straus_prepare(dalek_b200_ctx *ctx, cudaStream_t st, const uint32_t *d_scalars, const void *d_points, int point_kind, size_t n,
                   int8_t *d_nafs, ge_pniels_packed *d_tables)
{
    if (!n) return 0;
    const unsigned grid = (unsigned)((n + 63) / 64);
    if (point_kind == PK_NIELS) k_straus_prepare<PK_NIELS><<<grid, 64, 0, st>>>(d_scalars, d_points, n, d_nafs, d_tables);
    else k_straus_prepare<PK_PNIELS><<<grid, 64, 0, st>>>(d_scalars, d_points, n, d_nafs, d_tables);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return 0;
}

// sum scalars[i] * points[i] for n < 2^16 prepared points (PK_NIELS / PK_PNIELS); result like msm_full
int straus_vartime_msm(dalek_b200_ctx *ctx, const uint32_t *d_scalars, const void *d_points, int point_kind, size_t n,
                       MsmResult *d_result)
{
    int rc;
    cudaStream_t st = ctx->stream;
    const size_t n1 = n ? n : 1, nwarps = (n + 7) / 8;
    if ((rc = ws_reserve(ctx, ctx->digits, n1 * NAF_LEN))) return rc;
    if ((rc = ws_reserve(ctx, ctx->red_a, n1 * 8 * sizeof(ge_pniels_packed)))) return rc;
    if ((rc = ws_reserve(ctx, ctx->red_b, (nwarps ? nwarps : 1) * sizeof(ge_p3_raw)))) return rc;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_a, st));             // ev_a .. ev_b: the Straus kernels (also recorded for n = 0)
    if (n) {
        if ((rc = straus_prepare(ctx, st, d_scalars, d_points, point_kind, n, (int8_t *)ctx->digits.p, (ge_pniels_packed *)ctx->red_a.p))) return rc;
        k_straus_vartime<<<(unsigned)nwarps, 32, 0, st>>>((const int8_t *)ctx->digits.p, (const ge_pniels_packed *)ctx->red_a.p, n, (ge_p3_raw *)ctx->red_b.p);
        ctx->launches++;
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_b, st));
    ctx->last_kernel_launches = 1;
    CUDA_TRY(ctx, cudaGetLastError());
    return msm_combine_windows(ctx, (const ge_p3_raw *)ctx->red_b.p, (int)nwarps, 1, 1, d_result);   // nwin = 1: plain sum of the warps' results
}
