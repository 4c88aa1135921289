// warp4_f64.cuh -- the 4-lane point operations of warp4.cuh over the FP64-pipe field (fe64.cuh).
//
// The final Horner pass over the bucket windows (pippenger.rs:159) is ~250 DEPENDENT doublings: its
// latency is (instructions per doubling) x (issue interval of one lone warp).  The four independent
// field multiplications of each half of a point operation run in the four lanes of a group, as in
// warp4.cuh (the SIMT form of docs/parallel-formulas.md:51-76), but on five balanced FP64 limbs: a
// squaring is 15 split products instead of 55 IMAD.WIDE plus pre-multiplications, an element is ten
// 32-bit registers to select and shuffle instead of ten limbs with masks.  All 32 lanes of a warp must
// execute these calls together (full-mask shuffles).
//
// The lane primitives are wrapped (w4_lane / w4_shfl / w4_shfl_down / w4_any) so that tests/host can run
// the very same code on an emulated warp of host threads, with the operand-rule assertions of the host
// field model switched on.
#pragma once
#include "ge64.cuh"

#if defined(__CUDACC__)
#define W4_DEV __device__ __forceinline__
W4_DEV uint32_t w4_lane() { return threadIdx.x & 31u; }
W4_DEV uint32_t w4_shfl(uint32_t v, int src) { return __shfl_sync(0xffffffffu, v, src); }
W4_DEV uint32_t w4_shfl_down(uint32_t v, int delta) { return __shfl_down_sync(0xffffffffu, v, delta); }
W4_DEV bool w4_any(bool p) { return __any_sync(0xffffffffu, p) != 0; }
W4_DEV long long w4_bits(double d) { return __double_as_longlong(d); }
W4_DEV double w4_from_bits(long long b) { return __longlong_as_double(b); }
#else
#include <string.h>
#define W4_DEV static inline
uint32_t w4_lane();                          // the host emulation of one warp (tests/host/w4_host_check.cpp)
uint32_t w4_shfl(uint32_t v, int src);
uint32_t w4_shfl_down(uint32_t v, int delta);
bool w4_any(bool p);
W4_DEV long long w4_bits(double d) { long long b; memcpy(&b, &d, 8); return b; }
W4_DEV double w4_from_bits(long long b) { double d; memcpy(&d, &b, 8); return d; }
#endif

struct w4f_point { fe64 X, Y, Z, T; };       // extended point, coordinates of scale 1, replicated in the 4 lanes

W4_DEV void fe64_sel4(fe64 &o, const fe64 &a0, const fe64 &a1, const fe64 &a2, const fe64 &a3, uint32_t role)
{
#pragma unroll
    for (int i = 0; i < 5; i++) {
        const double lo = role & 1 ? a1.v[i] : a0.v[i], hi = role & 1 ? a3.v[i] : a2.v[i];
        o.v[i] = role & 2 ? hi : lo;
    }
}

// value held by lane `i` of this lane's group
W4_DEV void fe64_gbcast(fe64 &o, const fe64 &mine, int i)
{
    const int src = (int)((w4_lane() & 28u) | (uint32_t)i);
#pragma unroll
    for (int k = 0; k < 5; k++) {
        const long long v = w4_bits(mine.v[k]);
        const uint32_t lo = w4_shfl((uint32_t)v, src), hi = w4_shfl((uint32_t)(v >> 32), src);
        o.v[k] = w4_from_bits((long long)(((uint64_t)hi << 32) | lo));
    }
}

// scale-1 integer limbs (fe.cuh) -> balanced doubles of scale 1
FE_HD void fe64_from_fe_limbs(fe64 &h, const fe &f)
{
    fe64 t;
#pragma unroll
    for (int k = 0; k < 5; k++) {
        const uint64_t l = (uint64_t)f.v[2 * k] + ((uint64_t)f.v[2 * k + 1] << 26);       // < 2^51 + 2^26: exact in a double
#if FE64_DEV
        t.v[k] = __longlong_as_double((long long)l | FE64_E52) - FE64_TWO52;
#else
        t.v[k] = (double)l;
#endif
    }
    fe64_carry(h, t);
}

W4_DEV void w4f_identity(w4f_point &p) { fe64_0(p.X); fe64_1(p.Y); fe64_1(p.Z); fe64_0(p.T); }

W4_DEV void w4f_load(w4f_point &p, const ge_p3_raw *src)
{
    ge_p3 q;
    ge_p3_raw r;
#if defined(__CUDA_ARCH__)
    const uint4 *s = reinterpret_cast<const uint4 *>(src);
#pragma unroll
    for (int k = 0; k < 10; k++) { uint4 v = s[k]; r.w[4 * k] = v.x; r.w[4 * k + 1] = v.y; r.w[4 * k + 2] = v.z; r.w[4 * k + 3] = v.w; }
#else
    r = *src;
#endif
    ge_p3_load_raw(q, r);
    fe64_from_fe_limbs(p.X, q.X); fe64_from_fe_limbs(p.Y, q.Y); fe64_from_fe_limbs(p.Z, q.Z); fe64_from_fe_limbs(p.T, q.T);
}

// p <- 2p (curve_models.rs:381-397 + :365-372).  T is refreshed only when want_t (the doubling before an addition).
W4_DEV void w4f_dbl(w4f_point &p, uint32_t role, bool want_t)
{
    fe64 S, in, r, XX, YY, ZZ, S2, Yp, Ym, E, F, f, g;
    fe64_add(S, p.X, p.Y); fe64_carry(S, S);                  // squaring needs scale < 2
    fe64_sel4(in, p.X, p.Y, p.Z, S, role);
    fe64_sq(r, in);
    fe64_gbcast(XX, r, 0); fe64_gbcast(YY, r, 1); fe64_gbcast(ZZ, r, 2); fe64_gbcast(S2, r, 3);
    fe64_add(Yp, YY, XX);                                     // 2
    fe64_sub(Ym, YY, XX);                                     // 2
    fe64_sub(E, S2, Yp);                                      // 3   (X+Y)^2 - Y^2 - X^2
    fe64_add(F, ZZ, ZZ); fe64_sub(F, F, Ym);                  // 4   2Z^2 - (Y^2 - X^2)
    fe64_carry(F, F);                                         // 1
    fe64_sel4(f, E, Yp, Ym, E, role);                         // X3 = E F, Y3 = Yp Ym, Z3 = Ym F, T3 = E Yp
    fe64_sel4(g, F, Ym, F, Yp, role);
    fe64_mul(r, f, g);                                        // <= 3 x 2
    fe64_gbcast(p.X, r, 0); fe64_gbcast(p.Y, r, 1); fe64_gbcast(p.Z, r, 2);
    if (want_t) fe64_gbcast(p.T, r, 3);
}

// shared second half of the additions: a, b, c (scale 1), D (scale 2); neg swaps the roles of D + c and D - c
W4_DEV void w4f_add_tail(w4f_point &p, const fe64 &a, const fe64 &b, const fe64 &c, const fe64 &D, uint32_t neg, uint32_t role)
{
    fe64 E, H, DpC, DmC, F, G, f, g, r;
    fe64_sub(E, b, a); fe64_add(H, b, a);                     // 2, 2
    fe64_add(DpC, D, c); fe64_sub(DmC, D, c);                 // 3, 3
    fe64_carry(DmC, DmC);                                     // 1   (3 x 3 would break the operand rule of DmC * DpC)
    F = DmC; fe64_cmov(F, DpC, neg);                          // T of the completed point
    G = DpC; fe64_cmov(G, DmC, neg);                          // Z of the completed point
    fe64_sel4(f, F, G, DmC, E, role);                         // X3 = F E, Y3 = G H, Z3 = DmC DpC, T3 = E H
    fe64_sel4(g, E, H, DpC, H, role);
    fe64_mul(r, f, g);                                        // <= 3 x 2
    fe64_gbcast(p.X, r, 0); fe64_gbcast(p.Y, r, 1); fe64_gbcast(p.Z, r, 2); fe64_gbcast(p.T, r, 3);
}

// p <- p + q, both extended (edwards.rs:795-800 = :528-535 + curve_models.rs:411-430, :365-372); d2 = 2d as fe64
W4_DEV void w4f_add(w4f_point &p, const w4f_point &q, const fe64 &d2, uint32_t role)
{
    fe64 qYpX, qYmX, qT2d, A, B, f, g, r, a, b, c, zz, D;
    fe64_add(qYpX, q.Y, q.X);                                 // 2
    fe64_sub(qYmX, q.Y, q.X);                                 // 2
    fe64_sub(A, p.Y, p.X); fe64_add(B, p.Y, p.X);             // 2, 2
    fe64_mul(qT2d, q.T, d2);                                  // as_projective_niels (replicated in the four lanes)
    fe64_sel4(f, A, B, p.T, p.Z, role);                       // a = A qYmX, b = B qYpX, c = T qT2d, zz = Z qZ
    fe64_sel4(g, qYmX, qYpX, qT2d, q.Z, role);
    fe64_mul(r, f, g);                                        // <= 2 x 2
    fe64_gbcast(a, r, 0); fe64_gbcast(b, r, 1); fe64_gbcast(c, r, 2); fe64_gbcast(zz, r, 3);
    fe64_add(D, zz, zz);                                      // 2
    w4f_add_tail(p, a, b, c, D, 0u, role);
}

// p <- p + q or p - q for a projective Niels point whose coordinates have scale <= 2 (curve_models.rs:411-452 + :365-372)
W4_DEV void w4f_padd_pn(w4f_point &p, const ge64_pniels &q, uint32_t neg, uint32_t role)
{
    fe64 qp = q.YpX, qm = q.YmX;
    { fe64 t = qp; fe64_cmov(qp, qm, neg); fe64_cmov(qm, t, neg); }
    fe64 A, B, f, g, r, a, b, c, zz, D;
    fe64_sub(A, p.Y, p.X); fe64_add(B, p.Y, p.X);             // 2, 2
    fe64_sel4(f, A, B, p.T, p.Z, role);
    fe64_sel4(g, qm, qp, q.T2d, q.Z, role);
    fe64_mul(r, f, g);                                        // <= 2 x 2
    fe64_gbcast(a, r, 0); fe64_gbcast(b, r, 1); fe64_gbcast(c, r, 2); fe64_gbcast(zz, r, 3);
    fe64_add(D, zz, zz);
    w4f_add_tail(p, a, b, c, D, neg, role);
}

// the same for a packed projective Niels point
W4_DEV void w4f_padd(w4f_point &p, const ge_pniels_packed &pk, uint32_t neg, uint32_t role)
{
    ge64_pniels q; ge64_pniels_unpack(q, pk);                 // coordinates in [0, 2^51): scale 2
    w4f_padd_pn(p, q, neg, role);
}

// copy of the point held by the group `delta_lanes` lanes above (delta_lanes a multiple of 4)
W4_DEV void w4f_shfl_down(w4f_point &o, const w4f_point &p, int delta_lanes)
{
    const fe64 *src[4] = {&p.X, &p.Y, &p.Z, &p.T};
    fe64 *dst[4] = {&o.X, &o.Y, &o.Z, &o.T};
#pragma unroll
    for (int c = 0; c < 4; c++)
#pragma unroll
        for (int k = 0; k < 5; k++) {
            const long long v = w4_bits(src[c]->v[k]);
            const uint32_t lo = w4_shfl_down((uint32_t)v, delta_lanes), hi = w4_shfl_down((uint32_t)(v >> 32), delta_lanes);
            dst[c]->v[k] = w4_from_bits((long long)(((uint64_t)hi << 32) | lo));
        }
}

W4_DEV void w4f_to_p3(ge_p3 &o, const w4f_point &p)
{
    fe64_to_fe(o.X, p.X); fe64_to_fe(o.Y, p.Y); fe64_to_fe(o.Z, p.Z); fe64_to_fe(o.T, p.T);
}

// 2d (u64/constants.rs:54) as balanced doubles
FE_HD void fe64_const_2d(fe64 &d2) { fe k; fe_const_2d(k); fe64_from_fe_limbs(d2, k); }

// ---- 20-lane doubling chain: the LIMBS of a point spread over lanes -----------------------------------------------
// A run of doublings without additions (the c doublings between two windows of the Horner pass, 240 of them per MSM, all
// dependent) is bound by the instruction count of ONE doubling on ONE warp.  In the 4-lane form every lane still runs a
// whole 25-product field multiplication.  Here lane 5 g + i holds ONE double: limb i of coordinate g (X, Y, Z, T); a field
// multiplication is then five products per lane (row i of the schoolbook matrix), a transpose-sum over the five lanes of
// the group with shuffles, and ONE parallel round of carries:
//     lane i:  U[e] = (lo(a_i b_e) + 2 f(a_i b_{e-1})) * (19 if i + e >= 5),   U[0] = lo(a_i b_0) + 38 f(a_i b_4)
//     limb k = sum_d U_{lane (k - d) mod 5}[d];   q_k = round(limb_k / 2^51);   limb_k <- limb_k - q_k 2^51 + q_{k-1} (19 q_4)
// (p = f 2^52 + lo is the exact split of fe64_mul).  |column| < 2^60, so |q| < 2^9 and limbs end within 2^50 + 2^14: scale 1
// under the operand rule.  About 270 instructions per doubling instead of about 700.  Lanes 20..31 mirror lanes 0..11.
struct w20_role { uint32_t g, i, base; };
W4_DEV w20_role w20_roles() { const uint32_t l = w4_lane(); w20_role r; r.g = (l / 5u) & 3u; r.i = l % 5u; r.base = 5u * r.g; return r; }

W4_DEV double w20_shfl(double v, uint32_t src)
{
    const long long b = w4_bits(v);
    const uint32_t lo = w4_shfl((uint32_t)b, (int)src), hi = w4_shfl((uint32_t)((uint64_t)b >> 32), (int)src);
    return w4_from_bits((long long)(((uint64_t)hi << 32) | lo));
}
W4_DEV long long w20_shfl_ll(long long b, uint32_t src)
{
    const uint32_t lo = w4_shfl((uint32_t)b, (int)src), hi = w4_shfl((uint32_t)((uint64_t)b >> 32), (int)src);
    return (long long)(((uint64_t)hi << 32) | lo);
}

// fe64_carry on a limb-distributed element (every lane of a group holds its limb of the same element)
W4_DEV double w20_carry(double f, const w20_role &r)
{
#if FE64_DEV
    const double C = 6755399441055744.0;                                 // 1.5 * 2^52
    const double q = __fma_rn(f, 1.0 / 2251799813685248.0, C) - C;       // round(f / 2^51)
    const double rr = __fma_rn(q, -2251799813685248.0, f);
#else
    const double q = nearbyint(f / 2251799813685248.0), rr = f - q * 2251799813685248.0;
#endif
    const double qp = w20_shfl(q, r.base + (r.i + 4u) % 5u);
    return rr + (r.i == 0 ? 19.0 * qp : qp);
}

// exact split of one limb product: p = a b = f 2^52 + lo, f = floor(p / 2^52), 0 <= lo < 2^52   (|p| < 2^103)
W4_DEV void w20_split(long long &f, long long &lo, double a, double b, double b_scaled /* b 2^-52 */)
{
#if FE64_DEV
    const double M1 = 6755399441055744.0;                               // 1.5 * 2^52
    const double K = 6755399441055744.0 * 4503599627370496.0 + 4503599627370496.0;
    const double t = __fma_rz(a, b_scaled, M1);
    const double u = __fma_rn(t, -4503599627370496.0, K);
    const double l = __fma_rn(a, b, u);
    f = __double_as_longlong(t) - (FE64_E52 + (1LL << 51));
    lo = __double_as_longlong(l) - FE64_E52;
#else
    (void)b_scaled;
    const __int128 p = (__int128)(long long)a * (__int128)(long long)b, lim = (__int128)1 << 103;
    assert(p < lim && p > -lim);
    f = (long long)(p >> 52);
    lo = (long long)(p - ((__int128)f << 52));
#endif
}

// limb i of A * B from limb i of A and limb i of B (both limb-distributed over the lanes of the group)
W4_DEV double w20_mul(double a_own, double b_own, const w20_role &r)
{
    double b[5];
#pragma unroll
    for (uint32_t j = 0; j < 5; j++) b[j] = w20_shfl(b_own, r.base + j);
    long long f[5], lo[5];
#pragma unroll
    for (int d = 0; d < 5; d++) w20_split(f[d], lo[d], a_own, b[d], b[d] * (1.0 / 4503599627370496.0));
    long long U[5];
    U[0] = lo[0] + 38 * f[4];
#pragma unroll
    for (uint32_t e = 1; e < 5; e++) {
        const long long v = lo[e] + 2 * f[e - 1];
        U[e] = r.i + e >= 5u ? 19 * v : v;
    }
    long long R = U[0];
#pragma unroll
    for (uint32_t d = 1; d < 5; d++) R += w20_shfl_ll(U[d], r.base + (r.i + 5u - d) % 5u);
    const long long q = (R + (1LL << 50)) >> 51;
    const long long rr = R - q * (1LL << 51);
    long long qp = (long long)(int32_t)w4_shfl((uint32_t)(int32_t)q, (int)(r.base + (r.i + 4u) % 5u));
    if (r.i == 0) qp *= 19;
    const long long limb = rr + qp;
#if FE64_DEV
    return __longlong_as_double((limb + (1LL << 51)) | FE64_E52) - (FE64_TWO52 + FE64_TWO51);
#else
    assert(limb < (1LL << 50) + (1LL << 15) && limb > -(1LL << 50) - (1LL << 15));
    return (double)limb;
#endif
}

// own limb of the replicated point / back (c = limb i of coordinate g)
W4_DEV double w20_take(const w4f_point &p, const w20_role &r)
{
    double v = 0.0;
#pragma unroll
    for (uint32_t k = 0; k < 5; k++) {
        const double x = r.g == 0 ? p.X.v[k] : r.g == 1 ? p.Y.v[k] : r.g == 2 ? p.Z.v[k] : p.T.v[k];
        if (r.i == k) v = x;
    }
    return v;
}
W4_DEV void w20_give(w4f_point &p, double c)
{
#pragma unroll
    for (uint32_t k = 0; k < 5; k++) {
        p.X.v[k] = w20_shfl(c, k); p.Y.v[k] = w20_shfl(c, 5u + k); p.Z.v[k] = w20_shfl(c, 10u + k); p.T.v[k] = w20_shfl(c, 15u + k);
    }
}

// c <- limb of 2P (curve_models.rs:381-397 + :365-372; the same formulas and scales as w4f_dbl); T is not read
W4_DEV void w20_dbl(double &c, const w20_role &r)
{
    const double x = w20_shfl(c, r.i), y = w20_shfl(c, 5u + r.i);
    const double s = w20_carry(x + y, r);                               // squaring operand of scale 1
    const double in = r.g == 3 ? s : c;
    const double sq = w20_mul(in, in, r);                               // XX, YY, ZZ, (X+Y)^2 in groups 0..3
    const double xx = w20_shfl(sq, r.i), yy = w20_shfl(sq, 5u + r.i), zz = w20_shfl(sq, 10u + r.i), s2 = w20_shfl(sq, 15u + r.i);
    const double Yp = yy + xx, Ym = yy - xx;                            // 2, 2
    const double E = s2 - Yp;                                           // 3
    const double F = w20_carry(zz + zz - Ym, r);                        // 4 -> 1
    const double a = r.g == 1 ? Yp : r.g == 2 ? Ym : E;                 // X3 = E F, Y3 = Yp Ym, Z3 = Ym F, T3 = E Yp
    const double b = r.g == 1 ? Ym : r.g == 3 ? Yp : F;
    c = w20_mul(a, b, r);                                               // <= 3 x 2
}

// p <- 2^k p
W4_DEV void w20_dbl_n(w4f_point &p, int k)
{
    const w20_role r = w20_roles();
    double c = w20_take(p, r);
#if FE64_DEV
#pragma unroll 1
#endif
    for (int t = 0; t < k; t++) w20_dbl(c, r);
    w20_give(p, c);
}

// Horner over windows (pippenger.rs:159): total = total * 2^c + sum over ranks of window w, from the top window down.
// windows: rank-major (ranks x nwin raw points).  The result is replicated in the four lanes of every group.
W4_DEV void w4f_horner(w4f_point &tot, const ge_p3_raw *windows, int ranks, int nwin, int c, uint32_t role)
{
    fe64 d2; fe64_const_2d(d2);
    w4f_point x;
    w4f_identity(tot);
    // Leading windows that are empty contribute nothing and doubling the identity is wasted latency: the top window of
    // every MSM over canonical scalars (< 2^253) is the carry window of the signed recoding, always empty; short scalars
    // (verify_batch's 128-bit z_i) leave more.  `started` is uniform over the warp (every lane loads the same points).
    bool started = false;
#pragma unroll 1
    for (int w = nwin - 1; w >= 0; w--) {
        if (started) {
            w20_dbl_n(tot, c);
        } else {
            bool any = false;
#pragma unroll 1
            for (int r = 0; r < ranks; r++) {
                ge_p3 q; ge_p3_raw raw;
#if defined(__CUDA_ARCH__)
                const uint4 *s4 = reinterpret_cast<const uint4 *>(windows + (size_t)r * nwin + w);
#pragma unroll
                for (int k = 0; k < 10; k++) { uint4 v = s4[k]; raw.w[4 * k] = v.x; raw.w[4 * k + 1] = v.y; raw.w[4 * k + 2] = v.z; raw.w[4 * k + 3] = v.w; }
#else
                raw = windows[(size_t)r * nwin + w];
#endif
                ge_p3_load_raw(q, raw);
                any |= !ge_is_identity(q);
            }
            if (!any) continue;
            started = true;
        }
#pragma unroll 1
        for (int r = 0; r < ranks; r++) { w4f_load(x, windows + (size_t)r * nwin + w); w4f_add(tot, x, d2, role); }
    }
}
