// straus_vt.cuh -- device code of the variable-time Straus path for small inputs (straus_vt.cu): the width-5
// non-adjacent form (scalar.rs:955-1007), the table of odd multiples (window.rs:201-211) and the per-warp main
// loop (straus.rs:181-197).  In a header so that tests/host runs the same code on an emulated warp.
#pragma once
#include "warp4_f64.cuh"

// Scalar::non_adjacent_form(5), scalar.rs:955-1007, on four 64-bit words.  The reference requires bit 255 clear
// (debug_assert, scalar.rs:960) and produces 256 digits; this boundary takes any 256-bit value, so NAF_LEN digits are
// produced: for reference-legal scalars the digits beyond 255 are zero and the first 256 are the reference's.
#define NAF_LEN 264
FE_HD void naf5(int8_t *naf /* NAF_LEN */, const uint32_t s[8])
{
    uint64_t x[6];
#pragma unroll
    for (int i = 0; i < 4; i++) x[i] = (uint64_t)s[2 * i] | ((uint64_t)s[2 * i + 1] << 32);
    x[4] = 0; x[5] = 0;
    const uint64_t width = 32, window_mask = 31;
    uint32_t pos = 0;
    uint64_t carry = 0;
    for (int i = 0; i < NAF_LEN; i++) naf[i] = 0;
    while (pos < NAF_LEN - 5) {
        const uint32_t idx = pos >> 6, bit = pos & 63;
        uint64_t bit_buf;
        if (bit < 64 - 5) bit_buf = x[idx] >> bit;
        else bit_buf = (x[idx] >> bit) | (x[idx + 1] << (64 - bit));
        const uint64_t window = carry + (bit_buf & window_mask);
        if ((window & 1) == 0) { pos += 1; continue; }              // scalar.rs:990-996
        if (window < width / 2) { carry = 0; naf[pos] = (int8_t)window; }
        else { carry = 1; naf[pos] = (int8_t)((int64_t)window - (int64_t)width); }
        pos += 5;
    }
}

// EdwardsPoint::as_projective_niels (edwards.rs:528-535) with canonical 32-byte coordinates
FE_HD void ge64_pack_pniels(ge_pniels_packed &pk, const ge64_p3 &p, const fe64 &d2)
{
    fe64 ypx, ymx, t2d;
    fe64_add(ypx, p.Y, p.X); fe64_sub(ymx, p.Y, p.X); fe64_mul(t2d, p.T, d2);
    ge_pniels n;
    fe64_to_fe(n.YpX, ypx); fe64_to_fe(n.YmX, ymx); fe64_to_fe(n.Z, p.Z); fe64_to_fe(n.T2d, t2d);
    ge_pniels_pack(pk, n);
}

// NafLookupTable5::from (window.rs:201-211): tab = [A, 3A, 5A, ..., 15A] as projective Niels points
FE_HD void straus_table5(ge_pniels_packed tab[8], const ge64_p3 &A)
{
    fe64 d2; fe64_const_2d(d2);
    ge64_p3 A2, acc = A;
    ge64_dbl(A2, A);                                               // window.rs:206
    ge64_pniels A2n;
    fe64_add(A2n.YpX, A2.Y, A2.X); fe64_sub(A2n.YmX, A2.Y, A2.X); A2n.Z = A2.Z; fe64_mul(A2n.T2d, A2.T, d2);
    ge64_pack_pniels(tab[0], acc, d2);                             // Ai[0] = A
#if FE64_DEV
#pragma unroll 1
#endif
    for (int i = 1; i < 8; i++) {                                  // Ai[i] = A2 + Ai[i-1]  (window.rs:207-209)
        ge64_padd(acc, acc, A2n, 0u);
        ge64_pack_pniels(tab[i], acc, d2);
    }
}

// One warp, eight points (group g handles point 8 * warp + g): for i from the top non-zero digit down to 0
//   Q <- 2Q;  Q <- Q +/- table[|naf_i| / 2] when naf_i != 0          (straus.rs:181-197, window.rs:187-192)
// then the eight accumulators of the warp are added.  The sum is replicated in the lanes of group 0 on return.
W4_DEV void straus_warp(w4f_point &Q, const int8_t *nafs, const ge_pniels_packed *tables, size_t n, size_t warp, uint32_t role, uint32_t grp)
{
    const size_t j = warp * 8 + grp;
    const bool live = j < n;
    const int8_t *naf = nafs + NAF_LEN * (live ? j : 0);
    const ge_pniels_packed *tab = tables + 8 * (live ? j : 0);
    fe64 d2; fe64_const_2d(d2);
    w4f_identity(Q);
    // leading zero digits: doubling the identity changes nothing (straus.rs:181-190 starts from the identity)
    int top = -1;
    for (int i = NAF_LEN - 1; i >= 0; i--) {
        const int d = live ? naf[i] : 0;
        if (w4_any(d != 0)) { top = i; break; }
    }
#if FE64_DEV
#pragma unroll 1
#endif
    for (int i = top; i >= 0; i--) {
        const int d = live ? naf[i] : 0;
        const bool any = w4_any(d != 0);
        if (i != top) w4f_dbl(Q, role, any || i == 0);             // the sums below read T of the final Q
        if (any) {                                                 // uniform per warp: full-mask shuffles inside
            const uint32_t neg = d < 0, e = (uint32_t)(neg ? -d : d) >> 1;      // window.rs:187-192: entry |x| / 2
            ge_pniels_packed pk;
#if defined(__CUDA_ARCH__)
            const uint4 *src = reinterpret_cast<const uint4 *>(tab + (d ? e : 0));
#pragma unroll
            for (int k = 0; k < 8; k++) { uint4 v = src[k]; pk.w[4 * k] = v.x; pk.w[4 * k + 1] = v.y; pk.w[4 * k + 2] = v.z; pk.w[4 * k + 3] = v.w; }
#else
            pk = tab[d ? e : 0];
#endif
            w4f_point R = Q;
            w4f_padd(R, pk, neg, role);
            if (d != 0) Q = R;                                     // groups with a zero digit keep Q
        }
    }
    for (int delta = 16; delta >= 4; delta >>= 1) {                // the warp's eight accumulators -> one point
        w4f_point X; w4f_shfl_down(X, Q, delta);
        w4f_add(Q, X, d2, role);
    }
}
