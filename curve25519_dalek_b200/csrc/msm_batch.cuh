// msm_batch.cuh -- device routine and host planner of the batched vartime MSM (msm_batch.cu): m independent
// VartimeMultiscalarMul::optional_multiscalar_mul calls (traits.rs:196-262) in one call.  In a header so that
// tests/host runs the same code (the planner, and the group routine on an emulated warp).
#pragma once
#include <stdint.h>

#include <algorithm>
#include <vector>

#include "straus_vt.cuh"

// ---- plan (host): a pure function of the segment lengths, the bucket threshold and the SM count -------------------
struct BatchTask { uint32_t pair, len; };     // pairs [pair, pair + len) of the piece, all of ONE segment
struct BatchSum { uint32_t off, len; };       // tasks [off, off + len) of the piece: one segment (k_plain_sum's descriptor)
struct BatchPiece {
    uint64_t pair0, pair1;                     // pairs of the piece
    size_t seg0, seg1;                         // segments of the piece (consecutive)
    bool bucket;                               // one segment of >= bucket_min pairs: the bucket pipeline (msm.cu)
    std::vector<BatchTask> tasks;              // Straus pieces: the tasks of every segment, in segment order
    std::vector<BatchSum> sums;                // Straus pieces: one per segment seg0 .. seg1
};
struct BatchPlan { uint32_t p = 1; std::vector<BatchPiece> pieces; };

#define BATCH_PIECE_PAIRS ((uint64_t)1 << 20)   // Straus workspace per piece: 264 B of digits + 1 KiB of table per pair
#define BATCH_MAX_PAIRS_PER_TASK 64u

// Pairs per task: as many as keep about 64 groups of four lanes (full occupancy) per SM busy.  More pairs per task share
// more doublings (256 per task), fewer leave SMs idle.
inline uint32_t batch_pairs_per_task(uint64_t straus_pairs, int sm_count)
{
    const uint64_t want = (uint64_t)(sm_count > 0 ? sm_count : 1) * 64;
    uint32_t p = 1;
    while (p < BATCH_MAX_PAIRS_PER_TASK && straus_pairs / (2 * (uint64_t)p) >= want) p *= 2;
    return p;
}

// Segment k = pairs [offs[k], offs[k+1]).  Segments shorter than bucket_min (>= 1) and no longer than piece_cap run on the
// segmented Straus path in pieces of at most piece_cap pairs, cut at segment boundaries; every other segment is a piece
// of its own on the bucket pipeline (so the Straus workspace stays bounded whatever bucket_min is).  p_force > 0
// overrides the pairs per task (tests).
inline void batch_plan(BatchPlan &plan, const uint64_t *offs, size_t m, uint64_t bucket_min, int sm_count, uint64_t piece_cap,
                       uint32_t p_force = 0)
{
    plan.pieces.clear();
    uint64_t straus_pairs = 0;
    auto bucket = [&](uint64_t len) { return len >= bucket_min || len > piece_cap; };
    for (size_t k = 0; k < m; k++) if (!bucket(offs[k + 1] - offs[k])) straus_pairs += offs[k + 1] - offs[k];
    const uint32_t p = p_force ? p_force : batch_pairs_per_task(straus_pairs, sm_count);
    plan.p = p;
    BatchPiece cur;
    bool open = false;
    for (size_t k = 0; k < m; k++) {
        const uint64_t len = offs[k + 1] - offs[k];
        if (bucket(len)) {
            if (open) { plan.pieces.push_back(std::move(cur)); open = false; }
            BatchPiece b;
            b.pair0 = offs[k]; b.pair1 = offs[k + 1]; b.seg0 = k; b.seg1 = k + 1; b.bucket = true;
            plan.pieces.push_back(std::move(b));
            continue;
        }
        if (open && cur.pair1 - cur.pair0 + len > piece_cap) { plan.pieces.push_back(std::move(cur)); open = false; }
        if (!open) {
            cur = BatchPiece();
            cur.pair0 = cur.pair1 = offs[k]; cur.seg0 = cur.seg1 = k; cur.bucket = false;
            open = true;
        }
        BatchSum s{(uint32_t)cur.tasks.size(), 0};
        for (uint64_t a = 0; a < len; a += p) {
            cur.tasks.push_back(BatchTask{(uint32_t)(offs[k] + a - cur.pair0), (uint32_t)std::min<uint64_t>(p, len - a)});
            s.len++;
        }
        cur.sums.push_back(s);
        cur.pair1 = offs[k + 1]; cur.seg1 = k + 1;
    }
    if (open) plan.pieces.push_back(std::move(cur));
}

// ---- segmented vartime Straus: one 4-lane group per task ------------------------------------------------------------
// The group keeps ONE accumulator over the task's pairs, as the reference's Straus does (straus.rs:181-197): for i from
// the top non-zero digit down to 0, Q <- 2Q, then Q <- Q +/- table_j[|naf_j[i]| / 2] for every pair j with a non-zero
// digit (window.rs:187-192).  The 256 doublings are paid once per task.
//
// Uniform op stream: every step of every group is the complete unified addition (curve_models.rs:411-452) -- of Q itself
// (a doubling) or of the group's next table entry -- so the eight groups of a warp run the same instructions whatever
// their digits are, and the warp runs max over its groups of (doublings + additions) steps instead of paying an addition
// whenever any group needs one.  A group whose stream has ended keeps its Q.  All 32 lanes must call this together.
W4_DEV void straus_task_group(w4f_point &Q, const int8_t *nafs, const ge_pniels_packed *tables, uint32_t pair, uint32_t len,
                              bool live, uint32_t role)
{
    fe64 d2; fe64_const_2d(d2);
    w4f_identity(Q);
    if (!live) len = 0;
    const int8_t *naf = nafs + (size_t)NAF_LEN * pair;
    const ge_pniels_packed *tab = tables + (size_t)8 * pair;
    int top = -1;                                                  // leading zero digits: doubling the identity is a no-op
    for (uint32_t j = 0; j < len; j++)
        for (int i = NAF_LEN - 1; i > top; i--)
            if (naf[(size_t)NAF_LEN * j + i]) { top = i; break; }
    int i = top;
    uint32_t j = 0;
    bool dbl = false;                                              // a doubling is due before the additions of bit i
#if FE64_DEV
#pragma unroll 1
#endif
    for (;;) {
        int op = 0, d = 0;                                         // 0: stream ended, 1: doubling, 2: addition of pair jj
        uint32_t jj = 0;
        while (i >= 0) {
            if (dbl) { dbl = false; op = 1; break; }
            while (j < len && naf[(size_t)NAF_LEN * j + i] == 0) j++;
            if (j < len) { d = naf[(size_t)NAF_LEN * j + i]; jj = j++; op = 2; break; }
            i--; j = 0; dbl = true;
        }
        if (!w4_any(op != 0)) break;
        ge64_pniels q;                                             // Q as projective Niels (scale <= 2), as w4f_add forms it
        fe64_add(q.YpX, Q.Y, Q.X); fe64_sub(q.YmX, Q.Y, Q.X); q.Z = Q.Z; fe64_mul(q.T2d, Q.T, d2);
        uint32_t neg = 0;
        if (op == 2) {
            neg = d < 0;
            const uint32_t e = (uint32_t)(neg ? -d : d) >> 1;
            ge_pniels_packed pk;
#if defined(__CUDA_ARCH__)
            const uint4 *src = reinterpret_cast<const uint4 *>(tab + 8 * (size_t)jj + e);
#pragma unroll
            for (int k = 0; k < 8; k++) { uint4 v = src[k]; pk.w[4 * k] = v.x; pk.w[4 * k + 1] = v.y; pk.w[4 * k + 2] = v.z; pk.w[4 * k + 3] = v.w; }
#else
            pk = tab[8 * (size_t)jj + e];
#endif
            ge64_pniels_unpack(q, pk);
        }
        w4f_point R = Q;
        w4f_padd_pn(R, q, neg, role);
        if (op) Q = R;
    }
}
