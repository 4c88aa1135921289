// Host checks of the batched vartime MSM (csrc/msm_batch.cuh): the planner's invariants, and the segmented Straus group
// routine (straus_task_group) on the emulated warp of w4_host_check.cpp with the operand-rule assertions switched on.
// TEST INFRASTRUCTURE (tests/test_msm_batch_host.py): not a CPU fallback of the product.
#include "w4_host_check.cpp"                   // the emulated warp (run_warp, lane primitives) and the point helpers
#include "../../curve25519_dalek_b200/csrc/msm_batch.cuh"

extern "C" {

// Plan of the segments offs[0..m] and its invariants.  path[k] = 0 (segmented Straus) or 1 (bucket pipeline).
// Returns 1 if every invariant holds, a negative code naming the first one that does not.
int h_plan(const uint64_t *offs, size_t m, uint64_t bucket_min, int sm_count, uint64_t cap, uint8_t *path, uint64_t *npieces,
           uint32_t *p_out)
{
    BatchPlan plan;
    batch_plan(plan, offs, m, bucket_min, sm_count, cap);
    *npieces = plan.pieces.size();
    *p_out = plan.p;
    if (plan.p < 1 || plan.p > BATCH_MAX_PAIRS_PER_TASK) return -1;
    std::vector<uint8_t> covered(offs[m], 0);
    size_t seg = 0;
    for (const BatchPiece &pc : plan.pieces) {
        if (pc.seg0 != seg || pc.seg1 <= pc.seg0 || pc.seg1 > m) return -2;               // consecutive segments, none skipped
        if (pc.pair0 != offs[pc.seg0] || pc.pair1 != offs[pc.seg1]) return -3;              // pieces end at segment boundaries
        seg = pc.seg1;
        if (pc.bucket) {
            const uint64_t len = offs[pc.seg1] - offs[pc.seg0];
            if (pc.seg1 != pc.seg0 + 1 || (len < bucket_min && len <= cap)) return -4;
            path[pc.seg0] = 1;
            for (uint64_t a = pc.pair0; a < pc.pair1; a++) covered[a]++;
            continue;
        }
        if (pc.pair1 - pc.pair0 > cap) return -5;                                            // workspace bound
        if (pc.sums.size() != pc.seg1 - pc.seg0) return -6;
        uint32_t next_task = 0;
        for (size_t k = pc.seg0; k < pc.seg1; k++) {
            if (offs[k + 1] - offs[k] >= bucket_min) return -7;
            path[k] = 0;
            const BatchSum s = pc.sums[k - pc.seg0];
            if (s.off != next_task || s.off + s.len > pc.tasks.size()) return -8;
            uint64_t at = offs[k];
            for (uint32_t t = s.off; t < s.off + s.len; t++) {
                const BatchTask tk = pc.tasks[t];
                if (tk.len < 1 || tk.len > plan.p || pc.pair0 + tk.pair != at) return -9;      // tasks tile the segment in order
                for (uint32_t j = 0; j < tk.len; j++) covered[at + j]++;
                at += tk.len;
            }
            if (at != offs[k + 1]) return -10;
            next_task = s.off + s.len;
        }
        if (next_task != pc.tasks.size()) return -11;
    }
    if (seg != m) return -12;
    for (uint8_t c : covered) if (c != 1) return -13;                                         // every pair exactly once
    return 1;
}

// Segments offs[0..m] of compressed points, all on the segmented Straus path with p pairs per task: tables and NAFs as
// k_straus_prepare makes them, straus_task_group on emulated warps of eight tasks (so warps span segments and the last
// one is partly filled), the per-segment sum of the task accumulators.  out: m x 32 B compressed.
int h_straus_segmented(uint8_t *out, const uint8_t *scalars, const uint8_t *points, const uint64_t *offs, size_t m, uint32_t p)
{
    BatchPlan plan;
    batch_plan(plan, offs, m, ~0ull, 148, ~0ull, p);
    if (plan.pieces.size() != (m ? 1u : 0u)) return -1;
    const size_t n = offs[m];
    std::vector<int8_t> nafs((size_t)NAF_LEN * (n ? n : 1));
    std::vector<ge_pniels_packed> tables((size_t)8 * (n ? n : 1));
    for (size_t j = 0; j < n; j++) {
        uint32_t s[8]; memcpy(s, scalars + 32 * j, 32);
        naf5(&nafs[(size_t)NAF_LEN * j], s);
        ge_p3 pt, q; if (!load_point(pt, points + 32 * j)) return 0;
        blind(q, pt);
        ge_pniels pn; ge_p3_to_pniels(pn, q);
        ge_pniels_packed pk; ge_pniels_pack(pk, pn);
        ge64_pniels pn64; ge64_pniels_unpack(pn64, pk);
        ge64_p3 A; ge64_identity(A);
        ge64_padd(A, A, pn64, 0u);                                     // as k_straus_prepare does
        straus_table5(&tables[(size_t)8 * j], A);
    }
    const BatchPiece &pc = plan.pieces[0];
    const size_t ntasks = pc.tasks.size();
    std::vector<ge_p3> partial(ntasks ? ntasks : 1);
    for (size_t w = 0; w < (ntasks + 7) / 8; w++) {
        std::vector<uint8_t> agree(32, 1);
        std::vector<uint32_t> words(32 * 8);
        run_warp([&](uint32_t lane) {
            const size_t t = 8 * w + (lane >> 2);
            const bool live = t < ntasks;
            const BatchTask tk = pc.tasks[live ? t : 0];
            w4f_point Q;
            straus_task_group(Q, nafs.data(), tables.data(), tk.pair, tk.len, live, lane & 3);
            ge_p3 o; w4f_to_p3(o, Q);
            uint32_t c[8]; ge_compress(c, o);
            memcpy(&words[8 * lane], c, 32);
            if (live && (lane & 3) == 0) partial[t] = o;
        });
        for (uint32_t l = 0; l < 32; l++) if (memcmp(&words[8 * l], &words[8 * (l & ~3u)], 32)) return -2;   // replicated in the group
    }
    for (size_t k = 0; k < m; k++) {
        const BatchSum s = pc.sums[k];
        ge_p3 acc; ge_p3_identity(acc);
        for (uint32_t t = s.off; t < s.off + s.len; t++) ge_add(acc, acc, partial[t]);
        store_point(out + 32 * k, acc);
    }
    return 1;
}

}  // extern "C"
