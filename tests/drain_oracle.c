/*
 * drain_oracle.c — CPU restatement of node drains (include/simon_gpu.h, "node drains"): the checker of simon_drain_run.
 *
 * TEST INFRASTRUCTURE ONLY.  It builds on the unchanged CPU oracle (oracle/simon_oracle.c, included below, so the drain uses the
 * very schedule_one / commit the oracle pins) and adds one entry point, simon_oracle_drain.  tests/drain_oracle.py compiles this
 * file into a shared library of its own (a temporary directory) and binds it.
 */
#include "../oracle/simon_oracle.c"


/* ---------------------------------------------------------------------------------------------------------------
 * Node drain (include/simon_gpu.h, "node drains"): the checker of simon_drain_run, restated from the definition alone.  The
 * reference has the use case (README.md:16) and the primitives - NodeInfo.RemovePod (K8S/framework/types.go:539-585) for the pods
 * of the removed nodes and nodeTree.removeNode (K8S/internal/cache/node_tree.go:70-100) for the node order, which the caller passes
 * as `survivors` - but no implementation.  On the oracle's current state (the live run: every pod placed, placement[p] = its node):
 *   1. every pod on a drained node (not in survivors) is classified: DaemonSet pod (pinned class or guard node) -> counts[3],
 *      pre-bound pod (pod_fixed_node >= 0) -> counts[4], else evicted -> counts[0]; all of them give their counter increments back
 *      (the oracle keeps only the sig < 0 entries, see commit());
 *   2. the node set becomes `survivors` in that order, and the evicted pods are scheduled again in ascending pod index, each
 *      through schedule_one + commit with GPU-share Reserve: out_pod / out_node / out_fail_counts per evicted pod (failure
 *      histogram zero for placed pods), counts[1] placed, counts[2] unschedulable;
 *   3. out_sums = satisfyResourceSetting's sums over the survivors (req_mcpu, alloc_mcpu, req_mem, alloc_mem);
 *   4. the dynamic state and the active node set are restored: a drain is a what-if.
 * The output arrays hold up to n_pods entries. */
int simon_oracle_drain(simon_oracle *o, const int32_t *placement, const uint32_t *survivors, uint32_t n_surv, uint32_t *out_counts,
                       uint32_t *out_pod, int32_t *out_node, uint32_t *out_fail_counts, int64_t *out_sums) {
    const uint32_t N = o->N, P = o->p.n_pods;
    const uint32_t K = o->s.n_scalars ? o->s.n_scalars : 1;
    const uint64_t cw_words = o->cnt_off[o->p.n_counters];
    if (n_surv > N) return SIMON_ERR_INVALID;
    uint8_t *alive = (uint8_t *)calloc(N + 1, 1);
    for (uint32_t i = 0; i < n_surv; i++) {
        if (survivors[i] >= N || alive[survivors[i]]) { free(alive); return SIMON_ERR_INVALID; }
        alive[survivors[i]] = 1;
    }
    /* 1. save the dynamic state and the node set */
    int64_t *sv64[7] = {o->req_mcpu, o->req_mem, o->req_eph, o->nz_mcpu, o->nz_mem, o->req_scalar, o->gpu_used};
    const uint64_t n64[7] = {N, N, N, N, N, (uint64_t)K * N, (uint64_t)SIMON_MAX_GPU_DEV * N};
    int64_t *save64[7];
    for (int q = 0; q < 7; q++) { save64[q] = (int64_t *)malloc(8 * n64[q] + 8); memcpy(save64[q], sv64[q], 8 * n64[q]); }
    int32_t *save_np = (int32_t *)malloc(4ull * N + 4); memcpy(save_np, o->num_pods, 4ull * N);
    int32_t *save_cnt = (int32_t *)malloc(4 * cw_words + 4); memcpy(save_cnt, o->cnt, 4 * cw_words);
    int64_t *save_tot = (int64_t *)malloc(8ull * o->p.n_counters + 8); memcpy(save_tot, o->cnt_total, 8ull * o->p.n_counters);
    uint32_t *save_order = (uint32_t *)malloc(4ull * N + 4); memcpy(save_order, o->order, 4ull * N);
    uint8_t *save_active = (uint8_t *)malloc(N + 1); memcpy(save_active, o->active, N);
    const uint32_t save_na = o->n_active;
    const int64_t save_pin = o->cur_pin;
    /* 2. classify the pods of the drained nodes, release their counter increments */
    uint32_t n_ev = 0, n_daemon = 0, n_bound = 0, n_ok = 0, n_fail = 0;
    for (uint32_t p = 0; p < P; p++) {
        const int32_t a = placement[p];
        if (a < 0 || (uint32_t)a >= N || alive[a]) continue;
        const int64_t *cw = CW(o, o->p.pod_class[p]);
        int64_t guard = cw[SCW_GUARD_NODE];
        if (guard == -3) guard = o->p.pod_pin_node ? o->p.pod_pin_node[p] : -1;
        if ((cw[SCW_FLAGS] & SIMON_CLS_PINNED) || guard >= 0) n_daemon++;
        else if (o->p.pod_fixed_node[p] >= 0) n_bound++;
        else out_pod[n_ev++] = p;
        const int64_t *inc = cw + cw[SCW_OFF_INC];
        for (int64_t i = 0; i < cw[SCW_N_INC]; i++) {
            const int64_t k = inc[3 * i], t = inc[3 * i + 1], sig = inc[3 * i + 2];
            const int32_t d = dom_of(o, t, (uint32_t)a);
            if (sig >= 0 || d < 0) continue;
            o->cnt[o->cnt_off[k] + (uint32_t)d] -= 1;
            o->cnt_total[k] -= 1;
        }
    }
    /* 3. the survivors in their order; the evicted pods again, in pod order */
    simon_oracle_set_active(o, survivors, n_surv);
    int rc = SIMON_OK;
    for (uint32_t j = 0; j < n_ev; j++) {
        const uint32_t p = out_pod[j];
        const uint32_t cls = (uint32_t)o->p.pod_class[p];
        o->cur_pin = o->p.pod_pin_node ? o->p.pod_pin_node[p] : -1;
        uint32_t hist[SIMON_N_FAIL_CODES];
        int64_t score = 0;
        const int64_t g = schedule_one(o, cls, &score, hist);
        if (g == -2) { rc = SIMON_ERR_LIMIT; break; }
        if (g >= 0) { commit(o, CW(o, cls), (uint32_t)g, 1); memset(hist, 0, sizeof(hist)); n_ok++; }
        else n_fail++;
        out_node[j] = (int32_t)g;
        if (out_fail_counts) memcpy(out_fail_counts + (uint64_t)j * SIMON_N_FAIL_CODES, hist, sizeof(hist));
    }
    /* 4. sums over the survivors */
    int64_t sums[4] = {0, 0, 0, 0};
    for (uint32_t r = 0; r < n_surv; r++) {
        const uint32_t g = survivors[r];
        sums[0] += o->req_mcpu[g]; sums[1] += o->s.alloc_mcpu[g]; sums[2] += o->req_mem[g]; sums[3] += o->s.alloc_mem[g];
    }
    if (out_sums) memcpy(out_sums, sums, sizeof(sums));
    if (out_counts) { out_counts[0] = n_ev; out_counts[1] = n_ok; out_counts[2] = n_fail; out_counts[3] = n_daemon; out_counts[4] = n_bound; }
    /* 5. restore */
    for (int q = 0; q < 7; q++) { memcpy(sv64[q], save64[q], 8 * n64[q]); free(save64[q]); }
    memcpy(o->num_pods, save_np, 4ull * N); memcpy(o->cnt, save_cnt, 4 * cw_words); memcpy(o->cnt_total, save_tot, 8ull * o->p.n_counters);
    memcpy(o->order, save_order, 4ull * N); memcpy(o->active, save_active, N);
    o->n_active = save_na;
    o->cur_pin = save_pin;
    free(save_np); free(save_cnt); free(save_tot); free(save_order); free(save_active); free(alive);
    return rc;
}
