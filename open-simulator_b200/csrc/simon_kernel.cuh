// simon_kernel.cuh — persistent thread-block-cluster placement kernel (sm_100a): shared declarations.
//
// One scenario = one thread-block cluster (up to 16 CTAs, DSMEM).  Every node of the scenario is owned by
// one thread slot for the whole kernel; its static columns, its dynamic NodeInfo aggregates and the values
// cached for the current pod class live in that CTA's shared memory, so a placement decision touches no
// global memory on its critical path: filter -> score -> cluster-wide reductions over DSMEM (st.async + mbarrier,
// no barrier.cluster) -> argmax -> commit.
//
// Semantics follow oracle/simon_oracle.c line by line (which cites the reference file:line of every
// plugin); the data layout is include/simon_gpu.h.  Integer work is exact; the float64 plugin formulas use
// IEEE double with contraction disabled (-fmad=false) and truncation by cast.
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/simon_gpu.h"

namespace cg = cooperative_groups;

#define SK_MAX_ENT 32       // list entries (ports + constraints + terms) cached per node for one class
#define SK_MAX_HARD 8
#define SK_MAX_SOFT 8
#define SK_MAX_CS 16
#define SK_MAXW 6           // domain-bitmask words available per decision
#define SK_NV 16            // max values per all-reduce
#define SK_PLW 5            // payload: up to 10 int32 packed in 5 u64 (T domains + flags); only (T + 2) / 2 of them are sent
#define SK_MAX_WARPS 16     // threads per CTA <= 512 (the shipped variants use <= 320)
#define SK_AUX_W 324          // per-class tables built at upload (SkParams::cls_aux): [0..32] compact commit list (+ count word),
                              //   [33..64] counter bases of the commit list, pad, [68..323] entry table as int32 rows [ER_ROWS][SK_MAX_ENT]
#define SK_AUX_INCB 33
#define SK_AUX_ENT 68
#define SK_CSUM_W 26          // valid, 8 sizes, 6 summary scalars, last winner: rank, ignored, 8 domains (+1 spare)

enum { EK_PORT = 0, EK_HARD, EK_SOFT, EK_AFF, EK_ANTI, EK_EXIST, EK_SCORE };
enum { ER_KIND = 0, ER_K, ER_T, ER_A, ER_B, ER_INC, ER_WOFF, ER_BASE, ER_ROWS };   // ER_BASE: offset of the counter in cnt[]

// 64-bit per-node arrays
enum { A_ALLOC_MCPU = 0, A_ALLOC_MEM, A_ALLOC_EPH, A_REQ_MCPU, A_REQ_MEM, A_REQ_EPH, A_NZ_MCPU, A_NZ_MEM, A_SIMON,
       A_INV_MCPU, A_INV_MEM, A_N64 };
// 32-bit per-node arrays (followed by T domain rows and emax cached counter rows)
enum { B_ALLOC_PODS = 0, B_NUM_PODS, B_NODE_G, B_NODE_CLASS, B_RAW_NA, B_RAW_TT, B_EXTRA, B_RAW_PTS, B_RAW_IPA, B_OWN, B_SNORM, B_N32 };
// 8-bit per-node arrays
enum { C_ST_CODE = 0, C_NFLAGS, C_REGBITS, C_N8 };

#define NF_SEL_OK 1
#define NF_IGNORED 2
#define NF_HARDKEYS 4
#define NF_COUNTED 8
#define NF_FEASIBLE 16
#define NF_VALID 32
#define NF_FIT_OK 64
#define NF_STATIC_FAIL 128

struct SkScenario {
    const uint32_t *order;     // [n_active] scenario order -> node index (nullptr: identity)
    const int32_t *rank_of;    // [N] node index -> scenario rank or -1 (nullptr: identity)
    uint32_t n_active;
    uint32_t pad;
    // dynamic state, node-indexed
    int64_t *req_mcpu, *req_mem, *req_eph, *nz_mcpu, *nz_mem, *req_scalar, *gpu_used;
    int32_t *num_pods;
    int32_t *cnt;              // counters, all domains
    int32_t *cnt_total;        // [n_counters]
    // scratch tables [SK_MAX_SOFT or SK_MAX_HARD][max_dom]
    int32_t *tp, *fcount, *size;   // size: [SK_MAX_SOFT]
    long long *csum;           // [n_classes][SK_CSUM_W] feasible-set summary per class as of its last visit
    unsigned long long *ocache; // [n_classes][N] own-state score cache: {node version (num_pods + 1):32, fit:1, own score:31}; 0 = empty
    uint8_t *fbits;            // [n_classes][N] NF_FEASIBLE|NF_COUNTED per node as of that visit (what csum is exact for)
    uint8_t *hard_reg;
    // outputs
    int32_t *out_node;         // [P]
    int64_t *out_score;        // [P] or nullptr
    uint32_t *out_gpu;         // [P] or nullptr: GPU-share devices reserved for the pod, 4 bits per device = slots taken on it
    uint32_t *fail_counts;     // [max_fail][SIMON_N_FAIL_CODES]
    uint32_t *fail_pod;        // [max_fail]
    uint32_t *n_fail;          // [1]
    uint32_t *n_sched;         // [1]
    unsigned long long *clk;   // [2] start/stop globaltimer of this cluster (optional)
};

struct SkParams {
    // snapshot
    uint32_t N, K, WL, WT, T, NC, n_log, max_dom;
    const uint32_t *topo_ndom;
    const int64_t *alloc_mcpu, *alloc_mem, *alloc_eph, *alloc_scalar;
    const int32_t *alloc_pods;
    const uint32_t *node_flags;
    const uint64_t *label_bits, *taint_hard, *taint_soft;
    const int32_t *topo_dom, *node_class, *gpu_count;
    const int64_t *gpu_dev_mem, *gpu_total_mem;
    const double *log_table;
    // pod set
    uint32_t n_classes, n_pods, n_counters, max_blob_words;
    const uint64_t *class_off;
    const int64_t *class_blob;
    const int32_t *pod_class, *pod_fixed, *pod_guard;
    const uint32_t *cls_aux;       // [n_classes][SK_AUX_W] per-class commit / entry tables (built at upload)
    const uint64_t *cnt_off;
    const int64_t *simon_raw;
    const int32_t *extra_score;
    // launch
    uint32_t first, count, max_fail, npt, emax, record_scores;
    const SkScenario *scen;    // [gridDim.x / cluster size]
    unsigned long long *stats; // optional [8]: decisions, class changes, summary rebuilds, redone decisions
    // static cache: per (static signature, node) verdicts, filled on first use
    uint32_t n_sigs, use_scache;
    uint32_t simon32, pad32;       // simon32: every raw Simon score lies in [0, 2^31) -> reduced as a 32-bit word
    unsigned char *gnode;          // large-cluster variant: per-node arrays, one slice of gnode_stride bytes per CTA
    size_t gnode_stride;
    uint32_t dump_pod, pad_d;      // debug: pod index whose per-node totals / filter reasons are written out (0xffffffff: none)
    long long *dump_total;         // [N]
    int32_t *dump_code;            // [N] 0 = feasible, else the reason bitmask
    unsigned long long *scache;    // [n_sigs][N] packed {st_code, flags, tt, 0, na:int32}
    // pod-list variants (LIST, drains): scenario s places pods list_pods[list_off[s] .. list_off[s + 1]) in that order; its
    // out_node / fail records are indexed by position in the list.  Appended last: the fields above keep their offsets.
    const uint64_t *list_off;
    const uint32_t *list_pods;
};

__host__ __device__ inline size_t sk_align(size_t x) { return (x + 15) & ~(size_t)15; }

// shared memory carve-up (per CTA).  L = npt * blockDim.x node slots.
struct SkSmem {
    int64_t *a64;        // [A_N64][L]
    int32_t *a32;        // [B_N32 + T + emax][L]
    uint8_t *a8;         // [C_N8][L]
    int64_t *blob;       // [max_blob_words]
    unsigned long long *box;     // [2][SK_NV][nslots] reduction inbox: one slot per CTA of the cluster, double buffered
    unsigned long long *wpart;   // [SK_NV][SK_MAX_WARPS] per-warp partials of the CTA-level fold (u64, or 2*SK_NV rows of u32)
    int32_t *ent;        // [ER_ROWS][SK_MAX_ENT]
    uint32_t *tnd;       // [SIMON_MAX_TOPOS] topo_ndom copy
    uint32_t *inc;       // [SK_MAX_ENT + 1] compact list of the entries the current class increments; [SK_MAX_ENT] = count
    long long *pred;     // [SK_CSUM_W] the entered class's stored summary record (one global read per CTA)
    int32_t *lastdom;    // [SIMON_MAX_TOPOS] topology domains of the last winner (single-node flip fast path)
    uint32_t *incb;      // [32] counter base offsets (cnt_off) of the first 32 entries of the class's commit list
    double *soft_w;      // [SK_MAX_SOFT] log weights of the current class's soft constraints (uniform)
    SkScenario *scen;    // this cluster's scenario descriptor
    unsigned long long *mbar;    // [2] mbarriers guarding the two inbox buffers
    uint32_t L, T, nslots;
};

// bytes of the per-node arrays of one CTA (shared memory normally; a slice of SkParams::gnode in the large-cluster variant)
__host__ __device__ inline size_t sk_node_bytes(uint32_t L, uint32_t T, uint32_t emax) {
    return sk_align(8ull * A_N64 * L) + sk_align(4ull * (B_N32 + T + emax) * L) + sk_align(1ull * C_N8 * L);
}

__host__ __device__ inline size_t sk_smem_bytes(uint32_t L, uint32_t T, uint32_t emax, uint32_t blob_words, uint32_t nslots, bool node_arrays = true) {
    size_t b = 0;
    if (node_arrays) b += sk_node_bytes(L, T, emax);
    b += sk_align(8ull * blob_words);
    b += sk_align(8ull * 2 * SK_NV * nslots) + sk_align(8ull * SK_NV * SK_MAX_WARPS);
    b += sk_align(4ull * ER_ROWS * SK_MAX_ENT);
    b += sk_align(4ull * SIMON_MAX_TOPOS) + sk_align(4ull * (SK_MAX_ENT + 1)) + sk_align(4ull * 32) + sk_align(4ull * SIMON_MAX_TOPOS) + sk_align(8ull * SK_CSUM_W);
    b += sk_align(8ull * SK_MAX_SOFT) + sk_align(sizeof(SkScenario));
    b += sk_align(8ull * 2);
    return b + 64;
}

// gnode == nullptr: everything in shared memory.  Otherwise the per-node arrays live in this CTA's slice of global memory
// (large-cluster variant: the same code, the node state served by L1 / L2 instead of shared memory).
__device__ inline void sk_carve(SkSmem &S, unsigned char *base, uint32_t L, uint32_t T, uint32_t emax, uint32_t blob_words, uint32_t nslots,
                                unsigned char *gnode = nullptr) {
    unsigned char *p = base;
    unsigned char *q = gnode ? gnode : p;
    S.a64 = (int64_t *)q; q += sk_align(8ull * A_N64 * L);
    S.a32 = (int32_t *)q; q += sk_align(4ull * (B_N32 + T + emax) * L);
    S.a8 = (uint8_t *)q; q += sk_align(1ull * C_N8 * L);
    if (!gnode) p = q;
    S.blob = (int64_t *)p; p += sk_align(8ull * blob_words);
    S.box = (unsigned long long *)p; p += sk_align(8ull * 2 * SK_NV * nslots);
    S.wpart = (unsigned long long *)p; p += sk_align(8ull * SK_NV * SK_MAX_WARPS);
    S.ent = (int32_t *)p; p += sk_align(4ull * ER_ROWS * SK_MAX_ENT);
    S.tnd = (uint32_t *)p; p += sk_align(4ull * SIMON_MAX_TOPOS);
    S.inc = (uint32_t *)p; p += sk_align(4ull * (SK_MAX_ENT + 1));
    S.incb = (uint32_t *)p; p += sk_align(4ull * 32);
    S.lastdom = (int32_t *)p; p += sk_align(4ull * SIMON_MAX_TOPOS);
    S.pred = (long long *)p; p += sk_align(8ull * SK_CSUM_W);
    S.soft_w = (double *)p; p += sk_align(8ull * SK_MAX_SOFT);
    S.scen = (SkScenario *)p; p += sk_align(sizeof(SkScenario));
    S.mbar = (unsigned long long *)p;
    S.L = L; S.T = T; S.nslots = nslots;
}

// ---------------------------------------------------------------------------------------------------------
// warp / cluster reductions on unsigned 64-bit values built from 32-bit redux.sync (one instruction per step)
enum { OP_SUM32 = 0, OP_MINU = 1, OP_MAXU = 2, OP_OR = 3 };

__device__ __forceinline__ unsigned long long sk_enc(long long x) { return (unsigned long long)x ^ 0x8000000000000000ull; }
__device__ __forceinline__ long long sk_dec(unsigned long long x) { return (long long)(x ^ 0x8000000000000000ull); }

__device__ __forceinline__ unsigned long long warp_maxu64(unsigned long long x) {
    unsigned hi = (unsigned)(x >> 32), lo = (unsigned)x;
    unsigned mh = __reduce_max_sync(0xffffffffu, hi);
    unsigned ml = __reduce_max_sync(0xffffffffu, hi == mh ? lo : 0u);
    return ((unsigned long long)mh << 32) | ml;
}
__device__ __forceinline__ unsigned long long warp_minu64(unsigned long long x) {
    unsigned hi = (unsigned)(x >> 32), lo = (unsigned)x;
    unsigned mh = __reduce_min_sync(0xffffffffu, hi);
    unsigned ml = __reduce_min_sync(0xffffffffu, hi == mh ? lo : 0xffffffffu);
    return ((unsigned long long)mh << 32) | ml;
}
__device__ __forceinline__ unsigned long long warp_oru64(unsigned long long x) {
    unsigned hi = __reduce_or_sync(0xffffffffu, (unsigned)(x >> 32));
    unsigned lo = __reduce_or_sync(0xffffffffu, (unsigned)x);
    return ((unsigned long long)hi << 32) | lo;
}
__device__ __forceinline__ unsigned long long warp_op(unsigned long long x, int op) {
    if (op == OP_SUM32) return (unsigned long long)__reduce_add_sync(0xffffffffu, (unsigned)x);
    if (op == OP_MINU) return warp_minu64(x);
    if (op == OP_MAXU) return warp_maxu64(x);
    return warp_oru64(x);
}
__device__ __forceinline__ unsigned long long sk_ident(int op) { return op == OP_MINU ? ~0ull : 0ull; }

struct SkRed {
    SkSmem *S;
    cg::cluster_group *cluster;
    uint32_t crank, CS;
    uint32_t mph;      // reduction phase counter (selects inbox buffer, mbarrier and parity)
    long long *prof;   // profiling variants: [0] cycles in the reductions' __syncthreads, [1] from there to the mbarrier release, [2] count
};

// ---------------------------------------------------------------------------------------------------------
// Cluster reductions without barrier.cluster and without __syncthreads.
//   warp redux.sync -> per-warp partials in shared memory -> ONE __syncthreads -> warp 0 folds them and its lanes
//   0..CS-1 push the CTA's partials into EVERY CTA's inbox with st.async (a DSMEM store that completes a transaction
//   on the destination's mbarrier) -> all threads wait on the LOCAL mbarrier (armed by thread 0 with the byte count
//   of all CS messages) -> every warp folds the CS partials itself.
//   (Measured on B200: sending per-warp partials directly, 128 x 16 messages, is slower than this two-level form.)
// A reduction is still an execution barrier for the cluster (nobody returns before every warp has sent), but it does
// NOT order global memory: code that exchanges data through global memory fences and uses cluster.sync() explicitly.
// Inbox buffer, mbarrier and parity alternate with the phase counter; a warp can be at most one phase ahead of any
// other warp of the cluster, so two buffers suffice.
__device__ __forceinline__ uint32_t sk_saddr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void sk_mbar_init(unsigned long long *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(sk_saddr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void sk_mbar_expect(unsigned long long *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sk_saddr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void sk_mbar_wait(unsigned long long *bar, uint32_t parity) {
    uint32_t a = sk_saddr(bar), ok = 0;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ uint32_t sk_mapa(uint32_t laddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(laddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void sk_st_async(uint32_t raddr, unsigned long long v, uint32_t rbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];" ::"r"(raddr), "l"(v), "r"(rbar) : "memory");
}
__device__ __forceinline__ unsigned long long sk_comb(unsigned long long a, unsigned long long b, int op) {
    if (op == OP_SUM32) return a + b;
    if (op == OP_MINU) return a < b ? a : b;
    if (op == OP_MAXU) return a > b ? a : b;
    return a | b;
}

// must be called once by every thread of the cluster before the first reduction
__device__ inline void sk_red_init(SkRed &R) {
    SkSmem &S = *R.S;
    if (threadIdx.x == 0) {
        sk_mbar_init(&S.mbar[0], 1);
        sk_mbar_init(&S.mbar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    R.cluster->sync();
}

// All-reduce NVAL values over the cluster; every thread returns with the reduced values in v[].
// Two levels: warps -> CTA partial through shared memory (one __syncthreads, folded by warp 0), CTA partials ->
// every CTA's inbox with st.async; all threads wait on the local mbarrier and fold the CS partials themselves.
template <int NVAL>
__device__ __forceinline__ void sk_allreduce(SkRed &R, unsigned long long (&v)[NVAL], const int (&op)[NVAL]) {
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
    SkSmem &S = *R.S;
    const uint32_t ph = R.mph, buf = ph & 1, parity = (ph >> 1) & 1, ns = S.nslots;
    if (threadIdx.x == 0) sk_mbar_expect(&S.mbar[buf], ns * NVAL * 8u);
#pragma unroll
    for (int i = 0; i < NVAL; i++) v[i] = warp_op(v[i], op[i]);
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < NVAL; i++) S.wpart[i * SK_MAX_WARPS + warp] = v[i];
    }
    __syncthreads();
    if (warp == 0) {
        unsigned long long c[NVAL];
#pragma unroll
        for (int i = 0; i < NVAL; i++) c[i] = warp_op(lane < nwarp ? S.wpart[i * SK_MAX_WARPS + lane] : sk_ident(op[i]), op[i]);
        if (lane < R.CS) {
            const uint32_t rbar = sk_mapa(sk_saddr(&S.mbar[buf]), lane);
            const uint32_t rbox = sk_mapa(sk_saddr(S.box + (size_t)buf * SK_NV * ns + R.crank), lane);
#pragma unroll
            for (int i = 0; i < NVAL; i++) sk_st_async(rbox + 8u * i * ns, c[i], rbar);
        }
    }
    sk_mbar_wait(&S.mbar[buf], parity);
    const unsigned long long *bx = S.box + (size_t)buf * SK_NV * ns;
#pragma unroll
    for (int i = 0; i < NVAL; i++) v[i] = warp_op(lane < ns ? bx[i * ns + lane] : sk_ident(op[i]), op[i]);
    R.mph++;
}

// The same all-reduce over 32-bit words (native single-instruction redux.sync per word and stage; two words per
// st.async message).  This is the form the placement loop uses: scores, counts and domain bitmasks are 32-bit.
enum { W_SUM = 0, W_MIN = 1, W_MAX = 2, W_OR = 3 };
__device__ __forceinline__ uint32_t warp_w(uint32_t x, int op) {
    if (op == W_SUM) return __reduce_add_sync(0xffffffffu, x);
    if (op == W_MIN) return __reduce_min_sync(0xffffffffu, x);
    if (op == W_MAX) return __reduce_max_sync(0xffffffffu, x);
    return __reduce_or_sync(0xffffffffu, x);
}
__device__ __forceinline__ uint32_t w_ident(int op) { return op == W_MIN ? 0xffffffffu : 0u; }
__device__ __forceinline__ uint32_t w_enc(int32_t x) { return (uint32_t)x ^ 0x80000000u; }     // order-preserving int32 -> uint32
__device__ __forceinline__ int32_t w_dec(uint32_t x) { return (int32_t)(x ^ 0x80000000u); }

template <int NW>
__device__ __forceinline__ void sk_allreduce_w(SkRed &R, uint32_t (&w)[NW], const int (&op)[NW]) {
    constexpr int NM = (NW + 1) / 2;
    static_assert(NM <= SK_NV && NW <= 2 * SK_NV, "message too long for the inbox");
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
    SkSmem &S = *R.S;
    const uint32_t ph = R.mph, buf = ph & 1, parity = (ph >> 1) & 1, ns = S.nslots;
    if (threadIdx.x == 0) sk_mbar_expect(&S.mbar[buf], ns * NM * 8u);
#pragma unroll
    for (int i = 0; i < NW; i++) w[i] = warp_w(w[i], op[i]);
    uint32_t *wp = (uint32_t *)S.wpart;
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < NW; i++) wp[i * SK_MAX_WARPS + warp] = w[i];
    }
    const long long pt0 = R.prof ? clock64() : 0;
    __syncthreads();
    const long long pt1 = R.prof ? clock64() : 0;
    if (warp == 0) {
        uint32_t c[NW];
#pragma unroll
        for (int i = 0; i < NW; i++) c[i] = warp_w(lane < nwarp ? wp[i * SK_MAX_WARPS + lane] : w_ident(op[i]), op[i]);
        if (lane < R.CS) {
            const uint32_t rbar = sk_mapa(sk_saddr(&S.mbar[buf]), lane);
            const uint32_t rbox = sk_mapa(sk_saddr(S.box + (size_t)buf * SK_NV * ns + R.crank), lane);
#pragma unroll
            for (int m = 0; m < NM; m++) {
                const uint32_t hi = 2 * m + 1 < NW ? c[2 * m + 1 < NW ? 2 * m + 1 : 0] : 0u;
                sk_st_async(rbox + 8u * m * ns, ((unsigned long long)hi << 32) | c[2 * m], rbar);
            }
        }
    }
    sk_mbar_wait(&S.mbar[buf], parity);
    if (R.prof) { R.prof[0] += pt1 - pt0; R.prof[1] += clock64() - pt1; R.prof[2] += 1; }
    const unsigned long long *bx = S.box + (size_t)buf * SK_NV * ns;
#pragma unroll
    for (int m = 0; m < NM; m++) {
        const bool in = lane < ns;
        const unsigned long long x = in ? bx[m * ns + lane] : 0ull;
        w[2 * m] = warp_w(in ? (uint32_t)x : w_ident(op[2 * m]), op[2 * m]);
        if (2 * m + 1 < NW) w[2 * m + 1 < NW ? 2 * m + 1 : 0] = warp_w(in ? (uint32_t)(x >> 32) : w_ident(op[2 * m + 1 < NW ? 2 * m + 1 : 0]), op[2 * m + 1 < NW ? 2 * m + 1 : 0]);
    }
    R.mph++;
}

// Arg-max: value 0 of the message is the key (0 = no candidate); values 1..SK_PLW carry the payload of the CTA-local
// winner (its topology domains + node flags, read from this CTA's shared memory by warp 0).  Split in two so that the
// caller can work while the messages travel: sk_argmax_send returns the WARP-level maximum of the keys,
// sk_argmax_wait the winning key; `who` addresses the winner's message for sk_wpay().
__device__ __forceinline__ unsigned long long sk_argmax_send(SkRed &R, unsigned long long key, uint32_t CT, uint32_t TPB) {
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
    SkSmem &S = *R.S;
    const uint32_t ph = R.mph, buf = ph & 1, ns = S.nslots;
    const uint32_t plw = (S.T + 2u) >> 1;          // payload rows in use: T domains + the flags word, two per message
    if (threadIdx.x == 0) sk_mbar_expect(&S.mbar[buf], ns * (1 + plw) * 8u);
    key = warp_maxu64(key);
    if (lane == 0) S.wpart[warp] = key;
    const long long pt0 = R.prof ? clock64() : 0;
    __syncthreads();
    if (R.prof) R.prof[3] += clock64() - pt0;
    if (warp == 0) {
        const unsigned long long k = warp_maxu64(lane < nwarp ? S.wpart[lane] : 0ull);
        int32_t pw = -1;
        if (k != 0) {
            uint32_t r = 0xFFFFFFu - (uint32_t)(k & 0xFFFFFFu);
            uint32_t idx = (r / CT) * TPB + (r % CT) % TPB;
            if (lane < S.T) pw = S.a32[(B_N32 + lane) * S.L + idx];
            else if (lane == S.T) pw = S.a8[C_NFLAGS * S.L + idx];
        }
        unsigned long long w[SK_PLW];
#pragma unroll
        for (int j = 0; j < SK_PLW; j++) {
            unsigned lo = (unsigned)__shfl_sync(0xffffffffu, pw, 2 * j), hi = (unsigned)__shfl_sync(0xffffffffu, pw, 2 * j + 1);
            w[j] = ((unsigned long long)hi << 32) | lo;
        }
        if (lane < R.CS) {
            const uint32_t rbar = sk_mapa(sk_saddr(&S.mbar[buf]), lane);
            const uint32_t rbox = sk_mapa(sk_saddr(S.box + (size_t)buf * SK_NV * ns + R.crank), lane);
            sk_st_async(rbox, k, rbar);
#pragma unroll
            for (int j = 0; j < SK_PLW; j++)
                if ((uint32_t)j < plw) sk_st_async(rbox + 8u * (1 + j) * ns, w[j], rbar);
        }
    }
    return key;
}
__device__ __forceinline__ unsigned long long sk_argmax_wait(SkRed &R, uint32_t &who) {
    const unsigned lane = threadIdx.x & 31;
    SkSmem &S = *R.S;
    const uint32_t ph = R.mph, buf = ph & 1, parity = (ph >> 1) & 1, ns = S.nslots;
    const long long pt1 = R.prof ? clock64() : 0;
    sk_mbar_wait(&S.mbar[buf], parity);
    if (R.prof) { R.prof[4] += clock64() - pt1; R.prof[5] += 1; }
    const unsigned long long *bx = S.box + (size_t)buf * SK_NV * ns;
    const unsigned long long y = lane < ns ? bx[lane] : 0ull;
    const unsigned long long m = warp_maxu64(y);
    who = buf * SK_NV * ns + (__ffs(__ballot_sync(0xffffffffu, y == m)) - 1);
    R.mph++;
    return m;
}
__device__ __forceinline__ unsigned long long sk_argmax(SkRed &R, unsigned long long key, uint32_t CT, uint32_t TPB, uint32_t &who) {
    sk_argmax_send(R, key, CT, TPB);
    return sk_argmax_wait(R, who);
}
// word j of the winner's payload: j < T -> domain of topology j, j == T -> node flags
__device__ __forceinline__ int32_t sk_wpay(const SkSmem &S, uint32_t who, uint32_t j) {
    return ((const int32_t *)(S.box + who + (size_t)(1 + (j >> 1)) * S.nslots))[j & 1];
}
