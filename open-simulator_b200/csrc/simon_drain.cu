// simon_drain.cu — the fork of a node-drain batch (include/simon_gpu.h, "node drains"; DESIGN.md §3.5).
//
// A drain scenario starts from the live single-scenario state, not from empty.  For a chunk of m scenarios the fork
//   1. broadcasts the live per-node columns and counters into every scenario's slot of the pooled batch buffers: each word of the
//      live state is read once and written m times (simon_drain_bcast);
//   2. takes back the counter increments of every pod that ran on one of the scenario's drained nodes (NodeInfo.RemovePod,
//      K8S/framework/types.go:539-585): one thread per (scenario, removed pod), atomics on that scenario's counters, with the
//      domain and eligibility rules of the import kernel (simon_drain_release).
// The aggregates of a drained node stay as they were: no scenario reads them (the node is not in its order).  The placement
// kernel then runs each scenario's evicted pods with the LIST variant of simon_place_body.
#include "simon_kernel.cuh"

#define SD_MAX_SEG 12

struct SdSegment {
    const uint32_t *src;   // live column (32-bit words)
    uint32_t *dst;         // slot 0 of the pooled column; slot s at dst + s * stride
    uint64_t words, stride;
};
struct SdFork {
    SdSegment seg[SD_MAX_SEG];
    uint32_t n_seg, n_scen;
};

// blockIdx.y = segment; grid-stride over its words; every word read once and stored into all n_scen slots
__global__ void __launch_bounds__(256) simon_drain_bcast(const __grid_constant__ SdFork F) {
    const SdSegment &g = F.seg[blockIdx.y];
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < g.words; w += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t v = __ldg(g.src + w);
        uint32_t *d = g.dst + w;
        #pragma unroll 4
        for (uint32_t s = 0; s < F.n_scen; s++) __stcs(d + (uint64_t)s * g.stride, v);
    }
}

// rm_pods[j] ran on node rm_node[j], a drained node of scenario rm_scen[j] (chunk-relative): release its counter increments in
// that scenario's copy.  Eligibility-restricted entries (sig >= 0) are tested as at placement time, with the pod's pin.
__global__ void __launch_bounds__(256) simon_drain_release(const __grid_constant__ SkParams P, const uint32_t *rm_pods, const int32_t *rm_node,
                                                           const uint32_t *rm_scen, uint32_t n_rm) {
    const uint32_t N = P.N;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_rm; j += gridDim.x * blockDim.x) {
        const uint32_t q = rm_pods[j], g = (uint32_t)rm_node[j];
        const SkScenario &SC = P.scen[rm_scen[j]];
        const int32_t guard = P.pod_guard[q];
        const ReqCtx RC{P.label_bits, N, guard >= 0 ? guard : -1};
        const int64_t *cw = P.class_blob + P.class_off[P.pod_class[q]];
        const int64_t *inc = cw + cw[SCW_OFF_INC];
        for (int64_t u = 0; u < cw[SCW_N_INC]; u++) {
            const int64_t k = inc[3 * u], t = inc[3 * u + 1], sig = inc[3 * u + 2];
            const int32_t d = P.topo_dom[(uint64_t)t * N + g];
            if (d < 0) continue;
            if (sig >= 0 && !elig_eval(P, sig, RC, g)) continue;
            atomicSub(&SC.cnt[P.cnt_off[k] + d], 1);
            atomicSub(&SC.cnt_total[k], 1);
        }
    }
}
