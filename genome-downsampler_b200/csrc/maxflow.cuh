// maxflow.cuh — K3: bulk-synchronous push-relabel with on-device global relabelling.
//
// Replaces push_relabel_kernel + host global_relabel + driver loop of the reference
// (quasi_mcp_cuda_max_flow_solver.cu:12-79, :101-155, :366-405) with a different design:
//   * one CTA per connected component (K4), persistent over a work counter; all state stays in
//     HBM/L2 for the whole solve, nothing goes back to the host between rounds;
//   * state is packed so a push costs few DEPENDENT memory trips (rounds are latency-bound):
//     NodeRec = one 32-byte sector per node, BundleRec = 16 bytes per bundle (graph.cuh);
//   * frontier queues staged in shared memory (first QCAP entries) with a global spill slice;
//     appends are warp-aggregated (one shared-memory atomic per coalesced group);
//   * every round is a pure function of the previous state (DESIGN.md §4): phase A pushes along
//     admissible arcs using the labels of the round start, received excess is accumulated with
//     commutative atomics in NodeRec.eadd; phase B merges it, relabels from a label SNAPSHOT and
//     builds the next frontier.  The schedule is therefore independent of thread timing and the
//     CPU oracle (oracle/gds_oracle.cpp: sync_solve_component) replays it bit-exactly;
//   * global relabel = level-synchronous reverse BFS from the sink inside the same CTA, triggered
//     by a deterministic state-only rule;
//   * source arcs are consumed by the preflow (initial excess), the sink is implicit (snk).
//     On this network every active node always has a residual path to the sink (SURVEY App. A.1),
//     so no excess ever has to return to the source.
#pragma once
#include <cooperative_groups.h>

#include "common.cuh"
#include "graph.cuh"

namespace gds {
namespace cg = cooperative_groups;

// Launch shapes of the same kernel (the schedule does not depend on the thread count).  Every
// round is latency-bound with a small frontier, so throughput comes from running ALL components
// concurrently: the host picks the widest CTA whose resident count (CTAs/SM x 148) still covers
// the number of components; beyond 8 CTAs/SM the work counter hands out the rest in waves.
//   1024 threads x 1/SM (4096-entry staged queues) ... 128 threads x 8/SM (1024-entry queues)
struct MfShape {
    int threads, ctas_per_sm;
    uint32_t qcap;
};
constexpr MfShape kMfShapes[4] = {{1024, 1, 4096}, {512, 2, 2048}, {256, 4, 1024}, {128, 8, 1024}};

struct MfGraph {
    NodeRec* node;           // [n_nodes + 1] (sentinel closes the CSR ranges)
    uint32_t* d_snap;        // [n_nodes] label snapshot read by relabels
    BundleRec* bund;         // [B] sorted by (start node, key)
    const uint32_t* in_bid;  // [B] bundle ids ordered by (end node, bundle id)
    const uint32_t* in_src;  // [B] start node of in_bid[k]: the first relabel needs nothing else
    const int32_t* dem;      // [n_nodes] demand: the initial excess / sink capacity come from it
    const uint32_t* in1;     // [n_nodes] start node of a node's ONLY in-arc, kIn1None without in-arcs,
                             // kIn1Multi with several: one trip less per level of the first relabel
};
constexpr uint32_t kIn1None = 0xffffffffu, kIn1Multi = 0xfffffffeu;

struct SolveParams {
    uint32_t gr_interval_min, gr_levels_pct, gr_relabel_pct, max_rounds;
};

// Sums / maxima over the components of one call, accumulated on the device so that the host needs
// no per-component readback (gds_result's counters come from here).
struct MfTotals {
    unsigned long long rounds_total, rounds_max, pushes, relabels, grs, bfs_levels, max_frontier;
    long long sink_flow, stuck;
    unsigned long long n_solved;
};
__device__ __forceinline__ void mf_totals_add(MfTotals* T, unsigned long long rounds,
                                              unsigned long long pushes, unsigned long long relabels,
                                              unsigned long long grs, unsigned long long bfs_levels,
                                              unsigned long long max_frontier, long long sink_flow,
                                              long long stuck) {
    atomicAdd(&T->rounds_total, rounds);
    atomicMax(&T->rounds_max, rounds);
    atomicAdd(&T->pushes, pushes);
    atomicAdd(&T->relabels, relabels);
    atomicAdd(&T->grs, grs);
    atomicAdd(&T->bfs_levels, bfs_levels);
    atomicMax(&T->max_frontier, max_frontier);
    atomicAdd(reinterpret_cast<unsigned long long*>(&T->sink_flow), (unsigned long long)sink_flow);
    atomicAdd(reinterpret_cast<unsigned long long*>(&T->stuck), (unsigned long long)stuck);
    atomicAdd(&T->n_solved, 1ull);
}

struct CompStats {
    unsigned long long rounds, pushes, relabels, grs, bfs_levels, max_frontier;
    long long sink_flow, stuck;
    unsigned long long cycles, frontier_sum;  // diagnostics: SM clocks spent, sum of frontier sizes
    // diagnostics: clocks of the first global relabel's label reset, its BFS levels, its snapshot
    // copy, and of the initial frontier scan
    unsigned long long cyc_gr_init, cyc_gr_bfs, cyc_gr_snap, cyc_front, cyc_gr_later;
};

// Record loads.  A component is owned by ONE CTA, i.e. one SM: plain (L1-allocating) loads are
// coherent with the stores and atomics of the other threads of the CTA across __syncthreads, and
// measured faster than L2-only loads (__ldcg).
__device__ __forceinline__ void ld_node(const NodeRec* p, uint4& lo, uint4& hi) {
    const uint4* q = reinterpret_cast<const uint4*>(p);
    lo = q[0];  // d, stamp, e, eadd
    hi = q[1];  // snk, g, out_ptr, in_ptr
}
__device__ __forceinline__ uint4 ld_bundle(const BundleRec* p) {  // t, mult, f, s
    return *reinterpret_cast<const uint4*>(p);
}
__device__ __forceinline__ uint32_t ld_u32(const uint32_t* p) { return *p; }

template <uint32_t QCAP>
struct Queue {
    uint32_t* sm;  // QCAP entries in shared memory
    uint32_t* gl;  // global spill (indexed by the same position)
    __device__ __forceinline__ uint32_t get(uint32_t i) const { return i < QCAP ? sm[i] : gl[i]; }
    __device__ __forceinline__ void put(uint32_t i, uint32_t v) const {
        if (i < QCAP) sm[i] = v;
        else gl[i] = v;
    }
};

// warp-aggregated append from divergent code
template <uint32_t QCAP>
__device__ __forceinline__ void q_append(const Queue<QCAP>& q, uint32_t* count, uint32_t v) {
    auto g = cg::coalesced_threads();
    uint32_t base = 0;
    if (g.thread_rank() == 0) base = atomicAdd(count, g.size());
    base = g.shfl(base, 0);
    q.put(base + g.thread_rank(), v);
}

template <uint32_t QCAP>
struct MfShared {
    uint32_t qa[QCAP], qb[QCAP], qc[QCAP], qd[QCAP];
    uint32_t nF, nT, nN, nH;
    uint32_t lc[3];  // rotating level counters of the first global relabel
    uint32_t relabels_since;
    uint32_t comp;
    unsigned long long pushes, relabels;
    long long sink_flow, stuck;
};

// Nodes with more than kHeavyDeg incident bundles are not walked by one thread (a serial chain of
// dependent loads per bundle — variable read lengths give tens of bundles per node): the thread
// pass puts them on the heavy list H and a second pass gives each a whole WARP, 32 bundles per
// trip.  Semantics are unchanged: the sequential "push until the excess is gone" over the bundles
// in their fixed order is an exclusive prefix sum of the admissible residuals across the lanes.
constexpr uint32_t kHeavyDeg = 6;

__device__ __forceinline__ uint32_t warp_excl_sum(uint32_t v, uint32_t& total) {
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if ((int)lane_id() >= o) incl += t;
    }
    total = __shfl_sync(0xffffffffu, incl, 31);
    return incl - v;
}

// reverse BFS from the sink; T/N are used as the level queues.  returns the level counter.
// Three rotating level counters (this level / next level / being reset) leave one barrier per
// level; the label snapshot is written when a node is labelled.
// 16-bit claim of an unlabelled node in the shared-memory label array (two labels per word)
__device__ __forceinline__ bool mf_claim16(uint16_t* lab, uint32_t idx, uint32_t nl) {
    uint32_t* word = reinterpret_cast<uint32_t*>(lab) + (idx >> 1);
    const uint32_t sh16 = (idx & 1u) * 16;
    for (;;) {
        const uint32_t old = *reinterpret_cast<volatile uint32_t*>(word);
        if (((old >> sh16) & 0xffffu) != 0xffffu) return false;
        const uint32_t want = (old & ~(0xffffu << sh16)) | (nl << sh16);
        if (atomicCAS(word, old, want) == old) return true;
    }
}

template <int THREADS, uint32_t QCAP, bool LAB>
__device__ uint32_t mf_global_relabel(const MfGraph& G, uint32_t lo, uint32_t hi, Queue<QCAP> T,
                                      Queue<QCAP> N, Queue<QCAP> H, MfShared<QCAP>& sh,
                                      unsigned long long& bfs_levels, bool warp_mode,
                                      uint16_t* lab /* LAB: [hi-lo+1] shared-memory labels */) {
    const uint32_t tid = threadIdx.x;
    if (tid == 0) {
        sh.lc[0] = 0;
        sh.lc[1] = 0;
        sh.lc[2] = 0;
        sh.nH = 0;
    }
    if (LAB) {
        uint32_t* lab32 = reinterpret_cast<uint32_t*>(lab);
        for (uint32_t i = tid; i < (hi - lo + 2) / 2; i += THREADS) lab32[i] = 0xffffffffu;
    }
    __syncthreads();
    for (uint32_t v = lo + tid; v <= hi; v += THREADS) {
        const bool is_sink = (int32_t)ld_u32(reinterpret_cast<const uint32_t*>(&G.node[v].snk)) > 0;
        if (LAB) {
            if (is_sink) lab[v - lo] = 1;
        } else {
            G.node[v].d = is_sink ? 1u : kLabelInf;
            G.d_snap[v] = is_sink ? 1u : kLabelInf;
        }
        if (is_sink) q_append(T, &sh.lc[0], v);
    }
    __syncthreads();
    uint32_t level = 1;
    for (;;) {
        const uint32_t cnt = sh.lc[(level - 1) % 3];
        if (cnt == 0) break;
        ++bfs_levels;
        const uint32_t nl = level + 1;
        uint32_t* nxt = &sh.lc[level % 3];
        if (tid == 0) sh.lc[(level + 1) % 3] = 0;  // last level's counter: everyone has read it
        auto visit = [&](uint32_t u) {
            if constexpr (LAB) {
                if (mf_claim16(lab, u - lo, nl)) q_append(N, nxt, u);
            } else {
                if (atomicCAS(&G.node[u].d, kLabelInf, nl) == kLabelInf) {
                    G.d_snap[u] = nl;
                    q_append(N, nxt, u);
                }
            }
        };
        for (uint32_t i = tid; i < cnt && !warp_mode; i += THREADS) {
            const uint32_t w = T.get(i);
            uint4 lo4, hi4;
            ld_node(&G.node[w], lo4, hi4);
            // CSR range ends live in the next record (w + 1 <= n_nodes: the sentinel exists)
            const uint4 nx_hi = *(reinterpret_cast<const uint4*>(&G.node[w + 1]) + 1);
            if (w < hi) visit(w + 1);                              // back arc (w+1) -> w: residual
            if (w > lo && (int32_t)hi4.y > 0) visit(w - 1);        // reverse of back arc w -> w-1
            if ((nx_hi.w - hi4.w) + (nx_hi.z - hi4.z) > kHeavyDeg) {
                q_append(H, &sh.nH, w);  // bundles of a heavy node: warp pass below
                continue;
            }
            for (uint32_t k = hi4.w, ke = nx_hi.w; k < ke; ++k) {  // bundles s -> w with residual
                const uint4 b = ld_bundle(&G.bund[ld_u32(&G.in_bid[k])]);
                if (b.z < b.y) visit(b.w);
            }
            for (uint32_t b = hi4.z, be = nx_hi.z; b < be; ++b) {  // reverse arcs t -> w
                const uint4 r = ld_bundle(&G.bund[b]);
                if (r.z > 0) visit(r.x);
            }
        }
        if (!warp_mode) __syncthreads();
        const uint32_t nH = warp_mode ? cnt : sh.nH;  // uniform
        if (nH) {
            const uint32_t lane = lane_id();
            for (uint32_t h = tid >> 5; h < nH; h += THREADS / 32) {
                const uint32_t w = warp_mode ? T.get(h) : H.get(h);
                const uint4 hi4 = *(reinterpret_cast<const uint4*>(&G.node[w]) + 1);
                const uint4 nx_hi = *(reinterpret_cast<const uint4*>(&G.node[w + 1]) + 1);
                if (warp_mode && lane == 0) {  // the thread pass was skipped: neighbours here
                    if (w < hi) visit(w + 1);
                    if (w > lo && (int32_t)hi4.y > 0) visit(w - 1);
                }
                for (uint32_t k = hi4.w + lane; k < nx_hi.w; k += 32) {
                    const uint4 b = ld_bundle(&G.bund[ld_u32(&G.in_bid[k])]);
                    if (b.z < b.y) visit(b.w);
                }
                for (uint32_t b = hi4.z + lane; b < nx_hi.z; b += 32) {
                    const uint4 r = ld_bundle(&G.bund[b]);
                    if (r.z > 0) visit(r.x);
                }
            }
            __syncthreads();
            if (!warp_mode) {
                if (tid == 0) sh.nH = 0;
                __syncthreads();
            }
        }
        Queue<QCAP> tmp = T;
        T = N;
        N = tmp;
        ++level;
    }
    __syncthreads();
    if (LAB) {
        for (uint32_t v = lo + tid; v <= hi; v += THREADS) {
            const uint32_t d16 = lab[v - lo];
            const uint32_t d = d16 == 0xffffu ? kLabelInf : d16;
            G.node[v].d = d;
            G.d_snap[v] = d;
        }
    }
    if (tid == 0) {
        sh.nT = 0;
        sh.nN = 0;
    }
    __syncthreads();
    return level;
}

// The FIRST global relabel of a component.  No flow exists yet (f = 0, g = 0), every bundle arc
// is residual and there are no reverse arcs, all labels are still kLabelInf (k_node_finalize): the
// reverse BFS needs only the in-CSR ranges and the start node of every in-arc (in_src).  A level's
// critical path is node range -> in_src -> CAS (three dependent memory trips instead of five), the
// CAS on the right neighbour is in flight meanwhile, the label snapshot is written as nodes are
// labelled, and three rotating level counters leave ONE barrier per level.  Labels are exact BFS
// distances, so they equal what mf_global_relabel computes (and the oracle's replay).
template <int THREADS, uint32_t QCAP, bool LAB>
__device__ uint32_t mf_first_relabel(const MfGraph& G, uint32_t lo, uint32_t hi, Queue<QCAP> T,
                                     Queue<QCAP> N, Queue<QCAP> H, MfShared<QCAP>& sh,
                                     unsigned long long& bfs_levels, bool warp_mode,
                                     uint16_t* lab /* LAB: [hi-lo+1] shared-memory labels */) {
    const uint32_t tid = threadIdx.x;
    constexpr uint32_t kInf16 = 0xffffu;
    if (tid == 0) {
        sh.lc[0] = 0;
        sh.lc[1] = 0;
        sh.lc[2] = 0;
        sh.nH = 0;
    }
    if (LAB) {  // 16-bit labels of the whole component next to the SM: the CAS of a level becomes
                // a shared-memory operation (~60 cycles instead of a ~800-cycle L2 round trip)
        uint32_t* lab32 = reinterpret_cast<uint32_t*>(lab);
        for (uint32_t i = tid; i < (hi - lo + 2) / 2; i += THREADS) lab32[i] = 0xffffffffu;
    }
    __syncthreads();
    for (uint32_t v = lo + tid; v <= hi; v += THREADS) {
        if ((int32_t)ld_u32(reinterpret_cast<const uint32_t*>(&G.node[v].snk)) > 0) {
            if (LAB) {
                lab[v - lo] = 1;
            } else {
                G.node[v].d = 1u;
                G.d_snap[v] = 1u;
            }
            q_append(T, &sh.lc[0], v);
        }
    }
    __syncthreads();
    uint32_t level = 1;
    for (;;) {
        const uint32_t cnt = sh.lc[(level - 1) % 3];
        if (cnt == 0) break;
        ++bfs_levels;
        const uint32_t nl = level + 1;
        uint32_t* nxt = &sh.lc[level % 3];
        if (tid == 0) sh.lc[(level + 1) % 3] = 0;  // last level's counter: everyone has read it
        auto label = [&](uint32_t u) {
            if (!LAB) G.d_snap[u] = nl;
            q_append(N, nxt, u);
        };
        // true: u was unlabelled and now carries nl (exactly one caller wins)
        auto claim = [&](uint32_t u) -> bool {
            if constexpr (!LAB) {
                return atomicCAS(&G.node[u].d, kLabelInf, nl) == kLabelInf;
            } else {
                return mf_claim16(lab, u - lo, nl);
            }
        };
        for (uint32_t i = tid; i < cnt && !warp_mode; i += THREADS) {
            const uint32_t w = T.get(i);
            const uint32_t one = ld_u32(&G.in1[w]);  // most nodes have one in-arc: its start node
            // back arc (w+1) -> w.  Global labels: the CAS is issued here and its answer is only
            // looked at after the in-arcs, so it is in flight meanwhile
            uint32_t old_r = 0;
            bool got_r = false;
            if constexpr (LAB) got_r = w < hi && claim(w + 1);
            else if (w < hi) old_r = atomicCAS(&G.node[w + 1].d, kLabelInf, nl);
            if (one < kIn1Multi) {
                if (claim(one)) label(one);
            } else if (one == kIn1Multi) {
                const uint32_t in_lo = ld_u32(&G.node[w].in_ptr), in_hi = ld_u32(&G.node[w + 1].in_ptr);
                if (in_hi - in_lo > kHeavyDeg) {
                    q_append(H, &sh.nH, w);
                } else {
                    for (uint32_t k = in_lo; k < in_hi; ++k) {
                        const uint32_t s = ld_u32(&G.in_src[k]);
                        if (s != 0xffffffffu && claim(s)) label(s);  // (forced bundles are no arcs)
                    }
                }
            }
            if constexpr (!LAB) got_r = w < hi && old_r == kLabelInf;
            if (got_r) label(w + 1);
        }
        if (!warp_mode) __syncthreads();
        const uint32_t nH = warp_mode ? cnt : sh.nH;  // uniform
        if (nH) {  // in-arcs of heavy nodes (warp mode: of every node), one warp each
            const uint32_t lane = lane_id();
            for (uint32_t h = tid >> 5; h < nH; h += THREADS / 32) {
                const uint32_t w = warp_mode ? T.get(h) : H.get(h);
                const uint32_t in_lo = ld_u32(&G.node[w].in_ptr), in_hi = ld_u32(&G.node[w + 1].in_ptr);
                if (warp_mode && lane == 0 && w < hi && claim(w + 1)) label(w + 1);
                for (uint32_t k = in_lo + lane; k < in_hi; k += 32) {
                    const uint32_t s = ld_u32(&G.in_src[k]);
                    if (s != 0xffffffffu && claim(s)) label(s);
                }
            }
            __syncthreads();
            if (!warp_mode) {
                if (tid == 0) sh.nH = 0;
                __syncthreads();
            }
        }
        Queue<QCAP> tmp = T;
        T = N;
        N = tmp;
        ++level;
    }
    __syncthreads();
    if (LAB) {  // labels and their snapshot go to the node records in one coalesced pass
        for (uint32_t v = lo + tid; v <= hi; v += THREADS) {
            const uint32_t d16 = lab[v - lo];
            const uint32_t d = d16 == kInf16 ? kLabelInf : d16;
            G.node[v].d = d;
            G.d_snap[v] = d;
        }
    }
    if (tid == 0) {
        sh.nT = 0;
        sh.nN = 0;
    }
    __syncthreads();
    return level;
}

template <int THREADS, uint32_t QCAP, int MIN_CTAS>
__global__ void __launch_bounds__(THREADS, MIN_CTAS)
k_maxflow(MfGraph G, const uint32_t* __restrict__ comp_lo, const uint32_t* __restrict__ comp_hi,
          uint32_t* work_counter, uint32_t* qF_g, uint32_t* qT_g, uint32_t* qN_g,
          uint32_t* qH_g, SolveParams P, CompStats* __restrict__ stats,
          uint32_t lab_cap /* nodes the shared-memory label array behind MfShared holds (0: none) */,
          const uint32_t* __restrict__ comp_list /* null: all components; else the ids to solve */,
          const uint32_t* __restrict__ comp_list_n, const uint32_t* __restrict__ n_comp_dev,
          MfTotals* __restrict__ totals,
          uint16_t* __restrict__ lab_g /* [2 * n_nodes + 2]: compact 16-bit labels in GLOBAL
              memory for the relabel BFS of components whose labels get no shared memory — the BFS
              then claims 16 nodes per sector instead of one 32-byte record per node */) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    MfShared<QCAP>& sh = *reinterpret_cast<MfShared<QCAP>*>(smem_raw);
    uint16_t* lab_smem = reinterpret_cast<uint16_t*>(smem_raw + sizeof(MfShared<QCAP>));
    const uint32_t tid = threadIdx.x;
    // all components, or those k_maxflow_sm left for this kernel
    const uint32_t n_comp = comp_list ? *comp_list_n : *n_comp_dev;

    for (;;) {
        if (tid == 0) sh.comp = atomicAdd(work_counter, 1u);
        __syncthreads();
        const uint32_t ticket = sh.comp;
        if (ticket >= n_comp) break;
        const uint32_t c = comp_list ? comp_list[ticket] : ticket;
        const uint32_t lo = comp_lo[c], hi = comp_hi[c];
        const uint32_t ncomp = hi - lo + 1;
        // 16-bit labels during a relabel: shared memory when the launch has it, else the compact
        // global array (base 2*lo: 4-byte aligned, components never overlap)
        uint16_t* lab_base = lab_smem;
        uint32_t lcap = lab_cap;
        if (ncomp > lcap && ncomp < 0xfff0u) {
            lab_base = lab_g + 2 * (size_t)lo;
            lcap = 0xfff0u;
        }
        Queue<QCAP> F{sh.qa, qF_g + lo}, T{sh.qb, qT_g + lo}, N{sh.qc, qN_g + lo},
            H{sh.qd, qH_g + lo};
        if (tid == 0) {
            sh.nF = 0;
            sh.relabels_since = 0;
            sh.pushes = 0;
            sh.relabels = 0;
            sh.sink_flow = 0;
            sh.stuck = 0;
        }
        unsigned long long bfs_levels = 0, grs = 1, rounds = 0, max_frontier = 0, frontier_sum = 0;
        const long long t_begin = clock64();
        if (comp_list) {
            // components k_maxflow_sm left behind: the first half of their node records holds K2's
            // in-arc hints (graph.cuh); make it this kernel's {d, stamp, e, eadd} again
            for (uint32_t v = lo + tid; v <= hi; v += THREADS) {
                const int32_t dm = G.dem[v];
                *reinterpret_cast<uint4*>(&G.node[v]) =
                    make_uint4(kLabelInf, 0u, (uint32_t)(dm < 0 ? -dm : 0), 0u);
            }
            __syncthreads();
        }
        unsigned long long my_pushes = 0, my_relabels = 0;
        long long my_sink = 0, my_stuck = 0;
        // Components whose nodes are mostly "heavy" (variable read lengths: tens of bundles per
        // node) skip the per-thread passes: every frontier node goes straight to a warp, one pass
        // and two barriers fewer per phase.  Same schedule (the warp pass is the thread pass's
        // arithmetic spread over lanes).
        const bool warp_mode =
            2ull * (ld_u32(&G.node[hi + 1].out_ptr) - ld_u32(&G.node[lo].out_ptr)) >
            (unsigned long long)kHeavyDeg * ncomp;
        long long tparts[3] = {0, 0, 0};
        const long long t_gr = clock64();
        uint32_t last_levels =
            ncomp <= lcap
                ? mf_first_relabel<THREADS, QCAP, true>(G, lo, hi, T, N, H, sh, bfs_levels, warp_mode,
                                                        lab_base)
                : mf_first_relabel<THREADS, QCAP, false>(G, lo, hi, T, N, H, sh, bfs_levels,
                                                         warp_mode, nullptr);
        tparts[1] = clock64() - t_gr;
        const long long t_front = clock64();
        for (uint32_t v = lo + tid; v <= hi; v += THREADS) {
            if ((int32_t)ld_u32(reinterpret_cast<const uint32_t*>(&G.node[v].e)) > 0) {
                G.node[v].stamp = 1;
                q_append(F, &sh.nF, v);
            }
        }
        __syncthreads();
        const long long cyc_front = clock64() - t_front;
        uint32_t round = 0;
        unsigned long long rounds_since = 0;
        for (;;) {
            const uint32_t cntF = sh.nF;
            if (cntF == 0) break;
            if (P.max_rounds && rounds >= P.max_rounds) break;
            unsigned long long interval = (unsigned long long)last_levels * P.gr_levels_pct / 100;
            if (interval < P.gr_interval_min) interval = P.gr_interval_min;
            if (rounds_since >= interval &&
                (unsigned long long)sh.relabels_since * 100 >=
                    (unsigned long long)P.gr_relabel_pct * ncomp) {
                __syncthreads();  // everyone has read relabels_since
                last_levels = ncomp <= lcap
                                  ? mf_global_relabel<THREADS, QCAP, true>(G, lo, hi, T, N, H, sh,
                                                                           bfs_levels, warp_mode, lab_base)
                                  : mf_global_relabel<THREADS, QCAP, false>(G, lo, hi, T, N, H, sh,
                                                                            bfs_levels, warp_mode, nullptr);
                ++grs;
                if (tid == 0) sh.relabels_since = 0;
                rounds_since = 0;
                __syncthreads();
            }
            ++round;
            ++rounds;
            ++rounds_since;
            if (cntF > max_frontier) max_frontier = cntF;
            frontier_sum += cntF;

            // ---------------- phase A: pushes ----------------
            // Labels and stamps are constant during this phase (only phase B writes them); a bundle
            // flow or a back-arc flow is written only by the one node whose push/cancel is
            // admissible this round (the two directions exclude each other by their labels).
            for (uint32_t i = tid; i < cntF && !warp_mode; i += THREADS) {
                const uint32_t v = F.get(i);
                uint4 lo4, hi4, r_lo, r_hi;
                ld_node(&G.node[v], lo4, hi4);
                ld_node(&G.node[v + 1], r_lo, r_hi);  // neighbours' sectors come with the own one
                const uint4 l_lo = v > lo ? *reinterpret_cast<const uint4*>(&G.node[v - 1])
                                          : make_uint4(kLabelInf, 0, 0, 0);  // d, stamp of v-1
                const uint32_t dv = lo4.x;
                G.d_snap[v] = dv;  // re-sync the snapshot of a node relabelled last round
                if (dv >= kLabelInf) continue;
                if ((r_hi.z - hi4.z) + (r_hi.w - hi4.w) > kHeavyDeg) {
                    q_append(H, &sh.nH, v);  // many bundles: a whole warp takes it below
                    continue;
                }
                int32_t ex = (int32_t)lo4.z;
                auto give = [&](uint32_t w, int32_t dl, uint32_t w_stamp) {
                    // eadd is 0 between rounds and every delta is positive: the first giver of the
                    // round sees 0 and queues w, unless w is already in the frontier
                    const int32_t old = atomicAdd(&G.node[w].eadd, dl);
                    if (old == 0 && w_stamp != round) q_append(T, &sh.nT, w);
                    ++my_pushes;
                };
                if (dv == 1) {  // 1. sink arc
                    const int32_t s = (int32_t)hi4.x;
                    if (s > 0) {
                        const int32_t dl = min(ex, s);
                        G.node[v].snk = s - dl;
                        ex -= dl;
                        my_sink += dl;
                        ++my_pushes;
                    }
                }
                // 2. own bundles, farthest end first
                {
                    const uint32_t ob = hi4.z;
                    for (uint32_t b = r_hi.z; ex > 0 && b-- > ob;) {
                        const uint4 br = ld_bundle(&G.bund[b]);
                        const uint32_t r = br.y - br.z;
                        if (r == 0) continue;
                        const uint32_t td = ld_u32(&G.node[br.x].d);
                        const uint32_t tstamp = ld_u32(&G.node[br.x].stamp);
                        if (td + 1 != dv) continue;
                        const int32_t dl = (int32_t)min((uint32_t)ex, r);
                        G.bund[b].f = br.z + dl;
                        ex -= dl;
                        give(br.x, dl, tstamp);
                    }
                }
                // 3. cancel back-flow towards the right neighbour
                if (ex > 0 && v < hi && r_lo.x + 1 == dv) {
                    const int32_t gr = (int32_t)r_hi.y;
                    if (gr > 0) {
                        const int32_t dl = min(ex, gr);
                        G.node[v + 1].g = gr - dl;
                        ex -= dl;
                        give(v + 1, dl, r_lo.y);
                    }
                }
                // 4. back arc to the left neighbour (infinite capacity)
                if (ex > 0 && v > lo && l_lo.x + 1 == dv) {
                    G.node[v].g = (int32_t)hi4.y + ex;
                    give(v - 1, ex, l_lo.y);
                    ex = 0;
                }
                // 5. cancel flow on incoming bundles, nearest start first
                if (ex > 0) {
                    const uint32_t ib = hi4.w;
                    for (uint32_t k = r_hi.w; ex > 0 && k-- > ib;) {
                        const uint32_t b = ld_u32(&G.in_bid[k]);
                        const uint4 br = ld_bundle(&G.bund[b]);
                        if (br.z == 0) continue;
                        const uint32_t sd = ld_u32(&G.node[br.w].d);
                        const uint32_t sstamp = ld_u32(&G.node[br.w].stamp);
                        if (sd + 1 != dv) continue;
                        const int32_t dl = (int32_t)min((uint32_t)ex, br.z);
                        G.bund[b].f = br.z - dl;
                        ex -= dl;
                        give(br.w, dl, sstamp);
                    }
                }
                G.node[v].e = ex;
            }
            if (!warp_mode) __syncthreads();
            const uint32_t nHA = warp_mode ? cntF : sh.nH;  // uniform
            if (nHA) {  // ---- heavy nodes (warp mode: the whole frontier), one warp each
                const uint32_t nH = nHA, lane = lane_id();
                for (uint32_t h = tid >> 5; h < nH; h += THREADS / 32) {
                    const uint32_t v = warp_mode ? F.get(h) : H.get(h);
                    uint4 lo4, hi4, r_lo, r_hi;  // every lane loads the same sectors (broadcast)
                    ld_node(&G.node[v], lo4, hi4);
                    ld_node(&G.node[v + 1], r_lo, r_hi);
                    const uint4 l_lo = v > lo ? *reinterpret_cast<const uint4*>(&G.node[v - 1])
                                              : make_uint4(kLabelInf, 0, 0, 0);
                    const uint32_t dv = lo4.x;
                    if (warp_mode) {  // what the skipped thread pass does first
                        if (lane == 0) G.d_snap[v] = dv;
                        if (dv >= kLabelInf) continue;
                    }
                    int32_t ex = (int32_t)lo4.z;  // uniform across the warp throughout
                    auto give = [&](uint32_t w, int32_t dl, uint32_t w_stamp) {
                        const int32_t old = atomicAdd(&G.node[w].eadd, dl);
                        if (old == 0 && w_stamp != round) q_append(T, &sh.nT, w);
                        ++my_pushes;
                    };
                    if (dv == 1) {  // 1. sink arc
                        const int32_t sk = (int32_t)hi4.x;
                        if (sk > 0) {
                            const int32_t dl = min(ex, sk);
                            ex -= dl;
                            if (lane == 0) {
                                G.node[v].snk = sk - dl;
                                my_sink += dl;
                                ++my_pushes;
                            }
                        }
                    }
                    // 2. own bundles, farthest end first: lane i looks at bundle (top - 1 - i);
                    // "push until the excess is gone" = exclusive prefix sum of the residuals
                    for (uint32_t top = r_hi.z; ex > 0 && top > hi4.z;
                         top = top - hi4.z > 32 ? top - 32 : hi4.z) {
                        const bool have = top - hi4.z > lane;
                        const uint32_t b = top - 1 - lane;
                        uint4 br = make_uint4(0, 0, 0, 0);
                        uint32_t r = 0, tstamp = 0;
                        if (have) {
                            br = ld_bundle(&G.bund[b]);
                            r = br.y - br.z;
                            if (r) {
                                const uint32_t td = ld_u32(&G.node[br.x].d);
                                tstamp = ld_u32(&G.node[br.x].stamp);
                                if (td + 1 != dv) r = 0;
                            }
                        }
                        uint32_t tot;
                        const uint32_t pre = warp_excl_sum(r, tot);
                        if (r && pre < (uint32_t)ex) {
                            const int32_t dl = (int32_t)min(r, (uint32_t)ex - pre);
                            G.bund[b].f = br.z + dl;
                            give(br.x, dl, tstamp);
                        }
                        ex -= (int32_t)min((uint32_t)ex, tot);
                    }
                    // 3. cancel back-flow towards the right neighbour
                    if (ex > 0 && v < hi && r_lo.x + 1 == dv) {
                        const int32_t gr = (int32_t)r_hi.y;
                        if (gr > 0) {
                            const int32_t dl = min(ex, gr);
                            ex -= dl;
                            if (lane == 0) {
                                G.node[v + 1].g = gr - dl;
                                give(v + 1, dl, r_lo.y);
                            }
                        }
                    }
                    // 4. back arc to the left neighbour (infinite capacity)
                    if (ex > 0 && v > lo && l_lo.x + 1 == dv) {
                        if (lane == 0) {
                            G.node[v].g = (int32_t)hi4.y + ex;
                            give(v - 1, ex, l_lo.y);
                        }
                        ex = 0;
                    }
                    // 5. cancel flow on incoming bundles, nearest start first
                    for (uint32_t top = r_hi.w; ex > 0 && top > hi4.w;
                         top = top - hi4.w > 32 ? top - 32 : hi4.w) {
                        const bool have = top - hi4.w > lane;
                        uint32_t b = 0, r = 0, sstamp = 0;
                        uint4 br = make_uint4(0, 0, 0, 0);
                        if (have) {
                            b = ld_u32(&G.in_bid[top - 1 - lane]);
                            br = ld_bundle(&G.bund[b]);
                            r = br.z;
                            if (r) {
                                const uint32_t sd = ld_u32(&G.node[br.w].d);
                                sstamp = ld_u32(&G.node[br.w].stamp);
                                if (sd + 1 != dv) r = 0;
                            }
                        }
                        uint32_t tot;
                        const uint32_t pre = warp_excl_sum(r, tot);
                        if (r && pre < (uint32_t)ex) {
                            const int32_t dl = (int32_t)min(r, (uint32_t)ex - pre);
                            G.bund[b].f = br.z - dl;
                            give(br.w, dl, sstamp);
                        }
                        ex -= (int32_t)min((uint32_t)ex, tot);
                    }
                    if (lane == 0) G.node[v].e = ex;
                }
                __syncthreads();
                if (!warp_mode) {
                    if (tid == 0) sh.nH = 0;
                    __syncthreads();
                }
            }
            const uint32_t cntT = sh.nT;

            // ---------------- phase B: merge, relabel from snapshot, next frontier ----------------
            for (uint32_t i = tid; i < cntF + cntT; i += THREADS) {
                const bool in_front = i < cntF;
                const uint32_t w = in_front ? F.get(i) : T.get(i - cntF);
                uint4 lo4, hi4;
                ld_node(&G.node[w], lo4, hi4);
                const int32_t left = (int32_t)lo4.z;
                const uint32_t dw = lo4.x;
                bool frozen = dw >= kLabelInf;
                if (in_front && left > 0 && !frozen) {
                    const uint4 r_hi = *(reinterpret_cast<const uint4*>(&G.node[w + 1]) + 1);
                    if ((r_hi.z - hi4.z) + (r_hi.w - hi4.w) > kHeavyDeg) {
                        q_append(H, &sh.nH, w);  // the min over many bundles: warp pass below
                    } else {
                        uint32_t mn = kLabelInf;
                        if ((int32_t)hi4.x > 0) mn = 0;
                        for (uint32_t b = hi4.z, be = r_hi.z; b < be; ++b) {
                            const uint4 br = ld_bundle(&G.bund[b]);
                            if (br.z < br.y) mn = min(mn, ld_u32(&G.d_snap[br.x]));
                        }
                        if (w < hi && (int32_t)r_hi.y > 0) mn = min(mn, ld_u32(&G.d_snap[w + 1]));
                        if (w > lo) mn = min(mn, ld_u32(&G.d_snap[w - 1]));
                        for (uint32_t k = hi4.w, ke = r_hi.w; k < ke; ++k) {
                            const uint4 br = ld_bundle(&G.bund[ld_u32(&G.in_bid[k])]);
                            if (br.z > 0) mn = min(mn, ld_u32(&G.d_snap[br.w]));
                        }
                        G.node[w].d = mn >= kLabelInf ? kLabelInf : mn + 1;
                    }
                    ++my_relabels;
                    atomicAdd(&sh.relabels_since, 1u);
                    frozen = false;  // stays queued one more round so its snapshot is re-synced
                }
                const int32_t tot = left + (int32_t)lo4.w;
                // e and eadd in one 8-byte store (no atomics are in flight in this phase)
                *reinterpret_cast<int2*>(&G.node[w].e) = make_int2(tot, 0);
                if (tot > 0) {
                    if (frozen) {
                        my_stuck += tot;
                    } else {
                        G.node[w].stamp = round + 1;
                        q_append(N, &sh.nN, w);
                    }
                }
            }
            __syncthreads();
            if (sh.nH) {  // ---- relabels of heavy nodes, one warp each (labels come from d_snap,
                          //      bundle flows and g are not written in this phase)
                const uint32_t nH = sh.nH, lane = lane_id();
                for (uint32_t h = tid >> 5; h < nH; h += THREADS / 32) {
                    const uint32_t w = H.get(h);
                    const uint4 hi4 = *(reinterpret_cast<const uint4*>(&G.node[w]) + 1);
                    const uint4 r_hi = *(reinterpret_cast<const uint4*>(&G.node[w + 1]) + 1);
                    uint32_t mn = kLabelInf;
                    if ((int32_t)hi4.x > 0) mn = 0;
                    for (uint32_t b = hi4.z + lane; b < r_hi.z; b += 32) {
                        const uint4 br = ld_bundle(&G.bund[b]);
                        if (br.z < br.y) mn = min(mn, ld_u32(&G.d_snap[br.x]));
                    }
                    if (w < hi && (int32_t)r_hi.y > 0) mn = min(mn, ld_u32(&G.d_snap[w + 1]));
                    if (w > lo) mn = min(mn, ld_u32(&G.d_snap[w - 1]));
                    for (uint32_t k = hi4.w + lane; k < r_hi.w; k += 32) {
                        const uint4 br = ld_bundle(&G.bund[ld_u32(&G.in_bid[k])]);
                        if (br.z > 0) mn = min(mn, ld_u32(&G.d_snap[br.w]));
                    }
                    mn = __reduce_min_sync(0xffffffffu, mn);
                    if (lane == 0) G.node[w].d = mn >= kLabelInf ? kLabelInf : mn + 1;
                }
                __syncthreads();
                if (tid == 0) sh.nH = 0;
            }
            {
                Queue<QCAP> tmp = F;
                F = N;
                N = tmp;
            }
            const uint32_t nn = sh.nN;
            __syncthreads();
            if (tid == 0) {
                sh.nF = nn;
                sh.nN = 0;
                sh.nT = 0;
            }
            __syncthreads();
        }
        // ---- per-component statistics ----
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            my_pushes += __shfl_xor_sync(0xffffffffu, my_pushes, o);
            my_relabels += __shfl_xor_sync(0xffffffffu, my_relabels, o);
            my_sink += __shfl_xor_sync(0xffffffffu, my_sink, o);
            my_stuck += __shfl_xor_sync(0xffffffffu, my_stuck, o);
        }
        if (lane_id() == 0) {
            atomicAdd(&sh.pushes, my_pushes);
            atomicAdd(&sh.relabels, my_relabels);
            atomicAdd((unsigned long long*)&sh.sink_flow, (unsigned long long)my_sink);
            atomicAdd((unsigned long long*)&sh.stuck, (unsigned long long)my_stuck);
        }
        __syncthreads();
        if (tid == 0) mf_totals_add(totals, rounds, sh.pushes, sh.relabels, grs, bfs_levels, max_frontier,
                                    sh.sink_flow, sh.stuck);
        if (tid == 0 && stats) {  // per-component records: diagnostics only (GDS_DUMP_COMP)
            CompStats cs;
            cs.rounds = rounds;
            cs.pushes = sh.pushes;
            cs.relabels = sh.relabels;
            cs.grs = grs;
            cs.bfs_levels = bfs_levels;
            cs.max_frontier = max_frontier;
            cs.sink_flow = sh.sink_flow;
            cs.stuck = sh.stuck;
            cs.cycles = (unsigned long long)(clock64() - t_begin);
            cs.frontier_sum = frontier_sum;
            cs.cyc_gr_init = (unsigned long long)tparts[0];
            cs.cyc_gr_bfs = (unsigned long long)tparts[1];
            cs.cyc_gr_snap = (unsigned long long)tparts[2];
            cs.cyc_front = (unsigned long long)cyc_front;
            cs.cyc_gr_later = 0;
            stats[c] = cs;
        }
        __syncthreads();
    }
}

}  // namespace gds
