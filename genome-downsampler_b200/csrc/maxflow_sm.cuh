// maxflow_sm.cuh — K3, shared-memory-resident design (round 2).
//
// Same deterministic bulk-synchronous schedule as maxflow.cuh (DESIGN.md §4; the CPU replay is
// oracle/gds_oracle.cpp: sync_solve_component) — rounds, pushes, relabels, BFS levels and the kept
// set are bit-identical — but the state a dependent step waits on no longer lives in HBM/L2:
//
//   * one 32-bit word per node in SHARED memory: low half = 16-bit label, high half = excess
//     received during the current round.  A push is LDS (label of the target) + ATOMS (its excess);
//     the value the atomic returns tells the first giver of a round (it queues the target).  The
//     excess a node owns between rounds travels in its frontier-queue entry (excess << 16 | node),
//     so no second per-node array exists;
//   * 16-bit out-CSR row starts of the component in shared memory (when its bundle count fits):
//     node record and first bundle record are then fetched in ONE memory trip instead of two;
//   * the FIRST global relabel (no flow yet) runs entirely on shared memory: during that BFS the
//     high half of a node's word holds the start node of its only in-arc (0xffff none, 0xfffe
//     several -> in-CSR in global memory), so a level is queue -> word -> CAS with no global load;
//   * only what a push really changes stays in global memory (L2): bundle flows, back-arc flows,
//     sink capacities — written fire-and-forget, read with loads that do not depend on each other.
//
// Why not a thread-block cluster with the state spread over DSMEM (round-1 review, item 4): a
// remote shared-memory access costs ~215 cycles and cluster.sync ~380 (B300_MICROARCH.md, CGA/DSMEM
// table) against ~250 for an L2 hit and ~40 for a CTA barrier — a cluster buys capacity, not
// latency, and this kernel is a chain of ~550 dependent steps per component.  One CTA per
// component with 4-6 bytes of shared memory per node holds a 30 kb sample (180 KB) on one SM.
//
// Eligibility (checked per component inside the kernel): node count fits the shared memory of the
// launch, node ids fit 16 bits, and the component's total supply is <= 65535 (bounds every excess
// and every per-round receipt, SURVEY App. A.1: excess never exceeds the supply).  Anything else
// is put on a fallback list and solved by k_maxflow (global-memory state) right after.
#pragma once
#include "maxflow.cuh"

namespace gds {

constexpr uint32_t kInf16 = 0xffffu;
constexpr uint32_t kIn16None = 0xffffu, kIn16Multi = 0xfffeu;
constexpr uint32_t kMf2MaxNodes = 0xfff0u;  // relative node ids and in16 codes stay below 0xfffe

struct Mf2Graph {
    NodeRec* node;           // [n_nodes + 1]  {.., snk, g, out_ptr, in_ptr}: the mutable snk/g live here
    BundleRec* bund;         // [B]
    const uint32_t* in_bid;  // [B]
    const uint32_t* in_src;  // [B]
    const uint32_t* out_ptr;  // [n_nodes + 1]  SoA copies for the coalesced set-up pass
    const uint32_t* in_ptr;   // [n_nodes + 1]
    const int32_t* dem;       // [n_nodes]      demand (< 0 supply, > 0 sink capacity)
    // the express schedule (below): per-sample layout to tell segments of a cut reference from whole
    // samples; express_on = the call allows it; classic_ok = components that do not take the express
    // schedule may run here too (otherwise they go to k_maxflow)
    const VSample* vs;
    uint32_t n_samples, express_on, classic_ok;
    const uint8_t* dead;  // [n_nodes] 1 = the node has no live bundle of its own (null without express)
};

// The EXPRESS schedule (oracle/gds_oracle.cpp: express_component, sync_solve_component): in the
// distance labels a back arc v -> v-1 has length 0, every other residual arc length 1.  A segment of
// a cut reference has all its supply at its left end and all its sinks at its right end: M units
// have to spread over the read "lanes" (start modulo read length) and gather again, and changing
// lane means stepping left.  With unit-length back arcs every step is a round and a label; with
// length 0 a unit walks left past saturated nodes within ONE round (phase A, rule 4) and the relabel
// BFS has one level per read hop instead of one per hop plus one per step.  Config 4: 370 -> 165
// rounds and 290 -> 110 BFS levels per segment, no second global relabel, and the 1 400-round tail
// of the last segment is gone.  Which components take it is decided from the data alone.
constexpr uint32_t kExpressMaxNodes = 40961, kExpressEdge = 512, kExpressMinSupply = 128;

// Layout of the per-node arrays of an n-node component, in 32-bit words from `word`:
//   word[n] | inF bitmap [W] | (16-byte aligned) BFS bitmap A [W4] | saturated bits: snapshot [W4],
//   next [W4] (express schedule) | optr u16[n+1]
struct Mf2Layout {
    uint32_t W, W4, o_inF, o_A, o_B, o_Sn, o_optr, words;
};
__host__ __device__ constexpr Mf2Layout mf2_layout(uint32_t n, bool optr) {
    Mf2Layout L{};
    L.W = (n + 31u) / 32u;
    L.W4 = (L.W + 3u) & ~3u;
    L.o_inF = n;
    L.o_A = (n + L.W + 3u) & ~3u;
    L.o_B = L.o_A + L.W4;
    L.o_Sn = L.o_B + L.W4;
    L.o_optr = L.o_Sn + L.W4;
    L.words = L.o_optr + (optr ? (n + 2u) / 2u : 0u);
    return L;
}
__host__ __device__ constexpr uint32_t mf2_node_bytes(uint32_t n, bool optr) {
    return 4u * mf2_layout(n, optr).words;
}

// Global-memory accesses of this kernel name their state space: the graph pointers reach the
// non-inlined paths through a struct in shared memory, where the compiler would otherwise fall
// back to generic loads.
__device__ __forceinline__ uint4 g_ld4(const void* p) {
    uint4 v;
    asm volatile("ld.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t g_ld(const void* p) {
    uint32_t v;
    asm volatile("ld.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void g_st(void* p, uint32_t v) {
    asm volatile("st.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// fire-and-forget add (several walkers of one round may add to the same back-arc flow)
__device__ __forceinline__ void g_red_add(void* p, uint32_t v) {
    asm volatile("red.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// Shared-memory arrays are addressed by BYTE OFFSET from the dynamic shared-memory base, never by
// a pointer that went through memory: a pointer loaded from a struct is a generic pointer, and the
// compiler then emits generic loads, ATOM.E (global-path atomics) and system-scope stores for it —
// measured 5 800 clocks per BFS level instead of ~300 (profiles/r02_k3_notes.md).
__device__ __forceinline__ uint32_t* mf2_smem(uint32_t byte_off) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    return reinterpret_cast<uint32_t*>(smem_raw + byte_off);
}

struct Q2 {
    uint32_t sm_off;  // byte offset of the staged part
    uint32_t* gl;     // global spill (indexed by the same position)
    uint32_t cap;
    __device__ __forceinline__ uint32_t get(uint32_t i) const { return i < cap ? mf2_smem(sm_off)[i] : g_ld(gl + i); }
    __device__ __forceinline__ void put(uint32_t i, uint32_t v) const {
        if (i < cap) mf2_smem(sm_off)[i] = v;
        else g_st(gl + i, v);
    }
};
// One shared-memory atomic per entry (37 clocks with its return value, tools/lat_probe.cu).  The
// warp-aggregated append of maxflow.cuh costs ~190 clocks per call through cooperative groups and
// only pays when many lanes append at once; frontiers here are a handful of nodes.
__device__ __forceinline__ void q2_append(const Q2& q, uint32_t* count, uint32_t v) {
    q.put(atomicAdd(count, 1u), v);
}

__device__ __forceinline__ uint4 ld_node_hi(const NodeRec* p) {  // snk, g, out_ptr, in_ptr
    return g_ld4(reinterpret_cast<const uint4*>(p) + 1);
}
__device__ __forceinline__ uint4 ld_node_lo(const NodeRec* p) {  // in_src_last, in_bid_last, -, -
    return g_ld4(p);
}
__device__ __forceinline__ uint4 ld_bund(const BundleRec* p) { return g_ld4(p); }  // t, mult, f, s

// What the phases of one component share, in shared memory (one LDS away for every helper).
// Two rules this kernel follows, both measured (profiles/r02_k3_notes.md):
//   * NO local memory in the loops.  With the whole L1 carved out as shared memory a stack access
//     (a spill, a by-reference argument of a real call, registers saved around a call) costs a
//     trip to L2/DRAM: a BFS level whose shared-memory work is ~300 clocks took 5 700 with five
//     LDL/STL in it.  So every helper is force-inlined, counters stay in registers, and the launch
//     bound leaves the register file to the one CTA the shared memory admits anyway;
//   * each helper is expanded at ONE call site (the relabel BFS serves the first and the later
//     relabels through a flag) and inner loops are not unrolled, which keeps the code small.
struct Mf2Comp {
    Mf2Graph G;
    uint32_t lo, n, obase;
    uint32_t word_off, inF_off, bmA_off, bmB_off, optr_off;  // byte offsets (mf2_smem)
    uint32_t W4;
    uint32_t have_optr, express;
    uint32_t satn_off;  // bmB_off holds the snapshot the walkers read
    Q2 F, T, N, H;
};

struct Mf2Shared {
    uint32_t nF, nT, nN, nH;
    uint32_t relabels_since;
    uint32_t comp;
    uint32_t supply;
    uint32_t seg_sample;  // the component's sample is a cut reference (express schedule)
    uint32_t not_benign;  // a supply beyond the left edge or a sink before the right edge
    uint32_t lc[3];  // rotating level counters of the relabel BFS
    unsigned long long pushes, relabels;
    long long sink_flow, stuck;
    Mf2Comp C;
};
constexpr uint32_t kMf2HeaderBytes = (sizeof(Mf2Shared) + 15u) & ~15u;

__device__ __forceinline__ uint32_t mf2_label(const uint32_t* word, uint32_t w) { return word[w] & 0xffffu; }

// (Prefetching the records of next round's frontier nodes into L1 was tried twice: as loads nobody
// waits for — which ptxas removes, so that version never ran — and as prefetch.global.L1 (CCTL.PF1):
// config 1's phase A 2 560 -> 2 690 clocks per round, the "hole" shape 6 850 -> 7 460, config 4
// 5 640 -> 5 470.  Not kept.)
// receive dl units at node w: the first giver of the round queues w unless it is in the frontier
__device__ __forceinline__ void mf2_give(Mf2Shared& sh, uint32_t w, uint32_t dl) {
    const Mf2Comp& C = sh.C;
    const uint32_t old = atomicAdd(&mf2_smem(C.word_off)[w], dl << 16);
    if ((old >> 16) == 0 && !((mf2_smem(C.inF_off)[w >> 5] >> (w & 31)) & 1u)) {
        q2_append(C.T, &sh.nT, w);
    }
}

// express schedule, "saturated" bits: no sink capacity and no residual on any own bundle, as far as
// the three update rules know (0 is always safe).  Walkers read the snapshot of the round start
// (bmB), updates go to the next one (satn), copied over at the end of the round.
__device__ __forceinline__ void mf2_sat_set(const Mf2Comp& C, uint32_t v, bool on) {
    uint32_t* p = mf2_smem(C.satn_off) + (v >> 5);
    if (on) atomicOr(p, 1u << (v & 31));
    else atomicAnd(p, ~(1u << (v & 31)));
}
// phase A rule 4, express: ex units leave v over the chain of zero-length back arcs and stop at the
// first node that is not known to be saturated (or where the chain of equal labels ends).
__device__ __forceinline__ uint32_t mf2_walk_left(const Mf2Comp& C, uint32_t v, uint32_t ex) {
    const uint32_t* word = mf2_smem(C.word_off);
    const uint32_t* sat = mf2_smem(C.bmB_off);
    NodeRec* nr = C.G.node + C.lo;
    uint32_t u = v;
    uint32_t du = word[v] & 0xffffu;
#pragma unroll 1
    for (;;) {
        g_red_add(&nr[u].g, ex);
        --u;
        if (u == 0 || !((sat[u >> 5] >> (u & 31)) & 1u)) break;
        if ((word[u - 1] & 0xffffu) != du) break;  // (labels along the chain are all equal to du)
    }
    return u;
}

// One level of the relabel BFS: label to hand out, counter and queue of the next level.
// Queue slot a thread starts at: consecutive slots go to different WARPS (lane 0 of every warp
// first).  Frontiers are a handful of nodes whose pushes take different branches; in one warp those
// branches run one after the other, in different warps side by side (phase A of a 30 kb sample:
// 2 550 -> see profiles/r02_k3_notes.md).
template <int THREADS>
__device__ __forceinline__ uint32_t mf2_slot() {
    return (threadIdx.x & 31u) * (THREADS / 32) + (threadIdx.x >> 5);
}

struct Mf2Lvl {
    uint32_t nl;
    uint32_t* cnt;
    Q2 N;
};
// Claim node x for the next level: one ATOMS.OR on the visited bitmap (its return value decides, no
// compare-and-swap loop; a plain read first keeps already-visited nodes off the atomic unit), then
// the 16-bit label store and the queue slot.  tools/bfs_probe.cu measured this against a CAS on the
// label word (995 clocks per level of a 30 kb sample), against ballot-aggregated appends (1 150) and
// against a queue-free formulation on two bitmaps (2 340): 904.
__device__ __forceinline__ void mf2_mark(const Mf2Comp& C, const Mf2Lvl& L, uint32_t x) {
    uint32_t* vis = mf2_smem(C.bmA_off) + (x >> 5);
    const uint32_t bit = 1u << (x & 31);
    if (*vis & bit) return;
    if (atomicOr(vis, bit) & bit) return;
    reinterpret_cast<uint16_t*>(mf2_smem(C.word_off))[2 * x] = (uint16_t)L.nl;
    q2_append(L.N, L.cnt, x);
}

// ---- rarely taken paths: real functions ------------------------------------------------------

// first relabel, node u with several in-arcs: mark their start nodes (many: one warp, later)
__device__ __forceinline__ void mf2_expand_multi(Mf2Shared& sh, const Mf2Lvl& nxt, uint32_t u) {
    const Mf2Comp& C = sh.C;
    const uint32_t in_lo = g_ld(&C.G.in_ptr[C.lo + u]), in_hi = g_ld(&C.G.in_ptr[C.lo + u + 1]);
    if (in_hi - in_lo > kHeavyDeg) {
        q2_append(C.H, &sh.nH, u);
        return;
    }
    uint32_t src[kHeavyDeg];  // all loads first: one memory trip instead of one per in-arc
#pragma unroll
    for (uint32_t q = 0; q < kHeavyDeg; ++q) src[q] = in_lo + q < in_hi ? g_ld(&C.G.in_src[in_lo + q]) : 0xffffffffu;
#pragma unroll
    for (uint32_t q = 0; q < kHeavyDeg; ++q)
        if (src[q] != 0xffffffffu) mf2_mark(C, nxt, src[q] - C.lo);
}

// later relabels (flow exists), node u: residual arcs into u come from global memory
__device__ __forceinline__ void mf2_expand_flow(Mf2Shared& sh, const Mf2Lvl& nxt, uint32_t u) {
    const Mf2Comp& C = sh.C;
    const uint32_t lo = C.lo;
    const NodeRec* nr = C.G.node + lo + u;
    const uint4 lo4 = ld_node_lo(nr);
    const uint4 hi4 = ld_node_hi(nr);
    const uint4 nx = ld_node_hi(nr + 1);
    if (u > 0 && (int32_t)hi4.y > 0) mf2_mark(C, nxt, u - 1);  // reverse of back arc u -> u-1
    if ((nx.w - hi4.w) + (nx.z - hi4.z) > kHeavyDeg) {
        q2_append(C.H, &sh.nH, u);
        return;
    }
    uint4 b0 = make_uint4(0, 0, 0, 0), r0 = make_uint4(0, 0, 0, 0);
    if (nx.w > hi4.w) b0 = ld_bund(&C.G.bund[lo4.y]);  // nearest in-bundle and first out-bundle:
    if (nx.z > hi4.z) r0 = ld_bund(&C.G.bund[hi4.z]);  // fetched together
    if (nx.w > hi4.w) {  // in-bundles s -> u with residual capacity
        if (b0.z < b0.y) mf2_mark(C, nxt, lo4.x - lo);
#pragma unroll 1
        for (uint32_t k = hi4.w; k + 1 < nx.w; ++k) {
            const uint4 b2 = ld_bund(&C.G.bund[g_ld(&C.G.in_bid[k])]);
            if (b2.z < b2.y) mf2_mark(C, nxt, b2.w - lo);
        }
    }
#pragma unroll 1
    for (uint32_t b = hi4.z; b < nx.z; ++b) {  // reverse arcs t -> u (flow that can be cancelled)
        const uint4 r = b == hi4.z ? r0 : ld_bund(&C.G.bund[b]);
        if (r.z > 0) mf2_mark(C, nxt, r.x - lo);
    }
}

// relabel BFS, nodes with many arcs: one warp each.  First relabel: a warp takes up to eight of the
// level's heavy nodes at once — their in-CSR ranges in one memory trip (one lane per node), then the
// first 64 in-arcs of all eight in a second one (16 loads in flight per lane) — because a level of a
// component with variable read lengths holds ~150 nodes with ~40 in-arcs each and, taken one node
// after the other, costs two dependent trips per node (config 2: 13 600 clocks per level in k_maxflow).
template <int THREADS>
__device__ __forceinline__ void mf2_bfs_heavy(Mf2Shared& sh, const Mf2Lvl& nxt, uint32_t nH, bool first) {
    const Mf2Comp& C = sh.C;
    const uint32_t lane = lane_id(), lo = C.lo, warp = threadIdx.x >> 5;
    constexpr uint32_t NW = THREADS / 32, kBatch = 8;
    if (first) {
#pragma unroll 1
        for (uint32_t base = warp; base < nH; base += NW * kBatch) {
            // lane j < kBatch owns node (base + j * NW): its in-CSR range
            uint32_t my_lo = 0, my_hi = 0;
            if (lane < kBatch && base + lane * NW < nH) {
                const uint32_t u = C.H.get(base + lane * NW);
                my_lo = g_ld(&C.G.in_ptr[lo + u]);
                my_hi = g_ld(&C.G.in_ptr[lo + u + 1]);
            }
            uint32_t src[kBatch][2];
#pragma unroll
            for (uint32_t j = 0; j < kBatch; ++j) {
                const uint32_t in_lo = __shfl_sync(0xffffffffu, my_lo, j);
                const uint32_t in_hi = __shfl_sync(0xffffffffu, my_hi, j);
                const uint32_t k0 = in_lo + lane, k1 = k0 + 32;
                src[j][0] = k0 < in_hi ? g_ld(&C.G.in_src[k0]) : 0xffffffffu;
                src[j][1] = k1 < in_hi ? g_ld(&C.G.in_src[k1]) : 0xffffffffu;
            }
#pragma unroll
            for (uint32_t j = 0; j < kBatch; ++j) {
                if (src[j][0] != 0xffffffffu) mf2_mark(C, nxt, src[j][0] - lo);
                if (src[j][1] != 0xffffffffu) mf2_mark(C, nxt, src[j][1] - lo);
                const uint32_t in_lo = __shfl_sync(0xffffffffu, my_lo, j);
                const uint32_t in_hi = __shfl_sync(0xffffffffu, my_hi, j);
#pragma unroll 1
                for (uint32_t k = in_lo + 64 + lane; k < in_hi; k += 32)  // beyond 64 in-arcs
                {
                    const uint32_t sa = g_ld(&C.G.in_src[k]);
                    if (sa != 0xffffffffu) mf2_mark(C, nxt, sa - lo);
                }
            }
        }
        return;
    }
#pragma unroll 1
    for (uint32_t h = warp; h < nH; h += NW) {
        const uint32_t u = C.H.get(h);
        const uint4 hi4 = ld_node_hi(C.G.node + lo + u);
        const uint4 nx = ld_node_hi(C.G.node + lo + u + 1);
#pragma unroll 1
        for (uint32_t k = hi4.w + lane; k < nx.w; k += 32) {
            const uint4 b = ld_bund(&C.G.bund[g_ld(&C.G.in_bid[k])]);
            if (b.z < b.y) mf2_mark(C, nxt, b.w - lo);
        }
#pragma unroll 1
        for (uint32_t b = hi4.z + lane; b < nx.z; b += 32) {
            const uint4 r = ld_bund(&C.G.bund[b]);
            if (r.z > 0) mf2_mark(C, nxt, r.x - lo);
        }
    }
}

// phase A, nodes with many bundles, one warp each.  The sequential
// "push until the excess is gone" over the bundles in their fixed order is an exclusive prefix sum
// of the admissible residuals across the lanes (maxflow.cuh).  Memory trips per node: its records;
// then its last 64 out-bundles and the start nodes of its last 64 in-arcs together (two of each per
// lane in flight); the flow of an in-bundle only when the labels admit cancelling it.
template <int THREADS>
__device__ __forceinline__ void mf2_push_heavy(Mf2Shared& sh, uint32_t nH, unsigned long long& my_pushes,
                                            long long& my_sink) {
    const Mf2Comp& C = sh.C;
    const uint32_t lane = lane_id(), lo = C.lo, n = C.n;
    const uint32_t* word = mf2_smem(C.word_off);
#pragma unroll 1
    for (uint32_t h = threadIdx.x >> 5; h < nH; h += THREADS / 32) {
        const uint32_t i = C.H.get(h);
        const uint32_t ent = C.F.get(i);
        const uint32_t v = ent & 0xffffu;
        uint32_t ex = ent >> 16;  // uniform across the warp throughout
        const uint32_t dv = mf2_label(word, v);
        if (dv == kInf16) continue;
        NodeRec* nr = C.G.node + lo + v;
        const uint4 hi4 = ld_node_hi(nr);
        const uint4 r_hi = ld_node_hi(nr + 1);
        const uint32_t ob = hi4.z, oe = r_hi.z, ib = hi4.w, ie = r_hi.w;
        // second trip: everything the five steps may look at, at once
        uint4 pre_b[2];
        uint32_t pre_s[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const uint32_t off = lane + 32u * q;
            pre_b[q] = oe - ob > off ? ld_bund(&C.G.bund[oe - 1 - off]) : make_uint4(0, 0, 0, 0);
            pre_s[q] = ie - ib > off ? g_ld(&C.G.in_src[ie - 1 - off]) : 0xffffffffu;
        }
        const uint32_t dL = v > 0 ? mf2_label(word, v - 1) : kInf16;
        const uint32_t dR = v + 1 < n ? mf2_label(word, v + 1) : kInf16;
        int32_t snk_now = (int32_t)hi4.x;
        if (dv == 1) {  // 1. sink arc
            const int32_t sk = (int32_t)hi4.x;
            if (sk > 0) {
                const uint32_t dl = min(ex, (uint32_t)sk);
                snk_now = sk - (int32_t)dl;
                ex -= dl;
                if (lane == 0) {
                    g_st(&nr->snk, (uint32_t)(sk - (int32_t)dl));
                    my_sink += dl;
                    ++my_pushes;
                    if (C.express && snk_now == 0 && C.G.dead[lo + v]) mf2_sat_set(C, v, true);  // U4
                }
            }
        }
        // 2. own bundles, farthest end first: lane j looks at bundle (top - 1 - j)
        uint32_t chunk = 0;
#pragma unroll 1
        for (uint32_t top = oe; ex > 0 && top > ob; top = top - ob > 32 ? top - 32 : ob, ++chunk) {
            const bool have = top - ob > lane;
            const uint32_t b = top - 1 - lane;
            uint4 br = make_uint4(0, 0, 0, 0);
            uint32_t r = 0;
            if (have) {
                br = chunk == 0 ? pre_b[0] : chunk == 1 ? pre_b[1] : ld_bund(&C.G.bund[b]);
                r = br.y - br.z;
                if (r && mf2_label(word, br.x - lo) + 1 != dv) r = 0;
            }
            uint32_t tot;
            const uint32_t pre = warp_excl_sum(r, tot);
            if (r && pre < ex) {
                const uint32_t dl = min(r, ex - pre);
                g_st(&C.G.bund[b].f, br.z + dl);
                mf2_give(sh, br.x - lo, dl);
                ++my_pushes;
                if (C.express && dl == r && oe - ob == 1 && snk_now == 0) mf2_sat_set(C, v, true);  // U1
            }
            ex -= min(ex, tot);
        }
        // 3. cancel back-flow towards the right neighbour
        if (ex > 0 && v + 1 < n && dR + 1 == dv) {
            const int32_t gr = (int32_t)r_hi.y;
            if (gr > 0) {
                const uint32_t dl = min(ex, (uint32_t)gr);
                ex -= dl;
                if (lane == 0) {
                    g_st(&(nr + 1)->g, (uint32_t)(gr - (int32_t)dl));
                    mf2_give(sh, v + 1, dl);
                    ++my_pushes;
                }
            }
        }
        // 4. back arc to the left neighbour
        if (ex > 0 && v > 0 && dL + (C.express ? 0u : 1u) == dv) {
            if (lane == 0) {
                if (C.express) {
                    mf2_give(sh, mf2_walk_left(C, v, ex), ex);
                } else {
                    g_st(&nr->g, hi4.y + ex);
                    mf2_give(sh, v - 1, ex);
                }
                ++my_pushes;
            }
            ex = 0;
        }
        // 5. cancel flow on incoming bundles, nearest start first
        chunk = 0;
#pragma unroll 1
        for (uint32_t top = ie; ex > 0 && top > ib; top = top - ib > 32 ? top - 32 : ib, ++chunk) {
            const bool have = top - ib > lane;
            uint32_t b = 0, r = 0, s = 0;
            if (have) {
                const uint32_t sa = chunk == 0 ? pre_s[0] : chunk == 1 ? pre_s[1] : g_ld(&C.G.in_src[top - 1 - lane]);
                s = sa - lo;
                // (a forced bundle's slot holds no start node: it carries nothing that could be cancelled)
                if (sa != 0xffffffffu && mf2_label(word, s) + 1 == dv) {  // only then is the flow worth a memory trip
                    b = g_ld(&C.G.in_bid[top - 1 - lane]);
                    r = g_ld(&C.G.bund[b].f);
                }
            }
            uint32_t tot;
            const uint32_t pre = warp_excl_sum(r, tot);
            if (r && pre < ex) {
                const uint32_t dl = min(r, ex - pre);
                g_st(&C.G.bund[b].f, r - dl);
                mf2_give(sh, s, dl);
                ++my_pushes;
                if (C.express) mf2_sat_set(C, s, false);  // U2
            }
            ex -= min(ex, tot);
        }
        if (lane == 0) C.F.put(i, (ex << 16) | v);
    }
}

// phase B1, relabel of nodes with many bundles, one warp each: the new label waits in the high half.
// Trips: the records; the first 64 out-bundles and the ids of the first 64 in-bundles together; the
// in-bundles themselves.
template <int THREADS>
__device__ __forceinline__ void mf2_relabel_heavy(Mf2Shared& sh, uint32_t nH) {
    const Mf2Comp& C = sh.C;
    const uint32_t lane = lane_id(), lo = C.lo, n = C.n;
    uint32_t* word = mf2_smem(C.word_off);
#pragma unroll 1
    for (uint32_t h = threadIdx.x >> 5; h < nH; h += THREADS / 32) {
        const uint32_t v = C.F.get(C.H.get(h)) & 0xffffu;
        const NodeRec* nr = C.G.node + lo + v;
        const uint4 hi4 = ld_node_hi(nr);
        const uint4 r_hi = ld_node_hi(nr + 1);
        uint4 ob2[2];
        uint32_t id2[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const uint32_t b = hi4.z + lane + 32u * q, k = hi4.w + lane + 32u * q;
            ob2[q] = b < r_hi.z ? ld_bund(&C.G.bund[b]) : make_uint4(0, 0, 0, 0);
            id2[q] = k < r_hi.w ? g_ld(&C.G.in_bid[k]) : 0xffffffffu;
        }
        uint4 ib2[2];
#pragma unroll
        for (int q = 0; q < 2; ++q)
            ib2[q] = id2[q] != 0xffffffffu ? ld_bund(&C.G.bund[id2[q]]) : make_uint4(0, 0, 0, 0);
        uint32_t mn = kInf16;
        bool res_any = false;  // some own bundle has residual capacity
        if ((int32_t)hi4.x > 0) mn = 0;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            if (ob2[q].z < ob2[q].y) {  // (0,0): not taken
                mn = min(mn, mf2_label(word, ob2[q].x - lo));
                res_any = true;
            }
            if (ib2[q].z > 0) mn = min(mn, mf2_label(word, ib2[q].w - lo));
        }
#pragma unroll 1
        for (uint32_t b = hi4.z + 64 + lane; b < r_hi.z; b += 32) {
            const uint4 br = ld_bund(&C.G.bund[b]);
            if (br.z < br.y) {
                mn = min(mn, mf2_label(word, br.x - lo));
                res_any = true;
            }
        }
        if (v + 1 < n && (int32_t)r_hi.y > 0) mn = min(mn, mf2_label(word, v + 1));
        if (v > 0) mn = min(mn, mf2_label(word, v - 1) - (C.express ? 1u : 0u));  // labels are >= 1
#pragma unroll 1
        for (uint32_t k = hi4.w + 64 + lane; k < r_hi.w; k += 32) {
            const uint4 br = ld_bund(&C.G.bund[g_ld(&C.G.in_bid[k])]);
            if (br.z > 0) mn = min(mn, mf2_label(word, br.w - lo));
        }
        if (C.express) {  // U3: every own bundle has just been looked at
            const bool any = __any_sync(0xffffffffu, res_any) || (int32_t)hi4.x > 0;
            if (lane == 0) mf2_sat_set(C, v, !any);
        }
        mn = __reduce_min_sync(0xffffffffu, mn);
        const uint32_t nl = mn >= kInf16 - 1 ? kInf16 : mn + 1;
        if (lane == 0) word[v] = (nl << 16) | (word[v] & 0xffffu);
    }
}

// Reverse BFS from the sinks = global relabel, level-synchronous, labels and visited bitmap in shared
// memory, one barrier per level (three rotating level counters).  first (no flow yet): the
// in-neighbour of a node with one in-arc comes from the high half of its word (in16), so a level
// touches shared memory only; otherwise residual arcs are read from global memory.
// Precondition: sinks labelled 1, visited and queued in T with sh.lc[0] = their number.
// Returns (deepest level + 1) like the oracle's sync_global_relabel.
template <int THREADS>
__device__ __forceinline__ uint32_t mf2_bfs(Mf2Shared& sh, bool first, unsigned long long& bfs_levels) {
    const Mf2Comp& C = sh.C;
    const uint32_t tid = threadIdx.x;
    const uint32_t* word = mf2_smem(C.word_off);
    const uint32_t n = C.n;
    Q2 T = C.T, N = C.N;
    const bool express = C.express;
    uint32_t level = 1;
    for (;;) {
        uint32_t cnt = sh.lc[(level - 1) % 3];
        if (cnt == 0) break;
        ++bfs_levels;
        if (express) {
            // zero-length back arcs: the level is closed under "right neighbour" first: the run from
            // a seed to the next visited node gets the seed's label and its visited bits and joins
            // this level's queue (runs of different seeds are disjoint).  On dense data a level is
            // the previous one shifted by a read length and nearly every seed's right neighbour is
            // already visited: one thread per seed checks that bit and walks the rare run itself.
            uint32_t* vis = mf2_smem(C.bmA_off);
            uint16_t* lab = reinterpret_cast<uint16_t*>(mf2_smem(C.word_off));
            const uint32_t wn = (n + 31u) >> 5;
#pragma unroll 1
            for (uint32_t i = mf2_slot<THREADS>(); i < cnt; i += THREADS) {
                const uint32_t x = T.get(i) + 1;  // first node of the run
                if (x >= n) continue;
                uint32_t wi = x >> 5;
                uint32_t m = vis[wi] & (0xffffffffu << (x & 31));
                if ((m >> (x & 31)) & 1u) continue;  // no run
#pragma unroll 1
                while (m == 0 && ++wi < wn) m = vis[wi];
                uint32_t e = m ? (wi << 5) + (uint32_t)__ffs((int)m) - 1u : n;
                if (e > n) e = n;
                const uint32_t base = atomicAdd(&sh.lc[(level - 1) % 3], e - x);
#pragma unroll 1
                for (uint32_t j = x; j < e; ++j) {
                    lab[2 * j] = (uint16_t)level;
                    T.put(base + (j - x), j);
                }
#pragma unroll 1
                for (uint32_t w2 = x >> 5; w2 <= ((e - 1) >> 5); ++w2) {
                    uint32_t mask = 0xffffffffu;
                    if (w2 == (x >> 5)) mask &= 0xffffffffu << (x & 31);
                    if (w2 == ((e - 1) >> 5)) mask &= 0xffffffffu >> (31u - ((e - 1) & 31));
                    atomicOr(&vis[w2], mask);
                }
            }
            __syncthreads();
            cnt = sh.lc[(level - 1) % 3];
        }
        const Mf2Lvl L{level + 1, &sh.lc[level % 3], N};
        if (tid == 0) sh.lc[(level + 1) % 3] = 0;  // last level's counter: everyone has read it
#pragma unroll 1
        for (uint32_t i = mf2_slot<THREADS>(); i < cnt; i += THREADS) {
            const uint32_t u = T.get(i);
            if (!express && u + 1 < n) mf2_mark(C, L, u + 1);  // back arc (u+1) -> u: always residual
            if (first) {
                const uint32_t code = word[u] >> 16;
                if (code < kIn16Multi) mf2_mark(C, L, code);
                else if (code == kIn16Multi) mf2_expand_multi(sh, L, u);
            } else {
                mf2_expand_flow(sh, L, u);
            }
        }
        __syncthreads();
        const uint32_t nH = sh.nH;  // uniform
        if (nH) {  // nodes with many arcs: one warp each
            mf2_bfs_heavy<THREADS>(sh, L, nH, first);
            __syncthreads();
            if (tid == 0) sh.nH = 0;
            __syncthreads();
        }
        const Q2 tmp = T;
        T = N;
        N = tmp;
        ++level;
    }
    return level;
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? 2 : 1)
k_maxflow_sm(Mf2Graph G, const uint32_t* __restrict__ comp_lo, const uint32_t* __restrict__ comp_hi,
             uint32_t* work_counter, uint32_t* qF_g, uint32_t* qT_g, uint32_t* qN_g,
             uint32_t* qH_g, SolveParams P, CompStats* __restrict__ stats, uint32_t smem_bytes,
             uint32_t qcap, uint32_t* __restrict__ fb_list, uint32_t* fb_count, uint32_t allow_optr,
             const uint32_t* __restrict__ n_comp_dev,
             MfTotals* __restrict__ totals) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Mf2Shared& sh = *reinterpret_cast<Mf2Shared*>(smem_raw);
    const uint32_t word_off = kMf2HeaderBytes + 16u * qcap;
    uint32_t* const word = reinterpret_cast<uint32_t*>(smem_raw + word_off);
    const uint32_t node_cap_bytes = smem_bytes - kMf2HeaderBytes - 16u * qcap;
    const uint32_t tid = threadIdx.x;
    const uint32_t lane = lane_id();
    const uint32_t n_comp = *n_comp_dev;

    for (;;) {
        if (tid == 0) sh.comp = atomicAdd(work_counter, 1u);
        __syncthreads();
        const uint32_t c = sh.comp;
        if (c >= n_comp) break;
        const uint32_t lo = comp_lo[c], hi = comp_hi[c];
        const uint32_t n = hi - lo + 1;
        const uint32_t obase = G.out_ptr[lo];
        const uint32_t n_bund = G.out_ptr[hi + 1] - obase;
        const bool fits = n <= kMf2MaxNodes && mf2_node_bytes(n, false) <= node_cap_bytes;
        const bool have_optr = allow_optr && fits && n_bund <= 0xffffu &&
                               mf2_node_bytes(n, true) <= node_cap_bytes;
        const Mf2Layout lay = mf2_layout(n, have_optr);
        uint32_t* const inF = word + lay.o_inF;
        uint16_t* const optr = reinterpret_cast<uint16_t*>(word + lay.o_optr);
        const long long t_begin = clock64();
        if (tid == 0) {
            sh.nF = 0;
            sh.nT = 0;
            sh.nN = 0;
            sh.nH = 0;
            sh.relabels_since = 0;
            sh.supply = 0;
            sh.seg_sample = 0;
            sh.not_benign = 0;
            sh.lc[0] = 0;
            sh.lc[1] = 0;
            sh.lc[2] = 0;
            sh.pushes = 0;
            sh.relabels = 0;
            sh.sink_flow = 0;
            sh.stuck = 0;
            Mf2Comp& C = sh.C;
            C.G = G;
            C.lo = lo;
            C.n = n;
            C.obase = obase;
            C.word_off = word_off;
            C.inF_off = word_off + 4u * lay.o_inF;
            C.bmA_off = word_off + 4u * lay.o_A;
            C.bmB_off = word_off + 4u * lay.o_B;
            C.satn_off = word_off + 4u * lay.o_Sn;
            C.express = 0;
            C.optr_off = word_off + 4u * lay.o_optr;
            C.W4 = lay.W4;
            C.have_optr = have_optr;
            C.F = Q2{kMf2HeaderBytes, qF_g + lo, qcap};
            C.T = Q2{kMf2HeaderBytes + 4u * qcap, qT_g + lo, qcap};
            C.N = Q2{kMf2HeaderBytes + 8u * qcap, qN_g + lo, qcap};
            C.H = Q2{kMf2HeaderBytes + 12u * qcap, qH_g + lo, qcap};
        }
        // k_maxflow takes what does not fit, and the components whose nodes are mostly heavy (variable
        // read lengths, tens of bundles per node): their time is the per-bundle global traffic of the
        // warp passes, which shared-memory labels do not shorten (gds_api.cu: launch_mf2_shape)
        if (!fits || 2ull * n_bund > (unsigned long long)kHeavyDeg * n) {
            if (tid == 0) fb_list[atomicAdd(fb_count, 1u)] = c;
            __syncthreads();
            continue;
        }
        if (fits)  // the bitmaps (inF, BFS A, saturated x 2) are contiguous
            for (uint32_t i = lay.o_inF + tid; i < lay.o_optr; i += THREADS) word[i] = 0;
        __syncthreads();
        Q2 F = sh.C.F, N = sh.C.N;
        const Q2 T = sh.C.T, H = sh.C.H;

        // ---- set-up pass: one coalesced sweep over the SoA node arrays, four nodes in flight ----
        // word = (in16 << 16) | 0xffff; sinks become the level-1 candidates of the first relabel;
        // the supplies become the initial frontier.
        {
            uint32_t my_supply = 0;
            uint32_t* bmA = word + lay.o_A;
#pragma unroll 1
            for (uint32_t v0 = tid; v0 < n; v0 += 4 * THREADS) {
                int32_t dm[4];
                uint32_t ip[4], ip1[4], op[4], src[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const uint32_t v = v0 + q * THREADS;
                    const bool ok = v < n;
                    dm[q] = ok ? G.dem[lo + v] : 0;
                    ip[q] = ok && fits ? G.in_ptr[lo + v] : 0;
                    ip1[q] = ok && fits ? G.in_ptr[lo + v + 1] : 0;
                    op[q] = ok && have_optr ? G.out_ptr[lo + v] : 0;
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) src[q] = ip1[q] - ip[q] == 1 ? G.in_src[ip[q]] : 0;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const uint32_t v = v0 + q * THREADS;
                    if (v >= n) continue;
                    if (dm[q] < 0) my_supply += (uint32_t)(-dm[q]);
                    if ((dm[q] < 0 && v >= kExpressEdge) || (dm[q] > 0 && n - 1 - v >= kExpressEdge))
                        sh.not_benign = 1;
                    if (!fits) continue;
                    uint32_t code = kIn16None;
                    if (ip1[q] - ip[q] == 1) code = src[q] == 0xffffffffu ? kIn16None : src[q] - lo;
                    else if (ip1[q] - ip[q] > 1) code = kIn16Multi;
                    word[v] = (code << 16) | (dm[q] > 0 ? 1u : kInf16);
                    if (have_optr) optr[v] = (uint16_t)(op[q] - obase);
                    if (dm[q] > 0) {  // sinks: level 1 of the first relabel
                        atomicOr(&bmA[v >> 5], 1u << (v & 31));
                        q2_append(T, &sh.lc[0], v);
                    }
                    if (dm[q] < 0) {
                        q2_append(F, &sh.nF, ((uint32_t)(-dm[q]) << 16) | v);
                        atomicOr(&inF[v >> 5], 1u << (v & 31));
                    }
                }
            }
            if (have_optr && tid == 0) optr[n] = (uint16_t)n_bund;
            my_supply = __reduce_add_sync(0xffffffffu, my_supply);
            if (lane == 0 && my_supply) atomicAdd(&sh.supply, min(my_supply, 0x10000u));
        }
        __syncthreads();
        // the express schedule: decided from the data alone (oracle: express_component)
        const bool express = G.express_on && (G.express_on == 2 || sh.supply >= kExpressMinSupply) &&
                             !sh.not_benign && n <= kExpressMaxNodes && sh.supply <= 0xffffu;
        const uint32_t bl = express ? 0u : 1u;  // length of a back arc in the labels
        if (sh.supply > 0xffffu || (!express && !G.classic_ok)) {  // nothing has been written to global memory yet
            __syncthreads();
            if (tid == 0) fb_list[atomicAdd(fb_count, 1u)] = c;
            __syncthreads();
            continue;
        }
        if (tid == 0) sh.C.express = express;
        __syncthreads();
        unsigned long long bfs_levels = 0, grs = 1, rounds = 0, max_frontier = 0, frontier_sum = 0;
        (void)t_begin;
        unsigned long long my_pushes = 0, my_relabels = 0;
        long long my_sink = 0, my_stuck = 0;

        // ---- rounds; the first global relabel (no flow yet, shared memory only) opens them ----
        const long long t_gr = clock64();
        uint32_t last_levels = 0;
        bool first = true;
        unsigned long long rounds_since = 0;
        long long cyc_gr = 0, cyc_a = 0, cyc_b = 0, cyc_g = 0;  // diagnostics: clocks per part
        for (;;) {
            const uint32_t cntF = sh.nF;
            bool relabel = first;
            if (!first && cntF != 0 && !(P.max_rounds && rounds >= P.max_rounds)) {
                // (express: a level is a whole read hop, and lane changes cost rounds but no levels)
                unsigned long long interval = (unsigned long long)last_levels * P.gr_levels_pct / 100 * (2u - bl);
                if (interval < P.gr_interval_min) interval = P.gr_interval_min;
                relabel = rounds_since >= interval &&
                          (unsigned long long)sh.relabels_since * 100 >=
                              (unsigned long long)P.gr_relabel_pct * n;
            }
            if (relabel) {
                const long long t_g = clock64();
                if (!first) {  // flow exists: labels start over, the nodes with sink capacity left seed
                    __syncthreads();
                    uint32_t* bmA = word + lay.o_A;
                    for (uint32_t i = tid; i < lay.W4; i += THREADS) bmA[i] = 0;
                    if (tid == 0) {
                        sh.lc[0] = 0;
                        sh.lc[1] = 0;
                        sh.lc[2] = 0;
                    }
                    __syncthreads();
#pragma unroll 1
                    for (uint32_t v = tid; v < n; v += THREADS) {
                        const bool is_sink = (int32_t)g_ld(&G.node[lo + v].snk) > 0;
                        word[v] = is_sink ? 1u : kInf16;
                        if (is_sink) {
                            atomicOr(&bmA[v >> 5], 1u << (v & 31));
                            q2_append(T, &sh.lc[0], v);
                        }
                    }
                    __syncthreads();
                    ++grs;
                }
                last_levels = mf2_bfs<THREADS>(sh, first, bfs_levels);
                if (first) {  // the in16 halves become the per-round receipts: clear them
#pragma unroll 1
                    for (uint32_t v = tid; v < n; v += THREADS) word[v] &= 0xffffu;
                }
                if (tid == 0) sh.relabels_since = 0;
                rounds_since = 0;
                __syncthreads();
                if (first) cyc_gr = clock64() - t_g;
                else cyc_g += clock64() - t_g;
                first = false;
            }
            if (cntF == 0) break;
            if (P.max_rounds && rounds >= P.max_rounds) break;
            ++rounds;
            ++rounds_since;
            if (cntF > max_frontier) max_frontier = cntF;
            frontier_sum += cntF;
            const bool one_each = cntF <= THREADS;  // a thread owns one frontier node all round
            uint32_t c_bid = 0;                     // its nearest in-arc, kept from phase A for B1

            // ---------------- phase A: pushes (labels are constant in this phase) ----------------
            const long long t_a = clock64();
#pragma unroll 1
            for (uint32_t i = mf2_slot<THREADS>(); i < cntF; i += THREADS) {
                const uint32_t ent = F.get(i);
                const uint32_t v = ent & 0xffffu;
                uint32_t ex = ent >> 16;
                const uint32_t dv = mf2_label(word, v);
                if (dv == kInf16) continue;
                NodeRec* nr = G.node + lo + v;
                // every load below is independent of the others: one memory trip
                uint32_t ob = 0, oe = 0;
                uint4 br0 = make_uint4(0, 0, 0, 0);
                if (have_optr) {
                    ob = obase + optr[v];
                    oe = obase + optr[v + 1];
                    if (oe > ob) br0 = ld_bund(&G.bund[oe - 1]);
                }
                const uint4 lo4 = ld_node_lo(nr);
                const uint4 hi4 = ld_node_hi(nr);
                const uint4 r_hi = ld_node_hi(nr + 1);
                if (!have_optr) {
                    ob = hi4.z;
                    oe = r_hi.z;
                }
                const uint32_t ib = hi4.w, ie = r_hi.w;
                c_bid = ie > ib ? lo4.y : 0u;  // nodes without in-arcs carry no valid id
                if ((oe - ob) + (ie - ib) > kHeavyDeg) {
                    q2_append(H, &sh.nH, i);
                    continue;
                }
                const uint32_t dL = v > 0 ? mf2_label(word, v - 1) : kInf16;
                const uint32_t dR = v + 1 < n ? mf2_label(word, v + 1) : kInf16;
                int32_t snk_now = (int32_t)hi4.x;
                if (dv == 1) {  // 1. sink arc
                    const int32_t s = (int32_t)hi4.x;
                    if (s > 0) {
                        const uint32_t dl = min(ex, (uint32_t)s);
                        g_st(&nr->snk, (uint32_t)(s - (int32_t)dl));
                        snk_now = s - (int32_t)dl;
                        ex -= dl;
                        my_sink += dl;
                        ++my_pushes;
                        // U4: the sink of a node without a live bundle of its own is full: walkers pass it
                        if (express && snk_now == 0 && G.dead[lo + v]) mf2_sat_set(sh.C, v, true);
                    }
                }
                // 2. own bundles, farthest end first
#pragma unroll 1
                for (uint32_t b = oe; ex > 0 && b-- > ob;) {
                    const uint4 br = (have_optr && b == oe - 1) ? br0 : ld_bund(&G.bund[b]);
                    const uint32_t r = br.y - br.z;
                    if (r == 0) continue;
                    const uint32_t t = br.x - lo;
                    if (mf2_label(word, t) + 1 != dv) continue;
                    const uint32_t dl = min(ex, r);
                    g_st(&G.bund[b].f, br.z + dl);
                    ex -= dl;
                    mf2_give(sh, t, dl);
                    ++my_pushes;
                    // U1: the owner filled its only bundle (nobody else touches it this round)
                    if (express && dl == r && oe - ob == 1 && snk_now == 0) mf2_sat_set(sh.C, v, true);
                }
                // 3. cancel back-flow towards the right neighbour
                if (ex > 0 && v + 1 < n && dR + 1 == dv) {
                    const int32_t gr = (int32_t)r_hi.y;
                    if (gr > 0) {
                        const uint32_t dl = min(ex, (uint32_t)gr);
                        g_st(&(nr + 1)->g, (uint32_t)(gr - (int32_t)dl));
                        ex -= dl;
                        mf2_give(sh, v + 1, dl);
                        ++my_pushes;
                    }
                }
                // 4. back arc to the left neighbour (infinite capacity)
                if (ex > 0 && v > 0 && dL + bl == dv) {
                    if (express) {
                        mf2_give(sh, mf2_walk_left(sh.C, v, ex), ex);
                    } else {
                        g_st(&nr->g, hi4.y + ex);
                        mf2_give(sh, v - 1, ex);
                    }
                    ++my_pushes;
                    ex = 0;
                }
                // 5. cancel flow on incoming bundles, nearest start first.  The nearest one comes
                //    with the node record; its flow is only fetched when its label admits the push
#pragma unroll 1
                for (uint32_t k = ie; ex > 0 && k-- > ib;) {
                    uint32_t s, b;
                    if (k + 1 == ie) {
                        s = lo4.x;
                        b = lo4.y;
                    } else {
                        s = g_ld(&G.in_src[k]);
                        b = 0xffffffffu;
                    }
                    // a forced bundle (its start may lie in another component): nothing to cancel
                    if (s == 0xffffffffu) continue;
                    if (mf2_label(word, s - lo) + 1 != dv) continue;
                    if (b == 0xffffffffu) b = g_ld(&G.in_bid[k]);
                    const uint4 br = ld_bund(&G.bund[b]);
                    if (br.z == 0) continue;
                    const uint32_t dl = min(ex, br.z);
                    g_st(&G.bund[b].f, br.z - dl);
                    ex -= dl;
                    mf2_give(sh, s - lo, dl);
                    ++my_pushes;
                    if (express) mf2_sat_set(sh.C, s - lo, false);  // U2: s has residual capacity again
                }
                F.put(i, (ex << 16) | v);
            }
            __syncthreads();
            const uint32_t nH = sh.nH;  // uniform
            if (nH) {  // ---- heavy nodes, one warp each
                mf2_push_heavy<THREADS>(sh, nH, my_pushes, my_sink);
                __syncthreads();
                if (tid == 0) sh.nH = 0;
                __syncthreads();
            }
            const uint32_t cntT = sh.nT;
            const long long t_b = clock64();
            cyc_a += t_b - t_a;

            // ---- phase B1: fold the receipts, decide relabels from the labels of the round ----
            // (new labels are parked in the high half of the node's word until B2, so every
            //  relabel of this round reads the labels the round started with)
#pragma unroll 1
            for (uint32_t i = mf2_slot<THREADS>(); i < cntF + cntT; i += THREADS) {
                if (i >= cntF) {  // a node that only received
                    const uint32_t w = T.get(i - cntF);
                    const uint32_t ww = word[w];
                    const uint32_t tot = ww >> 16, dw = ww & 0xffffu;
                    word[w] = dw;
                    if (tot > 0) {
                        if (dw == kInf16) {
                            my_stuck += tot;
                        } else {
                            q2_append(N, &sh.nN, (tot << 16) | w);
                            atomicOr(&inF[w >> 5], 1u << (w & 31));
                        }
                    }
                    continue;
                }
                const uint32_t ent = F.get(i);
                const uint32_t v = ent & 0xffffu, left = ent >> 16;
                const uint32_t wv = word[v];
                const uint32_t dv = wv & 0xffffu;
                const uint32_t tot = left + (wv >> 16);
                uint32_t nl = 0;
                if (left > 0 && dv != kInf16) {
                    ++my_relabels;
                    atomicAdd(&sh.relabels_since, 1u);
                    const NodeRec* nr = G.node + lo + v;
                    // residual arcs of v: again loads that do not depend on each other
                    uint4 bo = make_uint4(0, 0, 0, 0), bi = make_uint4(0, 0, 0, 0);
                    uint32_t ob = 0, oe = 0;
                    if (have_optr) {
                        ob = obase + optr[v];
                        oe = obase + optr[v + 1];
                        if (oe > ob) bo = ld_bund(&G.bund[ob]);
                    }
                    if (one_each) bi = ld_bund(&G.bund[c_bid]);  // used only if v has in-arcs
                    const uint4 hi4 = ld_node_hi(nr);
                    const uint4 r_hi = ld_node_hi(nr + 1);
                    if (!have_optr) {
                        ob = hi4.z;
                        oe = r_hi.z;
                    }
                    if ((oe - ob) + (r_hi.w - hi4.w) > kHeavyDeg) {
                        q2_append(H, &sh.nH, i);  // the min over many bundles: warp pass below
                    } else {
                        uint32_t mn = kInf16;
                        bool res_any = (int32_t)hi4.x > 0;
                        if ((int32_t)hi4.x > 0) mn = 0;
#pragma unroll 1
                        for (uint32_t b = ob; b < oe; ++b) {
                            const uint4 br = (have_optr && b == ob) ? bo : ld_bund(&G.bund[b]);
                            if (br.z < br.y) {
                                mn = min(mn, mf2_label(word, br.x - lo));
                                res_any = true;
                            }
                        }
                        if (express) mf2_sat_set(sh.C, v, !res_any);  // U3: exact, after the barrier
                        if (v + 1 < n && (int32_t)r_hi.y > 0) mn = min(mn, mf2_label(word, v + 1));
                        if (v > 0) mn = min(mn, mf2_label(word, v - 1) - (1u - bl));  // labels are >= 1
#pragma unroll 1
                        for (uint32_t k = hi4.w; k < r_hi.w; ++k) {
                            const uint4 br = (one_each && k + 1 == r_hi.w)
                                                 ? bi
                                                 : ld_bund(&G.bund[g_ld(&G.in_bid[k])]);
                            if (br.z > 0) mn = min(mn, mf2_label(word, br.w - lo));
                        }
                        nl = mn >= kInf16 - 1 ? kInf16 : mn + 1;
                    }
                }
                word[v] = (nl << 16) | dv;
                F.put(i, (tot << 16) | v);
            }
            __syncthreads();
            if (sh.nH) {  // relabels of heavy nodes, one warp each
                mf2_relabel_heavy<THREADS>(sh, sh.nH);
                __syncthreads();
                if (tid == 0) sh.nH = 0;
            }
            // ---- phase B2: apply the new labels, next frontier from the old one ----
#pragma unroll 1
            for (uint32_t i = mf2_slot<THREADS>(); i < cntF; i += THREADS) {
                const uint32_t ent = F.get(i);
                const uint32_t v = ent & 0xffffu, tot = ent >> 16;
                const uint32_t wv = word[v];
                const uint32_t nl = wv >> 16;
                const uint32_t dnew = nl ? nl : (wv & 0xffffu);
                if (nl) word[v] = nl;
                if (tot > 0 && dnew != kInf16) {
                    q2_append(N, &sh.nN, ent);  // (its records are in L1 since phase A)
                } else {
                    if (tot > 0) my_stuck += tot;
                    atomicAnd(&inF[v >> 5], ~(1u << (v & 31)));
                }
            }
            if (express) {  // the saturation bits the next round's walkers read
                const uint32_t* satn = mf2_smem(sh.C.satn_off);
                uint32_t* sat = mf2_smem(sh.C.bmB_off);
#pragma unroll 1
                for (uint32_t i = tid; i < lay.W4; i += THREADS) sat[i] = satn[i];
            }
            __syncthreads();
            {
                Q2 tmp = F;
                F = N;
                N = tmp;
            }
            if (tid == 0) {
                sh.nF = sh.nN;
                sh.nN = 0;
                sh.nT = 0;
                sh.C.F = F;  // the non-inlined paths read the queues from shared memory
                sh.C.N = N;
            }
            __syncthreads();
            cyc_b += clock64() - t_b;
        }
        // ---- per-component statistics ----
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            my_pushes += __shfl_xor_sync(0xffffffffu, my_pushes, o);
            my_relabels += __shfl_xor_sync(0xffffffffu, my_relabels, o);
            my_sink += __shfl_xor_sync(0xffffffffu, my_sink, o);
            my_stuck += __shfl_xor_sync(0xffffffffu, my_stuck, o);
        }
        if (lane == 0) {
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
            cs.cyc_gr_init = (unsigned long long)(t_gr - t_begin);
            cs.cyc_gr_bfs = (unsigned long long)cyc_gr;
            cs.cyc_gr_snap = (unsigned long long)cyc_a;
            cs.cyc_front = (unsigned long long)cyc_b;
            cs.cyc_gr_later = (unsigned long long)cyc_g;
            stats[c] = cs;
        }
        __syncthreads();
    }
}

}  // namespace gds
