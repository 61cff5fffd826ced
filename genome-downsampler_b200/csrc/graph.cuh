// graph.cuh — K2 (coverage flow graph over reference positions) and K4 (zero-coverage cuts).
//
// Network restated from quasi_mcp_cpu_max_flow_solver.cpp:30-87 (identical construction in
// quasi_mcp_cuda_max_flow_solver.cu:157-259), on read BUNDLES (all reads with equal
// (start node, end node) share one arc of capacity = multiplicity):
//   * sort reads by key (start node, length)  -> bundles, ascending read index inside a bundle
//   * difference array over nodes from the bundles (+mult at s, -mult at t) -> scan -> coverage,
//     capped coverage, demand, initial excess (source arcs pre-saturated), sink capacities
//   * out-CSR (bundles by start) and in-CSR (bundle ids by end, ascending start)
//   * components = maximal runs of covered positions (a back arc over an uncovered position can
//     carry no flow in any maximum flow, so it is cut)
#pragma once
#include <cstddef>
#include "common.cuh"
#include "prep.cuh"
#include "radix_sort.cuh"
#include "scan.cuh"

namespace gds {

// Per-sample layout of the virtual node space.  A reference longer than seg positions is cut
// into nseg segments (the zero-coverage split of SURVEY App. A.3, generalised): a read crossing
// a cut becomes two arcs truncated at the cut node, one per segment, and is kept if either part
// carries flow.  Virtual id of original node x in segment j = vbase + j*W + P + (x - j*seg),
// W = P + seg + 1, with P = maxlen-1 phantom ids in front of every segment.  Arc items are keyed
// by (fake start id, original length); the right part of a crossing read uses the fake start
// (end node - length), which lands on a phantom id, so the key width does not grow.  Decoding
// clamps to the real node range of the segment.  nseg == 1: virtual == original, P = W = 0.
// Restated on the CPU in oracle/gds_oracle.cpp: build_sync_graph.
struct VSample {
    uint32_t obase, vbase, L, nseg, P, W;
};

struct VLayout {
    const VSample* vs;    // [n_samples]
    const uint64_t* off;  // [n_samples+1] read offsets
    uint32_t n_samples;
    uint32_t seg;
    __device__ __forceinline__ uint32_t fake_primary(const VSample& v, uint32_t s) const {
        if (v.nseg == 1) return v.vbase + s;
        uint32_t js = s / seg;
        return v.vbase + js * v.W + v.P + (s - js * seg);
    }
    __device__ __forceinline__ bool crosses(const VSample& v, uint32_t s, uint32_t e) const {
        return v.nseg > 1 && e + 1u != s && e / seg > s / seg;  // a read of length 0 crosses nothing
    }
    __device__ __forceinline__ uint32_t fake_right(const VSample& v, uint32_t s, uint32_t e) const {
        uint32_t je = e / seg;
        uint32_t vt = v.vbase + je * v.W + v.P + (e + 1 - je * seg);
        return vt - (e - s + 1);
    }
    // real node range [first, last] of the segment holding virtual id vid
    __device__ __forceinline__ void seg_range(const VSample& v, uint32_t vid, uint32_t& first,
                                              uint32_t& last) const {
        if (v.nseg == 1) {
            first = v.vbase;
            last = v.vbase + v.L;
            return;
        }
        uint32_t j = (vid - v.vbase) / v.W;
        first = v.vbase + j * v.W + v.P;
        last = first + min(seg, v.L - j * seg);
    }
    __device__ __forceinline__ uint32_t to_orig(const VSample& v, uint32_t vid) const {
        if (v.nseg == 1) return v.obase + (vid - v.vbase);
        uint32_t j = (vid - v.vbase) / v.W;
        return v.obase + j * seg + ((vid - v.vbase) - j * v.W - v.P);
    }
};

// First-pass key source of the arc sort.  Items [0, n_reads) are the reads themselves (left part
// if they cross a cut), items [n_reads, n_reads + n_cross) the right parts of crossing reads
// (cross_idx = their read indices, ascending).  key = (fake start << lenbits) | (len - minlen);
// value = owner read index.
//   LOCAL  (no sample is segmented): the sort is segmented by sample, so the key is relative to
//          the sample — simply (start << lenbits) | (len - minlen): branch-free, no lookups;
//   global (some sample is segmented): one group, key on the global virtual node id.
template <typename K, bool LOCAL>
struct ReadKeys {
    typedef uint2 Raw;  // (start, end) of the owner read
    const uint32_t* S;
    const uint32_t* E;
    VLayout vl;
    const uint32_t* cross_idx;
    size_t n_reads;
    int lenbits;
    uint32_t minlen;
    // validation fused into the first histogram pass when the caller gave read-length hints
    // (LOCAL keys only): range check against the sample's reference length + the hints themselves
    const uint32_t* ref_len;  // [n_samples], null = no fused validation
    uint32_t* stats;          // [2] += range errors, [3] += reads outside the hinted lengths
    uint32_t hint_min, hint_max;
    __device__ __forceinline__ bool checks() const { return LOCAL && ref_len != nullptr; }
    __device__ __forceinline__ uint32_t check(Raw r, uint32_t group) const {
        const uint32_t len = r.y - r.x + 1;
        if (!read_in_range(r.x, r.y, ref_len[group])) return 1u;
        return (len < hint_min || len > hint_max) ? 0x10000u : 0u;
    }
    __device__ __forceinline__ uint32_t* check_stats() const { return stats; }
    __device__ __forceinline__ Raw load(size_t i) const {
        if (LOCAL) return make_uint2(ld_stream(S + i), ld_stream(E + i));
        size_t rd = i < n_reads ? i : (size_t)cross_idx[i - n_reads];
        return make_uint2(S[rd], E[rd]);
    }
    __device__ __forceinline__ K make(Raw r, size_t i) const {
        const K low = (K)(r.y - r.x + 1 - minlen);
        if (LOCAL) return ((K)r.x << lenbits) | low;
        if (i < n_reads) {
            uint32_t k = vl.n_samples == 1 ? 0 : find_sample(vl.off, vl.n_samples, i);
            return ((K)vl.fake_primary(vl.vs[k], r.x) << lenbits) | low;
        }
        uint32_t rd = cross_idx[i - n_reads];
        uint32_t k = vl.n_samples == 1 ? 0 : find_sample(vl.off, vl.n_samples, rd);
        return ((K)vl.fake_right(vl.vs[k], r.x, r.y) << lenbits) | low;
    }
    __device__ __forceinline__ uint32_t owner(size_t i) const {
        if (LOCAL) return (uint32_t)i;
        return i < n_reads ? (uint32_t)i : cross_idx[i - n_reads];
    }
};

// crossing reads -> ascending list of their indices (tile counts -> scan -> write)
constexpr int kCrossThreads = 256;
constexpr int kCrossItems = 8;
constexpr int kCrossTile = kCrossThreads * kCrossItems;

__global__ void __launch_bounds__(kCrossThreads)
k_cross_count(const uint32_t* __restrict__ S, const uint32_t* __restrict__ E, size_t n, VLayout vl,
              uint32_t* __restrict__ tile_counts) {
    size_t base = (size_t)blockIdx.x * kCrossTile + (size_t)threadIdx.x * kCrossItems;
    uint32_t c = 0;
#pragma unroll
    for (int q = 0; q < kCrossItems; ++q) {
        size_t i = base + q;
        if (i < n) {
            uint32_t k = vl.n_samples == 1 ? 0 : find_sample(vl.off, vl.n_samples, i);
            c += vl.crosses(vl.vs[k], S[i], E[i]) ? 1u : 0u;
        }
    }
    c = __reduce_add_sync(0xffffffffu, c);
    __shared__ uint32_t tot;
    if (threadIdx.x == 0) tot = 0;
    __syncthreads();
    if (lane_id() == 0 && c) atomicAdd(&tot, c);
    __syncthreads();
    if (threadIdx.x == 0) tile_counts[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(kCrossThreads)
k_cross_write(const uint32_t* __restrict__ S, const uint32_t* __restrict__ E, size_t n, VLayout vl,
              const uint32_t* __restrict__ tile_offs, uint32_t* __restrict__ cross_idx) {
    __shared__ uint32_t total;
    size_t base = (size_t)blockIdx.x * kCrossTile + (size_t)threadIdx.x * kCrossItems;
    bool hit[kCrossItems];
    uint32_t c = 0;
#pragma unroll
    for (int q = 0; q < kCrossItems; ++q) {
        size_t i = base + q;
        hit[q] = false;
        if (i < n) {
            uint32_t k = vl.n_samples == 1 ? 0 : find_sample(vl.off, vl.n_samples, i);
            hit[q] = vl.crosses(vl.vs[k], S[i], E[i]);
        }
        c += hit[q] ? 1u : 0u;
    }
    uint32_t ex = block_excl_scan(c, &total) + tile_offs[blockIdx.x];
#pragma unroll
    for (int q = 0; q < kCrossItems; ++q)
        if (hit[q]) cross_idx[ex++] = (uint32_t)(base + q);
}

// Bundle heads over the sorted keys: item j starts a bundle if it is the first item of its group
// or its key differs from its predecessor's.  Same tile geometry as the sort (tiles never
// straddle a group).
constexpr int kHeadThreads = 1024;
constexpr int kHeadRows = kRsTile / kHeadThreads;  // warp w owns items [w*32*rows, (w+1)*32*rows)

// head flags of this lane's items, one ballot word per row (coalesced 128-byte row loads; the
// predecessor comes from the neighbouring lane, lane 0 re-reads one key)
template <typename K>
__device__ __forceinline__ void head_ballots(const K* __restrict__ keys, const TilePos& tp,
                                             uint32_t (&bal)[kHeadRows]) {
    const uint32_t lane = lane_id();
    const uint32_t wofs = (threadIdx.x >> 5) * 32 * kHeadRows;
    K kk[kHeadRows];
#pragma unroll
    for (int r = 0; r < kHeadRows; ++r) {
        uint32_t j = wofs + r * 32 + lane;
        kk[r] = keys[tp.first + (j < tp.n_valid ? j : 0u)];
    }
    // predecessor of the warp chunk's first item (unless it is the first item of the group)
    K prev_chunk = (K)0;
    const bool chunk_has_prev = !(wofs == 0 && tp.tile_in_g == 0) && wofs < tp.n_valid;
    if (lane == 0 && chunk_has_prev) prev_chunk = keys[tp.first + wofs - 1];
#pragma unroll
    for (int r = 0; r < kHeadRows; ++r) {
        uint32_t j = wofs + r * 32 + lane;
        K up = __shfl_up_sync(0xffffffffu, kk[r], 1);
        K last_prev_row = __shfl_sync(0xffffffffu, r ? kk[r ? r - 1 : 0] : prev_chunk, r ? 31 : 0);
        K pred = lane ? up : last_prev_row;
        bool first_of_group = j == 0 && tp.tile_in_g == 0;
        bool head = j < tp.n_valid && (first_of_group || kk[r] != pred);
        bal[r] = __ballot_sync(0xffffffffu, head);
    }
}

// pass 1: head flags of every item as a bitmap (one word per 32 consecutive items of a tile, tiles
// padded to kRsTile/32 words) + heads per tile.  pass 2 reads the bitmap, not the keys again.
template <typename K>
__global__ void __launch_bounds__(kHeadThreads)
k_heads_count(const K* __restrict__ keys, TileMap tm, uint32_t* __restrict__ tile_counts,
              uint32_t* __restrict__ head_bits) {
    const TilePos tp = locate_tile(tm, blockIdx.x);
    uint32_t bal[kHeadRows];
    head_ballots<K>(keys, tp, bal);
    const uint32_t warp = threadIdx.x >> 5, lane = lane_id();
    uint32_t c = 0;
#pragma unroll
    for (int r = 0; r < kHeadRows; ++r) c += __popc(bal[r]);
    if (lane < kHeadRows) {
        uint32_t w = bal[0];
#pragma unroll
        for (int r = 1; r < kHeadRows; ++r) w = lane == r ? bal[r] : w;
        head_bits[(size_t)blockIdx.x * (kRsTile / 32) + warp * kHeadRows + lane] = w;
    }
    __shared__ uint32_t tot;
    if (threadIdx.x == 0) tot = 0;
    __syncthreads();
    if (lane == 0 && c) atomicAdd(&tot, c);
    __syncthreads();
    if (threadIdx.x == 0) tile_counts[blockIdx.x] = tot;
}

// pass 2: one lane per bitmap word (32 items): 256 threads cover a tile.  Only the keys at head
// positions are gathered.
constexpr int kHeadWriteThreads = kRsTile / 32;

template <typename K>
__global__ void __launch_bounds__(kHeadWriteThreads)
k_heads_write(const K* __restrict__ keys, TileMap tm, const uint32_t* __restrict__ tile_offs,
              const uint32_t* __restrict__ head_bits, uint32_t* __restrict__ b_first,
              K* __restrict__ b_key) {
    __shared__ uint32_t wtot[kHeadWriteThreads / 32];
    const TilePos tp = locate_tile(tm, blockIdx.x);
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    uint32_t bits = head_bits[(size_t)blockIdx.x * (kRsTile / 32) + threadIdx.x];
    const uint32_t c = __popc(bits);
    const uint32_t incl = warp_incl_scan(c);
    if (lane == 31) wtot[warp] = incl;
    __syncthreads();
    uint32_t slot = tile_offs[blockIdx.x] + incl - c;
#pragma unroll
    for (int w = 0; w < kHeadWriteThreads / 32; ++w) slot += (w < (int)warp) ? wtot[w] : 0u;
    const size_t base = tp.first + (size_t)threadIdx.x * 32;
    while (bits) {
        const int b = __ffs(bits) - 1;
        bits &= bits - 1;
        b_first[slot] = (uint32_t)(base + b);
        b_key[slot] = keys[base + b];
        ++slot;
    }
}

// Max-flow state, one 32-byte sector per node and one 16-byte record per bundle, so that a
// push touches: own node (1 sector, neighbours v-1 / v+1 adjacent) -> bundle (1 load) -> target
// node (1 sector).  Everything a round decides on comes from these records; d_snap (the label
// snapshot relabels read) is the only side array.
// The first 16 bytes have two uses: {d, stamp, e, eadd} for k_maxflow (state in global memory), as
// k_node_finalize writes them; when k_maxflow_sm runs (labels and excess in shared memory), k_in_src
// puts {start node, bundle id} of the node's NEAREST in-arc over d and stamp, and k_maxflow restores
// the four fields for the components it is handed afterwards.
struct __align__(32) NodeRec {
    uint32_t d;        // label                                      | start node of the nearest in-arc
    uint32_t stamp;    // round in which v is in the frontier        | its bundle id
    int32_t e;         // excess                                    (e, eadd: one aligned 8-byte
    int32_t eadd;      // excess received during the current round   store in phase B; 0 between rounds)
    int32_t snk;       // remaining sink-arc capacity
    int32_t g;         // flow on the back arc v -> v-1
    uint32_t out_ptr;  // first bundle starting at v (bundles are sorted by start)
    uint32_t in_ptr;   // first in-CSR slot of bundles ending at v
};
struct __align__(16) BundleRec {
    uint32_t t, mult, f, s;  // end node, capacity, flow, start node
};

// Per bundle: decode the key to the real (s, t) of its segment, multiplicity, and accumulate the
// node-level difference array (virtual space, and original space when some sample is split) and
// the CSR degree counters.  One atomic group per BUNDLE, not per read.
template <typename K>
__global__ void __launch_bounds__(256)
k_bundle_fill(const K* __restrict__ b_key, uint32_t* __restrict__ b_first,
              const uint32_t* __restrict__ sorted_owner, uint32_t B, uint32_t n_items, int lenbits,
              uint32_t minlen, VLayout vl, bool local_keys, BundleRec* __restrict__ bund,
              uint32_t* __restrict__ b_t, int32_t* __restrict__ diff,
              uint32_t* __restrict__ outdeg, uint32_t* __restrict__ indeg,
              int32_t* __restrict__ odiff /* null when virtual == original */) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    K key = b_key[b];
    uint32_t fake = (uint32_t)(key >> lenbits);
    uint32_t len = (uint32_t)(key & (((K)1 << lenbits) - 1)) + minlen;
    uint32_t first_item = b_first[b];
    uint32_t owner = sorted_owner[first_item];
    uint32_t k = vl.n_samples == 1 ? 0 : find_sample(vl.off, vl.n_samples, owner);
    const VSample v = vl.vs[k];
    if (local_keys) fake += v.vbase;  // the segmented sort keys are relative to the sample
    uint32_t first, last;
    vl.seg_range(v, fake, first, last);
    uint32_t s = max(fake, first);
    uint32_t t = min(fake + len, last);
    uint32_t nxt = (b + 1 < B) ? b_first[b + 1] : n_items;
    uint32_t mult = nxt - first_item;
    reinterpret_cast<uint4*>(bund)[b] = make_uint4(t, mult, 0u, s);  // {t, mult, f = 0, s}
    b_t[b] = t;  // key of the in-CSR sort
    atomicAdd(&diff[s], (int32_t)mult);
    atomicAdd(&diff[t], -(int32_t)mult);
    atomicAdd(&outdeg[s], 1u);
    atomicAdd(&indeg[t], 1u);
    if (odiff) {
        atomicAdd(&odiff[vl.to_orig(v, s)], (int32_t)mult);
        atomicAdd(&odiff[vl.to_orig(v, t)], -(int32_t)mult);
    }
}

// Original-space outputs when some sample is split: capped coverage, demand
// (create_demand_function, quasi_mcp_cpu_max_flow_solver.cpp:75-87) and F* = sum of source
// capacities of the ORIGINAL network (totals[3]).
__global__ void __launch_bounds__(256)
k_orig_outputs(const uint32_t* __restrict__ oexcl, const int32_t* __restrict__ odiff,
               uint32_t n_onodes, uint32_t M, uint32_t* __restrict__ cov_capped_out,
               int32_t* __restrict__ demand_out, unsigned long long* __restrict__ totals) {
    uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long src = 0;
    if (v < n_onodes) {
        uint32_t covL = oexcl[v];
        uint32_t covR = covL + (uint32_t)odiff[v];
        int32_t dem = (int32_t)min(covL, M) - (int32_t)min(covR, M);
        if (cov_capped_out) cov_capped_out[v] = min(covR, M);
        if (demand_out) demand_out[v] = dem;
        if (dem < 0) src = (unsigned long long)(-dem);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) src += __shfl_xor_sync(0xffffffffu, src, o);
    if (lane_id() == 0 && src) atomicAdd(&totals[3], src);
}

// Flow that passes straight through the cut nodes when the segment flows are stitched into a
// flow of the original network: min(cov'(x-1), cov'(x)) per cut node x (totals[4]).
__global__ void k_cut_through(const uint32_t* __restrict__ cut_nodes, uint32_t n_cuts,
                              const uint32_t* __restrict__ oexcl, const int32_t* __restrict__ odiff,
                              uint32_t M, unsigned long long* __restrict__ totals) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_cuts) return;
    uint32_t x = cut_nodes[i];
    uint32_t covL = oexcl[x];
    uint32_t covR = covL + (uint32_t)odiff[x];
    atomicAdd(&totals[4], (unsigned long long)min(min(covL, M), min(covR, M)));
}

// covL[v] = coverage of the position left of node v = exclusive prefix; covR = inclusive prefix.
// totals[0] (u64) accumulates F*.
__global__ void __launch_bounds__(256)
k_node_finalize(const uint32_t* __restrict__ excl, const int32_t* __restrict__ diff,
                const uint32_t* __restrict__ out_ptr, const uint32_t* __restrict__ in_ptr,
                uint32_t n_nodes, uint32_t M, NodeRec* __restrict__ node,
                uint32_t* __restrict__ d_snap, uint32_t* __restrict__ comp_start,
                uint32_t* __restrict__ comp_end, uint32_t* __restrict__ cov_capped_out,
                int32_t* __restrict__ demand_out, int32_t* __restrict__ dem_v /* [n_nodes] always */,
                unsigned long long* __restrict__ totals,
                const int32_t* __restrict__ adj /* null or: what the forced bundles add to the demand */,
                uint32_t cut_at /* v and v+1 belong to one component iff covR[v] > cut_at (0 or M) */,
                unsigned long long* __restrict__ res_supply /* += supply of the residual problem */,
                uint8_t* __restrict__ dead /* null or: |= 1 for nodes without bundles of their own */) {
    uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long src = 0, rsrc = 0;
    if (v == n_nodes) {  // sentinel record: closes the CSR ranges of the last node
        uint4* r = reinterpret_cast<uint4*>(&node[v]);
        r[0] = make_uint4(0u, 0u, 0u, 0u);
        r[1] = make_uint4(0u, 0u, out_ptr[v], in_ptr[v]);
    }
    static_assert(sizeof(NodeRec) == 32 && offsetof(NodeRec, e) == 8 && offsetof(NodeRec, snk) == 16,
                  "NodeRec layout is relied on by the vector loads in maxflow.cuh");
    if (v < n_nodes) {
        uint32_t covL = excl[v];
        uint32_t covR = covL + (uint32_t)diff[v];
        int32_t dem = (int32_t)min(covL, M) - (int32_t)min(covR, M);
        // what K3 solves: the demand with the forced bundles' fixed flows taken out
        const int32_t dk = dem + (adj ? adj[v] : 0);
        uint4* r = reinterpret_cast<uint4*>(&node[v]);
        r[0] = make_uint4(kLabelInf, 0u, (uint32_t)(dk < 0 ? -dk : 0), 0u);  // d, stamp, e, eadd
        r[1] = make_uint4((uint32_t)(dk > 0 ? dk : 0), 0u, out_ptr[v], in_ptr[v]);  // snk, g, ptrs
        d_snap[v] = kLabelInf;
        dem_v[v] = dk;
        comp_start[v] = (covL <= cut_at && covR > cut_at) ? 1u : 0u;
        comp_end[v] = (covL > cut_at && covR <= cut_at) ? 1u : 0u;
        if (cov_capped_out) cov_capped_out[v] = min(covR, M);
        if (demand_out) demand_out[v] = dem;
        if (dem < 0) src = (unsigned long long)(-dem);
        if (dk < 0) rsrc = (unsigned long long)(-dk);
        if (dead && out_ptr[v + 1] == out_ptr[v]) dead[v] = 1;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        src += __shfl_xor_sync(0xffffffffu, src, o);
        rsrc += __shfl_xor_sync(0xffffffffu, rsrc, o);
    }
    if (lane_id() == 0 && src) atomicAdd(&totals[0], src);
    if (lane_id() == 0 && rsrc) atomicAdd(res_supply, rsrc);
}

// start node of every in-CSR slot (the first global relabel of K3 walks only this array), and for
// every node with in-arcs {start node, bundle id} of its last in-CSR slot — the nearest start, the
// first one a cancel tries — next to its other fields, so a push needs no in-CSR lookup
__global__ void __launch_bounds__(256)
k_in_src(const BundleRec* __restrict__ bund, const uint32_t* __restrict__ in_bid,
         const uint32_t* __restrict__ in_ptr, const uint32_t* __restrict__ B_dev,
         uint32_t* __restrict__ in_src,
         NodeRec* __restrict__ node /* null: k_maxflow only, the records keep {d, stamp, e, eadd} */,
         uint32_t* __restrict__ in1 /* [n_nodes], preset to 0xffffffff: start node of a node's only
                                       in-arc, 0xfffffffe when it has several */) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= *B_dev) return;
    const uint32_t b = in_bid[k];
    const uint4 r = reinterpret_cast<const uint4*>(bund)[b];  // t, mult, f, s
    // a forced bundle (capacity 0 while K3 runs) is no arc of the residual graph: the relabels that
    // walk in_src without looking at the bundles must not see it
    const bool inert = r.y == 0;
    in_src[k] = inert ? 0xffffffffu : r.w;
    if (k == in_ptr[r.x]) {
        if (k + 1 != in_ptr[r.x + 1]) in1[r.x] = 0xfffffffeu;
        else if (!inert) in1[r.x] = r.w;
    }
    if (node && k + 1 == in_ptr[r.x + 1])
        *reinterpret_cast<uint2*>(&node[r.x]) = make_uint2(inert ? 0xffffffffu : r.w, b);
}

// Components are disjoint runs, so starts and ends alternate: the end at v closes the component
// opened by the last start before it, index (number of starts before v) - 1 — one scan serves both.
__global__ void __launch_bounds__(256)
k_comp_write(const uint32_t* __restrict__ comp_start, const uint32_t* __restrict__ comp_end,
             const uint32_t* __restrict__ start_idx, uint32_t n_nodes,
             uint32_t* __restrict__ comp_lo, uint32_t* __restrict__ comp_hi) {
    uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_nodes) return;
    if (comp_start[v]) comp_lo[start_idx[v]] = v;
    if (comp_end[v]) comp_hi[start_idx[v] - 1] = v;
}

// ---- forced reads out, cuts in (DESIGN.md §4) -------------------------------------------------
// A bundle that covers a position with cov <= M is in every valid answer: its flow is fixed at its
// multiplicity.  flag -> exclusive scan = number of such positions left of a node; a bundle s -> t
// is forced iff the count differs between t and s.  Forced bundles get capacity 0 for the solve
// (their multiplicity waits in fmult), their ends' demands absorb the fixed flow (adj), and
// k_node_finalize cuts the components at every such position.
__global__ void __launch_bounds__(256)
k_uncapped_flags(const uint32_t* __restrict__ excl, const int32_t* __restrict__ diff, uint32_t n_nodes,
                 uint32_t M, uint32_t* __restrict__ flag /* [n_nodes + 1] */) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v > n_nodes) return;
    flag[v] = v < n_nodes && excl[v] + (uint32_t)diff[v] <= M ? 1u : 0u;
}

// One thread per NODE: if no uncapped position lies within maxlen of v none of its bundles can be
// forced — two reads of the prefix count and nothing else (config 4: all but the genome's two ends).
// Otherwise its out-bundles are tested one by one.  fmult[b] is written for every bundle of such a
// node (0 when the bundle is not forced) and read back, after K3, by the same test: it needs no
// clearing.
__device__ __forceinline__ bool node_may_be_forced(const uint32_t* __restrict__ unc, uint32_t v,
                                                   uint32_t n_nodes, uint32_t maxlen) {
    return unc[v] != unc[min(v + maxlen, n_nodes)];
}

__global__ void __launch_bounds__(256)
k_forced_bundles(BundleRec* __restrict__ bund, const uint32_t* __restrict__ out_ptr, uint32_t n_nodes,
                 uint32_t maxlen, const uint32_t* __restrict__ unc, int32_t* __restrict__ adj,
                 uint32_t* __restrict__ fmult,
                 uint8_t* __restrict__ dead /* [n_nodes], zero on entry: 1 = every own bundle is forced */) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_nodes || !node_may_be_forced(unc, v, n_nodes, maxlen)) return;
    const uint32_t uv = unc[v];
    bool live = false;
    for (uint32_t b = out_ptr[v]; b < out_ptr[v + 1]; ++b) {
        const uint4 r = reinterpret_cast<const uint4*>(bund)[b];  // t, mult, f, s
        const bool forced = unc[r.x] != uv;
        fmult[b] = forced ? r.y : 0u;
        if (forced) {
            bund[b].mult = 0;
            atomicAdd(&adj[v], (int32_t)r.y);
            atomicAdd(&adj[r.x], -(int32_t)r.y);
        } else {
            live = true;
        }
    }
    if (!live) dead[v] = 1;
}

// after K3: the forced bundles come back with their fixed flow (K5 keeps all their reads)
__global__ void __launch_bounds__(256)
k_forced_restore(BundleRec* __restrict__ bund, const uint32_t* __restrict__ out_ptr, uint32_t n_nodes,
                 uint32_t maxlen, const uint32_t* __restrict__ unc, const uint32_t* __restrict__ fmult) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_nodes || !node_may_be_forced(unc, v, n_nodes, maxlen)) return;
    for (uint32_t b = out_ptr[v]; b < out_ptr[v + 1]; ++b) {
        const uint32_t m = fmult[b];
        if (m) {
            bund[b].mult = m;
            bund[b].f = m;
        }
    }
}

}  // namespace gds
