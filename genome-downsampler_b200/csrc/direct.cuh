// direct.cuh — sort-free K2 (bundles) and K5 (selection) for samples whose key space fits in the
// shared memory of one SM.
//
// A bundle is the set of reads with one (start node, length) key (graph.cuh).  When all reads of
// the call have one length, the key is the start node, and when a sample has at most kDirectMaxKeys
// nodes (30 001 for a 30 kb reference: configs 1, 3, 5 of SURVEY §8) its bundle multiplicities are
// a HISTOGRAM of the reads: one shared-memory atomic per read, every input byte read exactly once
// at HBM speed (tools/hist_probe.cu: 7.0 TB/s on B200 — the atomic unit keeps up with the loads),
// instead of the two-pass radix sort's 48 bytes per read.  Restates the same network as the sort path
// (quasi_mcp_cpu_max_flow_solver.cpp:30-87 on bundles) — bundle order, node ids, difference array
// and CSR are identical, so K3 and every parity test see the same graph.
// Several read lengths take the global-memory histogram at the end of this file: (ref_len + 1) x
// #lengths counters fit one SM only for short references (a 30 kb sample with two lengths already
// has 60 002), so no realistic input with several lengths ever fitted here.
//
// K5 without a sorted read order: see the K5 section below.
#pragma once
#include "common.cuh"
#include "graph.cuh"
#include "prep.cuh"
#include "scan.cuh"

namespace gds {

constexpr uint32_t kDirectMaxKeys = 48 * 1024;  // u32 counters: 192 KB of shared memory
constexpr int kDhThreads = 1024;
constexpr int kDirectUnroll = 4;  // 16-byte loads per array in flight per thread
constexpr int kDkThreads = 256;   // key tiles of the bundle kernels: 4 keys per thread
constexpr int kDkTile = kDkThreads * 4;

struct DirectLayout {
    const uint64_t* off;       // [ns+1] read offsets
    const uint32_t* ref_len;   // [ns]
    const uint32_t* node_base; // [ns+1] first node id of sample k
    const uint32_t* kbase;     // [ns+1] first histogram slot of sample k (regions padded to 32)
    const uint32_t* item_off;  // [ns+1] first work item (sample part) of sample k
    uint32_t ns, minlen;       // minlen: the one read length R
};

__device__ __forceinline__ uint32_t find_u32(const uint32_t* __restrict__ off, uint32_t n,
                                             uint32_t i) {
    uint32_t lo = 0, hi = n;  // invariant: off[lo] <= i < off[hi]
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (off[mid] <= i) lo = mid;
        else hi = mid;
    }
    return lo;
}

// ---- K2 direct: per-sample histogram of read keys -------------------------------------------
// Work item = one part of one sample (parts balance the SMs when there are few samples).  The CTA
// counts the part in shared memory and adds its non-zero counters to the sample's region of the
// global histogram (coalesced reductions; the region must be zero on entry).  Validation (range,
// length hints) rides along: bad reads are counted, never touch the histogram.
__global__ void __launch_bounds__(kDhThreads, 1)
k_direct_hist(const uint32_t* __restrict__ S, const uint32_t* __restrict__ E, DirectLayout dl,
              uint32_t n_items, uint32_t* __restrict__ work_counter, uint32_t* __restrict__ ghist,
              uint32_t kmax, uint32_t* __restrict__ stats) {
    extern __shared__ uint32_t h[];
    __shared__ uint32_t s_item;
    const uint32_t tid = threadIdx.x;
    for (uint32_t i = tid; i < kmax; i += kDhThreads) h[i] = 0;
    uint32_t bad_range = 0, bad_hint = 0;
    const uint32_t R = dl.minlen;
    for (;;) {
        if (tid == 0) s_item = atomicAdd(work_counter, 1u);
        __syncthreads();
        const uint32_t item = s_item;
        if (item >= n_items) break;
        const uint32_t k = find_u32(dl.item_off, dl.ns, item);
        const uint32_t parts = dl.item_off[k + 1] - dl.item_off[k];
        const uint32_t p = item - dl.item_off[k];
        const uint64_t o0 = dl.off[k], o1 = dl.off[k + 1];
        const uint64_t plen = (((o1 - o0) + parts - 1) / parts + 3) & ~3ull;
        const uint64_t a = o0 + p * plen;
        const uint64_t b = min(a + plen, o1);
        const uint32_t L = dl.ref_len[k];
        auto count = [&](uint32_t s, uint32_t e) {
            if (!read_in_range(s, e, L)) {
                ++bad_range;
                return;
            }
            if (e - s + 1 != R) {
                ++bad_hint;
                return;
            }
            atomicAdd(&h[s], 1u);
        };
        if (a < b) {
            // unaligned head and tail by single loads, the body by 16-byte loads
            const uint64_t a4 = min((uint64_t)((a + 3) & ~3ull), b), b4 = max((uint64_t)(b & ~3ull), a4);
            if (tid < a4 - a) count(S[a + tid], E[a + tid]);
            if (tid < b - b4) count(S[b4 + tid], E[b4 + tid]);
            const uint4* S4 = reinterpret_cast<const uint4*>(S);
            const uint4* E4 = reinterpret_cast<const uint4*>(E);
            uint64_t j = a4 / 4 + tid;
            const uint64_t jend = b4 / 4;
            // all loads of a round are issued before the first atomic (8 x 16 B in flight per
            // thread: the kernel is bound by bytes in flight per SM, not by the atomics)
            for (; j + (kDirectUnroll - 1) * kDhThreads < jend; j += kDirectUnroll * kDhThreads) {
                uint4 s[kDirectUnroll], e[kDirectUnroll];
#pragma unroll
                for (int u = 0; u < kDirectUnroll; ++u) {
                    s[u] = ld_stream4(S4 + j + u * kDhThreads);
                    e[u] = ld_stream4(E4 + j + u * kDhThreads);
                }
#pragma unroll
                for (int u = 0; u < kDirectUnroll; ++u) {
                    count(s[u].x, e[u].x);
                    count(s[u].y, e[u].y);
                    count(s[u].z, e[u].z);
                    count(s[u].w, e[u].w);
                }
            }
            for (; j < jend; j += kDhThreads) {
                const uint4 s = ld_stream4(S4 + j), e = ld_stream4(E4 + j);
                count(s.x, e.x);
                count(s.y, e.y);
                count(s.z, e.z);
                count(s.w, e.w);
            }
        }
        __syncthreads();
        uint32_t* gh = ghist + dl.kbase[k];
        const uint32_t kk = dl.kbase[k + 1] - dl.kbase[k];
        for (uint32_t i = tid; i < kk; i += kDhThreads) {
            const uint32_t c = h[i];
            if (c) {
                atomicAdd(gh + i, c);
                h[i] = 0;
            }
        }
        __syncthreads();
    }
    bad_range = __reduce_add_sync(0xffffffffu, bad_range);
    bad_hint = __reduce_add_sync(0xffffffffu, bad_hint);
    if (lane_id() == 0) {
        if (bad_range) atomicAdd(&stats[2], bad_range);
        if (bad_hint) atomicAdd(&stats[3], bad_hint);
    }
}

// ---- bundles = non-zero counters, in key order (sample, start, length) -------------------------
__global__ void __launch_bounds__(kDkThreads)
k_direct_count(const uint32_t* __restrict__ ghist, uint32_t ktot, uint32_t* __restrict__ tile_counts) {
    const uint32_t i = (blockIdx.x * kDkThreads + threadIdx.x) * 4;
    uint32_t c = 0;
    if (i < ktot) {  // ktot is a multiple of 32
        const uint4 v = reinterpret_cast<const uint4*>(ghist)[i / 4];
        c = (v.x != 0) + (v.y != 0) + (v.z != 0) + (v.w != 0);
    }
    c = __reduce_add_sync(0xffffffffu, c);
    __shared__ uint32_t tot;
    if (threadIdx.x == 0) tot = 0;
    __syncthreads();
    if (lane_id() == 0 && c) atomicAdd(&tot, c);
    __syncthreads();
    if (threadIdx.x == 0) tile_counts[blockIdx.x] = tot;
}

// Writes what k_bundle_fill writes on the sort path (bundle record, in-CSR key, difference array,
// CSR degrees) plus the bundle's histogram slot (K5 puts the bundle's flow there) and the identity
// in-CSR.  k_direct_graph below does all of it in one pass, except with forced cuts: the
// forced-bundle test compares the uncapped-position count at a bundle's end, R nodes to the right of
// a node, which a left-to-right pass does not have yet.  This kernel serves that case.
__global__ void __launch_bounds__(kDkThreads)
k_direct_bundles(const uint32_t* __restrict__ ghist, uint32_t ktot, DirectLayout dl,
                 const uint32_t* __restrict__ tile_offs, BundleRec* __restrict__ bund,
                 uint32_t* __restrict__ b_t, uint32_t* __restrict__ b_slot,
                 uint32_t* __restrict__ in_bid, int32_t* __restrict__ diff,
                 uint32_t* __restrict__ outdeg, uint32_t* __restrict__ indeg) {
    __shared__ uint32_t total;
    const uint32_t i = (blockIdx.x * kDkThreads + threadIdx.x) * 4;
    uint32_t v[4] = {0, 0, 0, 0};
    if (i < ktot) {
        const uint4 q = reinterpret_cast<const uint4*>(ghist)[i / 4];
        v[0] = q.x;
        v[1] = q.y;
        v[2] = q.z;
        v[3] = q.w;
    }
    const uint32_t c = (v[0] != 0) + (v[1] != 0) + (v[2] != 0) + (v[3] != 0);
    uint32_t b = block_excl_scan(c, &total) + tile_offs[blockIdx.x];
    if (i >= ktot) return;
    const uint32_t k = find_u32(dl.kbase, dl.ns, i);  // regions are 32-aligned: same k for all 4
    const uint32_t local = i - dl.kbase[k];
    const uint32_t nb = dl.node_base[k];
    // key == start node, so the difference array needs no atomics —
    // diff[v] = (reads starting at v) - (reads ending before v) = hist[v] - hist[v - len];
    // every node of the sample is written (the region covers ref_len + 1 slots)
    const uint32_t L = dl.ref_len[k], len = dl.minlen;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint32_t j = local + q;
        if (j > L) continue;
        const uint32_t ends = j >= len ? ghist[i + q - len] : 0u;
        diff[nb + j] = (int32_t)v[q] - (int32_t)ends;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        if (!v[q]) continue;
        const uint32_t s = nb + local + q;
        const uint32_t t = s + len;
        reinterpret_cast<uint4*>(bund)[b] = make_uint4(t, v[q], 0u, s);
        b_t[b] = t;
        b_slot[b] = i + q;
        in_bid[b] = b;
        outdeg[s] = 1u;  // at most one bundle starts / ends at a node
        indeg[t] = 1u;
        ++b;
    }
}

// ---- one read length: the whole flow graph in one pass --------------------------------------------
// With one read length R and no forced cuts, every node and bundle array K3, K5 and K6 read follows
// from the histogram h alone.  Node v of sample k is slot j = v - node_base[k] of the sample's region:
//   diff[v]  = h[j] - h[j-R]         (reads starting at v minus reads ending at v)
//   out-arc  iff h[j] != 0, in-arc iff h[j-R] != 0   (at most one bundle starts / ends at a node)
//   the in-CSR order is the bundle order, so the in-arc of v is bundle indeg[v] and starts at v - R.
// One pass over tiles of the node space carries four exclusive prefixes with the decoupled look-back
// of scan.cuh (status words tile*4 + 0..3): coverage, bundles starting before v, bundles ending
// before v, and components starting before v.  The first three are published as soon as the tile
// has its loads; a component starts where the coverage rises from 0, so that word follows once the
// tile knows its coverage prefix.  Coverage does not leak from one sample into the next: each
// sample's diff sums to 0.  Every output is written once, the same as the chain it replaces
// (direct_count, its scan, direct_bundles, the node scans, node_finalize, the component scan,
// comp_write and in_src) wrote it.
// A lane holds 4 x 4 consecutive nodes (4-aligned: the node arrays take 16-byte stores); 4 tiles of
// 64 registers per thread sit on each SM, so one tile's look-back is covered by the others' loads.
constexpr int kDgThreads = 256;
constexpr int kDgRows = 4;
constexpr int kDgWarpSpan = 32 * 4 * kDgRows;
constexpr int kDgTile = kDgThreads / 32 * kDgWarpSpan;  // 4096 nodes

struct DirectGraphOut {
    BundleRec* bund;
    uint32_t *b_t, *b_slot, *ident, *in_src;
    int32_t* diff;
    uint32_t *excl, *outdeg, *indeg;
    NodeRec* node;
    uint32_t* d_snap;
    int32_t* dem_v;
    uint32_t* in1;
    uint32_t *comp_lo, *comp_hi;
    uint32_t* cov_capped;  // null unless the call asks for it
    int32_t* demand;       // likewise
    uint32_t *n_bundles, *n_comp;
    unsigned long long *fstar, *res_supply;
};

// Histogram slot and sample-local index of nodes v0 .. v0+3 (the four may run into the next
// sample; past the last node they mean nothing).  Samples k0 .. k1 hold the tile's nodes.
__device__ __forceinline__ void dg_locate(const DirectLayout& dl, uint32_t k0, uint32_t k1, uint32_t v0,
                                          uint32_t n_nodes, uint32_t (&slot)[4], uint32_t (&j)[4]) {
    const uint32_t vs = min(v0, n_nodes - 1);
    uint32_t lo = k0, hi = k1 + 1;  // node_base[lo] <= vs < node_base[hi]
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (dl.node_base[mid] <= vs) lo = mid;
        else hi = mid;
    }
    uint32_t k = lo, nb = dl.node_base[k], nb1 = dl.node_base[k + 1], kb = dl.kbase[k];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint32_t v = v0 + q;
        if (v >= nb1 && v < n_nodes) {
            do {
                ++k;
            } while (dl.node_base[k + 1] <= v);
            nb = dl.node_base[k];
            nb1 = dl.node_base[k + 1];
            kb = dl.kbase[k];
        }
        j[q] = v - nb;
        slot[q] = kb + j[q];
    }
}

// Tiles cover nodes [0, n_nodes]: node n_nodes is the sentinel that closes the CSR ranges.
__global__ void __launch_bounds__(kDgThreads, 4)
k_direct_graph(const uint32_t* __restrict__ ghist, DirectLayout dl, uint32_t n_nodes, uint32_t M,
               uint32_t in_first /* k_maxflow_sm runs: {start, bundle} of the in-arc over {d, stamp} */,
               DirectGraphOut o, unsigned long long* __restrict__ status, uint32_t* __restrict__ ticket,
               uint32_t epoch, uint32_t n_tiles) {
    __shared__ uint32_t s_tile, s_k0, s_k1;
    __shared__ uint32_t s_prefix[4];
    __shared__ uint32_t wtot[3][kDgThreads / 32];
    __shared__ uint4 s_h[kDgTile / 4], s_hin[kDgTile / 4];  // h[j] and h[j-R] of the tile's nodes
    // a row's bundles (start node, multiplicity, slot) on their way to coalesced stores
    __shared__ uint32_t s_bv[kDgThreads / 32][128], s_bm[kDgThreads / 32][128], s_bs[kDgThreads / 32][128];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    // tiles are handed out in launch order, so every predecessor of a tile is already running
    if (threadIdx.x == 0) {
        const uint32_t t = atomicAdd(ticket, 1u);
        s_tile = t;
        s_k0 = find_u32(dl.node_base, dl.ns, min(t * kDgTile, n_nodes - 1));
        s_k1 = find_u32(dl.node_base, dl.ns, min(t * kDgTile + kDgTile - 1, n_nodes - 1));
    }
    __syncthreads();
    const uint32_t tile = s_tile, k0 = s_k0, k1 = s_k1;
    const uint32_t R = dl.minlen;
    const uint32_t wbase = tile * kDgTile + warp * kDgWarpSpan;
    // this lane's 4 nodes of row r sit at s_h[row(r)] (each thread reads back only what it wrote)
    auto row = [&](int r) { return warp * (kDgWarpSpan / 4) + r * 32 + lane; };
    uint32_t hv[4], hin[4];
    auto fetch = [&](int r) {
        const uint4 a = s_h[row(r)], b = s_hin[row(r)];
        hv[0] = a.x; hv[1] = a.y; hv[2] = a.z; hv[3] = a.w;
        hin[0] = b.x; hin[1] = b.y; hin[2] = b.z; hin[3] = b.w;
    };
    {  // loads warp-striped (32 consecutive nodes per load), stored where the row layout reads them
        uint32_t* sh = reinterpret_cast<uint32_t*>(s_h) + warp * kDgWarpSpan;
        uint32_t* si = reinterpret_cast<uint32_t*>(s_hin) + warp * kDgWarpSpan;
        uint32_t lo = k0, hi = k1 + 1;  // the sample of the warp's first node
        const uint32_t vs = min(wbase, n_nodes - 1);
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (dl.node_base[mid] <= vs) lo = mid;
            else hi = mid;
        }
        uint32_t k = lo, nb = dl.node_base[k], nb1 = dl.node_base[k + 1], kb = dl.kbase[k];
        if (wbase + kDgWarpSpan <= nb1) {  // the warp's nodes lie in one sample (and before the end)
            const uint32_t j0 = wbase - nb + lane;
            const uint32_t* h = ghist + kb + j0;
#pragma unroll
            for (int m = 0; m < kDgWarpSpan / 32; ++m) {
                sh[m * 32 + lane] = h[m * 32];
                si[m * 32 + lane] = j0 + m * 32 >= R ? h[m * 32 - (int)R] : 0u;
            }
        } else {
#pragma unroll 4
            for (int m = 0; m < kDgWarpSpan / 32; ++m) {
                const uint32_t v = wbase + m * 32 + lane;
                uint32_t x = 0, y = 0;
                if (v < n_nodes) {
                    while (v >= nb1) {  // nodes only grow with m
                        ++k;
                        nb = dl.node_base[k];
                        nb1 = dl.node_base[k + 1];
                        kb = dl.kbase[k];
                    }
                    const uint32_t j = v - nb;
                    x = ghist[kb + j];
                    y = j >= R ? ghist[kb + j - R] : 0u;
                }
                sh[m * 32 + lane] = x;
                si[m * 32 + lane] = y;
            }
        }
        __syncwarp();
    }
    // lane offsets within the warp, row by row: coverage, and (out-arcs | in-arcs << 16)
    uint32_t rd[kDgRows], ro[kDgRows], wd = 0, wo = 0;
#pragma unroll
    for (int r = 0; r < kDgRows; ++r) {
        fetch(r);
        uint32_t sd = 0, so = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            sd += hv[q] - hin[q];
            so += (hv[q] != 0 ? 1u : 0u) + (hin[q] != 0 ? 0x10000u : 0u);
        }
        const uint32_t id = warp_incl_scan(sd), io = warp_incl_scan(so);
        rd[r] = wd + id - sd;
        ro[r] = wo + io - so;
        wd += __shfl_sync(0xffffffffu, id, 31);
        wo += __shfl_sync(0xffffffffu, io, 31);
    }
    if (lane == 0) {
        wtot[0][warp] = wd;
        wtot[1][warp] = wo;
    }
    __syncthreads();
    uint32_t offd = 0, offo = 0, totd = 0, toto = 0;
#pragma unroll
    for (int w = 0; w < kDgThreads / 32; ++w) {
        const uint32_t td = wtot[0][w], to = wtot[1][w];
        offd += w < (int)warp ? td : 0u;
        offo += w < (int)warp ? to : 0u;
        totd += td;
        toto += to;
    }
    if (warp < 3) {
        const uint32_t total = warp == 0 ? totd : warp == 1 ? (toto & 0xffffu) : (toto >> 16);
        const uint32_t p = lookback_prefix(status, tile * 4 + warp, 4, tile == 0, total, epoch);
        if (lane == 0) s_prefix[warp] = p;
    }
    __syncthreads();
    const uint32_t pd = s_prefix[0] + offd;
    const uint32_t po = s_prefix[1] + (offo & 0xffffu), pi = s_prefix[2] + (offo >> 16);
    // components start where the coverage rises from 0 (past the last node it stays 0)
    uint32_t rc[kDgRows], wc = 0;
#pragma unroll
    for (int r = 0; r < kDgRows; ++r) {
        fetch(r);
        uint32_t cov = pd + rd[r], sc = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint32_t covR = cov + hv[q] - hin[q];
            sc += (cov == 0 && covR != 0) ? 1u : 0u;
            cov = covR;
        }
        const uint32_t ic = warp_incl_scan(sc);
        rc[r] = wc + ic - sc;
        wc += __shfl_sync(0xffffffffu, ic, 31);
    }
    if (lane == 0) wtot[2][warp] = wc;
    __syncthreads();
    uint32_t offc = 0, totc = 0;
#pragma unroll
    for (int w = 0; w < kDgThreads / 32; ++w) {
        const uint32_t t = wtot[2][w];
        offc += w < (int)warp ? t : 0u;
        totc += t;
    }
    if (warp == 3) {
        const uint32_t p = lookback_prefix(status, tile * 4 + 3, 4, tile == 0, totc, epoch);
        if (lane == 0) s_prefix[3] = p;
    }
    __syncthreads();
    const uint32_t pc = s_prefix[3] + offc;
    unsigned long long src = 0;
    // (one row at a time: unrolled, the rows' stores would need 96 registers)
    auto pick = [](const uint32_t (&a)[kDgRows], int r) {
        uint32_t x = a[0];
#pragma unroll
        for (int i = 1; i < kDgRows; ++i) x = r == i ? a[i] : x;
        return x;
    };
#pragma unroll 1
    for (int r = 0; r < kDgRows; ++r) {
        fetch(r);
        const uint32_t v0 = wbase + r * 128 + lane * 4;
        const uint32_t rdr = pick(rd, r), ror = pick(ro, r), rcr = pick(rc, r);
        const uint32_t cov0 = pd + rdr, b0 = po + (ror & 0xffffu), ib0 = pi + (ror >> 16);
        // the node arrays, one at a time (16-byte stores; the end of the last tile one by one)
        auto put = [&](uint32_t* a, uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3, uint32_t last) {
            if (v0 + 3 < n_nodes) {
                *reinterpret_cast<uint4*>(a + v0) = make_uint4(x0, x1, x2, x3);
            } else {
                if (v0 <= last) a[v0] = x0;
                if (v0 + 1 <= last) a[v0 + 1] = x1;
                if (v0 + 2 <= last) a[v0 + 2] = x2;
                if (v0 + 3 <= last) a[v0 + 3] = x3;
            }
        };
        const uint32_t d0 = hv[0] - hin[0], d1 = hv[1] - hin[1], d2 = hv[2] - hin[2],
                       d3 = hv[3] - hin[3];
        const uint32_t c1 = cov0 + d0, c2 = c1 + d1, c3 = c2 + d2, c4 = c3 + d3;  // covR of each node
        put(reinterpret_cast<uint32_t*>(o.diff), d0, d1, d2, d3, n_nodes);
        put(o.excl, cov0, c1, c2, c3, n_nodes);
        auto dem = [&](uint32_t l, uint32_t rr) { return (uint32_t)((int32_t)min(l, M) - (int32_t)min(rr, M)); };
        put(reinterpret_cast<uint32_t*>(o.dem_v), dem(cov0, c1), dem(c1, c2), dem(c2, c3), dem(c3, c4), n_nodes - 1);
        auto nz = [&](uint32_t x) { return x != 0 ? 1u : 0u; };
        const uint32_t o1 = b0 + nz(hv[0]), o2 = o1 + nz(hv[1]), o3 = o2 + nz(hv[2]);
        put(o.outdeg, b0, o1, o2, o3, n_nodes);
        const uint32_t i1 = ib0 + nz(hin[0]), i2 = i1 + nz(hin[1]), i3 = i2 + nz(hin[2]);
        put(o.indeg, ib0, i1, i2, i3, n_nodes);
        // start node of the node's only in-arc
        auto src_of = [&](uint32_t hi, uint32_t v) { return hi ? v - R : 0xffffffffu; };
        put(o.in1, src_of(hin[0], v0), src_of(hin[1], v0 + 1), src_of(hin[2], v0 + 2),
            src_of(hin[3], v0 + 3), n_nodes);
        put(o.d_snap, kLabelInf, kLabelInf, kLabelInf, kLabelInf, n_nodes - 1);
        // per node: the record, the components, the bundle
        uint32_t slot[4], j[4];
        dg_locate(dl, k0, k1, v0, n_nodes, slot, j);
        uint32_t cov = cov0, b = b0, ib = ib0, cs = pc + rcr;
        const uint32_t rb = __shfl_sync(0xffffffffu, b0, 0);  // the row's first bundle
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint32_t v = v0 + q, h = hv[q], hi = hin[q];
            const uint32_t covR = cov + h - hi;
            const int32_t dm = (int32_t)min(cov, M) - (int32_t)min(covR, M);
            const bool start = cov == 0 && covR != 0;
            if (v < n_nodes) {
                uint4* nr = reinterpret_cast<uint4*>(&o.node[v]);
                const bool inf = !(in_first && hi);
                nr[0] = make_uint4(inf ? kLabelInf : v - R, inf ? 0u : ib, (uint32_t)(dm < 0 ? -dm : 0), 0u);
                nr[1] = make_uint4((uint32_t)(dm > 0 ? dm : 0), 0u, b, ib);
                if (o.cov_capped) o.cov_capped[v] = min(covR, M);
                if (o.demand) o.demand[v] = dm;
                if (dm < 0) src += (unsigned long long)(-dm);
                // components are disjoint runs: the end at v closes the one opened last
                if (start) o.comp_lo[cs] = v;
                if (cov != 0 && covR == 0) o.comp_hi[cs - 1] = v;
                if (h) {
                    s_bv[warp][b - rb] = v;
                    s_bm[warp][b - rb] = h;
                    s_bs[warp][b - rb] = slot[q];
                }
            } else if (v == n_nodes) {  // sentinel record; the counts stay on the device
                uint4* nr = reinterpret_cast<uint4*>(&o.node[v]);
                nr[0] = make_uint4(0u, 0u, 0u, 0u);
                nr[1] = make_uint4(0u, 0u, b, ib);
                *o.n_bundles = b;
                *o.n_comp = cs;
            }
            cs += start ? 1u : 0u;
            b += h != 0 ? 1u : 0u;
            ib += hi != 0 ? 1u : 0u;
            cov = covR;
        }
        // the row's bundles are consecutive: written by consecutive lanes (one lane per bundle and
        // its own 4-node group scattered every store over 16-32 sectors)
        const uint32_t nrow = __shfl_sync(0xffffffffu, b, 31) - rb;
        __syncwarp();
        for (uint32_t x = lane; x < nrow; x += 32) {
            const uint32_t bb = rb + x, v = s_bv[warp][x];
            reinterpret_cast<uint4*>(o.bund)[bb] = make_uint4(v + R, s_bm[warp][x], 0u, v);  // {t, mult, f, s}
            o.b_t[bb] = v + R;
            o.b_slot[bb] = s_bs[warp][x];
            o.ident[bb] = bb;
            o.in_src[bb] = v;
        }
        __syncwarp();
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) src += __shfl_xor_sync(0xffffffffu, src, s);
    if (lane == 0 && src) {
        atomicAdd(o.fstar, src);
        atomicAdd(o.res_supply, src);
    }
    if (threadIdx.x == 0 && tile == n_tiles - 1) *ticket = 0;  // every ticket is out by now
}

// ---- K5 direct ---------------------------------------------------------------------------------
// "A bundle with flow f keeps its f lowest-index reads" (select.cuh) without a sorted read order.
// Push-relabel saturates most bundles it uses, so after K3 a key is in one of three states:
//   f == 0        none of its reads is kept                                       (code 0)
//   f == mult     all of its reads are kept — no order needed                     (code 1)
//   0 < f < mult  "partial": the f lowest of its mult read indices are kept       (code 2)
// k_direct_classify writes the 2-bit code of every key (16 per word; a 30 kb sample's table is
// 7.5 KB) and gives every partial bundle a segment of mult slots in a candidate buffer.
// k_direct_mark streams the reads' starts once more, in parallel parts like the histogram: code 1
// sets the kept bit, code 2 appends the read index to the bundle's segment.  k_direct_partial then
// ranks each partial bundle's candidates, one warp per bundle whatever its size.  If the candidates
// do not fit their buffer, ctl[2] is raised and the host repeats the selection with the buffer grown
// to ctl[1].
constexpr uint32_t kSatCode = 1, kPartCode = 2;
// 512 threads x 3 CTAs per SM at 40 registers: the kernel is bound by neither issue slots nor HBM
// but by its stalls per instruction, so more resident warps pay — 1.27 ms with one CTA of 1024
// threads (48 registers, half occupancy), 1.14 ms this way (config 5)
constexpr int kDmThreads = 512;
constexpr int kDmCtasPerSm = 3;
constexpr uint32_t kDmSplit = 3;

// ctl: [0] number of partial bundles, [1] candidate slots handed out, [2] flags: the mark and
// ranking kernels do nothing when any is set — 2 the candidates do not fit cand_cap (the host grows
// the buffer and repeats the selection), 4 K2 counted bad reads (the call fails; the mark kernels
// do not re-validate)
__global__ void __launch_bounds__(256)
k_direct_classify(const BundleRec* __restrict__ bund, const uint32_t* __restrict__ b_slot,
                  uint32_t* __restrict__ ghist, uint32_t* __restrict__ kstat,
                  uint32_t* __restrict__ pb_off, uint32_t* __restrict__ pb_f,
                  uint32_t* __restrict__ pb_fill, uint32_t* __restrict__ ctl,
                  const uint32_t* __restrict__ B_dev, uint32_t cand_cap,
                  const uint32_t* __restrict__ stats) {
    __shared__ uint32_t tot_n, tot_m, base_n, base_m;
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t B = *B_dev;
    if (b == 0 && (stats[2] | stats[3])) atomicOr(&ctl[2], 4u);
    uint32_t mult = 0, f = 0;
    if (b < B) {
        const uint4 r = reinterpret_cast<const uint4*>(bund)[b];  // {t, mult, f, s}
        mult = r.y;
        f = r.z;
    }
    const bool partial = f != 0 && f < mult;
    // one pair of global atomics per block hands out bundle ids and candidate segments
    const uint32_t my_n = block_excl_scan(partial ? 1u : 0u, &tot_n);
    const uint32_t my_m = block_excl_scan(partial ? mult : 0u, &tot_m);
    if (threadIdx.x == 0 && tot_n) {
        base_n = atomicAdd(&ctl[0], tot_n);
        base_m = atomicAdd(&ctl[1], tot_m);
        if ((unsigned long long)base_m + tot_m > cand_cap) atomicOr(&ctl[2], 2u);
    }
    __syncthreads();
    if (f == 0) return;
    const uint32_t slot = b_slot[b];
    uint32_t code = kSatCode;
    if (partial) {
        code = kPartCode;
        const uint32_t pid = base_n + my_n;
        const uint32_t o = base_m + my_m;
        pb_off[pid] = o;
        pb_f[pid] = f;
        pb_fill[pid] = 0;
        ghist[slot] = pid;
    }
    atomicOr(&kstat[slot >> 4], code << (2 * (slot & 15)));
}

// Reads of partial bundles are rare (~2 %) but each costs a chain of dependent global accesses
// (bundle id -> segment -> atomic slot -> store).  Taken inline that chain stalls the warp once per
// hit; instead every warp parks its hits (key, read index) in its own shared-memory queue and
// drains the queue 32 entries at a time when it is nearly full and at the end of the part.
// The kernel was issue-bound in its first version (ncu: 43 instructions per read, 62 % issue
// slots busy): the codes are expanded to one BYTE per key in shared memory (one LDS per read),
// indices are 32-bit offsets from the part start, and nothing is re-validated (K2 already failed
// the call on any bad read).
// ncu of the second version: issue slots 50 % busy, long-scoreboard stalls, 3.6 TB/s.  Neither
// doubling the loads in flight (8 x 16 B per thread: 1.24 -> 1.21 ms) nor draining 4 x 32 entries
// per chain of dependent accesses (1.21 -> 1.39 ms, register pressure) nor keeping the next batch's
// loads in flight while this one is looked up (1.27 -> 1.32 ms, 64 registers) helped, and parking
// the hits of a group warp-wide (ballots give every hit its queue slot, register counter, no
// divergent per-hit path: 1.14 -> 1.27 ms) was slower than letting the few lanes with a hit diverge; what remains is the
// scattered traffic of 20 M candidates.  The queue does not have to hold a whole round: a hit that
// finds it full takes the slow chain inline (only adversarial inputs get there).
// Switching the parking off altogether (wrong results, timing only) takes 25 % off the kernel and
// the kept-bit reductions cost nothing: what remains is one random shared-memory lookup per read,
// 3.5 reads per clock and SM — the kernel handles 1.0 T reads/s where the histogram, at the HBM
// bound with twice the bytes per read, handles 0.8 T.
constexpr int kDmUnroll = 4;                                    // 512 reads per warp and round
constexpr uint32_t kDmQueue = 256;                              // entries per warp
constexpr uint32_t kDmQueueBytes = (kDmThreads / 32) * kDmQueue * 8;

__global__ void __launch_bounds__(kDmThreads, kDmCtasPerSm)
k_direct_mark(const uint32_t* __restrict__ S, DirectLayout dl, uint32_t n_items,
              uint32_t* __restrict__ work_counter,
              const uint32_t* __restrict__ ghist, const uint32_t* __restrict__ kstat,
              const uint32_t* __restrict__ pb_off, uint32_t* __restrict__ pb_fill,
              uint32_t* __restrict__ cand, const uint32_t* __restrict__ ctl,
              uint32_t* __restrict__ bitmap, unsigned long long* __restrict__ totals) {
    extern __shared__ __align__(16) uint32_t dm_smem[];
    uint2* wq = reinterpret_cast<uint2*>(dm_smem) + (threadIdx.x >> 5) * kDmQueue;  // this warp's queue
    uint32_t* st32 = dm_smem + kDmQueueBytes / 4;
    const uint8_t* st = reinterpret_cast<const uint8_t*>(st32);  // code of every key of the sample
    __shared__ uint32_t s_item;
    __shared__ uint32_t wcnt[kDmThreads / 32];
    if (ctl[2]) return;
    const uint32_t tid = threadIdx.x, lane = lane_id(), warp = threadIdx.x >> 5;
    constexpr int kU = kDmUnroll;
    uint32_t kept = 0;
    if (lane == 0) wcnt[warp] = 0;
    __syncwarp();
    for (;;) {
        if (tid == 0) s_item = atomicAdd(work_counter, 1u);
        __syncthreads();
        // the histogram's parts are cut in kDmSplit pieces each: three CTAs per SM share the work
        // counter here, and with whole parts the last of ~3.5 items per CTA set the pace
        if (s_item >= n_items * kDmSplit) break;
        const uint32_t item = s_item / kDmSplit, sub = s_item % kDmSplit;
        const uint32_t k = find_u32(dl.item_off, dl.ns, item);
        const uint32_t parts = dl.item_off[k + 1] - dl.item_off[k];
        const uint32_t p = item - dl.item_off[k];
        const uint64_t o0 = dl.off[k], o1 = dl.off[k + 1];
        const uint64_t plen = (((o1 - o0) + parts - 1) / parts + 3) & ~3ull;
        const uint64_t pa = min(o0 + p * plen, o1), pb_ = min(pa + plen, o1);
        const uint64_t slen = (((pb_ - pa) + kDmSplit - 1) / kDmSplit + 3) & ~3ull;
        const uint64_t a = min(pa + sub * slen, pb_);
        const uint64_t b = min(a + slen, pb_);
        const uint32_t kb = dl.kbase[k];
        const uint32_t kk = dl.kbase[k + 1] - kb;
        for (uint32_t i = tid; i < (kk >> 4); i += kDmThreads) {  // 16 two-bit codes -> 16 bytes
            const uint32_t w = kstat[(kb >> 4) + i];
            uint32_t o[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t x = w >> (8 * q);
                o[q] = (x & 3u) | ((x & 12u) << 6) | ((x & 48u) << 12) | ((x & 192u) << 18);
            }
            reinterpret_cast<uint4*>(st32)[i] = make_uint4(o[0], o[1], o[2], o[3]);
        }
        __syncthreads();
        // the key is the start: in range on validated input; never read past the table
        auto key_of = [&](uint32_t s) { return min(s, kk - 1); };
        // converged warp: hand the parked reads to their bundles' candidate segments
        auto park = [&](uint32_t key, uint32_t g) {
            const uint32_t pid = ghist[kb + key];
            const uint32_t pos = atomicAdd(&pb_fill[pid], 1u);
            cand[pb_off[pid] + pos] = g;
        };
        auto drain = [&](uint32_t min_pending) {
            __syncwarp();
            const uint32_t n = min(wcnt[warp], kDmQueue);
            if (n <= min_pending) return;
            for (uint32_t i = lane; i < n; i += 32) {
                const uint2 q = wq[i];
                park(q.x, q.y);
            }
            __syncwarp();
            if (lane == 0) wcnt[warp] = 0;
            __syncwarp();
        };
        // rare path: some read of the group carries a key with flow
        auto hit = [&](uint64_t g, uint32_t key, uint32_t code) -> uint32_t {
            if (code == kPartCode) {
                const uint32_t slot = atomicAdd(&wcnt[warp], 1u);
                if (slot < kDmQueue) wq[slot] = make_uint2(key, (uint32_t)g);
                else park(key, (uint32_t)g);  // queue full: take the chain now
            }
            return code == kSatCode ? 1u : 0u;
        };
        if (a < b) {
            const uint64_t a4 = min((uint64_t)((a + 3) & ~3ull), b), b4 = max((uint64_t)(b & ~3ull), a4);
            for (int side = 0; side < 2; ++side) {  // unaligned head and tail
                const uint64_t lo = side ? b4 : a, hi = side ? b : a4;
                if (tid < hi - lo) {
                    const uint64_t g = lo + tid;
                    const uint32_t key = key_of(S[g]);
                    if (hit(g, key, st[key])) {
                        atomicOr(&bitmap[g >> 5], 1u << (g & 31));
                        ++kept;
                    }
                }
            }
            const uint4* S4 = reinterpret_cast<const uint4*>(S) + a4 / 4;
            auto mark4 = [&](uint32_t j, const uint4& s) {
                const uint32_t k0 = key_of(s.x), k1 = key_of(s.y), k2 = key_of(s.z), k3 = key_of(s.w);
                const uint32_t c0 = st[k0], c1 = st[k1], c2 = st[k2], c3 = st[k3];
                if ((c0 | c1 | c2 | c3) == 0) return;  // 94 % of the groups
                const uint64_t g = a4 + 4ull * j;
                const uint32_t nib = hit(g, k0, c0) | hit(g + 1, k1, c1) << 1 | hit(g + 2, k2, c2) << 2 |
                                     hit(g + 3, k3, c3) << 3;
                if (nib) {
                    atomicOr(&bitmap[g >> 5], nib << (g & 31));
                    kept += __popc(nib);
                }
            };
            // the trip count is the same for every lane of a warp (the drain needs the warp
            // converged): lanes past the end process nothing
            const uint32_t jend = (uint32_t)((b4 - a4) / 4);
            for (uint32_t jw = warp * 32; jw < jend; jw += kU * kDmThreads) {
                uint4 s[kU];
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    const uint32_t j = jw + lane + u * kDmThreads;
                    if (j < jend) s[u] = ld_stream4(S4 + j);
                }
#pragma unroll
                for (int u = 0; u < kU; ++u) {
                    const uint32_t j = jw + lane + u * kDmThreads;
                    if (j < jend) mark4(j, s[u]);
                }
                drain(kDmQueue / 2);
            }
        }
        drain(0);  // the next part may belong to another sample
        __syncthreads();
    }
    kept = __reduce_add_sync(0xffffffffu, kept);
    if (lane == 0 && kept) atomicAdd(&totals[1], (unsigned long long)kept);
}

// Partial bundles: keep the f lowest of a bundle's candidate read indices.  Up to 16 candidates (the
// common case with segments: config 4 has 1.7 M partial bundles of ~10 reads) take HALF a warp — two
// bundles per warp and step, ranked against each other through 16 shuffles (0.29 -> 0.20 ms there);
// larger ones get the whole warp: up to 32 candidates the same way, beyond that the f-th lowest index
// by bisection on the index value (count = ballots over the candidates, in registers up to 128 of
// them).  (Packing a bundle's segment start and fill count into one 64-bit word, parked with one
// 64-bit atomic instead of a load and a 32-bit atomic, was measured too: the mark kernel of config 4
// went 0.71 -> 0.79 ms.  Not kept.)
// HALF = false (bundles of whole 30 kb samples hold ~67 reads: config 5): one warp per bundle only.
template <bool HALF>
__global__ void __launch_bounds__(256)
k_direct_partial(const uint32_t* __restrict__ pb_off, const uint32_t* __restrict__ pb_f,
                 const uint32_t* __restrict__ pb_fill, const uint32_t* __restrict__ cand,
                 const uint32_t* __restrict__ ctl, uint32_t* __restrict__ bitmap,
                 unsigned long long* __restrict__ totals) {
    if (ctl[2]) return;
    const uint32_t n_partial = ctl[0];
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t lane = lane_id();
    uint32_t kept = 0;
    auto keep = [&](uint32_t v) {  // a read cut in two by a segment cut can be chosen twice
        const uint32_t bit = 1u << (v & 31);
        kept += (atomicOr(&bitmap[v >> 5], bit) & bit) ? 0u : 1u;
    };
    constexpr int kReg = 4;
    // the whole warp on one bundle
    auto whole_warp = [&](uint32_t pid, uint32_t n) {
        const uint32_t* c = cand + pb_off[pid];
        const uint32_t f = pb_f[pid];
        if (n <= 32) {
            const uint32_t x = lane < n ? c[lane] : 0xffffffffu;
            uint32_t rank = 0;
            for (uint32_t j = 0; j < n; ++j) rank += __shfl_sync(0xffffffffu, x, j) < x;
            if (lane < n && rank < f) keep(x);
            return;
        }
        uint32_t x[kReg];
        uint32_t mn = 0xffffffffu, mx = 0;
#pragma unroll
        for (int r = 0; r < kReg; ++r) {
            x[r] = r * 32 + lane < n ? c[r * 32 + lane] : 0xffffffffu;  // padding is never counted
            if (r * 32 + lane < n) {
                mn = min(mn, x[r]);
                mx = max(mx, x[r]);
            }
        }
        for (uint32_t i = kReg * 32 + lane; i < n; i += 32) {
            mn = min(mn, c[i]);
            mx = max(mx, c[i]);
        }
        uint32_t lo = __reduce_min_sync(0xffffffffu, mn), hi = __reduce_max_sync(0xffffffffu, mx);
        while (lo < hi) {  // smallest T with #{c <= T} >= f  (indices are distinct)
            const uint32_t mid = lo + (hi - lo) / 2;
            uint32_t cnt = 0;
#pragma unroll
            for (int r = 0; r < kReg; ++r) cnt += __popc(__ballot_sync(0xffffffffu, x[r] <= mid));
            if (n > kReg * 32) {
                uint32_t mine = 0;
                for (uint32_t i = kReg * 32 + lane; i < n; i += 32) mine += c[i] <= mid;
                cnt += __reduce_add_sync(0xffffffffu, mine);
            }
            if (cnt >= f) hi = mid;
            else lo = mid + 1;
        }
#pragma unroll
        for (int r = 0; r < kReg; ++r)
            if (x[r] <= lo) keep(x[r]);  // the padding value is above every index
        for (uint32_t i = kReg * 32 + lane; i < n; i += 32)
            if (c[i] <= lo) keep(c[i]);
    };
    if (!HALF) {
        for (uint32_t pid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; pid < n_partial; pid += warps)
            whole_warp(pid, pb_fill[pid]);
    }
    const uint32_t half = lane >> 4, hl = lane & 15u;
    for (uint32_t p0 = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 2; HALF && p0 < n_partial;
         p0 += 2 * warps) {
        const uint32_t pid = p0 + half;
        const bool valid = pid < n_partial;
        const uint32_t n = valid ? pb_fill[pid] : 0u;
        const bool small = valid && n <= 16;
        if (__any_sync(0xffffffffu, small)) {  // (config 5's bundles hold ~67 candidates: never)
            const uint32_t f = small ? pb_f[pid] : 0u;
            const uint32_t x = small && hl < n ? cand[pb_off[pid] + hl] : 0xffffffffu;
            uint32_t rank = 0;
#pragma unroll
            for (uint32_t j = 0; j < 16; ++j) rank += __shfl_sync(0xffffffffu, x, (lane & 16u) | j) < x;
            if (small && hl < n && rank < f) keep(x);
        }
        // bundles beyond half a warp: one after the other, all lanes
        const uint32_t big = __ballot_sync(0xffffffffu, valid && !small && hl == 0);
        const uint32_t n0 = __shfl_sync(0xffffffffu, n, 0), n1 = __shfl_sync(0xffffffffu, n, 16);
        if (big & 1u) whole_warp(p0, n0);
        if (big & 0x10000u) whole_warp(p0 + 1, n1);
    }
    kept = __reduce_add_sync(0xffffffffu, kept);
    if (lane == 0 && kept) atomicAdd(&totals[1], (unsigned long long)kept);
}

// ---- the same idea with the histogram in global memory ------------------------------------------
// When the reads have several lengths (config 2), a sample does not fit one SM, or the reference is
// cut into segments (config 4), the counters live in global memory instead: up to kGDirectMaxKeys
// of them (96 MB, resident in the 126 MB L2), one RED.ADD per read (tools/hist_probe.cu: 170 G
// keys/s) and a second one for the right part of a read that crosses a segment cut.  Keys are the
// sort path's keys, (virtual fake start id, length) — graph.cuh: ReadKeys / VLayout — so bundles
// come out in the same order with the same clamping to the segment's node range.
constexpr unsigned long long kGDirectMaxKeys = 24ull << 20;
constexpr int kGdThreads = 256;
constexpr int kGdItems = 8;
constexpr int kGdTile = kGdThreads * kGdItems;

struct GDirectLayout {
    VLayout vl;
    uint32_t nlen, minlen, maxlen;
};

// largest k with vs[k].vbase <= vid
__device__ __forceinline__ uint32_t find_vsample(const VLayout& vl, uint32_t vid) {
    uint32_t lo = 0, hi = vl.n_samples;
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (vl.vs[mid].vbase <= vid) lo = mid;
        else hi = mid;
    }
    return lo;
}

// per block: a tile of consecutive reads; sample lookups once per block when the tile lies in one
// sample.  f(i, sample, start, end) is called for every read of the tile by the thread that owns it
// (thread t owns reads base + q*256 + t: a warp covers 32 consecutive reads per q).
template <typename F>
__device__ __forceinline__ void gd_for_tile(const uint32_t* __restrict__ S,
                                            const uint32_t* __restrict__ E, size_t n,
                                            const VLayout& vl, F f) {
    __shared__ uint32_t krange[2];
    const size_t base = (size_t)blockIdx.x * kGdTile;
    if (threadIdx.x == 0) {
        const size_t last = min(base + kGdTile, n) - 1;
        krange[0] = vl.n_samples == 1 ? 0 : find_sample(vl.off, vl.n_samples, base);
        krange[1] = vl.n_samples == 1 ? 0 : find_sample(vl.off, vl.n_samples, last);
    }
    __syncthreads();
    const uint32_t k0 = krange[0];
    const bool one = k0 == krange[1];
    const VSample v0 = vl.vs[k0];
    uint32_t s[kGdItems], e[kGdItems];
#pragma unroll
    for (int q = 0; q < kGdItems; ++q) {
        const size_t i = base + (size_t)q * kGdThreads + threadIdx.x;
        const size_t ii = i < n ? i : base;
        s[q] = ld_stream(S + ii);
        e[q] = ld_stream(E + ii);
    }
#pragma unroll
    for (int q = 0; q < kGdItems; ++q) {
        const size_t i = base + (size_t)q * kGdThreads + threadIdx.x;
        const bool in = i < n;
        const VSample v = (one || !in) ? v0 : vl.vs[find_sample(vl.off, vl.n_samples, i)];
        f(q, i, in, v, s[q], e[q]);
    }
}

__global__ void __launch_bounds__(kGdThreads)
k_gdirect_hist(const uint32_t* __restrict__ S, const uint32_t* __restrict__ E, size_t n,
               GDirectLayout gl, uint32_t* __restrict__ ghist, uint32_t* __restrict__ stats) {
    uint32_t bad_range = 0, bad_hint = 0, n_cross = 0;
    gd_for_tile(S, E, n, gl.vl, [&](int, size_t, bool in, const VSample& v, uint32_t s, uint32_t e) {
        if (!in) return;
        if (!read_in_range(s, e, v.L)) {
            ++bad_range;
            return;
        }
        const uint32_t len = e - s + 1;
        if (len < gl.minlen || len > gl.maxlen) {
            ++bad_hint;
            return;
        }
        const uint32_t dl = len - gl.minlen;
        atomicAdd(&ghist[gl.vl.fake_primary(v, s) * gl.nlen + dl], 1u);
        if (gl.vl.crosses(v, s, e)) {
            atomicAdd(&ghist[gl.vl.fake_right(v, s, e) * gl.nlen + dl], 1u);
            ++n_cross;
        }
    });
    bad_range = __reduce_add_sync(0xffffffffu, bad_range);
    bad_hint = __reduce_add_sync(0xffffffffu, bad_hint);
    n_cross = __reduce_add_sync(0xffffffffu, n_cross);
    if (lane_id() == 0) {
        if (bad_range) atomicAdd(&stats[2], bad_range);
        if (bad_hint) atomicAdd(&stats[3], bad_hint);
        if (n_cross) atomicAdd(&stats[4], n_cross);  // reads cut in two (gds_result.n_arc_items)
    }
}

// bundles = non-zero counters in key order; decoding as k_bundle_fill (graph.cuh)
__global__ void __launch_bounds__(kDkThreads)
k_gdirect_bundles(const uint32_t* __restrict__ ghist, uint32_t ktot, GDirectLayout gl,
                  const uint32_t* __restrict__ tile_offs, BundleRec* __restrict__ bund,
                  uint32_t* __restrict__ b_t, uint32_t* __restrict__ b_slot,
                  uint32_t* __restrict__ in_bid /* identity when nlen == 1, else null */,
                  int32_t* __restrict__ diff, uint32_t* __restrict__ outdeg,
                  uint32_t* __restrict__ indeg, int32_t* __restrict__ odiff) {
    __shared__ uint32_t total;
    const uint32_t i = (blockIdx.x * kDkThreads + threadIdx.x) * 4;
    uint32_t cnt[4] = {0, 0, 0, 0};
    if (i < ktot) {
        const uint4 q = reinterpret_cast<const uint4*>(ghist)[i / 4];
        cnt[0] = q.x;
        cnt[1] = q.y;
        cnt[2] = q.z;
        cnt[3] = q.w;
    }
    const uint32_t c = (cnt[0] != 0) + (cnt[1] != 0) + (cnt[2] != 0) + (cnt[3] != 0);
    uint32_t b = block_excl_scan(c, &total) + tile_offs[blockIdx.x];
    if (c == 0) return;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        if (!cnt[q]) continue;
        const uint32_t key = i + q;
        const uint32_t fake = key / gl.nlen;
        const uint32_t len = gl.minlen + key % gl.nlen;
        const VSample v = gl.vl.vs[find_vsample(gl.vl, fake)];
        uint32_t first, last;
        gl.vl.seg_range(v, fake, first, last);
        const uint32_t s = max(fake, first);
        const uint32_t t = min(fake + len, last);
        const uint32_t mult = cnt[q];
        reinterpret_cast<uint4*>(bund)[b] = make_uint4(t, mult, 0u, s);
        b_t[b] = t;
        b_slot[b] = key;
        if (in_bid) in_bid[b] = b;
        atomicAdd(&diff[s], (int32_t)mult);
        atomicAdd(&diff[t], -(int32_t)mult);
        atomicAdd(&outdeg[s], 1u);
        atomicAdd(&indeg[t], 1u);
        if (odiff) {
            atomicAdd(&odiff[gl.vl.to_orig(v, s)], (int32_t)mult);
            atomicAdd(&odiff[gl.vl.to_orig(v, t)], -(int32_t)mult);
        }
        ++b;
    }
}

// K5: codes from the global 2-bit table (L1/L2 resident), one kept-bitmap word per warp and q.
// With segments of a long reference a third of the reads belong to partial bundles (config 4:
// 19 M of 50 M), so the candidate chain (bundle id -> segment, slot -> store) is staged across the
// thread's 8 reads: all lookups of a stage are in flight together.  The right part of a read that
// crosses a cut (1 % of the reads) takes the chain inline.
__global__ void __launch_bounds__(kGdThreads)
k_gdirect_mark(const uint32_t* __restrict__ S, const uint32_t* __restrict__ E, size_t n,
               GDirectLayout gl, const uint32_t* __restrict__ ghist,
               const uint32_t* __restrict__ kstat, const uint32_t* __restrict__ pb_off,
               uint32_t* __restrict__ pb_fill, uint32_t* __restrict__ cand,
               uint32_t* __restrict__ bitmap, unsigned long long* __restrict__ totals,
               const uint32_t* __restrict__ ctl) {
    __shared__ uint32_t krange[2];
    if (ctl[2]) return;
    const VLayout& vl = gl.vl;
    const size_t base = (size_t)blockIdx.x * kGdTile;
    if (threadIdx.x == 0) {
        const size_t last = min(base + kGdTile, n) - 1;
        krange[0] = vl.n_samples == 1 ? 0 : find_sample(vl.off, vl.n_samples, base);
        krange[1] = vl.n_samples == 1 ? 0 : find_sample(vl.off, vl.n_samples, last);
    }
    __syncthreads();
    const uint32_t k0 = krange[0];
    const bool one = k0 == krange[1];
    const VSample v0 = vl.vs[k0];
    constexpr uint32_t kNone = 0xffffffffu;
    uint32_t s[kGdItems], e[kGdItems], key[kGdItems], code[kGdItems];
#pragma unroll
    for (int q = 0; q < kGdItems; ++q) {
        const size_t i = base + (size_t)q * kGdThreads + threadIdx.x;
        const size_t ii = i < n ? i : base;
        s[q] = ld_stream(S + ii);
        e[q] = ld_stream(E + ii);
    }
    auto sample_of = [&](size_t i) { return one ? v0 : vl.vs[find_sample(vl.off, vl.n_samples, i)]; };
    uint32_t cross = 0;  // bit q: the read crosses a segment cut
#pragma unroll
    for (int q = 0; q < kGdItems; ++q) {
        const size_t i = base + (size_t)q * kGdThreads + threadIdx.x;
        key[q] = kNone;
        if (i < n) {
            const VSample v = sample_of(i);
            const uint32_t dl = e[q] - s[q] + 1 - gl.minlen;
            if (s[q] <= e[q] && e[q] < v.L && dl < gl.nlen) {  // validated by K2; never index with garbage
                key[q] = vl.fake_primary(v, s[q]) * gl.nlen + dl;
                if (vl.crosses(v, s[q], e[q])) cross |= 1u << q;
            }
        }
    }
#pragma unroll
    for (int q = 0; q < kGdItems; ++q)
        code[q] = key[q] != kNone ? (kstat[key[q] >> 4] >> (2 * (key[q] & 15))) & 3u : 0u;
    uint32_t pid[kGdItems], off[kGdItems], pos[kGdItems];
#pragma unroll
    for (int q = 0; q < kGdItems; ++q)
        if (code[q] == kPartCode) pid[q] = ghist[key[q]];
#pragma unroll
    for (int q = 0; q < kGdItems; ++q)
        if (code[q] == kPartCode) {
            off[q] = pb_off[pid[q]];
            pos[q] = atomicAdd(&pb_fill[pid[q]], 1u);
        }
    uint32_t kept = 0;
#pragma unroll
    for (int q = 0; q < kGdItems; ++q) {
        const size_t i = base + (size_t)q * kGdThreads + threadIdx.x;
        if (code[q] == kPartCode) cand[off[q] + pos[q]] = (uint32_t)i;
        bool keep = code[q] == kSatCode;
        if (cross >> q & 1) {  // right part: its own bundle
            const VSample v = sample_of(i);
            const uint32_t k2 = vl.fake_right(v, s[q], e[q]) * gl.nlen + (e[q] - s[q] + 1 - gl.minlen);
            const uint32_t c2 = (kstat[k2 >> 4] >> (2 * (k2 & 15))) & 3u;
            if (c2 == kPartCode) {
                const uint32_t p2 = ghist[k2];
                cand[pb_off[p2] + atomicAdd(&pb_fill[p2], 1u)] = (uint32_t)i;
            }
            keep |= c2 == kSatCode;
        }
        // tiles start at multiples of 32 reads: the 32 lanes of a warp hold one bitmap word
        const uint32_t w = __ballot_sync(0xffffffffu, keep);
        if (lane_id() == 0 && w) {
            atomicOr(&bitmap[i >> 5], w);
            kept += __popc(w);
        }
    }
    kept = __reduce_add_sync(0xffffffffu, kept);
    if (lane_id() == 0 && kept) atomicAdd(&totals[1], (unsigned long long)kept);
}

}  // namespace gds
