// sweep.cuh — K3': the minimum-cardinality solve (gds_params.algorithm = 1).
//
// What the reference's `mcp-cpu` computes with OR-Tools' cost-scaling min-cost flow
// (mcp_cpu_cost_scaling_solver.cpp:33-67: the quasi-MCP network with cost 1 on every read arc and 0 on
// the back arcs, so the optimum is the FEWEST reads with cov_S >= min(cov, M)) has, on this network,
// a direct exact algorithm: greedy interval multicover — sweep the positions left to right and, on
// a deficit, take the available read that ends farthest (SURVEY §8c: equal to the network-simplex
// optimum on 300/300 random instances; oracle/gds_oracle.cpp: orc_greedy_multicover).  Any set S with
// cov_S >= min(cov, M) is also a maximum flow of the quasi-MCP network (flow 1 on S, back-arc flow
// cov_S - cov'), so F*, demand and capped coverage are the same as on the push-relabel path; only the
// kept set differs — it is the smallest one.
//
// On the bundled graph of K2 the sweep needs no priority queue: reads that have started are pooled
// BY END NODE (two reads with one end are interchangeable for covering the current position), the
// pool is a ring of maxlen+1 counters in shared memory, "farthest end" is a pointer that only moves
// down until new reads arrive.  Afterwards the reads taken with end node t are handed to the bundles
// ending at t in in-CSR order (earliest start first: a read with the same end and an earlier start
// covers a superset), and K5 keeps the lowest-index reads of every bundle as always.
//
// One WARP per component (a sweep is sequential), every component of the call concurrent: lanes
// fetch 32 positions' CSR rows and coverage with one coalesced load, the chunk's bundle records are
// staged in shared memory with cp.async one chunk ahead, lane-parallel arrivals, warp-uniform picks.
// Deterministic; restated on the CPU in oracle/gds_oracle.cpp: orc_sweep_solve.
#pragma once
#include "graph.cuh"

namespace gds {

struct SweepGraph {
    const uint32_t* excl;     // [n_nodes + 1] coverage left of node v
    const int32_t* diff;      // [n_nodes + 1] coverage change at node v
    const uint32_t* out_ptr;  // [n_nodes + 1]
    const BundleRec* bund;    // [B] {t, mult, f, s}
    uint32_t* taken;          // [n_nodes + 1] reads taken per END node (zeroed by the caller)
};

constexpr int kSweepWarps = 4;  // warps (= components in flight) per CTA

__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(a), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.wait_all;" ::: "memory");
}

// W: ring size (power of two, > longest bundle in nodes); CAP: staged bundle records per chunk.
// The sweep itself is sequential: lane 0 walks the positions of a chunk with everything it needs in
// shared memory and no warp-level synchronisation inside the walk (the first version kept all 32
// lanes in step through shuffles and __syncwarp: 630 clocks per position; this one ~100); the other
// lanes fetch — rows and coverage of the next chunk with one coalesced load, its bundle records
// with cp.async — while lane 0 walks.
template <int W, int CAP>
__global__ void __launch_bounds__(kSweepWarps * 32)
k_sweep(SweepGraph G, const uint32_t* __restrict__ comp_lo, const uint32_t* __restrict__ comp_hi,
        const uint32_t* __restrict__ n_comp_dev, uint32_t M, uint32_t* work_counter,
        unsigned long long* __restrict__ fail /* += positions whose pool ran dry (never) */) {
    extern __shared__ __align__(16) unsigned char sw_raw[];
    const uint32_t warp = threadIdx.x >> 5, lane = lane_id();
    // per warp: pool[W], pend[W], stage[2][CAP] of {t, mult}, rows[2][34], need[2][32]
    constexpr uint32_t kWords = 2 * W + 4 * CAP + 2 * 34 + 2 * 32;
    uint32_t* pool = reinterpret_cast<uint32_t*>(sw_raw) + (size_t)warp * kWords;
    uint32_t* pend = pool + W;
    uint2* stage = reinterpret_cast<uint2*>(pend + W);
    uint32_t* rows = reinterpret_cast<uint32_t*>(stage + 2 * CAP);
    uint32_t* needs = rows + 2 * 34;
    const uint32_t n_comp = *n_comp_dev;
    for (;;) {
        uint32_t c = 0;
        if (lane == 0) c = atomicAdd(work_counter, 1u);
        c = __shfl_sync(0xffffffffu, c, 0);
        if (c >= n_comp) break;
        const uint32_t lo = comp_lo[c], hi = comp_hi[c];
        for (uint32_t i = lane; i < 2 * W; i += 32) pool[i] = 0;  // pool and pend
        uint32_t have = 0, top = lo;
        unsigned long long dry = 0;
        // stage chunk [p0, p0 + 32): rows (out-CSR starts, one more than positions), capped coverage,
        // and the chunk's bundle records; buffers alternate
        auto stage_chunk = [&](uint32_t p0, uint32_t bufi) {
            const uint32_t p = min(p0 + lane, hi);
            const uint32_t op = G.out_ptr[p];
            const uint32_t cov = G.excl[p] + (uint32_t)G.diff[p];
            rows[bufi * 34 + lane] = op;
            needs[bufi * 32 + lane] = p0 + lane < hi ? min(cov, M) : 0u;
            const uint32_t cnt = min(32u, hi - p0);
            const uint32_t b0 = __shfl_sync(0xffffffffu, op, 0);
            uint32_t b1 = G.out_ptr[min(p0 + cnt, hi)];  // same address in every lane
            if (lane == 0) rows[bufi * 34 + 32] = b1;
            const uint32_t nb = min(b1 - b0, (uint32_t)CAP);
            for (uint32_t i = lane; i < nb; i += 32) cp_async8(stage + bufi * CAP + i, G.bund + b0 + i);
        };
        stage_chunk(lo, 0);
        uint32_t buf = 0;
        for (uint32_t p0 = lo; p0 < hi; p0 += 32, buf ^= 1) {
            cp_async_wait_all();  // this chunk's bundle records have landed
            __syncwarp();         // ... and its rows are visible to lane 0
            if (p0 + 32 < hi) stage_chunk(p0 + 32, buf ^ 1);  // in flight while lane 0 walks
            if (lane == 0) {
                const uint32_t cnt = min(32u, hi - p0);
                const uint32_t* rw = rows + buf * 34;
                const uint32_t* nd_ = needs + buf * 32;
                const uint2* st = stage + buf * CAP;
                const uint32_t cb0 = rw[0];
                for (uint32_t j = 0; j < cnt; ++j) {
                    const uint32_t p = p0 + j, slot = p & (W - 1);
                    // reads whose end node is p stop covering here; their count is final
                    const uint32_t exp = pend[slot];
                    if (exp) {
                        G.taken[p] = exp;
                        pend[slot] = 0;
                        have -= exp;
                    }
                    pool[slot] = 0;
                    // arrivals: the bundles starting at p join the pool of their end node
                    const uint32_t b0 = rw[j], b1 = j + 1 < cnt ? rw[j + 1] : rw[32];
                    for (uint32_t b = b0; b < b1; ++b) {
                        const uint32_t k = b - cb0;
                        const uint2 r = k < (uint32_t)CAP ? st[k]
                                                          : *reinterpret_cast<const uint2*>(G.bund + b);
                        if (r.x != p) {  // a read of length 0 covers nothing
                            pool[r.x & (W - 1)] += r.y;
                            top = max(top, r.x);
                        }
                    }
                    // picks: farthest end first
                    const uint32_t nd = nd_[j];
                    while (have < nd) {
                        while (top > p && pool[top & (W - 1)] == 0) --top;
                        if (top <= p) {
                            ++dry;
                            break;
                        }
                        const uint32_t k = min(nd - have, pool[top & (W - 1)]);
                        pool[top & (W - 1)] -= k;
                        pend[top & (W - 1)] += k;
                        have += k;
                    }
                }
            }
        }
        __syncwarp();
        if (lane == 0) {  // reads that end at the component's last node
            const uint32_t exp = pend[hi & (W - 1)];
            if (exp) G.taken[hi] = exp;
            if (dry) atomicAdd(fail, dry);
        }
        __syncwarp();
    }
}

// The warp-synchronous form of the same sweep, for components with MANY bundles per position
// (variable read lengths: ~40 arrivals per position, added to the pool by the lanes in parallel): all
// 32 lanes walk the positions together — 630 clocks per position whatever the arrivals, where the
// one-lane walk above pays ~130 per arrival (config 2: 17 ms against 80 ms).
template <int W, int CAP>
__global__ void __launch_bounds__(kSweepWarps * 32)
k_sweep_warp(SweepGraph G, const uint32_t* __restrict__ comp_lo, const uint32_t* __restrict__ comp_hi,
        const uint32_t* __restrict__ n_comp_dev, uint32_t M, uint32_t* work_counter,
        unsigned long long* __restrict__ fail /* += positions whose pool ran dry (never) */) {
    extern __shared__ __align__(16) unsigned char sw_raw[];
    const uint32_t warp = threadIdx.x >> 5, lane = lane_id();
    // per warp: pool[W], pend[W], stage[2][CAP] of {t, mult}
    uint32_t* pool = reinterpret_cast<uint32_t*>(sw_raw) + (size_t)warp * (2 * W + 4 * CAP);
    uint32_t* pend = pool + W;
    uint2* stage = reinterpret_cast<uint2*>(pend + W);
    const uint32_t n_comp = *n_comp_dev;
    for (;;) {
        uint32_t c = 0;
        if (lane == 0) c = atomicAdd(work_counter, 1u);
        c = __shfl_sync(0xffffffffu, c, 0);
        if (c >= n_comp) break;
        const uint32_t lo = comp_lo[c], hi = comp_hi[c];
        for (uint32_t i = lane; i < 2 * W; i += 32) pool[i] = 0;  // pool and pend
        __syncwarp();
        uint32_t have = 0, top = lo;
        unsigned long long dry = 0;
        // chunk pipeline: rows/coverage of chunk k+1 in registers, bundles of chunk k+1 in flight
        auto load_rows = [&](uint32_t p0, uint32_t& op, uint32_t& op1, uint32_t& need) {
            const uint32_t p = min(p0 + lane, hi);
            op = G.out_ptr[p];
            op1 = G.out_ptr[min(p + 1, hi)];
            const uint32_t cov = G.excl[p] + (uint32_t)G.diff[p];
            need = p0 + lane < hi ? min(cov, M) : 0u;
        };
        auto stage_bundles = [&](uint32_t b0, uint32_t b1, uint2* dst) {
            const uint32_t nb = min(b1 - b0, (uint32_t)CAP);
            for (uint32_t i = lane; i < nb; i += 32) cp_async8(dst + i, G.bund + b0 + i);
        };
        uint32_t op, op1, need, opn, op1n, needn;
        load_rows(lo, op, op1, need);
        {
            const uint32_t b0 = __shfl_sync(0xffffffffu, op, 0);
            const uint32_t b1 = __shfl_sync(0xffffffffu, op1, min(31u, hi - lo - 1));
            stage_bundles(b0, b1, stage);
        }
        uint32_t buf = 0;
        for (uint32_t p0 = lo; p0 < hi; p0 += 32, buf ^= 1) {
            const uint32_t cnt = min(32u, hi - p0);
            const uint32_t cb0 = __shfl_sync(0xffffffffu, op, 0);  // first bundle of this chunk
            const bool more = p0 + 32 < hi;
            if (more) load_rows(p0 + 32, opn, op1n, needn);
            cp_async_wait_all();  // this chunk's bundle records have landed
            __syncwarp();
            if (more) {  // next chunk's records: in flight while this chunk is swept
                const uint32_t nb0 = __shfl_sync(0xffffffffu, opn, 0);
                const uint32_t nb1 = __shfl_sync(0xffffffffu, op1n, min(31u, hi - (p0 + 32) - 1));
                stage_bundles(nb0, nb1, stage + (buf ^ 1) * CAP);
            }
            const uint2* st = stage + buf * CAP;
            for (uint32_t j = 0; j < cnt; ++j) {
                const uint32_t p = p0 + j;
                const uint32_t b0 = __shfl_sync(0xffffffffu, op, j), b1 = __shfl_sync(0xffffffffu, op1, j);
                const uint32_t nd = __shfl_sync(0xffffffffu, need, j);
                // reads whose end node is p stop covering here; their count is final
                const uint32_t slot = p & (W - 1);
                const uint32_t exp = pend[slot];
                __syncwarp();
                if (lane == 0) {
                    if (exp) G.taken[p] = exp;
                    pend[slot] = 0;
                    pool[slot] = 0;
                }
                have -= exp;
                // arrivals: the bundles starting at p join the pool of their end node
                uint32_t tmax = 0;
                for (uint32_t b = b0 + lane; b < b1; b += 32) {
                    const uint32_t k = b - cb0;
                    uint2 r;
                    if (k < (uint32_t)CAP) r = st[k];
                    else r = *reinterpret_cast<const uint2*>(G.bund + b);  // chunk larger than the stage
                    if (r.x != p) {  // a read of length 0 covers nothing
                        // (two keys of one start can be clamped to one end node at a segment cut)
                        atomicAdd(&pool[r.x & (W - 1)], r.y);
                        tmax = max(tmax, r.x);
                    }
                }
                __syncwarp();
                if (b1 > b0) top = max(top, __reduce_max_sync(0xffffffffu, tmax));
                // picks: farthest end first
                while (have < nd) {
                    while (top > p && pool[top & (W - 1)] == 0) --top;
                    if (top <= p) {
                        ++dry;
                        break;
                    }
                    const uint32_t k = min(nd - have, pool[top & (W - 1)]);
                    __syncwarp();
                    if (lane == 0) {
                        pool[top & (W - 1)] -= k;
                        pend[top & (W - 1)] += k;
                    }
                    __syncwarp();
                    have += k;
                }
            }
            op = opn;
            op1 = op1n;
            need = needn;
        }
        // reads that end at the component's last node
        {
            const uint32_t exp = pend[hi & (W - 1)];
            if (lane == 0 && exp) G.taken[hi] = exp;
        }
        if (lane == 0 && dry) atomicAdd(fail, dry);
        __syncwarp();
    }
}

// Reads taken per end node -> bundle flows: the bundles ending at t, earliest start first.
__global__ void __launch_bounds__(256)
k_sweep_distribute(const uint32_t* __restrict__ taken, const uint32_t* __restrict__ in_ptr,
                   const uint32_t* __restrict__ in_bid, BundleRec* __restrict__ bund, uint32_t n_nodes,
                   unsigned long long* __restrict__ fail) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_nodes) return;
    uint32_t rem = taken[t];
    if (rem == 0) return;
    for (uint32_t k = in_ptr[t], ke = in_ptr[t + 1]; k < ke && rem; ++k) {
        const uint32_t b = in_bid[k];
        const uint4 r = reinterpret_cast<const uint4*>(bund)[b];  // t, mult, f, s
        if (r.w == r.x) continue;
        const uint32_t x = min(rem, r.y);
        bund[b].f = x;
        rem -= x;
    }
    if (rem) atomicAdd(fail, (unsigned long long)rem);
}

}  // namespace gds
