// radix_sort.cuh — stable, SEGMENTED LSD radix sort of (key, uint32 value) pairs, 8 bits per pass.
//
// Stability is what makes read selection deterministic: after sorting by (start node, length)
// the reads of one bundle appear in ascending read index.
//
// Segmented: the items come pre-grouped (group = sample; its reads are contiguous in the input),
// so the group id is an implicit, already sorted key prefix and only the key bits INSIDE a group
// are sorted.  Tiles of kRsTile items never straddle a group; the per-tile digit histograms are
// laid out [group][digit][tile in group], so one exclusive scan over that array yields, for every
// (group, digit, tile), the global position of the tile's first key with that digit.  A batch of
// 512 samples x 30 kb therefore sorts 15-bit keys in 2 passes instead of 24-bit keys in 3.
//
// Per pass: k_rs_hist (per-tile digit counts) -> exclusive scan -> k_rs_scatter.  The scatter
// ranks keys with warp match_any + per-warp running counts (stable), reorders the whole tile by
// digit in shared memory and writes each digit run as one contiguous, coalesced segment
// (a direct scatter wrote 30 sectors per 32-lane store; this writes ~5).
#pragma once
#include "common.cuh"
#include "prep.cuh"
#include "scan.cuh"

#include <algorithm>
#include <cstdlib>

namespace gds {

constexpr int kRsThreads = 512;
constexpr int kRsWarps = kRsThreads / 32;
constexpr int kRsItems = 16;
constexpr int kRsTile = kRsThreads * kRsItems;  // 8192 keys per tile

// Where the tiles are.  n_groups == 1: items [0, n_items) in tiles of kRsTile.  Otherwise group g
// owns items [item_off[g], item_off[g+1]) and tiles [tile_off[g], tile_off[g+1]).
struct TileMap {
    const uint32_t* tile_off;  // [n_groups+1], device
    const uint64_t* item_off;  // [n_groups+1], device
    uint32_t n_groups;
    uint32_t n_tiles;
    size_t n_items;
};

struct TilePos {
    size_t first;        // first item of the tile
    uint32_t n_valid;    // items in the tile
    uint32_t hist_base;  // index of hist[group][digit 0][tile 0]
    uint32_t tiles_g;    // tiles in the group
    uint32_t tile_in_g;
    uint32_t group;
};

// executed by every thread of the block (uniform result); the binary search is ~9 L1-cached steps
__device__ __forceinline__ TilePos locate_tile(const TileMap& tm, uint32_t tile) {
    TilePos p;
    if (tm.n_groups == 1) {
        p.first = (size_t)tile * kRsTile;
        p.n_valid = (uint32_t)min((size_t)kRsTile, tm.n_items - p.first);
        p.hist_base = 0;
        p.tiles_g = tm.n_tiles;
        p.tile_in_g = tile;
        p.group = 0;
        return p;
    }
    uint32_t lo = 0, hi = tm.n_groups;  // largest g with tile_off[g] <= tile
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (tm.tile_off[mid] <= tile) lo = mid;
        else hi = mid;
    }
    const uint32_t t0 = tm.tile_off[lo];
    const uint64_t i0 = tm.item_off[lo], i1 = tm.item_off[lo + 1];
    p.tile_in_g = tile - t0;
    p.tiles_g = tm.tile_off[lo + 1] - t0;
    p.first = (size_t)i0 + (size_t)p.tile_in_g * kRsTile;
    p.n_valid = (uint32_t)min((uint64_t)kRsTile, i1 - p.first);
    p.hist_base = 256u * t0;
    p.group = lo;
    return p;
}

// Key sources: a plain array, or a functor that builds the key from the reads (first pass).
// Two-step interface so the kernels can issue ALL loads of a thread before any use:
//   Raw load(i)      — the global loads, nothing else (branch-free on the hot paths)
//   K   make(raw, i) — arithmetic on the loaded values
template <typename K>
struct ArrayKeys {
    typedef K Raw;
    const K* keys;
    __device__ __forceinline__ Raw load(size_t i) const { return keys[i]; }
    __device__ __forceinline__ K make(Raw r, size_t) const { return r; }
    __device__ __forceinline__ uint32_t owner(size_t i) const { return (uint32_t)i; }
    // nothing to validate in a plain key array
    __device__ __forceinline__ bool checks() const { return false; }
    __device__ __forceinline__ uint32_t check(Raw, uint32_t) const { return 0; }
    __device__ __forceinline__ uint32_t* check_stats() const { return nullptr; }
};

template <typename K, typename KS>
__global__ void __launch_bounds__(kRsThreads)
k_rs_hist(KS ks, TileMap tm, int shift, uint32_t* __restrict__ tile_hist) {
    __shared__ uint32_t h[kRsWarps][256];  // per-warp counts: conflicts only inside a warp
    for (int i = threadIdx.x; i < kRsWarps * 256; i += kRsThreads) (&h[0][0])[i] = 0;
    const TilePos tp = locate_tile(tm, blockIdx.x);
    __syncthreads();
    const uint32_t warp = threadIdx.x >> 5;
    typename KS::Raw raw[kRsItems];
#pragma unroll
    for (int k = 0; k < kRsItems; ++k) {
        uint32_t j = (uint32_t)k * kRsThreads + threadIdx.x;
        // out-of-range lanes re-read the tile's first item: the load stays unconditional
        raw[k] = ks.load(tp.first + (j < tp.n_valid ? j : 0u));
    }
    uint32_t bad = 0;  // input validation fused into the first pass (low half: range, high: hints)
#pragma unroll
    for (int k = 0; k < kRsItems; ++k) {
        uint32_t j = (uint32_t)k * kRsThreads + threadIdx.x;
        // lanes past the tile's end get the first item's index too: make() may index side arrays
        // (the crossing-read list of the global key source) with it
        K key = ks.make(raw[k], tp.first + (j < tp.n_valid ? j : 0u));
        if (j < tp.n_valid) {
            atomicAdd(&h[warp][(uint32_t)(key >> shift) & 255u], 1u);
            if (ks.checks()) bad += ks.check(raw[k], tp.group);
        }
    }
    if (ks.checks()) {
        bad = __reduce_add_sync(0xffffffffu, bad);
        if (bad && lane_id() == 0) {
            if (bad & 0xffffu) atomicAdd(&ks.check_stats()[2], bad & 0xffffu);
            if (bad >> 16) atomicAdd(&ks.check_stats()[3], bad >> 16);
        }
    }
    __syncthreads();
    if (threadIdx.x < 256) {
        uint32_t s = 0;
#pragma unroll
        for (int w = 0; w < kRsWarps; ++w) s += h[w][threadIdx.x];
        tile_hist[(size_t)tp.hist_base + (size_t)threadIdx.x * tp.tiles_g + tp.tile_in_g] = s;
    }
}

// Lanes holding the same 8-bit digit, from 8 ballots (fixed latency; the MATCH.ANY instruction
// measured ~35% slower here: it iterates once per distinct value, ~30 times for random digits).
// Per bit: test, vote, conditional complement, and — hand-written so ptxas keeps it at 4 SASS.
// Only the low `nbits` bits of the digit can be set in this pass (uniform), the rest is skipped.
__device__ __forceinline__ uint32_t match_digit(uint32_t d, uint32_t valid_mask, int nbits) {
    uint32_t peers = valid_mask;
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        if (b >= nbits) break;
        asm("{\n"
            ".reg .pred p;\n"
            ".reg .b32 m;\n"
            "and.b32 m, %1, %2;\n"
            "setp.ne.u32 p, m, 0;\n"
            "vote.sync.ballot.b32 m, p, 0xffffffff;\n"
            "@!p not.b32 m, m;\n"
            "and.b32 %0, %0, m;\n"
            "}\n"
            : "+r"(peers)
            : "r"(d), "r"(1u << b));
    }
    return peers;
}

// ------------------------------------------------------------------------------------------
// Stable ranks from ONE shared-memory atomic per key.  When several lanes of a warp instruction
// atomicAdd the same shared word, B200 serialises them in ascending lane order (measured:
// 0 violations over 1.6e9 conflicting lanes, tools/atoms_order_probe.cu), so the value returned
// to a lane is exactly its stable rank among the equal digits seen so far by the warp.  That
// replaces ~45 instructions of ballot matching per 32 keys by one ATOMS.  The order is not an
// architectural guarantee, so every context PROBES it once (k_atoms_order_probe below) and
// falls back to the ballot ranking if a single violation shows up.
__global__ void k_atoms_order_probe(uint32_t seed, int iters, unsigned int* violations) {
    __shared__ uint32_t cnt[32][256];
    const uint32_t warp = threadIdx.x >> 5, lane = lane_id();
    uint32_t x = seed ^ (blockIdx.x * 9781u + threadIdx.x * 6271u + 1u);
    uint32_t v = 0;
    for (int it = 0; it < iters; ++it) {
        for (int i = lane; i < 256; i += 32) cnt[warp][i] = 0;
        __syncwarp();
        x = x * 1664525u + 1013904223u;
        const uint32_t nbins = (it & 3) == 0 ? 256u : (it & 3) == 1 ? 128u : (it & 3) == 2 ? 7u : 1u;
        const uint32_t d = (x >> 13) % nbins;
        const bool active = (it & 4) ? ((x >> 5) & 3) != 0 : true;  // divergent callers too
        uint32_t r = 0;
        if (active) r = atomicAdd(&cnt[warp][d], 1u);
        __syncwarp();
        const uint32_t peers = match_digit(d, __ballot_sync(0xffffffffu, active), 8);
        if (active && r != (uint32_t)__popc(peers & lanemask_lt())) ++v;
        __syncwarp();
    }
    if (v) atomicAdd(violations, v);
}

// true if shared-memory atomics hand out ranks in lane order on `device` (probed once per process
// and device; GDS_RANK=ballot|atomic overrides)
inline bool atomic_rank_is_stable(int device, cudaStream_t st) {
    static int cached[64];  // 0 unknown, 1 stable, 2 not stable
    if (const char* f = getenv("GDS_RANK")) {
        if (f[0] == 'b') return false;
        if (f[0] == 'a') return true;
    }
    int& c = cached[device & 63];
    if (c == 0) {
        unsigned int* d = nullptr;
        unsigned int h = 1;
        if (cudaMalloc(&d, sizeof h) == cudaSuccess) {
            cudaMemsetAsync(d, 0, sizeof h, st);
            k_atoms_order_probe<<<kNumSMs, 1024, 0, st>>>(0x9e3779b9u, 512, d);
            if (cudaMemcpyAsync(&h, d, sizeof h, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaStreamSynchronize(st) != cudaSuccess)
                h = 1;
            cudaFree(d);
        }
        cudaGetLastError();
        c = h == 0 ? 1 : 2;
    }
    return c == 1;
}

template <typename K>
struct RsSmem {
    K skey[kRsTile];
    uint32_t sval[kRsTile];
    uint32_t whist[kRsWarps][256];  // per-warp digit counts, then first slot per (warp, digit)
    uint32_t gbase[256];            // global position of the digit's run minus its first slot
    uint32_t dstart[256];
    uint32_t wsum[8];
};

// vals_in is read when HAS_VALS, else the value is what the key source says (the owner read).
template <typename K, typename KS, bool HAS_VALS, bool ATOMIC_RANK, int MIN_CTAS>
__global__ void __launch_bounds__(kRsThreads, MIN_CTAS)
k_rs_scatter(KS ks, const uint32_t* __restrict__ vals_in, K* __restrict__ keys_out,
             uint32_t* __restrict__ vals_out, TileMap tm, int shift, int nbits,
             const uint32_t* __restrict__ tile_off_scanned) {
    extern __shared__ __align__(16) unsigned char rs_smem_raw[];
    RsSmem<K>& sm = *reinterpret_cast<RsSmem<K>*>(rs_smem_raw);
    const uint32_t warp = threadIdx.x >> 5, lane = lane_id();
    for (int i = threadIdx.x; i < kRsWarps * 256; i += kRsThreads) (&sm.whist[0][0])[i] = 0;
    const TilePos tp = locate_tile(tm, blockIdx.x);
    if (threadIdx.x < 256)
        sm.gbase[threadIdx.x] = tile_off_scanned[(size_t)tp.hist_base +
                                                 (size_t)threadIdx.x * tp.tiles_g + tp.tile_in_g];

    // warp w owns the contiguous chunk [w*32*kRsItems, (w+1)*32*kRsItems) of the tile; row k
    // covers 32 consecutive keys, so (warp, row, lane) order == input order.  Loads are batched 8
    // rows at a time (register budget) and never predicated: short tiles re-read their first item.
    const uint32_t wofs = warp * 32 * kRsItems + lane;
    const bool full = tp.n_valid == (uint32_t)kRsTile;
    const size_t gfirst = tp.first + wofs;
    K key[kRsItems];
    constexpr int kHalf = kRsItems / 2;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        typename KS::Raw raw[kHalf];
#pragma unroll
        for (int k = 0; k < kHalf; ++k) {
            const uint32_t jo = (uint32_t)(h * kHalf + k) * 32;
            raw[k] = ks.load((full || wofs + jo < tp.n_valid) ? gfirst + jo : tp.first);
        }
#pragma unroll
        for (int k = 0; k < kHalf; ++k) {
            const uint32_t jo = (uint32_t)(h * kHalf + k) * 32;
            key[h * kHalf + k] =
                ks.make(raw[k], (full || wofs + jo < tp.n_valid) ? gfirst + jo : tp.first);
        }
    }
    __syncthreads();  // whist zeroed

    // ---- stable ranks: peers by ballots (independent across rows), then one shared-memory
    // atomic per peer group, issued by its lowest lane, hands out the group's base rank
    uint32_t rank2[kRsItems / 2];  // two 16-bit ranks per register
    if (ATOMIC_RANK) {
        // one ATOMS per key: same-digit lanes are served in lane order (probed), so the returned
        // count is the stable rank; the 16 atomics of a thread are independent and pipeline
#pragma unroll
        for (int k = 0; k < kRsItems / 2; ++k) rank2[k] = 0;
#pragma unroll
        for (int kk = 0; kk < kRsItems; ++kk) {
            const uint32_t d = (uint32_t)(key[kk] >> shift) & 255u;
            uint32_t r = 0;
            if (full || wofs + (uint32_t)kk * 32 < tp.n_valid) r = atomicAdd(&sm.whist[warp][d], 1u);
            rank2[kk >> 1] |= r << (16 * (kk & 1));
        }
    } else
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        uint32_t peers[kHalf];
#pragma unroll
        for (int k = 0; k < kHalf; ++k) {
            const int kk = h * kHalf + k;
            const uint32_t d = (uint32_t)(key[kk] >> shift) & 255u;
            const uint32_t vm = full ? 0xffffffffu
                                     : __ballot_sync(0xffffffffu, wofs + (uint32_t)kk * 32 < tp.n_valid);
            peers[k] = match_digit(d, vm, nbits);
        }
#pragma unroll
        for (int k = 0; k < kHalf; ++k) {
            const int kk = h * kHalf + k;
            const uint32_t d = (uint32_t)(key[kk] >> shift) & 255u;
            const uint32_t before = __popc(peers[k] & lanemask_lt());
            const bool valid = full || wofs + (uint32_t)kk * 32 < tp.n_valid;
            uint32_t prev = 0;
            if (valid && before == 0) prev = atomicAdd(&sm.whist[warp][d], __popc(peers[k]));
            prev = __shfl_sync(0xffffffffu, prev, __ffs(peers[k] | (valid ? 0u : 1u << lane)) - 1);
            const uint32_t r = prev + before;
            if (kk & 1) rank2[kk >> 1] |= r << 16;
            else rank2[kk >> 1] = r;
        }
    }
    __syncthreads();
    // ---- first slot of every (warp, digit) in the reordered tile
    uint32_t tot = 0;
    if (threadIdx.x < 256) {
#pragma unroll
        for (int w = 0; w < kRsWarps; ++w) tot += sm.whist[w][threadIdx.x];
        uint32_t incl = warp_incl_scan(tot);  // exclusive scan of the 256 digit totals (8 warps)
        if (lane == 31) sm.wsum[warp] = incl;
        sm.dstart[threadIdx.x] = incl - tot;
    }
    __syncthreads();
    if (threadIdx.x < 256) {
        uint32_t run = sm.dstart[threadIdx.x];
#pragma unroll
        for (int w = 0; w < 8; ++w) run += (w < (int)warp) ? sm.wsum[w] : 0u;
        sm.gbase[threadIdx.x] -= run;
#pragma unroll
        for (int w = 0; w < kRsWarps; ++w) {
            uint32_t c = sm.whist[w][threadIdx.x];
            sm.whist[w][threadIdx.x] = run;
            run += c;
        }
    }
    __syncthreads();
    // ---- reorder the tile by digit in shared memory
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        uint32_t val[kHalf];
#pragma unroll
        for (int k = 0; k < kHalf; ++k) {
            const uint32_t jo = (uint32_t)(h * kHalf + k) * 32;
            const size_t i = (full || wofs + jo < tp.n_valid) ? gfirst + jo : tp.first;
            val[k] = HAS_VALS ? vals_in[i] : ks.owner(i);
        }
#pragma unroll
        for (int k = 0; k < kHalf; ++k) {
            const int kk = h * kHalf + k;
            if (full || wofs + (uint32_t)kk * 32 < tp.n_valid) {
                const uint32_t d = (uint32_t)(key[kk] >> shift) & 255u;
                const uint32_t p = sm.whist[warp][d] + ((rank2[kk >> 1] >> (16 * (kk & 1))) & 0xffffu);
                sm.skey[p] = key[kk];
                sm.sval[p] = val[k];
            }
        }
    }
    __syncthreads();
    // ---- every digit run goes out as one contiguous segment
    K* const ko = keys_out;
    uint32_t* const vo = vals_out;
#pragma unroll 4
    for (uint32_t j = threadIdx.x; j < tp.n_valid; j += kRsThreads) {
        const K kk = sm.skey[j];
        const uint32_t dst = sm.gbase[(uint32_t)(kk >> shift) & 255u] + j;
        ko[dst] = kk;
        vo[dst] = sm.sval[j];
    }
}

struct RadixTemp {
    DevBuf hist;
    ScanTemp scan;
};

inline uint32_t tiles_for(size_t n) { return (uint32_t)((n + kRsTile - 1) / kRsTile); }

template <typename K, typename KS>
inline void launch_scatter(const char* name, unsigned long long bytes, const KS& ks,
                           const uint32_t* vals_in, K* kout, uint32_t* vout, const TileMap& t,
                           int shift, int nbits, const uint32_t* hist, bool atomic_rank,
                           cudaStream_t st) {
    constexpr int kMinCtas = sizeof(K) == 4 ? 2 : 1;
    constexpr int smem = (int)sizeof(RsSmem<K>);
    auto go = [&](auto kern) {
        GDS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        launch(name, bytes, kern, t.n_tiles, kRsThreads, smem, st, ks, vals_in, kout, vout, t, shift,
               nbits, hist);
    };
    if (vals_in) {
        if (atomic_rank) go(k_rs_scatter<K, KS, true, true, kMinCtas>);
        else go(k_rs_scatter<K, KS, true, false, kMinCtas>);
    } else {
        if (atomic_rank) go(k_rs_scatter<K, KS, false, true, kMinCtas>);
        else go(k_rs_scatter<K, KS, false, false, kMinCtas>);
    }
}

// Sorts the pairs by the low `bits` bits of the key inside every group.  Buffers ping-pong; returns
// 0 if the result is in (keys_a, vals_a), 1 if in (keys_b, vals_b).  The first pass takes key and
// value from *first_ks when it is non-null, else from keys_a with value = item index.
template <typename K, typename KS0 = ArrayKeys<K>>
inline int radix_sort_pairs(K* keys_a, uint32_t* vals_a, K* keys_b, uint32_t* vals_b,
                            const TileMap& tm, int bits, RadixTemp& tmp, cudaStream_t st,
                            bool atomic_rank, int* passes_out = nullptr,
                            const KS0* first_ks = nullptr) {
    int passes = (bits + 7) / 8;
    if (passes == 0) passes = 1;  // still need vals materialised
    if (passes_out) *passes_out = passes;
    const size_t n = tm.n_items;
    if (n == 0 || tm.n_tiles == 0) return 0;
    uint32_t* hist = tmp.hist.get<uint32_t>((size_t)256 * tm.n_tiles);
    int cur = 0;
    for (int p = 0; p < passes; ++p) {
        K* kin = cur ? keys_b : keys_a;
        K* kout = cur ? keys_a : keys_b;
        uint32_t* vin = cur ? vals_b : vals_a;
        uint32_t* vout = cur ? vals_a : vals_b;
        int shift = 8 * p;
        const int nbits = std::max(1, std::min(8, bits - shift));  // significant digit bits
        if (p == 0 && first_ks) {
            launch("rs_hist_reads", 8ull * n, k_rs_hist<K, KS0>, tm.n_tiles, kRsThreads, 0, st,
                   *first_ks, tm, shift, hist);
            exclusive_scan_u32(hist, hist, (size_t)256 * tm.n_tiles, tmp.scan, st);
            launch_scatter<K, KS0>("rs_scatter_reads", (8ull + sizeof(K) + 4) * n, *first_ks, nullptr,
                                   kout, vout, tm, shift, nbits, hist, atomic_rank, st);
        } else {
            ArrayKeys<K> ak{kin};
            const uint32_t* vsrc = p == 0 ? nullptr : vin;
            launch("rs_hist", sizeof(K) * (unsigned long long)n, k_rs_hist<K, ArrayKeys<K>>, tm.n_tiles,
                   kRsThreads, 0, st, ak, tm, shift, hist);
            exclusive_scan_u32(hist, hist, (size_t)256 * tm.n_tiles, tmp.scan, st);
            launch_scatter<K, ArrayKeys<K>>("rs_scatter", (2ull * sizeof(K) + (vsrc ? 8 : 4)) * n, ak,
                                            vsrc, kout, vout, tm, shift, nbits, hist, atomic_rank, st);
        }
        cur ^= 1;
    }
    return cur;
}

}  // namespace gds
