// scan.cuh — device-wide exclusive prefix sum over uint32 (wrap-around add, so it also serves
// int32 difference arrays).  One pass with decoupled look-back (each tile publishes its aggregate,
// then its inclusive prefix, in one 64-bit status word; a tile's first warp walks back over its
// predecessors' words): the data is read once and written once, 8 bytes per element.  Inputs of
// one k_scan_tiles tile or less are scanned by a single block.
// Integer addition is associative, so the result does not depend on which tiles were ready when.
#pragma once
#include "common.cuh"

namespace gds {

constexpr int kScanThreads = 1024;
constexpr int kScanItems = 4;
constexpr int kScanTile = kScanThreads * kScanItems;

__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, v, o);
        if ((int)lane_id() >= o) v += t;
    }
    return v;
}

// exclusive scan of a block-wide value; returns exclusive prefix, *total = block sum
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t* total) {
    __shared__ uint32_t warp_sums[32];
    uint32_t incl = warp_incl_scan(v);
    uint32_t w = threadIdx.x >> 5;
    if (lane_id() == 31) warp_sums[w] = incl;
    __syncthreads();
    if (w == 0) {
        uint32_t nw = (blockDim.x + 31) >> 5;
        uint32_t s = lane_id() < nw ? warp_sums[lane_id()] : 0;
        uint32_t si = warp_incl_scan(s);
        warp_sums[lane_id()] = si - s;  // exclusive warp offsets
        if (lane_id() == 31) *total = si;
    }
    __syncthreads();
    uint32_t r = warp_sums[w] + incl - v;
    __syncthreads();
    return r;
}

// n <= kScanTile, one block
__global__ void __launch_bounds__(kScanThreads)
k_scan_tiles(const uint32_t* in, uint32_t* out /* may alias in: in-place scans */, size_t n) {
    __shared__ uint32_t total;
    const size_t base = (size_t)threadIdx.x * kScanItems;
    uint32_t v[kScanItems];
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) {
        v[k] = base + k < n ? in[base + k] : 0u;
        s += v[k];
    }
    uint32_t ex = block_excl_scan(s, &total);
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) {
        if (base + k < n) out[base + k] = ex;
        ex += v[k];
    }
}

// Up to three equally long arrays scanned by one launch (the node arrays of the graph build).
struct ScanArrays {
    const uint32_t* in[3];
    uint32_t* out[3];  // out[k] may alias in[k]
};

// status word: [63:34] epoch of the launch, [33:32] 1 = aggregate / 2 = inclusive prefix, [31:0] value.
// The epoch makes stale words of earlier launches invalid, so the array is never cleared.
__device__ __forceinline__ unsigned long long scan_status(uint32_t epoch, uint32_t flag, uint32_t v) {
    return ((unsigned long long)epoch << 34) | ((unsigned long long)flag << 32) | v;
}

// Decoupled look-back of one value, run by one whole warp of the tile holding ticket tk; the tile
// before it in the same sequence holds tk - stride.  Publishes the tile's aggregate, adds up the
// predecessors' words back to the nearest inclusive prefix, publishes the tile's inclusive prefix
// and returns its exclusive prefix (on every lane).
__device__ __forceinline__ uint32_t lookback_prefix(unsigned long long* status, uint32_t tk,
                                                    uint32_t stride, bool first_tile, uint32_t total,
                                                    uint32_t epoch) {
    const uint32_t lane = lane_id();
    volatile unsigned long long* st = status;
    if (first_tile) {
        if (lane == 0) st[tk] = scan_status(epoch, 2, total);
        return 0;
    }
    if (lane == 0) st[tk] = scan_status(epoch, 1, total);
    uint32_t prefix = 0;
    long long idx = (long long)tk - stride;
    for (;;) {
        const long long my = idx - (long long)lane * stride;
        uint32_t flag = 2, val = 0;  // before the first tile: an inclusive prefix of zero
        if (my >= 0) {
            unsigned long long w;
            do {
                w = st[my];
            } while ((uint32_t)(w >> 34) != epoch || ((w >> 32) & 3) == 0);
            flag = (uint32_t)(w >> 32) & 3;
            val = (uint32_t)w;
        }
        const uint32_t incl = __ballot_sync(0xffffffffu, flag == 2);
        const int first = __ffs(incl) - 1;  // nearest predecessor that knows its prefix
        prefix += __reduce_add_sync(0xffffffffu, (first < 0 || (int)lane <= first) ? val : 0u);
        if (first >= 0) break;
        idx -= 32ll * stride;
    }
    if (lane == 0) st[tk] = scan_status(epoch, 2, prefix + total);
    return prefix;
}

// 256 threads x 16 elements per step, kLbSub steps per tile: a tile is 64 KB, read twice (the
// second time from L2): once to publish its aggregate, once to scan and write.  Six or more tiles
// per SM are resident, so the wait of one tile for its predecessors is covered by the loads of the
// others.  Two earlier shapes, measured on config 5 (15.4 M entries per array): 1024 threads x 4
// elements with two tiles per SM had too few bytes in flight (1.3 TB/s, slower than the
// three-kernel scan); 16 KB tiles were bound by the look-back relay itself — inclusive prefixes
// travel 32 tiles per L2 round trip, 3 751 tiles took 117 trips = 48 us (ncu: 54 barrier-stall
// cycles per issue) — hence the larger tile.  A warp owns 512 consecutive elements of a step and
// reads them as four fully coalesced 512-byte rows; lane l holds the l-th 16 bytes of each row.
constexpr int kLbThreads = 256;
constexpr int kLbRows = 4;
constexpr int kLbWarpSpan = 32 * 4 * kLbRows;
constexpr int kLbStep = kLbThreads / 32 * kLbWarpSpan;  // 4096 elements
constexpr int kLbSub = 4;
constexpr int kLbTile = kLbStep * kLbSub;

__global__ void __launch_bounds__(kLbThreads, 6)
k_scan_lookback(ScanArrays a, uint32_t n_arr, size_t n, uint32_t n_tiles,
                unsigned long long* __restrict__ status, uint32_t* __restrict__ ticket, uint32_t epoch) {
    __shared__ uint32_t s_ticket, s_prefix;
    __shared__ uint32_t warp_tot[kLbThreads / 32];
    // tiles are handed out in launch order, so every predecessor of a tile is already running
    if (threadIdx.x == 0) s_ticket = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tk = s_ticket;
    const uint32_t tile = tk / n_arr, arr = tk - tile * n_arr;
    const uint32_t* in = arr == 0 ? a.in[0] : arr == 1 ? a.in[1] : a.in[2];
    uint32_t* out = arr == 0 ? a.out[0] : arr == 1 ? a.out[1] : a.out[2];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t tbase = (size_t)tile * kLbTile + (size_t)warp * kLbWarpSpan;
    const bool aligned = (reinterpret_cast<uintptr_t>(in) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    uint32_t v[kLbRows][4];
    auto load = [&](size_t wbase, bool vec) {  // vec is the same for a whole warp
        if (vec) {
            const uint4* in4 = reinterpret_cast<const uint4*>(in + wbase);
#pragma unroll
            for (int r = 0; r < kLbRows; ++r) {
                const uint4 q = in4[r * 32 + lane];
                v[r][0] = q.x; v[r][1] = q.y; v[r][2] = q.z; v[r][3] = q.w;
            }
        } else {
#pragma unroll
            for (int r = 0; r < kLbRows; ++r)
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const size_t i = wbase + (size_t)(r * 32 + lane) * 4 + k;
                    v[r][k] = i < n ? in[i] : 0u;
                }
        }
    };
    // pass 1: the tile's aggregate
    uint32_t sum = 0;
#pragma unroll 1
    for (int sub = 0; sub < kLbSub; ++sub) {
        const size_t wbase = tbase + (size_t)sub * kLbStep;
        if (wbase >= n) break;
        load(wbase, aligned && wbase + kLbWarpSpan <= n);
#pragma unroll
        for (int r = 0; r < kLbRows; ++r) sum += v[r][0] + v[r][1] + v[r][2] + v[r][3];
    }
    sum = __reduce_add_sync(0xffffffffu, sum);
    if (lane == 0) warp_tot[warp] = sum;
    __syncthreads();
    if (warp == 0) {
        uint32_t total = 0;
#pragma unroll
        for (int w = 0; w < kLbThreads / 32; ++w) total += warp_tot[w];
        // the tile before this one in the same array holds ticket tk - n_arr
        const uint32_t prefix = lookback_prefix(status, tk, n_arr, tile == 0, total, epoch);
        if (lane == 0) s_prefix = prefix;
    }
    __syncthreads();
    // pass 2: scan and write, step by step, carrying the running prefix
    uint32_t carry = s_prefix;
#pragma unroll 1
    for (int sub = 0; sub < kLbSub; ++sub) {
        const size_t wbase = tbase + (size_t)sub * kLbStep;
        if ((size_t)tile * kLbTile + (size_t)sub * kLbStep >= n) break;  // the same for the whole CTA
        const bool vec = aligned && wbase + kLbWarpSpan <= n;
        load(wbase, vec);
        uint32_t ex[kLbRows], wsum = 0;
#pragma unroll
        for (int r = 0; r < kLbRows; ++r) {
            const uint32_t s = v[r][0] + v[r][1] + v[r][2] + v[r][3];
            const uint32_t incl = warp_incl_scan(s);
            ex[r] = wsum + incl - s;
            wsum += __shfl_sync(0xffffffffu, incl, 31);
        }
        __syncthreads();  // warp_tot of the previous step (or of pass 1) has been read by everyone
        if (lane == 0) warp_tot[warp] = wsum;
        __syncthreads();
        uint32_t woff = 0, total = 0;
#pragma unroll
        for (int w = 0; w < kLbThreads / 32; ++w) {
            const uint32_t t = warp_tot[w];
            woff += w < (int)warp ? t : 0u;
            total += t;
        }
        const uint32_t base_ex = carry + woff;
        carry += total;
        if (vec) {
            uint4* out4 = reinterpret_cast<uint4*>(out + wbase);
#pragma unroll
            for (int r = 0; r < kLbRows; ++r) {
                uint4 q;
                q.x = base_ex + ex[r];
                q.y = q.x + v[r][0];
                q.z = q.y + v[r][1];
                q.w = q.z + v[r][2];
                out4[r * 32 + lane] = q;
            }
        } else {
#pragma unroll
            for (int r = 0; r < kLbRows; ++r) {
                uint32_t e = base_ex + ex[r];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const size_t i = wbase + (size_t)(r * 32 + lane) * 4 + k;
                    if (i < n) out[i] = e;
                    e += v[r][k];
                }
            }
        }
    }
    if (threadIdx.x == 0 && tk == n_tiles * n_arr - 1) *ticket = 0;  // every ticket is out by now
}

struct ScanTemp {
    DevBuf status, ticket;
    size_t status_cap = 0;
    uint32_t epoch = 0;
};

inline void scan_one_tile(const uint32_t* in, uint32_t* out, size_t n, cudaStream_t st) {
    launch("scan_u32", 8ull * n, k_scan_tiles, 1, kScanThreads, 0, st, in, out, n);
}

// The status words and the ticket of one look-back launch, and its epoch.  The ticket is zero
// between launches (the last tile of a launch resets it).
struct LookbackWords {
    unsigned long long* status;
    uint32_t* ticket;
    uint32_t epoch;
};

inline LookbackWords lookback_words(ScanTemp& tmp, size_t n_words, cudaStream_t st) {
    unsigned long long* status = tmp.status.get<unsigned long long>(n_words);
    uint32_t* ticket = tmp.ticket.get<uint32_t>(1);
    if (tmp.status_cap != tmp.status.cap || tmp.epoch >= (1u << 30) - 1) {  // new buffer or epoch wrap
        GDS_CUDA(cudaMemsetAsync(tmp.status.p, 0, tmp.status.cap, st));
        GDS_CUDA(cudaMemsetAsync(ticket, 0, 4, st));
        tmp.status_cap = tmp.status.cap;
        tmp.epoch = 0;
    }
    return LookbackWords{status, ticket, ++tmp.epoch};
}

// k equally long arrays in one launch; arrays of one tile are scanned one by one
inline void exclusive_scan_u32_multi(const ScanArrays& a, int n_arr, size_t n, ScanTemp& tmp,
                                     cudaStream_t st) {
    if (n == 0 || n_arr <= 0) return;
    if (n <= (size_t)kScanTile) {
        for (int k = 0; k < n_arr; ++k) scan_one_tile(a.in[k], a.out[k], n, st);
        return;
    }
    const size_t tl = (n + kLbTile - 1) / kLbTile;
    const LookbackWords lw = lookback_words(tmp, tl * n_arr, st);
    launch("scan_u32", 8ull * n * n_arr, k_scan_lookback, (unsigned)(tl * n_arr), kLbThreads, 0, st, a,
           (uint32_t)n_arr, n, (uint32_t)tl, lw.status, lw.ticket, lw.epoch);
}

// out may alias in.  Callers that need the grand total read out[n-1] + in[n-1] themselves or scan
// n+1 elements with a trailing zero.
inline void exclusive_scan_u32(const uint32_t* in, uint32_t* out, size_t n, ScanTemp& tmp,
                               cudaStream_t st) {
    ScanArrays a{{in, nullptr, nullptr}, {out, nullptr, nullptr}};
    exclusive_scan_u32_multi(a, 1, n, tmp, st);
}

}  // namespace gds
