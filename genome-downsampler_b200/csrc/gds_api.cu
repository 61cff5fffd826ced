// gds_api.cu — C ABI (include/gds.h) and host-side orchestration of the device pipeline.
// No CPU fallback exists: without a usable CUDA device every entry point fails.
#include "../../include/gds.h"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"
#include "direct.cuh"
#include "graph.cuh"
#include "maxflow.cuh"
#include "maxflow_sm.cuh"
#include "prep.cuh"
#include "radix_sort.cuh"
#include "scan.cuh"
#include "select.cuh"
#include "sweep.cuh"

using namespace gds;

namespace {
enum Ev { EV_BEGIN = 0, EV_H2D, EV_FILTER, EV_GRAPH, EV_MAXFLOW, EV_SELECT, EV_VERIFY, EV_END, EV_COUNT };
}

struct gds_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    std::string err;
    cudaEvent_t ev[EV_COUNT] = {};
    void* pinned = nullptr;  // small readback area
    static constexpr size_t kPinnedBytes = 1 << 16;

    DevBuf in_start, in_end, in_mapq, in_len, in_raw;
    DevBuf off_d, reflen_d, base_d, foff_d, amp_s, amp_e;
    DevBuf pair_pass, flag32, fS, fE;
    DevBuf small;  // uint32 stats[8] + u64 totals[4]
    DevBuf keysA, keysB, valsA, valsB, tile_counts;
    RadixTemp radix;
    ScanTemp scan;
    DevBuf b_first, b_key, b_t, bund;
    DevBuf diff, outdeg, indeg, excl;
    DevBuf tkA, tkB, tvA, tvB;
    DevBuf node_rec, n_dsnap;
    DevBuf comp_start, comp_end, comp_sidx, comp_lo, comp_hi;
    DevBuf qF, qT, qN, qH, work_counter, comp_stats;
    DevBuf bitmap, cov_tmp, dem_tmp, vdiff, vexcl;
    DevBuf vs_d, cross_idx, cross_tc, odiff, oexcl, cut_nodes, tile_off_d, head_bits;
    DevBuf unc, adj, fmult, dead;  // forced reads out, cuts in (graph.cuh)
    DevBuf dhist, dlay, b_slot, ident, dwork;  // direct (sort-free) bundle path
    DevBuf kstat, pbund, cand, dctl, in_src, dem_v, fb_list, in1, lab_g, taken;
    unsigned sweep_smem_set = 0;  // bit i: the sweep launch shape i has its shared memory set up
    int mf2_smem_set[2] = {0, 0};
    unsigned direct_attr = 0;                  // bytes of dynamic smem the direct kernels are set up for
    int mf_smem_set[4] = {0, 0, 0, 0};  // dynamic shared memory the launch shapes are set up for
    bool atomic_rank = false;  // shared-memory atomics rank in lane order on this device (probed)
    Profiler prof;

};

namespace {

struct InputFail {  // bad input discovered on the device in the middle of the pipeline
    int code;
    uint32_t count;
    const char* what;
};

int fail(gds_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg;
    return code;
}

int fail_cuda(gds_ctx* ctx, const CudaFail& f) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s failed: %s (%s:%d)", f.what, cudaGetErrorString(f.err), f.file,
             f.line);
    ctx->err = buf;
    cudaGetLastError();  // clear sticky-free errors
    return f.err == cudaErrorMemoryAllocation ? GDS_ERR_NOMEM : GDS_ERR_CUDA;
}

template <typename T>
void d2h_sync(gds_ctx* c, T* host_dst, const T* dev_src, size_t n) {
    size_t bytes = n * sizeof(T);
    if (bytes <= gds_ctx::kPinnedBytes) {
        GDS_CUDA(cudaMemcpyAsync(c->pinned, dev_src, bytes, cudaMemcpyDeviceToHost, c->stream));
        GDS_CUDA(cudaStreamSynchronize(c->stream));
        memcpy(host_dst, c->pinned, bytes);
    } else {
        GDS_CUDA(cudaMemcpyAsync(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost, c->stream));
        GDS_CUDA(cudaStreamSynchronize(c->stream));
    }
}

// copy a device array to the caller's buffer (host or device)
template <typename T>
void deliver(gds_ctx* c, T* dst, const T* dev_src, size_t n, bool dst_on_device) {
    if (!dst || n == 0 || dst == dev_src) return;
    GDS_CUDA(cudaMemcpyAsync(dst, dev_src, n * sizeof(T),
                             dst_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost,
                             c->stream));
}

template <int I>
void launch_maxflow_shape(gds_ctx* c, const MfGraph& mg,
                          const uint32_t* comp_lo, const uint32_t* comp_hi, uint32_t n_comp,
                          uint32_t* wc, uint32_t* qF, uint32_t* qT, uint32_t* qN, uint32_t* qH,
                          const SolveParams& sp, CompStats* cstats, uint32_t max_comp_nodes,
                          const uint32_t* comp_list, const uint32_t* comp_list_n,
                          const uint32_t* n_comp_dev, MfTotals* mft, uint16_t* lab_g) {
    constexpr MfShape sh = kMfShapes[I];
    auto kern = k_maxflow<sh.threads, sh.qcap, sh.ctas_per_sm>;
    // 16-bit labels of a whole component in shared memory for the first global relabel, when
    // every resident CTA of this shape can have them (maxflow.cuh: mf_first_relabel)
    uint32_t lab_cap = 0;
    int smem = (int)sizeof(MfShared<sh.qcap>);
    if (max_comp_nodes && max_comp_nodes < 0xfff0u) {
        const int lab_bytes = (int)((2 * max_comp_nodes + 4 + 15) & ~15u);
        // ... and the SM keeps at least ~100 KB of L1 for the rounds' plain loads (measured: with
        // 4 x 49 KB per SM config 4 lost 13 %)
        if ((smem + lab_bytes) * sh.ctas_per_sm <= 132 * 1024) {
            smem += lab_bytes;
            lab_cap = max_comp_nodes;
        }
    }
    if (c->mf_smem_set[I] < smem) {
        GDS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        c->mf_smem_set[I] = smem;
    }
    int grid = std::min<uint32_t>(n_comp, (uint32_t)kNumSMs * sh.ctas_per_sm);
    kern<<<grid, sh.threads, smem, c->stream>>>(mg, comp_lo, comp_hi, n_comp, wc, qF, qT, qN, qH, sp,
                                                cstats, lab_cap, comp_list, comp_list_n, n_comp_dev, mft,
                                                lab_g);
}

void launch_maxflow(gds_ctx* c, const MfGraph& mg,
                    const uint32_t* comp_lo, const uint32_t* comp_hi, uint32_t n_comp, uint32_t* wc,
                    uint32_t* qF, uint32_t* qT, uint32_t* qN, uint32_t* qH, const SolveParams& sp,
                    CompStats* cstats, unsigned long long alg_bytes, uint32_t max_comp_nodes,
                    const uint32_t* n_comp_dev, MfTotals* mft, uint16_t* lab_g,
                    const uint32_t* comp_list = nullptr, const uint32_t* comp_list_n = nullptr) {
    KScope ks("maxflow", alg_bytes, c->stream);
    const uint32_t sms = (uint32_t)kNumSMs;
    int shape = 3;
    for (int i = 0; i < 3; ++i)
        if (n_comp <= sms * kMfShapes[i].ctas_per_sm) {
            shape = i;
            break;
        }
    switch (shape) {
        case 0: launch_maxflow_shape<0>(c, mg, comp_lo, comp_hi, n_comp, wc, qF, qT, qN, qH, sp, cstats, max_comp_nodes, comp_list, comp_list_n, n_comp_dev, mft, lab_g); break;
        case 1: launch_maxflow_shape<1>(c, mg, comp_lo, comp_hi, n_comp, wc, qF, qT, qN, qH, sp, cstats, max_comp_nodes, comp_list, comp_list_n, n_comp_dev, mft, lab_g); break;
        case 2: launch_maxflow_shape<2>(c, mg, comp_lo, comp_hi, n_comp, wc, qF, qT, qN, qH, sp, cstats, max_comp_nodes, comp_list, comp_list_n, n_comp_dev, mft, lab_g); break;
        default: launch_maxflow_shape<3>(c, mg, comp_lo, comp_hi, n_comp, wc, qF, qT, qN, qH, sp, cstats, max_comp_nodes, comp_list, comp_list_n, n_comp_dev, mft, lab_g); break;
    }
    GDS_KERNEL_CHECK();
}

// K3 with the hot state in shared memory (maxflow_sm.cuh).  Returns false when no component of
// this call can fit (then k_maxflow solves everything).  Components the kernel finds ineligible
// (too large for the launch, supply beyond 16 bits) land on fb_list for k_maxflow.
// Components whose nodes are mostly heavy (variable read lengths: tens of bundles per node) go to
// k_maxflow: their frontiers hold tens of nodes with ~40 bundles each, the time is the per-bundle
// global traffic of the warp passes, and 32 warps of 64 registers (k_maxflow) beat 16 warps with the
// labels in shared memory (config 2 without its filter: 2.6 ms there, 3.0 ms here after batching the
// loads of eight nodes per warp; 3.4 ms before).  GDS_MF_WARP=1 keeps them here (tests, measurements).
inline uint32_t mf2_allow_warp() {
    const char* e = getenv("GDS_MF_WARP");
    return (e && e[0] == '1') ? 1u : 0u;
}

constexpr int kMf2MaxSmem = 227 * 1024;
template <int THREADS, int SLOT>
void launch_mf2_shape(gds_ctx* c, const Mf2Graph& g, const uint32_t* comp_lo, const uint32_t* comp_hi,
                      uint32_t n_comp, uint32_t* wc, uint32_t* qF, uint32_t* qT, uint32_t* qN,
                      uint32_t* qH, const SolveParams& sp, CompStats* cstats, int smem, uint32_t qcap,
                      uint32_t* fb_list, uint32_t* fb_count, bool optr, int ctas_per_sm,
                      const uint32_t* n_comp_dev, MfTotals* mft) {
    auto kern = k_maxflow_sm<THREADS>;
    if (c->mf2_smem_set[SLOT] < smem) {
        GDS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        c->mf2_smem_set[SLOT] = smem;
    }
    // with the count on the device n_comp is an estimate (one component per sample or segment); the
    // cuts at cov <= M can make many more (the reference's "low sides" shape: 11 from one sample,
    // which a grid of one CTA solved one after the other).  A CTA without work exits at once.
    const int grid = (int)std::min<uint32_t>(n_comp_dev ? 0xffffffffu : n_comp,
                                             (uint32_t)(kNumSMs * ctas_per_sm));
    kern<<<grid, THREADS, smem, c->stream>>>(g, comp_lo, comp_hi, n_comp, wc, qF, qT, qN, qH, sp, cstats,
                                             (uint32_t)smem, qcap, fb_list, fb_count, optr ? 1u : 0u,
                                             n_comp_dev, mft, mf2_allow_warp());
}

// Whether this call's components go to k_maxflow_sm, and with which launch shape.
// gds_params.seg_len == 0 (include/gds.h): 16 384 positions, stretched by up to a quarter when that
// lets every segment of the batch be resident at once.  k_maxflow_sm keeps two components per SM
// resident (296 on a B200); 306 segments would run as 296 + a second wave of 10 that starts when
// the first components finish, i.e. ~1.3x the time of 296 slightly longer ones.  The constant is
// part of the deterministic schedule (the oracle has the same rule), NOT a property of the device
// the call happens to run on: the same input gives the same kept set everywhere.
constexpr uint32_t kSegBase = 16384, kSegResident = 296;
uint32_t default_seg_len(uint32_t n_samples, const uint32_t* ref_len) {
    auto count = [&](uint32_t seg) {
        unsigned long long n = 0;
        for (uint32_t k = 0; k < n_samples; ++k)
            n += (unsigned long long)ref_len[k] > 2ull * seg ? ((unsigned long long)ref_len[k] + seg - 1) / seg : 1;
        return n;
    };
    const unsigned long long n0 = count(kSegBase);
    if (n0 <= kSegResident || n0 > kSegResident + kSegResident / 4) return kSegBase;
    for (uint32_t seg = kSegBase + 128; seg <= kSegBase + kSegBase / 4; seg += 128)
        if (count(seg) <= kSegResident) return seg;
    return kSegBase;
}

struct Mf2Plan {
    bool on = false;
    bool classic_ok = false;  // components outside the express schedule may run in k_maxflow_sm too
    int smem = 0, per_sm = 1;  // two CTAs per SM run 256 threads each, one runs 512
    uint32_t qcap = 0;
    bool optr = false;
};

Mf2Plan plan_maxflow_sm(uint32_t n_comp, uint32_t max_comp_nodes, bool express_possible) {
    Mf2Plan pl;
    const char* env = getenv("GDS_MF");  // =global: the round-1 kernel only; =sm: this one whenever it fits
    // (components of the express schedule exist only in k_maxflow_sm: with them in the call the
    //  kernel always runs, and GDS_MF=global is ignored)
    if (env && !strcmp(env, "global") && !express_possible) return pl;
    // shared memory per CTA: header + 4 staged queues + the node arrays of the largest component
    // that should still fit.  Prefer the out-CSR cache unless leaving it out lets all components
    // be resident at once (a batch of segments) where they otherwise would not be.
    auto need = [&](uint32_t nodes, bool optr, uint32_t qcap) {
        return (long long)kMf2HeaderBytes + 16ll * qcap + mf2_node_bytes(nodes, optr);
    };
    const uint32_t nmax = std::min<uint32_t>(max_comp_nodes, kMf2MaxNodes);
    if (nmax == 0 || n_comp == 0) return pl;
    uint32_t qcap = 2048;
    bool optr = true;
    if (const char* e = getenv("GDS_MF_OPTR")) optr = e[0] != '0';
    // the queues shrink before the node arrays do
    while (qcap > 256 && need(nmax, optr, qcap) > kMf2MaxSmem) qcap >>= 1;
    if (need(nmax, optr, qcap) > kMf2MaxSmem) optr = false;
    if (need(nmax, optr, qcap) > kMf2MaxSmem && max_comp_nodes > nmax) return pl;
    long long smem_ll = need(nmax, optr, qcap);
    if (smem_ll > kMf2MaxSmem) smem_ll = kMf2MaxSmem;  // the largest does not fit; smaller ones may
    // CTAs per SM: by shared memory, and never more than two (128 registers x 256 threads each)
    auto resident = [&](long long bytes) {
        return std::min(2, std::max(1, (int)((228 * 1024) / (bytes + 1024))));
    };
    int per_sm = resident(smem_ll);
    if (optr && n_comp > (uint32_t)kNumSMs * per_sm) {
        uint32_t q2 = qcap;
        while (q2 > 512 && resident(need(nmax, false, q2)) <= per_sm) q2 >>= 1;
        const int alt = resident(need(nmax, false, q2));
        if (alt > per_sm) {
            optr = false;
            qcap = q2;
            smem_ll = need(nmax, false, qcap);
            per_sm = alt;
        }
    }
    // One CTA per component with the component's labels next to the SM is a LATENCY design: it wins
    // while (nearly) all components are resident at once.  A batch beyond that (config 5: 512
    // samples of 180 KB each, one per SM, four waves: 3.2 ms) is faster on k_maxflow, whose state
    // lives in L2/HBM but which runs every component concurrently (1.84 ms).
    const bool forced = env && !strcmp(env, "sm");
    pl.classic_ok = !(env && !strcmp(env, "global")) &&
                    (forced || (unsigned long long)n_comp * 2 <= 3ull * kNumSMs * per_sm);
    if (!pl.classic_ok && !express_possible) return pl;
    pl.on = true;
    pl.smem = (int)((smem_ll + 15) & ~15ll);
    pl.per_sm = per_sm;
    pl.qcap = qcap;
    pl.optr = optr;
    return pl;
}

void launch_maxflow_sm(gds_ctx* c, const Mf2Plan& pl, const Mf2Graph& g, const uint32_t* comp_lo,
                       const uint32_t* comp_hi, uint32_t n_comp, uint32_t* wc, uint32_t* qF,
                       uint32_t* qT, uint32_t* qN, uint32_t* qH, const SolveParams& sp,
                       CompStats* cstats, unsigned long long alg_bytes, uint32_t* fb_list,
                       uint32_t* fb_count, const uint32_t* n_comp_dev, MfTotals* mft) {
    KScope ks("maxflow", alg_bytes, c->stream);
    if (pl.per_sm >= 2)
        launch_mf2_shape<256, 0>(c, g, comp_lo, comp_hi, n_comp, wc, qF, qT, qN, qH, sp, cstats, pl.smem, pl.qcap, fb_list, fb_count, pl.optr, pl.per_sm, n_comp_dev, mft);
    else
        launch_mf2_shape<512, 1>(c, g, comp_lo, comp_hi, n_comp, wc, qF, qT, qN, qH, sp, cstats, pl.smem, pl.qcap, fb_list, fb_count, pl.optr, pl.per_sm, n_comp_dev, mft);
    GDS_KERNEL_CHECK();
}

// K3' (sweep.cuh): the minimum-cardinality solve.  One warp per component.
template <int W, int CAP, bool WARP, int SLOT>
void launch_sweep_shape(gds_ctx* c, const SweepGraph& g, const uint32_t* comp_lo, const uint32_t* comp_hi,
                        uint32_t n_comp, const uint32_t* n_comp_dev, uint32_t M, uint32_t* wc,
                        unsigned long long* fail) {
    constexpr int smem = kSweepWarps * (2 * W + 4 * CAP + 2 * 34 + 2 * 32) * 4;
    const int grid = std::max(1, std::min<int>(div_up(n_comp, kSweepWarps), kNumSMs * 8));
    auto kern = WARP ? k_sweep_warp<W, CAP> : k_sweep<W, CAP>;
    if (!(c->sweep_smem_set & (1u << SLOT))) {
        GDS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        c->sweep_smem_set |= 1u << SLOT;
    }
    kern<<<grid, kSweepWarps * 32, smem, c->stream>>>(g, comp_lo, comp_hi, n_comp, n_comp_dev, M, wc, fail);
}

void launch_sweep(gds_ctx* c, const SweepGraph& g, const uint32_t* comp_lo, const uint32_t* comp_hi,
                  uint32_t n_comp, const uint32_t* n_comp_dev, uint32_t M, uint32_t* wc,
                  unsigned long long* fail, uint32_t maxlen, bool one_len,
                  unsigned long long alg_bytes) {
    KScope ks("sweep", alg_bytes, c->stream);
    // one read length: at most a few bundles per position -> one lane walks; several lengths: tens of
    // arrivals per position -> the warp-synchronous walk adds them in parallel
    const int w = maxlen < 256 ? 0 : maxlen < 1024 ? 1 : 2;
    switch (w * 2 + (one_len ? 0 : 1)) {
        case 0: launch_sweep_shape<256, 64, false, 0>(c, g, comp_lo, comp_hi, n_comp, n_comp_dev, M, wc, fail); break;
        case 1: launch_sweep_shape<256, 1024, true, 1>(c, g, comp_lo, comp_hi, n_comp, n_comp_dev, M, wc, fail); break;
        case 2: launch_sweep_shape<1024, 64, false, 2>(c, g, comp_lo, comp_hi, n_comp, n_comp_dev, M, wc, fail); break;
        case 3: launch_sweep_shape<1024, 1024, true, 3>(c, g, comp_lo, comp_hi, n_comp, n_comp_dev, M, wc, fail); break;
        case 4: launch_sweep_shape<4096, 64, false, 4>(c, g, comp_lo, comp_hi, n_comp, n_comp_dev, M, wc, fail); break;
        default: launch_sweep_shape<4096, 1024, true, 5>(c, g, comp_lo, comp_hi, n_comp, n_comp_dev, M, wc, fail); break;
    }
    GDS_KERNEL_CHECK();
}

template <typename K>
void build_bundles(gds_ctx* c, const uint32_t* S, const uint32_t* E, const VLayout& vl,
                   const uint32_t* cross_idx, size_t N, const TileMap& tm, bool local_keys,
                   uint32_t n_nodes, int keybits, int lenbits, uint32_t minlen, int32_t* odiff,
                   const uint32_t* fused_ref_len, uint32_t* stats, uint32_t hint_min,
                   uint32_t hint_max, uint32_t& B_out, uint32_t*& sorted_idx_out, int& passes_out) {
    cudaStream_t st = c->stream;
    const size_t n_items = tm.n_items;
    K* kA = c->keysA.get<K>(n_items);
    K* kB = c->keysB.get<K>(n_items);
    uint32_t* vA = c->valsA.get<uint32_t>(n_items);
    uint32_t* vB = c->valsB.get<uint32_t>(n_items);
    int where;
    if (local_keys) {
        ReadKeys<K, true> rk{S, E, vl, cross_idx, N, lenbits, minlen, fused_ref_len, stats,
                             hint_min, hint_max};
        where = radix_sort_pairs<K, ReadKeys<K, true>>(kA, vA, kB, vB, tm, keybits, c->radix, st,
                                                       c->atomic_rank, &passes_out, &rk);
    } else {
        ReadKeys<K, false> rk{S, E, vl, cross_idx, N, lenbits, minlen, nullptr, stats, 0, 0};
        where = radix_sort_pairs<K, ReadKeys<K, false>>(kA, vA, kB, vB, tm, keybits, c->radix, st,
                                                        c->atomic_rank, &passes_out, &rk);
    }
    const K* keys = where ? kB : kA;
    sorted_idx_out = where ? vB : vA;
    // bundle heads
    const uint32_t n_tiles = tm.n_tiles;
    uint32_t* tc = c->tile_counts.get<uint32_t>(n_tiles + 1);
    GDS_CUDA(cudaMemsetAsync(tc + n_tiles, 0, sizeof(uint32_t), st));
    uint32_t* head_bits = c->head_bits.get<uint32_t>((size_t)n_tiles * (kRsTile / 32));
    {
        KScope ks("heads_count", (sizeof(K) * 8ull + 1ull) * n_items / 8, st);
        k_heads_count<K><<<n_tiles, kHeadThreads, 0, st>>>(keys, tm, tc, head_bits);
        GDS_KERNEL_CHECK();
    }
    exclusive_scan_u32(tc, tc, n_tiles + 1, c->scan, st);
    uint32_t B = 0;
    d2h_sync(c, &B, tc + n_tiles, 1);
    B_out = B;
    if (fused_ref_len) {  // verdict of the validation fused into the first histogram pass
        uint32_t hs[4];
        d2h_sync(c, hs, stats, 4);
        if (hs[2]) throw InputFail{GDS_ERR_RANGE, hs[2], "reads with start > end or end >= ref_len"};
        if (hs[3]) throw InputFail{GDS_ERR_ARG, hs[3], "reads outside the len_min/len_max hints"};
    }
    uint32_t* b_first = c->b_first.get<uint32_t>(B + 1);
    K* b_key = c->b_key.get<K>(B + 1);
    {
        KScope ks("heads_write", n_items / 8ull + (4ull + 2 * sizeof(K)) * B, st);
        k_heads_write<K><<<n_tiles, kHeadWriteThreads, 0, st>>>(keys, tm, tc, head_bits, b_first,
                                                                  b_key);
        GDS_KERNEL_CHECK();
    }
    BundleRec* bund = c->bund.get<BundleRec>(B + 1);
    uint32_t* b_t = c->b_t.get<uint32_t>(B + 1);
    int32_t* diff = c->diff.get<int32_t>(n_nodes + 1);
    uint32_t* outdeg = c->outdeg.get<uint32_t>(n_nodes + 1);
    uint32_t* indeg = c->indeg.get<uint32_t>(n_nodes + 1);
    GDS_CUDA(cudaMemsetAsync(diff, 0, (n_nodes + 1) * sizeof(int32_t), st));
    GDS_CUDA(cudaMemsetAsync(outdeg, 0, (n_nodes + 1) * sizeof(uint32_t), st));
    GDS_CUDA(cudaMemsetAsync(indeg, 0, (n_nodes + 1) * sizeof(uint32_t), st));
    if (B) {
        KScope ks("bundle_fill", (sizeof(K) + 8ull + 12ull + 16ull) * B, st);
        k_bundle_fill<K><<<div_up(B, 256), 256, 0, st>>>(b_key, b_first, sorted_idx_out, B,
                                                         (uint32_t)n_items, lenbits, minlen, vl,
                                                         local_keys, bund, b_t, diff, outdeg, indeg,
                                                         odiff);
        GDS_KERNEL_CHECK();
    }
}

// Sort-free K2 (direct.cuh).  Eligible when no sample is segmented and every sample's key space
// (ref_len x number of distinct read lengths) fits in one SM's shared memory.
struct DirectPlan {
    bool on = false;
    DirectLayout dl{};
    uint32_t* ghist = nullptr;
    uint32_t ktot = 0, kmax = 0, n_items = 0;
    uint32_t* in_bid = nullptr;  // identity in-CSR (single read length), else null
    bool global = false;         // counters in global memory (several lengths / segmented reference)
    GDirectLayout gl{};
    // lazy: no readback between the kernels — B is an upper bound on the host, the exact count
    // lives in *B_dev, and input errors are looked at with the final readback
    bool lazy = false;
    const uint32_t* B_dev = nullptr;
};

// slots of the small device array `stats` (uint32 x 64) beyond the validation counters [0..4] and the
// 64-bit totals at [8..19]: counts that stay on the device in lazy mode, and the K3 totals
constexpr int kStatB = 20, kStatNComp = 21, kStatCtl = 24, kStatMf = 32, kStatRes = 52, kStatWords = 64;

bool direct_eligible(const gds_reads* rd, uint32_t ns, uint32_t minlen, uint32_t maxlen,
                     const uint32_t* S, const uint32_t* E) {
    if (((uintptr_t)S | (uintptr_t)E) & 15) return false;  // 16-byte loads
    const uint64_t nlen = (uint64_t)maxlen - minlen + 1;
    uint64_t tot = 0;
    for (uint32_t k = 0; k < ns; ++k) {
        const uint64_t kk = ((uint64_t)rd->ref_len[k] + 1) * nlen;  // one slot row per node
        if (kk > kDirectMaxKeys) return false;
        tot += (kk + 31) & ~31ull;
    }
    return tot < (1ull << 31);
}

void build_bundles_direct(gds_ctx* c, const gds_reads* rd, const uint32_t* S, const uint32_t* E,
                          const uint64_t* foff_dev, const std::vector<uint64_t>& foff_host,
                          const uint32_t* reflen_d, const uint32_t* base_d, uint32_t ns, size_t N,
                          uint32_t n_nodes, uint32_t minlen, uint32_t maxlen, uint32_t* stats,
                          DirectPlan& plan, uint32_t& B_out) {
    cudaStream_t st = c->stream;
    const uint32_t nlen = maxlen - minlen + 1;
    // host-side layout: histogram regions and work items (sample parts)
    std::vector<uint32_t> lay(2 * (ns + 1), 0);
    uint32_t* kbase = lay.data();
    uint32_t* item_off = lay.data() + ns + 1;
    const uint64_t part_len = std::max<uint64_t>(65536, (N + 8ull * kNumSMs - 1) / (8ull * kNumSMs));
    uint32_t kmax = 32;
    for (uint32_t k = 0; k < ns; ++k) {
        const uint32_t kk = ((rd->ref_len[k] + 1) * nlen + 31u) & ~31u;
        kmax = std::max(kmax, kk);
        kbase[k + 1] = kbase[k] + kk;
        const uint64_t nk = foff_host[k + 1] - foff_host[k];
        item_off[k + 1] = item_off[k] + (uint32_t)((nk + part_len - 1) / part_len);
    }
    const uint32_t ktot = kbase[ns], n_items = item_off[ns];
    uint32_t* lay_d = c->dlay.get<uint32_t>(lay.size());
    // on the solve's own stream: a copy on the legacy stream is not ordered against it (pageable
    // sources are staged before the call returns, so the vector may go out of scope)
    GDS_CUDA(cudaMemcpyAsync(lay_d, lay.data(), lay.size() * 4, cudaMemcpyHostToDevice, st));
    uint32_t* ghist = c->dhist.get<uint32_t>(ktot);
    uint32_t* wc = c->dwork.get<uint32_t>(2);
    GDS_CUDA(cudaMemsetAsync(ghist, 0, (size_t)ktot * 4, st));
    GDS_CUDA(cudaMemsetAsync(wc, 0, 8, st));
    DirectLayout dl{foff_dev, reflen_d, base_d, lay_d, lay_d + ns + 1, ns, nlen, minlen, maxlen};
    const unsigned smem = kmax * 4;
    if (smem > c->direct_attr) {
        GDS_CUDA(cudaFuncSetAttribute(k_direct_hist, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(kDirectMaxKeys * 4)));
        GDS_CUDA(cudaFuncSetAttribute(k_direct_select, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(kDirectMaxKeys * 4)));
        GDS_CUDA(cudaFuncSetAttribute(k_direct_mark<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(kDmQueueBytes + kDirectMaxKeys)));
        GDS_CUDA(cudaFuncSetAttribute(k_direct_mark<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(kDmQueueBytes + kDirectMaxKeys)));
        c->direct_attr = kDirectMaxKeys * 4;
    }
    {
        KScope ks("direct_hist", 8ull * N + 4ull * ktot, st);
        const int grid = (int)std::min<uint32_t>(n_items, (uint32_t)kNumSMs);
        k_direct_hist<<<grid, kDhThreads, smem, st>>>(S, E, dl, n_items, wc, ghist, kmax, stats);
        GDS_KERNEL_CHECK();
    }
    const uint32_t n_tiles = (uint32_t)div_up(ktot, kDkTile);
    uint32_t* tc = c->tile_counts.get<uint32_t>(n_tiles + 1);
    GDS_CUDA(cudaMemsetAsync(tc + n_tiles, 0, sizeof(uint32_t), st));
    {
        KScope ks("direct_count", 4ull * ktot, st);
        k_direct_count<<<n_tiles, kDkThreads, 0, st>>>(ghist, ktot, tc);
        GDS_KERNEL_CHECK();
    }
    exclusive_scan_u32(tc, tc, n_tiles + 1, c->scan, st);
    uint32_t B = 0;
    if (plan.lazy) {  // the count stays on the device (stats[kStatB]); size everything by its bound
        GDS_CUDA(cudaMemcpyAsync(stats + kStatB, tc + n_tiles, 4, cudaMemcpyDeviceToDevice, st));
        plan.B_dev = stats + kStatB;
        B = (uint32_t)std::min<uint64_t>(ktot, N);
    } else {
        d2h_sync(c, &B, tc + n_tiles, 1);
        uint32_t hs[4];
        d2h_sync(c, hs, stats, 4);
        if (hs[2]) throw InputFail{GDS_ERR_RANGE, hs[2], "reads with start > end or end >= ref_len"};
        if (hs[3]) throw InputFail{GDS_ERR_ARG, hs[3], "reads outside the len_min/len_max hints"};
    }
    B_out = B;
    BundleRec* bund = c->bund.get<BundleRec>(B + 1);
    uint32_t* b_t = c->b_t.get<uint32_t>(B + 1);
    uint32_t* b_slot = c->b_slot.get<uint32_t>(B + 1);
    uint32_t* ident = nlen == 1 ? c->ident.get<uint32_t>(B + 1) : nullptr;
    int32_t* diff = c->diff.get<int32_t>(n_nodes + 1);
    uint32_t* outdeg = c->outdeg.get<uint32_t>(n_nodes + 1);
    uint32_t* indeg = c->indeg.get<uint32_t>(n_nodes + 1);
    // one read length: k_direct_bundles writes the difference array of every node itself
    if (nlen == 1 && B) GDS_CUDA(cudaMemsetAsync(diff + n_nodes, 0, sizeof(int32_t), st));
    else GDS_CUDA(cudaMemsetAsync(diff, 0, (n_nodes + 1) * sizeof(int32_t), st));
    GDS_CUDA(cudaMemsetAsync(outdeg, 0, (n_nodes + 1) * sizeof(uint32_t), st));
    GDS_CUDA(cudaMemsetAsync(indeg, 0, (n_nodes + 1) * sizeof(uint32_t), st));
    if (B) {
        KScope ks("direct_bundles", 4ull * ktot + 40ull * B, st);
        k_direct_bundles<<<n_tiles, kDkThreads, 0, st>>>(ghist, ktot, dl, tc, bund, b_t, b_slot,
                                                        ident, diff, outdeg, indeg);
        GDS_KERNEL_CHECK();
    }
    plan.on = true;
    plan.dl = dl;
    plan.ghist = ghist;
    plan.ktot = ktot;
    plan.kmax = kmax;
    plan.n_items = n_items;
    plan.in_bid = ident;
}

// The same with the counters in global memory (direct.cuh: k_gdirect_*): any layout whose key space
// (virtual nodes x read lengths) stays L2-sized.
void build_bundles_gdirect(gds_ctx* c, const uint32_t* S, const uint32_t* E, const VLayout& vl,
                           size_t N, uint32_t n_nodes, uint32_t minlen, uint32_t maxlen,
                           int32_t* odiff, uint32_t* stats, DirectPlan& plan, uint32_t& B_out,
                           uint64_t& n_cross_out) {
    cudaStream_t st = c->stream;
    const uint32_t nlen = maxlen - minlen + 1;
    const uint32_t ktot = (uint32_t)((((uint64_t)n_nodes * nlen) + 31) & ~31ull);
    uint32_t* ghist = c->dhist.get<uint32_t>(ktot);
    GDS_CUDA(cudaMemsetAsync(ghist, 0, (size_t)ktot * 4, st));
    GDirectLayout gl{vl, nlen, minlen, maxlen};
    {
        KScope ks("gdirect_hist", 8ull * N + 4ull * ktot, st);
        k_gdirect_hist<<<div_up((long long)N, kGdTile), kGdThreads, 0, st>>>(S, E, N, gl, ghist, stats);
        GDS_KERNEL_CHECK();
    }
    const uint32_t n_tiles = (uint32_t)div_up(ktot, kDkTile);
    uint32_t* tc = c->tile_counts.get<uint32_t>(n_tiles + 1);
    GDS_CUDA(cudaMemsetAsync(tc + n_tiles, 0, sizeof(uint32_t), st));
    {
        KScope ks("direct_count", 4ull * ktot, st);
        k_direct_count<<<n_tiles, kDkThreads, 0, st>>>(ghist, ktot, tc);
        GDS_KERNEL_CHECK();
    }
    exclusive_scan_u32(tc, tc, n_tiles + 1, c->scan, st);
    uint32_t B = 0;
    if (plan.lazy) {
        GDS_CUDA(cudaMemcpyAsync(stats + kStatB, tc + n_tiles, 4, cudaMemcpyDeviceToDevice, st));
        plan.B_dev = stats + kStatB;
        B = (uint32_t)std::min<uint64_t>(ktot, 2 * (uint64_t)N);  // a read crossing a cut counts twice
        n_cross_out = 0;  // known with the final readback
    } else {
        d2h_sync(c, &B, tc + n_tiles, 1);
        uint32_t hs[5];
        d2h_sync(c, hs, stats, 5);
        if (hs[2]) throw InputFail{GDS_ERR_RANGE, hs[2], "reads with start > end or end >= ref_len"};
        if (hs[3]) throw InputFail{GDS_ERR_ARG, hs[3], "reads outside the len_min/len_max hints"};
        n_cross_out = hs[4];
    }
    B_out = B;
    BundleRec* bund = c->bund.get<BundleRec>(B + 1);
    uint32_t* b_t = c->b_t.get<uint32_t>(B + 1);
    uint32_t* b_slot = c->b_slot.get<uint32_t>(B + 1);
    uint32_t* ident = nlen == 1 ? c->ident.get<uint32_t>(B + 1) : nullptr;
    int32_t* diff = c->diff.get<int32_t>(n_nodes + 1);
    uint32_t* outdeg = c->outdeg.get<uint32_t>(n_nodes + 1);
    uint32_t* indeg = c->indeg.get<uint32_t>(n_nodes + 1);
    GDS_CUDA(cudaMemsetAsync(diff, 0, (n_nodes + 1) * sizeof(int32_t), st));
    GDS_CUDA(cudaMemsetAsync(outdeg, 0, (n_nodes + 1) * sizeof(uint32_t), st));
    GDS_CUDA(cudaMemsetAsync(indeg, 0, (n_nodes + 1) * sizeof(uint32_t), st));
    if (B) {
        KScope ks("gdirect_bundles", 4ull * ktot + 40ull * B, st);
        k_gdirect_bundles<<<n_tiles, kDkThreads, 0, st>>>(ghist, ktot, gl, tc, bund, b_t, b_slot, ident,
                                                         diff, outdeg, indeg, odiff);
        GDS_KERNEL_CHECK();
    }
    plan.on = true;
    plan.global = true;
    plan.gl = gl;
    plan.ghist = ghist;
    plan.ktot = ktot;
    plan.in_bid = ident;
}

// K5 on the direct path (direct.cuh): classify the bundles, mark the reads of saturated bundles in
// one parallel streaming pass, rank the candidates of partial bundles; the ordered walk is the
// fallback when the candidates do not fit (or GDS_DIRECT_SELECT=walk asks for it).
// force_walk: the ordered walk right away (the lazy path's second attempt after ctl flag 1).
// Lazy mode (dp.lazy): nothing is read back here.  The candidate buffer keeps the size it has
// (never below N/8 slots); k_direct_classify raises ctl flag 2 when the candidates do not fit and
// flag 1 for a partial bundle too large for one warp, the mark / ranking kernels then do nothing,
// and gds_solve — which sees the flags with its one final readback — repeats the selection.
void direct_select(gds_ctx* c, const DirectPlan& dp, const uint32_t* S, const uint32_t* E,
                   uint32_t ns, size_t N, uint32_t B, uint32_t* bm, unsigned long long* totals,
                   uint32_t* stats, gds_result* out, bool force_walk, size_t cand_need) {
    cudaStream_t st = c->stream;
    BundleRec* bund = c->bund.as<BundleRec>();
    uint32_t* b_slot = c->b_slot.as<uint32_t>();
    const char* env = getenv("GDS_DIRECT_SELECT");
    bool walk = !dp.global && (force_walk || (env && !strcmp(env, "walk")));
    uint32_t* ctl = c->dctl.get<uint32_t>(4);
    GDS_CUDA(cudaMemsetAsync(ctl, 0, 16, st));
    if (!walk) {
        uint32_t* kstat = c->kstat.get<uint32_t>(dp.ktot / 16 + 1);
        uint32_t* pb = c->pbund.get<uint32_t>(3 * ((size_t)B + 1));
        uint32_t* fill = pb + 2 * ((size_t)B + 1);
        GDS_CUDA(cudaMemsetAsync(kstat, 0, ((size_t)dp.ktot / 16 + 1) * 4, st));
        // never below N/8 slots: the share of reads in partial bundles varies from call to call
        // and regrowing the arena is expensive
        size_t cand_cap = std::max<size_t>({cand_need, N / 8, c->cand.cap / 4, (size_t)1});
        cand_cap = std::min<size_t>(cand_cap, 0xffffffffu);
        uint32_t* cand = dp.lazy ? c->cand.get<uint32_t>(cand_cap) : nullptr;
        {
            // a partial bundle beyond kMaxPartialMult reads sends the shared-memory path to the
            // ordered walk; the global path has no walk and lets one warp grind through it
            KScope ks("direct_classify", 20ull * B, st);
            k_direct_classify<<<div_up(B, 256), 256, 0, st>>>(
                bund, b_slot, B, dp.ghist, kstat, pb, pb + B + 1, fill, ctl,
                dp.global ? 0xffffffffu : kMaxPartialMult, dp.B_dev,
                dp.lazy ? (uint32_t)cand_cap : 0xffffffffu, stats);
            GDS_KERNEL_CHECK();
        }
        uint32_t hctl[4] = {1, 0, 0, 0};  // lazy: the ranking kernel is launched unconditionally
        if (!dp.lazy) {
            d2h_sync(c, hctl, ctl, 4);  // candidate buffer sized exactly
            out->partial_bundles = hctl[0];
            out->partial_candidates = hctl[1];
            walk = (hctl[2] & 1u) != 0;
            if (!walk) cand = c->cand.get<uint32_t>(std::max<size_t>((size_t)hctl[1] + 1, N / 8));
        }
        if (!walk) {
            const unsigned long long per_read = (dp.global || dp.dl.nlen > 1) ? 8 : 4;
            if (dp.global) {
                KScope ks("gdirect_mark", per_read * N + dp.ktot / 4 + 8ull * N / 32, st);
                k_gdirect_mark<<<div_up((long long)N, kGdTile), kGdThreads, 0, st>>>(
                    S, E, N, dp.gl, dp.ghist, kstat, pb, fill, cand, bm, totals, ctl);
                GDS_KERNEL_CHECK();
            } else {
                KScope ks("direct_mark", per_read * N + dp.ktot / 4 + 8ull * N / 32, st);
                uint32_t* wc = c->dwork.as<uint32_t>() + 1;
                GDS_CUDA(cudaMemsetAsync(wc, 0, 4, st));
                const int grid = (int)std::min<uint32_t>(
                    dp.n_items * kDmSplit, (uint32_t)kNumSMs * (dp.dl.nlen == 1 ? kDmCtasPerSm : 2));
                const unsigned smem = kDmQueueBytes + dp.kmax;
                if (dp.dl.nlen == 1)
                    k_direct_mark<true><<<grid, kDmThreads, smem, st>>>(S, E, dp.dl, dp.n_items, wc,
                                                                       dp.ghist, kstat, pb, fill, cand,
                                                                       ctl, bm, totals);
                else
                    k_direct_mark<false><<<grid, kDmThreads, smem, st>>>(S, E, dp.dl, dp.n_items, wc,
                                                                        dp.ghist, kstat, pb, fill, cand,
                                                                        ctl, bm, totals);
                GDS_KERNEL_CHECK();
            }
            if (hctl[0]) {
                KScope ks("direct_partial", dp.lazy ? 16ull * (N / 64) : 16ull * hctl[0] + 4ull * hctl[1], st);
                if (dp.global)  // segments of a long reference: ~10 reads per bundle, half a warp each
                    k_direct_partial<true><<<kNumSMs * 32, 256, 0, st>>>(pb, pb + B + 1, fill, cand, ctl,
                                                                        bm, totals);
                else
                    k_direct_partial<false><<<kNumSMs * 32, 256, 0, st>>>(pb, pb + B + 1, fill, cand, ctl,
                                                                         bm, totals);
                GDS_KERNEL_CHECK();
            }
            if (dp.lazy)
                GDS_CUDA(cudaMemcpyAsync(stats + kStatCtl, ctl, 16, cudaMemcpyDeviceToDevice, st));
            return;
        }
    }
    // ordered walk: one CTA per sample, quota per key in shared memory
    {
        KScope ks("direct_quota", 24ull * B, st);
        k_direct_quota<<<div_up(B, 256), 256, 0, st>>>(bund, b_slot, B, dp.ghist, dp.B_dev);
        GDS_KERNEL_CHECK();
    }
    {
        KScope ks("direct_walk", 4ull * dp.ktot + 8ull * N / 32, st);
        uint32_t* wc = c->dwork.as<uint32_t>() + 1;
        GDS_CUDA(cudaMemsetAsync(wc, 0, 4, st));
        const int grid = (int)std::min<uint32_t>(ns, (uint32_t)kNumSMs);
        k_direct_select<<<grid, kDsThreads, dp.kmax * 4, st>>>(S, E, dp.dl, wc, dp.ghist, bm, totals);
        GDS_KERNEL_CHECK();
    }
    if (dp.lazy) GDS_CUDA(cudaMemcpyAsync(stats + kStatCtl, ctl, 16, cudaMemcpyDeviceToDevice, st));
}

}  // namespace

extern "C" int gds_abi_version(void) { return GDS_ABI_VERSION; }

extern "C" int gds_create(int device, gds_ctx** out) {
    if (!out) return GDS_ERR_ARG;
    *out = nullptr;
    gds_ctx* c = new (std::nothrow) gds_ctx();
    if (!c) return GDS_ERR_NOMEM;
    c->device = device;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMallocHost(&c->pinned, gds_ctx::kPinnedBytes);
    for (int i = 0; i < EV_COUNT && e == cudaSuccess; ++i) e = cudaEventCreate(&c->ev[i]);
    if (e != cudaSuccess) {
        // no device, no driver, wrong arch: there is no CPU path to fall back to
        fprintf(stderr, "gds_create: CUDA device %d unusable: %s\n", device, cudaGetErrorString(e));
        cudaGetLastError();
        delete c;
        return GDS_ERR_CUDA;
    }
    c->stream = c->own_stream;
    c->atomic_rank = atomic_rank_is_stable(device, c->own_stream);
    *out = c;
    return GDS_OK;
}

extern "C" void gds_destroy(gds_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    c->prof.release();
    for (int i = 0; i < EV_COUNT; ++i)
        if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    if (c->pinned) cudaFreeHost(c->pinned);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

extern "C" void* gds_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

extern "C" void gds_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

extern "C" const char* gds_last_error(const gds_ctx* c) { return c ? c->err.c_str() : "null context"; }

extern "C" int gds_set_stream(gds_ctx* c, void* cuda_stream) {
    if (!c) return GDS_ERR_ARG;
    c->stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : c->own_stream;
    return GDS_OK;
}

extern "C" uint32_t gds_kernel_profile(gds_ctx* c, gds_kernel_stat* outp, uint32_t cap) {
    // aggregates the per-launch event pairs of the GDS_PROFILE_KERNELS calls since the last reset
    if (!c) return 0;
    std::vector<gds_kernel_stat> agg;
    for (const KRec& r : c->prof.recs) {
        float t = 0;
        if (cudaEventElapsedTime(&t, r.e0, r.e1) != cudaSuccess) {
            cudaGetLastError();
            continue;
        }
        gds_kernel_stat* hit = nullptr;
        for (auto& a : agg)
            if (!strncmp(a.name, r.name, sizeof a.name)) hit = &a;
        if (!hit) {
            gds_kernel_stat z{};
            strncpy(z.name, r.name, sizeof z.name - 1);
            agg.push_back(z);
            hit = &agg.back();
        }
        hit->ms += t;
        hit->bytes += r.bytes;
        hit->launches += 1;
    }
    for (uint32_t i = 0; i < agg.size() && i < cap && outp; ++i) outp[i] = agg[i];
    return (uint32_t)agg.size();
}

extern "C" void gds_kernel_profile_reset(gds_ctx* c) {
    if (c) c->prof.reset();
}

extern "C" uint64_t gds_bitmap_to_indices(const uint32_t* bitmap, uint64_t n_bits,
                                          uint64_t* indices, uint64_t cap) {
    // counts per chunk of words, then every chunk writes its slice: up to 16 host threads (a 50 M
    // read solve keeps 17 M indices = 134 MB; one thread needs longer for that than the device
    // for the whole path)
    const uint64_t words = (n_bits + 31) / 32;
    auto word_at = [&](uint64_t w) {
        uint32_t x = bitmap[w];
        if (w == words - 1 && (n_bits & 31)) x &= (1u << (n_bits & 31)) - 1u;  // bits past the end
        return x;
    };
    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    const unsigned nt = words < (1u << 16) ? 1u : std::min<unsigned>({hw, 16u, (unsigned)(words >> 14)});
    const uint64_t per = (words + nt - 1) / nt;
    std::vector<uint64_t> cnt(nt + 1, 0);
    auto run = [&](auto fn) {
        if (nt == 1) {
            fn(0u);
            return;
        }
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nt; ++t) th.emplace_back([=, &fn] { fn(t); });
        for (auto& t : th) t.join();
    };
    run([&](unsigned t) {
        uint64_t c = 0;
        for (uint64_t w = std::min(words, t * per), we = std::min(words, (t + 1) * per); w < we; ++w)
            c += (uint64_t)__builtin_popcount(word_at(w));
        cnt[t + 1] = c;
    });
    for (unsigned t = 0; t < nt; ++t) cnt[t + 1] += cnt[t];
    if (indices && cap) {
        run([&](unsigned t) {
            uint64_t o = cnt[t];
            for (uint64_t w = std::min(words, t * per), we = std::min(words, (t + 1) * per); w < we; ++w) {
                uint32_t x = word_at(w);
                while (x) {
                    const int bit = __builtin_ctz(x);
                    x &= x - 1;
                    if (o < cap) indices[o] = w * 32 + bit;
                    ++o;
                }
            }
        });
    }
    return cnt[nt];
}

extern "C" int gds_solve(gds_ctx* c, const gds_reads* rd, const gds_filter* flt,
                         uint32_t max_coverage, const gds_params* prm, uint32_t flags,
                         gds_result* out) {
    if (!c) return GDS_ERR_ARG;
    c->err.clear();
    if (!rd || !out || rd->n_samples == 0 || !rd->read_off || !rd->ref_len)
        return fail(c, GDS_ERR_ARG, "null reads/result or n_samples == 0");
    const uint32_t ns = rd->n_samples;
    const uint64_t P = rd->read_off[ns];
    if (rd->read_off[0] != 0) return fail(c, GDS_ERR_ARG, "read_off[0] must be 0");
    for (uint32_t k = 0; k < ns; ++k)
        if (rd->read_off[k + 1] < rd->read_off[k])
            return fail(c, GDS_ERR_ARG, "read_off must be non-decreasing");
    if (P > 0 && !rd->start && !rd->start16) return fail(c, GDS_ERR_ARG, "null start");
    const bool fixed_len = rd->len_min != 0 && rd->len_min == rd->len_max;
    if (P > 0 && !rd->end && !fixed_len)
        return fail(c, GDS_ERR_ARG, "end may only be omitted with len_min == len_max != 0");
    if (rd->start16)
        for (uint32_t k = 0; k < ns; ++k)
            if (rd->ref_len[k] > 65536u)
                return fail(c, GDS_ERR_ARG, "start16 needs every ref_len <= 65536");
    const bool compact = P > 0 && (rd->start16 || !rd->end);
    if (P >= (1ull << 32) - 64) return fail(c, GDS_ERR_RANGE, "more than 2^32 reads in one call");
    const bool use_filter = flt != nullptr;
    if (use_filter) {
        if (P > 0 && (!rd->mapq || !rd->seq_len))
            return fail(c, GDS_ERR_ARG, "filter needs mapq and seq_len");
        for (uint32_t k = 0; k <= ns; ++k)
            if (rd->read_off[k] & 1)
                return fail(c, GDS_ERR_ARG, "filter needs an even read count per sample (mates adjacent)");
        if (flt->n_amplicons && (!flt->amp_start || !flt->amp_end))
            return fail(c, GDS_ERR_ARG, "null amplicon table");
    }
    if (flags & GDS_FIND_PAIRS)  // mates are read 2i and 2i+1 of a sample: a pair must not straddle two
        for (uint32_t k = 0; k <= ns; ++k)
            if (rd->read_off[k] & 1)
                return fail(c, GDS_ERR_ARG, "GDS_FIND_PAIRS needs an even read count per sample (mates adjacent)");
    uint64_t nn64 = 0;
    std::vector<uint32_t> base(ns + 1, 0);  // original node space: sample k owns ref_len[k]+1 nodes
    for (uint32_t k = 0; k < ns; ++k) {
        nn64 += (uint64_t)rd->ref_len[k] + 1;
        if (nn64 >= kLabelInf) return fail(c, GDS_ERR_RANGE, "total reference length beyond 2^30 nodes");
        base[k + 1] = (uint32_t)nn64;
    }
    const uint32_t n_onodes = (uint32_t)nn64;
    uint32_t n_nodes = n_onodes;  // virtual node space (grows when long references are segmented)
    const bool in_dev = flags & GDS_INPUT_ON_DEVICE;
    const bool out_dev = flags & GDS_OUTPUT_ON_DEVICE;
    SolveParams sp{64, 150, 1, 0};
    if (prm && (prm->gr_interval_min | prm->gr_levels_pct | prm->gr_relabel_pct | prm->max_rounds)) {
        sp.gr_interval_min = prm->gr_interval_min;
        sp.gr_levels_pct = prm->gr_levels_pct;
        sp.gr_relabel_pct = prm->gr_relabel_pct;
        sp.max_rounds = prm->max_rounds;
    }
    uint32_t seg_len =
        (prm && prm->seg_len) ? prm->seg_len : default_seg_len(rd->n_samples, rd->ref_len);
    const uint32_t algorithm = prm ? prm->algorithm : 0u;
    uint32_t schedule = prm ? prm->schedule : 0u;
    if (schedule > 3) return fail(c, GDS_ERR_ARG, "gds_params.schedule must be 0, 1, 2 or 3");
    // a call that filters by an amplicon table works on amplicon-tiled coverage, which dips between
    // the amplicons whatever M is: the default then is the graph reduction at every M (config 2:
    // 6.1 -> 3.6 ms).  A call-level choice like the filter itself, never a property of the batch.
    if (schedule == 0 && flt && flt->n_amplicons > 0) schedule = 3;
    if (algorithm > 1) return fail(c, GDS_ERR_ARG, "gds_params.algorithm must be 0 (quasi-MCP) or 1 (minimum cardinality)");
    // scalars of the result start clean (buffers are left alone)
    {
        gds_result keep = *out;
        memset(out, 0, sizeof *out);
        out->kept_bitmap = keep.kept_bitmap;
        out->pair_pass = keep.pair_pass;
        out->filt_off = keep.filt_off;
        out->cov_capped = keep.cov_capped;
        out->demand = keep.demand;
    }
    out->seg_len = seg_len;
    out->n_reads_in = P;
    out->n_nodes = n_onodes;

    struct ProfGuard {
        ProfGuard(Profiler* p) { cur_prof() = p; }
        ~ProfGuard() { cur_prof() = nullptr; }
    } prof_guard(&c->prof);
    c->prof.on = (flags & GDS_PROFILE_KERNELS) != 0;
    if (!c->prof.on) c->prof.reset();  // profiled calls accumulate until gds_kernel_profile_reset
    const unsigned long long launches0 = launch_counter();
    try {
        GDS_CUDA(cudaSetDevice(c->device));
        cudaStream_t st = c->stream;
        GDS_CUDA(cudaEventRecord(c->ev[EV_BEGIN], st));

        // ---------------- inputs ----------------
        const uint32_t *dS, *dE, *dLen = nullptr;
        const uint8_t* dQ = nullptr;
        if (in_dev || P == 0) {
            dS = rd->start;
            dE = rd->end;
            dQ = rd->mapq;
            dLen = rd->seq_len;
        } else {
            // compact transport: only the narrow start column (and the ends, if given) cross PCIe
            uint32_t* s = c->in_start.get<uint32_t>(P);
            uint32_t* e = c->in_end.get<uint32_t>(P);
            if (rd->start16) {
                uint16_t* raw = c->in_raw.get<uint16_t>(P + 8);
                GDS_CUDA(cudaMemcpyAsync(raw, rd->start16, P * 2, cudaMemcpyHostToDevice, st));
            } else {
                GDS_CUDA(cudaMemcpyAsync(s, rd->start, P * 4, cudaMemcpyHostToDevice, st));
            }
            if (rd->end) GDS_CUDA(cudaMemcpyAsync(e, rd->end, P * 4, cudaMemcpyHostToDevice, st));
            dS = s;
            dE = e;
            if (use_filter) {
                uint8_t* q = c->in_mapq.get<uint8_t>(P);
                uint32_t* l = c->in_len.get<uint32_t>(P);
                GDS_CUDA(cudaMemcpyAsync(q, rd->mapq, P, cudaMemcpyHostToDevice, st));
                GDS_CUDA(cudaMemcpyAsync(l, rd->seq_len, P * 4, cudaMemcpyHostToDevice, st));
                dQ = q;
                dLen = l;
            }
        }
        if (compact) {  // widen to the 32-bit columns (k_expand_reads)
            const uint16_t* s16 = nullptr;
            const uint32_t* s32 = nullptr;
            const uint32_t* e32 = nullptr;
            uint32_t* s = c->in_start.get<uint32_t>(P);
            uint32_t* e = c->in_end.get<uint32_t>(P);
            if (in_dev) {
                s16 = rd->start16;
                s32 = rd->start16 ? nullptr : rd->start;
                e32 = rd->end;
            } else {
                s16 = rd->start16 ? c->in_raw.as<uint16_t>() : nullptr;
                s32 = rd->start16 ? nullptr : s;
                e32 = rd->end ? e : nullptr;
            }
            uint32_t* So = (s32 && ((uintptr_t)s32 & 15) == 0) ? const_cast<uint32_t*>(s32) : s;
            uint32_t* Eo = e32 ? const_cast<uint32_t*>(e32) : e;
            {
                KScope ks("expand_reads", (s16 ? 2ull : 4ull) * P + (So != s32 ? 4ull : 0ull) * P +
                                              (e32 ? 0ull : 4ull) * P, st);
                k_expand_reads<<<div_up((long long)P, 256 * 8), 256, 0, st>>>(s16, s32, e32, rd->len_min,
                                                                             P, So, Eo);
                GDS_KERNEL_CHECK();
            }
            dS = So;
            dE = Eo;
        }
        uint64_t* off_d = c->off_d.get<uint64_t>(ns + 1);
        uint32_t* reflen_d = c->reflen_d.get<uint32_t>(ns);
        uint32_t* base_d = c->base_d.get<uint32_t>(ns + 1);
        GDS_CUDA(cudaMemcpyAsync(off_d, rd->read_off, (ns + 1) * 8, cudaMemcpyHostToDevice, st));
        GDS_CUDA(cudaMemcpyAsync(reflen_d, rd->ref_len, ns * 4, cudaMemcpyHostToDevice, st));
        GDS_CUDA(cudaMemcpyAsync(base_d, base.data(), (ns + 1) * 4, cudaMemcpyHostToDevice, st));
        uint32_t* stats = c->small.get<uint32_t>(kStatWords);
        unsigned long long* totals = reinterpret_cast<unsigned long long*>(stats + 8);
        MfTotals* mft = reinterpret_cast<MfTotals*>(stats + kStatMf);
        static_assert(kStatMf * 4 + sizeof(MfTotals) <= kStatWords * 4 && kStatMf % 2 == 0, "stats layout");
        {
            uint32_t init[kStatWords] = {};
            init[0] = 0xffffffffu;
            memcpy(c->pinned, init, sizeof init);
            GDS_CUDA(cudaMemcpyAsync(stats, c->pinned, sizeof init, cudaMemcpyHostToDevice, st));
        }
        GDS_CUDA(cudaEventRecord(c->ev[EV_H2D], st));

        // ---------------- K1: filter ----------------
        const uint32_t* S = dS;
        const uint32_t* E = dE;
        const uint64_t* foff_dev = off_d;
        uint64_t N = P;
        std::vector<uint64_t> foff_host(rd->read_off, rd->read_off + ns + 1);
        if (use_filter && P > 0) {
            const size_t n_pairs = P / 2;
            FilterArgs fa{flt->min_seq_length, flt->min_mapq, flt->n_amplicons, nullptr, nullptr};
            std::vector<uint32_t> as, ae;  // must outlive the async upload
            if (flt->n_amplicons) {
                std::vector<std::pair<uint32_t, uint32_t>> amps(flt->n_amplicons);
                for (uint32_t i = 0; i < flt->n_amplicons; ++i)
                    amps[i] = {flt->amp_start[i], flt->amp_end[i]};
                std::sort(amps.begin(), amps.end());
                as.resize(amps.size());
                ae.resize(amps.size());
                uint32_t run = 0;
                for (size_t i = 0; i < amps.size(); ++i) {
                    run = std::max(run, amps[i].second);
                    as[i] = amps[i].first;
                    ae[i] = run;
                }
                uint32_t* das = c->amp_s.get<uint32_t>(as.size());
                uint32_t* dae = c->amp_e.get<uint32_t>(ae.size());
                GDS_CUDA(cudaMemcpyAsync(das, as.data(), as.size() * 4, cudaMemcpyHostToDevice, st));
                GDS_CUDA(cudaMemcpyAsync(dae, ae.data(), ae.size() * 4, cudaMemcpyHostToDevice, st));
                fa.amp_start_sorted = das;
                fa.amp_end_runmax = dae;
            }
            uint8_t* pp = (out_dev && out->pair_pass) ? out->pair_pass
                                                      : c->pair_pass.get<uint8_t>(n_pairs);
            uint32_t* f32 = c->flag32.get<uint32_t>(n_pairs);
            int grid = std::min<long long>(div_up(n_pairs, 256), kNumSMs * 16);
            {
                KScope ks("filter_flags", 13ull * P + 5ull * n_pairs, st);
                k_filter_flags<<<grid, 256, 0, st>>>(dS, dE, dQ, dLen, n_pairs, fa, pp, f32);
                GDS_KERNEL_CHECK();
            }
            exclusive_scan_u32(f32, f32, n_pairs, c->scan, st);
            uint64_t* foff = c->foff_d.get<uint64_t>(ns + 1);
            {
                KScope ks("filter_offsets", 16ull * (ns + 1), st);
                k_filter_offsets<<<div_up(ns + 1, 128), 128, 0, st>>>(off_d, ns, f32, pp, n_pairs, foff);
                GDS_KERNEL_CHECK();
            }
            d2h_sync(c, foff_host.data(), foff, ns + 1);
            N = foff_host[ns];
            uint32_t* fS = c->fS.get<uint32_t>(N);
            uint32_t* fE = c->fE.get<uint32_t>(N);
            {
                KScope ks("filter_compact", 5ull * n_pairs + 16ull * N, st);
                k_filter_compact<<<grid, 256, 0, st>>>(dS, dE, pp, f32, n_pairs, fS, fE);
                GDS_KERNEL_CHECK();
            }
            S = fS;
            E = fE;
            foff_dev = foff;
            if (!out_dev) deliver(c, out->pair_pass, pp, n_pairs, false);
        }
        out->n_filtered = N;
        if (out->filt_off) memcpy(out->filt_off, foff_host.data(), (ns + 1) * 8);
        GDS_CUDA(cudaEventRecord(c->ev[EV_FILTER], st));

        // ---------------- K2: coverage flow graph ----------------
        uint32_t B = 0, n_comp = 0;
        uint32_t* sorted_idx = nullptr;
        int sort_passes = 0;
        uint32_t minlen = 1, maxlen = 1;
        int lenbits = 0;
        // exact read-length bounds from the caller (the host adapter has them for free from its
        // narrowing loop) let the validation ride on the first histogram pass of the sort
        const bool have_hints = rd->len_max != 0 && rd->len_min != 0 && rd->len_min <= rd->len_max;
        bool fused_validation = false;
        if (N > 0 && have_hints) {
            minlen = rd->len_min;
            maxlen = rd->len_max;
            lenbits = bits_for(maxlen - minlen);
            fused_validation = true;
        } else if (N > 0) {
            {
                KScope ks("validate", 8ull * N, st);
                k_validate<<<div_up(N, kValTile), kValThreads, 0, st>>>(S, E, N, foff_dev, reflen_d,
                                                                        ns, stats);
                GDS_KERNEL_CHECK();
            }
            uint32_t hstats[3];
            d2h_sync(c, hstats, stats, 3);
            if (hstats[2] != 0) {
                char buf[128];
                snprintf(buf, sizeof buf, "%u reads with start > end or end >= ref_len", hstats[2]);
                return fail(c, GDS_ERR_RANGE, buf);
            }
            minlen = hstats[0];
            maxlen = hstats[1];
            lenbits = bits_for(maxlen - minlen);
        }
        // K4 (generalised): virtual node space — references longer than seg are cut into segments
        // default rule, one read length R: a whole number of reads per segment.  Every node then
        // reaches the segment's end in the same number of read hops as its neighbours within one
        // "lane block", the cut node's bundles are all admissible at once, and a segment of config 4
        // needs 175 rounds instead of 255 (tools/k3_tail.py).  The oracle rounds the same way.
        if (!(prm && prm->seg_len) && minlen == maxlen && maxlen > 1)
            seg_len = (seg_len + maxlen - 1) / maxlen * maxlen;
        out->seg_len = seg_len;
        const uint32_t seg = seg_len >= maxlen ? seg_len : 0xffffffffu;  // a read crosses <= 1 cut
        std::vector<VSample> hvs(ns);
        std::vector<uint32_t> hcuts;
        bool split = false;
        {
            uint64_t vb = 0;
            for (uint32_t k = 0; k < ns; ++k) {
                VSample& v = hvs[k];
                v.obase = base[k];
                v.vbase = (uint32_t)vb;
                v.L = rd->ref_len[k];
                // only references longer than two segments are cut (a 30 kb sample stays whole)
                v.nseg = (uint64_t)v.L > 2ull * seg ? (uint32_t)(((uint64_t)v.L + seg - 1) / seg) : 1;
                v.P = v.nseg > 1 ? maxlen - 1 : 0;
                v.W = v.nseg > 1 ? v.P + seg + 1 : 0;
                uint64_t vn = v.nseg == 1 ? (uint64_t)v.L + 1
                                          : (uint64_t)(v.nseg - 1) * v.W + v.P +
                                                (v.L - (uint64_t)(v.nseg - 1) * seg) + 1;
                vb += vn;
                if (vb >= kLabelInf)
                    return fail(c, GDS_ERR_RANGE, "segmented reference beyond 2^30 nodes");
                if (v.nseg > 1) {
                    split = true;
                    for (uint32_t j = 1; j < v.nseg; ++j) hcuts.push_back(v.obase + j * seg);
                }
            }
            n_nodes = (uint32_t)vb;
        }
        VSample* vs_d = c->vs_d.get<VSample>(ns);
        GDS_CUDA(cudaMemcpyAsync(vs_d, hvs.data(), ns * sizeof(VSample), cudaMemcpyHostToDevice, st));
        VLayout vl{vs_d, foff_dev, ns, seg};
        const int nodebits = bits_for(n_nodes ? n_nodes - 1 : 0);
        out->key_bits = nodebits + lenbits;
        int32_t* odiff = nullptr;
        uint32_t* oexcl = nullptr;
        if (split) {
            odiff = c->odiff.get<int32_t>(n_onodes + 1);
            oexcl = c->oexcl.get<uint32_t>(n_onodes + 1);
            GDS_CUDA(cudaMemsetAsync(odiff, 0, ((size_t)n_onodes + 1) * 4, st));
        }
        // how K2 finds the bundles: shared-memory histogram, global-memory histogram, radix sort
        // 0 = choose, 1 = always the radix sort, 2 = the direct histogram whenever eligible
        const int bmode = prm ? (int)prm->bundle_mode : 0;
        const bool use_direct =
            N > 0 && !split && bmode != 1 && direct_eligible(rd, ns, minlen, maxlen, S, E);
        const bool use_gdirect = N > 0 && !use_direct && bmode != 1 &&
                                 (uint64_t)n_nodes * ((uint64_t)maxlen - minlen + 1) <= kGDirectMaxKeys;
        size_t n_items = N;
        uint32_t* cross_idx = nullptr;
        if (split && N > 0 && !use_gdirect) {  // right parts of the reads that cross a cut
            uint32_t n_ct = (uint32_t)((N + kCrossTile - 1) / kCrossTile);
            uint32_t* ctc = c->cross_tc.get<uint32_t>(n_ct + 1);
            GDS_CUDA(cudaMemsetAsync(ctc + n_ct, 0, 4, st));
            {
                KScope ks("cross_count", 8ull * N, st);
                k_cross_count<<<n_ct, kCrossThreads, 0, st>>>(S, E, N, vl, ctc);
                GDS_KERNEL_CHECK();
            }
            exclusive_scan_u32(ctc, ctc, n_ct + 1, c->scan, st);
            uint32_t X = 0;
            d2h_sync(c, &X, ctc + n_ct, 1);
            cross_idx = c->cross_idx.get<uint32_t>(X + 1);
            if (X) {
                KScope ks("cross_write", 8ull * N + 4ull * X, st);
                k_cross_write<<<n_ct, kCrossThreads, 0, st>>>(S, E, N, vl, ctc, cross_idx);
                GDS_KERNEL_CHECK();
            }
            n_items = N + X;
            if (n_items >= (1ull << 32) - 64)
                return fail(c, GDS_ERR_RANGE, "more than 2^32 arc items after segmentation");
        }
        out->n_arc_items = n_items;
        DirectPlan direct;
        // Lazy mode: one read length (the in-CSR is the identity, no second sort to size) on a
        // histogram path, caller-provided length hints (no validation readback): nothing is read
        // back until the end of the call, so the ~25 launches queue up behind each other instead
        // of waiting for the host five times.  GDS_SYNC=1 keeps the readbacks (measurements).
        {
            const char* e = getenv("GDS_SYNC");
            direct.lazy = (use_direct || use_gdirect) && fused_validation && minlen == maxlen &&
                          !use_filter && !(e && e[0] == '1');
        }
        if (use_direct) {
            build_bundles_direct(c, rd, S, E, foff_dev, foff_host, reflen_d, base_d, ns, N, n_nodes,
                                 minlen, maxlen, stats, direct, B);
            out->key_bits = bits_for(direct.kmax - 1);
            out->bundle_path = 1;
        } else if (use_gdirect) {
            uint64_t n_cross = 0;
            build_bundles_gdirect(c, S, E, vl, N, n_nodes, minlen, maxlen, odiff, stats, direct, B,
                                  n_cross);
            out->n_arc_items = N + n_cross;
            out->key_bits = bits_for((uint64_t)direct.ktot - 1);
            out->bundle_path = 2;
        } else if (N > 0) {
            // the arc sort is segmented by sample unless some sample is cut into segments (then the
            // right parts live after all reads and one group with global keys is sorted)
            const bool local_keys = !split;
            // the hinted path validates inside the first histogram pass; a segmented reference
            // (global keys, rare) keeps the stand-alone validation kernel
            if (fused_validation && !local_keys) {
                KScope ks("validate", 8ull * N, st);
                k_validate<<<div_up(N, kValTile), kValThreads, 0, st>>>(S, E, N, foff_dev, reflen_d,
                                                                        ns, stats);
                GDS_KERNEL_CHECK();
                uint32_t hstats[3];
                d2h_sync(c, hstats, stats, 3);
                if (hstats[2] != 0) throw InputFail{GDS_ERR_RANGE, hstats[2],
                                                    "reads with start > end or end >= ref_len"};
                if (hstats[0] < minlen || hstats[1] > maxlen)
                    throw InputFail{GDS_ERR_ARG, 1, "reads outside the len_min/len_max hints"};
            }
            const uint32_t* fused_ref = (fused_validation && local_keys) ? reflen_d : nullptr;
            TileMap tm{nullptr, nullptr, 1, tiles_for(n_items), n_items};
            int keybits = nodebits + lenbits;
            if (local_keys && ns > 1) {
                std::vector<uint32_t> toff(ns + 1, 0);
                uint32_t maxvn = 1;
                for (uint32_t k = 0; k < ns; ++k) {
                    const uint64_t nk = foff_host[k + 1] - foff_host[k];
                    toff[k + 1] = toff[k] + tiles_for(nk);
                    maxvn = std::max(maxvn, rd->ref_len[k] + 1);
                }
                uint32_t* toff_d = c->tile_off_d.get<uint32_t>(ns + 1);
                GDS_CUDA(cudaMemcpyAsync(toff_d, toff.data(), toff.size() * 4, cudaMemcpyHostToDevice, st));
                tm = TileMap{toff_d, foff_dev, ns, toff[ns], n_items};
                keybits = bits_for(maxvn - 1) + lenbits;
            }
            out->key_bits = keybits;
            if (keybits <= 32)
                build_bundles<uint32_t>(c, S, E, vl, cross_idx, N, tm, local_keys, n_nodes,
                                        keybits, lenbits, minlen, odiff, fused_ref, stats, minlen,
                                        maxlen, B, sorted_idx, sort_passes);
            else
                build_bundles<unsigned long long>(c, S, E, vl, cross_idx, N, tm, local_keys,
                                                  n_nodes, keybits, lenbits, minlen, odiff,
                                                  fused_ref, stats, minlen, maxlen, B, sorted_idx,
                                                  sort_passes);
        } else {
            int32_t* diff = c->diff.get<int32_t>(n_nodes + 1);
            uint32_t* outdeg = c->outdeg.get<uint32_t>(n_nodes + 1);
            uint32_t* indeg = c->indeg.get<uint32_t>(n_nodes + 1);
            GDS_CUDA(cudaMemsetAsync(diff, 0, (n_nodes + 1) * 4, st));
            GDS_CUDA(cudaMemsetAsync(outdeg, 0, (n_nodes + 1) * 4, st));
            GDS_CUDA(cudaMemsetAsync(indeg, 0, (n_nodes + 1) * 4, st));
            c->b_first.get<uint32_t>(1);
            c->b_t.get<uint32_t>(1);
            c->bund.get<BundleRec>(1);
        }
        out->n_bundles = B;
        out->sort_passes = sort_passes;
        int32_t* diff = c->diff.as<int32_t>();
        uint32_t* out_ptr = c->outdeg.as<uint32_t>();
        uint32_t* in_ptr = c->indeg.as<uint32_t>();
        uint32_t* excl = c->excl.get<uint32_t>(n_nodes + 1);
        {  // coverage from the difference array and both CSR row starts: one launch
            ScanArrays sa{{reinterpret_cast<const uint32_t*>(diff), out_ptr, in_ptr}, {excl, out_ptr, in_ptr}};
            exclusive_scan_u32_multi(sa, 3, n_nodes + 1, c->scan, st);
        }
        NodeRec* node = c->node_rec.get<NodeRec>((size_t)n_nodes + 1);
        uint32_t* d_snap = c->n_dsnap.get<uint32_t>(n_nodes);
        int32_t* dem_v = c->dem_v.get<int32_t>((size_t)n_nodes + 1);
        uint32_t* cstart = c->comp_start.get<uint32_t>(n_nodes + 1);
        uint32_t* cend = c->comp_end.get<uint32_t>(n_nodes + 1);
        GDS_CUDA(cudaMemsetAsync(cstart + n_nodes, 0, 4, st));
        GDS_CUDA(cudaMemsetAsync(cend + n_nodes, 0, 4, st));
        // cov_capped / demand are reported on the ORIGINAL node space
        uint32_t* cov_dev = nullptr;
        int32_t* dem_dev = nullptr;
        if (out->cov_capped) cov_dev = out_dev ? out->cov_capped : c->cov_tmp.get<uint32_t>(n_onodes);
        if (out->demand) dem_dev = out_dev ? out->demand : c->dem_tmp.get<int32_t>(n_onodes);
        // Forced reads out, cuts in (graph.cuh, DESIGN.md §4): bundles that cover a position with
        // cov <= M get capacity 0 for the solve and their fixed flow goes into the demand; components
        // are cut at every such position.  Not for the minimum-cardinality sweep (it walks all
        // bundles itself) and not with gds_params.schedule = 1 (round 1's graph and schedule).
        // ... and not below the supply at which the express schedule starts (kExpressMinSupply):
        // with M = 100 (configs 1, 2, 5) the classic schedule on the uncut graph needs no more
        // rounds than hops, and the three extra passes over nodes and bundles would cost config 5
        // 0.25 ms of 5.75 (measured); gds_params.schedule = 2 applies them regardless.
        const bool forced_cuts = !(flags & GDS_NO_SOLVE) && algorithm == 0 && schedule != 1 &&
                           (schedule >= 2 || max_coverage >= kExpressMinSupply);
        int32_t* adj = nullptr;
        uint32_t* fmult = nullptr;
        uint8_t* dead = nullptr;  // nodes without a live bundle of their own (express rule U4)
        static_assert(kStatRes % 2 == 0 && kStatRes + 2 <= kStatWords, "stats layout");
        unsigned long long* res_supply = reinterpret_cast<unsigned long long*>(stats + kStatRes);
        if (forced_cuts && B) {
            uint32_t* unc = c->unc.get<uint32_t>((size_t)n_nodes + 1);
            adj = c->adj.get<int32_t>((size_t)n_nodes + 1);
            fmult = c->fmult.get<uint32_t>((size_t)B + 1);
            dead = c->dead.get<uint8_t>((size_t)n_nodes + 1);
            GDS_CUDA(cudaMemsetAsync(adj, 0, ((size_t)n_nodes + 1) * 4, st));
            GDS_CUDA(cudaMemsetAsync(dead, 0, (size_t)n_nodes + 1, st));
            {
                KScope ks("uncapped_flags", 12ull * n_nodes, st);
                k_uncapped_flags<<<div_up((long long)n_nodes + 1, 256), 256, 0, st>>>(excl, diff, n_nodes,
                                                                                     max_coverage, unc);
                GDS_KERNEL_CHECK();
            }
            exclusive_scan_u32(unc, unc, (size_t)n_nodes + 1, c->scan, st);
            {
                KScope ks("forced_bundles", 8ull * n_nodes, st);
                k_forced_bundles<<<div_up((long long)n_nodes, 256), 256, 0, st>>>(
                    c->bund.as<BundleRec>(), out_ptr, n_nodes, maxlen, unc, adj, fmult, dead);
                GDS_KERNEL_CHECK();
            }
        }
        {
            KScope ks("node_finalize", 60ull * n_nodes, st);
            k_node_finalize<<<div_up((long long)n_nodes + 1, 256), 256, 0, st>>>(
                excl, diff, out_ptr, in_ptr, n_nodes, max_coverage, node, d_snap, cstart, cend,
                split ? nullptr : cov_dev, split ? nullptr : dem_dev, dem_v, totals, adj,
                forced_cuts ? max_coverage : 0u, res_supply, dead);
            GDS_KERNEL_CHECK();
        }
        if (split) {
            exclusive_scan_u32(reinterpret_cast<const uint32_t*>(odiff), oexcl, (size_t)n_onodes + 1,
                               c->scan, st);
            {
                KScope ks("orig_outputs", 16ull * n_onodes, st);
                k_orig_outputs<<<div_up(n_onodes, 256), 256, 0, st>>>(oexcl, odiff, n_onodes,
                                                                      max_coverage, cov_dev, dem_dev,
                                                                      totals);
                GDS_KERNEL_CHECK();
            }
            uint32_t* cuts_d = c->cut_nodes.get<uint32_t>(hcuts.size());
            GDS_CUDA(cudaMemcpyAsync(cuts_d, hcuts.data(), hcuts.size() * 4, cudaMemcpyHostToDevice,
                                     st));
            {
                KScope ks("cut_through", 12ull * hcuts.size(), st);
                k_cut_through<<<div_up(hcuts.size(), 128), 128, 0, st>>>(
                    cuts_d, (uint32_t)hcuts.size(), oexcl, odiff, max_coverage, totals);
                GDS_KERNEL_CHECK();
            }
        }
        uint32_t* sidx = c->comp_sidx.get<uint32_t>(n_nodes + 1);
        exclusive_scan_u32(cstart, sidx, n_nodes + 1, c->scan, st);
        const bool lazy = direct.lazy;
        const uint32_t* n_comp_dev = nullptr;
        if (lazy) {
            // the count stays on the device; on the host an ESTIMATE (one component per sample or
            // segment — zero-coverage gaps add more, empty samples take some away) picks the K3
            // kernel and the grid, and the arrays are sized by the bound (a component has >= 2 nodes)
            GDS_CUDA(cudaMemcpyAsync(stats + kStatNComp, sidx + n_nodes, 4, cudaMemcpyDeviceToDevice, st));
            n_comp_dev = stats + kStatNComp;
            uint64_t est = 0;
            for (const VSample& v : hvs) est += v.nseg;
            n_comp = (uint32_t)std::min<uint64_t>(est, n_nodes / 2 + 1);
        } else {
            d2h_sync(c, &n_comp, sidx + n_nodes, 1);  // also fences hvs/hcuts uploads
        }
        out->n_components = n_comp;
        const uint32_t n_comp_cap = lazy ? n_nodes / 2 + 1 : n_comp;
        uint32_t* comp_lo = c->comp_lo.get<uint32_t>(n_comp_cap + 1);
        uint32_t* comp_hi = c->comp_hi.get<uint32_t>(n_comp_cap + 1);
        if (n_comp) {
            {
                KScope ks("comp_write", 16ull * n_nodes, st);
                k_comp_write<<<div_up(n_nodes, 256), 256, 0, st>>>(cstart, cend, sidx, n_nodes,
                comp_lo, comp_hi);
                GDS_KERNEL_CHECK();
            }
        }
        // in-CSR: bundle ids ordered by (end node, bundle id) = stable sort of ids by b_t
        uint32_t* in_bid = direct.in_bid;  // single read length: bundle order is end order too
        if (B && !in_bid) {
            uint32_t* tkA = c->tkA.get<uint32_t>(B);
            uint32_t* tkB = c->tkB.get<uint32_t>(B);
            uint32_t* tvA = c->tvA.get<uint32_t>(B);
            uint32_t* tvB = c->tvB.get<uint32_t>(B);
            GDS_CUDA(cudaMemcpyAsync(tkA, c->b_t.as<uint32_t>(), (size_t)B * 4,
                                     cudaMemcpyDeviceToDevice, st));
            TileMap btm{nullptr, nullptr, 1, tiles_for(B), B};
            int w = radix_sort_pairs<uint32_t>(tkA, tvA, tkB, tvB, btm, nodebits, c->radix, st,
                                               c->atomic_rank);
            in_bid = w ? tvB : tvA;
        }
        if (!out_dev) {
            deliver(c, out->cov_capped, cov_dev, n_onodes, false);
            deliver(c, out->demand, dem_dev, n_onodes, false);
        }
        GDS_CUDA(cudaEventRecord(c->ev[EV_GRAPH], st));

        // ---------------- K3: max flow ----------------
        // no component is larger than a whole unsegmented sample or one segment
        uint32_t max_comp_nodes = 0;
        for (const VSample& v : hvs)
            max_comp_nodes = std::max(max_comp_nodes, v.nseg == 1 ? v.L + 1 : seg + 1);
        const bool do_solve = !(flags & GDS_NO_SOLVE);
        if (do_solve && algorithm == 1 && maxlen >= 4096)
            return fail(c, GDS_ERR_ARG, "algorithm 1 (minimum cardinality) takes reads of up to 4095 positions");
        // the express schedule (maxflow_sm.cuh): components with a supply of kExpressMinSupply or
        // more — none when M is below that, and then nothing about the launch changes
        uint32_t express_on = schedule == 1 ? 0u : schedule == 2 ? 2u : 1u;  // (3: the usual supply rule)
        if (!forced_cuts || (express_on == 1 && max_coverage < kExpressMinSupply)) express_on = 0;
        const bool express_possible = express_on != 0;
        const Mf2Plan mf2 = do_solve && algorithm == 0
                                ? plan_maxflow_sm(n_comp, max_comp_nodes, express_possible)
                                : Mf2Plan{};
        uint32_t* in_src = c->in_src.get<uint32_t>((size_t)B + 1);
        uint32_t* in1 = c->in1.get<uint32_t>((size_t)n_nodes + 1);
        GDS_CUDA(cudaMemsetAsync(in1, 0xff, ((size_t)n_nodes + 1) * 4, st));
        if (B) {
            KScope ks("in_src", 24ull * B, st);
            k_in_src<<<div_up(B, 256), 256, 0, st>>>(c->bund.as<BundleRec>(), in_bid, in_ptr, B, in_src,
                                                     mf2.on ? node : nullptr, direct.B_dev, in1);
            GDS_KERNEL_CHECK();
        }
        MfGraph mg{node, d_snap, c->bund.as<BundleRec>(), in_bid, in_src, dem_v, in1};
        // per-component records only for the diagnostics dump; gds_result's counters are summed on
        // the device (MfTotals)
        const char* dump_comp = getenv("GDS_DUMP_COMP");
        CompStats* cstats = dump_comp ? c->comp_stats.get<CompStats>(n_comp_cap + 1) : nullptr;
        if (do_solve && n_comp && algorithm == 1) {
            // K3': greedy interval multicover, one warp per component, then bundle flows
            uint32_t* wc = c->work_counter.get<uint32_t>(4);
            GDS_CUDA(cudaMemsetAsync(wc, 0, 16, st));
            uint32_t* taken = c->taken.get<uint32_t>((size_t)n_nodes + 2);
            GDS_CUDA(cudaMemsetAsync(taken, 0, ((size_t)n_nodes + 2) * 4, st));
            SweepGraph sg{excl, diff, out_ptr, c->bund.as<BundleRec>(), taken};
            launch_sweep(c, sg, comp_lo, comp_hi, n_comp, n_comp_dev, max_coverage, wc, totals + 5, maxlen,
                         minlen == maxlen, 12ull * n_nodes + 8ull * B);
            if (B) {
                KScope ks("sweep_distribute", 12ull * n_nodes + 24ull * B, st);
                k_sweep_distribute<<<div_up((long long)n_nodes, 256), 256, 0, st>>>(
                    taken, in_ptr, in_bid, c->bund.as<BundleRec>(), n_nodes, totals + 5);
                GDS_KERNEL_CHECK();
            }
        } else if (do_solve && n_comp) {
            uint32_t* qF = c->qF.get<uint32_t>(n_nodes);
            uint32_t* qT = c->qT.get<uint32_t>(n_nodes);
            uint32_t* qN = c->qN.get<uint32_t>(n_nodes);
            uint32_t* qH = c->qH.get<uint32_t>(n_nodes);
            uint32_t* wc = c->work_counter.get<uint32_t>(4);  // [0] sm kernel, [1] fallback, [2] list size
            GDS_CUDA(cudaMemsetAsync(wc, 0, 16, st));
            const unsigned long long mf_bytes = 36ull * n_nodes + 20ull * B;
            // compact labels for k_maxflow's relabels
            uint16_t* lab_g = c->lab_g.get<uint16_t>(2 * (size_t)n_nodes + 4);
            if (mf2.on) {
                uint32_t* fb_list = c->fb_list.get<uint32_t>(n_comp_cap + 1);
                Mf2Graph g2{node, c->bund.as<BundleRec>(), in_bid, in_src, out_ptr, in_ptr, dem_v,
                            vs_d, ns, express_on, mf2.classic_ok ? 1u : 0u, dead};
                launch_maxflow_sm(c, mf2, g2, comp_lo, comp_hi, n_comp, wc, qF, qT, qN, qH, sp, cstats,
                                  mf_bytes, fb_list, wc + 2, n_comp_dev, mft);
                // whatever the shared-memory kernel could not take (grid: at most one wave)
                // (with the count on the device the list may be longer than the estimate says)
                launch_maxflow(c, mg, comp_lo, comp_hi,
                               mf2.classic_ok && !n_comp_dev ? std::min<uint32_t>(n_comp, kNumSMs)
                                                             : std::max<uint32_t>(n_comp, kNumSMs),
                               wc + 1, qF,
                               qT, qN, qH, sp, cstats, 0, max_comp_nodes, n_comp_dev, mft, lab_g,
                               fb_list, wc + 2);
            } else {
                launch_maxflow(c, mg, comp_lo, comp_hi,
                               n_comp_dev ? std::max<uint32_t>(n_comp, kNumSMs) : n_comp, wc, qF, qT, qN, qH,
                               sp, cstats, mf_bytes, max_comp_nodes, n_comp_dev, mft, lab_g);
            }
        }
        if (fmult) {  // the forced bundles come back with their fixed flow: K5 keeps all their reads
            KScope ks("forced_restore", 8ull * n_nodes, st);
            k_forced_restore<<<div_up((long long)n_nodes, 256), 256, 0, st>>>(
                c->bund.as<BundleRec>(), out_ptr, n_nodes, maxlen, c->unc.as<uint32_t>(), fmult);
            GDS_KERNEL_CHECK();
        }
        GDS_CUDA(cudaEventRecord(c->ev[EV_MAXFLOW], st));

        // ---------------- K5 / K6 / results ----------------
        // One pass in the normal case.  In lazy mode the selection may have to be repeated once: the
        // final readback is the first time the host sees that the candidates of the partial bundles
        // did not fit their buffer (it grows) or that a partial bundle needs the ordered walk.
        const size_t n_words = (N + 31) / 32;
        uint32_t* bm = (out_dev && out->kept_bitmap) ? out->kept_bitmap
                                                     : c->bitmap.get<uint32_t>(n_words + 1);
        uint32_t hstat[kStatWords] = {};
        unsigned long long* htot = reinterpret_cast<unsigned long long*>(hstat + 8);
        bool force_walk = false;
        size_t cand_need = 0;
        for (int attempt = 0;; ++attempt) {
            if (do_solve) {
                GDS_CUDA(cudaMemsetAsync(bm, 0, n_words * 4, st));
                if (attempt) GDS_CUDA(cudaMemsetAsync(totals + 1, 0, 16, st));  // n_kept, violations
                if (B && direct.on)
                    direct_select(c, direct, S, E, ns, N, B, bm, totals, stats, out, force_walk, cand_need);
                else if (B) {
                    KScope ks("select", 8ull * B + 8ull * N / 32, st);
                    k_select<<<div_up(B, 256), 256, 0, st>>>(c->b_first.as<uint32_t>(),
                                                             c->bund.as<BundleRec>(), sorted_idx, B, bm,
                                                             totals);
                    GDS_KERNEL_CHECK();
                }
            }
            if (!attempt) GDS_CUDA(cudaEventRecord(c->ev[EV_SELECT], st));

            // K6: verification (before find_pairs widens the set), on the original node space:
            // compares with the input coverage (odiff when segmented)
            if (do_solve && (flags & GDS_VERIFY)) {
                int32_t* vdiff = c->vdiff.get<int32_t>((size_t)n_onodes + 1);
                uint32_t* vexcl = c->vexcl.get<uint32_t>((size_t)n_onodes + 1);
                GDS_CUDA(cudaMemsetAsync(vdiff, 0, ((size_t)n_onodes + 1) * 4, st));
                if (n_words) {
                    KScope ks("verify_accumulate", 4ull * n_words, st);
                    k_verify_accumulate<<<div_up(n_words, 256), 256, 0, st>>>(bm, S, E, N, foff_dev,
                                                                              base_d, ns, vdiff);
                    GDS_KERNEL_CHECK();
                }
                exclusive_scan_u32(reinterpret_cast<const uint32_t*>(vdiff), vexcl,
                                   (size_t)n_onodes + 1, c->scan, st);
                {
                    KScope ks("verify_compare", 16ull * n_onodes, st);
                    k_verify_compare<<<div_up(n_onodes, 256), 256, 0, st>>>(
                        vexcl, vdiff, split ? oexcl : excl, split ? odiff : diff, n_onodes,
                        max_coverage, totals);
                    GDS_KERNEL_CHECK();
                }
            }
            if (do_solve && (flags & GDS_FIND_PAIRS) && n_words) {
                KScope ks("find_pairs", 8ull * n_words, st);
                k_find_pairs<<<div_up(n_words, 256), 256, 0, st>>>(bm, n_words);
                GDS_KERNEL_CHECK();
            }
            if (!attempt) GDS_CUDA(cudaEventRecord(c->ev[EV_VERIFY], st));

            if (do_solve && !out_dev) deliver(c, out->kept_bitmap, bm, n_words, false);
            d2h_sync(c, hstat, stats, (size_t)kStatWords);  // THE readback of a lazy call
            if (!lazy) break;
            if (hstat[2]) throw InputFail{GDS_ERR_RANGE, hstat[2], "reads with start > end or end >= ref_len"};
            if (hstat[3]) throw InputFail{GDS_ERR_ARG, hstat[3], "reads outside the len_min/len_max hints"};
            const uint32_t cflags = do_solve && B && direct.on ? hstat[kStatCtl + 2] : 0;
            if (attempt || !(cflags & 3u)) break;
            force_walk = (cflags & 1u) != 0;                  // ordered walk (shared-memory path)
            cand_need = (size_t)hstat[kStatCtl + 1] + 1;      // or the buffer the candidates need
        }
        if (lazy) {
            out->n_bundles = hstat[kStatB];
            n_comp = hstat[kStatNComp];
            out->n_components = n_comp;
            out->partial_bundles = hstat[kStatCtl];
            out->partial_candidates = hstat[kStatCtl + 1];
            if (direct.global) out->n_arc_items = N + hstat[4];
        }
        // htot[0] = source capacity of the (virtual) network the kernel solved; when references
        // were segmented the closed-form F* of the ORIGINAL network is htot[3] and htot[4] units
        // pass straight through the cut nodes once the segment flows are stitched together
        const long long fstar_virtual = (long long)htot[0];
        out->fstar = (int64_t)(split ? htot[3] : htot[0]);
        out->n_kept = htot[1];
        out->verify_violations = htot[2];
        long long stuck = 0;
        if (do_solve) {
            MfTotals ht;
            memcpy(&ht, hstat + kStatMf, sizeof ht);
            // sink inflow of the residual problem + the forced bundles' fixed flows: whatever the
            // residual problem left undelivered (nothing, on valid input) is missing from F*
            unsigned long long hres = 0;
            memcpy(&hres, hstat + kStatRes, sizeof hres);
            out->flow_value = forced_cuts ? fstar_virtual - ((long long)hres - ht.sink_flow) : ht.sink_flow;
            out->rounds_total = ht.rounds_total;
            out->rounds_max = ht.rounds_max;
            out->pushes = ht.pushes;
            out->relabels = ht.relabels;
            out->global_relabels = ht.grs;
            out->bfs_levels = ht.bfs_levels;
            out->max_frontier = ht.max_frontier;
            stuck = ht.stuck;
            if (algorithm == 1) {
                // the sweep's cover IS a maximum flow (flow 1 on the kept reads, back arcs take the
                // surplus); htot[5] counts deficits it could not fill and reads it could not place
                out->flow_value = htot[5] ? -1 : fstar_virtual;
                stuck = (long long)htot[5];
            } else if (ht.n_solved != n_comp) {
                stuck += 1;  // a component was never taken: cannot happen
            }
        }
        if (do_solve && n_comp && dump_comp) {  // diagnostics only
            std::vector<CompStats> hs(n_comp);
            d2h_sync(c, hs.data(), cstats, n_comp);
            if (FILE* fp = fopen(dump_comp, "w")) {
                fprintf(fp, "comp rounds pushes relabels grs bfs_levels max_frontier frontier_sum cycles gr_init gr_bfs gr_snap front gr_later\n");
                for (uint32_t i = 0; i < n_comp; ++i)
                    fprintf(fp, "%u %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu\n", i,
                            hs[i].rounds, hs[i].pushes, hs[i].relabels, hs[i].grs, hs[i].bfs_levels,
                            hs[i].max_frontier, hs[i].frontier_sum, hs[i].cycles, hs[i].cyc_gr_init,
                            hs[i].cyc_gr_bfs, hs[i].cyc_gr_snap, hs[i].cyc_front, hs[i].cyc_gr_later);
                fclose(fp);
            }
        }
        GDS_CUDA(cudaEventRecord(c->ev[EV_END], st));
        GDS_CUDA(cudaStreamSynchronize(st));
        auto ms = [&](int a, int b) {
            float t = 0;
            cudaEventElapsedTime(&t, c->ev[a], c->ev[b]);
            return t;
        };
        out->ms_h2d = ms(EV_BEGIN, EV_H2D);
        out->ms_filter = ms(EV_H2D, EV_FILTER);
        out->ms_graph = ms(EV_FILTER, EV_GRAPH);
        out->ms_maxflow = ms(EV_GRAPH, EV_MAXFLOW);
        out->ms_select = ms(EV_MAXFLOW, EV_SELECT);
        out->ms_verify = ms(EV_SELECT, EV_VERIFY);
        out->ms_d2h = ms(EV_VERIFY, EV_END);
        out->ms_total = ms(EV_BEGIN, EV_END);
        out->kernel_launches = launch_counter() - launches0;
        const bool converged = out->flow_value == fstar_virtual && stuck == 0;
        if (split) out->flow_value -= (int64_t)htot[4];
        if (do_solve && !converged) {
            char buf[160];
            snprintf(buf, sizeof buf, "max-flow did not converge: sink inflow %lld, F* %lld, stuck %lld",
                     (long long)out->flow_value, (long long)out->fstar, stuck);
            return fail(c, GDS_ERR_NOCONVERGE, buf);
        }
        return GDS_OK;
    } catch (const InputFail& f) {
        char buf[160];
        snprintf(buf, sizeof buf, "%u %s", f.count, f.what);
        return fail(c, f.code, buf);
    } catch (const CudaFail& f) {
        return fail_cuda(c, f);
    } catch (const std::bad_alloc&) {
        return fail(c, GDS_ERR_NOMEM, "host allocation failed");
    }
}
