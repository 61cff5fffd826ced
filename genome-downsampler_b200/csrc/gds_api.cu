// gds_api.cu — C ABI (include/gds.h) and host-side orchestration of the device pipeline.
// No CPU fallback exists: without a usable CUDA device every entry point fails.
#include "../../include/gds.h"

#include <algorithm>
#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
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
    DevBuf small;  // one StatsBlock
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
    bool atomic_rank = false;  // shared-memory atomics rank in lane order on this device (probed)
    Profiler prof;

};

namespace {

struct InputFail {  // bad input discovered on the device in the middle of the pipeline
    int code;
    uint32_t count;
    const char* what;
};
constexpr const char* kBadRange = "reads with start > end or end >= ref_len";
constexpr const char* kBadHints = "reads outside the len_min/len_max hints";

struct CallFail {  // a call the pipeline finds it cannot take, after the argument checks
    int code;
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

// Diagnostic knobs for tests and measurements.  Read once per call: tests change them between calls.
struct Knobs {
    bool mf_global;         // GDS_MF=global: the round-1 kernel only
    bool mf_optr;           // GDS_MF_OPTR=0: k_maxflow_sm without the out-CSR cache
    const char* dump_comp;  // GDS_DUMP_COMP=<file>: per-component K3 records
    static Knobs read() {
        const char* mf = getenv("GDS_MF");
        const char* optr = getenv("GDS_MF_OPTR");
        return Knobs{mf && !strcmp(mf, "global"), !optr || optr[0] != '0', getenv("GDS_DUMP_COMP")};
    }
};

// The small device block gds_ctx::small.  Kernels get it as uint32_t* (the validation words) and
// unsigned long long* (the totals); the host reads it by name.
struct StatsBlock {
    uint32_t len_min, len_max;       // read-length bounds found by the validation
    uint32_t bad_range, bad_hints;   // reads with start > end or end >= ref_len / outside the hints
    uint32_t n_cross;                // reads crossing a cut (global-memory histogram path)
    uint32_t pad0[3];
    // F* of the virtual network, reads kept, verification violations, F* of the original network,
    // units through the cut nodes, what the minimum-cardinality sweep could not fill or place
    unsigned long long fstar_virtual, n_kept, violations, fstar_orig, through_flow, sweep_fail;
    uint32_t n_bundles, n_comp;      // the counts stay on the device until the final readback
    uint32_t pad1[2];
    uint32_t ctl[4];                 // K5 control words of the histogram path (direct_select)
    uint32_t pad2[4];
    MfTotals mf;                     // K3 sums over the components
    unsigned long long res_supply;   // supply of the residual problem (forced cuts)
    uint32_t pad3[10];
};
static_assert(offsetof(StatsBlock, len_min) == 0 && offsetof(StatsBlock, len_max) == 4 &&
              offsetof(StatsBlock, bad_range) == 8 && offsetof(StatsBlock, bad_hints) == 12 &&
              offsetof(StatsBlock, n_cross) == 16 && offsetof(StatsBlock, fstar_virtual) == 32 &&
              offsetof(StatsBlock, n_kept) == 40 && offsetof(StatsBlock, violations) == 48 &&
              offsetof(StatsBlock, fstar_orig) == 56 && offsetof(StatsBlock, through_flow) == 64 &&
              offsetof(StatsBlock, sweep_fail) == 72 && offsetof(StatsBlock, n_bundles) == 80 &&
              offsetof(StatsBlock, n_comp) == 84 && offsetof(StatsBlock, ctl) == 96 &&
              offsetof(StatsBlock, mf) == 128 && offsetof(StatsBlock, res_supply) == 208 &&
              sizeof(StatsBlock) == 256, "stats layout (the kernels index it as words)");

void input_verdict(const StatsBlock& h) {
    if (h.bad_range) throw InputFail{GDS_ERR_RANGE, h.bad_range, kBadRange};
    if (h.bad_hints) throw InputFail{GDS_ERR_ARG, h.bad_hints, kBadHints};
}

// reads back the validation words (a synchronisation) and throws on bad input
StatsBlock read_input_verdict(gds_ctx* c, const StatsBlock* ds) {
    StatsBlock h{};
    d2h_sync(c, &h.len_min, &ds->len_min, 5);
    input_verdict(h);
    return h;
}

// What both K3 kernels are given (host side; every launch shape passes it on)
struct K3Args {
    const uint32_t *comp_lo, *comp_hi;
    uint32_t n_comp;  // the host's estimate: it picks the launch shape and the grid
    uint32_t* wc;
    uint32_t *qF, *qT, *qN, *qH;
    SolveParams sp;
    CompStats* cstats;
    const uint32_t* n_comp_dev;  // the count itself
    MfTotals* mft;
};

struct MfArgs {  // k_maxflow
    MfGraph g;
    K3Args k;
    uint32_t max_comp_nodes;
    const uint32_t *comp_list, *comp_list_n;
    uint16_t* lab_g;
};

// The dynamic shared memory a kernel may take is an attribute of the kernel on the device, shared by
// every gds_ctx (and host thread) there.  It is only ever raised, under one lock: a record kept per
// context would let a context with small components lower the limit below what another context's
// next launch needs, and that launch would fail with "invalid argument".
void raise_smem_limit(const void* kern, int device, int bytes) {
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, int> limit;
    std::lock_guard<std::mutex> lock(mu);
    int& cur = limit[{kern, device}];
    if (bytes > cur) {
        GDS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        cur = bytes;
    }
}

template <int I>
void launch_maxflow_shape(gds_ctx* c, const MfArgs& a, unsigned long long alg_bytes) {
    constexpr MfShape sh = kMfShapes[I];
    auto kern = k_maxflow<sh.threads, sh.qcap, sh.ctas_per_sm>;
    // 16-bit labels of a whole component in shared memory for the first global relabel, when
    // every resident CTA of this shape can have them (maxflow.cuh: mf_first_relabel)
    uint32_t lab_cap = 0;
    int smem = (int)sizeof(MfShared<sh.qcap>);
    if (a.max_comp_nodes && a.max_comp_nodes < 0xfff0u) {
        const int lab_bytes = (int)((2 * a.max_comp_nodes + 4 + 15) & ~15u);
        // ... and the SM keeps at least ~100 KB of L1 for the rounds' plain loads (measured: with
        // 4 x 49 KB per SM config 4 lost 13 %)
        if ((smem + lab_bytes) * sh.ctas_per_sm <= 132 * 1024) {
            smem += lab_bytes;
            lab_cap = a.max_comp_nodes;
        }
    }
    raise_smem_limit(reinterpret_cast<const void*>(kern), c->device, smem);
    const K3Args& k = a.k;
    int grid = std::min<uint32_t>(k.n_comp, (uint32_t)kNumSMs * sh.ctas_per_sm);
    launch("maxflow", alg_bytes, kern, grid, sh.threads, smem, c->stream, a.g, k.comp_lo, k.comp_hi,
           k.wc, k.qF, k.qT, k.qN, k.qH, k.sp, k.cstats, lab_cap, a.comp_list, a.comp_list_n,
           k.n_comp_dev, k.mft, a.lab_g);
}

void launch_maxflow(gds_ctx* c, const MfArgs& a, unsigned long long alg_bytes) {
    using Launch = void (*)(gds_ctx*, const MfArgs&, unsigned long long);
    static constexpr Launch kShapes[4] = {launch_maxflow_shape<0>, launch_maxflow_shape<1>,
                                          launch_maxflow_shape<2>, launch_maxflow_shape<3>};
    int shape = 3;
    for (int i = 0; i < 3; ++i)
        if (a.k.n_comp <= (uint32_t)kNumSMs * kMfShapes[i].ctas_per_sm) {
            shape = i;
            break;
        }
    kShapes[shape](c, a, alg_bytes);
}

constexpr int kMf2MaxSmem = 227 * 1024;
constexpr uint32_t kMf2MinQcap = 256;  // staged entries per frontier queue, at the least
// The express schedule runs only in k_maxflow_sm, and a component the launch cannot hold goes to
// k_maxflow: every launch, even one clamped to kMf2MaxSmem with the smallest queues, must hold the
// largest express component, or its schedule would depend on the other components of the call.
static_assert(kMf2HeaderBytes + 16u * kMf2MinQcap + mf2_node_bytes(kExpressMaxNodes, false) <=
                  (uint32_t)kMf2MaxSmem,
              "an express component must fit every k_maxflow_sm launch");

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

Mf2Plan plan_maxflow_sm(uint32_t n_comp, uint32_t max_comp_nodes, bool express_possible,
                        const Knobs& knobs) {
    Mf2Plan pl;
    // (components of the express schedule exist only in k_maxflow_sm: with them in the call the
    //  kernel always runs, and GDS_MF=global is ignored)
    if (knobs.mf_global && !express_possible) return pl;
    // shared memory per CTA: header + 4 staged queues + the node arrays of the largest component
    // that should still fit.  Prefer the out-CSR cache unless leaving it out lets all components
    // be resident at once (a batch of segments) where they otherwise would not be.
    auto need = [&](uint32_t nodes, bool optr, uint32_t qcap) {
        return (long long)kMf2HeaderBytes + 16ll * qcap + mf2_node_bytes(nodes, optr);
    };
    const uint32_t nmax = std::min<uint32_t>(max_comp_nodes, kMf2MaxNodes);
    if (nmax == 0 || n_comp == 0) return pl;
    uint32_t qcap = 2048;
    bool optr = knobs.mf_optr;
    // the queues shrink before the node arrays do
    while (qcap > kMf2MinQcap && need(nmax, optr, qcap) > kMf2MaxSmem) qcap >>= 1;
    if (need(nmax, optr, qcap) > kMf2MaxSmem) optr = false;
    long long smem_ll = need(nmax, optr, qcap);
    // the largest does not fit (beyond 50 672 nodes): the launch takes all an SM has, which holds
    // every express component (static_assert above); the kernel puts the longer ones on fb_list
    if (smem_ll > kMf2MaxSmem) smem_ll = kMf2MaxSmem;
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
    pl.classic_ok = !knobs.mf_global && (unsigned long long)n_comp * 2 <= 3ull * kNumSMs * per_sm;
    if (!pl.classic_ok && !express_possible) return pl;
    pl.on = true;
    pl.smem = (int)((smem_ll + 15) & ~15ll);
    pl.per_sm = per_sm;
    pl.qcap = qcap;
    pl.optr = optr;
    return pl;
}

// K3 with the hot state in shared memory (maxflow_sm.cuh).  Components the kernel finds ineligible
// (too large for the launch, supply beyond 16 bits) land on fb_list for k_maxflow.
// Components whose nodes are mostly heavy (variable read lengths: tens of bundles per node) go to
// k_maxflow: their frontiers hold tens of nodes with ~40 bundles each, the time is the per-bundle
// global traffic of the warp passes, and 32 warps of 64 registers (k_maxflow) beat 16 warps with the
// labels in shared memory (config 2 without its filter: 2.6 ms there, 3.0 ms here after batching the
// loads of eight nodes per warp; 3.4 ms before).
template <int THREADS, int SLOT>
void launch_mf2_shape(gds_ctx* c, const Mf2Plan& pl, const Mf2Graph& g, const K3Args& k,
                      uint32_t* fb_list, uint32_t* fb_count, unsigned long long alg_bytes) {
    auto kern = k_maxflow_sm<THREADS>;
    raise_smem_limit(reinterpret_cast<const void*>(kern), c->device, pl.smem);
    // one full wave: k.n_comp is an estimate (one component per sample or segment), and the cuts at
    // cov <= M can make many more (the reference's "low sides" shape: 11 from one sample, which a
    // grid of one CTA solved one after the other).  A CTA without work exits at once.
    const int grid = kNumSMs * pl.per_sm;
    launch("maxflow", alg_bytes, kern, grid, THREADS, pl.smem, c->stream, g, k.comp_lo, k.comp_hi,
           k.wc, k.qF, k.qT, k.qN, k.qH, k.sp, k.cstats, (uint32_t)pl.smem, pl.qcap, fb_list,
           fb_count, pl.optr ? 1u : 0u, k.n_comp_dev, k.mft);
}

// K3' (sweep.cuh): the minimum-cardinality solve.  One warp per component.
struct SweepArgs {
    SweepGraph g;
    const uint32_t *comp_lo, *comp_hi;
    uint32_t n_comp;  // the host's estimate, for the grid
    const uint32_t* n_comp_dev;
    uint32_t M;
    uint32_t* wc;
    unsigned long long* fail;
};

template <int W, int CAP, bool WARP>
void launch_sweep_shape(gds_ctx* c, const SweepArgs& a, unsigned long long alg_bytes) {
    constexpr int smem = kSweepWarps * (2 * W + 4 * CAP + 2 * 34 + 2 * 32) * 4;
    const int grid = std::max(1, std::min<int>(div_up(a.n_comp, kSweepWarps), kNumSMs * 8));
    auto kern = WARP ? k_sweep_warp<W, CAP> : k_sweep<W, CAP>;
    raise_smem_limit(reinterpret_cast<const void*>(kern), c->device, smem);
    launch("sweep", alg_bytes, kern, grid, kSweepWarps * 32, smem, c->stream, a.g, a.comp_lo,
           a.comp_hi, a.n_comp_dev, a.M, a.wc, a.fail);
}

void launch_sweep(gds_ctx* c, const SweepArgs& a, uint32_t maxlen, bool one_len,
                  unsigned long long alg_bytes) {
    using Launch = void (*)(gds_ctx*, const SweepArgs&, unsigned long long);
    static constexpr Launch kShapes[6] = {
        launch_sweep_shape<256, 64, false>,  launch_sweep_shape<256, 1024, true>,
        launch_sweep_shape<1024, 64, false>, launch_sweep_shape<1024, 1024, true>,
        launch_sweep_shape<4096, 64, false>, launch_sweep_shape<4096, 1024, true>};
    // one read length: at most a few bundles per position -> one lane walks; several lengths: tens of
    // arrivals per position -> the warp-synchronous walk adds them in parallel
    const int w = maxlen < 256 ? 0 : maxlen < 1024 ? 1 : 2;
    kShapes[w * 2 + (one_len ? 0 : 1)](c, a, alg_bytes);
}

// Sort-free K2 (direct.cuh).  The shared-memory histogram is eligible when all reads have one
// length, no sample is segmented and every sample's ref_len + 1 nodes fit in one SM's shared memory.
struct DirectPlan {
    bool on = false;
    DirectLayout dl{};
    uint32_t* ghist = nullptr;
    uint32_t ktot = 0, kmax = 0, n_items = 0;
    uint32_t* in_bid = nullptr;  // identity in-CSR (one read length), else null
    bool global = false;         // counters in global memory (several lengths / segmented reference)
    GDirectLayout gl{};
};

// How the virtual node space is laid out: references longer than two segments are cut into
// segments of `seg` positions, each its own component.  A pure function of the call's arguments
// and read lengths.
struct SegPlan {
    uint32_t seg_len;  // gds_result.seg_len
    uint32_t seg;      // the cut length, 0xffffffff when no reference is cut
    std::vector<VSample> hvs;
    std::vector<uint32_t> hcuts;  // original node of every cut
    bool split;
    uint32_t n_nodes;
    uint32_t max_comp_nodes;  // no component is larger than a whole unsegmented sample or one segment
    // one component per sample or segment (zero-coverage gaps add more, empty samples take some
    // away): the host's ESTIMATE of the component count, which stays on the device
    uint32_t comp_estimate;
};

struct Degrees {
    int32_t* diff;
    uint32_t *outdeg, *indeg;
};

// One gds_solve call: its arguments, the values derived from them and the device arrays one stage
// hands to the next.
struct SolveCall {
    const gds_reads* rd;
    const gds_filter* flt;
    const gds_params* prm;
    uint32_t flags;
    uint32_t M;
    gds_result* out;
    Knobs knobs;
    // argument checks
    uint32_t ns;
    uint64_t P;
    uint32_t n_onodes;
    std::vector<uint32_t> base;  // original node space: sample k owns ref_len[k]+1 nodes
    bool out_dev, do_solve;
    SolveParams sp;
    uint32_t algorithm, schedule;
    cudaStream_t st;
    // inputs on the device
    const uint32_t *dS, *dE, *dLen;
    const uint8_t* dQ;
    uint64_t* off_d;
    uint32_t *reflen_d, *base_d;
    StatsBlock* ds;
    // the reads K2 sees (after the filter)
    const uint32_t *S, *E;
    const uint64_t* foff_dev;
    uint64_t N;
    std::vector<uint64_t> foff_host;
    uint32_t minlen, maxlen;
    int lenbits;
    bool fused_validation;
    // virtual node space
    SegPlan plan;
    VSample* vs_d;
    VLayout vl;
    int nodebits;
    int32_t* odiff;
    uint32_t* oexcl;
    // what K3 will run, decided before the graph is built (plan_solve)
    bool forced_cuts;
    uint32_t express_on;
    Mf2Plan mf2;
    // K2
    DirectPlan direct;
    bool direct_graph;  // k_direct_graph builds the nodes, components and in-arcs (no forced cuts)
    uint32_t B;  // exact when the host needs it (radix sorts over the bundles), else a bound
    uint32_t* sorted_idx;
    int sort_passes;
    // nodes and components
    uint32_t* excl;
    Degrees deg;
    NodeRec* node;
    uint32_t* d_snap;
    int32_t* dem_v;
    uint32_t* fmult;
    uint8_t* dead;
    uint32_t n_comp_cap;  // a bound; the count is ds->n_comp
    uint32_t *comp_lo, *comp_hi, *in_bid;
    CompStats* cstats;
    // K5 and the final readback
    uint32_t* bm;
    StatsBlock hstat;

    uint32_t* stats() const { return reinterpret_cast<uint32_t*>(ds); }
    unsigned long long* totals() const { return &ds->fstar_virtual; }
};

// k_validate: read-length bounds and the coordinate check in a pass of its own
StatsBlock validate_reads(gds_ctx* c, const SolveCall& sc) {
    launch("validate", 8ull * sc.N, k_validate, div_up(sc.N, kValTile), kValThreads, 0, sc.st, sc.S,
           sc.E, sc.N, sc.foff_dev, sc.reflen_d, sc.ns, sc.stats());
    return read_input_verdict(c, sc.ds);
}

// K2's per-node outputs: the difference array of the coverage and the out/in degrees
Degrees degree_buffers(gds_ctx* c, uint32_t n_nodes) {
    return Degrees{c->diff.get<int32_t>(n_nodes + 1), c->outdeg.get<uint32_t>(n_nodes + 1),
                   c->indeg.get<uint32_t>(n_nodes + 1)};
}

// ... cleared
Degrees alloc_degrees(gds_ctx* c, cudaStream_t st, uint32_t n_nodes, bool clear_diff = true) {
    const Degrees d = degree_buffers(c, n_nodes);
    if (clear_diff) GDS_CUDA(cudaMemsetAsync(d.diff, 0, (n_nodes + 1) * sizeof(int32_t), st));
    else GDS_CUDA(cudaMemsetAsync(d.diff + n_nodes, 0, sizeof(int32_t), st));
    GDS_CUDA(cudaMemsetAsync(d.outdeg, 0, (n_nodes + 1) * sizeof(uint32_t), st));
    GDS_CUDA(cudaMemsetAsync(d.indeg, 0, (n_nodes + 1) * sizeof(uint32_t), st));
    return d;
}

template <typename K>
void build_bundles(gds_ctx* c, SolveCall& sc, const TileMap& tm, const uint32_t* cross_idx,
                   bool local_keys, int keybits, const uint32_t* fused_ref_len) {
    cudaStream_t st = sc.st;
    const size_t n_items = tm.n_items;
    const uint32_t n_nodes = sc.plan.n_nodes, minlen = sc.minlen;
    const int lenbits = sc.lenbits;
    K* kA = c->keysA.get<K>(n_items);
    K* kB = c->keysB.get<K>(n_items);
    uint32_t* vA = c->valsA.get<uint32_t>(n_items);
    uint32_t* vB = c->valsB.get<uint32_t>(n_items);
    int where;
    if (local_keys) {
        ReadKeys<K, true> rk{sc.S, sc.E, sc.vl, cross_idx, sc.N, lenbits, minlen, fused_ref_len,
                             sc.stats(), minlen, sc.maxlen};
        where = radix_sort_pairs<K, ReadKeys<K, true>>(kA, vA, kB, vB, tm, keybits, c->radix, st,
                                                       c->atomic_rank, &sc.sort_passes, &rk);
    } else {
        ReadKeys<K, false> rk{sc.S, sc.E, sc.vl, cross_idx, sc.N, lenbits, minlen, nullptr,
                              sc.stats(), 0, 0};
        where = radix_sort_pairs<K, ReadKeys<K, false>>(kA, vA, kB, vB, tm, keybits, c->radix, st,
                                                        c->atomic_rank, &sc.sort_passes, &rk);
    }
    const K* keys = where ? kB : kA;
    sc.sorted_idx = where ? vB : vA;
    // bundle heads
    const uint32_t n_tiles = tm.n_tiles;
    uint32_t* tc = c->tile_counts.get<uint32_t>(n_tiles + 1);
    GDS_CUDA(cudaMemsetAsync(tc + n_tiles, 0, sizeof(uint32_t), st));
    uint32_t* head_bits = c->head_bits.get<uint32_t>((size_t)n_tiles * (kRsTile / 32));
    launch("heads_count", (sizeof(K) * 8ull + 1ull) * n_items / 8, k_heads_count<K>, n_tiles,
           kHeadThreads, 0, st, keys, tm, tc, head_bits);
    exclusive_scan_u32(tc, tc, n_tiles + 1, c->scan, st);
    GDS_CUDA(cudaMemcpyAsync(&sc.ds->n_bundles, tc + n_tiles, 4, cudaMemcpyDeviceToDevice, st));
    uint32_t B = 0;
    d2h_sync(c, &B, tc + n_tiles, 1);  // the sort path sizes and launches by the exact count
    sc.B = B;
    if (fused_ref_len) read_input_verdict(c, sc.ds);  // validation fused into the first histogram pass
    uint32_t* b_first = c->b_first.get<uint32_t>(B + 1);
    K* b_key = c->b_key.get<K>(B + 1);
    launch("heads_write", n_items / 8ull + (4ull + 2 * sizeof(K)) * B, k_heads_write<K>, n_tiles,
           kHeadWriteThreads, 0, st, keys, tm, tc, head_bits, b_first, b_key);
    BundleRec* bund = c->bund.get<BundleRec>(B + 1);
    uint32_t* b_t = c->b_t.get<uint32_t>(B + 1);
    const Degrees d = alloc_degrees(c, st, n_nodes);
    if (B)
        launch("bundle_fill", (sizeof(K) + 8ull + 12ull + 16ull) * B, k_bundle_fill<K>, div_up(B, 256),
               256, 0, st, b_key, b_first, sc.sorted_idx, B, (uint32_t)n_items, lenbits, minlen,
               sc.vl, local_keys, bund, b_t, d.diff, d.outdeg, d.indeg, sc.odiff);
}

// K2 by radix sort of the arc items
void sort_bundles(gds_ctx* c, SolveCall& sc, const uint32_t* cross_idx, size_t n_items) {
    const uint32_t ns = sc.ns;
    // the arc sort is segmented by sample unless some sample is cut into segments (then the
    // right parts live after all reads and one group with global keys is sorted)
    const bool local_keys = !sc.plan.split;
    // the hinted path validates inside the first histogram pass; a segmented reference
    // (global keys, rare) keeps the stand-alone validation kernel
    if (sc.fused_validation && !local_keys) {
        const StatsBlock h = validate_reads(c, sc);
        if (h.len_min < sc.minlen || h.len_max > sc.maxlen) throw InputFail{GDS_ERR_ARG, 1, kBadHints};
    }
    const uint32_t* fused_ref = (sc.fused_validation && local_keys) ? sc.reflen_d : nullptr;
    TileMap tm{nullptr, nullptr, 1, tiles_for(n_items), n_items};
    int keybits = sc.nodebits + sc.lenbits;
    if (local_keys && ns > 1) {
        std::vector<uint32_t> toff(ns + 1, 0);
        uint32_t maxvn = 1;
        for (uint32_t k = 0; k < ns; ++k) {
            const uint64_t nk = sc.foff_host[k + 1] - sc.foff_host[k];
            toff[k + 1] = toff[k] + tiles_for(nk);
            maxvn = std::max(maxvn, sc.rd->ref_len[k] + 1);
        }
        uint32_t* toff_d = c->tile_off_d.get<uint32_t>(ns + 1);
        GDS_CUDA(cudaMemcpyAsync(toff_d, toff.data(), toff.size() * 4, cudaMemcpyHostToDevice, sc.st));
        tm = TileMap{toff_d, sc.foff_dev, ns, toff[ns], n_items};
        keybits = bits_for(maxvn - 1) + sc.lenbits;
    }
    sc.out->key_bits = keybits;
    if (keybits <= 32)
        build_bundles<uint32_t>(c, sc, tm, cross_idx, local_keys, keybits, fused_ref);
    else
        build_bundles<unsigned long long>(c, sc, tm, cross_idx, local_keys, keybits, fused_ref);
}

bool direct_eligible(const gds_reads* rd, uint32_t ns, const uint32_t* S, const uint32_t* E) {
    if (((uintptr_t)S | (uintptr_t)E) & 15) return false;  // 16-byte loads
    uint64_t tot = 0;
    for (uint32_t k = 0; k < ns; ++k) {
        const uint64_t kk = (uint64_t)rd->ref_len[k] + 1;  // one slot per node
        if (kk > kDirectMaxKeys) return false;
        tot += (kk + 31) & ~31ull;
    }
    return tot < (1ull << 31);
}

// What the bundle kernel of either histogram path writes to
struct BundleOut {
    uint32_t n_tiles;
    const uint32_t* tc;  // bundles before each tile
    BundleRec* bund;
    uint32_t *b_t, *b_slot, *ident;
    Degrees d;
};

// The bundle buffers of a histogram path, sized for B bundles; the identity in-CSR when there is
// one read length (always on the shared-memory path)
void bundle_buffers(gds_ctx* c, SolveCall& sc, DirectPlan& plan, uint32_t B, BundleOut& o) {
    sc.B = B;
    o.bund = c->bund.get<BundleRec>(B + 1);
    o.b_t = c->b_t.get<uint32_t>(B + 1);
    o.b_slot = c->b_slot.get<uint32_t>(B + 1);
    o.ident = sc.minlen == sc.maxlen ? c->ident.get<uint32_t>(B + 1) : nullptr;
    plan.on = true;
    plan.in_bid = o.ident;
}

// What both histogram paths do once plan.ghist holds the counts: count the non-empty keys per
// tile, scan, the bundle count (on the device; b_bound sizes the buffers), the bundle buffers and
// the cleared degree arrays (k_direct_bundles writes the whole difference array itself).
BundleOut histogram_bundles(gds_ctx* c, SolveCall& sc, DirectPlan& plan, uint64_t b_bound) {
    cudaStream_t st = sc.st;
    const uint32_t ktot = plan.ktot;
    const uint32_t n_tiles = (uint32_t)div_up(ktot, kDkTile);
    uint32_t* tc = c->tile_counts.get<uint32_t>(n_tiles + 1);
    GDS_CUDA(cudaMemsetAsync(tc + n_tiles, 0, sizeof(uint32_t), st));
    launch("direct_count", 4ull * ktot, k_direct_count, n_tiles, kDkThreads, 0, st, plan.ghist, ktot, tc);
    exclusive_scan_u32(tc, tc, n_tiles + 1, c->scan, st);
    GDS_CUDA(cudaMemcpyAsync(&sc.ds->n_bundles, tc + n_tiles, 4, cudaMemcpyDeviceToDevice, st));
    uint32_t B = (uint32_t)std::min<uint64_t>(ktot, b_bound);
    if (sc.minlen != sc.maxlen) {
        // several read lengths (global memory): the in-CSR order comes from a radix sort of the
        // bundles (build_nodes), which needs their exact number; the input verdict comes with the
        // same synchronisation
        d2h_sync(c, &B, tc + n_tiles, 1);
        read_input_verdict(c, sc.ds);
    }
    BundleOut o{n_tiles, tc};
    bundle_buffers(c, sc, plan, B, o);
    o.d = alloc_degrees(c, st, sc.plan.n_nodes, plan.global || !B);
    return o;
}

void build_bundles_direct(gds_ctx* c, SolveCall& sc) {
    cudaStream_t st = sc.st;
    DirectPlan& plan = sc.direct;
    const uint32_t ns = sc.ns;
    const uint64_t N = sc.N;
    // host-side layout: histogram regions and work items (sample parts)
    std::vector<uint32_t> lay(2 * (ns + 1), 0);
    uint32_t* kbase = lay.data();
    uint32_t* item_off = lay.data() + ns + 1;
    const uint64_t part_len = std::max<uint64_t>(65536, (N + 8ull * kNumSMs - 1) / (8ull * kNumSMs));
    uint32_t kmax = 32;
    for (uint32_t k = 0; k < ns; ++k) {
        const uint32_t kk = (sc.rd->ref_len[k] + 1 + 31u) & ~31u;
        kmax = std::max(kmax, kk);
        kbase[k + 1] = kbase[k] + kk;
        const uint64_t nk = sc.foff_host[k + 1] - sc.foff_host[k];
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
    const DirectLayout dl{sc.foff_dev, sc.reflen_d, sc.base_d, lay_d, lay_d + ns + 1, ns, sc.minlen};
    const unsigned smem = kmax * 4;
    raise_smem_limit(reinterpret_cast<const void*>(k_direct_hist), c->device,
                     (int)(kDirectMaxKeys * 4));
    raise_smem_limit(reinterpret_cast<const void*>(k_direct_mark), c->device,
                     (int)(kDmQueueBytes + kDirectMaxKeys));
    launch("direct_hist", 8ull * N + 4ull * ktot, k_direct_hist,
           (int)std::min<uint32_t>(n_items, (uint32_t)kNumSMs), kDhThreads, smem, st, sc.S, sc.E, dl,
           n_items, wc, ghist, kmax, sc.stats());
    plan.dl = dl;
    plan.ghist = ghist;
    plan.ktot = ktot;
    plan.kmax = kmax;
    plan.n_items = n_items;
    if (sc.direct_graph) {  // k_direct_graph (build_nodes) writes the bundles and every node array
        BundleOut o{};
        bundle_buffers(c, sc, plan, (uint32_t)std::min<uint64_t>(ktot, N), o);
        degree_buffers(c, sc.plan.n_nodes);
        return;
    }
    const BundleOut o = histogram_bundles(c, sc, plan, N);
    if (sc.B)
        launch("direct_bundles", 4ull * ktot + 40ull * sc.B, k_direct_bundles, o.n_tiles, kDkThreads, 0,
               st, ghist, ktot, dl, o.tc, o.bund, o.b_t, o.b_slot, o.ident, o.d.diff, o.d.outdeg,
               o.d.indeg);
}

// The same with the counters in global memory (direct.cuh: k_gdirect_*): any layout whose key space
// (virtual nodes x read lengths) stays L2-sized.
void build_bundles_gdirect(gds_ctx* c, SolveCall& sc) {
    cudaStream_t st = sc.st;
    DirectPlan& plan = sc.direct;
    const uint64_t N = sc.N;
    const uint32_t nlen = sc.maxlen - sc.minlen + 1;
    const uint32_t ktot = (uint32_t)((((uint64_t)sc.plan.n_nodes * nlen) + 31) & ~31ull);
    uint32_t* ghist = c->dhist.get<uint32_t>(ktot);
    GDS_CUDA(cudaMemsetAsync(ghist, 0, (size_t)ktot * 4, st));
    const GDirectLayout gl{sc.vl, nlen, sc.minlen, sc.maxlen};
    launch("gdirect_hist", 8ull * N + 4ull * ktot, k_gdirect_hist, div_up((long long)N, kGdTile),
           kGdThreads, 0, st, sc.S, sc.E, N, gl, ghist, sc.stats());
    plan.global = true;
    plan.gl = gl;
    plan.ghist = ghist;
    plan.ktot = ktot;
    // a read crossing a cut counts twice
    const BundleOut o = histogram_bundles(c, sc, plan, 2 * N);
    if (sc.B)
        launch("gdirect_bundles", 4ull * ktot + 40ull * sc.B, k_gdirect_bundles, o.n_tiles, kDkThreads,
               0, st, ghist, ktot, gl, o.tc, o.bund, o.b_t, o.b_slot, o.ident, o.d.diff, o.d.outdeg,
               o.d.indeg, sc.odiff);
}

// K5 on the direct path (direct.cuh): classify the bundles, mark the reads of saturated bundles in
// one parallel streaming pass, rank the candidates of partial bundles.  Nothing is read back here.
// The candidate buffer keeps the size it has (never below N/8 slots or cand_need);
// k_direct_classify raises ctl flag 2 when the candidates do not fit, the mark / ranking kernels
// then do nothing, and select_reads — which sees the flag with the final readback — repeats the
// selection with a larger buffer.
void direct_select(gds_ctx* c, SolveCall& sc, size_t cand_need) {
    cudaStream_t st = sc.st;
    const DirectPlan& dp = sc.direct;
    const uint32_t B = sc.B;
    const uint32_t* B_dev = &sc.ds->n_bundles;
    const size_t N = sc.N;
    uint32_t* bm = sc.bm;
    unsigned long long* totals = sc.totals();
    BundleRec* bund = c->bund.as<BundleRec>();
    uint32_t* b_slot = c->b_slot.as<uint32_t>();
    uint32_t* ctl = c->dctl.get<uint32_t>(4);
    GDS_CUDA(cudaMemsetAsync(ctl, 0, 16, st));
    uint32_t* kstat = c->kstat.get<uint32_t>(dp.ktot / 16 + 1);
    uint32_t* pb = c->pbund.get<uint32_t>(3 * ((size_t)B + 1));
    uint32_t* fill = pb + 2 * ((size_t)B + 1);
    GDS_CUDA(cudaMemsetAsync(kstat, 0, ((size_t)dp.ktot / 16 + 1) * 4, st));
    // never below N/8 slots: the share of reads in partial bundles varies from call to call
    // and regrowing the arena is expensive
    size_t cand_cap = std::max<size_t>({cand_need, N / 8, c->cand.cap / 4, (size_t)1});
    cand_cap = std::min<size_t>(cand_cap, 0xffffffffu);
    uint32_t* cand = c->cand.get<uint32_t>(cand_cap);
    launch("direct_classify", 20ull * B, k_direct_classify, div_up(B, 256), 256, 0, st, bund,
           b_slot, dp.ghist, kstat, pb, pb + B + 1, fill, ctl, B_dev, (uint32_t)cand_cap,
           sc.stats());
    if (dp.global) {
        launch("gdirect_mark", 8ull * N + dp.ktot / 4 + 8ull * N / 32, k_gdirect_mark,
               div_up((long long)N, kGdTile), kGdThreads, 0, st, sc.S, sc.E, N, dp.gl, dp.ghist,
               kstat, pb, fill, cand, bm, totals, ctl);
    } else {
        uint32_t* wc = c->dwork.as<uint32_t>() + 1;
        GDS_CUDA(cudaMemsetAsync(wc, 0, 4, st));
        const int grid = (int)std::min<uint32_t>(dp.n_items * kDmSplit, (uint32_t)kNumSMs * kDmCtasPerSm);
        launch("direct_mark", 4ull * N + dp.ktot / 4 + 8ull * N / 32, k_direct_mark, grid, kDmThreads,
               kDmQueueBytes + dp.kmax, st, sc.S, dp.dl, dp.n_items, wc, dp.ghist, kstat, pb, fill,
               cand, ctl, bm, totals);
    }
    // segments of a long reference (global path): ~10 reads per bundle, half a warp each
    launch("direct_partial", 16ull * (N / 64),
           dp.global ? k_direct_partial<true> : k_direct_partial<false>, kNumSMs * 32, 256, 0, st,
           pb, pb + B + 1, fill, cand, ctl, bm, totals);
    GDS_CUDA(cudaMemcpyAsync(sc.ds->ctl, ctl, 16, cudaMemcpyDeviceToDevice, st));
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

namespace {

// ---------------- the stages of gds_solve, in the order they run ----------------

// Argument checks: pure host, before any device work.  Fills the call's derived values.
int check_args(gds_ctx* c, SolveCall& sc) {
    const gds_reads* rd = sc.rd;
    const gds_filter* flt = sc.flt;
    const gds_params* prm = sc.prm;
    gds_result* out = sc.out;
    if (!rd || !out || rd->n_samples == 0 || !rd->read_off || !rd->ref_len)
        return fail(c, GDS_ERR_ARG, "null reads/result or n_samples == 0");
    const uint32_t ns = sc.ns = rd->n_samples;
    const uint64_t P = sc.P = rd->read_off[ns];
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
    if (P >= (1ull << 32) - 64) return fail(c, GDS_ERR_RANGE, "more than 2^32 reads in one call");
    if (flt) {
        if (P > 0 && (!rd->mapq || !rd->seq_len))
            return fail(c, GDS_ERR_ARG, "filter needs mapq and seq_len");
        for (uint32_t k = 0; k <= ns; ++k)
            if (rd->read_off[k] & 1)
                return fail(c, GDS_ERR_ARG, "filter needs an even read count per sample (mates adjacent)");
        if (flt->n_amplicons && (!flt->amp_start || !flt->amp_end))
            return fail(c, GDS_ERR_ARG, "null amplicon table");
    }
    if (sc.flags & GDS_FIND_PAIRS)  // mates are read 2i and 2i+1 of a sample: a pair must not straddle two
        for (uint32_t k = 0; k <= ns; ++k)
            if (rd->read_off[k] & 1)
                return fail(c, GDS_ERR_ARG, "GDS_FIND_PAIRS needs an even read count per sample (mates adjacent)");
    uint64_t nn64 = 0;
    sc.base.assign(ns + 1, 0);
    for (uint32_t k = 0; k < ns; ++k) {
        nn64 += (uint64_t)rd->ref_len[k] + 1;
        if (nn64 >= kLabelInf) return fail(c, GDS_ERR_RANGE, "total reference length beyond 2^30 nodes");
        sc.base[k + 1] = (uint32_t)nn64;
    }
    sc.n_onodes = (uint32_t)nn64;
    sc.out_dev = sc.flags & GDS_OUTPUT_ON_DEVICE;
    sc.do_solve = !(sc.flags & GDS_NO_SOLVE);
    sc.sp = SolveParams{64, 150, 1, 0};
    if (prm && (prm->gr_interval_min | prm->gr_levels_pct | prm->gr_relabel_pct | prm->max_rounds)) {
        sc.sp.gr_interval_min = prm->gr_interval_min;
        sc.sp.gr_levels_pct = prm->gr_levels_pct;
        sc.sp.gr_relabel_pct = prm->gr_relabel_pct;
        sc.sp.max_rounds = prm->max_rounds;
    }
    sc.algorithm = prm ? prm->algorithm : 0u;
    sc.schedule = prm ? prm->schedule : 0u;
    if (sc.schedule > 3) return fail(c, GDS_ERR_ARG, "gds_params.schedule must be 0, 1, 2 or 3");
    // a call that filters by an amplicon table works on amplicon-tiled coverage, which dips between
    // the amplicons whatever M is: the default then is the graph reduction at every M (config 2:
    // 6.1 -> 3.6 ms).  A call-level choice like the filter itself, never a property of the batch.
    if (sc.schedule == 0 && flt && flt->n_amplicons > 0) sc.schedule = 3;
    if (sc.algorithm > 1) return fail(c, GDS_ERR_ARG, "gds_params.algorithm must be 0 (quasi-MCP) or 1 (minimum cardinality)");
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
    out->n_reads_in = P;
    out->n_nodes = sc.n_onodes;
    return GDS_OK;
}

// Input upload and widening: 32-bit start and end columns on the device, the per-sample tables,
// and the stats block initialised.
void upload_inputs(gds_ctx* c, SolveCall& sc) {
    const gds_reads* rd = sc.rd;
    const uint64_t P = sc.P;
    const uint32_t ns = sc.ns;
    cudaStream_t st = sc.st;
    const bool in_dev = sc.flags & GDS_INPUT_ON_DEVICE;
    if (in_dev || P == 0) {
        sc.dS = rd->start;
        sc.dE = rd->end;
        sc.dQ = rd->mapq;
        sc.dLen = rd->seq_len;
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
        sc.dS = s;
        sc.dE = e;
        if (sc.flt) {
            uint8_t* q = c->in_mapq.get<uint8_t>(P);
            uint32_t* l = c->in_len.get<uint32_t>(P);
            GDS_CUDA(cudaMemcpyAsync(q, rd->mapq, P, cudaMemcpyHostToDevice, st));
            GDS_CUDA(cudaMemcpyAsync(l, rd->seq_len, P * 4, cudaMemcpyHostToDevice, st));
            sc.dQ = q;
            sc.dLen = l;
        }
    }
    if (P > 0 && (rd->start16 || !rd->end)) {  // compact columns: widen to 32 bits (k_expand_reads)
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
        launch("expand_reads", (s16 ? 2ull : 4ull) * P + (So != s32 ? 4ull : 0ull) * P +
                                   (e32 ? 0ull : 4ull) * P,
               k_expand_reads, div_up((long long)P, 256 * 8), 256, 0, st, s16, s32, e32, rd->len_min,
               P, So, Eo);
        sc.dS = So;
        sc.dE = Eo;
    }
    sc.off_d = c->off_d.get<uint64_t>(ns + 1);
    sc.reflen_d = c->reflen_d.get<uint32_t>(ns);
    sc.base_d = c->base_d.get<uint32_t>(ns + 1);
    GDS_CUDA(cudaMemcpyAsync(sc.off_d, rd->read_off, (ns + 1) * 8, cudaMemcpyHostToDevice, st));
    GDS_CUDA(cudaMemcpyAsync(sc.reflen_d, rd->ref_len, ns * 4, cudaMemcpyHostToDevice, st));
    GDS_CUDA(cudaMemcpyAsync(sc.base_d, sc.base.data(), (ns + 1) * 4, cudaMemcpyHostToDevice, st));
    sc.ds = c->small.get<StatsBlock>(1);
    {
        StatsBlock init{};
        init.len_min = 0xffffffffu;
        memcpy(c->pinned, &init, sizeof init);
        GDS_CUDA(cudaMemcpyAsync(sc.ds, c->pinned, sizeof init, cudaMemcpyHostToDevice, st));
    }
    GDS_CUDA(cudaEventRecord(c->ev[EV_H2D], st));
}

// K1: the pair filter (mapq, read length, amplicons) compacts the reads K2 sees
void filter_reads(gds_ctx* c, SolveCall& sc) {
    const gds_filter* flt = sc.flt;
    const uint32_t ns = sc.ns;
    const uint64_t P = sc.P;
    cudaStream_t st = sc.st;
    gds_result* out = sc.out;
    sc.S = sc.dS;
    sc.E = sc.dE;
    sc.foff_dev = sc.off_d;
    sc.N = P;
    sc.foff_host.assign(sc.rd->read_off, sc.rd->read_off + ns + 1);
    if (flt && P > 0) {
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
        uint8_t* pp = (sc.out_dev && out->pair_pass) ? out->pair_pass
                                                     : c->pair_pass.get<uint8_t>(n_pairs);
        uint32_t* f32 = c->flag32.get<uint32_t>(n_pairs);
        int grid = std::min<long long>(div_up(n_pairs, 256), kNumSMs * 16);
        launch("filter_flags", 13ull * P + 5ull * n_pairs, k_filter_flags, grid, 256, 0, st, sc.dS,
               sc.dE, sc.dQ, sc.dLen, n_pairs, fa, pp, f32);
        exclusive_scan_u32(f32, f32, n_pairs, c->scan, st);
        uint64_t* foff = c->foff_d.get<uint64_t>(ns + 1);
        launch("filter_offsets", 16ull * (ns + 1), k_filter_offsets, div_up(ns + 1, 128), 128, 0, st,
               sc.off_d, ns, f32, pp, n_pairs, foff);
        d2h_sync(c, sc.foff_host.data(), foff, ns + 1);
        const uint64_t N = sc.N = sc.foff_host[ns];
        uint32_t* fS = c->fS.get<uint32_t>(N);
        uint32_t* fE = c->fE.get<uint32_t>(N);
        launch("filter_compact", 5ull * n_pairs + 16ull * N, k_filter_compact, grid, 256, 0, st, sc.dS,
               sc.dE, pp, f32, n_pairs, fS, fE);
        sc.S = fS;
        sc.E = fE;
        sc.foff_dev = foff;
        if (!sc.out_dev) deliver(c, out->pair_pass, pp, n_pairs, false);
    }
    out->n_filtered = sc.N;
    if (out->filt_off) memcpy(out->filt_off, sc.foff_host.data(), (ns + 1) * 8);
    GDS_CUDA(cudaEventRecord(c->ev[EV_FILTER], st));
}

// Read-length bounds: exact ones from the caller (the host adapter has them for free from its
// narrowing loop) let the validation ride on the first histogram pass of K2; without them
// k_validate finds them.
void read_length_bounds(gds_ctx* c, SolveCall& sc) {
    const gds_reads* rd = sc.rd;
    sc.minlen = sc.maxlen = 1;
    if (sc.N == 0) return;
    if (rd->len_max != 0 && rd->len_min != 0 && rd->len_min <= rd->len_max) {
        sc.minlen = rd->len_min;
        sc.maxlen = rd->len_max;
        sc.fused_validation = true;
    } else {
        const StatsBlock h = validate_reads(c, sc);
        sc.minlen = h.len_min;
        sc.maxlen = h.len_max;
    }
    sc.lenbits = bits_for(sc.maxlen - sc.minlen);
}

// K4 (generalised): the virtual node space — references longer than two segments are cut.
SegPlan plan_segments(const gds_reads* rd, const gds_params* prm, const std::vector<uint32_t>& base,
                      uint32_t minlen, uint32_t maxlen) {
    const uint32_t ns = rd->n_samples;
    SegPlan pl{};
    pl.seg_len = (prm && prm->seg_len) ? prm->seg_len : default_seg_len(ns, rd->ref_len);
    // default rule, one read length R: a whole number of reads per segment.  Every node then
    // reaches the segment's end in the same number of read hops as its neighbours within one
    // "lane block", the cut node's bundles are all admissible at once, and a segment of config 4
    // needs 175 rounds instead of 255 (tools/k3_tail.py).  The oracle rounds the same way.
    if (!(prm && prm->seg_len) && minlen == maxlen && maxlen > 1)
        pl.seg_len = (pl.seg_len + maxlen - 1) / maxlen * maxlen;
    const uint32_t seg = pl.seg = pl.seg_len >= maxlen ? pl.seg_len : 0xffffffffu;  // a read crosses <= 1 cut
    pl.hvs.resize(ns);
    uint64_t vb = 0, est = 0;
    for (uint32_t k = 0; k < ns; ++k) {
        VSample& v = pl.hvs[k];
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
        if (vb >= kLabelInf) throw CallFail{GDS_ERR_RANGE, "segmented reference beyond 2^30 nodes"};
        if (v.nseg > 1) {
            pl.split = true;
            for (uint32_t j = 1; j < v.nseg; ++j) pl.hcuts.push_back(v.obase + j * seg);
        }
        pl.max_comp_nodes = std::max(pl.max_comp_nodes, v.nseg == 1 ? v.L + 1 : seg + 1);
        est += v.nseg;
    }
    pl.n_nodes = (uint32_t)vb;
    // (a component has >= 2 nodes)
    pl.comp_estimate = (uint32_t)std::min<uint64_t>(est, pl.n_nodes / 2 + 1);
    return pl;
}

// What K3 runs, from the call's arguments and the segment plan alone: the graph build writes the
// node records in the form the chosen kernel reads.
void plan_solve(SolveCall& sc) {
    // Forced reads out, cuts in (graph.cuh, DESIGN.md §4): bundles that cover a position with
    // cov <= M get capacity 0 for the solve and their fixed flow goes into the demand; components
    // are cut at every such position.  Not for the minimum-cardinality sweep (it walks all
    // bundles itself) and not with gds_params.schedule = 1 (round 1's graph and schedule).
    // ... and not below the supply at which the express schedule starts (kExpressMinSupply):
    // with M = 100 (configs 1, 2, 5) the classic schedule on the uncut graph needs no more
    // rounds than hops, and the three extra passes over nodes and bundles would cost config 5
    // 0.25 ms of 5.75 (measured); gds_params.schedule = 2 applies them regardless.
    sc.forced_cuts = sc.do_solve && sc.algorithm == 0 && sc.schedule != 1 &&
                     (sc.schedule >= 2 || sc.M >= kExpressMinSupply);
    // the express schedule (maxflow_sm.cuh): components with a supply of kExpressMinSupply or
    // more — none when M is below that, and then nothing about the launch changes
    uint32_t express_on = sc.schedule == 1 ? 0u : sc.schedule == 2 ? 2u : 1u;  // (3: the usual supply rule)
    if (!sc.forced_cuts || (express_on == 1 && sc.M < kExpressMinSupply)) express_on = 0;
    sc.express_on = express_on;
    sc.mf2 = sc.do_solve && sc.algorithm == 0
                 ? plan_maxflow_sm(sc.plan.comp_estimate, sc.plan.max_comp_nodes, express_on != 0, sc.knobs)
                 : Mf2Plan{};
}

// K2: the bundles (arcs of equal start, end and length) and the node degrees.  Shared-memory
// histogram, global-memory histogram or radix sort.
void find_bundles(gds_ctx* c, SolveCall& sc) {
    const SegPlan& pl = sc.plan;
    const uint32_t ns = sc.ns, n_nodes = pl.n_nodes, n_onodes = sc.n_onodes;
    const uint64_t N = sc.N;
    cudaStream_t st = sc.st;
    gds_result* out = sc.out;
    sc.vs_d = c->vs_d.get<VSample>(ns);
    GDS_CUDA(cudaMemcpyAsync(sc.vs_d, pl.hvs.data(), ns * sizeof(VSample), cudaMemcpyHostToDevice, st));
    sc.vl = VLayout{sc.vs_d, sc.foff_dev, ns, pl.seg};
    sc.nodebits = bits_for(n_nodes ? n_nodes - 1 : 0);
    out->key_bits = sc.nodebits + sc.lenbits;
    if (pl.split) {
        sc.odiff = c->odiff.get<int32_t>(n_onodes + 1);
        sc.oexcl = c->oexcl.get<uint32_t>(n_onodes + 1);
        GDS_CUDA(cudaMemsetAsync(sc.odiff, 0, ((size_t)n_onodes + 1) * 4, st));
    }
    // 0 = choose, 1 = always the radix sort, 2 = the direct histogram whenever eligible
    const int bmode = sc.prm ? (int)sc.prm->bundle_mode : 0;
    const bool use_direct = N > 0 && !pl.split && bmode != 1 && sc.minlen == sc.maxlen &&
                            direct_eligible(sc.rd, ns, sc.S, sc.E);
    const bool use_gdirect = N > 0 && !use_direct && bmode != 1 &&
                             (uint64_t)n_nodes * ((uint64_t)sc.maxlen - sc.minlen + 1) <= kGDirectMaxKeys;
    sc.direct_graph = use_direct && !sc.forced_cuts;
    size_t n_items = N;
    uint32_t* cross_idx = nullptr;
    if (pl.split && N > 0 && !use_gdirect) {  // right parts of the reads that cross a cut
        uint32_t n_ct = (uint32_t)((N + kCrossTile - 1) / kCrossTile);
        uint32_t* ctc = c->cross_tc.get<uint32_t>(n_ct + 1);
        GDS_CUDA(cudaMemsetAsync(ctc + n_ct, 0, 4, st));
        launch("cross_count", 8ull * N, k_cross_count, n_ct, kCrossThreads, 0, st, sc.S, sc.E, N, sc.vl, ctc);
        exclusive_scan_u32(ctc, ctc, n_ct + 1, c->scan, st);
        uint32_t X = 0;
        d2h_sync(c, &X, ctc + n_ct, 1);
        cross_idx = c->cross_idx.get<uint32_t>(X + 1);
        if (X)
            launch("cross_write", 8ull * N + 4ull * X, k_cross_write, n_ct, kCrossThreads, 0, st, sc.S,
                   sc.E, N, sc.vl, ctc, cross_idx);
        n_items = N + X;
        if (n_items >= (1ull << 32) - 64)
            throw CallFail{GDS_ERR_RANGE, "more than 2^32 arc items after segmentation"};
    }
    out->n_arc_items = n_items;  // (global histogram: N + n_cross, with the final readback)
    if (use_direct) {
        build_bundles_direct(c, sc);
        out->key_bits = bits_for(sc.direct.kmax - 1);
        out->bundle_path = 1;
    } else if (use_gdirect) {
        build_bundles_gdirect(c, sc);
        out->key_bits = bits_for((uint64_t)sc.direct.ktot - 1);
        out->bundle_path = 2;
    } else if (N > 0) {
        sort_bundles(c, sc, cross_idx, n_items);
    } else {
        alloc_degrees(c, st, n_nodes);
        c->b_first.get<uint32_t>(1);
        c->b_t.get<uint32_t>(1);
        c->bund.get<BundleRec>(1);
    }
    sc.deg = Degrees{c->diff.as<int32_t>(), c->outdeg.as<uint32_t>(), c->indeg.as<uint32_t>()};
    out->sort_passes = sc.sort_passes;
}

// The graph build of every path but k_direct_graph's: scans, forced cuts, node records, components,
// in-CSR order
void build_nodes_chain(gds_ctx* c, SolveCall& sc, uint32_t* cov_dev, int32_t* dem_dev) {
    const uint32_t n_nodes = sc.plan.n_nodes, n_onodes = sc.n_onodes, B = sc.B, M = sc.M;
    const bool split = sc.plan.split;
    cudaStream_t st = sc.st;
    unsigned long long* totals = sc.totals();
    const Degrees& d = sc.deg;
    uint32_t* excl = sc.excl;
    {  // coverage from the difference array and both CSR row starts: one launch
        ScanArrays sa{{reinterpret_cast<const uint32_t*>(d.diff), d.outdeg, d.indeg}, {excl, d.outdeg, d.indeg}};
        exclusive_scan_u32_multi(sa, 3, n_nodes + 1, c->scan, st);
    }
    uint32_t* cstart = c->comp_start.get<uint32_t>(n_nodes + 1);
    uint32_t* cend = c->comp_end.get<uint32_t>(n_nodes + 1);
    GDS_CUDA(cudaMemsetAsync(cstart + n_nodes, 0, 4, st));
    GDS_CUDA(cudaMemsetAsync(cend + n_nodes, 0, 4, st));
    int32_t* adj = nullptr;
    if (sc.forced_cuts && B) {
        uint32_t* unc = c->unc.get<uint32_t>((size_t)n_nodes + 1);
        adj = c->adj.get<int32_t>((size_t)n_nodes + 1);
        sc.fmult = c->fmult.get<uint32_t>((size_t)B + 1);
        sc.dead = c->dead.get<uint8_t>((size_t)n_nodes + 1);  // nodes without a live bundle of their own (express rule U4)
        GDS_CUDA(cudaMemsetAsync(adj, 0, ((size_t)n_nodes + 1) * 4, st));
        GDS_CUDA(cudaMemsetAsync(sc.dead, 0, (size_t)n_nodes + 1, st));
        launch("uncapped_flags", 12ull * n_nodes, k_uncapped_flags, div_up((long long)n_nodes + 1, 256),
               256, 0, st, excl, d.diff, n_nodes, M, unc);
        exclusive_scan_u32(unc, unc, (size_t)n_nodes + 1, c->scan, st);
        launch("forced_bundles", 8ull * n_nodes, k_forced_bundles, div_up((long long)n_nodes, 256), 256,
               0, st, c->bund.as<BundleRec>(), d.outdeg, n_nodes, sc.maxlen, unc, adj, sc.fmult, sc.dead);
    }
    launch("node_finalize", 60ull * n_nodes, k_node_finalize, div_up((long long)n_nodes + 1, 256), 256,
           0, st, excl, d.diff, d.outdeg, d.indeg, n_nodes, M, sc.node, sc.d_snap, cstart, cend,
           split ? nullptr : cov_dev, split ? nullptr : dem_dev, sc.dem_v, totals, adj,
           sc.forced_cuts ? M : 0u, &sc.ds->res_supply, sc.dead);
    if (split) {
        exclusive_scan_u32(reinterpret_cast<const uint32_t*>(sc.odiff), sc.oexcl, (size_t)n_onodes + 1,
                           c->scan, st);
        launch("orig_outputs", 16ull * n_onodes, k_orig_outputs, div_up(n_onodes, 256), 256, 0, st,
               sc.oexcl, sc.odiff, n_onodes, M, cov_dev, dem_dev, totals);
        const std::vector<uint32_t>& hcuts = sc.plan.hcuts;
        uint32_t* cuts_d = c->cut_nodes.get<uint32_t>(hcuts.size());
        GDS_CUDA(cudaMemcpyAsync(cuts_d, hcuts.data(), hcuts.size() * 4, cudaMemcpyHostToDevice, st));
        launch("cut_through", 12ull * hcuts.size(), k_cut_through, div_up(hcuts.size(), 128), 128, 0, st,
               cuts_d, (uint32_t)hcuts.size(), sc.oexcl, sc.odiff, M, totals);
    }
    uint32_t* sidx = c->comp_sidx.get<uint32_t>(n_nodes + 1);
    exclusive_scan_u32(cstart, sidx, n_nodes + 1, c->scan, st);
    GDS_CUDA(cudaMemcpyAsync(&sc.ds->n_comp, sidx + n_nodes, 4, cudaMemcpyDeviceToDevice, st));
    launch("comp_write", 16ull * n_nodes, k_comp_write, div_up(n_nodes, 256), 256, 0, st, cstart, cend,
           sidx, n_nodes, sc.comp_lo, sc.comp_hi);
    // in-CSR: bundle ids ordered by (end node, bundle id) = stable sort of ids by b_t
    if (B && !sc.in_bid) {
        uint32_t* tkA = c->tkA.get<uint32_t>(B);
        uint32_t* tkB = c->tkB.get<uint32_t>(B);
        uint32_t* tvA = c->tvA.get<uint32_t>(B);
        uint32_t* tvB = c->tvB.get<uint32_t>(B);
        GDS_CUDA(cudaMemcpyAsync(tkA, c->b_t.as<uint32_t>(), (size_t)B * 4,
                                 cudaMemcpyDeviceToDevice, st));
        TileMap btm{nullptr, nullptr, 1, tiles_for(B), B};
        int w = radix_sort_pairs<uint32_t>(tkA, tvA, tkB, tvB, btm, sc.nodebits, c->radix, st,
                                           c->atomic_rank);
        sc.in_bid = w ? tvB : tvA;
    }
}

// Coverage and CSR row starts, the forced cuts, the node records, the components and the in-CSR
void build_nodes(gds_ctx* c, SolveCall& sc) {
    const uint32_t n_nodes = sc.plan.n_nodes, n_onodes = sc.n_onodes, B = sc.B, M = sc.M;
    cudaStream_t st = sc.st;
    gds_result* out = sc.out;
    unsigned long long* totals = sc.totals();
    const Degrees& d = sc.deg;
    uint32_t* excl = sc.excl = c->excl.get<uint32_t>(n_nodes + 1);
    sc.node = c->node_rec.get<NodeRec>((size_t)n_nodes + 1);
    sc.d_snap = c->n_dsnap.get<uint32_t>(n_nodes);
    sc.dem_v = c->dem_v.get<int32_t>((size_t)n_nodes + 1);
    // cov_capped / demand are reported on the ORIGINAL node space
    uint32_t* cov_dev = nullptr;
    int32_t* dem_dev = nullptr;
    if (out->cov_capped) cov_dev = sc.out_dev ? out->cov_capped : c->cov_tmp.get<uint32_t>(n_onodes);
    if (out->demand) dem_dev = sc.out_dev ? out->demand : c->dem_tmp.get<int32_t>(n_onodes);
    // the count stays on the device; on the host SegPlan::comp_estimate picks the K3 kernel and the
    // grid, and the arrays are sized by the bound (a component has >= 2 nodes)
    sc.n_comp_cap = n_nodes / 2 + 1;
    sc.comp_lo = c->comp_lo.get<uint32_t>(sc.n_comp_cap + 1);
    sc.comp_hi = c->comp_hi.get<uint32_t>(sc.n_comp_cap + 1);
    sc.in_bid = sc.direct.in_bid;  // single read length: bundle order is end order too
    if (sc.direct_graph) {
        // one pass writes what the scans, node_finalize, comp_write and in_src write below
        // (no split, no forced cuts: virtual == original nodes, cut_at = 0, no adjustment)
        const uint32_t n_tiles = (uint32_t)div_up((long long)n_nodes + 1, kDgTile);
        const LookbackWords lw = lookback_words(c->scan, 4ull * n_tiles, st);
        const DirectGraphOut o{c->bund.as<BundleRec>(), c->b_t.as<uint32_t>(), c->b_slot.as<uint32_t>(),
                               sc.in_bid, c->in_src.get<uint32_t>((size_t)B + 1), d.diff, excl, d.outdeg,
                               d.indeg, sc.node, sc.d_snap, sc.dem_v,
                               c->in1.get<uint32_t>((size_t)n_nodes + 1), sc.comp_lo, sc.comp_hi, cov_dev,
                               dem_dev, &sc.ds->n_bundles, &sc.ds->n_comp, totals, &sc.ds->res_supply};
        // (B is the bound)
        launch("direct_graph", 4ull * sc.direct.ktot + 60ull * n_nodes + 32ull * B, k_direct_graph,
               n_tiles, kDgThreads, 0, st, sc.direct.ghist, sc.direct.dl, n_nodes, M,
               sc.mf2.on ? 1u : 0u, o, lw.status, lw.ticket, lw.epoch, n_tiles);
    } else {
        build_nodes_chain(c, sc, cov_dev, dem_dev);
    }
    if (!sc.out_dev) {
        deliver(c, out->cov_capped, cov_dev, n_onodes, false);
        deliver(c, out->demand, dem_dev, n_onodes, false);
    }
    GDS_CUDA(cudaEventRecord(c->ev[EV_GRAPH], st));
}

// K3: max flow (k_maxflow_sm and/or k_maxflow), or the sweep of the minimum-cardinality solve
void solve_flow(gds_ctx* c, SolveCall& sc) {
    const uint32_t n_nodes = sc.plan.n_nodes, B = sc.B, n_comp = sc.plan.comp_estimate;
    const uint32_t max_comp_nodes = sc.plan.max_comp_nodes;
    const uint32_t* n_comp_dev = &sc.ds->n_comp;
    cudaStream_t st = sc.st;
    BundleRec* bund = c->bund.as<BundleRec>();
    const Degrees& d = sc.deg;
    if (sc.do_solve && sc.algorithm == 1 && sc.maxlen >= 4096)
        throw CallFail{GDS_ERR_ARG, "algorithm 1 (minimum cardinality) takes reads of up to 4095 positions"};
    const uint32_t express_on = sc.express_on;
    const Mf2Plan& mf2 = sc.mf2;
    uint32_t* in_src = c->in_src.get<uint32_t>((size_t)B + 1);
    uint32_t* in1 = c->in1.get<uint32_t>((size_t)n_nodes + 1);
    if (!sc.direct_graph) {  // (k_direct_graph wrote both)
        GDS_CUDA(cudaMemsetAsync(in1, 0xff, ((size_t)n_nodes + 1) * 4, st));
        if (B)
            launch("in_src", 24ull * B, k_in_src, div_up(B, 256), 256, 0, st, bund, sc.in_bid, d.indeg,
                   &sc.ds->n_bundles, in_src, mf2.on ? sc.node : nullptr, in1);
    }
    // per-component records only for the diagnostics dump; gds_result's counters are summed on
    // the device (MfTotals)
    sc.cstats = sc.knobs.dump_comp ? c->comp_stats.get<CompStats>(sc.n_comp_cap + 1) : nullptr;
    if (sc.do_solve && sc.algorithm == 1) {
        // K3': greedy interval multicover, one warp per component, then bundle flows
        uint32_t* wc = c->work_counter.get<uint32_t>(4);
        GDS_CUDA(cudaMemsetAsync(wc, 0, 16, st));
        uint32_t* taken = c->taken.get<uint32_t>((size_t)n_nodes + 2);
        GDS_CUDA(cudaMemsetAsync(taken, 0, ((size_t)n_nodes + 2) * 4, st));
        const SweepArgs a{SweepGraph{sc.excl, d.diff, d.outdeg, bund, taken}, sc.comp_lo, sc.comp_hi,
                          n_comp, n_comp_dev, sc.M, wc, &sc.ds->sweep_fail};
        launch_sweep(c, a, sc.maxlen, sc.minlen == sc.maxlen, 12ull * n_nodes + 8ull * B);
        if (B)
            launch("sweep_distribute", 12ull * n_nodes + 24ull * B, k_sweep_distribute,
                   div_up((long long)n_nodes, 256), 256, 0, st, taken, d.indeg, sc.in_bid, bund, n_nodes,
                   &sc.ds->sweep_fail);
    } else if (sc.do_solve) {
        uint32_t* wc = c->work_counter.get<uint32_t>(4);  // [0] sm kernel, [1] fallback, [2] list size
        GDS_CUDA(cudaMemsetAsync(wc, 0, 16, st));
        // k_maxflow gets at least one wave: the estimate may be low
        K3Args k{sc.comp_lo, sc.comp_hi, std::max<uint32_t>(n_comp, kNumSMs), wc,
                 c->qF.get<uint32_t>(n_nodes), c->qT.get<uint32_t>(n_nodes),
                 c->qN.get<uint32_t>(n_nodes), c->qH.get<uint32_t>(n_nodes), sc.sp, sc.cstats,
                 n_comp_dev, &sc.ds->mf};
        const unsigned long long mf_bytes = 36ull * n_nodes + 20ull * B;
        // compact labels for k_maxflow's relabels
        uint16_t* lab_g = c->lab_g.get<uint16_t>(2 * (size_t)n_nodes + 4);
        const MfGraph mg{sc.node, sc.d_snap, bund, sc.in_bid, in_src, sc.dem_v, in1};
        if (mf2.on) {
            uint32_t* fb_list = c->fb_list.get<uint32_t>(sc.n_comp_cap + 1);
            const Mf2Graph g2{sc.node, bund, sc.in_bid, in_src, d.outdeg, d.indeg, sc.dem_v,
                              sc.vs_d, sc.ns, express_on, mf2.classic_ok ? 1u : 0u, sc.dead};
            (mf2.per_sm >= 2 ? launch_mf2_shape<256, 0> : launch_mf2_shape<512, 1>)(
                c, mf2, g2, k, fb_list, wc + 2, mf_bytes);
            // whatever the shared-memory kernel could not take
            k.wc = wc + 1;
            launch_maxflow(c, MfArgs{mg, k, max_comp_nodes, fb_list, wc + 2, lab_g}, 0);
        } else {
            launch_maxflow(c, MfArgs{mg, k, max_comp_nodes, nullptr, nullptr, lab_g}, mf_bytes);
        }
    }
    if (sc.fmult)  // the forced bundles come back with their fixed flow: K5 keeps all their reads
        launch("forced_restore", 8ull * n_nodes, k_forced_restore, div_up((long long)n_nodes, 256), 256,
               0, st, bund, d.outdeg, n_nodes, sc.maxlen, c->unc.as<uint32_t>(), sc.fmult);
    GDS_CUDA(cudaEventRecord(c->ev[EV_MAXFLOW], st));
}

// K5 (selection), K6 (verification) and the final readback.  One pass in the normal case.  On a
// histogram path the selection may have to be repeated once: the final readback is the first time
// the host sees that the candidates of the partial bundles did not fit their buffer (it grows).
void select_reads(gds_ctx* c, SolveCall& sc) {
    const uint32_t B = sc.B, n_onodes = sc.n_onodes;
    const uint64_t N = sc.N;
    const bool split = sc.plan.split;
    cudaStream_t st = sc.st;
    gds_result* out = sc.out;
    unsigned long long* totals = sc.totals();
    const size_t n_words = (N + 31) / 32;
    uint32_t* bm = sc.bm = (sc.out_dev && out->kept_bitmap) ? out->kept_bitmap
                                                            : c->bitmap.get<uint32_t>(n_words + 1);
    StatsBlock& h = sc.hstat;
    size_t cand_need = 0;
    for (int attempt = 0;; ++attempt) {
        if (sc.do_solve) {
            GDS_CUDA(cudaMemsetAsync(bm, 0, n_words * 4, st));
            if (attempt) GDS_CUDA(cudaMemsetAsync(&sc.ds->n_kept, 0, 16, st));  // n_kept, violations
            if (B && sc.direct.on)
                direct_select(c, sc, cand_need);
            else if (B)
                launch("select", 8ull * B + 8ull * N / 32, k_select, div_up(B, 256), 256, 0, st,
                       c->b_first.as<uint32_t>(), c->bund.as<BundleRec>(), sc.sorted_idx, B, bm, totals);
        }
        if (!attempt) GDS_CUDA(cudaEventRecord(c->ev[EV_SELECT], st));

        // K6: verification (before find_pairs widens the set), on the original node space:
        // compares with the input coverage (odiff when segmented)
        if (sc.do_solve && (sc.flags & GDS_VERIFY)) {
            int32_t* vdiff = c->vdiff.get<int32_t>((size_t)n_onodes + 1);
            uint32_t* vexcl = c->vexcl.get<uint32_t>((size_t)n_onodes + 1);
            GDS_CUDA(cudaMemsetAsync(vdiff, 0, ((size_t)n_onodes + 1) * 4, st));
            if (n_words)
                launch("verify_accumulate", 4ull * n_words, k_verify_accumulate, div_up(n_words, 256), 256,
                       0, st, bm, sc.S, sc.E, N, sc.foff_dev, sc.base_d, sc.ns, vdiff);
            exclusive_scan_u32(reinterpret_cast<const uint32_t*>(vdiff), vexcl, (size_t)n_onodes + 1,
                               c->scan, st);
            launch("verify_compare", 16ull * n_onodes, k_verify_compare, div_up(n_onodes, 256), 256, 0, st,
                   vexcl, vdiff, split ? sc.oexcl : sc.excl, split ? sc.odiff : sc.deg.diff, n_onodes, sc.M,
                   totals);
        }
        if (sc.do_solve && (sc.flags & GDS_FIND_PAIRS) && n_words)
            launch("find_pairs", 8ull * n_words, k_find_pairs, div_up(n_words, 256), 256, 0, st, bm, n_words);
        if (!attempt) GDS_CUDA(cudaEventRecord(c->ev[EV_VERIFY], st));

        if (sc.do_solve && !sc.out_dev) deliver(c, out->kept_bitmap, bm, n_words, false);
        d2h_sync(c, &h, sc.ds, 1);
        input_verdict(h);
        const uint32_t cflags = sc.do_solve && B && sc.direct.on ? h.ctl[2] : 0;
        if (attempt || !(cflags & 2u)) break;
        cand_need = (size_t)h.ctl[1] + 1;  // the buffer the candidates need
    }
    out->n_bundles = h.n_bundles;
    out->n_components = h.n_comp;
    out->partial_bundles = h.ctl[0];
    out->partial_candidates = h.ctl[1];
    if (sc.direct.global) out->n_arc_items = N + h.n_cross;
}

// The result: flow and counters from the final readback, stage times, convergence
int finish(gds_ctx* c, SolveCall& sc, unsigned long long launches0) {
    gds_result* out = sc.out;
    const StatsBlock& h = sc.hstat;
    const bool split = sc.plan.split;
    const uint32_t n_comp = h.n_comp;
    // fstar_virtual = source capacity of the (virtual) network the kernel solved; when references
    // were segmented the closed-form F* of the ORIGINAL network is fstar_orig and through_flow
    // units pass straight through the cut nodes once the segment flows are stitched together
    const long long fstar_virtual = (long long)h.fstar_virtual;
    out->fstar = (int64_t)(split ? h.fstar_orig : h.fstar_virtual);
    out->n_kept = h.n_kept;
    out->verify_violations = h.violations;
    long long stuck = 0;
    if (sc.do_solve) {
        const MfTotals& ht = h.mf;
        // sink inflow of the residual problem + the forced bundles' fixed flows: whatever the
        // residual problem left undelivered (nothing, on valid input) is missing from F*
        out->flow_value = sc.forced_cuts ? fstar_virtual - ((long long)h.res_supply - ht.sink_flow)
                                         : ht.sink_flow;
        out->rounds_total = ht.rounds_total;
        out->rounds_max = ht.rounds_max;
        out->pushes = ht.pushes;
        out->relabels = ht.relabels;
        out->global_relabels = ht.grs;
        out->bfs_levels = ht.bfs_levels;
        out->max_frontier = ht.max_frontier;
        stuck = ht.stuck;
        if (sc.algorithm == 1) {
            // the sweep's cover IS a maximum flow (flow 1 on the kept reads, back arcs take the
            // surplus); sweep_fail counts deficits it could not fill and reads it could not place
            out->flow_value = h.sweep_fail ? -1 : fstar_virtual;
            stuck = (long long)h.sweep_fail;
        } else if (ht.n_solved != n_comp) {
            stuck += 1;  // a component was never taken: cannot happen
        }
    }
    if (sc.do_solve && n_comp && sc.knobs.dump_comp) {  // diagnostics only
        std::vector<CompStats> hs(n_comp);
        d2h_sync(c, hs.data(), sc.cstats, n_comp);
        if (FILE* fp = fopen(sc.knobs.dump_comp, "w")) {
            fprintf(fp, "comp rounds pushes relabels grs bfs_levels max_frontier frontier_sum cycles gr_init gr_bfs gr_snap front gr_later\n");
            for (uint32_t i = 0; i < n_comp; ++i)
                fprintf(fp, "%u %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu\n", i,
                        hs[i].rounds, hs[i].pushes, hs[i].relabels, hs[i].grs, hs[i].bfs_levels,
                        hs[i].max_frontier, hs[i].frontier_sum, hs[i].cycles, hs[i].cyc_gr_init,
                        hs[i].cyc_gr_bfs, hs[i].cyc_gr_snap, hs[i].cyc_front, hs[i].cyc_gr_later);
            fclose(fp);
        }
    }
    GDS_CUDA(cudaEventRecord(c->ev[EV_END], sc.st));
    GDS_CUDA(cudaStreamSynchronize(sc.st));
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
    if (split) out->flow_value -= (int64_t)h.through_flow;
    if (sc.do_solve && !converged) {
        char buf[160];
        snprintf(buf, sizeof buf, "max-flow did not converge: sink inflow %lld, F* %lld, stuck %lld",
                 (long long)out->flow_value, (long long)out->fstar, stuck);
        return fail(c, GDS_ERR_NOCONVERGE, buf);
    }
    return GDS_OK;
}

}  // namespace

extern "C" int gds_solve(gds_ctx* c, const gds_reads* rd, const gds_filter* flt,
                         uint32_t max_coverage, const gds_params* prm, uint32_t flags,
                         gds_result* out) {
    if (!c) return GDS_ERR_ARG;
    c->err.clear();
    SolveCall sc{rd, flt, prm, flags, max_coverage, out, Knobs::read()};
    if (const int rc = check_args(c, sc)) return rc;

    struct ProfGuard {
        ProfGuard(Profiler* p) { cur_prof() = p; }
        ~ProfGuard() { cur_prof() = nullptr; }
    } prof_guard(&c->prof);
    c->prof.on = (flags & GDS_PROFILE_KERNELS) != 0;
    if (!c->prof.on) c->prof.reset();  // profiled calls accumulate until gds_kernel_profile_reset
    const unsigned long long launches0 = launch_counter();
    try {
        GDS_CUDA(cudaSetDevice(c->device));
        sc.st = c->stream;
        GDS_CUDA(cudaEventRecord(c->ev[EV_BEGIN], sc.st));
        upload_inputs(c, sc);
        filter_reads(c, sc);
        read_length_bounds(c, sc);
        sc.plan = plan_segments(rd, prm, sc.base, sc.minlen, sc.maxlen);
        out->seg_len = sc.plan.seg_len;
        plan_solve(sc);
        find_bundles(c, sc);
        build_nodes(c, sc);
        solve_flow(c, sc);
        select_reads(c, sc);
        return finish(c, sc, launches0);
    } catch (const InputFail& f) {
        char buf[160];
        snprintf(buf, sizeof buf, "%u %s", f.count, f.what);
        return fail(c, f.code, buf);
    } catch (const CallFail& f) {
        return fail(c, f.code, f.what);
    } catch (const CudaFail& f) {
        return fail_cuda(c, f);
    } catch (const std::bad_alloc&) {
        return fail(c, GDS_ERR_NOMEM, "host allocation failed");
    }
}
