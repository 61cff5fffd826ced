/*
 * gds.h — C ABI of the B200-native quasi-MCP downsampler (libgds_b200.so).
 *
 * This is the drop-in boundary for ONE path of migoox/genome-downsampler: what a
 * qmcp::Solver::solve(max_coverage, BamApi&) implementation
 * (libs/qmcp-solver/include/qmcp-solver/solver.hpp:15-20) needs from the device:
 *   filter -> coverage/demand -> flow graph -> max-flow -> read selection.
 * Plain pointers and sizes only; no C++ or torch types cross it.  Every entry point cites the
 * reference interface it replaces.  There is NO CPU fallback: every call fails with
 * GDS_ERR_CUDA when no sm_100 device / driver is usable.
 *
 * Index conventions are the reference's: positions are 0-based inclusive [start, end]
 * (libs/bam-api/include/bam-api/read.hpp:19-30), mates are adjacent (first at even index,
 * libs/bam-api/src/bam_api.cpp:456-461), returned read indices refer to the POST-FILTER arrays
 * (what BamApi::get_paired_reads_soa() would hold, bam_api.cpp:212-233).
 */
#ifndef GDS_H
#define GDS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GDS_ABI_VERSION 7

/* status codes (the reference has none: it logs and exits, cuda_helpers.cuh:13-21) */
enum {
    GDS_OK = 0,
    GDS_ERR_ARG = 1,       /* null pointer, odd read count with a filter, bad sizes */
    GDS_ERR_RANGE = 2,     /* end >= ref_len, start > end, L or N beyond 32-bit device limits */
    GDS_ERR_CUDA = 3,      /* CUDA runtime error (message in gds_last_error) */
    GDS_ERR_NOMEM = 4,     /* device allocation failed */
    GDS_ERR_NOCONVERGE = 5 /* max_rounds hit or sink inflow != F* (never on valid input) */
};

/* flags for gds_solve */
enum {
    GDS_INPUT_ON_DEVICE = 1u << 0,  /* start/end/mapq/seq_len are device pointers */
    GDS_OUTPUT_ON_DEVICE = 1u << 1, /* kept_bitmap/pair_pass/cov/demand are device pointers */
    GDS_VERIFY = 1u << 2,           /* recompute coverage of the kept set on device and compare */
    GDS_FIND_PAIRS = 1u << 3,       /* also OR each kept read's mate into the bitmap
                                       (BamApi::find_pairs, bam_api.cpp:239-273).  The mate of read i
                                       is i ^ 1 inside its sample, so every read_off must be even
                                       (GDS_ERR_ARG otherwise).  The reference looks at is_first_read
                                       (id + 1 or id - 1): the same thing whenever the first mate sits
                                       at the even index, which is how BamApi lays pairs out
                                       (bam_api.cpp:456-461).  gds_result.n_kept stays the number of
                                       reads the flow selected, before their mates are added. */
    GDS_NO_SOLVE = 1u << 4,         /* stop after coverage/demand/graph (K1+K2 only) */
    GDS_PROFILE_KERNELS = 1u << 5   /* bracket every kernel with CUDA events (gds_kernel_profile) */
};

typedef struct gds_ctx gds_ctx;

/* Input reads.  Replaces bam_api::SOAPairedReads (soa_paired_reads.hpp:18-24) narrowed to
 * 32-bit; a batch is n_samples independent samples/contigs concatenated.  read_off and ref_len
 * are always HOST arrays. */
typedef struct {
    uint32_t n_samples;       /* >= 1 */
    const uint64_t* read_off; /* [n_samples+1], read_off[0] = 0 */
    const uint32_t* ref_len;  /* [n_samples]  PairedReads::ref_genome_length */
    const uint32_t* start;    /* [n_reads]    Read::start_ind (ignored when start16 is given) */
    const uint32_t* end;      /* [n_reads]    Read::end_ind (inclusive); NULL = every read has
                                 length len_min == len_max (fixed-length reads: end = start+len-1) */
    const uint8_t* mapq;      /* [n_reads]    Read::quality (MAPQ); NULL if no filter */
    const uint32_t* seq_len;  /* [n_reads]    Read::seq_length (l_qseq); NULL if no filter */
    /* optional: exact bounds of end-start+1 over all reads (0,0 = unknown).  A caller that
     * narrows the reference's size_t arrays anyway has them for free; with them the device folds
     * input validation into the first pass of the sort instead of a separate pass over the
     * reads.  Reads outside the bounds fail the call with GDS_ERR_ARG.  The bounds have to be the
     * exact minimum and maximum: the default segment length of a long reference depends on whether
     * all reads have one length (gds_params.seg_len), so looser bounds may select another — equally
     * valid — kept set than a call without them. */
    uint32_t len_min, len_max;
    /* optional compact transport of the start column: 16-bit starts (every ref_len <= 65536).
     * With fixed-length reads (end == NULL) a read then crosses PCIe as 2 bytes instead of 8; the
     * device widens the columns again before anything else runs.  Same pointer kind (host or
     * device) as start/end. */
    const uint16_t* start16;
} gds_reads;

/* Pre-filter.  Replaces BamApi::should_be_filtered_out (bam_api.cpp:311-332) and the amplicon
 * table built by set_amplicon_filter (bam_api.cpp:53-95).  n_amplicons == 0 means
 * AmpliconBehaviour::IGNORE; otherwise FILTER.  Amplicon bounds are inclusive (amplicon.cpp:5-7).
 * Host arrays. */
typedef struct {
    uint32_t min_seq_length; /* -l, BamApiConfig::min_seq_length */
    uint32_t min_mapq;       /* -q, BamApiConfig::min_mapq */
    uint32_t n_amplicons;
    const uint32_t* amp_start;
    const uint32_t* amp_end;
} gds_filter;

/* Deterministic schedule knobs (DESIGN.md §4).  Zero-initialised = defaults (64, 150, 1, 0),
 * seg_len 0, bundle_mode 0.  seg_len: a reference longer than 2*seg_len positions is cut into
 * independent segments of seg_len positions (reads crossing a cut are truncated into one arc per
 * segment and kept if either part carries flow) — the zero-coverage split generalised;
 * 0xffffffff = never cut.  Shorter segments mean fewer dependent max-flow rounds per component and
 * at most max_coverage extra kept reads per cut (config 4: +0.5 % reads, K3 2.4x faster than
 * 32768).  0 = the default rule: 16384, stretched in steps of 128 by up to a quarter when that
 * brings the number of segments of the whole batch down to 296 — two resident components per SM of
 * a B200, so that no second wave of a few left-over segments runs (config 4: 5 Mb -> 296 segments
 * of 16896 instead of 306), then rounded up to a whole number of reads when all reads have one
 * length (16950 = 113 x 150: 295 segments).  The rule is a constant of the schedule, not a device
 * query: the same input gives the same kept set on every device.  gds_result.seg_len reports the
 * value used. */
typedef struct {
    uint32_t gr_interval_min;
    uint32_t gr_levels_pct;
    uint32_t gr_relabel_pct;
    uint32_t max_rounds;
    uint32_t seg_len;
    /* how K2 finds the bundles (reads with one (start, length) key): 0 = choose, 1 = always the
     * segmented radix sort, 2 = a sort-free histogram whenever one is eligible: counters in shared
     * memory (one read length, no sample segmented, ref_len + 1 <= 49152 per sample, 16-byte
     * aligned start/end) or else in global memory (virtual nodes x #read-lengths <= 24 Mi).  All
     * three give the same graph and the same kept set; gds_result.bundle_path tells which one ran. */
    uint32_t bundle_mode;
    /* which solve runs on the graph:
     *   0  quasi-MCP — maximum flow by push-relabel (quasi_mcp_cpu_max_flow_solver.cpp:11-100);
     *   1  minimum cardinality — the objective of `mcp-cpu` (mcp_cpu_cost_scaling_solver.cpp:33-67:
     *      the same network with cost 1 on every read arc), solved exactly by the greedy interval
     *      multicover sweep (csrc/sweep.cuh).  Same F*, demand vector and capped coverage; the kept
     *      set is the smallest one (per segment, when a long reference is cut).  Reads of up to 4095
     *      positions.  rounds / pushes / relabels stay 0. */
    uint32_t algorithm;
    /* graph reduction and push-relabel schedule of algorithm 0 (csrc/graph.cuh, csrc/maxflow_sm.cuh,
     * DESIGN.md §4; the oracle replays all three: orc_sync_params.schedule):
     *   0  from max_coverage = 128 on: (a) FORCED READS OUT, CUTS IN — a read that covers a position
     *      with coverage <= max_coverage is in every valid answer, so its flow is fixed and it leaves
     *      the network, and the back arc over such a position carries nothing in any valid answer, so
     *      the components are cut there (the zero-coverage rule with "<= max_coverage" for "== 0");
     *      (b) the EXPRESS schedule for components with a supply of 128 or more that fit one SM: back
     *      arcs have length 0 in the distance labels, flow changes read "lanes" within one round.
     *      The reference's hole / low-sides / zero-sides shapes at M = 8000: 2 100-4 300 rounds ->
     *      155-430, 13-19 ms -> 1.1-2.4 ms; config 4: 370 -> 175 rounds per segment.
     *      Below 128 (configs 1, 5: M = 100) the graph and the schedule are round 1's — except
     *      in a call that carries an amplicon table (gds_filter.n_amplicons > 0: amplicon-tiled
     *      coverage dips between the amplicons), which gets (a) at every max_coverage, like 3;
     *   1  round 1's graph and classic schedule always;
     *   2  (a) and (b) whatever max_coverage and the supply are (experiments);
     *   3  (a) at every max_coverage, (b) by the usual rule.  Worth asking for when the coverage
     *      dips below a SMALL max_coverage in many places and the batch is not huge (config 2 —
     *      amplicon tiling, M = 100: 6.1 -> 3.6 ms; the three extra passes over nodes and bundles
     *      cost config 5's 15 M nodes 0.25 ms, which is why 0 does not do it below 128).
     * Every choice is a function of the data and these fields alone, never of the device or the
     * batch a sample travels in. */
    uint32_t schedule;
} gds_params;

/* Results.  Buffers are caller-owned and optional (NULL = not wanted). */
typedef struct {
    /* ---- buffers ---- */
    uint32_t* kept_bitmap;   /* [ceil(n_filtered/32)] bit i = post-filter read i kept
                                (quasi_mcp_cpu_max_flow_solver.cpp:89-100) */
    uint8_t* pair_pass;      /* [n_reads/2] 1 = pair survived the filter */
    uint64_t* filt_off;      /* [n_samples+1] HOST: post-filter read offsets per sample */
    uint32_t* cov_capped;    /* [n_nodes] min(cov, M) of the position right of each node */
    int32_t* demand;         /* [n_nodes] create_demand_function (…cpu_max_flow_solver.cpp:75-87) */
    /* ---- scalars ---- */
    uint64_t n_reads_in, n_filtered, n_kept, n_bundles;
    uint64_t n_arc_items;    /* sorted arc items = n_filtered + reads cut in two by a segment cut */
    uint32_t n_nodes, n_components;
    int64_t fstar;           /* closed form: sum of source capacities */
    int64_t flow_value;      /* value of the flow found, on the original network (== fstar) */
    uint64_t rounds_total, rounds_max, pushes, relabels, global_relabels, bfs_levels, max_frontier;
    uint64_t verify_violations; /* GDS_VERIFY: positions with min(cov_out,M) != min(cov_in,M) */
    uint32_t key_bits, sort_passes;
    uint64_t kernel_launches; /* kernels this call launched (counted at the launch sites) */
    /* direct (histogram) path, K5: bundles with 0 < flow < multiplicity and the reads that carry
     * their keys (ranked by index; every other kept read belongs to a saturated bundle) */
    uint64_t partial_bundles, partial_candidates;
    uint32_t bundle_path; /* how K2 found the bundles: 0 radix sort, 1 histogram in shared memory,
                             2 histogram in global memory (gds_params.bundle_mode) */
    uint32_t seg_len;     /* the segment length this call used (gds_params.seg_len or the default rule) */
    /* device-event milliseconds per phase */
    float ms_h2d, ms_filter, ms_graph, ms_maxflow, ms_select, ms_verify, ms_d2h, ms_total;
} gds_result;

/* lifecycle: one context per host thread / per GPU; device arenas grow-only and are reused
 * across calls (the reference re-enters one solver instance 5x, coverage_tester.cpp:28-43) */
int gds_create(int device, gds_ctx** out);
void gds_destroy(gds_ctx* ctx);
const char* gds_last_error(const gds_ctx* ctx);
int gds_abi_version(void);
/* run all work on this cudaStream_t (as void*); NULL = the context's own stream */
int gds_set_stream(gds_ctx* ctx, void* cuda_stream);

/* Page-locked host memory for staging buffers (a host-only caller needs no CUDA headers):
 * gds_solve copies from/to pinned buffers at full PCIe speed, pageable ones take a bounce copy.
 * The reference's CUDA solver copies from pageable std::vector (cuda_helpers.cuh:33-48). */
void* gds_host_alloc(size_t bytes);
void gds_host_free(void* p);

/* The whole hot path.  Replaces QuasiMcpCpuMaxFlowSolver::solve
 * (quasi_mcp_cpu_max_flow_solver.cpp:11-28) and QuasiMcpCudaMaxFlowSolver::solve
 * (quasi_mcp_cuda_max_flow_solver.cu:319-435) plus the filter of BamApi::read_bam. */
int gds_solve(gds_ctx* ctx, const gds_reads* reads, const gds_filter* filter /* NULL = none */,
              uint32_t max_coverage, const gds_params* params /* NULL = defaults */,
              uint32_t flags, gds_result* out);

/* Per-kernel device time of the gds_solve calls that ran with GDS_PROFILE_KERNELS since the last
 * gds_kernel_profile_reset (a call without the flag also resets), aggregated by kernel name: CUDA-event milliseconds, launches, and the algorithmic bytes (once-through reads +
 * writes) those launches had to move.  Returns the number of distinct kernels. */
typedef struct {
    char name[32];
    float ms;
    uint32_t launches;
    uint64_t bytes;
} gds_kernel_stat;
uint32_t gds_kernel_profile(gds_ctx* ctx, gds_kernel_stat* out, uint32_t cap);
void gds_kernel_profile_reset(gds_ctx* ctx);

/* Expand a HOST bitmap into ascending indices (qmcp::Solution order).  Returns count. */
uint64_t gds_bitmap_to_indices(const uint32_t* bitmap, uint64_t n_bits, uint64_t* indices,
                               uint64_t cap);

#ifdef __cplusplus
}
#endif
#endif
