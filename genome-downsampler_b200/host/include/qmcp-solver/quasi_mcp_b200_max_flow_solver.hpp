// qmcp::QuasiMcpB200MaxFlowSolver — the new algorithm ("quasi-mcp-b200") behind the reference's
// Solver interface.  Host-only translation unit: it talks to the device exclusively through the
// C ABI of include/gds.h (libgds_b200.so).  No CPU fallback: if the library cannot create a
// device context the solver logs and exits like the reference's CUDA helpers do
// (libs/qmcp-solver/include/qmcp-solver/cuda_helpers.cuh:13-21).
#pragma once
#include <cstdint>
#include <memory>
#include <vector>

#include "gds.h"
#include "qmcp-solver/solver.hpp"

namespace qmcp {

class QuasiMcpB200MaxFlowSolver : public Solver {
   public:
    explicit QuasiMcpB200MaxFlowSolver(int device = 0, uint32_t algorithm = 0)
        : device_(device), algorithm_(algorithm) {}
    ~QuasiMcpB200MaxFlowSolver() override;
    std::unique_ptr<Solution> solve(uint32_t max_coverage, bam_api::BamApi& bam_api) override;
    bool uses_quality_of_reads() override { return false; }

    // A batch of independent samples (contigs, runs) in ONE device call: one narrowing loop over all
    // samples fills one pinned staging area on the host threads, gds_solve gets n_samples = size of
    // the batch, and every sample's ascending kept indices come back as its own Solution — what
    // calling solve() on each BamApi in turn returns, minus a device round trip per sample.
    // BamApis with a pending pair filter are solved one by one through solve().
    std::vector<std::unique_ptr<Solution>> solve_batch(uint32_t max_coverage,
                                                       const std::vector<bam_api::BamApi*>& bam_apis);

    // last call's device-side report (flow value, kept count, per-phase milliseconds, ...)
    const gds_result& last_result() const { return last_; }
    void set_verify(bool v) { verify_ = v; }
    // gds_params.seg_len (include/gds.h): references longer than twice this many positions are solved
    // as independent segments — same F*, demand and capped coverage as the reference's network, at
    // most max_coverage extra kept reads per cut (+0.5 % at 50 M reads / 5 Mb).  0xffffffff = never cut
    // (the reference's own network, ~120x slower on a 5 Mb reference); 0 = the library's default.
    // The environment variable GDS_SEG_LEN sets it for a solver that came out of SolverManager.
    void set_segment_length(uint32_t positions) { seg_len_ = positions; }

   private:
    // The device call of solve() and solve_batch(): the samples' size_t columns, laid end to end,
    // are narrowed into the staging buffers and solved in one gds_solve; any failure logs and
    // exits.  `filter` = the BamApi whose pending filter the device applies (one sample only).
    // Leaves the report in last_, the kept bitmap in bitmap_ and, filtered, the pair verdicts in
    // pair_pass_.  Returns the samples' read offsets (n_samples + 1 entries).
    std::vector<uint64_t> solve_on_device(uint32_t max_coverage,
                                          const std::vector<const bam_api::SOAPairedReads*>& samples,
                                          const bam_api::BamApi* filter);

    // grow-only page-locked staging buffer (gds_host_alloc): the narrowing loop writes straight
    // into it and the library copies from it at full PCIe speed
    struct Pinned {
        void* p = nullptr;
        size_t cap = 0;
        template <typename T>
        T* get(size_t n) {
            size_t bytes = (n ? n : 1) * sizeof(T);
            if (bytes > cap) {
                gds_host_free(p);
                p = gds_host_alloc(bytes + bytes / 8);
                cap = p ? bytes + bytes / 8 : 0;
            }
            return static_cast<T*>(p);
        }
        ~Pinned() { gds_host_free(p); }
    };
    Pinned start_, start16_, end_, mapq_, seq_len_, bitmap_, pair_pass_;

    int device_;
    gds_ctx* ctx_ = nullptr;  // created lazily, reused across solve() calls
    gds_result last_{};
    bool verify_ = true;
    uint32_t seg_len_ = 0;
    uint32_t algorithm_ = 0;  // gds_params.algorithm
};

// "mcp-b200": the same adapter with gds_params.algorithm = 1 — the kept set of minimum size (what
// mcp-cpu's min-cost flow with unit read costs returns as its optimal cost,
// mcp_cpu_cost_scaling_solver.cpp:33-67).  Like mcp-cpu it does not look at read qualities.
class McpB200SweepSolver : public QuasiMcpB200MaxFlowSolver {
   public:
    explicit McpB200SweepSolver(int device = 0) : QuasiMcpB200MaxFlowSolver(device, 1) {}
};

}  // namespace qmcp
