// Adapter: qmcp::Solver::solve(max_coverage, BamApi&) -> C ABI (include/gds.h) -> ascending
// kept indices.  Narrowing size_t -> uint32 happens once, here, with range checks.
#include "qmcp-solver/quasi_mcp_b200_max_flow_solver.hpp"

#include <algorithm>
#include <cstdlib>
#include <limits>
#include <thread>
#include <vector>

#include "logging/log.hpp"

namespace qmcp {

namespace {
// The narrowing loop reads the reference's size_t columns once (32 bytes per read): at 50 M reads
// that is 1.6 GB of host memory traffic, a multiple of the device time when one thread does it.
// fn(begin, end, chunk) runs on up to kMaxThreads threads over disjoint index ranges.
constexpr unsigned kMaxThreads = 16;
template <typename F>
void parallel_chunks(uint64_t n, unsigned& n_chunks, F fn) {
    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    n_chunks = n < (1u << 18) ? 1u : std::min<unsigned>({hw, kMaxThreads, (unsigned)(n >> 16)});
    if (n_chunks <= 1) {
        n_chunks = 1;
        fn(uint64_t{0}, n, 0u);
        return;
    }
    // chunk boundaries on multiples of 64 reads: no two threads share a cache line of an output
    const uint64_t per = ((n + n_chunks - 1) / n_chunks + 63) & ~uint64_t{63};
    std::vector<std::thread> th;
    for (unsigned c = 0; c < n_chunks; ++c) {
        const uint64_t b = std::min<uint64_t>(n, (uint64_t)c * per), e = std::min<uint64_t>(n, b + per);
        th.emplace_back([=, &fn] { fn(b, e, c); });
    }
    for (auto& t : th) t.join();
}
}  // namespace

// kept indices are written as the library's uint64_t
static_assert(sizeof(bam_api::ReadIndex) == sizeof(uint64_t), "ReadIndex must be 64-bit");

QuasiMcpB200MaxFlowSolver::~QuasiMcpB200MaxFlowSolver() {
    if (ctx_) gds_destroy(ctx_);
}

std::vector<uint64_t> QuasiMcpB200MaxFlowSolver::solve_on_device(
    uint32_t max_coverage, const std::vector<const bam_api::SOAPairedReads*>& samples,
    const bam_api::BamApi* filter) {
    if (!ctx_ && gds_create(device_, &ctx_) != GDS_OK) {
        LOG_WITH_LEVEL(logging::ERROR)
            << "quasi-mcp-b200: no usable CUDA device " << device_ << " (there is no CPU fallback)";
        std::exit(EXIT_FAILURE);
    }
    const uint32_t ns = static_cast<uint32_t>(samples.size());
    constexpr uint64_t kMax32 = std::numeric_limits<uint32_t>::max();
    std::vector<uint64_t> off(ns + 1, 0);
    std::vector<uint32_t> ref_len(ns);
    // compact transport (gds_reads.start16): references of up to 65536 positions fit 16-bit
    // starts; the column is written by the same narrowing loop
    bool narrow16 = true;
    for (uint32_t k = 0; k < ns; ++k) {
        const uint64_t L = samples[k]->ref_genome_length;
        off[k + 1] = off[k] + samples[k]->get_reads_count();
        // the library takes fewer than 2^32 - 64 reads in one call
        if (L > kMax32 - 4 || off[k + 1] > kMax32 - 64) {
            LOG_WITH_LEVEL(logging::ERROR) << "quasi-mcp-b200: input beyond 32-bit device limits";
            std::exit(EXIT_FAILURE);
        }
        ref_len[k] = static_cast<uint32_t>(L);
        narrow16 &= L <= 65536;
    }
    const uint64_t n = off[ns];
    uint32_t* start = start_.get<uint32_t>(n);
    uint32_t* end = end_.get<uint32_t>(n);
    uint16_t* start16 = narrow16 ? start16_.get<uint16_t>(n) : nullptr;
    uint32_t* seq_len = filter ? seq_len_.get<uint32_t>(n) : nullptr;
    uint8_t* mapq = filter ? mapq_.get<uint8_t>(n) : nullptr;
    uint8_t* pair_pass = filter ? pair_pass_.get<uint8_t>(n / 2 + 1) : nullptr;
    uint32_t* bitmap = bitmap_.get<uint32_t>((n + 31) / 32 + 1);
    if (!start || !end || (narrow16 && !start16) || (filter && (!seq_len || !mapq || !pair_pass)) ||
        !bitmap) {
        LOG_WITH_LEVEL(logging::ERROR) << "quasi-mcp-b200: cannot allocate pinned staging buffers";
        std::exit(EXIT_FAILURE);
    }
    // the narrowing loop also yields the exact read-length bounds the library can use to fold its
    // input validation into the first sort pass (gds_reads.len_min / len_max)
    struct Part {
        uint32_t len_min = 0xffffffffu, len_max = 0;
        bool lens_ok = true;
        bool fits16 = true;  // a start beyond 16 bits is an input error the device has to see as such
    };
    Part parts[kMaxThreads];
    unsigned n_chunks = 1;
    parallel_chunks(n, n_chunks, [&](uint64_t b, uint64_t e, unsigned c) {
        Part p;
        // a chunk may begin inside a sample: the last sample that starts at or before b
        size_t k = std::upper_bound(off.begin(), off.end(), b) - off.begin() - 1;
        for (uint64_t i = b; i < e; ++k) {
            const bam_api::SOAPairedReads& in = *samples[k];
            const uint64_t o = off[k], stop = std::min(e, off[k + 1]);
            for (; i < stop; ++i) {
                const uint64_t s64 = in.start_inds[i - o];
                const uint32_t s = static_cast<uint32_t>(s64);
                const uint32_t t = static_cast<uint32_t>(std::min<uint64_t>(in.end_inds[i - o], kMax32));
                start[i] = s;
                end[i] = t;
                if (narrow16) {
                    p.fits16 &= s64 <= 0xffff;
                    start16[i] = static_cast<uint16_t>(s64);
                }
                if (t < s) {
                    p.lens_ok = false;  // the library reports it as GDS_ERR_RANGE
                } else {
                    p.len_min = std::min(p.len_min, t - s + 1);
                    p.len_max = std::max(p.len_max, t - s + 1);
                }
                if (filter) {
                    seq_len[i] = in.seq_lengths[i - o];
                    mapq[i] = static_cast<uint8_t>(std::min<uint32_t>(in.qualities[i - o], 255));
                }
            }
        }
        parts[c] = p;
    });
    uint32_t len_min = 0xffffffffu, len_max = 0;
    bool lens_ok = n > 0, fits16 = true;
    for (unsigned c = 0; c < n_chunks; ++c) {
        len_min = std::min(len_min, parts[c].len_min);
        len_max = std::max(len_max, parts[c].len_max);
        lens_ok &= parts[c].lens_ok;
        fits16 &= parts[c].fits16;
    }
    gds_reads rd{ns, off.data(), ref_len.data(), start, end, mapq, seq_len,
                 lens_ok ? len_min : 0, lens_ok ? len_max : 0, nullptr};
    // fixed-length reads (reads-gen, most short-read runs): the end column is implied; with
    // 16-bit starts a read crosses PCIe as 2 bytes instead of 8.
    if (lens_ok && len_min == len_max) {
        rd.end = nullptr;
        if (narrow16 && fits16) {
            rd.start16 = start16;
            rd.start = nullptr;
        }
    }
    gds_filter flt{};
    std::vector<uint32_t> amp_s, amp_e;
    if (filter) {
        flt.min_seq_length = filter->min_seq_length();
        flt.min_mapq = std::min<uint32_t>(filter->min_mapq(), 256);  // > 255 can never pass anyway
        if (filter->amplicon_behaviour() == bam_api::AmpliconBehaviour::FILTER) {
            for (const auto& a : filter->amplicon_set().amplicons) {
                amp_s.push_back(static_cast<uint32_t>(std::min<uint64_t>(a.start, kMax32)));
                amp_e.push_back(static_cast<uint32_t>(std::min<uint64_t>(a.end, kMax32)));
            }
            if (amp_s.empty()) {  // FILTER with an empty set drops every pair (any_of over nothing)
                amp_s.push_back(1);
                amp_e.push_back(0);
            }
            flt.n_amplicons = static_cast<uint32_t>(amp_s.size());
            flt.amp_start = amp_s.data();
            flt.amp_end = amp_e.data();
        }
    }
    last_ = gds_result{};
    last_.kept_bitmap = bitmap;
    last_.pair_pass = pair_pass;
    gds_params prm{};  // zero = the library's defaults
    prm.seg_len = seg_len_;
    prm.algorithm = algorithm_;
    if (const char* e = std::getenv("GDS_SEG_LEN")) prm.seg_len = static_cast<uint32_t>(std::strtoul(e, nullptr, 0));
    int rc = gds_solve(ctx_, &rd, filter ? &flt : nullptr, max_coverage, &prm,
                       verify_ ? GDS_VERIFY : 0, &last_);
    last_.kept_bitmap = nullptr;
    last_.pair_pass = nullptr;
    if (rc != GDS_OK) {
        LOG_WITH_LEVEL(logging::ERROR) << "quasi-mcp-b200: " << gds_last_error(ctx_);
        std::exit(EXIT_FAILURE);
    }
    if (verify_ && last_.verify_violations != 0) {
        LOG_WITH_LEVEL(logging::ERROR) << "quasi-mcp-b200: device verification found "
                                       << last_.verify_violations << " bad positions";
        std::exit(EXIT_FAILURE);
    }
    return off;
}

std::unique_ptr<Solution> QuasiMcpB200MaxFlowSolver::solve(uint32_t max_coverage,
                                                           bam_api::BamApi& bam_api) {
    const bool device_filter = bam_api.has_pending_filter();
    const bam_api::SOAPairedReads& in =
        device_filter ? bam_api.unfiltered_soa() : bam_api.get_paired_reads_soa();
    const uint64_t n = solve_on_device(max_coverage, {&in}, device_filter ? &bam_api : nullptr)[1];
    if (device_filter) {  // BamApi now holds the post-filter arrays
        const uint8_t* pair_pass = static_cast<const uint8_t*>(pair_pass_.p);
        bam_api.apply_pair_filter(std::vector<uint8_t>(pair_pass, pair_pass + n / 2));
    }
    auto sol = std::make_unique<Solution>(last_.n_kept);
    uint64_t k = gds_bitmap_to_indices(static_cast<const uint32_t*>(bitmap_.p), last_.n_filtered,
                                       reinterpret_cast<uint64_t*>(sol->data()), sol->size());
    sol->resize(std::min<uint64_t>(k, sol->size()));
    LOG_WITH_LEVEL(logging::DEBUG) << "quasi-mcp-b200: F*=" << last_.fstar << " kept=" << last_.n_kept
                                   << " rounds=" << last_.rounds_total << " device ms=" << last_.ms_total;
    return sol;
}

std::vector<std::unique_ptr<Solution>> QuasiMcpB200MaxFlowSolver::solve_batch(
    uint32_t max_coverage, const std::vector<bam_api::BamApi*>& bam_apis) {
    std::vector<std::unique_ptr<Solution>> out(bam_apis.size());
    bool plain = !bam_apis.empty();
    for (auto* a : bam_apis) plain &= a != nullptr && !a->has_pending_filter();
    if (!plain) {  // the device filter rewrites each BamApi: keep the one-by-one path for it
        for (size_t k = 0; k < bam_apis.size(); ++k) out[k] = solve(max_coverage, *bam_apis[k]);
        return out;
    }
    const uint32_t ns = static_cast<uint32_t>(bam_apis.size());
    std::vector<const bam_api::SOAPairedReads*> soa(ns);
    for (uint32_t k = 0; k < ns; ++k) soa[k] = &bam_apis[k]->get_paired_reads_soa();
    const std::vector<uint64_t> off = solve_on_device(max_coverage, soa, nullptr);
    const uint32_t* bitmap = static_cast<const uint32_t*>(bitmap_.p);
    // per-sample ascending indices: samples on the host threads, bits walked in place (sample
    // boundaries need not be word-aligned)
    auto expand = [&](uint32_t k) {
        auto sol = std::make_unique<Solution>();
        const uint64_t b = off[k], e = off[k + 1];
        uint64_t cnt = 0;
        for (uint64_t w = b / 32; w <= (e ? (e - 1) / 32 : 0) && b < e; ++w) {
            uint32_t x = bitmap[w];
            if (w == b / 32) x &= ~0u << (b % 32);
            if (w == (e - 1) / 32 && (e % 32)) x &= (1u << (e % 32)) - 1u;
            cnt += __builtin_popcount(x);
        }
        sol->reserve(cnt);
        for (uint64_t w = b / 32; w <= (e ? (e - 1) / 32 : 0) && b < e; ++w) {
            uint32_t x = bitmap[w];
            if (w == b / 32) x &= ~0u << (b % 32);
            if (w == (e - 1) / 32 && (e % 32)) x &= (1u << (e % 32)) - 1u;
            while (x) {
                sol->push_back(w * 32 + __builtin_ctz(x) - b);
                x &= x - 1;
            }
        }
        out[k] = std::move(sol);
    };
    const unsigned nt = std::min<unsigned>({std::max(1u, std::thread::hardware_concurrency()), 32u, ns});
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nt; ++t)
        th.emplace_back([&, t] {
            for (uint32_t k = t; k < ns; k += nt) expand(k);
        });
    for (auto& t : th) t.join();
    return out;
}

}  // namespace qmcp
