// kernel_harness.cu — test-only entry points into the production kernels of scan.cuh,
// radix_sort.cuh and select.cuh (included unchanged), loaded by tests/test_kernels.py with ctypes.
//
// Every wrapper takes host arrays, runs the kernels on the default stream, copies the results back
// and returns the CUDA status (0 = success).  Every device buffer a wrapper allocates lies between
// kGuardBytes of guard words on either side, filled with a known pattern; *intact reports whether
// all of them (and any padding in front of a misaligned array) still hold it afterwards.  This is
// how the tests catch out-of-bounds writes without a memory checker.
#include "../../genome-downsampler_b200/csrc/radix_sort.cuh"
#include "../../genome-downsampler_b200/csrc/scan.cuh"
#include "../../genome-downsampler_b200/csrc/select.cuh"

#include <cstring>
#include <vector>

using namespace gds;

namespace {

constexpr size_t kGuardBytes = 256;  // keeps an array without offset 256-byte aligned

// One device array of `len` bytes, `pad` bytes past the end of the front guard, between guards.
struct GuardBuf {
    unsigned char* d = nullptr;
    size_t lo = 0, len = 0, total = 0;
    std::vector<unsigned char> pat;
    GuardBuf() = default;
    GuardBuf(const GuardBuf&) = delete;
    GuardBuf& operator=(const GuardBuf&) = delete;
    ~GuardBuf() {
        if (d) cudaFree(d);
    }
    void init(size_t len_bytes, size_t pad = 0) {
        lo = kGuardBytes + pad;
        len = len_bytes;
        total = lo + len + kGuardBytes;
        pat.resize(total);
        uint32_t x = 0x9e3779b9u ^ (uint32_t)total;
        for (size_t i = 0; i < total; ++i) {
            x = x * 1664525u + 1013904223u;
            pat[i] = (unsigned char)(x >> 24);
        }
        GDS_CUDA(cudaMalloc(&d, total));
        GDS_CUDA(cudaMemcpy(d, pat.data(), total, cudaMemcpyHostToDevice));
    }
    template <typename T>
    T* ptr() const {
        return reinterpret_cast<T*>(d + lo);
    }
    void upload(const void* h) {
        if (len) GDS_CUDA(cudaMemcpy(d + lo, h, len, cudaMemcpyHostToDevice));
    }
    void download(void* h) const {
        if (len) GDS_CUDA(cudaMemcpy(h, d + lo, len, cudaMemcpyDeviceToHost));
    }
    bool intact() const {
        std::vector<unsigned char> now(total);
        GDS_CUDA(cudaMemcpy(now.data(), d, total, cudaMemcpyDeviceToHost));
        return !memcmp(now.data(), pat.data(), lo) &&
               !memcmp(now.data() + lo + len, pat.data() + lo + len, total - lo - len);
    }
};

// Runs body(); returns the CUDA status: the first failed call, else whatever the kernels left.
template <typename F>
int run(F&& body) {
    try {
        body();
        GDS_CUDA(cudaDeviceSynchronize());
        return (int)cudaGetLastError();
    } catch (const CudaFail& f) {
        return (int)f.err;
    }
}

template <typename K>
int sort_pairs(const K* keys, const uint64_t* group_size, uint32_t n_groups, int bits,
               int atomic_rank, K* keys_out, uint32_t* vals_out, int* passes, int* intact) {
    *intact = 0;
    return run([&] {
        size_t n = 0;
        for (uint32_t g = 0; g < n_groups; ++g) n += group_size[g];
        GuardBuf ka, kb, va, vb, toff_b, ioff_b;
        ka.init(n * sizeof(K));
        kb.init(n * sizeof(K));
        va.init(n * 4);
        vb.init(n * 4);
        ka.upload(keys);
        // the segmented map exactly as sort_bundles (gds_api.cu) builds it; one group is the
        // plain map there
        TileMap tm{nullptr, nullptr, 1, tiles_for(n), n};
        if (n_groups > 1) {
            std::vector<uint32_t> toff(n_groups + 1, 0);
            std::vector<uint64_t> ioff(n_groups + 1, 0);
            for (uint32_t k = 0; k < n_groups; ++k) {
                toff[k + 1] = toff[k] + tiles_for(group_size[k]);
                ioff[k + 1] = ioff[k] + group_size[k];
            }
            toff_b.init(toff.size() * 4);
            ioff_b.init(ioff.size() * 8);
            toff_b.upload(toff.data());
            ioff_b.upload(ioff.data());
            tm = TileMap{toff_b.ptr<uint32_t>(), ioff_b.ptr<uint64_t>(), n_groups, toff[n_groups], n};
        }
        RadixTemp tmp;
        const int where = radix_sort_pairs<K>(ka.ptr<K>(), va.ptr<uint32_t>(), kb.ptr<K>(),
                                              vb.ptr<uint32_t>(), tm, bits, tmp, 0, atomic_rank != 0,
                                              passes);
        GDS_CUDA(cudaDeviceSynchronize());
        (where ? kb : ka).download(keys_out);
        (where ? vb : va).download(vals_out);
        bool ok = ka.intact() && kb.intact() && va.intact() && vb.intact();
        if (n_groups > 1) ok = ok && toff_b.intact() && ioff_b.intact();
        *intact = ok;
    });
}

}  // namespace

extern "C" {

// ---- look-back scan: a ScanTemp the caller keeps across calls (status words, epoch)
void* kh_scan_temp_new() { return new ScanTemp(); }
void kh_scan_temp_free(void* t) { delete static_cast<ScanTemp*>(t); }
uint32_t kh_scan_temp_epoch(void* t) { return static_cast<ScanTemp*>(t)->epoch; }

// exclusive_scan_u32_multi over n_arr (1-3) arrays of n elements (in/out: n_arr x n, row-major).
// Array k is read from `in_off` and written at `out_off` elements past a 256-byte-aligned address;
// in_place scans each array in its own buffer (in_off is used).  epoch >= 0 sets the ScanTemp's
// epoch before the call.
int kh_scan(void* t, const uint32_t* in, uint32_t* out, int n_arr, uint64_t n, uint32_t in_off,
            uint32_t out_off, int in_place, long long epoch, int* intact) {
    *intact = 0;
    ScanTemp& tmp = *static_cast<ScanTemp*>(t);
    return run([&] {
        GuardBuf bi[3], bo[3];
        ScanArrays a{{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};
        for (int k = 0; k < n_arr; ++k) {
            bi[k].init(n * 4, 4ull * in_off);
            bi[k].upload(in + (size_t)k * n);
            a.in[k] = bi[k].ptr<uint32_t>();
            if (in_place) {
                a.out[k] = bi[k].ptr<uint32_t>();
            } else {
                bo[k].init(n * 4, 4ull * out_off);
                a.out[k] = bo[k].ptr<uint32_t>();
            }
        }
        if (epoch >= 0) tmp.epoch = (uint32_t)epoch;
        exclusive_scan_u32_multi(a, n_arr, n, tmp, 0);
        GDS_CUDA(cudaDeviceSynchronize());
        bool ok = true;
        for (int k = 0; k < n_arr; ++k) {
            (in_place ? bi[k] : bo[k]).download(out + (size_t)k * n);
            ok = ok && bi[k].intact() && (in_place || bo[k].intact());
        }
        *intact = ok;
    });
}

// ---- radix_sort_pairs on the groups [group_size[0], group_size[1], ...] (one group: the plain
// tile map).  Values start as the item index; the sorted keys and values come back.
int kh_sort_u32(const uint32_t* keys, const uint64_t* group_size, uint32_t n_groups, int bits,
                int atomic_rank, uint32_t* keys_out, uint32_t* vals_out, int* passes, int* intact) {
    return sort_pairs<uint32_t>(keys, group_size, n_groups, bits, atomic_rank, keys_out, vals_out,
                                passes, intact);
}
int kh_sort_u64(const unsigned long long* keys, const uint64_t* group_size, uint32_t n_groups,
                int bits, int atomic_rank, unsigned long long* keys_out, uint32_t* vals_out,
                int* passes, int* intact) {
    return sort_pairs<unsigned long long>(keys, group_size, n_groups, bits, atomic_rank, keys_out,
                                          vals_out, passes, intact);
}

// ---- K5: k_select on B bundles (first slot in sorted_idx, flow) into a cleared bitmap of n_words
int kh_select(const uint32_t* b_first, const uint32_t* flow, uint32_t B, const uint32_t* sorted_idx,
              uint64_t n_sorted, uint64_t n_words, uint32_t* bitmap_out, unsigned long long* n_kept,
              int* intact) {
    *intact = 0;
    return run([&] {
        std::vector<BundleRec> recs(B);
        for (uint32_t b = 0; b < B; ++b) recs[b] = BundleRec{0u, flow[b], flow[b], 0u};
        GuardBuf fb, bb, sb, bm, tb;
        fb.init(B * 4ull);
        bb.init(B * sizeof(BundleRec));
        sb.init(n_sorted * 4);
        bm.init(n_words * 4);
        tb.init(3 * sizeof(unsigned long long));
        fb.upload(b_first);
        bb.upload(recs.data());
        sb.upload(sorted_idx);
        GDS_CUDA(cudaMemset(bm.ptr<uint32_t>(), 0, n_words * 4));
        GDS_CUDA(cudaMemset(tb.ptr<unsigned long long>(), 0, 3 * sizeof(unsigned long long)));
        if (B)
            launch("select", 0, k_select, div_up(B, 256), 256, 0, 0, fb.ptr<uint32_t>(),
                   bb.ptr<BundleRec>(), sb.ptr<uint32_t>(), B, bm.ptr<uint32_t>(),
                   tb.ptr<unsigned long long>());
        GDS_CUDA(cudaDeviceSynchronize());
        unsigned long long tot[3];
        tb.download(tot);
        *n_kept = tot[1];
        bm.download(bitmap_out);
        *intact = fb.intact() && bb.intact() && sb.intact() && bm.intact() && tb.intact();
    });
}

// ---- k_find_pairs on a bitmap of n_words, in place
int kh_find_pairs(uint32_t* bitmap, uint64_t n_words, int* intact) {
    *intact = 0;
    return run([&] {
        GuardBuf bm;
        bm.init(n_words * 4);
        bm.upload(bitmap);
        if (n_words)
            launch("find_pairs", 0, k_find_pairs, div_up(n_words, 256), 256, 0, 0, bm.ptr<uint32_t>(),
                   (size_t)n_words);
        GDS_CUDA(cudaDeviceSynchronize());
        bm.download(bitmap);
        *intact = bm.intact();
    });
}

// ---- K6 on n reads of n_samples samples (read_off[n_samples+1], ref_len[n_samples]) and a kept
// bitmap of (n+31)/32 words.  The input side, diff_in and its exclusive scan excl_in over the
// n_onodes + 1 nodes of the batch (sample k owns ref_len[k] + 1 nodes), comes from the caller.  The
// kept side is computed by the production sequence of select_reads (gds_api.cu:1512-1522):
// k_verify_accumulate, exclusive_scan_u32, k_verify_compare.
int kh_verify(const uint32_t* bitmap, const uint32_t* S, const uint32_t* E, uint64_t n,
              const uint64_t* read_off, const uint32_t* ref_len, uint32_t n_samples,
              const int32_t* diff_in, const uint32_t* excl_in, uint32_t M,
              unsigned long long* violations, int* intact) {
    *intact = 0;
    return run([&] {
        std::vector<uint32_t> base(n_samples + 1, 0);
        for (uint32_t k = 0; k < n_samples; ++k) base[k + 1] = base[k] + ref_len[k] + 1;
        const uint32_t n_onodes = base[n_samples];
        const size_t n_words = (n + 31) / 32;
        GuardBuf bm, sb, eb, ob, bb, di, xi, vdiff, vexcl, tb;
        bm.init(n_words * 4);
        sb.init(n * 4);
        eb.init(n * 4);
        ob.init((n_samples + 1) * 8ull);
        bb.init((n_samples + 1) * 4ull);
        di.init((n_onodes + 1) * 4ull);
        xi.init((n_onodes + 1) * 4ull);
        vdiff.init((n_onodes + 1) * 4ull);
        vexcl.init((n_onodes + 1) * 4ull);
        tb.init(3 * sizeof(unsigned long long));
        bm.upload(bitmap);
        sb.upload(S);
        eb.upload(E);
        ob.upload(read_off);
        bb.upload(base.data());
        di.upload(diff_in);
        xi.upload(excl_in);
        GDS_CUDA(cudaMemset(tb.ptr<unsigned long long>(), 0, 3 * sizeof(unsigned long long)));
        ScanTemp scan;
        int32_t* vd = vdiff.ptr<int32_t>();
        uint32_t* vx = vexcl.ptr<uint32_t>();
        GDS_CUDA(cudaMemsetAsync(vd, 0, ((size_t)n_onodes + 1) * 4, 0));
        if (n_words)
            launch("verify_accumulate", 0, k_verify_accumulate, div_up(n_words, 256), 256, 0, 0,
                   bm.ptr<uint32_t>(), sb.ptr<uint32_t>(), eb.ptr<uint32_t>(), (size_t)n,
                   ob.ptr<uint64_t>(), bb.ptr<uint32_t>(), n_samples, vd);
        exclusive_scan_u32(reinterpret_cast<const uint32_t*>(vd), vx, (size_t)n_onodes + 1, scan, 0);
        launch("verify_compare", 0, k_verify_compare, div_up(n_onodes, 256), 256, 0, 0, vx, vd,
               xi.ptr<uint32_t>(), di.ptr<int32_t>(), n_onodes, M, tb.ptr<unsigned long long>());
        GDS_CUDA(cudaDeviceSynchronize());
        unsigned long long tot[3];
        tb.download(tot);
        *violations = tot[2];
        *intact = bm.intact() && sb.intact() && eb.intact() && ob.intact() && bb.intact() &&
                  di.intact() && xi.intact() && vdiff.intact() && vexcl.intact() && tb.intact();
    });
}

}  // extern "C"
