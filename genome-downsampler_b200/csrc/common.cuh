// common.cuh — shared helpers for the sm_100a kernels of libgds_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cstdio>
#include <string>
#include <utility>
#include <vector>

namespace gds {

constexpr uint32_t kLabelInf = 0x3fffffffu;
constexpr int kNumSMs = 148;  // B200

struct CudaFail {
    cudaError_t err;
    const char* what;
    const char* file;
    int line;
};

#define GDS_CUDA(call)                                                   \
    do {                                                                 \
        cudaError_t _e = (call);                                         \
        if (_e != cudaSuccess) throw gds::CudaFail{_e, #call, __FILE__, __LINE__}; \
    } while (0)

// kernels this thread has launched; gds_result.kernel_launches is its growth over one call
inline unsigned long long& launch_counter() {
    static thread_local unsigned long long n = 0;
    return n;
}

// Per-launch accounting.  When profiling is on (GDS_PROFILE_KERNELS), a KScope brackets a launch
// with CUDA events on the launching stream so bench.py can report per-kernel time and achieved
// bytes/s measured live.  launch() opens it and counts the launch.
struct KRec {
    const char* name;
    unsigned long long bytes;
    cudaEvent_t e0, e1;
};
struct Profiler {
    bool on = false;
    std::vector<KRec> recs;
    std::vector<cudaEvent_t> pool;
    size_t used = 0;
    cudaEvent_t ev() {
        if (used == pool.size()) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            pool.push_back(e);
        }
        return pool[used++];
    }
    void reset() {
        recs.clear();
        used = 0;
    }
    void release() {
        for (cudaEvent_t e : pool) cudaEventDestroy(e);
        pool.clear();
    }
};
inline Profiler*& cur_prof() {
    static thread_local Profiler* p = nullptr;
    return p;
}
struct KScope {
    cudaStream_t st;
    cudaEvent_t e1 = nullptr;
    KScope(const char* name, unsigned long long bytes, cudaStream_t s) : st(s) {
        Profiler* p = cur_prof();
        if (!p) return;
        if (p->on) {
            KRec r{name, bytes, p->ev(), p->ev()};
            cudaEventRecord(r.e0, st);
            e1 = r.e1;
            p->recs.push_back(r);
        }
    }
    ~KScope() {
        if (e1) cudaEventRecord(e1, st);
    }
};

// Every kernel launch of the solve path: profiled under `name` with its algorithmic `bytes`, counted
// (gds_result.kernel_launches) and checked.
template <typename... Params, typename... Args>
inline void launch(const char* name, unsigned long long bytes, void (*kernel)(Params...), dim3 grid,
                   dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    KScope ks(name, bytes, st);
    kernel<<<grid, block, smem, st>>>(std::forward<Args>(args)...);
    ++launch_counter();
    GDS_CUDA(cudaGetLastError());
}

// Grow-only device buffer (arena slot).  Reused across gds_solve calls, freed with its owner.
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() {
        if (p) cudaFree(p);
    }
    template <typename T>
    T* get(size_t n) {
        size_t bytes = n * sizeof(T);
        if (bytes == 0) bytes = sizeof(T);
        if (bytes > cap) {
            if (p) cudaFree(p);
            p = nullptr;
            // geometric growth: a context that is re-entered with slowly growing inputs (the
            // reference's tester solves five cases on one instance) must not pay a cudaFree +
            // cudaMalloc — tens of milliseconds with a device synchronisation — on every call
            size_t want = std::max(bytes + bytes / 8 + 256, cap + cap / 2);
            cudaError_t e = cudaMalloc(&p, want);
            if (e != cudaSuccess) {
                cap = 0;
                p = nullptr;
                throw CudaFail{e, "cudaMalloc", __FILE__, __LINE__};
            }
            cap = want;
        }
        return reinterpret_cast<T*>(p);
    }
    template <typename T>
    T* as() const {
        return reinterpret_cast<T*>(p);
    }
};

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ uint32_t lanemask_lt() {
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// Warp-aggregated append: every calling lane with pred==true gets a distinct slot of *counter.
// Must be called by all 32 lanes of the warp (converged).
__device__ __forceinline__ uint32_t warp_agg_slot(bool pred, uint32_t* counter) {
    uint32_t mask = __ballot_sync(0xffffffffu, pred);
    uint32_t base = 0;
    if (mask != 0) {
        int leader = __ffs(mask) - 1;
        if ((int)lane_id() == leader) base = atomicAdd(counter, __popc(mask));
        base = __shfl_sync(0xffffffffu, base, leader);
    }
    return base + __popc(mask & lanemask_lt());
}

// streaming loads that do not pollute L1 (inputs are read once)
__device__ __forceinline__ uint32_t ld_stream(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint4 ld_stream4(const uint4* p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p));
    return v;
}

inline int div_up(long long a, long long b) { return (int)((a + b - 1) / b); }
inline int bits_for(uint64_t max_value) {  // bits needed to represent values 0..max_value
    int b = 0;
    while (max_value) {
        ++b;
        max_value >>= 1;
    }
    return b;
}

}  // namespace gds
