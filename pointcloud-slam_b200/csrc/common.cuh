// b200reg — shared device/host helpers.  sm_100a only; compiled with -fmad=false so every
// fp32 op is a separately rounded IEEE op (the reference is built without FMA,
// jueying_lio/CMakeLists.txt:10-11, and neighbour sets must be bit-exact).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <cstdio>
#include <cstdlib>
#include <atomic>
#include <cstring>
#include <string>

#include "../../include/b200reg.h"

namespace b200 {

extern thread_local std::string g_last_error;
extern std::atomic<int64_t> g_kernel_launches;  // counted by every launch site (bench.py "gpu_launches"); handles may live on different threads

inline int32_t fail(int32_t code, const char* what, const char* file, int line) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s (%s:%d)", what, file, line);
    g_last_error = buf;
    return code;
}
#define B200_FAIL(code, what) return ::b200::fail((code), (what), __FILE__, __LINE__)
#define CUDA_TRY(expr)                                                                   \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) return ::b200::fail(B200_ERR_CUDA, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)
#define LAUNCH_COUNT(n) (::b200::g_kernel_launches.fetch_add((n), std::memory_order_relaxed))
// Entry of a public call: select the handle's device and drop a stale "last error" left behind by an earlier, unrelated
// runtime call in this process (ours or anybody else's), so that it is not mistaken for a failure of this call.
inline void drop_stale_error(const char* file, int line) {
    const cudaError_t e = cudaGetLastError();
    static const bool dbg = getenv("B200_DEBUG") != nullptr;
    if (e != cudaSuccess && dbg) fprintf(stderr, "[b200reg] stale CUDA error dropped at %s:%d: %s\n", file, line, cudaGetErrorString(e));
}
#define CUDA_SET_DEVICE(dev)                              \
    do {                                                  \
        ::b200::drop_stale_error(__FILE__, __LINE__);     \
        CUDA_TRY(cudaSetDevice(dev));                     \
    } while (0)

// ---- programmatic dependent launch (PDL): a kernel launched with the attribute may start while its predecessor on the
// stream is still draining; pdl_wait() blocks until the predecessor grid has completed and its writes are visible (a
// no-op when the kernel was launched normally), pdl_trigger() lets the successor's blocks be scheduled early.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
inline bool pdl_enabled() {
    static const bool on = !(getenv("B200_PDL") && atoi(getenv("B200_PDL")) == 0);
    return on;
}
template <class... Params, class... Args>
inline cudaError_t launch_k(void (*kernel)(Params...), dim3 grid, dim3 block, cudaStream_t stream, bool pdl, Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = 0;
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = (pdl && pdl_enabled()) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<Params>(args)...);
}

template <class T>
struct DevBuf {  // grow-only device buffer
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        size_t ncap = n + n / 4 + 64;
        T* q = nullptr;
        cudaError_t e = cudaMalloc(&q, ncap * sizeof(T));
        if (e != cudaSuccess) return e;
        if (p) cudaFree(p);
        p = q;
        cap = ncap;
        return cudaSuccess;
    }
    // grow but keep the first `keep` elements
    cudaError_t reserve_keep(size_t n, size_t keep, cudaStream_t s, bool exact = false) {
        if (n <= cap) return cudaSuccess;
        size_t ncap = exact ? n : n + n / 2 + 64;
        T* q = nullptr;
        cudaError_t e = cudaMalloc(&q, ncap * sizeof(T));
        if (e != cudaSuccess) return e;
        if (p && keep) {
            e = cudaMemcpyAsync(q, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, s);
            if (e != cudaSuccess) return e;
            cudaStreamSynchronize(s);
        }
        if (p) cudaFree(p);
        p = q;
        cap = ncap;
        return cudaSuccess;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

template <class T>
struct PinnedBuf {
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        size_t ncap = n + n / 4 + 64;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cudaError_t e = cudaMallocHost(&p, ncap * sizeof(T));
        cap = e == cudaSuccess ? ncap : 0;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

// ---- voxel keys: three 21-bit biased cell coordinates packed into 63 bits ----------------
constexpr int kKeyBias = 1 << 20;
constexpr uint64_t kEmptyKey = 0xFFFFFFFFFFFFFFFFull;
__host__ __device__ inline bool cell_in_range(int x, int y, int z) {
    return (unsigned)(x + kKeyBias) < (1u << 21) && (unsigned)(y + kKeyBias) < (1u << 21) && (unsigned)(z + kKeyBias) < (1u << 21);
}
__host__ __device__ inline uint64_t pack_key(int x, int y, int z) {
    return ((uint64_t)(uint32_t)(x + kKeyBias) << 42) | ((uint64_t)(uint32_t)(y + kKeyBias) << 21) | (uint64_t)(uint32_t)(z + kKeyBias);
}
// Table placement with 2 x 2 x 2-voxel locality: the eight voxels of an aligned 2x2x2 block hash to ONE 128-byte line of the
// table (8 entries of 16 bytes, position inside the line = the low bit of each cell coordinate), so the 27 probes of a
// stencil search touch the lines of at most 8 blocks instead of 27 scattered 32-byte sectors, and z-neighbours share a
// sector.  A collision steps 9 slots on: to the next line and the next position inside it, so a probe sequence visits
// every slot of the table (9 is odd) even when all voxels share coordinate parities (a flat floor fills only half of
// the in-line positions).
__host__ __device__ inline uint32_t hash_key(uint64_t k) {  // 32-bit multiply-xorshift mix of the block key, times 8, plus the in-block index
    const uint32_t lo = (uint32_t)k, hi = (uint32_t)(k >> 32);
    const uint32_t idx = ((hi >> 10) & 1u) << 2 | ((lo >> 21) & 1u) << 1 | (lo & 1u);  // low bits of x (bit 42), y (bit 21), z (bit 0)
    uint32_t h = (lo & ~0x00200001u) * 0x9E3779B1u ^ (hi & ~0x00000400u) * 0x85EBCA77u;
    h ^= h >> 15;
    h *= 0x2C1B3C6Du;
    h ^= h >> 13;
    return (h << 3) | idx;
}
__host__ __device__ inline uint32_t next_slot(uint32_t slot, uint32_t tmask) { return (slot + 9u) & tmask; }

// Pass a strided host cloud through a pinned staging buffer as packed float4 (x,y,z,0).
inline void pack_xyz_float4(const float* xyz, int64_t n, int64_t stride, float4* dst) {
    const char* src = (const char*)xyz;
    for (int64_t i = 0; i < n; ++i) {
        const float* p = (const float*)(src + i * stride);
        dst[i] = make_float4(p[0], p[1], p[2], 0.0f);
    }
}

}  // namespace b200
