// Shared helpers for libp2s_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <stdexcept>
#include <atomic>
#include <memory>
#include <utility>
#include <vector>

#include "../../include/p2s_b200.h"

namespace p2s {

extern thread_local std::string g_last_error;
extern std::atomic<uint64_t> g_launches;

struct Error : std::runtime_error {
    using std::runtime_error::runtime_error;
};

#define P2S_CUDA(call)                                                                             \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            char _buf[512];                                                                        \
            snprintf(_buf, sizeof(_buf), "%s:%d: %s failed: %s", __FILE__, __LINE__, #call,       \
                     cudaGetErrorString(_e));                                                      \
            throw ::p2s::Error(_buf);                                                              \
        }                                                                                          \
    } while (0)

#define P2S_CHECK(cond, msg)                                                                       \
    do {                                                                                           \
        if (!(cond)) {                                                                             \
            char _buf[512];                                                                        \
            snprintf(_buf, sizeof(_buf), "%s:%d: check failed (%s): %s", __FILE__, __LINE__,      \
                     #cond, msg);                                                                  \
            throw ::p2s::Error(_buf);                                                              \
        }                                                                                          \
    } while (0)

// every kernel launch goes through this so that p2s_launch_count() is honest
#define P2S_LAUNCH(kernel, grid, block, smem, stream, ...)                                         \
    do {                                                                                           \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);                                \
        ::p2s::g_launches.fetch_add(1, std::memory_order_relaxed);                                 \
        P2S_CUDA(cudaGetLastError());                                                              \
    } while (0)

template <class F>
static inline int guarded(F&& f) {
    try {
        f();
        return 0;
    } catch (const std::exception& e) {
        g_last_error = e.what();
        return 1;
    }
}

static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Optional coarse stage timing (env P2S_STAGE_TIMING=1): synchronises the stream around every stage and
// accumulates host wall-clock per label; printed by p2s_model_destroy.  Diagnostics only.
struct StageTimer {
    static bool enabled();
    static void add(const char* label, double ms);
    static void report();
};
struct StageScope {
    const char* label; cudaStream_t st; double t0 = 0.0; bool on;
    StageScope(const char* l, cudaStream_t s);
    ~StageScope();
};

// grow-only device scratch buffer
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    void* get(size_t need) {
        if (need > bytes) {
            if (p) P2S_CUDA(cudaFree(p));
            p = nullptr;
            size_t want = need + need / 8;
            P2S_CUDA(cudaMalloc(&p, want));
            bytes = want;
        }
        return p;
    }
    template <class T>
    T* as(size_t count) { return reinterpret_cast<T*>(get(count * sizeof(T))); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
};

// Cell index of a cloud for the weighted sub-sampler (assemble.cu): device pointers into DeviceCtx::cloud_ws
struct CloudIndex {
    const float* meta;      // [6] bounding-box low corner, cells per unit length
    const float* spts;      // [N,3] points in cell order
    const int32_t* perm;    // [N]   original id of sorted point i
    const int32_t* start;   // [C+1] first sorted point of each cell
    const float* cbox;      // [C,6] tight bounding box of each cell's points
};

// Host-side state of the library for one CUDA device, one context per calling thread and device (device_ctx()).
// Device memory and kernel attributes belong to one device, so a launcher takes them from the context of the device it
// launches on; per thread, so that two threads never share scratch.  Two streams of one thread do share it: calls that
// use the same scratch on two streams must be ordered by the caller.
struct DeviceCtx {
    int device = 0;
    int sm_count = 0;
    int* err_flag = nullptr;                      // device int: selection failure of kNN / ball query / sub-sample
    int knn_slots_small = 0, knn_slots_big = 0;   // co-resident CTAs of the two kNN kernels (0 = not yet queried)
    DevBuf grid_ws;                               // candidate grid (grid.cu)
    DevBuf vol_ws;                                // sign propagation (volume.cu)
    DevBuf mc_ws;                                 // marching cubes (mc.cu)
    DevBuf mesh_area, mesh_cum, mesh_cub, mesh_best, mesh_red;   // mesh sampling and metric (meshdist.cu)
    DevBuf cloud_ws;                              // cell index of the last cloud (assemble.cu) ...
    CloudIndex cloud_index{};                     // ... and its pointers, valid until the next cloud_index_build
    DevBuf train_wimg, train_zero_bias;           // weight image and 4096 zeros of the training GEMMs (fc_tc.cu)
    DevBuf wait_stats;                            // P2S_TC_WAITSTATS counters (net_tc.cu)
    std::vector<std::pair<const void*, int>> smem_limits;   // dynamic shared-memory limits raised so far

    // raises the dynamic shared-memory limit of kernel `fn` to `bytes` unless this device already allows that much
    void set_max_dynamic_smem(const void* fn, int bytes);
};
// the context of the calling thread's current CUDA device, created on first use
DeviceCtx& device_ctx();

// ---- Philox4x32-10 (Salmon et al. 2011), counter-based: (key, counter) -> 4 x u32 ----
__host__ __device__ inline void philox4x32_10(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1,
                                              uint32_t c2, uint32_t c3, uint32_t out[4]) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
        uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

}  // namespace p2s
