// Shared helpers for the tgp_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>

#define TGP_WARP 32

namespace tgp {

// last error text, returned by tgp_last_error()
extern char g_last_error[512];

inline int set_error(int code, const char* msg) {
    snprintf(g_last_error, sizeof(g_last_error), "%s", msg);
    return code;
}

extern long g_launch_count;      // kernels launched by this library (tgp_launch_count())

inline int check_launch(const char* what) {
    ++g_launch_count;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(g_last_error, sizeof(g_last_error), "%s: %s", what, cudaGetErrorString(e));
        return -100;
    }
    return 0;
}

#define TGP_TRY(expr) do { int _rc = (expr); if (_rc != 0) return _rc; } while (0)

// Concurrency of the per-step factorisation with K_xz generation.  tgp_prepare is a chain of ~80 small, mostly single-CTA
// kernels (1.2-1.4 ms at M = 1024) that leaves the GPU almost idle; K_xz generation of the coming forward needs only the
// transformed parameters.  With TGP_OPT_OVERLAP_KGEN (default) tgp_prepare forks: the factorisation runs on a library-owned
// HIGHEST-priority stream (its short kernels are dispatched ahead of the K_xz tiles), the caller's stream continues;
// tgp_qf_forward enqueues K_xz generation on the caller's stream and only then joins.  Every other consumer of the step
// workspace joins first (join_factor).  The 4-byte pivot status is copied to pinned host memory on the factorisation's
// stream; tgp_factor_status() blocks the host on that copy alone.  Host objects only — no device memory is allocated.
struct SideStream {
    cudaStream_t hp = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_factor = nullptr, ev_status = nullptr;
    int* status_host = nullptr;
    bool pending = false;        // a factorisation is in flight on `hp` and the consumer stream has not joined yet
    bool status_valid = false;   // ev_status was recorded outside graph capture
};
inline SideStream& side_stream() {
    static SideStream s[64];
    int dev = 0;
    cudaGetDevice(&dev);
    SideStream& x = s[dev >= 0 && dev < 64 ? dev : 0];
    if (!x.hp) {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        cudaStreamCreateWithPriority(&x.hp, cudaStreamNonBlocking, hi);
        cudaEventCreateWithFlags(&x.ev_fork, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&x.ev_factor, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&x.ev_status, cudaEventDisableTiming);
        cudaHostAlloc(reinterpret_cast<void**>(&x.status_host), sizeof(int), cudaHostAllocDefault);
    }
    return x;
}
inline bool stream_is_capturing(cudaStream_t st) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { cudaGetLastError(); return false; }
    return cs != cudaStreamCaptureStatusNone;
}
// the consumer stream waits for the factorisation in flight (no-op when there is none)
inline int join_factor(cudaStream_t st) {
    SideStream& ss = side_stream();
    if (ss.pending) {
        ss.pending = false;
        if (cudaStreamWaitEvent(st, ss.ev_factor, 0) != cudaSuccess) return -100;
    }
    return 0;
}
extern int g_overlap_kgen;       // TGP_OPT_OVERLAP_KGEN

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <typename T>
__device__ __forceinline__ T warp_max(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__host__ __device__ inline long cdiv(long a, long b) { return (a + b - 1) / b; }

// Carves typed views out of a caller-owned workspace in declaration order, each starting on a 256-byte ABSOLUTE address
// (callers of the staged entry points may pass any alignment; cp.async, vector loads and TMA need 16 bytes).  With a NULL
// base it only measures: `used` starts at 256, so bytes() covers a carve of the same pieces from a base of any alignment.
// Every workspace size the library reports is bytes() of the layout function that the entry points carve with.
struct Carve {
    char* base;
    size_t used;
    explicit Carve(void* b) : base(static_cast<char*>(b)), used(b ? 0 : 256) {}
    template <class T> T* take(size_t n) {
        const uintptr_t b = reinterpret_cast<uintptr_t>(base), at = (b + used + 255) & ~uintptr_t(255);
        used = at - b + n * sizeof(T);
        return reinterpret_cast<T*>(at);
    }
    size_t bytes() const { return used; }
};

// cudaFuncSetAttribute is per DEVICE: one-time kernel configuration is tracked per (site, device), so that a second GPU
// used from the same process gets its own opt-in to large dynamic shared memory.
struct PerDeviceOnce {
    bool done[64] = {};
    bool first() {
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev < 0 || dev >= 64) return true;
        if (done[dev]) return false;
        done[dev] = true;
        return true;
    }
};

// softplus and its derivative as torch.nn.functional.softplus (beta=1, threshold=20) evaluates them
__device__ __forceinline__ double softplus_d(double x) { return x > 20.0 ? x : log1p(exp(x)); }
__device__ __forceinline__ double sigmoid_d(double x) { return x > 20.0 ? 1.0 : 1.0 / (1.0 + exp(-x)); }

}  // namespace tgp
