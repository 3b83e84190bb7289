// Shared helpers for the tgp_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include <type_traits>
#include "../../../include/tgp_b200.h"

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

// ---- covariance functions ------------------------------------------------------------------------------------------
// k(x, z) = s phi(r), r^2 = d2 = sum_d (x_d / l_d - z_d / l_d)^2 (direct differences), TgpModel.kernel = KIND:
//   RBF         phi = exp(-d2 / 2)                          psi = phi
//   MATERN12    phi = exp(-r)                               psi = exp(-r) / r          (0 for d2 <= 1e-30)
//   MATERN32    phi = (1 + sqrt3 r) exp(-sqrt3 r)           psi = 3 exp(-sqrt3 r)
//   MATERN52    phi = (1 + sqrt5 r + 5 r^2 / 3) exp(-sqrt5 r)   psi = 5/3 (1 + sqrt5 r) exp(-sqrt5 r)
// with psi = -2 dphi / d(d2): the kernel gradients are dk/dz = s psi (x - z) / l^2 and dk/dl = s psi (x - z)^2 / l^3.
// phi(0) = 1 and 0 <= phi <= 1 for every kind.  psi of MATERN12 is singular at r = 0 (a minibatch row on an inducing
// point, the K_zz diagonal): such a pair contributes nothing to the Z / lengthscale gradients, which is what
// sqrt(clamp_min(d2, 1e-30)) yields under autograd.  The other kinds take r = 0 there as well (their psi is smooth).
// Three flavours, one per consumer:
//   phi / phi_psi        FP64 (K tiles, FP64 kernel gradients);
//   kf                   FP64 distance and argument, FP32 exponential exp(a) = expf(a_hi) (1 + a_lo), times s (TF32 planes);
//   phi_psi_f            FP32 throughout (the FP32 kernel-gradient pass of the tensor-core mode).
template <int KIND> struct Cov;

template <> struct Cov<TGP_KERNEL_RBF> {
    static __device__ __forceinline__ double phi(double d2) { return exp(-0.5 * d2); }
    static __device__ __forceinline__ void phi_psi(double d2, double& ph, double& ps) { ph = exp(-0.5 * d2); ps = ph; }
    static __device__ __forceinline__ float kf(double d2, float s) {
        const double arg = -0.5 * d2;
        const float ahi = (float)arg;
        return s * expf(ahi) * (1.0f + (float)(arg - (double)ahi));
    }
    static __device__ __forceinline__ void phi_psi_f(float d2, float& ph, float& ps) { ph = expf(-0.5f * d2); ps = ph; }
};

constexpr double COV_R2_MIN = 1e-30;      // d2 at or below this counts as r = 0
__device__ __forceinline__ double cov_r(double d2) { return d2 > COV_R2_MIN ? sqrt(d2) : 0.0; }
__device__ __forceinline__ float cov_rf(float d2) { return d2 > (float)COV_R2_MIN ? sqrtf(d2) : 0.f; }
__device__ __forceinline__ float exp_split(double a) {      // exp(a) with the argument kept in FP64, to FP32 accuracy
    const float ahi = (float)a;
    return expf(ahi) * (1.0f + (float)(a - (double)ahi));
}

template <> struct Cov<TGP_KERNEL_MATERN12> {
    static __device__ __forceinline__ double phi(double d2) { return exp(-cov_r(d2)); }
    static __device__ __forceinline__ void phi_psi(double d2, double& ph, double& ps) {
        const double r = cov_r(d2);
        ph = exp(-r);
        ps = r > 0.0 ? ph / r : 0.0;
    }
    static __device__ __forceinline__ float kf(double d2, float s) { return s * exp_split(-cov_r(d2)); }
    static __device__ __forceinline__ void phi_psi_f(float d2, float& ph, float& ps) {
        const float r = cov_rf(d2);
        ph = expf(-r);
        ps = r > 0.f ? ph / r : 0.f;
    }
};

template <> struct Cov<TGP_KERNEL_MATERN32> {
    static constexpr double C = 1.7320508075688772;          // sqrt(3)
    static __device__ __forceinline__ double phi(double d2) { const double a = C * cov_r(d2); return (1.0 + a) * exp(-a); }
    static __device__ __forceinline__ void phi_psi(double d2, double& ph, double& ps) {
        const double a = C * cov_r(d2), e = exp(-a);
        ph = (1.0 + a) * e;
        ps = 3.0 * e;
    }
    static __device__ __forceinline__ float kf(double d2, float s) {
        const double a = C * cov_r(d2);
        return s * exp_split(-a) * (float)(1.0 + a);
    }
    static __device__ __forceinline__ void phi_psi_f(float d2, float& ph, float& ps) {
        const float a = (float)C * cov_rf(d2), e = expf(-a);
        ph = (1.f + a) * e;
        ps = 3.f * e;
    }
};

template <> struct Cov<TGP_KERNEL_MATERN52> {
    static constexpr double C = 2.23606797749979;            // sqrt(5)
    static __device__ __forceinline__ double phi(double d2) {
        const double a = C * cov_r(d2);
        return (1.0 + a + a * a / 3.0) * exp(-a);
    }
    static __device__ __forceinline__ void phi_psi(double d2, double& ph, double& ps) {
        const double a = C * cov_r(d2), e = exp(-a);
        ph = (1.0 + a + a * a / 3.0) * e;
        ps = (5.0 / 3.0) * (1.0 + a) * e;
    }
    static __device__ __forceinline__ float kf(double d2, float s) {
        const double a = C * cov_r(d2);
        return s * exp_split(-a) * (float)(1.0 + a + a * a / 3.0);
    }
    static __device__ __forceinline__ void phi_psi_f(float d2, float& ph, float& ps) {
        const float a = (float)C * cov_rf(d2), e = expf(-a);
        ph = (1.f + a + a * a / 3.f) * e;
        ps = (5.f / 3.f) * (1.f + a) * e;
    }
};

inline bool kernel_kind_valid(int kind) { return kind >= TGP_KERNEL_RBF && kind <= TGP_KERNEL_MATERN52; }

// Runs f(std::integral_constant<int, KIND>{}) for the runtime kind: the one place a driver turns TgpModel.kernel into the
// template parameter of its kernels (validate() has rejected unknown kinds before any driver runs)
template <class F> inline int with_kernel(int kind, F&& f) {
    switch (kind) {
        case TGP_KERNEL_MATERN12: return f(std::integral_constant<int, TGP_KERNEL_MATERN12>{});
        case TGP_KERNEL_MATERN32: return f(std::integral_constant<int, TGP_KERNEL_MATERN32>{});
        case TGP_KERNEL_MATERN52: return f(std::integral_constant<int, TGP_KERNEL_MATERN52>{});
        default: return f(std::integral_constant<int, TGP_KERNEL_RBF>{});
    }
}

}  // namespace tgp
