// Input-dependent flow parameters (ID_TGP): the small MLPs  x_n -> theta(x_n)  evaluated on the device, with MC-dropout.
//
// Reference: code/dsp/models/flow.py:853-871 builds, per flow parameter, nn.Sequential(apply_linear(in, H, act, drop=p) x
// num_H, apply_linear(H, 1, 'linear')) and :949-950 evaluates them once per call on X (MB, D); dropout stays ACTIVE in
// training (sparse_MF_SP.py:133-134).  apply_linear comes from the un-vendored pytorchlib; layer order
// Linear -> activation -> Dropout is the documented assumption (SURVEY.md §8c).
//
// One warp per row, hidden units over the lanes (H <= 64), the weights of the current net in shared memory.
// Dropout: keep-mask m in {0,1}, output a * m / (1 - p)  (torch.nn.Dropout semantics).  Three mask modes:
//   0  no dropout (eval / p = 0);
//   1  Philox-4x32-10 counter RNG keyed by (seed; row, net, layer, unit block, call offset) — the mask is EXPORTED so that
//      the backward (and a parity harness) sees exactly the mask of the forward;
//   2  explicit mask supplied by the caller (parity mode: the reference's masks come from torch's global RNG and cannot
//      be regenerated, SURVEY.md §7.7).
// The backward recomputes the forward of each row, then back-propagates analytically; weight gradients are accumulated
// per CTA in shared memory (FP64 shared atomics) and flushed with one global atomic per weight per CTA.  Input gradients
// (dX, optional, k_flow_mlp<true, true>) are added per row by the warp that owns the row.
#pragma once
#include "common.cuh"
#include "../../../include/tgp_b200.h"

namespace tgp {

constexpr int MLP_MAX_H = 64, MLP_MAX_LAYERS = 4, MLP_WARPS = 8, MLP_THREADS = 32 * MLP_WARPS;

struct MlpArgs {
    int n_nets, n_in, H, L, act, mask_mode;
    double p_drop;
    long R;
    const double* W;            // n_nets x net_size
    const double* X;            // R x n_in
    const unsigned char* mask_in;   // (n_nets, L, R, H) keep flags (mode 2; backward: the forward's mask for modes 1, 2)
    unsigned char* mask_out;        // forward, mode 1 (required) / mode 2 (optional copy)
    unsigned long long seed;
    const unsigned long long* offset_dev;
    double* out;                // forward: R x n_nets
    const double* dout;         // backward: R x n_nets
    double* dW;                 // backward: n_nets x net_size, accumulated
    double* dX;                 // backward: R x n_in, accumulated; NULL = not computed
};

__host__ __device__ inline int mlp_net_size(int n_in, int H, int L) { return H * n_in + H + (L - 1) * (H * H + H) + H + 1; }
__host__ __device__ inline int mlp_layer_off(int n_in, int H, int l) { return l == 0 ? 0 : H * n_in + H + (l - 1) * (H * H + H); }

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                              uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// keep flag of hidden unit h of (row, net, layer): one Philox block serves four consecutive units
__device__ __forceinline__ bool philox_keep(unsigned long long seed, unsigned long long offset, long row, int net, int layer,
                                            int h, double p) {
    uint32_t r[4];
    philox4x32_10((uint32_t)row, (uint32_t)((unsigned long long)row >> 32) ^ ((uint32_t)(net * MLP_MAX_LAYERS + layer) << 8) ^ (uint32_t)(h >> 2),
                  (uint32_t)offset, (uint32_t)(offset >> 32), (uint32_t)seed, (uint32_t)(seed >> 32), r);
    return (double)r[h & 3] * 2.3283064365386963e-10 >= p;          // P(keep) = 1 - p
}

__device__ __forceinline__ double mlp_act(int act, double z, double& dz) {
    if (act == 0) { dz = z > 0.0 ? 1.0 : 0.0; return z > 0.0 ? z : 0.0; }          // relu
    if (act == 1) { const double t = tanh(z); dz = 1.0 - t * t; return t; }          // tanh
    if (act == 2) { const double s = 1.0 / (1.0 + exp(-z)); dz = s * (1.0 - s); return s; }   // sigmoid
    dz = 1.0; return z;                                                              // linear
}

// DX (backward only): also the input gradients, in an instantiation of its own, so that the forward and the plain backward
// compile exactly as without it
template <bool BWD, bool DX = false>
__global__ void __launch_bounds__(MLP_THREADS) k_flow_mlp(MlpArgs a) {
    extern __shared__ double sm_mlp[];
    const int nsz = mlp_net_size(a.n_in, a.H, a.L);
    double* w = sm_mlp;                               // [nsz]
    double* gw = w + nsz;                             // [nsz] (backward only)
    double* scratch = BWD ? gw + nsz : w + nsz;       // per warp: xs[64], act[L][64], dfac[L][64], dz[2][64]
    const int per_warp = 64 * (1 + 2 * MLP_MAX_LAYERS + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* xs = scratch + warp * per_warp;
    double* actv = xs + 64;
    double* dfac = actv + 64 * MLP_MAX_LAYERS;
    double* dzb = dfac + 64 * MLP_MAX_LAYERS;
    const int H = a.H, L = a.L, nin = a.n_in;
    const double inv_keep = a.mask_mode != 0 ? 1.0 / (1.0 - a.p_drop) : 1.0;
    const unsigned long long offset = (a.mask_mode == 1 && a.offset_dev) ? a.offset_dev[0] : 0ull;
    const int wo_off = mlp_layer_off(nin, H, L), bo_off = wo_off + H;

    for (int net = 0; net < a.n_nets; ++net) {
        __syncthreads();
        for (int i = threadIdx.x; i < nsz; i += MLP_THREADS) { w[i] = a.W[(long)net * nsz + i]; if (BWD) gw[i] = 0.0; }
        __syncthreads();
        for (long row = (long)blockIdx.x * MLP_WARPS + warp; row < a.R; row += (long)gridDim.x * MLP_WARPS) {
            for (int d = lane; d < nin; d += 32) xs[d] = a.X[row * nin + d];
            __syncwarp();
            // ---- forward ----
            for (int l = 0; l < L; ++l) {
                const int np = l == 0 ? nin : H;
                const double* inp = l == 0 ? xs : actv + 64 * (l - 1);
                const double* Wl = w + mlp_layer_off(nin, H, l);
                const double* bl = Wl + H * np;
                for (int h = lane; h < H; h += 32) {
                    double z = bl[h];
                    for (int k = 0; k < np; ++k) z = fma(Wl[h * np + k], inp[k], z);
                    double dz;
                    const double av = mlp_act(a.act, z, dz);
                    bool keep = true;
                    const long midx = (((long)net * L + l) * a.R + row) * H + h;
                    if (a.mask_mode == 1 && !BWD) keep = philox_keep(a.seed, offset, row, net, l, h, a.p_drop);
                    else if (a.mask_mode != 0) keep = a.mask_in[midx] != 0;
                    if (!BWD && a.mask_out && a.mask_mode != 0) a.mask_out[midx] = keep ? 1 : 0;
                    actv[64 * l + h] = keep ? av * inv_keep : 0.0;
                    dfac[64 * l + h] = keep ? dz * inv_keep : 0.0;
                }
                __syncwarp();
            }
            const double* last = actv + 64 * (L - 1);
            double o = 0.0;
            for (int h = lane; h < H; h += 32) o = fma(w[wo_off + h], last[h], o);
            o = warp_sum(o) + w[bo_off];
            if (!BWD) {
                if (lane == 0) a.out[row * a.n_nets + net] = o;
                continue;
            }
            // ---- backward ----
            const double g = a.dout[row * a.n_nets + net];
            for (int h = lane; h < H; h += 32) {
                atomicAdd(&gw[wo_off + h], g * last[h]);
                dzb[h] = g * w[wo_off + h] * dfac[64 * (L - 1) + h];
            }
            if (lane == 0) atomicAdd(&gw[bo_off], g);
            __syncwarp();
            int cur = 0;
            for (int l = L - 1; l >= 0; --l) {
                const int np = l == 0 ? nin : H;
                const double* inp = l == 0 ? xs : actv + 64 * (l - 1);
                const int off = mlp_layer_off(nin, H, l);
                const double* dz = dzb + 64 * cur;
                for (int h = lane; h < H; h += 32) {
                    const double d = dz[h];
                    atomicAdd(&gw[off + H * np + h], d);
                    for (int k = 0; k < np; ++k) atomicAdd(&gw[off + h * np + k], d * inp[k]);
                }
                if (l > 0) {
                    double* nz = dzb + 64 * (cur ^ 1);
                    for (int k = lane; k < H; k += 32) {
                        double s = 0.0;
                        for (int h = 0; h < H; ++h) s = fma(w[off + h * np + k], dz[h], s);
                        nz[k] = s * dfac[64 * (l - 1) + k];
                    }
                    cur ^= 1;
                }
                __syncwarp();
            }
            if constexpr (DX) {     // dX[row] += W_0^T dz_0: a row belongs to one warp for every net, so no atomics
                const double* dz0 = dzb + 64 * cur;
                for (int k = lane; k < nin; k += 32) {
                    double s = 0.0;
#pragma unroll 1
                    for (int h = 0; h < H; ++h) s = fma(w[h * nin + k], dz0[h], s);
                    a.dX[row * nin + k] += s;
                }
            }
        }
        if (BWD) {
            __syncthreads();
            for (int i = threadIdx.x; i < nsz; i += MLP_THREADS) {
                const double v = gw[i];
                if (v != 0.0) atomicAdd(a.dW + (long)net * nsz + i, v);
            }
        }
    }
}

__global__ void k_bump_offset(unsigned long long* c) { c[0] += 1; }

inline int mlp_validate(const TgpMlp* m) {
    if (!m) return set_error(-1, "mlp description is NULL");
    if (m->n_nets < 1 || m->n_in < 1 || m->n_in > MLP_MAX_H) return set_error(-1, "flow MLP: n_nets >= 1 and 1 <= n_in <= 64 required");
    if (m->hidden < 1 || m->hidden > MLP_MAX_H) return set_error(-1, "flow MLP: hidden width must be in 1..64");
    if (m->n_hidden_layers < 1 || m->n_hidden_layers > MLP_MAX_LAYERS) return set_error(-1, "flow MLP: 1..4 hidden layers");
    if (m->activation < 0 || m->activation > 3) return set_error(-1, "flow MLP: unknown activation");
    if (m->mask_mode < 0 || m->mask_mode > 2) return set_error(-1, "flow MLP: mask_mode must be 0, 1 or 2");
    if (m->mask_mode != 0 && !(m->p_drop >= 0.0 && m->p_drop < 1.0)) return set_error(-1, "flow MLP: dropout p must be in [0, 1)");
    return 0;
}

inline int launch_flow_mlp(const TgpMlp* m, MlpArgs a, bool bwd, cudaStream_t st) {
    const int nsz = mlp_net_size(m->n_in, m->hidden, m->n_hidden_layers);
    const size_t smem = ((size_t)nsz * (bwd ? 2 : 1) + (size_t)MLP_WARPS * 64 * (1 + 2 * MLP_MAX_LAYERS + 2)) * sizeof(double);
    if (smem > 200 * 1024) return set_error(-2, "flow MLP too large for shared memory");
    static PerDeviceOnce once_f, once_b, once_dx;
    if (bwd && a.dX) { if (once_dx.first()) cudaFuncSetAttribute(k_flow_mlp<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); }
    else if (bwd) { if (once_b.first()) cudaFuncSetAttribute(k_flow_mlp<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); }
    else { if (once_f.first()) cudaFuncSetAttribute(k_flow_mlp<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); }
    long blocks = cdiv(a.R, MLP_WARPS);
    if (blocks > 148 * 2) blocks = 148 * 2;
    if (blocks < 1) blocks = 1;
    if (bwd && a.dX) k_flow_mlp<true, true><<<(unsigned)blocks, MLP_THREADS, smem, st>>>(a);
    else if (bwd) k_flow_mlp<true><<<(unsigned)blocks, MLP_THREADS, smem, st>>>(a);
    else k_flow_mlp<false><<<(unsigned)blocks, MLP_THREADS, smem, st>>>(a);
    return check_launch("k_flow_mlp");
}

}  // namespace tgp
