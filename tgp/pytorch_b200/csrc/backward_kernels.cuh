// Backward-side kernels (FP64): upstream row gradients -> operand of the data/weight-gradient GEMMs, kernel-matrix
// derivatives w.r.t. Z / lengthscale / outputscale (K tiles recomputed on the fly), final raw-parameter gradients.
// Mathematics: SURVEY.md Appendix B (derived from sparse_MF_SP.py:352-382 and autograd through them).
#pragma once
#include <type_traits>
#include "common.cuh"

namespace tgp {

// [A | B] (ld 2M): B -> Bbar = 2 g_v*B in place, A is kept; Abar[n,j] (ld M) = g_mu*m - 2 g_v*A; accumulates
// dm[j] += sum_n g_mu[n]*A[n,j] and (block column 0) dos += sum_n g_v[n]   (K_xx diag = outputscale).
constexpr int ABB_ROWS = 64, ABB_COLS = 128;
__global__ void __launch_bounds__(ABB_COLS) k_make_abbar(double* __restrict__ AB, double* __restrict__ Abar,
                                                         const double* __restrict__ g_mu, const double* __restrict__ g_v,
                                                         const double* __restrict__ m, long R, int M,
                                                         double* __restrict__ dm, double* __restrict__ dos) {
    const int j = blockIdx.x * ABB_COLS + threadIdx.x;
    const long n0 = (long)blockIdx.y * ABB_ROWS, n1 = min(n0 + ABB_ROWS, R);
    const double mj = j < M ? m[j] : 0.0;
    double acc = 0.0, accv = 0.0;
    for (long n = n0; n < n1; ++n) {
        const double gm = g_mu[n], gv = g_v[n];
        accv += gv;
        if (j < M) {
            double* row = AB + n * 2 * M;
            const double a = row[j], b = row[M + j];
            acc = fma(gm, a, acc);
            Abar[n * M + j] = gm * mj - 2.0 * gv * a;
            row[M + j] = 2.0 * gv * b;
        }
    }
    if (j < M) atomicAdd(dm + j, acc);
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(dos, accv);
}

// Accumulates, for t[n,j] = Kbar[n,j] * os * psi(x_n, z_j) (psi: Cov<KIND>, common.cuh; psi = phi for the RBF):
//   dZ[j,d]  += zscale * sum_n t * (xs[n,d] - zs[j,d]) / ls[d]
//   dls[d]   += sum_{n,j} t * (xs[n,d] - zs[j,d])^2 / ls[d]
//   dos      += sum_{n,j} Kbar[n,j] * k(x_n, z_j) / os
// sym = 1 reads Kbar symmetrised, 0.5*(Kbar[n,j] + Kbar[j,n]) (the K_zz case, where X = Zs and R = M).
// 256 rows per CTA: every CTA ends with one FP64 atomic per (column, dimension), so taller CTAs mean fewer
// same-address atomics on dZ (128 row-blocks per 8192-row chunk serialised on each address with 64-row CTAs)
constexpr int KG_TC = 64, KG_TR = 4, KG_THREADS = KG_TC * KG_TR;
__host__ __device__ constexpr int kg_rows(int maxd) { return maxd <= 16 ? 256 : 64; }      // static shared memory stays below 48 KiB
// Kval / Kfhi + Kflo: the forward's K tile, still resident, replaces the distance and the exponential.  RBF only, where
// psi = phi; the launcher drops them for the other kinds, which recompute the tile from X and Z.
template <int MAXD, typename KBT, int KIND>
__global__ void __launch_bounds__(KG_THREADS) k_kernel_grads(const KBT* __restrict__ Kbar, long ldk,
                                                             const double* __restrict__ X, int x_scaled,
                                                             const double* __restrict__ Zs, const double* __restrict__ ls,
                                                             const double* __restrict__ os, long R, int M, int D, int sym,
                                                             double zscale, double* __restrict__ dZ,
                                                             double* __restrict__ dls, double* __restrict__ dos,
                                                             const double* __restrict__ Kval, long ldkv,
                                                             const float* __restrict__ Kfhi, const float* __restrict__ Kflo,
                                                             long ldkf) {
    constexpr int KG_ROWS = kg_rows(MAXD);
    __shared__ double xs[KG_ROWS][MAXD + 1];
    __shared__ double red[KG_THREADS];
    const int tid = threadIdx.x, c = tid % KG_TC, ry = tid / KG_TC;
    const int j = blockIdx.x * KG_TC + c;
    const long n0 = (long)blockIdx.y * KG_ROWS, n1 = min(n0 + KG_ROWS, R);
    for (int i = tid; i < KG_ROWS * D; i += KG_THREADS) {
        const int r = i / D, d = i % D;
        const long n = n0 + r;
        xs[r][d] = n < R ? (x_scaled ? X[n * D + d] : X[n * D + d] / ls[d]) : 0.0;
    }
    // FP32 mode (Kbar arrives as float from the tensor-core GEMM): differences, exponential and the <= 16 per-thread
    // partial sums run in FP32; everything that crosses threads is accumulated in FP64
    using AccT = typename std::conditional<std::is_same<KBT, float>::value, float, double>::type;
    double zj[MAXD];
    AccT az[MAXD], al[MAXD];
#pragma unroll
    for (int d = 0; d < MAXD; ++d) { zj[d] = (d < D && j < M) ? Zs[(long)j * D + d] : 0.0; az[d] = 0; al[d] = 0; }
    __syncthreads();
    const double s = os[0];
    AccT asum = 0;
    if (j < M) {
        // FP64 variant: four rows per iteration, their Kbar / K loads issued together (it is load-latency bound otherwise);
        // the FP32 variant measured slower that way (4.54 vs 4.22 ms backward at cfg4) and keeps one row per iteration
        constexpr int UR = std::is_same<KBT, float>::value ? 1 : 4;
        for (long nb = n0 + ry; nb < n1; nb += UR * KG_TR) {
            double kbr[UR], kvr[UR];
#pragma unroll
            for (int u = 0; u < UR; ++u) {
                const long n = nb + u * KG_TR;
                const bool ok = n < n1;
                kbr[u] = ok ? (double)Kbar[n * ldk + j] : 0.0;
                if (sym && ok) kbr[u] = 0.5 * (kbr[u] + (double)Kbar[(long)j * ldk + n]);
                if constexpr (std::is_same<KBT, float>::value)       // FP32 planes: value = hi + lo exactly
                    kvr[u] = (KIND == TGP_KERNEL_RBF && Kfhi && ok) ? (double)(Kfhi[n * ldkf + j] + Kflo[n * ldkf + j]) : 0.0;
                else
                    kvr[u] = (KIND == TGP_KERNEL_RBF && Kval && ok) ? Kval[n * ldkv + j] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < UR; ++u) {
                const long n = nb + u * KG_TR;
                if (n >= n1) break;
                const int r = (int)(n - n0);
                const double kb = kbr[u];
                if constexpr (std::is_same<KBT, float>::value) {
                    float df[MAXD];
#pragma unroll
                    for (int d = 0; d < MAXD; ++d) if (d < D) df[d] = (float)(xs[r][d] - zj[d]);
                    float t, tk;
                    if (KIND == TGP_KERNEL_RBF && Kfhi) {     // the forward's K planes are still resident
                        t = (float)kb * (float)kvr[u];
                        tk = t;
                    } else {
                        float q = 0.f;
#pragma unroll
                        for (int d = 0; d < MAXD; ++d) if (d < D) q = fmaf(df[d], df[d], q);
                        float ph, ps;
                        Cov<KIND>::phi_psi_f(q, ph, ps);
                        t = (float)kb * (float)s * ps;
                        tk = KIND == TGP_KERNEL_RBF ? t : (float)kb * (float)s * ph;
                    }
                    asum += tk;
#pragma unroll
                    for (int d = 0; d < MAXD; ++d) if (d < D) { az[d] = fmaf(t, df[d], az[d]); al[d] = fmaf(t * df[d], df[d], al[d]); }
                } else {
                    double t, tk;
                    if (KIND == TGP_KERNEL_RBF && Kval) {     // the forward's K tile is still resident: no distance / exponential
                        t = kb * kvr[u];
                        tk = t;
                    } else {
                        double q = 0.0;
#pragma unroll
                        for (int d = 0; d < MAXD; ++d) if (d < D) { const double df = xs[r][d] - zj[d]; q = fma(df, df, q); }
                        double ph, ps;
                        Cov<KIND>::phi_psi(q, ph, ps);
                        t = kb * s * ps;
                        tk = KIND == TGP_KERNEL_RBF ? t : kb * s * ph;
                    }
                    asum += tk;
#pragma unroll
                    for (int d = 0; d < MAXD; ++d) if (d < D) {
                        const double df = xs[r][d] - zj[d];
                        az[d] = fma(t, df, az[d]);
                        al[d] = fma(t * df, df, al[d]);
                    }
                }
            }
        }
    }
    // dZ: reduce the KG_TR row-lanes of each column through shared memory
    for (int d = 0; d < D; ++d) {
        double vz = 0.0, vl = 0.0;
#pragma unroll
        for (int dd = 0; dd < MAXD; ++dd) if (dd == d) { vz = (double)az[dd]; vl = (double)al[dd]; }
        red[tid] = vz;
        __syncthreads();
        if (ry == 0 && j < M) {
            double t = 0.0;
            for (int r = 0; r < KG_TR; ++r) t += red[r * KG_TC + c];
            atomicAdd(dZ + (long)j * D + d, zscale * t / ls[d]);
        }
        __syncthreads();
        // dls[d]: full block reduction
        vl = warp_sum(vl);
        if ((tid & 31) == 0) red[tid >> 5] = vl;
        __syncthreads();
        if (tid == 0) {
            double t = 0.0;
            for (int w = 0; w < KG_THREADS / 32; ++w) t += red[w];
            atomicAdd(dls + d, t / ls[d]);
        }
        __syncthreads();
    }
    double asum_d = warp_sum((double)asum);
    if ((tid & 31) == 0) red[tid >> 5] = asum_d;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int w = 0; w < KG_THREADS / 32; ++w) t += red[w];
        atomicAdd(dos, t / s);
    }
}

template <int KIND, typename KBT>
inline int launch_kernel_grads(const KBT* Kbar, long ldk, const double* X, int x_scaled, const double* Zs,
                               const double* ls, const double* os, long R, int M, int D, int sym, double zscale,
                               double* dZ, double* dls, double* dos, cudaStream_t st, const double* Kval = nullptr,
                               long ldkv = 0, const float* Kfhi = nullptr, const float* Kflo = nullptr, long ldkf = 0) {
    if (KIND != TGP_KERNEL_RBF) { Kval = nullptr; Kfhi = Kflo = nullptr; }     // psi != phi: recompute the tile
#define TGP_KG(MD) k_kernel_grads<MD, KBT, KIND><<<dim3((unsigned)cdiv(M, KG_TC), (unsigned)cdiv(R, kg_rows(MD))), KG_THREADS, 0, st>>>(Kbar, ldk, X, x_scaled, Zs, ls, os, R, M, D, sym, \
                                                                  zscale, dZ, dls, dos, Kval, ldkv, Kfhi, Kflo, ldkf)
    if (D <= 4) TGP_KG(4);
    else if (D <= 8) TGP_KG(8);
    else if (D <= 16) TGP_KG(16);
    else if (D <= 32) TGP_KG(32);
    else if (D <= 64) TGP_KG(64);
    else return set_error(-2, "input dimension > 64 not supported by the kernel-gradient kernel");
#undef TGP_KG
    return check_launch("k_kernel_grads");
}

// Input gradients, the row-side twin of the dZ sum of k_kernel_grads:
//   dX[n,d] += -(1 / ls[d]) * sum_j t[n,j] * (xs[n,d] - zs[j,d]),     t = Kbar[n,j] * os * psi(x_n, z_j)
// Each warp owns ig_rows(MAXD) rows and loops over all M columns in tiles of 32, lane c taking column j0 + c: Kbar is read
// coalesced along j, and the tile's Zs rows are staged in shared memory once per CTA (read from L2 once per 8 warps).  No
// row is split across warps, so dX needs no atomics and the result does not depend on scheduling.  For D <= 16 the warp's
// scaled rows and each lane's Zs row are held in registers; wider inputs read both from shared memory per use to stay
// within the register file.  FP64 throughout (a float Kbar is widened); the distance is taken by direct differences, as the FP64 path of
// k_kernel_grads does.
constexpr int IG_WARPS = 8, IG_THREADS = 32 * IG_WARPS;
__host__ __device__ constexpr int ig_rows(int maxd) { return maxd <= 8 ? 2 : 1; }      // rows per warp
template <int MAXD, typename KBT, int KIND>
__global__ void __launch_bounds__(IG_THREADS) k_input_grads(const KBT* __restrict__ Kbar, long ldk, const double* __restrict__ X,
                                                            const double* __restrict__ Zs, const double* __restrict__ ls,
                                                            const double* __restrict__ os, long R, int M, int D,
                                                            double* __restrict__ dX) {
    constexpr int UR = ig_rows(MAXD), ROWS = IG_WARPS * UR;
    constexpr bool REG = MAXD <= 16;
    __shared__ double xsh[ROWS][MAXD];
    __shared__ double zt[32][MAXD + 1];               // the CTA's current tile of Zs rows, shared by its 8 warps
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long n0 = (long)blockIdx.x * ROWS;
    for (int i = tid; i < ROWS * D; i += IG_THREADS) {
        const int r = i / D, d = i % D;
        const long n = n0 + r;
        xsh[r][d] = n < R ? X[n * D + d] / ls[d] : 0.0;
    }
    __syncthreads();
    const long nw = n0 + warp * UR;                   // first row of this warp
    double xr[REG ? UR : 1][REG ? MAXD : 1];
    if constexpr (REG) {
#pragma unroll
        for (int u = 0; u < UR; ++u)
#pragma unroll
            for (int d = 0; d < MAXD; ++d) xr[u][d] = d < D ? xsh[warp * UR + u][d] : 0.0;
    }
    const double s = os[0];
    double acc[UR][MAXD];
#pragma unroll
    for (int u = 0; u < UR; ++u)
#pragma unroll
        for (int d = 0; d < MAXD; ++d) acc[u][d] = 0.0;
    for (int j0 = 0; j0 < M; j0 += 32) {
        __syncthreads();                              // the previous tile has been read
        for (int i = tid; i < 32 * D; i += IG_THREADS) {
            const int c = i / D, d = i % D;
            zt[c][d] = j0 + c < M ? Zs[(long)(j0 + c) * D + d] : 0.0;
        }
        __syncthreads();
        const int j = j0 + lane;
        if (nw >= R || j >= M) continue;
        double zj[REG ? MAXD : 1];
        if constexpr (REG) {
#pragma unroll
            for (int d = 0; d < MAXD; ++d) zj[d] = d < D ? zt[lane][d] : 0.0;
        }
        double kb[UR];
#pragma unroll
        for (int u = 0; u < UR; ++u) kb[u] = nw + u < R ? (double)Kbar[(nw + u) * ldk + j] : 0.0;
#pragma unroll
        for (int u = 0; u < UR; ++u) {          // rows past R carry kb = 0 and add nothing
            // wide inputs take the differences twice rather than hold them (the register file would not)
            auto diff = [&](int d) {
                if constexpr (REG) return xr[u][d] - zj[d];
                else return d < D ? xsh[warp * UR + u][d] - zt[lane][d] : 0.0;
            };
            double q = 0.0;
#pragma unroll
            for (int d = 0; d < MAXD; ++d) { const double df = diff(d); q = fma(df, df, q); }
            double ph, ps;
            Cov<KIND>::phi_psi(q, ph, ps);
            const double t = kb[u] * s * ps;
#pragma unroll
            for (int d = 0; d < MAXD; ++d) acc[u][d] = fma(t, diff(d), acc[u][d]);
        }
    }
#pragma unroll
    for (int u = 0; u < UR; ++u) {
        const long n = nw + u;
#pragma unroll
        for (int d = 0; d < MAXD; ++d) {
            if (d >= D) break;
            const double v = warp_sum(acc[u][d]);
            if (lane == 0 && n < R) dX[n * D + d] -= v / ls[d];
        }
    }
}

template <int KIND, typename KBT>
inline int launch_input_grads(const KBT* Kbar, long ldk, const double* X, const double* Zs, const double* ls, const double* os,
                              long R, int M, int D, double* dX, cudaStream_t st) {
#define TGP_IG(MD) k_input_grads<MD, KBT, KIND><<<(unsigned)cdiv(R, IG_WARPS * ig_rows(MD)), IG_THREADS, 0, st>>>(Kbar, ldk, X, Zs, ls, \
                                                                                                             os, R, M, D, dX)
    if (D <= 4) TGP_IG(4);
    else if (D <= 8) TGP_IG(8);
    else if (D <= 16) TGP_IG(16);
    else if (D <= 32) TGP_IG(32);
    else if (D <= 64) TGP_IG(64);
    else return set_error(-2, "input dimension > 64 not supported by the input-gradient kernel");
#undef TGP_IG
    return check_launch("k_input_grads");
}

// Final raw-parameter gradients of gE*ELL + gK*KL  (softplus' = sigmoid; KL: dm = m, dL_S = L_S - diag(1/L_ii)).
__global__ void k_finalize_small(const double* __restrict__ raw_ls, const double* __restrict__ raw_os,
                                 const double* __restrict__ m, int M, int D, int n_theta, double gE, double gK,
                                 const double* __restrict__ g_dev, const double* __restrict__ dls, const double* __restrict__ dos,
                                 const double* __restrict__ dm_ell, const double* __restrict__ dZ_acc,
                                 const double* __restrict__ dlogvar, const double* __restrict__ dtheta_acc,
                                 double* __restrict__ out_dZ, double* __restrict__ out_dls,
                                 double* __restrict__ out_dos, double* __restrict__ out_dm,
                                 double* __restrict__ out_dlogvar, double* __restrict__ out_dtheta) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (g_dev) { gE = g_dev[0]; gK = g_dev[1]; }
    if (i < M * D) out_dZ[i] = gE * dZ_acc[i];
    if (i < D) out_dls[i] = gE * dls[i] * sigmoid_d(raw_ls[i]);
    if (i == 0) { out_dos[0] = gE * dos[0] * sigmoid_d(raw_os[0]); if (out_dlogvar) out_dlogvar[0] = gE * dlogvar[0]; }
    if (i < M) out_dm[i] = gE * dm_ell[i] + gK * m[i];
    if (i < n_theta) out_dtheta[i] = gE * dtheta_acc[i];
}

// dL_raw[r,c] = gE*dLS[r,c] + gK*(LS[r,c] - (r==c)/LS[r,r]) for c <= r, else 0     (output ld = M)
__global__ void k_finalize_LS(const double* __restrict__ dLS, const double* __restrict__ LS, long ld, int M, double gE,
                              double gK, const double* __restrict__ g_dev, double* __restrict__ out) {
    const int r = blockIdx.x;
    if (g_dev) { gE = g_dev[0]; gK = g_dev[1]; }
    for (int c = threadIdx.x; c < M; c += blockDim.x) {
        double v = 0.0;
        if (c <= r) {
            const double l = LS[(long)r * ld + c];
            v = gE * dLS[(long)r * ld + c] + gK * (l - (r == c ? 1.0 / l : 0.0));
        }
        out[(long)r * M + c] = v;
    }
}

// Non-whitened q(u): the batch pass and the KL see the whitened pair (m~, P~) = (L^-1 m, L^-1 P).  For rows r < M, c <= r:
//   m~bar[r]  = gE dm_ell[r] + gK m~[r]                                     -> mbar
//   P~bar     = gE dLS + gK (P~ - diag(1 / P~_ii))                          (dLS in place)
//   Gtot      = gE Gtot + m~bar m^T                                         (in place; P~bar P^T is added by a GEMM)
// Gtot then is the complete dF/dL^-1 of F = gE ELL + gK KL, which the Murray chain carries to K_zz.
__global__ void __launch_bounds__(256) k_unwhiten_adjoints(double* __restrict__ dLS, const double* __restrict__ LSt,
                                                           double* __restrict__ Gtot, long ld, int M,
                                                           const double* __restrict__ dm_ell, const double* __restrict__ mt,
                                                           const double* __restrict__ m, double gE, double gK,
                                                           const double* __restrict__ g_dev, double* __restrict__ mbar) {
    const int r = blockIdx.x;
    if (g_dev) { gE = g_dev[0]; gK = g_dev[1]; }
    const double mb = gE * dm_ell[r] + gK * mt[r];
    if (threadIdx.x == 0) mbar[r] = mb;
    const double inv_d = 1.0 / LSt[(long)r * ld + r];
    for (int c = threadIdx.x; c <= r; c += blockDim.x) {
        const long i = (long)r * ld + c;
        dLS[i] = gE * dLS[i] + gK * (LSt[i] - (c == r ? inv_d : 0.0));
        Gtot[i] = gE * Gtot[i] + mb * m[c];
    }
}

// Final raw-parameter gradients of a non-whitened model.  The K_zz-side accumulators (acc_*) already carry gE and gK
// (through Gtot); the K_xz-side sums of the reduce buffer (rb_*) are scaled by gE here.  dm and dL_raw are written by the chain.
__global__ void k_finalize_small_unwhitened(const double* __restrict__ raw_ls, const double* __restrict__ raw_os, int M, int D,
                                            int n_theta, double gE, const double* __restrict__ g_dev,
                                            const double* __restrict__ acc_dZ, const double* __restrict__ acc_dls,
                                            const double* __restrict__ acc_dos, const double* __restrict__ rb_dZ,
                                            const double* __restrict__ rb_dls, const double* __restrict__ rb_dos,
                                            const double* __restrict__ rb_dlogvar, const double* __restrict__ rb_dtheta,
                                            double* __restrict__ out_dZ, double* __restrict__ out_dls, double* __restrict__ out_dos,
                                            double* __restrict__ out_dlogvar, double* __restrict__ out_dtheta) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (g_dev) gE = g_dev[0];
    if (i < M * D) out_dZ[i] = acc_dZ[i] + gE * rb_dZ[i];
    if (i < D) out_dls[i] = (acc_dls[i] + gE * rb_dls[i]) * sigmoid_d(raw_ls[i]);
    if (i == 0) {
        out_dos[0] = (acc_dos[0] + gE * rb_dos[0]) * sigmoid_d(raw_os[0]);
        if (out_dlogvar) out_dlogvar[0] = gE * rb_dlogvar[0];
    }
    if (i < n_theta) out_dtheta[i] = gE * rb_dtheta[i];
}

__global__ void k_copy_strided(const double* __restrict__ src, long lds, double* __restrict__ dst, long ldd, int M) {
    const int r = blockIdx.x;
    for (int c = threadIdx.x; c < M; c += blockDim.x) dst[(long)r * ldd + c] = src[(long)r * lds + c];
}

}  // namespace tgp
