// Per-step FP64 kernels: ARD-RBF tiles, blocked Cholesky of K_zz (+jitter) with explicit L^-1, KL pieces, and the
// small kernels of the Cholesky-backward chain.  Reference lines: sparse_MF_SP.py:313-330 (kernels + Cholesky),
// utils.py:222-270 (jitter), sparse_MF_SP.py:406-431 (whitened KL).
#pragma once
#include "common.cuh"
#include "gemm_f64.cuh"

namespace tgp {

constexpr int POTRF_NB = 64;
constexpr int POTRF_SMEM = (2 * POTRF_NB * (POTRF_NB + 1) + 3 * POTRF_NB + 2) * (int)sizeof(double);

// ls = softplus(raw_ls), os = softplus(raw_os), Zs = Z / ls      (gpytorch: x.div(lengthscale))
__global__ void k_transform_params(const double* __restrict__ Z, const double* __restrict__ raw_ls,
                                   const double* __restrict__ raw_os, int M, int D, double* __restrict__ ls,
                                   double* __restrict__ os, double* __restrict__ Zs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < D) ls[i] = softplus_d(raw_ls[i]);
    if (i == 0) os[0] = softplus_d(raw_os[0]);
    if (i < M * D) Zs[i] = Z[i] / softplus_d(raw_ls[i % D]);
}

// out[n*ldo + j] = os * phi(sum_d (X[n,d]/ls[d] - Zs[j,d])^2)   for n < R, j < M   (phi: Cov<KIND>, common.cuh)
// pad_identity: rows/cols in [M, Mp) get the identity (used for the padded K_zz); jitter is added on the diagonal.
// x_scaled: X is already divided by ls (K_zz case, X = Zs).
constexpr int RBF_TR = 32, RBF_TC = 64, RBF_THREADS = 256;
template <int KIND>
__global__ void __launch_bounds__(RBF_THREADS) k_rbf_tile(const double* __restrict__ X, const double* __restrict__ Zs,
                                                          const double* __restrict__ ls, const double* __restrict__ os,
                                                          int R, int M, int D, int x_scaled, double* __restrict__ out,
                                                          long ldo, int Rp, int Mp, double jitter) {
    extern __shared__ double sm_rbf[];
    const int DP = D + 1;
    double* xs = sm_rbf;                 // [RBF_TR][DP]
    double* zs = sm_rbf + RBF_TR * DP;   // [RBF_TC][DP]
    const int r0 = blockIdx.y * RBF_TR, c0 = blockIdx.x * RBF_TC, tid = threadIdx.x;
    for (int i = tid; i < RBF_TR * D; i += RBF_THREADS) {
        const int r = i / D, d = i % D, n = r0 + r;
        double v = 0.0;
        if (n < R) v = x_scaled ? X[(long)n * D + d] : X[(long)n * D + d] / ls[d];
        xs[r * DP + d] = v;
    }
    for (int i = tid; i < RBF_TC * D; i += RBF_THREADS) {
        const int c = i / D, d = i % D, j = c0 + c;
        zs[c * DP + d] = j < M ? Zs[(long)j * D + d] : 0.0;
    }
    __syncthreads();
    const double s = os[0];
    const int c = tid % RBF_TC, j = c0 + c;
    for (int r = tid / RBF_TC; r < RBF_TR; r += RBF_THREADS / RBF_TC) {
        const int n = r0 + r;
        if (n >= Rp || j >= Mp) continue;
        double val;
        if (n < R && j < M) {
            double acc = 0.0;
            for (int d = 0; d < D; ++d) { const double df = xs[r * DP + d] - zs[c * DP + d]; acc = fma(df, df, acc); }
            val = s * Cov<KIND>::phi(acc);
            if (n == j) val += jitter;
        } else {
            val = (n == j) ? 1.0 : 0.0;
        }
        out[(long)n * ldo + j] = val;
    }
}

// Register-blocked variant for D <= 64 (every shipped configuration): a thread owns one column j — its inducing point
// lives in registers, zero-padded to MAXD — and walks the tile's rows; the X rows are read from shared memory as
// warp-uniform 16-byte broadcasts (MAXD/2 LDS per element instead of 2*D 8-byte ones in the generic kernel above).
template <int MAXD, int KIND>
__global__ void __launch_bounds__(RBF_THREADS) k_rbf_tile_reg(const double* __restrict__ X, const double* __restrict__ Zs,
                                                              const double* __restrict__ ls, const double* __restrict__ os,
                                                              int R, int M, int D, int x_scaled, double* __restrict__ out,
                                                              long ldo, int Rp, int Mp, double jitter) {
    __shared__ __align__(16) double xs[RBF_TR][MAXD];
    const int r0 = blockIdx.y * RBF_TR, c0 = blockIdx.x * RBF_TC, tid = threadIdx.x;
    for (int i = tid; i < RBF_TR * MAXD; i += RBF_THREADS) {
        const int r = i / MAXD, d = i % MAXD, n = r0 + r;
        double v = 0.0;
        if (n < R && d < D) v = x_scaled ? X[(long)n * D + d] : X[(long)n * D + d] / ls[d];
        xs[r][d] = v;
    }
    const int c = tid % RBF_TC, j = c0 + c;
    double zj[MAXD];
#pragma unroll
    for (int d = 0; d < MAXD; ++d) zj[d] = (j < M && d < D) ? Zs[(long)j * D + d] : 0.0;
    __syncthreads();
    const double s = os[0];
    for (int r = tid / RBF_TC; r < RBF_TR; r += RBF_THREADS / RBF_TC) {
        const int n = r0 + r;
        if (n >= Rp || j >= Mp) continue;
        double val;
        if (n < R && j < M) {
            double acc = 0.0;
            const double2* xr = reinterpret_cast<const double2*>(xs[r]);
#pragma unroll
            for (int d = 0; d < MAXD / 2; ++d) {
                const double2 x2 = xr[d];
                const double d0 = x2.x - zj[2 * d], d1 = x2.y - zj[2 * d + 1];
                acc = fma(d0, d0, acc);
                acc = fma(d1, d1, acc);
            }
            val = s * Cov<KIND>::phi(acc);
            if (n == j) val += jitter;
        } else {
            val = (n == j) ? 1.0 : 0.0;
        }
        out[(long)n * ldo + j] = val;
    }
}

template <int KIND>
inline int launch_rbf(const double* X, const double* Zs, const double* ls, const double* os, int R, int M, int D,
                      int x_scaled, double* out, long ldo, int Rp, int Mp, double jitter, cudaStream_t st) {
    dim3 grid((unsigned)cdiv(Mp, RBF_TC), (unsigned)cdiv(Rp, RBF_TR));
#define TGP_RBF(MD) k_rbf_tile_reg<MD, KIND><<<grid, RBF_THREADS, 0, st>>>(X, Zs, ls, os, R, M, D, x_scaled, out, ldo, Rp, Mp, jitter)
    if (D <= 4) { TGP_RBF(4); return check_launch("k_rbf_tile_reg"); }
    if (D <= 8) { TGP_RBF(8); return check_launch("k_rbf_tile_reg"); }
    if (D <= 16) { TGP_RBF(16); return check_launch("k_rbf_tile_reg"); }
    if (D <= 32) { TGP_RBF(32); return check_launch("k_rbf_tile_reg"); }
    if (D <= 64) { TGP_RBF(64); return check_launch("k_rbf_tile_reg"); }
#undef TGP_RBF
    const size_t smem = (size_t)(RBF_TR + RBF_TC) * (D + 1) * sizeof(double);
    if (smem > 200 * 1024) return set_error(-2, "input dimension too large for the RBF tile kernel");
    if (smem > 48 * 1024)       // generic kernel for D > 64 only: set per call (per-device attribute, rare path)
        cudaFuncSetAttribute(k_rbf_tile<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    k_rbf_tile<KIND><<<grid, RBF_THREADS, smem, st>>>(X, Zs, ls, os, R, M, D, x_scaled, out, ldo, Rp, Mp, jitter);
    return check_launch("k_rbf_tile");
}

// Factor the kb-th 64x64 diagonal block of the (partially updated) matrix Aw: L_kk -> Lout (upper zero),
// L_kk^-1 -> Dinv (dense 64x64, upper zero) and -> the diagonal block of Linv.
// status[0] = 1-based index of the first non-positive / NaN pivot (0 = ok); only the first failure is recorded.
//
// One CTA on the critical path of the factorisation, written for latency.  Gauss-Jordan on the UNSCALED block: step j
// subtracts f_t = a[t][j] / d_j times row j from every row t > j, on the lower triangle of A (row j read through
// symmetry as column j) and on an identity (which turns into W = Lu^-1, A = Lu D Lu^T).  Row t then always has exactly
// t + 1 live entries, columns k <= j holding W[t][k] and columns k > j holding A[t][k]; so the assignment of entries to
// threads is static — thread (t, q) keeps entries k = q, q+8, ..., q+56 of row t in REGISTERS for the whole
// factorisation, and the only shared-memory traffic per step is the operand vector op[k] (= a[k][j] for k > j,
// = w[j][k] for k < j: one array, one formula val -= f * op[k]) that the owners of column j+1 / row j+1 publish for the
// next step.  The column loop is fully unrolled (entry indices, owner phases and buffer parities are compile-time
// constants): one barrier and ~30 instructions per warp per column.  What is left is the dependent FP64 chain of a
// column (f = a*rd, the update of the next pivot, its reciprocal by a hardware seed + two Newton steps): measured
// 1.21-1.25 ms per M = 1024 factorisation with 256 / 512 / 1024 threads alike (it was 2.04 ms with a two-barrier
// shared-memory version followed by a 64-step substitution for the inverse).
constexpr int POTRF_THREADS = 512;         // 64 rows x 8 column phases, 8 register-resident entries per thread
__device__ __forceinline__ double fast_rcp(double d) {   // reciprocal to ~1 ulp: hardware seed + two Newton steps
    double x;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
    x = fma(x, fma(-d, x, 1.0), x);
    x = fma(x, fma(-d, x, 1.0), x);
    return x;
}
__global__ void __launch_bounds__(POTRF_THREADS) k_potrf_diag(const double* __restrict__ Aw, double* __restrict__ Lout,
                                                              double* __restrict__ Linv, double* __restrict__ Dinv,
                                                              int kb, long ld, const double* __restrict__ os,
                                                              int* __restrict__ status) {
    constexpr int NB = POTRF_NB, LDS = NB + 1, NT = POTRF_THREADS, PH = NT / NB, NI = NB / PH;
    // a pivot that is not positive *to working precision* (relative to the kernel's diagonal k(z,z) = outputscale) counts
    // as a failed factorisation: exactly singular inputs (duplicated inducing rows) then take the jitter ladder
    // deterministically instead of depending on the sign of a 1e-16 rounding residue
    const double pivot_floor = 8.0 * 2.220446049250313e-16 * os[0];
    extern __shared__ double sm_potrf[];
    double* sa = sm_potrf;                 // [NB][LDS] staging: input block, later L
    double* sw = sa + NB * LDS;            // [NB][LDS] staging: L^-1
    double* op = sw + NB * LDS;            // [2][NB] operand vector of the current / next step
    double* dd = op + 2 * NB;              // [NB] pivots d_j
    double* rdv = dd + NB;                 // [2] 1 / d_j of the current / next step
    const int tid = threadIdx.x, t = tid & 63, q = tid >> 6;
    const long base = (long)kb * NB * ld + (long)kb * NB;
    for (int i = tid; i < NB * NB; i += NT) {
        const int r = i >> 6, c = i & 63;
        sa[r * LDS + c] = (c <= r) ? Aw[base + (long)r * ld + c] : 0.0;
    }
    __syncthreads();
    double val[NI], lsave[NI];
#pragma unroll
    for (int i = 0; i < NI; ++i) { val[i] = sa[t * LDS + q + PH * i]; lsave[i] = 0.0; }
    // Entries right of the diagonal (k > t) take part in the arithmetic but are never read: the loop body below has no
    // per-entry branches at all (the kernel is bound by the instruction latency of one warp per column, not by work).
    // Conventions that make this work: f = 0 for finished rows (t <= j); op[j] = 0 in step j, so that the entry that is
    // about to change type is left alone by the generic update.
    if (q == 0) {
        op[t] = t == 0 ? 0.0 : val[0];           // operands of step 0: column 0 of A
        if (t == 0) {
            const double d = val[0];
            if (!(d > pivot_floor)) atomicCAS(status, 0, kb * NB + 1);
            dd[0] = d;
            rdv[0] = fast_rcp(d);
        }
    }
    __syncthreads();
    // Fully unrolled over the 64 columns (j = PH*jo + ji): every entry index, owner phase and buffer parity is a
    // compile-time constant, so a column costs one warp ~20 instructions.
    const double* op_t = op + t;
    const double* op_q = op + q;
#pragma unroll
    for (int jo = 0; jo < NI; ++jo) {
#pragma unroll
        for (int ji = 0; ji < PH; ++ji) {
            const int j = PH * jo + ji;
            const int cur = (j & 1) * NB, nxt = ((j + 1) & 1) * NB;
            const double f = t > j ? op_t[cur] * rdv[j & 1] : 0.0;
#pragma unroll
            for (int i = 0; i < NI; ++i) val[i] = fma(-f, op_q[cur + PH * i], val[i]);
            if (q == ji && t > j) { lsave[jo] = val[jo]; val[jo] = -f; }     // a[t][j] is final; the entry becomes W[t][j]
            if (j + 1 < NB) {
                const int jn = j + 1, jno = jn / PH, jni = jn % PH;
                if (q == jni) {                    // warp-uniform: owners of column j+1 publish it for the next step
                    const double v = val[jno];
                    if (t > jn) op[nxt + t] = v;
                    else if (t == jn) {            // ... and its pivot
                        if (!(v > pivot_floor)) atomicCAS(status, 0, kb * NB + jn + 1);
                        dd[jn] = v;
                        rdv[jn & 1] = fast_rcp(v);
                        op[nxt + jn] = 0.0;
                    }
                }
                if (t == jn) {                     // row j+1 of W (left of the diagonal) is final
#pragma unroll
                    for (int i = 0; i < NI; ++i) if (q + PH * i <= j) op[nxt + q + PH * i] = val[i];
                }
            }
            __syncthreads();
        }
    }
    // A = Lu D Lu^T with a[t][k] = Lu[t][k] d_k, W = Lu^-1:   L = Lu D^1/2,   L^-1 = D^-1/2 W
    const double rst = rsqrt(dd[t]);
#pragma unroll
    for (int i = 0; i < NI; ++i) {
        const int k = q + PH * i;
        double l = 0.0, li = 0.0;
        if (k < t) { l = lsave[i] * rsqrt(dd[k]); li = val[i] * rst; }
        else if (k == t) { l = val[i] * rst; li = rst; }
        sa[t * LDS + k] = l;
        sw[t * LDS + k] = li;
    }
    __syncthreads();
    for (int i = tid; i < NB * NB; i += NT) {
        const int r = i >> 6, c = i & 63;
        Lout[base + (long)r * ld + c] = sa[r * LDS + c];
        Linv[base + (long)r * ld + c] = sw[r * LDS + c];
        Dinv[i] = sw[r * LDS + c];
    }
}

// LS = tril(L_raw) (ld -> ldo, rest zero) and the three KL reductions:
// kl[0] += sum_i log(L_ii^2)   kl[1] += sum_i m_i^2   kl[2] += ||tril(L_raw)||_F^2
__global__ void __launch_bounds__(256) k_tril_kl(const double* __restrict__ Lraw, const double* __restrict__ m, int M,
                                                 double* __restrict__ LS, long ldo, int Mp, double* __restrict__ kl) {
    const int r = blockIdx.x;
    double fro = 0.0;
    for (int c = threadIdx.x; c < Mp; c += blockDim.x) {
        double v = 0.0;
        if (r < M && c <= r) { v = Lraw[(long)r * M + c]; fro = fma(v, v, fro); }
        LS[(long)r * ldo + c] = v;
    }
    fro = warp_sum(fro);
    __shared__ double part[8];
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = fro;
    __syncthreads();
    if (threadIdx.x == 0 && r < M) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += part[w];
        const double d = Lraw[(long)r * M + r];
        atomicAdd(kl + 0, log(d * d));
        atomicAdd(kl + 1, m[r] * m[r]);
        atomicAdd(kl + 2, t);
    }
}

// kl_out = 0.5 * (-logdet + m'm + trace - M)
__global__ void k_kl_finish(const double* __restrict__ kl, int M, double* __restrict__ out) {
    out[0] = 0.5 * (-kl[0] + kl[1] + kl[2] - (double)M);
}

// sum of v over the 256 threads of the CTA, valid in thread 0
__device__ __forceinline__ double block_sum_256(double v) {
    __shared__ double part[8];
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < 8; ++w) t += part[w];
    return t;
}

// y = L x (trans = 0) or y = L^T x (trans = 1) for a lower-triangular L (M x M, ld ld); one CTA of 256 threads per element
__global__ void __launch_bounds__(256) k_trmv_lower(const double* __restrict__ L, long ld, int M, const double* __restrict__ x,
                                                    double* __restrict__ y, int trans) {
    const int i = blockIdx.x;
    double acc = 0.0;
    if (trans) for (int k = i + threadIdx.x; k < M; k += 256) acc = fma(L[(long)k * ld + i], x[k], acc);
    else for (int k = threadIdx.x; k <= i; k += 256) acc = fma(L[(long)i * ld + k], x[k], acc);
    acc = block_sum_256(acc);
    if (threadIdx.x == 0) y[i] = acc;
}

// The KL sums of k_tril_kl for a lower-triangular P (ld ld) that is already in place:
// kl[0] += sum_i log(P_ii^2)   kl[1] += sum_i m_i^2   kl[2] += ||P||_F^2
__global__ void __launch_bounds__(256) k_kl_rows(const double* __restrict__ P, long ld, const double* __restrict__ m, int M,
                                                 double* __restrict__ kl) {
    const int r = blockIdx.x;
    double fro = 0.0;
    for (int c = threadIdx.x; c <= r; c += 256) { const double v = P[(long)r * ld + c]; fro = fma(v, v, fro); }
    fro = block_sum_256(fro);
    if (threadIdx.x == 0) {
        const double d = P[(long)r * ld + r];
        atomicAdd(kl + 0, log(d * d));
        atomicAdd(kl + 1, m[r] * m[r]);
        atomicAdd(kl + 2, fro);
    }
}

__global__ void k_halve_diag(double* __restrict__ P, long ld, int M) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < M) P[(long)i * ld + i] *= 0.5;
}

struct StepView {       // carved views into the per-step workspace (all doubles)
    int M, Mp, D;
    int kind;           // TGP_KERNEL_* of the model (not part of the layout)
    double *ls, *os, *Zs, *kl3, *Dinv, *mvec;
    double *Kzz, *L, *Linv, *LS, *Cm, *S0, *S1, *S2, *S3;
    // TGP_QU_UNWHITENED only (nullptr otherwise): P = tril(L_raw), while LS and mvec hold the whitened pair L^-1 P, L^-1 m
    double* P;
};

inline int pad_M(int M) {
    int mp = POTRF_NB;
    while (mp < M) mp *= 2;
    return mp;
}

// The FP64 region of the step workspace.  The Mp x Mp matrices are multiples of 256 bytes, so they are contiguous:
// run_prepare zeroes L and Linv with one memset, and the region ends on a 256-byte boundary.
inline StepView step_view(Carve& c, int M, int D) {
    StepView v;
    v.M = M; v.D = D; v.Mp = pad_M(M); v.kind = TGP_KERNEL_RBF;
    const size_t mm = (size_t)v.Mp * v.Mp;
    v.ls = c.take<double>(D);
    v.os = c.take<double>(1);
    v.kl3 = c.take<double>(8);
    v.Zs = c.take<double>((size_t)M * D);
    v.mvec = c.take<double>(M);
    v.Dinv = c.take<double>(POTRF_NB * POTRF_NB);
    v.Kzz = c.take<double>(mm); v.L = c.take<double>(mm); v.Linv = c.take<double>(mm); v.LS = c.take<double>(mm);
    v.Cm = c.take<double>(mm);
    v.S0 = c.take<double>(mm); v.S1 = c.take<double>(mm); v.S2 = c.take<double>(mm); v.S3 = c.take<double>(mm);
    v.P = nullptr;      // carved last by step_layout for non-whitened models, so that no other offset depends on the form
    return v;
}

// Right-looking blocked Cholesky of the Np x Np lower triangle of Aw (Np a multiple of POTRF_NB, ld = Np); the panel solve
// is a GEMM with the inverted diagonal block.  L -> L (its upper triangle must hold zeros already), the diagonal blocks of
// L^-1 -> Linv (same ld; only block (kb, kb) of Linv + kb (NB ld + NB) is written), Dinv: POTRF_NB^2 scratch.  Aw's
// trailing blocks are overwritten.  status: first pivot not above 8 eps * scale[0] (tgp_prepare's meaning).
inline int blocked_cholesky(double* Aw, double* L, double* Linv, double* Dinv, int Np, const double* scale, int* status,
                            cudaStream_t st) {
    const int NB = POTRF_NB, nb = Np / NB;
    static PerDeviceOnce potrf_once;
    if (potrf_once.first()) cudaFuncSetAttribute(k_potrf_diag, cudaFuncAttributeMaxDynamicSharedMemorySize, POTRF_SMEM);
    for (int kb = 0; kb < nb; ++kb) {
        k_potrf_diag<<<1, POTRF_THREADS, POTRF_SMEM, st>>>(Aw, L, Linv, Dinv, kb, Np, scale, status);
        TGP_TRY(check_launch("k_potrf_diag"));
        const int rem = Np - (kb + 1) * NB;
        if (rem <= 0) break;
        const long off_panel = (long)(kb + 1) * NB * Np + (long)kb * NB;
        GemmArgs p = make_gemm(rem, NB, NB, Aw + off_panel, Np, 0, Dinv, NB, 0, L + off_panel, Np);
        p.b_tri = 1;
        TGP_TRY(gemm_f64(p, st));
        const long off_trail = (long)(kb + 1) * NB * Np + (long)(kb + 1) * NB;
        GemmArgs t = make_gemm(rem, rem, NB, L + off_panel, Np, 0, L + off_panel, Np, 0, Aw + off_trail, Np, -1.0, 1.0);
        t.c_lower = 1;
        TGP_TRY(gemm_f64(t, st));
    }
    return 0;
}

// K_zz (+jitter) -> L, L^-1 (explicit), C = L_S^T L^-1, KL.  Everything stays on `st`; no host sync.
// Non-whitened q(u) (v.P set): L_S = L^-1 P and mvec = L^-1 m, the whitened pair of the same q(u), and the KL of that pair.
inline int run_prepare(const StepView& v, const double* Z, const double* raw_ls, const double* raw_os,
                       const double* m, const double* Lraw, double jitter, double* kl_out, int* status,
                       bool need_C, cudaStream_t st, cudaStream_t (*fork)(cudaStream_t) = nullptr) {
    const int M = v.M, Mp = v.Mp, D = v.D, NB = POTRF_NB;
    const size_t mm = (size_t)Mp * Mp;
    const bool unwhitened = v.P != nullptr;
    cudaMemsetAsync(status, 0, sizeof(int), st);
    cudaMemsetAsync(v.kl3, 0, 8 * sizeof(double), st);
    // L and Linv are contiguous, and so is LS after them: the non-whitened transform writes its lower triangle only
    cudaMemsetAsync(v.L, 0, (unwhitened ? 3 : 2) * mm * sizeof(double), st);
    if (!unwhitened) cudaMemcpyAsync(v.mvec, m, (size_t)M * sizeof(double), cudaMemcpyDeviceToDevice, st);
    {
        const int n = max(M * D, D);
        k_transform_params<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(Z, raw_ls, raw_os, M, D, v.ls, v.os, v.Zs);
        TGP_TRY(check_launch("k_transform_params"));
    }
    // non-whitened: tril(L_raw) goes to P, and the sums of this kernel (of the untransformed pair) to unused slots of kl3
    k_tril_kl<<<Mp, 256, 0, st>>>(Lraw, m, M, unwhitened ? v.P : v.LS, Mp, Mp, unwhitened ? v.kl3 + 4 : v.kl3);
    TGP_TRY(check_launch("k_tril_kl"));
    if (!unwhitened) k_kl_finish<<<1, 1, 0, st>>>(v.kl3, M, kl_out);
    cudaStream_t fst = fork ? fork(st) : nullptr;
    // everything above stays on the caller's stream (a whitened model's kl_out is an output in stream order); the factorisation
    // proper forks onto the high-priority stream `fst` when the caller passed one (tgp_prepare), see common.cuh
    st = fst ? fst : st;
    TGP_TRY(with_kernel(v.kind, [&](auto k) {
        return launch_rbf<decltype(k)::value>(v.Zs, v.Zs, v.ls, v.os, M, M, D, 1, v.Kzz, Mp, Mp, Mp, jitter, st);
    }));

    TGP_TRY(blocked_cholesky(v.Kzz, v.L, v.Linv, v.Dinv, Mp, v.os, status, st));
    // explicit inverse by recursive doubling: inv([[A,0],[B,C]]) = [[A^-1,0],[-C^-1 B A^-1, C^-1]]
    for (int b = NB; b < Mp; b *= 2) {
        const int batch = Mp / (2 * b);
        const long stride = (long)2 * b * (Mp + 1);
        const long off_B = (long)b * Mp;                 // block (1,0) of each 2b x 2b diagonal block
        const long off_C = (long)b * Mp + b;             // block (1,1)
        GemmArgs t = make_gemm(b, b, b, v.L + off_B, Mp, 0, v.Linv, Mp, 1, v.S0 + off_B, Mp);   // T = B * A^-1
        t.b_tri = 2; t.batch = batch; t.strideA = t.strideB = t.strideC = stride;
        TGP_TRY(gemm_f64(t, st));
        GemmArgs x = make_gemm(b, b, b, v.Linv + off_C, Mp, 0, v.S0 + off_B, Mp, 1, v.Linv + off_B, Mp, -1.0, 0.0);
        x.a_tri = 1; x.batch = batch; x.strideA = x.strideB = x.strideC = stride;
        TGP_TRY(gemm_f64(x, st));
    }
    if (unwhitened) {
        // L_S = L^-1 P   (Aop[m,k] = Linv[m,k], nonzero k <= m;  Bop[n,k] = P[k,n], nonzero k >= n)
        GemmArgs t = make_gemm(M, M, M, v.Linv, Mp, 0, v.P, Mp, 1, v.LS, Mp);
        t.a_tri = 1; t.b_tri = 2; t.c_lower = 1;
        TGP_TRY(gemm_f64(t, st));
        k_trmv_lower<<<M, 256, 0, st>>>(v.Linv, Mp, M, m, v.mvec, 0);
        TGP_TRY(check_launch("k_trmv_lower"));
        // KL(N(m, P P^T) || N(0, L L^T)) = the whitened KL of (L^-1 m, L^-1 P): it needs L, so it is finished here
        k_kl_rows<<<M, 256, 0, st>>>(v.LS, Mp, v.mvec, M, v.kl3);
        TGP_TRY(check_launch("k_kl_rows"));
        k_kl_finish<<<1, 1, 0, st>>>(v.kl3, M, kl_out);
    }
    // C = L_S^T L^-1   (Aop[m,k] = LS[k,m], nonzero k >= m;  Bop[n,k] = Linv[k,n], nonzero k >= n)
    if (need_C) {      // only the tensor-core mode contracts with C; the FP64 mode applies L_S to A directly
        GemmArgs c = make_gemm(M, M, M, v.LS, Mp, 1, v.Linv, Mp, 1, v.Cm, Mp);
        c.a_tri = 2; c.b_tri = 2;
        TGP_TRY(gemm_f64(c, st));
    }
    return 0;
}

}  // namespace tgp
