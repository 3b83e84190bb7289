// Full covariance of q(f) over a test batch, its Cholesky factor and joint samples (tgp_qf_cov_forward, tgp_cov_cholesky,
// tgp_cov_sample).  Per output GP, whitened (DESIGN section 2), with A = K_xz L^-T and B = A L_S (R x M each):
//   mu = A m,   Sigma = s Phi(X, X) - A A^T + B B^T,   L_Sigma = chol(Sigma + jitter I),   f0 = mu + eps L_Sigma^T.
// Every product runs on the FP64 DMMA GEMM in every compute mode: this is an evaluation op, and the cancellation in
// K_xx - A A^T + B B^T wants the FP64 operands the step workspace already holds (L, L^-1, L_S, m).
#pragma once
#include "common.cuh"
#include "gemm_f64.cuh"
#include "step_kernels.cuh"
#include "row_kernels.cuh"
#include "backward_kernels.cuh"
#include "f64_driver.cuh"

namespace tgp {
namespace cov {

// Workspace of tgp_qf_cov_forward: O(R M), nothing R x R (Sigma is written straight into the caller's output)
struct CovView { double *K, *AB, *v; };
inline CovView cov_view(Carve& c, int M, long R) {
    CovView w;
    w.K = c.take<double>((size_t)R * M);          // K_xz
    w.AB = c.take<double>((size_t)R * 2 * M);     // [A | B], ld 2M
    w.v = c.take<double>(R);                      // the marginal variances k_row_stats writes next to mu (diag(Sigma) up to rounding)
    return w;
}

// Workspace of tgp_cov_cholesky: the padded work matrix and factor (Rp = R rounded up to the 64-block)
struct CholView { double *Aw, *L, *Dinv; int Rp; };
inline CholView chol_view(Carve& c, long R) {
    CholView w;
    w.Rp = (int)(cdiv(R, POTRF_NB) * POTRF_NB);
    const size_t rp = (size_t)w.Rp;
    w.Aw = c.take<double>(rp * rp);
    // one block row more than Rp: k_potrf_diag's diagonal block of L^-1 is pointed at the block below the diagonal block it
    // factors, which the panel GEMM overwrites right after (the last one lands in the spare row)
    w.L = c.take<double>((rp + POTRF_NB) * rp);
    w.Dinv = c.take<double>(POTRF_NB * POTRF_NB);
    return w;
}

// cov[i,j] = cov[j,i] = cov[i,j] + s phi(r_ij^2) for j <= i, on the lower triangle of -A A^T + B B^T the GEMMs wrote.
// r^2 by direct differences of the scaled rows X[n,d] / ls[d] (as the K tiles take them), so r_ii^2 = 0 and phi = 1 on the
// diagonal.  One CTA per 32 x 32 tile on or below the diagonal; the mirrored tile goes out through shared memory, so that
// both the lower and the upper write are coalesced, and both halves hold the same double (exact symmetry).
constexpr int COV_T = 32, COV_THREADS = 256;
template <int KIND>
__global__ void __launch_bounds__(COV_THREADS) k_cov_assemble(const double* __restrict__ X, const double* __restrict__ ls,
                                                              const double* __restrict__ os, int R, int D,
                                                              double* __restrict__ cov, long ldc) {
    const int bi = blockIdx.y, bj = blockIdx.x;
    if (bj > bi) return;
    extern __shared__ double sm_cov[];
    const int DP = D + 1;
    double* xi = sm_cov;                     // [COV_T][DP] rows of tile row bi
    double* xj = xi + COV_T * DP;            // [COV_T][DP] rows of tile column bj
    double* tr = xj + COV_T * DP;            // [COV_T][COV_T + 1] the finished tile, transposed
    const int i0 = bi * COV_T, j0 = bj * COV_T, tid = threadIdx.x;
    for (int e = tid; e < COV_T * D; e += COV_THREADS) {
        const int r = e / D, d = e % D;
        xi[r * DP + d] = i0 + r < R ? X[(long)(i0 + r) * D + d] / ls[d] : 0.0;
        xj[r * DP + d] = j0 + r < R ? X[(long)(j0 + r) * D + d] / ls[d] : 0.0;
    }
    __syncthreads();
    const double s = os[0];
    const int c = tid % COV_T;
    for (int r = tid / COV_T; r < COV_T; r += COV_THREADS / COV_T) {
        const int i = i0 + r, j = j0 + c;
        if (i < R && j <= i) {
            double acc = 0.0;
            for (int d = 0; d < D; ++d) { const double df = xi[r * DP + d] - xj[c * DP + d]; acc = fma(df, df, acc); }
            const double val = cov[(long)i * ldc + j] + s * Cov<KIND>::phi(acc);
            cov[(long)i * ldc + j] = val;
            tr[c * (COV_T + 1) + r] = val;
        }
    }
    __syncthreads();
    for (int r = tid / COV_T; r < COV_T; r += COV_THREADS / COV_T) {      // cov[j, i] for j < i: row j0 + r, column i0 + c
        const int j = j0 + r, i = i0 + c;
        if (i < R && j < i) cov[(long)j * ldc + i] = tr[r * (COV_T + 1) + c];
    }
}

template <int KIND>
inline int launch_cov_assemble(const double* X, const double* ls, const double* os, long R, int D, double* cov, long ldc,
                               cudaStream_t st) {
    const size_t smem = (size_t)(2 * COV_T * (D + 1) + COV_T * (COV_T + 1)) * sizeof(double);
    if (smem > 200 * 1024) return set_error(-2, "input dimension too large for the covariance kernel");
    if (smem > 48 * 1024) cudaFuncSetAttribute(k_cov_assemble<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const unsigned nt = (unsigned)cdiv(R, COV_T);
    k_cov_assemble<KIND><<<dim3(nt, nt), COV_THREADS, smem, st>>>(X, ls, os, (int)R, D, cov, ldc);
    return check_launch("k_cov_assemble");
}

// mu (R) and Sigma (R x R, ld ldc) at the rows of X from a prepared step workspace
inline int qf_cov_forward(const StepView& s, const CovView& w, const double* X, long R, double* mu, double* cov, long ldc,
                          cudaStream_t st) {
    const int M = s.M, D = s.D;
    // K_xz needs the transformed parameters only: enqueued before the join with the factorisation, as in qf_forward
    TGP_TRY(with_kernel(s.kind, [&](auto k) {
        return launch_rbf<decltype(k)::value>(X, s.Zs, s.ls, s.os, (int)R, M, D, 0, w.K, M, (int)R, M, 0.0, st);
    }));
    if (join_factor(st)) return set_error(-100, "join with the factorisation failed");
    TGP_TRY(f64::ab_rows(s, w.K, (int)R, w.AB, st));
    k_row_stats<<<row_grid(R), ROW_THREADS, 0, st>>>(w.AB, s.mvec, s.os, (int)R, M, mu, w.v);
    TGP_TRY(check_launch("k_row_stats"));
    // lower triangle of -A A^T, then += B B^T
    GemmArgs ga = make_gemm((int)R, (int)R, M, w.AB, 2 * M, 0, w.AB, 2 * M, 0, cov, ldc, -1.0, 0.0);
    ga.c_lower = 1;
    TGP_TRY(gemm_f64(ga, st));
    GemmArgs gb = make_gemm((int)R, (int)R, M, w.AB + M, 2 * M, 0, w.AB + M, 2 * M, 0, cov, ldc, 1.0, 1.0);
    gb.c_lower = 1;
    TGP_TRY(gemm_f64(gb, st));
    return with_kernel(s.kind, [&](auto k) { return launch_cov_assemble<decltype(k)::value>(X, s.ls, s.os, R, D, cov, ldc, st); });
}

// Aw = [[cov + jitter I, 0], [0, I]]  (Rp x Rp; one CTA per row)
__global__ void __launch_bounds__(256) k_cov_pad(const double* __restrict__ cov, long ldc, int R, int Rp, double jitter,
                                                 double* __restrict__ Aw) {
    const int r = blockIdx.x;
    for (int c = threadIdx.x; c < Rp; c += blockDim.x) {
        double v;
        if (r < R && c < R) v = cov[(long)r * ldc + c] + (r == c ? jitter : 0.0);
        else v = r == c ? 1.0 : 0.0;
        Aw[(long)r * Rp + c] = v;
    }
}

// L (R x R, ld ldl, upper triangle 0) = chol(cov + jitter I) by the blocked factorisation of tgp_prepare
inline int cholesky(const CholView& w, long R, const double* cov, long ldc, double jitter, const double* scale, double* L,
                    long ldl, int* status, cudaStream_t st) {
    const int Rp = w.Rp;
    cudaMemsetAsync(status, 0, sizeof(int), st);
    cudaMemsetAsync(w.L, 0, (size_t)(Rp + POTRF_NB) * Rp * sizeof(double), st);
    k_cov_pad<<<Rp, 256, 0, st>>>(cov, ldc, (int)R, Rp, jitter, w.Aw);
    TGP_TRY(check_launch("k_cov_pad"));
    TGP_TRY(blocked_cholesky(w.Aw, w.L, w.L + (long)POTRF_NB * Rp, w.Dinv, Rp, scale, status, st));
    k_copy_strided<<<(unsigned)R, 256, 0, st>>>(w.L, Rp, L, ldl, (int)R);
    return check_launch("k_copy_strided");
}

__global__ void k_cov_broadcast(const double* __restrict__ mu, long R, long n, double* __restrict__ out) {
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long)gridDim.x * blockDim.x) out[e] = mu[e % R];
}

// out (S x R) = mu + eps L^T: one broadcast of mu, then the GEMM with the triangular factor as its B operand and beta = 1
inline int sample(long R, int S, const double* mu, const double* L, long ldl, const double* eps, double* out, cudaStream_t st) {
    const long n = (long)S * R;
    const long blocks = cdiv(n, 256);
    k_cov_broadcast<<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, st>>>(mu, R, n, out);
    TGP_TRY(check_launch("k_cov_broadcast"));
    // Bop[n,k] = L[n,k], nonzero k <= n
    GemmArgs g = make_gemm(S, (int)R, (int)R, eps, R, 0, L, ldl, 0, out, R, 1.0, 1.0);
    g.b_tri = 1;
    return gemm_f64(g, st);
}

}  // namespace cov
}  // namespace tgp
