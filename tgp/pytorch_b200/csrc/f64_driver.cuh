// Host-side orchestration of compute mode TGP_F64: the batch contractions on the FP64 DMMA GEMM (gemm_f64.cuh), in the
// reference's form of two dependent triangular contractions (a = L^-1 k, b = L_S^T a).
#pragma once
#include "gemm_f64.cuh"
#include "step_kernels.cuh"
#include "backward_kernels.cuh"
#include "row_kernels.cuh"

namespace tgp {
namespace f64 {

inline long g_row_chunk = 32768;      // rows per launch of the batch contractions (Kbar / Abar staging); measured at cfg4:
                                      // 8192 -> 20.3 ms/step, 16384 -> 20.0, 32768 -> 19.6, 65536 -> 19.5

// AB = [A | B] (R x 2M) and K (R x M) are kept from the forward for the backward; Kbar / Abar are per-chunk staging
struct BatchView { double *AB, *Kbuf, *Kbar, *Abar; long Rc; };

inline long chunk_rows(long R) { return R < g_row_chunk ? R : g_row_chunk; }

inline BatchView batch_view(Carve& c, int M, long R) {
    BatchView b;
    b.Rc = chunk_rows(R);
    b.AB = c.take<double>(R * 2 * M);
    b.Kbuf = c.take<double>(R * M);
    b.Kbar = c.take<double>(b.Rc * M);
    b.Abar = c.take<double>(b.Rc * M);
    return b;
}

// The weight-gradient GEMMs have only (M/128)^2 output tiles but a reduction over thousands of rows: split the
// reduction so that the live CTAs fill whole waves of the 148 SMs (36 lower tiles x 4 splits = 144 CTAs at M = 1024).
inline int weight_splitk(int M, int rc, bool lower) {
    const long tiles = gemm_tiles(M, M, lower);
    const long max_split = rc / (8 * GBK) > 0 ? rc / (8 * GBK) : 1;
    auto util = [&](long s) { const long c = tiles * s; return (double)c / (double)(cdiv(c, GEMM_SLOTS) * GEMM_SLOTS); };
    double best_util = 0.0;
    for (long s = 1; s <= max_split && s <= 64; ++s) best_util = util(s) > best_util ? util(s) : best_util;
    int best = 1;
    for (long s = 1; s <= max_split && s <= 64; ++s)           // smallest split that fills the waves (fewest atomics)
        if (util(s) >= best_util - 0.03) { best = (int)s; break; }
    return best;
}

// [A | B] of rc rows (ld 2M) from their K_xz (ld M): the two triangular contractions of the forward.  Also the first stage
// of the full covariance over a test batch (cov_kernels.cuh), in every compute mode.
inline int ab_rows(const StepView& s, const double* K, int rc, double* AB, cudaStream_t st) {
    const int M = s.M;
    // A = K L^-T   (Bop[n,k] = Linv[n,k], nonzero k <= n)
    GemmArgs ga = make_gemm(rc, M, M, K, M, 0, s.Linv, s.Mp, 0, AB, 2 * M);
    ga.b_tri = 1;
    ga.tag = 1;
    TGP_TRY(gemm_f64(ga, st));
    // B = A L_S   (Bop[n,k] = L_S[k,n], nonzero k >= n) — the reference's two-contraction form, both triangular
    GemmArgs gb = make_gemm(rc, M, M, AB, 2 * M, 0, s.LS, s.Mp, 1, AB + M, 2 * M);
    gb.b_tri = 2;
    gb.tag = 1;
    return gemm_f64(gb, st);
}

// forward: K_xz per chunk -> A = K L^-T, B = A L_S -> row statistics
inline int qf_forward(const StepView& s, const BatchView& b, const double* X, long R, double* mu, double* v, cudaStream_t st) {
    const int M = s.M, D = s.D;
    // K_xz of every chunk depends on the transformed parameters only: it is enqueued BEFORE the join with the factorisation
    // (which may still be running on the library's high-priority stream, TGP_OPT_OVERLAP_KGEN) and runs under it
    TGP_TRY(with_kernel(s.kind, [&](auto k) {
        for (long r0 = 0; r0 < R; r0 += b.Rc) {
            const int rc = (int)((R - r0) < b.Rc ? (R - r0) : b.Rc);
            TGP_TRY(launch_rbf<decltype(k)::value>(X + r0 * D, s.Zs, s.ls, s.os, rc, M, D, 0, b.Kbuf + r0 * M, M, rc, M, 0.0, st));
        }
        return 0;
    }));
    if (join_factor(st)) return set_error(-100, "join with the factorisation failed");
    for (long r0 = 0; r0 < R; r0 += b.Rc) {
        const int rc = (int)((R - r0) < b.Rc ? (R - r0) : b.Rc);
        TGP_TRY(ab_rows(s, b.Kbuf + r0 * M, rc, b.AB + r0 * 2 * M, st));
    }
    k_row_stats<<<row_grid(R), ROW_THREADS, 0, st>>>(b.AB, s.mvec, s.os, (int)R, M, mu, v);
    return check_launch("k_row_stats");
}

// backward:
//   Bbar = 2 g_v B;  Abar = g_mu m - 2 g_v A + Bbar L_S^T;  Kbar = Abar L^-1;
//   Gbar += tril(Abar^T K);  dL_S += tril(A^T Bbar)   (accumulated in the `Cbar` slot of the reduce buffer)
template <int KIND>
inline int qf_backward_k(const StepView& s, const BatchView& b, const double* X, long R, const double* g_mu, const double* g_v,
                         double* dm, double* dos, double* dZ, double* dls, double* Gbar, double* Cbar, double* dX,
                         cudaStream_t st) {
    const int M = s.M, D = s.D;
    for (long r0 = 0; r0 < R; r0 += b.Rc) {
        const int rc = (int)((R - r0) < b.Rc ? (R - r0) : b.Rc);
        double* ABc = b.AB + r0 * 2 * M;
        {
            dim3 grid((unsigned)cdiv(M, ABB_COLS), (unsigned)cdiv(rc, ABB_ROWS));
            k_make_abbar<<<grid, ABB_COLS, 0, st>>>(ABc, b.Abar, g_mu + r0, g_v + r0, s.mvec, rc, M, dm, dos);
            TGP_TRY(check_launch("k_make_abbar"));
        }
        // Abar += Bbar * L_S^T   (Bop[n,k] = L_S[n,k], nonzero k <= n)
        GemmArgs g0 = make_gemm(rc, M, M, ABc + M, 2 * M, 0, s.LS, s.Mp, 0, b.Abar, M, 1.0, 1.0);
        g0.b_tri = 1; g0.tag = 1;
        TGP_TRY(gemm_f64(g0, st));
        const double* Kc = b.Kbuf + r0 * M;          // K_xz of these rows, kept by the forward
        // Kbar = Abar * Linv     (Bop[n,k] = Linv[k,n], nonzero k >= n)
        GemmArgs g1 = make_gemm(rc, M, M, b.Abar, M, 0, s.Linv, s.Mp, 1, b.Kbar, M);
        g1.b_tri = 2; g1.tag = 1;
        TGP_TRY(gemm_f64(g1, st));
        // the RBF reads K from Kc; the other kinds recompute it (launch_kernel_grads)
        TGP_TRY(launch_kernel_grads<KIND>(b.Kbar, M, X + r0 * D, 0, s.Zs, s.ls, s.os, rc, M, D, 0, 1.0, dZ, dls, dos, st, Kc, M));
        if (dX) TGP_TRY(launch_input_grads<KIND>(b.Kbar, M, X + r0 * D, s.Zs, s.ls, s.os, rc, M, D, dX + r0 * D, st));
        // Gbar += tril(Abar^T K)      (reduction over the rows of the chunk)
        GemmArgs g3 = make_gemm(M, M, rc, b.Abar, M, 1, Kc, M, 1, Gbar, s.Mp, 1.0, 1.0);
        g3.c_lower = 1; g3.splitk = weight_splitk(M, rc, true); g3.tag = 1;
        TGP_TRY(gemm_f64(g3, st));
        // dL_S += tril(A^T Bbar)
        GemmArgs g4 = make_gemm(M, M, rc, ABc, 2 * M, 1, ABc + M, 2 * M, 1, Cbar, s.Mp, 1.0, 1.0);
        g4.c_lower = 1; g4.splitk = weight_splitk(M, rc, true); g4.tag = 1;
        TGP_TRY(gemm_f64(g4, st));
    }
    return 0;
}

inline int qf_backward(const StepView& s, const BatchView& b, const double* X, long R, const double* g_mu, const double* g_v,
                       double* dm, double* dos, double* dZ, double* dls, double* Gbar, double* Cbar, double* dX,
                       cudaStream_t st) {
    return with_kernel(s.kind, [&](auto k) {
        return qf_backward_k<decltype(k)::value>(s, b, X, R, g_mu, g_v, dm, dos, dZ, dls, Gbar, Cbar, dX, st);
    });
}

}  // namespace f64
}  // namespace tgp
