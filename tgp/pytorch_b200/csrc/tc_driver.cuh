// Host-side orchestration of the FP32 / tensor-core mode (workspace carving + launch sequences).
#pragma once
#include "step_kernels.cuh"
#include "backward_kernels.cuh"
#include "tc_path.cuh"

namespace tgp {
namespace tc {

constexpr long TC_ROW_CHUNK = 16384;

struct StepPlanes { float *Whi, *Wlo, *Wthi, *Wtlo; double* u; long ldk, ld2m; };      // u = L^-T m (FP64, M)
struct BatchPlanes {
    float *AB;                       // (R x ld2m) saved forward -> backward
    float *Khi, *Klo;                // (R x ldk)  K_xz planes, kept from the forward (kernel gradients read hi + lo)
    float *KThi, *KTlo;              // per row chunk (M x ldt): transposed planes, kept for the weight contraction
    float *Phi, *Plo;                // (Rc x ld2m)
    float *PThi, *PTlo;              // (2M x ldt)
    float *Kbar;                     // (Rc x ldk)
    long Rc, ldk, ld2m, ldt;
};

inline long chunk_rows(long R) { return R < TC_ROW_CHUNK ? R : TC_ROW_CHUNK; }

// the planes of the step workspace, carved after its FP64 region
inline StepPlanes step_planes(Carve& c, int M) {
    StepPlanes s;
    s.ldk = pad4(M); s.ld2m = pad4(2L * M);
    s.Whi = c.take<float>(2L * M * s.ldk);
    s.Wlo = c.take<float>(2L * M * s.ldk);
    s.Wthi = c.take<float>((long)M * s.ld2m);
    s.Wtlo = c.take<float>((long)M * s.ld2m);
    s.u = c.take<double>(M);
    return s;
}

inline BatchPlanes batch_planes(Carve& c, int M, long R) {
    BatchPlanes b;
    b.Rc = chunk_rows(R); b.ldk = pad4(M); b.ld2m = pad4(2L * M); b.ldt = pad4(b.Rc);
    const long nch = (R + b.Rc - 1) / b.Rc;
    b.AB = c.take<float>(R * b.ld2m);
    b.Khi = c.take<float>(R * b.ldk); b.Klo = c.take<float>(R * b.ldk);
    b.KThi = c.take<float>(nch * (long)M * b.ldt); b.KTlo = c.take<float>(nch * (long)M * b.ldt);
    b.Phi = c.take<float>(b.Rc * b.ld2m); b.Plo = c.take<float>(b.Rc * b.ld2m);
    b.PThi = c.take<float>(2L * M * b.ldt); b.PTlo = c.take<float>(2L * M * b.ldt);
    b.Kbar = c.take<float>(b.Rc * b.ldk);
    return b;
}

inline int make_step_planes(const StepView& v, const StepPlanes& s, cudaStream_t st) {
    dim3 grid((unsigned)cdiv(v.M, 32), (unsigned)cdiv(v.M, 32));
    k_make_w_planes<<<grid, 256, 0, st>>>(v.Linv, v.Cm, v.Mp, v.M, s.Whi, s.Wlo, s.ldk, s.Wthi, s.Wtlo, s.ld2m);
    TGP_TRY(check_launch("k_make_w_planes"));
    k_linvT_m<<<(unsigned)cdiv(v.M, 32), 256, 0, st>>>(v.Linv, v.Mp, v.mvec, v.M, s.u);
    return check_launch("k_linvT_m");
}

inline int row_grid128(long R) {
    const long blocks = cdiv(R, 4);
    return (int)(blocks < 148 * 16 ? blocks : 148 * 16);
}

// forward: K planes per chunk -> [A | B] = K [Linv; C]^T on tcgen05 -> row statistics.  The K generation reads u = L^-T m:
// it joins the factorisation first.
inline int qf_forward(const StepView& s, const StepPlanes& sp, const BatchPlanes& b, const double* X, long R, double* mu, double* v,
                      cudaStream_t st) {
    const int M = s.M, D = s.D;
    if (join_factor(st)) return set_error(-100, "join with the factorisation failed");
    // mu = K_xz (L^-T m) is accumulated in FP64 by the K generation
    cudaMemsetAsync(mu, 0, (size_t)R * sizeof(double), st);
    TGP_TRY(with_kernel(s.kind, [&](auto k) {
        for (long r0 = 0; r0 < R; r0 += b.Rc) {
            const int rc = (int)((R - r0) < b.Rc ? (R - r0) : b.Rc);
            const long kt_off = (r0 / b.Rc) * (long)M * b.ldt;
            float *Khi = b.Khi + r0 * b.ldk, *Klo = b.Klo + r0 * b.ldk;
            TGP_TRY(launch_rbf_planes<decltype(k)::value>(X + r0 * D, s.Zs, s.ls, s.os, rc, M, D, Khi, Klo, b.ldk, b.KThi + kt_off,
                                                          b.KTlo + kt_off, b.ldt, st, sp.u, mu + r0));
            Params p{};
            p.Mrows = rc; p.Ncols = 2 * M; p.K = M;
            p.tri_mode = 1; p.tri_rows = M;
            p.out_mode = 0; p.lower_rows = 0; p.Cf = b.AB + r0 * b.ld2m; p.Cd = nullptr; p.ldc = b.ld2m; p.splitk = 1;
            Operand A{Khi, Klo, rc, M, b.ldk};
            Operand B{sp.Whi, sp.Wlo, 2L * M, M, sp.ldk};
            TGP_TRY(gemm_tf32x3(A, B, p, st));
        }
        return 0;
    }));
    k_row_stats_f32<<<row_grid128(R), 128, 0, st>>>(b.AB, b.ld2m, s.os, (int)R, M, v);
    return check_launch("k_row_stats_f32");
}

// backward: ABbar planes (+transposes), K^T planes; Kbar = ABbar Wt^T; kernel gradients; Gbar / Cbar += ABbar^T K
template <int KIND>
inline int qf_backward_k(const StepView& s, const StepPlanes& sp, const BatchPlanes& b, const double* X, long R, const double* g_mu,
                         const double* g_v, double* dm, double* dos, double* dZ, double* dls, double* Gbar, double* Cbar, double* dX,
                         cudaStream_t st) {
    const int M = s.M, D = s.D;
    for (long r0 = 0; r0 < R; r0 += b.Rc) {
        const int rc = (int)((R - r0) < b.Rc ? (R - r0) : b.Rc);
        {
            dim3 grid((unsigned)cdiv(M, 64), (unsigned)cdiv(rc, 32));
            k_make_abbar_planes<<<grid, 256, 0, st>>>(b.AB + r0 * b.ld2m, b.ld2m, g_mu + r0, g_v + r0, s.mvec, rc, M, b.Phi,
                                                      b.Plo, b.ld2m, b.PThi, b.PTlo, b.ldt, dm, dos);
            TGP_TRY(check_launch("k_make_abbar_planes"));
        }
        const long kt_off = (r0 / b.Rc) * (long)M * b.ldt;          // K^T planes of this chunk, kept by the forward
        float *KThi = b.KThi + kt_off, *KTlo = b.KTlo + kt_off;
        {   // Kbar (rc x M) = ABbar (rc x 2M) * Wt (M x 2M)^T ; for k < M only k >= n contributes
            Params p{};
            p.Mrows = rc; p.Ncols = M; p.K = 2 * M;
            p.tri_mode = 2; p.tri_rows = M;
            p.out_mode = 0; p.Cf = b.Kbar; p.ldc = b.ldk; p.splitk = 1;
            Operand A{b.Phi, b.Plo, rc, 2L * M, b.ld2m};
            Operand B{sp.Wthi, sp.Wtlo, M, 2L * M, sp.ld2m};
            TGP_TRY(gemm_tf32x3(A, B, p, st));
        }
        // the RBF reads K from the planes; the other kinds recompute it (launch_kernel_grads)
        TGP_TRY((launch_kernel_grads<KIND, float>(b.Kbar, b.ldk, X + r0 * D, 0, s.Zs, s.ls, s.os, rc, M, D, 0, 1.0, dZ, dls, dos, st,
                                                  nullptr, 0, b.Khi + r0 * b.ldk, b.Klo + r0 * b.ldk, b.ldk)));
        if (dX) TGP_TRY(launch_input_grads<KIND>(b.Kbar, b.ldk, X + r0 * D, s.Zs, s.ls, s.os, rc, M, D, dX + r0 * D, st));
        const int kblocks = (rc + BK - 1) / BK;
        int split = (int)cdiv(2 * 148, cdiv(M, BM) * cdiv(M, BN));
        if (split > kblocks / 8) split = kblocks / 8 > 0 ? kblocks / 8 : 1;
        {   // Gbar (M x M, lower) += Abar^T K : operands ABbar^T rows [0, M) and K^T, reduction over the chunk rows
            Params p{};
            p.Mrows = M; p.Ncols = M; p.K = rc;
            p.tri_mode = 0; p.out_mode = 1; p.lower_rows = M; p.Cd = Gbar; p.ldc = s.Mp; p.splitk = split;
            Operand A{b.PThi, b.PTlo, M, rc, b.ldt};
            Operand B{KThi, KTlo, M, rc, b.ldt};
            TGP_TRY(gemm_tf32x3(A, B, p, st));
        }
        {   // Cbar (M x M) += Bbar^T K
            Params p{};
            p.Mrows = M; p.Ncols = M; p.K = rc;
            p.tri_mode = 0; p.out_mode = 1; p.lower_rows = 0; p.Cd = Cbar; p.ldc = s.Mp; p.splitk = split;
            Operand A{b.PThi + (long)M * b.ldt, b.PTlo + (long)M * b.ldt, M, rc, b.ldt};
            Operand B{KThi, KTlo, M, rc, b.ldt};
            TGP_TRY(gemm_tf32x3(A, B, p, st));
        }
    }
    return 0;
}

inline int qf_backward(const StepView& s, const StepPlanes& sp, const BatchPlanes& b, const double* X, long R, const double* g_mu,
                       const double* g_v, double* dm, double* dos, double* dZ, double* dls, double* Gbar, double* Cbar, double* dX,
                       cudaStream_t st) {
    return with_kernel(s.kind, [&](auto k) {
        return qf_backward_k<decltype(k)::value>(s, sp, b, X, R, g_mu, g_v, dm, dos, dZ, dls, Gbar, Cbar, dX, st);
    });
}

}  // namespace tc
}  // namespace tgp
