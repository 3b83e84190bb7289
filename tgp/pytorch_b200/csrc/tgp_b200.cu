// C-ABI entry points (include/tgp_b200.h) — host-side orchestration of the sm_100a kernels.
#include <cstdlib>
#include "../../../include/tgp_b200.h"
#include "common.cuh"
#include "gemm_f64.cuh"
#include "step_kernels.cuh"
#include "row_kernels.cuh"
#include "backward_kernels.cuh"
#include "f64_driver.cuh"
#include "cov_kernels.cuh"
#include "tc_driver.cuh"
#include "flow_mlp.cuh"
#include "crt_driver.cuh"
#include "eval_kernels.cuh"
#include "kmeans.cuh"
#include "mc_kernels.cuh"

namespace tgp {
char g_last_error[512] = "";
long g_launch_count = 0;
GemmTimer g_gemm_timer;
int g_overlap_kgen = 1;

inline long even(long x) { return (x + 1) / 2 * 2; }

inline TgpReduceLayout reduce_layout(const TgpModel* md) {
    TgpReduceLayout l;
    const long Mp = pad_M(md->M);
    l.ell_sum = 0; l.dlogvar = 1; l.dos = 2;
    l.dls = 4;
    l.dtheta = l.dls + even(md->D);
    l.dm = l.dtheta + even(md->n_theta);
    l.dZ = l.dm + even(md->M);
    l.Gbar = l.dZ + even((long)md->M * md->D);
    l.Cbar = l.Gbar + Mp * Mp;
    l.total = l.Cbar + Mp * Mp;
    const long M = md->M, tri = M * (M + 1) / 2;
    l.packed_total = l.Gbar + tri + (md->dtype != TGP_F64 ? M * M : tri);
    return l;
}

// reduce buffer <-> tril-packed exchange buffer (one CTA per matrix row; dir 0 = pack, 1 = unpack)
__global__ void __launch_bounds__(256) k_reduce_pack(double* __restrict__ rb, double* __restrict__ packed, long small, long offG,
                                                     long offC, int M, long Mp, int second_dense, int dir) {
    const long tri = (long)M * (M + 1) / 2;
    const int r = blockIdx.x;
    if (r == M) {                                   // the small leading vector
        for (long i = threadIdx.x; i < small; i += blockDim.x) { if (dir) rb[i] = packed[i]; else packed[i] = rb[i]; }
        return;
    }
    double* pg = packed + small + (long)r * (r + 1) / 2;
    double* g = rb + offG + (long)r * Mp;
    for (int c = threadIdx.x; c <= r; c += blockDim.x) { if (dir) g[c] = pg[c]; else pg[c] = g[c]; }
    double* pc = packed + small + tri + (second_dense ? (long)r * M : (long)r * (r + 1) / 2);
    double* cc = rb + offC + (long)r * Mp;
    const int nc = second_dense ? M : r + 1;
    for (int c = threadIdx.x; c < nc; c += blockDim.x) { if (dir) cc[c] = pc[c]; else pc[c] = cc[c]; }
}

inline int reduce_pack(const TgpModel* md, double* rb, double* packed, int dir, cudaStream_t st) {
    const TgpReduceLayout l = reduce_layout(md);
    k_reduce_pack<<<md->M + 1, 256, 0, st>>>(rb, packed, l.Gbar, l.Gbar, l.Cbar, md->M, pad_M(md->M), md->dtype != TGP_F64, dir);
    return check_launch("k_reduce_pack");
}

inline int validate(const TgpModel* md) {
    if (!md) return set_error(-1, "model is NULL");
    if (md->dtype != TGP_F64 && md->dtype != TGP_F32 && md->dtype != TGP_F64_I8)
        return set_error(-1, "dtype must be TGP_F64, TGP_F32 or TGP_F64_I8");
    if (md->M < 1 || md->D < 1) return set_error(-1, "M and D must be positive");
    if (!kernel_kind_valid(md->kernel))
        return set_error(-1, "kernel must be TGP_KERNEL_RBF, TGP_KERNEL_MATERN12, TGP_KERNEL_MATERN32 or TGP_KERNEL_MATERN52");
    if (md->q_u_form != TGP_QU_WHITENED && md->q_u_form != TGP_QU_UNWHITENED)
        return set_error(-1, "q_u_form must be TGP_QU_WHITENED or TGP_QU_UNWHITENED");
    if (md->n_layers < 0 || md->n_layers > TGP_MAX_LAYERS) return set_error(-1, "too many flow layers");
    if (md->n_theta < 0 || md->n_theta > MAX_THETA) return set_error(-1, "too many global flow parameters");
    if (md->n_rowparams < 0 || md->n_rowparams > MAX_ROWP) return set_error(-1, "too many per-row flow parameters");
    if (md->likelihood < 0 || md->likelihood > TGP_LIK_GAUSS_WARPED) return set_error(-1, "unknown likelihood");
    if (md->likelihood == TGP_LIK_GAUSS_LINEAR && md->n_layers != 0)
        return set_error(-1, "the closed-form Gaussian likelihood takes an identity flow");
    if (md->likelihood != TGP_LIK_GAUSS_LINEAR && (md->n_quad < 1 || md->n_quad > 4096))
        return set_error(-1, "n_quad out of range");
    if (md->likelihood == TGP_LIK_GAUSS_WARPED) {
        if (md->n_rowparams != 0) return set_error(-1, "the warped likelihood takes a warp with global parameters only");
        for (int i = 0; i < md->n_layers; ++i)
            if (md->layers[i].flags & TGP_FLOW_PER_ROW)
                return set_error(-1, "input-dependent warps (TGP_FLOW_PER_ROW) are outside the warped likelihood");
    }
    for (int i = 0, left = 0; i < md->n_layers; ++i) {          // step groups: header + exactly n_steps member layers
        const TgpFlowLayer& L = md->layers[i];
        if (L.kind < 0 || L.kind > TGP_FLOW_STEP_GROUP) return set_error(-1, "unknown flow layer kind");
        if ((L.flags & TGP_FLOW_SWITCH) && (L.flags & TGP_FLOW_PER_ROW))
            return set_error(-1, "a switch_off member cannot take per-row parameters");
        if (L.kind == TGP_FLOW_STEP_GROUP) {
            if (left) return set_error(-1, "step groups cannot nest");
            if (L.n_steps < 1 || i + L.n_steps > md->n_layers - 1)
                return set_error(-1, "step group runs past the last layer");
            left = L.n_steps;
        } else if (left) {
            if (L.kind == TGP_FLOW_AFFINE || L.kind == TGP_FLOW_IDENTITY)
                return set_error(-1, "affine / identity layers cannot be step members");
            --left;
        } else if (L.flags & TGP_FLOW_SWITCH) return set_error(-1, "switch_off outside a step group");
    }
    return 0;
}

inline void fill_flow(FlowDesc& fd, const TgpModel* md) {
    fd.n_layers = md->n_layers;
    for (int i = 0; i < md->n_layers; ++i) fd.layers[i] = md->layers[i];
}

// M x M x M products of the per-step chain have only (M/128)^2 output tiles: split their reduction (FP64 atomics into a
// zeroed output) so that one launch fills the SMs instead of running 36-64 long CTAs.
inline int gemm_small(GemmArgs g, cudaStream_t st) {
    const long tiles = gemm_tiles(g.M, g.N, g.c_lower != 0);
    long split = tiles > 0 ? (GEMM_SLOTS + tiles - 1) / tiles : 1;
    const long max_split = g.K / (4 * GBK) > 0 ? g.K / (4 * GBK) : 1;
    if (split > max_split) split = max_split;
    if (split > 1 && g.batch == 1) {
        if (g.beta == 0.0) {
            cudaMemset2DAsync(g.C, (size_t)g.ldc * sizeof(double), 0, (size_t)g.N * sizeof(double), (size_t)g.M, st);
            g.beta = 1.0;
        }
        if (g.beta == 1.0) g.splitk = (int)split;
    }
    return gemm_f64(g, st);
}

// The step workspace: the FP64 region, then the planes of the active tensor-core mode (TGP_F64 has none), then tril(L_raw)
// of a non-whitened model
struct StepWorkspace { StepView f64; tc::StepPlanes tc; crt::StepPlanes crt; };
inline StepWorkspace step_layout(Carve& c, const TgpModel* md) {
    StepWorkspace w{};
    w.f64 = step_view(c, md->M, md->D);
    w.f64.kind = md->kernel;
    if (md->dtype == TGP_F32) w.tc = tc::step_planes(c, md->M);
    if (md->dtype == TGP_F64_I8) w.crt = crt::step_planes(c, md->M);
    if (md->q_u_form == TGP_QU_UNWHITENED) w.f64.P = c.take<double>((size_t)w.f64.Mp * w.f64.Mp);
    return w;
}
}  // namespace tgp

using namespace tgp;

extern "C" {

const char* tgp_last_error(void) { return g_last_error; }
int tgp_version(void) { return 102; }

size_t tgp_step_workspace_bytes(const TgpModel* md) {
    if (validate(md)) return 0;
    Carve c(nullptr);
    step_layout(c, md);
    return c.bytes();
}

size_t tgp_batch_workspace_bytes(const TgpModel* md, long R) {
    if (validate(md) || R < 0) return 0;
    Carve c(nullptr);
    if (md->dtype == TGP_F32) tc::batch_planes(c, md->M, R);
    else if (md->dtype == TGP_F64_I8) crt::batch_view(c, md->M, md->D, R);
    else f64::batch_view(c, md->M, R);
    return c.bytes();
}

int tgp_reduce_layout(const TgpModel* md, TgpReduceLayout* out) {
    TGP_TRY(validate(md));
    if (!out) return set_error(-1, "out is NULL");
    *out = reduce_layout(md);
    return 0;
}

// fork of tgp_prepare: the factorisation's stream (the library's high-priority stream, ordered after everything enqueued on
// `st` so far), or `st` itself when the overlap is off / the fork fails
static cudaStream_t g_factor_stream = nullptr;
static cudaStream_t fork_factor(cudaStream_t st) {
    g_factor_stream = st;
    if (!g_overlap_kgen) return st;
    SideStream& ss = side_stream();
    if (cudaEventRecord(ss.ev_fork, st) != cudaSuccess || cudaStreamWaitEvent(ss.hp, ss.ev_fork, 0) != cudaSuccess) {
        cudaGetLastError();
        return st;
    }
    g_factor_stream = ss.hp;
    return ss.hp;
}

int tgp_prepare(const TgpModel* md, const TgpParams* p, double jitter, void* step_ws, double* kl_out, int* status,
                void* stream) {
    TGP_TRY(validate(md));
    if (!p || !step_ws || !kl_out || !status) return set_error(-1, "NULL argument to tgp_prepare");
    cudaStream_t st = (cudaStream_t)stream;
    if (join_factor(st)) return set_error(-100, "join with the previous factorisation failed");      // it may still use this workspace
    Carve c(step_ws);
    const StepWorkspace w = step_layout(c, md);
    TGP_TRY(run_prepare(w.f64, (const double*)p->Z, (const double*)p->raw_lengthscale, (const double*)p->raw_outputscale,
                        (const double*)p->m, (const double*)p->L_raw, jitter, kl_out, status, md->dtype != TGP_F64, st, fork_factor));
    cudaStream_t fst = g_factor_stream;
    if (md->dtype == TGP_F32) TGP_TRY(tc::make_step_planes(w.f64, w.tc, fst));
    if (md->dtype == TGP_F64_I8) TGP_TRY(crt::make_step_planes(w.f64, w.crt, fst));
    SideStream& ss = side_stream();
    ss.status_valid = false;
    if (!stream_is_capturing(st)) {          // the pivot status travels to pinned host memory behind the factorisation alone
        cudaMemcpyAsync(ss.status_host, status, sizeof(int), cudaMemcpyDeviceToHost, fst);
        ss.status_valid = cudaEventRecord(ss.ev_status, fst) == cudaSuccess;
    }
    if (fst != st) {
        if (cudaEventRecord(ss.ev_factor, fst) != cudaSuccess) return set_error(-100, "recording the factorisation event failed");
        ss.pending = true;
    }
    return 0;
}

int tgp_factor_status(int* status_out) {
    SideStream& ss = side_stream();
    if (!status_out) return set_error(-1, "status_out is NULL");
    if (!ss.status_valid) return set_error(-1, "no factorisation status in flight (tgp_prepare under graph capture records none)");
    if (cudaEventSynchronize(ss.ev_status) != cudaSuccess) return set_error(-100, "waiting for the factorisation failed");
    *status_out = *ss.status_host;
    return 0;
}

// Each mode's qf_forward joins the factorisation as soon as it has enqueued the work that does not need it
int tgp_qf_forward(const TgpModel* md, const void* step_ws, void* batch_ws, const void* X, long R, void* mu, void* v,
                   void* stream) {
    TGP_TRY(validate(md));
    if (R <= 0) return 0;
    if (!step_ws || !batch_ws || !X || !mu || !v) return set_error(-1, "NULL argument to tgp_qf_forward");
    cudaStream_t st = (cudaStream_t)stream;
    const int M = md->M, D = md->D;
    Carve cs(const_cast<void*>(step_ws)), cb(batch_ws);
    const StepWorkspace w = step_layout(cs, md);
    const double* Xd = (const double*)X;
    if (md->dtype == TGP_F32) return tc::qf_forward(w.f64, w.tc, tc::batch_planes(cb, M, R), Xd, R, (double*)mu, (double*)v, st);
    if (md->dtype == TGP_F64_I8)
        return crt::qf_forward(w.f64, w.crt, crt::batch_view(cb, M, D, R), Xd, R, (double*)mu, (double*)v, st);
    return f64::qf_forward(w.f64, f64::batch_view(cb, M, R), Xd, R, (double*)mu, (double*)v, st);
}

size_t tgp_qf_cov_workspace_bytes(const TgpModel* md, long R) {
    if (validate(md) || R < 1) return 0;
    Carve c(nullptr);
    cov::cov_view(c, md->M, R);
    return c.bytes();
}

// Reads the step workspace only (any compute mode; the batch workspace is not touched), joins the factorisation after
// enqueuing the K_xz generation
int tgp_qf_cov_forward(const TgpModel* md, const void* step_ws, void* cov_ws, const void* X, long R, void* mu, void* cov,
                       long ldc, void* stream) {
    TGP_TRY(validate(md));
    if (R < 1) return set_error(-1, "R must be >= 1");
    if (ldc < R) return set_error(-1, "ldc must be >= R");
    if (!step_ws || !cov_ws || !X || !mu || !cov) return set_error(-1, "NULL argument to tgp_qf_cov_forward");
    Carve cs(const_cast<void*>(step_ws)), cw(cov_ws);
    const StepWorkspace w = step_layout(cs, md);
    return cov::qf_cov_forward(w.f64, cov::cov_view(cw, md->M, R), (const double*)X, R, (double*)mu, (double*)cov, ldc,
                               (cudaStream_t)stream);
}

size_t tgp_cov_cholesky_workspace_bytes(long R) {
    if (R < 1) return 0;
    Carve c(nullptr);
    cov::chol_view(c, R);
    return c.bytes();
}

int tgp_cov_cholesky(long R, const void* cov, long ldc, double jitter, const double* scale_dev, void* chol_ws, void* L, long ldl,
                     int* status, void* stream) {
    if (R < 1) return set_error(-1, "R must be >= 1");
    if (ldc < R || ldl < R) return set_error(-1, "ldc and ldl must be >= R");
    if (!(jitter >= 0.0)) return set_error(-1, "jitter must be >= 0");
    if (!cov || !scale_dev || !chol_ws || !L || !status) return set_error(-1, "NULL argument to tgp_cov_cholesky");
    Carve c(chol_ws);
    return cov::cholesky(cov::chol_view(c, R), R, (const double*)cov, ldc, jitter, scale_dev, (double*)L, ldl, status,
                         (cudaStream_t)stream);
}

int tgp_cov_sample(long R, int S, const void* mu, const void* L, long ldl, const void* eps, void* out, void* stream) {
    if (R < 1 || S < 1) return set_error(-1, "R and S must be >= 1");
    if (ldl < R) return set_error(-1, "ldl must be >= R");
    if (!mu || !L || !eps || !out) return set_error(-1, "NULL argument to tgp_cov_sample");
    return cov::sample(R, S, (const double*)mu, (const double*)L, ldl, (const double*)eps, (double*)out, (cudaStream_t)stream);
}

int tgp_ell_forward(const TgpModel* md, const TgpParams* p, const void* mu, const void* v, const void* Y,
                    const void* rowparams, long R, double scale, const void* quad_t, const void* quad_w, int want_grad,
                    void* ell_rows, void* g_mu, void* g_v, void* drowparams, double* reduce_buf, void* stream) {
    TGP_TRY(validate(md));
    if (R <= 0) return 0;
    if (!p || !mu || !v || !Y || !ell_rows || !reduce_buf) return set_error(-1, "NULL argument to tgp_ell_forward");
    if (want_grad && (!g_mu || !g_v)) return set_error(-1, "g_mu / g_v required when want_grad");
    if (md->n_rowparams > 0 && (!rowparams || (want_grad && !drowparams)))
        return set_error(-1, "rowparams / drowparams required for input-dependent flows");
    const bool warped = md->likelihood == TGP_LIK_GAUSS_WARPED;
    if (md->likelihood != TGP_LIK_GAUSS_LINEAR && !warped && (!quad_t || !quad_w)) return set_error(-1, "quadrature rule missing");
    if (warped && md->n_theta > 0 && !p->theta) return set_error(-1, "theta required for the warp");
    const TgpReduceLayout l = reduce_layout(md);
    RowQuadArgs a;
    a.R = (int)R; a.likelihood = md->likelihood; a.n_quad = md->n_quad; a.n_theta = md->n_theta;
    a.n_rowp = md->n_rowparams; a.want_grad = want_grad; a.scale = scale;
    a.mu = (const double*)mu; a.v = (const double*)v; a.y = (const double*)Y;
    a.log_var_noise = (const double*)p->log_var_noise; a.theta = (const double*)p->theta;
    a.rowp = md->n_rowparams > 0 ? (const double*)rowparams : nullptr;
    a.qt = (const double*)quad_t; a.qw = (const double*)quad_w;
    a.ell_rows = (double*)ell_rows; a.g_mu = (double*)g_mu; a.g_v = (double*)g_v;
    a.ell_sum = reduce_buf + l.ell_sum; a.dlogvar = reduce_buf + l.dlogvar; a.dtheta = reduce_buf + l.dtheta;
    a.drowp = (double*)drowparams;
    fill_flow(a.flow, md);
    if (warped) {
        const long blocks = cdiv(R, ROW_THREADS);
        k_row_warped<<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), ROW_THREADS, 0, (cudaStream_t)stream>>>(a);
        return check_launch("k_row_warped");
    }
    k_row_quad<<<row_grid(R), ROW_THREADS, 0, (cudaStream_t)stream>>>(a);
    return check_launch("k_row_quad");
}

int tgp_qf_backward(const TgpModel* md, const TgpParams* p, const void* step_ws, void* batch_ws, const void* X,
                    long R, const void* g_mu, const void* g_v, double* reduce_buf, void* stream) {
    return tgp_qf_backward_dx(md, p, step_ws, batch_ws, X, R, g_mu, g_v, reduce_buf, nullptr, stream);
}

int tgp_qf_backward_dx(const TgpModel* md, const TgpParams* p, const void* step_ws, void* batch_ws, const void* X,
                       long R, const void* g_mu, const void* g_v, double* reduce_buf, void* dX, void* stream) {
    TGP_TRY(validate(md));
    if (R <= 0) return 0;
    if (!p || !step_ws || !batch_ws || !X || !g_mu || !g_v || !reduce_buf)
        return set_error(-1, "NULL argument to tgp_qf_backward");
    if (dX && md->D > 64) return set_error(-2, "input gradients need D <= 64");
    cudaStream_t st = (cudaStream_t)stream;
    const int M = md->M, D = md->D;
    Carve cs(const_cast<void*>(step_ws)), cb(batch_ws);
    const StepWorkspace w = step_layout(cs, md);
    const TgpReduceLayout l = reduce_layout(md);
    const double* Xd = (const double*)X;
    const double *gm = (const double*)g_mu, *gv = (const double*)g_v;
    double *dm = reduce_buf + l.dm, *dos = reduce_buf + l.dos, *dZ = reduce_buf + l.dZ, *dls = reduce_buf + l.dls;
    double *Gbar = reduce_buf + l.Gbar, *Cbar = reduce_buf + l.Cbar;
    double* dXd = (double*)dX;
    if (join_factor(st)) return set_error(-100, "join with the factorisation failed");
    if (md->dtype == TGP_F32)
        return tc::qf_backward(w.f64, w.tc, tc::batch_planes(cb, M, R), Xd, R, gm, gv, dm, dos, dZ, dls, Gbar, Cbar, dXd, st);
    if (md->dtype == TGP_F64_I8)
        return crt::qf_backward(w.f64, w.crt, crt::batch_view(cb, M, D, R), Xd, R, gm, gv, dm, dos, dZ, dls, Gbar, Cbar, dXd, st);
    return f64::qf_backward(w.f64, f64::batch_view(cb, M, R), Xd, R, gm, gv, dm, dos, dZ, dls, Gbar, Cbar, dXd, st);
}

int tgp_chain_backward(const TgpModel* md, const TgpParams* p, void* step_ws, const double* reduce_buf, double gE,
                       double gK, const double* g_dev, void* dZ, void* draw_ls, void* draw_os, void* dm, void* dL_raw, void* dlogvar,
                       void* dtheta, void* stream) {
    TGP_TRY(validate(md));
    if (!p || !step_ws || !reduce_buf || !dZ || !draw_ls || !draw_os || !dm || !dL_raw)
        return set_error(-1, "NULL argument to tgp_chain_backward");
    if (md->n_theta > 0 && !dtheta) return set_error(-1, "dtheta required");
    cudaStream_t st = (cudaStream_t)stream;
    if (join_factor(st)) return set_error(-100, "join with the factorisation failed");
    const int M = md->M, D = md->D, Mp = pad_M(md->M);
    const size_t mm = (size_t)Mp * Mp;
    Carve c(step_ws);
    const StepView s = step_layout(c, md).f64;
    const TgpReduceLayout l = reduce_layout(md);
    const double* Cbar = reduce_buf + l.Cbar;
    double* Gtot = s.Kzz;                          // K_zz's buffer is free after the factorisation
    double* dZacc = s.S3;                          // (M*D) accumulators live at the head of S3 until Phi needs it

    if (md->dtype != TGP_F64) {
        // tensor-core modes carry C = L_S^T L^-1:  dLS = tril(Linv * Cbar^T),  Gtot = Gbar + tril(LS * Cbar)
        GemmArgs a1 = make_gemm(M, M, M, s.Linv, Mp, 0, Cbar, Mp, 0, s.S0, Mp);
        a1.a_tri = 1; a1.c_lower = 1;
        cudaMemsetAsync(s.S0, 0, mm * sizeof(double), st);
        TGP_TRY(gemm_small(a1, st));
        cudaMemcpyAsync(Gtot, reduce_buf + l.Gbar, mm * sizeof(double), cudaMemcpyDeviceToDevice, st);
        GemmArgs a2 = make_gemm(M, M, M, s.LS, Mp, 0, Cbar, Mp, 1, Gtot, Mp, 1.0, 1.0);
        a2.a_tri = 1; a2.c_lower = 1;
        TGP_TRY(gemm_small(a2, st));
    } else {
        // FP64 mode: the batch pass already accumulated dL_S (in the Cbar slot) and the complete Gbar
        cudaMemcpyAsync(s.S0, Cbar, mm * sizeof(double), cudaMemcpyDeviceToDevice, st);
        cudaMemcpyAsync(Gtot, reduce_buf + l.Gbar, mm * sizeof(double), cudaMemcpyDeviceToDevice, st);
    }
    const bool unwhitened = s.P != nullptr;
    if (unwhitened) {
        // S0 and Gtot hold dELL/dL_S and dELL/dL^-1 of the whitened pair (m~, P~) = (L^-1 m, L^-1 P).  With its adjoints
        // m~bar, P~bar (k_unwhiten_adjoints):  dm = L^-T m~bar,  dP = tril(L^-T P~bar),  dL^-1 = gE Gtot + tril(m~bar m^T + P~bar P^T).
        // gE and gK both enter Gtot here, before the Murray chain; the final kernel does not scale the K_zz side again.
        double* mbar = s.S3;                       // S3 is free until Phi
        k_unwhiten_adjoints<<<M, 256, 0, st>>>(s.S0, s.LS, Gtot, Mp, M, reduce_buf + l.dm, s.mvec, (const double*)p->m, gE, gK,
                                               g_dev, mbar);
        TGP_TRY(check_launch("k_unwhiten_adjoints"));
        // Gtot += tril(P~bar P^T)   (Aop[m,k] = P~bar[m,k], nonzero k <= m;  Bop[n,k] = P[n,k], nonzero k <= n)
        GemmArgs u1 = make_gemm(M, M, M, s.S0, Mp, 0, s.P, Mp, 0, Gtot, Mp, 1.0, 1.0);
        u1.a_tri = 1; u1.b_tri = 1; u1.c_lower = 1;
        TGP_TRY(gemm_small(u1, st));
        k_trmv_lower<<<M, 256, 0, st>>>(s.Linv, Mp, M, mbar, (double*)dm, 1);
        TGP_TRY(check_launch("k_trmv_lower"));
        // dL_raw = tril(L^-T P~bar)   (Aop[m,k] = Linv[k,m], nonzero k >= m;  Bop[n,k] = P~bar[k,n], nonzero k >= n)
        cudaMemsetAsync(dL_raw, 0, (size_t)M * M * sizeof(double), st);
        GemmArgs u2 = make_gemm(M, M, M, s.Linv, Mp, 1, s.S0, Mp, 1, (double*)dL_raw, M, 1.0, 1.0);
        u2.a_tri = 2; u2.b_tri = 2; u2.c_lower = 1;
        TGP_TRY(gemm_small(u2, st));
    }
    // T1 = Gtot * Linv^T
    GemmArgs a3 = make_gemm(M, M, M, Gtot, Mp, 0, s.Linv, Mp, 0, s.S1, Mp);
    a3.a_tri = 1; a3.b_tri = 1;
    TGP_TRY(gemm_small(a3, st));
    // Lbar = -tril(Linv^T * T1)
    cudaMemsetAsync(s.S2, 0, mm * sizeof(double), st);
    GemmArgs a4 = make_gemm(M, M, M, s.Linv, Mp, 1, s.S1, Mp, 1, s.S2, Mp, -1.0, 0.0);
    a4.a_tri = 2; a4.c_lower = 1;
    TGP_TRY(gemm_small(a4, st));
    // Phi = tril(L^T * Lbar), diagonal halved      (Murray 2016; equals torch's cholesky_backward)
    cudaMemsetAsync(s.S3, 0, mm * sizeof(double), st);
    GemmArgs a5 = make_gemm(M, M, M, s.L, Mp, 1, s.S2, Mp, 1, s.S3, Mp);
    a5.a_tri = 2; a5.b_tri = 2; a5.c_lower = 1;
    TGP_TRY(gemm_small(a5, st));
    k_halve_diag<<<(unsigned)cdiv(M, 256), 256, 0, st>>>(s.S3, Mp, M);
    // S1 = Phi * Linv ;  Kbar_zz = Linv^T * S1  (symmetrised on the fly by the gradient kernel)
    GemmArgs a6 = make_gemm(M, M, M, s.S3, Mp, 0, s.Linv, Mp, 1, s.S1, Mp);
    a6.a_tri = 1; a6.b_tri = 2;
    TGP_TRY(gemm_small(a6, st));
    GemmArgs a7 = make_gemm(M, M, M, s.Linv, Mp, 1, s.S1, Mp, 1, s.S2, Mp);
    a7.a_tri = 2;
    TGP_TRY(gemm_small(a7, st));
    // K_zz -> Z (both index roles: factor 2 on the symmetrised matrix), lengthscale, outputscale.
    // accumulators: start from the K_xz-side sums of the reduce buffer (whitened)
    dZacc = s.S3;   // Phi is dead now
    double* dls_acc = dZacc + even((long)M * D);
    double* dos_acc = dls_acc + even(D);
    if (unwhitened) {   // the K_zz side alone (it carries gE and gK); the final kernel adds gE times the K_xz-side sums
        cudaMemsetAsync(dZacc, 0, (size_t)(even((long)M * D) + even(D) + 1) * sizeof(double), st);
    } else {
        cudaMemcpyAsync(dZacc, reduce_buf + l.dZ, (size_t)M * D * sizeof(double), cudaMemcpyDeviceToDevice, st);
        cudaMemcpyAsync(dls_acc, reduce_buf + l.dls, (size_t)D * sizeof(double), cudaMemcpyDeviceToDevice, st);
        cudaMemcpyAsync(dos_acc, reduce_buf + l.dos, sizeof(double), cudaMemcpyDeviceToDevice, st);
    }
    TGP_TRY(with_kernel(s.kind, [&](auto k) {
        return launch_kernel_grads<decltype(k)::value>(s.S2, Mp, s.Zs, 1, s.Zs, s.ls, s.os, M, M, D, 1, 2.0, dZacc, dls_acc, dos_acc, st);
    }));
    if (unwhitened) {
        const int n = M * D > md->n_theta ? M * D : md->n_theta;
        k_finalize_small_unwhitened<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(
            (const double*)p->raw_lengthscale, (const double*)p->raw_outputscale, M, D, md->n_theta, gE, g_dev, dZacc, dls_acc,
            dos_acc, reduce_buf + l.dZ, reduce_buf + l.dls, reduce_buf + l.dos, reduce_buf + l.dlogvar, reduce_buf + l.dtheta,
            (double*)dZ, (double*)draw_ls, (double*)draw_os, (double*)dlogvar, (double*)dtheta);
        return check_launch("k_finalize_small_unwhitened");
    }
    {
        const int n = M * D > M ? M * D : M;
        const int nn = n > md->n_theta ? n : md->n_theta;
        k_finalize_small<<<(unsigned)cdiv(nn, 256), 256, 0, st>>>(
            (const double*)p->raw_lengthscale, (const double*)p->raw_outputscale, (const double*)p->m, M, D,
            md->n_theta, gE, gK, g_dev, dls_acc, dos_acc, reduce_buf + l.dm, dZacc, reduce_buf + l.dlogvar,
            reduce_buf + l.dtheta, (double*)dZ, (double*)draw_ls, (double*)draw_os, (double*)dm, (double*)dlogvar,
            (double*)dtheta);
        TGP_TRY(check_launch("k_finalize_small"));
        k_finalize_LS<<<M, 256, 0, st>>>(s.S0, s.LS, Mp, M, gE, gK, g_dev, (double*)dL_raw);
        TGP_TRY(check_launch("k_finalize_LS"));
    }
    return 0;
}

int tgp_test_rows(const TgpModel* md, const TgpParams* p, const void* mu, const void* v, const void* Y,
                  const void* rowparams, long R, int n_mc, double y_std, const void* quad_t, const void* quad_w,
                  const double* bern_std, void* logp_rows, void* m1, void* m2, void* stream) {
    TGP_TRY(validate(md));
    if (R <= 0) return 0;
    if (!p || !mu || !v || !logp_rows || !m1 || !m2) return set_error(-1, "NULL argument to tgp_test_rows");
    if (n_mc < 1) return set_error(-1, "n_mc must be >= 1");
    if (md->n_rowparams > 0 && !rowparams) return set_error(-1, "rowparams required for input-dependent flows");
    if (md->likelihood == TGP_LIK_BERNOULLI && md->n_layers > 0 && !bern_std)
        return set_error(-1, "bern_std required for Bernoulli with a non-identity flow");
    const bool warped = md->likelihood == TGP_LIK_GAUSS_WARPED;
    if (warped && (!quad_t || !quad_w)) return set_error(-1, "quadrature rule missing (the warped predictive moments use it)");
    if (warped && n_mc != 1) return set_error(-1, "the warped likelihood takes n_mc = 1");
    RowTestArgs a;
    a.R = (int)R; a.likelihood = md->likelihood; a.n_quad = md->n_quad; a.n_rowp = md->n_rowparams; a.n_mc = n_mc;
    a.y_std = y_std;
    a.mu = (const double*)mu; a.v = (const double*)v; a.y = (const double*)Y;
    a.log_var_noise = (const double*)p->log_var_noise; a.theta = (const double*)p->theta;
    a.rowp = md->n_rowparams > 0 ? (const double*)rowparams : nullptr;
    a.qt = (const double*)quad_t; a.qw = (const double*)quad_w; a.bern_std = bern_std;
    a.logp_rows = (double*)logp_rows; a.m1 = (double*)m1; a.m2 = (double*)m2;
    fill_flow(a.flow, md);
    if (warped) k_row_test<true><<<row_grid(R), ROW_THREADS, 0, (cudaStream_t)stream>>>(a);
    else k_row_test<false><<<row_grid(R), ROW_THREADS, 0, (cudaStream_t)stream>>>(a);
    return check_launch("k_row_test");
}

int tgp_flow_inverse(const TgpModel* md, const void* theta, const void* z, long R, void* out, int* n_fail, void* stream) {
    TGP_TRY(validate(md));
    for (int i = 0; i < md->n_layers; ++i)
        if (md->layers[i].flags & TGP_FLOW_PER_ROW) return set_error(-1, "tgp_flow_inverse takes flows with global parameters only");
    if (R <= 0) return 0;
    if (!z || !out || !n_fail || (md->n_theta > 0 && !theta)) return set_error(-1, "NULL argument to tgp_flow_inverse");
    FlowDesc fd;
    fill_flow(fd, md);
    const long blocks = cdiv(R, ROW_THREADS);
    k_flow_inverse<<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), ROW_THREADS, 0, (cudaStream_t)stream>>>(
        fd, (const double*)theta, (const double*)z, R, (double*)out, n_fail);
    return check_launch("k_flow_inverse");
}

int tgp_coverage_rows(const TgpModel* md, const TgpParams* p, const void* mu, const void* v, const void* Y, const void* rowparams,
                      long R, int n_mc, int S, unsigned long long seed, unsigned long long* offset_dev, double q_lo_p, double q_hi_p,
                      void* q_lo, void* q_hi, void* covered, void* samples, double* count, void* stream) {
    TGP_TRY(validate(md));
    if (R <= 0) return 0;
    if (md->likelihood == TGP_LIK_BERNOULLI) return set_error(-1, "coverage intervals are defined for the Gaussian likelihoods");
    if (md->likelihood == TGP_LIK_GAUSS_WARPED)
        return set_error(-1, "coverage intervals are not implemented for the warped likelihood (its samples need the inverse warp)");
    if (!p || !mu || !v || !Y || !q_lo || !q_hi || !covered || !p->log_var_noise) return set_error(-1, "NULL argument to tgp_coverage_rows");
    if (S < 2 || S > 128) return set_error(-1, "S must be in 2..128");
    if (n_mc != 1 && n_mc != S) return set_error(-1, "n_mc must be 1 or S");
    if (md->n_rowparams > 0 && !rowparams) return set_error(-1, "rowparams required for input-dependent flows");
    RowCoverArgs a;
    a.R = (int)R; a.n_rowp = md->n_rowparams; a.n_mc = n_mc; a.S = S;
    a.mu = (const double*)mu; a.v = (const double*)v; a.y = (const double*)Y; a.log_var_noise = (const double*)p->log_var_noise;
    a.theta = (const double*)p->theta; a.rowp = md->n_rowparams > 0 ? (const double*)rowparams : nullptr;
    a.seed = seed; a.offset_dev = offset_dev; a.q_lo_p = q_lo_p; a.q_hi_p = q_hi_p;
    a.q_lo = (double*)q_lo; a.q_hi = (double*)q_hi; a.covered = (double*)covered; a.samples = (double*)samples; a.count = count;
    fill_flow(a.flow, md);
    k_row_coverage<<<row_grid(R), ROW_THREADS, 0, (cudaStream_t)stream>>>(a);
    TGP_TRY(check_launch("k_row_coverage"));
    if (offset_dev) {
        k_bump_offset<<<1, 1, 0, (cudaStream_t)stream>>>(offset_dev);
        TGP_TRY(check_launch("k_bump_offset"));
    }
    return 0;
}

static int mc_softmax_launch(const TgpModel* md, int C, int S, long R, const void* mu, const void* v, const void* Y, const void* eps,
                             const void* theta, const void* rowparams, int want_grad, void* ell_rows, void* g_mu, void* g_v,
                             void* dtheta, void* drowparams, void* probs, void* stream) {
    McSoftmaxArgs a;
    a.R = (int)R; a.C = C; a.S = S; a.n_theta = md->n_theta; a.want_grad = want_grad;
    a.mu = (const double*)mu; a.v = (const double*)v; a.y = (const double*)Y; a.eps = (const double*)eps;
    a.theta = (const double*)theta;
    a.ell_rows = (double*)ell_rows; a.g_mu = (double*)g_mu; a.g_v = (double*)g_v; a.dtheta = (double*)dtheta; a.probs = (double*)probs;
    fill_flow(a.flow, md);
    a.n_rowp = md->n_rowparams; a.rowp = (const double*)rowparams; a.drowp = (double*)drowparams;
    const unsigned grid = (unsigned)((R + MC_THREADS - 1) / MC_THREADS);
    if (md->n_rowparams == 0) {
        const size_t smem = (size_t)C * 3 * (md->n_theta > 0 ? md->n_theta : 1) * sizeof(double);
        k_row_mc_softmax<false><<<grid, MC_THREADS, smem, (cudaStream_t)stream>>>(a);
    } else {
        // flow_prepare indexes its table by parameter slot over all layers, per-row ones included
        const size_t smem = (size_t)C * 3 * (md->n_theta + md->n_rowparams) * sizeof(double);
        k_row_mc_softmax<true><<<grid, MC_THREADS, smem, (cudaStream_t)stream>>>(a);
    }
    return check_launch("k_row_mc_softmax");
}

// the checks both Monte-Carlo softmax entry points share, after their class-count and sample-count checks
static int mc_softmax_check(const TgpModel* md, int C, const void* mu, const void* v, const void* Y, const void* eps,
                            const void* theta, int want_grad, void* ell_rows, void* g_mu, void* g_v, void* dtheta) {
    if ((long)C * md->n_theta > MC_MAX_ACC) return set_error(-1, "C * n_theta exceeds the per-thread gradient accumulator (256)");
    if (!mu || !v || !Y || !eps || !ell_rows || (md->n_theta > 0 && !theta))
        return set_error(-1, "NULL argument to tgp_mc_softmax_rows");
    if (want_grad && (!g_mu || !g_v || (md->n_theta > 0 && !dtheta))) return set_error(-1, "gradient outputs required");
    return 0;
}

int tgp_mc_softmax_rows(const TgpModel* md, int C, int S, long R, const void* mu, const void* v, const void* Y, const void* eps,
                        const void* theta, int want_grad, void* ell_rows, void* g_mu, void* g_v, void* dtheta, void* probs,
                        void* stream) {
    TGP_TRY(validate(md));
    if (R <= 0) return 0;
    if (C < 2 || C > MC_MAX_CLASSES) return set_error(-1, "number of classes out of range (2..32)");
    if (S < 1) return set_error(-1, "S must be positive");
    if (md->n_rowparams > 0) return set_error(-1, "the Monte-Carlo softmax likelihood takes flows with global parameters");
    TGP_TRY(mc_softmax_check(md, C, mu, v, Y, eps, theta, want_grad, ell_rows, g_mu, g_v, dtheta));
    for (int i = 0; i < md->n_layers; ++i)
        if (md->layers[i].flags & TGP_FLOW_PER_ROW) return set_error(-1, "per-row flow parameters are not supported here");
    return mc_softmax_launch(md, C, S, R, mu, v, Y, eps, theta, nullptr, want_grad, ell_rows, g_mu, g_v, dtheta, nullptr, probs, stream);
}

int tgp_mc_softmax_rows_rowp(const TgpModel* md, int C, int S, long R, const void* mu, const void* v, const void* Y, const void* eps,
                             const void* theta, int want_grad, void* ell_rows, void* g_mu, void* g_v, void* dtheta, void* probs,
                             const void* rowparams, void* drowparams, void* stream) {
    TGP_TRY(validate(md));
    if (R <= 0) return 0;
    if (C < 2 || C > MC_MAX_CLASSES) return set_error(-1, "number of classes out of range (2..32)");
    if (S < 1) return set_error(-1, "S must be positive");
    TGP_TRY(mc_softmax_check(md, C, mu, v, Y, eps, theta, want_grad, ell_rows, g_mu, g_v, dtheta));
    const int nr = md->n_rowparams;
    if (nr > MAX_ROWP) return set_error(-1, "too many per-row flow parameters (n_rowparams <= 16)");
    if ((long)C * nr > MC_MAX_ACC)
        return set_error(-1, "C * n_rowparams exceeds the per-thread per-row gradient accumulator (256)");
    if (nr > 0 && !rowparams) return set_error(-1, "rowparams required for input-dependent flows");
    if (want_grad && nr > 0 && !drowparams) return set_error(-1, "drowparams required for the gradient of input-dependent flows");
    return mc_softmax_launch(md, C, S, R, mu, v, Y, eps, theta, rowparams, want_grad, ell_rows, g_mu, g_v, dtheta, drowparams, probs,
                             stream);
}

int tgp_reduce_pack(const TgpModel* md, const double* reduce_buf, double* packed, void* stream) {
    TGP_TRY(validate(md));
    if (!reduce_buf || !packed) return set_error(-1, "NULL argument to tgp_reduce_pack");
    return reduce_pack(md, const_cast<double*>(reduce_buf), packed, 0, (cudaStream_t)stream);
}

int tgp_reduce_unpack(const TgpModel* md, const double* packed, double* reduce_buf, void* stream) {
    TGP_TRY(validate(md));
    if (!reduce_buf || !packed) return set_error(-1, "NULL argument to tgp_reduce_unpack");
    return reduce_pack(md, reduce_buf, const_cast<double*>(packed), 1, (cudaStream_t)stream);
}

long tgp_flow_mlp_net_doubles(const TgpMlp* m) {
    if (mlp_validate(m)) return 0;
    return mlp_net_size(m->n_in, m->hidden, m->n_hidden_layers);
}

int tgp_flow_mlp_forward(const TgpMlp* m, const void* weights, const void* X, long R, const unsigned char* mask_in,
                         unsigned char* mask_out, unsigned long long seed, unsigned long long* offset_dev, void* out,
                         void* stream) {
    TGP_TRY(mlp_validate(m));
    if (R <= 0) return 0;
    if (!weights || !X || !out) return set_error(-1, "NULL argument to tgp_flow_mlp_forward");
    if (m->mask_mode == 1 && (!mask_out || !offset_dev)) return set_error(-1, "Philox dropout needs mask_out and offset_dev");
    if (m->mask_mode == 2 && !mask_in) return set_error(-1, "explicit dropout needs mask_in");
    MlpArgs a{};
    a.n_nets = m->n_nets; a.n_in = m->n_in; a.H = m->hidden; a.L = m->n_hidden_layers; a.act = m->activation;
    a.mask_mode = m->mask_mode; a.p_drop = m->p_drop; a.R = R;
    a.W = (const double*)weights; a.X = (const double*)X; a.mask_in = mask_in; a.mask_out = mask_out; a.seed = seed;
    a.offset_dev = offset_dev; a.out = (double*)out;
    TGP_TRY(launch_flow_mlp(m, a, false, (cudaStream_t)stream));
    if (m->mask_mode == 1) {
        k_bump_offset<<<1, 1, 0, (cudaStream_t)stream>>>(offset_dev);
        TGP_TRY(check_launch("k_bump_offset"));
    }
    return 0;
}

int tgp_flow_mlp_backward(const TgpMlp* m, const void* weights, const void* X, long R, const unsigned char* mask,
                          const void* dout, void* dweights, void* stream) {
    return tgp_flow_mlp_backward_dx(m, weights, X, R, mask, dout, dweights, nullptr, stream);
}

int tgp_flow_mlp_backward_dx(const TgpMlp* m, const void* weights, const void* X, long R, const unsigned char* mask,
                             const void* dout, void* dweights, void* dX, void* stream) {
    TGP_TRY(mlp_validate(m));
    if (R <= 0) return 0;
    if (!weights || !X || !dout || !dweights) return set_error(-1, "NULL argument to tgp_flow_mlp_backward");
    if (m->mask_mode != 0 && !mask) return set_error(-1, "the backward needs the keep-mask of the forward");
    MlpArgs a{};
    a.n_nets = m->n_nets; a.n_in = m->n_in; a.H = m->hidden; a.L = m->n_hidden_layers; a.act = m->activation;
    a.mask_mode = m->mask_mode; a.p_drop = m->p_drop; a.R = R;
    a.W = (const double*)weights; a.X = (const double*)X; a.mask_in = mask; a.dout = (const double*)dout; a.dW = (double*)dweights;
    a.dX = (double*)dX;
    return launch_flow_mlp(m, a, true, (cudaStream_t)stream);
}

// ---- single-call interface ------------------------------------------------------------------------------------------
namespace tgp {
// Regions of the handle's workspace.  The step and batch regions are as large as the staged entry points' queries
// report, so those entry points carve them again from their own base.
struct HandleView {
    void *step, *batch;
    double *reduce, *packed;
    double *kl;                                  // the KL term of the last factorisation
    double *mu, *v, *g_mu, *g_v, *ell_rows;      // max_rows each
};
inline HandleView handle_view(Carve& c, const TgpModel* md, long max_rows) {
    const TgpReduceLayout l = reduce_layout(md);
    HandleView w;
    w.step = c.take<char>(tgp_step_workspace_bytes(md));
    w.batch = c.take<char>(tgp_batch_workspace_bytes(md, max_rows));
    w.reduce = c.take<double>(l.total);
    w.packed = c.take<double>(l.packed_total);
    w.kl = c.take<double>(1);
    w.mu = c.take<double>(max_rows);
    w.v = c.take<double>(max_rows);
    w.g_mu = c.take<double>(max_rows);
    w.g_v = c.take<double>(max_rows);
    w.ell_rows = c.take<double>(max_rows);
    return w;
}
}  // namespace tgp

struct TgpHandle {
    TgpModel model;
    long max_rows;
    bool bound;
    tgp::HandleView ws;          // regions of the bound workspace
    long last_R;                 // rows of the last forward (the backward must match)
    bool prepared;
};

namespace tgp {
__global__ void k_fwd_terms(const double* __restrict__ rb_ell, const double* __restrict__ kl, double scale, double* __restrict__ terms) {
    terms[0] = scale * rb_ell[0];
    terms[1] = kl[0];
}
__global__ void k_scale_by_dev(double* __restrict__ x, long n, const double* __restrict__ g) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] *= g[0];
}
inline int handle_ready(TgpHandle* h, const TgpBatch* b) {
    if (!h) return set_error(-1, "handle is NULL");
    if (!h->bound) return set_error(-1, "no workspace bound: call tgp_bind_workspace first");
    if (!b || b->R < 0 || b->R > h->max_rows) return set_error(-1, "batch rows exceed the max_rows the handle was created for");
    return 0;
}
}  // namespace tgp

size_t tgp_workspace_bytes(const TgpModel* md, long max_rows) {
    if (validate(md) || max_rows < 1) return 0;
    Carve c(nullptr);
    handle_view(c, md, max_rows);
    return c.bytes();
}

int tgp_create(const TgpModel* md, long max_rows, TgpHandle** out) {
    TGP_TRY(validate(md));
    if (!out || max_rows < 1) return set_error(-1, "tgp_create: out is NULL or max_rows < 1");
    TgpHandle* h = new TgpHandle();
    h->model = *md; h->max_rows = max_rows; h->bound = false; h->last_R = -1; h->prepared = false;
    *out = h;
    return 0;
}

void tgp_destroy(TgpHandle* h) { delete h; }

int tgp_bind_workspace(TgpHandle* h, void* workspace, size_t bytes) {
    if (!h || !workspace) return set_error(-1, "NULL argument to tgp_bind_workspace");
    // the size is asked for again: the row-chunk option may have changed since tgp_create
    if (bytes < tgp_workspace_bytes(&h->model, h->max_rows)) return set_error(-1, "workspace smaller than tgp_workspace_bytes()");
    if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) return set_error(-2, "workspace must be 256-byte aligned");
    Carve c(workspace);
    h->ws = handle_view(c, &h->model, h->max_rows);
    h->bound = true; h->prepared = false; h->last_R = -1;
    return 0;
}

int tgp_elbo_fwd(TgpHandle* h, const TgpParams* p, const TgpBatch* b, double jitter, const TgpFwdOut* out, void* stream) {
    TGP_TRY(handle_ready(h, b));
    if (!p || !out || !out->terms || !out->status) return set_error(-1, "NULL argument to tgp_elbo_fwd");
    const TgpModel* md = &h->model;
    cudaStream_t st = (cudaStream_t)stream;
    const TgpReduceLayout l = reduce_layout(md);
    const HandleView& w = h->ws;
    double* mu = out->mu ? (double*)out->mu : w.mu;
    double* v = out->v ? (double*)out->v : w.v;
    double* rows = out->ell_rows ? (double*)out->ell_rows : w.ell_rows;
    cudaMemsetAsync(w.reduce, 0, (size_t)l.total * sizeof(double), st);
    TGP_TRY(tgp_prepare(md, p, jitter, w.step, w.kl, out->status, stream));
    h->prepared = true;
    TGP_TRY(tgp_qf_forward(md, w.step, w.batch, b->X, b->R, mu, v, stream));
    TGP_TRY(tgp_ell_forward(md, p, mu, v, b->Y, b->rowparams, b->R, b->scale, b->quad_t, b->quad_w, 1, rows, w.g_mu, w.g_v,
                            nullptr, w.reduce, stream));
    k_fwd_terms<<<1, 1, 0, st>>>(w.reduce + l.ell_sum, w.kl, b->scale, out->terms);
    h->last_R = b->R;
    return check_launch("k_fwd_terms");
}

int tgp_elbo_bwd(TgpHandle* h, const TgpParams* p, const TgpBatch* b, const double* g_dev, const TgpGrads* g,
                 TgpAllReduceFn allreduce, void* user, void* stream) {
    TGP_TRY(handle_ready(h, b));
    if (!p || !g || !g_dev) return set_error(-1, "NULL argument to tgp_elbo_bwd");
    if (h->last_R != b->R) return set_error(-1, "tgp_elbo_bwd must follow tgp_elbo_fwd on the same batch");
    const TgpModel* md = &h->model;
    if (md->n_rowparams > 0)
        return set_error(-1, "input-dependent flows: use the staged entry points (drowparams flows back to the caller's MLP)");
    const TgpReduceLayout l = reduce_layout(md);
    const HandleView& w = h->ws;
    if (g->dX && cudaMemsetAsync(g->dX, 0, (size_t)b->R * md->D * sizeof(double), (cudaStream_t)stream) != cudaSuccess)
        return set_error(-100, "zeroing dX failed");
    TGP_TRY(tgp_qf_backward_dx(md, p, w.step, w.batch, b->X, b->R, w.g_mu, w.g_v, w.reduce, g->dX, stream));
    if (g->dX && b->R > 0) {         // dX is row-local (never all-reduced); the ELL weight g_dev[0] is applied here
        const long n = b->R * md->D;
        k_scale_by_dev<<<(unsigned)cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>((double*)g->dX, n, g_dev);
        TGP_TRY(check_launch("k_scale_by_dev"));
    }
    if (allreduce) {
        TGP_TRY(tgp_reduce_pack(md, w.reduce, w.packed, stream));
        if (allreduce(w.packed, l.packed_total, user, stream) != 0) return set_error(-103, "the all-reduce callback failed");
        TGP_TRY(tgp_reduce_unpack(md, w.packed, w.reduce, stream));
    }
    h->last_R = -1;
    return tgp_chain_backward(md, p, w.step, w.reduce, 0.0, 0.0, g_dev, g->dZ, g->draw_lengthscale, g->draw_outputscale, g->dm,
                              g->dL_raw, g->dlog_var_noise, g->dtheta, stream);
}

int tgp_test_nll_fwd(TgpHandle* h, const TgpParams* p, const TgpBatch* b, int refactor, int n_mc, double y_std,
                     const double* bern_std, void* logp_rows, void* m1, void* m2, void* mu_out, void* v_out, int* status,
                     void* stream) {
    TGP_TRY(handle_ready(h, b));
    if (!p || !logp_rows || !m1 || !m2) return set_error(-1, "NULL argument to tgp_test_nll_fwd");
    const TgpModel* md = &h->model;
    const HandleView& w = h->ws;
    if (refactor || !h->prepared) {
        if (!status) return set_error(-1, "status required when the factorisation is (re)computed");
        TGP_TRY(tgp_prepare(md, p, 0.0, w.step, w.kl, status, stream));
        h->prepared = true;
    }
    double* mu = mu_out ? (double*)mu_out : w.mu;
    double* v = v_out ? (double*)v_out : w.v;
    TGP_TRY(tgp_qf_forward(md, w.step, w.batch, b->X, b->R, mu, v, stream));
    h->last_R = -1;
    return tgp_test_rows(md, p, mu, v, b->Y, b->rowparams, b->R, n_mc, y_std, b->quad_t, b->quad_w, bern_std, logp_rows, m1,
                         m2, stream);
}

namespace tgp {
constexpr int ADAM_BLOCK = 4096;
__global__ void __launch_bounds__(256) k_adam(const void* const* __restrict__ tab, const long* __restrict__ sizes,
                                              const double* __restrict__ lr, const double* __restrict__ wd,
                                              const int* __restrict__ block_tensor, const long* __restrict__ block_offset,
                                              double beta1, double beta2, double eps, const long* __restrict__ step_dev) {
    const int t = block_tensor[blockIdx.x];
    const long off = block_offset[blockIdx.x], n = sizes[t];
    double* p = (double*)tab[4 * t];
    const double* g = (const double*)tab[4 * t + 1];
    double* m = (double*)tab[4 * t + 2];
    double* v = (double*)tab[4 * t + 3];
    const double step = (double)(step_dev[0] + 1);                 // this update's count; k_adam_count bumps it afterwards
    const double bc1 = 1.0 - pow(beta1, step), bc2 = 1.0 - pow(beta2, step);
    const double step_size = lr[t] / bc1, rsq2 = 1.0 / sqrt(bc2), w = wd[t];
    for (long i = off + threadIdx.x; i < min(off + (long)ADAM_BLOCK, n); i += 256) {
        const double pi = p[i];
        const double gi = g[i] + w * pi;
        const double mi = beta1 * m[i] + (1.0 - beta1) * gi;       // torch: exp_avg.lerp_(grad, 1 - beta1)
        const double vi = beta2 * v[i] + (1.0 - beta2) * gi * gi;  // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
        m[i] = mi; v[i] = vi;
        p[i] = pi - step_size * (mi / (sqrt(vi) * rsq2 + eps));    // param.addcdiv_(exp_avg, denom, value=-step_size)
    }
}
__global__ void k_adam_count(long* step_dev) { step_dev[0] += 1; }
}  // namespace tgp

int tgp_adam_step(int n_tensors, long n_blocks, const void* const* ptr_table, const long* sizes, const double* lr,
                  const double* weight_decay, const int* block_tensor, const long* block_offset, double beta1, double beta2,
                  double eps, long* step_dev, void* stream) {
    if (n_tensors <= 0 || n_blocks <= 0) return 0;
    if (!ptr_table || !sizes || !lr || !weight_decay || !block_tensor || !block_offset || !step_dev)
        return set_error(-1, "NULL argument to tgp_adam_step");
    cudaStream_t st = (cudaStream_t)stream;
    k_adam<<<(unsigned)n_blocks, 256, 0, st>>>(ptr_table, sizes, lr, weight_decay, block_tensor, block_offset, beta1, beta2, eps, step_dev);
    TGP_TRY(check_launch("k_adam"));
    k_adam_count<<<1, 1, 0, st>>>(step_dev);
    return check_launch("k_adam_count");
}

int tgp_kmeans_iteration(const void* X, long N, int D, void* Cc, int M, int* assign, double* sums, double* counts, double* inertia,
                         int update, void* stream) {
    if (!X || !Cc || !sums || !counts || !inertia) return set_error(-1, "NULL argument to tgp_kmeans_iteration");
    if (N < 1 || M < 1 || D < 1) return set_error(-1, "N, M, D must be positive");
    return kmeans_iteration((const double*)X, N, D, (double*)Cc, M, assign, sums, counts, inertia, update, (cudaStream_t)stream);
}

long tgp_launch_count(void) { return g_launch_count; }

int tgp_set_option(int key, int value) {
    if (key == TGP_OPT_OVERLAP_KGEN) { g_overlap_kgen = value != 0; return 0; }
    if (key == TGP_OPT_ROW_CHUNK) {
        if (value < 128) return set_error(-1, "row chunk must be >= 128");
        f64::g_row_chunk = value;
        return 0;
    }
    return set_error(-1, "unknown option");
}

int tgp_gemm_timing(int enable, double* ms_out, long* launches_out) {
    g_gemm_timer.flush();
    for (int i = 0; i < 3; ++i) {
        if (ms_out) ms_out[i] = g_gemm_timer.ms[i];
        if (launches_out) launches_out[i] = g_gemm_timer.launches[i];
    }
    if (enable >= 0) {
        g_gemm_timer.enabled = enable != 0;
        for (int i = 0; i < 3; ++i) { g_gemm_timer.ms[i] = 0; g_gemm_timer.launches[i] = 0; }
    }
    return 0;
}

int tgp_debug_gemm_f64(int M, int N, int K, const double* A, long lda, int a_layout, const double* B, long ldb,
                       int b_layout, double* C, long ldc, double alpha, double beta, int a_tri, int b_tri, int c_lower,
                       void* stream) {
    GemmArgs g = make_gemm(M, N, K, A, lda, a_layout, B, ldb, b_layout, C, ldc, alpha, beta);
    g.a_tri = a_tri; g.b_tri = b_tri; g.c_lower = c_lower;
    return gemm_f64(g, (cudaStream_t)stream);
}

int tgp_debug_gemm_tf32x3(int Mrows, int Ncols, int K, const float* Ahi, const float* Alo, long lda, const float* Bhi,
                          const float* Blo, long ldb, float* Cf, double* Cd, long ldc, int out_mode, int tri_mode,
                          int tri_rows, int lower_rows, int splitk, void* stream) {
    tc::Params p{};
    p.Mrows = Mrows; p.Ncols = Ncols; p.K = K; p.tri_mode = tri_mode; p.tri_rows = tri_rows; p.out_mode = out_mode;
    p.lower_rows = lower_rows; p.Cf = Cf; p.Cd = Cd; p.ldc = ldc; p.splitk = splitk;
    tc::Operand A{Ahi, Alo, Mrows, K, lda};
    tc::Operand B{Bhi, Blo, Ncols, K, ldb};
    return tc::gemm_tf32x3(A, B, p, (cudaStream_t)stream);
}

size_t tgp_debug_gemm_crt_bytes(long M, long N, long K, int T) {
    Carve c(nullptr);
    crt::debug_scratch(c, M, N, K, T);
    return c.bytes();
}

int tgp_debug_gemm_crt(long M, long N, long K, const double* A, long lda, const double* B, long ldb, double* C, long ldc, int T,
                       int tri_mode, int tri_rows, int lower_rows, int accumulate, int mn_major, void* scratch, void* stream) {
    if (T != 9 && T != 12 && T != 15 && T != 16) return set_error(-1, "T must be 9, 12, 15 or 16");
    if (!A || !B || !C || !scratch) return set_error(-1, "NULL argument to tgp_debug_gemm_crt");
    return crt::debug_matmul(M, N, K, A, lda, B, ldb, C, ldc, T, tri_mode, tri_rows, lower_rows, accumulate, mn_major, scratch,
                             (cudaStream_t)stream);
}

int tgp_debug_export_step(const TgpModel* md, const void* step_ws, double* L, double* Linv, double* C, void* stream) {
    TGP_TRY(validate(md));
    Carve c(const_cast<void*>(step_ws));
    const StepView s = step_layout(c, md).f64;
    cudaStream_t st = (cudaStream_t)stream;
    if (join_factor(st)) return set_error(-100, "join with the factorisation failed");
    if (L) k_copy_strided<<<md->M, 256, 0, st>>>(s.L, s.Mp, L, md->M, md->M);
    if (Linv) k_copy_strided<<<md->M, 256, 0, st>>>(s.Linv, s.Mp, Linv, md->M, md->M);
    if (C) k_copy_strided<<<md->M, 256, 0, st>>>(s.Cm, s.Mp, C, md->M, md->M);
    return check_launch("k_copy_strided");
}

}  // extern "C"
