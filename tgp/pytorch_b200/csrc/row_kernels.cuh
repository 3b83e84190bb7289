// Per-row kernels: q(f) marginal statistics and the likelihood epilogue (flow o Gauss-Hermite o likelihood) with its
// analytic gradients.  One warp per row; quadrature points are spread over the lanes and reduced with shuffles.
//
// Reference lines: GaussianNonLinearMean.py:64-150 (GH expected log-lik), GaussianLinearMean.py:60-87 (closed form),
// Bernoulli.py:50-95, utils.py:164-195 (expanded quadratic form, float32-rounded pi), flow.py:330-340 (affine),
// 755-773 + 1096-1103 (tanh steps), 904-905 + 965-977 (sinh-arcsinh), sparse_MF_SP.py:705-776 (test log-lik).
#pragma once
#include "common.cuh"
#include "../../../include/tgp_b200.h"

namespace tgp {

constexpr int MAX_THETA = 288;     // global flow scalars (largest shipped architecture: StepTanhL(15,4) = 270)
constexpr int MAX_ROWP = 16;       // per-row (input-dependent) flow parameters
constexpr int ROW_THREADS = 128;   // 4 warps = 4 rows per CTA pass

inline int row_grid(long R) {
    const long blocks = cdiv(R, ROW_THREADS / 32);
    return (int)(blocks < 148 * 16 ? blocks : 148 * 16);
}

// log(2*pi) with the reference's float32-rounded pi (code/dsp/config.py:71, utils.py:180) and exact 1/sqrt(pi)
__device__ constexpr double LOG_2PI_F32PI = 1.8378770942368803;
__device__ constexpr double INV_SQRT_PI = 0.5641895835477563;
__device__ constexpr double INV_SQRT_2PI = 0.3989422804014327;

struct FlowDesc {
    int n_layers;
    TgpFlowLayer layers[TGP_MAX_LAYERS];
};

// mu[n] = sum_j A[n,j] m[j];  v[n] = os - sum_j A^2 + sum_j B^2          (AB row = [A | B], ld = 2M)
__global__ void __launch_bounds__(ROW_THREADS) k_row_stats(const double* __restrict__ AB, const double* __restrict__ m,
                                                           const double* __restrict__ os, int R, int M,
                                                           double* __restrict__ mu, double* __restrict__ v) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    for (long n = (long)blockIdx.x * wpb + wid; n < R; n += (long)gridDim.x * wpb) {
        const double* a = AB + n * 2 * M;
        const double* b = a + M;
        double sm = 0.0, sa = 0.0, sb = 0.0;
        for (int j = lane; j < M; j += 32) {
            const double aj = a[j], bj = b[j];
            sm = fma(aj, __ldg(m + j), sm);
            sa = fma(aj, aj, sa);
            sb = fma(bj, bj, sb);
        }
        sm = warp_sum(sm); sa = warp_sum(sa); sb = warp_sum(sb);
        if (lane == 0) { mu[n] = sm; v[n] = os[0] - sa + sb; }
    }
}

// ---- flow evaluation for one quadrature location ---------------------------------------------------------------
// fetch parameter `idx` of a layer: global theta or this row's parameter vector
__device__ __forceinline__ double flow_param(const TgpFlowLayer& L, int idx, const double* __restrict__ theta,
                                             const double* __restrict__ rowp) {
    return (L.flags & TGP_FLOW_PER_ROW) ? rowp[L.p0 + idx] : theta[L.p0 + idx];
}

__device__ __forceinline__ int layer_nparams(const TgpFlowLayer& L);

// Node-independent transforms of the GLOBAL flow parameters, hoisted out of the (rows x quadrature nodes) loop: for every
// parameter slot s (layer-major, descriptor order) prep[3s] = the value the forward uses (softplus where restricted),
// prep[3s+1] = d(value)/d(raw) (sigmoid where restricted, else 1), prep[3s+2] = 1/value (used for the tanh widths: the
// per-node divisions by a constant become multiplications).  Per-row
// (input-dependent) parameters are not prepared; flow_forward transforms those per row.
constexpr int FLOW_PREP_DOUBLES = 3 * (MAX_THETA + MAX_ROWP);
__device__ __forceinline__ void flow_prepare(const FlowDesc& fd, const double* __restrict__ theta, double* prep) {
    int total = 0;
    for (int l = 0; l < fd.n_layers; ++l) total += layer_nparams(fd.layers[l]);
    for (int s = threadIdx.x; s < total; s += blockDim.x) {
        int l = 0, base = 0;
        while (s >= base + layer_nparams(fd.layers[l])) { base += layer_nparams(fd.layers[l]); ++l; }
        const TgpFlowLayer& L = fd.layers[l];
        if (L.flags & TGP_FLOW_PER_ROW) continue;
        const int idx = s - base;
        const double raw = theta[L.p0 + idx];
        double v0 = raw, v1 = 1.0;
        const bool res = L.flags & TGP_FLOW_RESTRICT;
        if ((L.flags & TGP_FLOW_SWITCH) && idx >= layer_nparams(L) - 2) {       // [softplus(scale), bias] of a step member
            if (idx == layer_nparams(L) - 2) { v0 = softplus_d(raw); v1 = sigmoid_d(raw); }
        } else if (L.kind == TGP_FLOW_AFFINE) {
            if (idx == 0 && res) { v0 = softplus_d(raw); v1 = sigmoid_d(raw); }
        } else if (L.kind == TGP_FLOW_TANH_STEP) {
            const int w = idx & 3;
            if (w == 1) { v0 = softplus_d(raw); v1 = sigmoid_d(raw); }
            else if (w == 3) { v0 = softplus_d(raw); v1 = sigmoid_d(raw); }
        } else if (L.kind == TGP_FLOW_SAL) {
            if (idx == 1 && res) { v0 = softplus_d(raw); v1 = sigmoid_d(raw); }
        } else if (L.kind == TGP_FLOW_ARCSINH) {
            if ((idx == 1 || idx == 3) && res) { v0 = softplus_d(raw); v1 = sigmoid_d(raw); }
        }
        prep[3 * s] = v0; prep[3 * s + 1] = v1; prep[3 * s + 2] = 1.0 / v0;
    }
    __syncthreads();
}

// Forward through all layers.  Returns G(f); *dG = G'(f).  If pg != nullptr, stores for every parameter slot k
// (layer-major, in descriptor order) dG_l/dtheta_k at this location into pg[], and the layer derivatives into dl[].
// prep: the table flow_prepare filled (shared memory).
//
// SECOND = true (the warped likelihood, which differentiates log G'(y)): pg and dl are required, and per layer l the sweep
// also stores d2l[l] = g_l''(x_l) and xpl[l] = dx_l/df (the derivative of the layer's input), and per slot pg2[k] =
// d g_l'(x_l) / dtheta_k.  A step group's members get dl = 1, d2l = 0 and the group's input derivative; its header gets the
// summed g' and g''.  A reverse sweep with adjoints (abar of h, bbar of h') then reads, layer by layer from the last:
//   dtheta_k += abar pg[k] + bbar pg2[k] xpl[l];   abar = abar dl[l] + bbar d2l[l] xpl[l];   bbar = bbar dl[l].
// Global parameters only (per-row layers take the first-order path).  SECOND = false compiles to the first-order sweep.
template <bool SECOND = false>
__device__ __forceinline__ double flow_forward(const FlowDesc& fd, double f, const double* __restrict__ theta,
                                               const double* __restrict__ rowp, double* dG, double* pg, double* dl,
                                               const double* prep, double* pg2 = nullptr, double* d2l = nullptr,
                                               double* xpl = nullptr) {
    double dtot = 1.0;
    int slot = 0;
    // step group (StepFlow, flow.py:1096-1103): the members are evaluated at the group's input and summed
    int group_left = 0, group_l = 0;
    double group_in = 0.0, group_acc = 0.0, group_d = 0.0, group_d2 = 0.0;
    for (int l = 0; l < fd.n_layers; ++l) {
        const TgpFlowLayer& L = fd.layers[l];
        if constexpr (SECOND) xpl[l] = dtot;
        if (L.kind == TGP_FLOW_STEP_GROUP) {
            group_left = L.n_steps; group_l = l; group_in = f;
            const bool add = L.flags & TGP_FLOW_ADD_F0;
            group_acc = add ? f : 0.0; group_d = add ? 1.0 : 0.0;
            if constexpr (SECOND) group_d2 = 0.0;
            if (group_left == 0) {
                f = group_acc; dtot *= group_d; if (dl) dl[l] = group_d;
                if constexpr (SECOND) d2l[l] = 0.0;
            }
            continue;
        }
        if (group_left) f = group_in;
        const int slot0 = slot;
        const bool per_row = L.flags & TGP_FLOW_PER_ROW;
        const bool res = L.flags & TGP_FLOW_RESTRICT;
        // transformed value / chain factor of parameter idx (restricted = through softplus)
        auto val = [&](int idx, bool restricted, double& chain) -> double {
            if (!per_row) { chain = prep[3 * (slot0 + idx) + 1]; return prep[3 * (slot0 + idx)]; }
            const double raw = rowp[L.p0 + idx];
            if (restricted) { chain = sigmoid_d(raw); return softplus_d(raw); }
            chain = 1.0;
            return raw;
        };
        double g, d, ch0, ch1;
        double d2 = 0.0;                                 // g''(f), SECOND only
        if (L.kind == TGP_FLOW_AFFINE) {
            const double a = val(0, res, ch0), b = val(1, false, ch1);
            g = a * f + b;
            d = a;
            if (pg) { pg[slot] = f * ch0; pg[slot + 1] = 1.0; }
            if constexpr (SECOND) { pg2[slot] = ch0; pg2[slot + 1] = 0.0; }
            slot += 2;
        } else if (L.kind == TGP_FLOW_TANH_STEP) {
            double acc = 0.0;
            d = 0.0;
            for (int i = 0; i < L.n_steps; ++i) {
                double chb, chd;
                const double a = val(4 * i, false, ch0), be = val(4 * i + 1, true, chb);
                const double c = val(4 * i + 2, false, ch0), de = val(4 * i + 3, true, chd);
                const double ide = per_row ? 1.0 / de : prep[3 * (slot + 4 * i + 3) + 2];
                const double u = (f - c) * ide;
                const double th = tanh(u);
                const double sech2 = 1.0 - th * th;
                acc += a + be * th;
                const double slope = be * sech2 * ide;
                d += slope;
                if (pg) {
                    pg[slot + 4 * i] = 1.0;
                    pg[slot + 4 * i + 1] = th * chb;
                    pg[slot + 4 * i + 2] = -slope;
                    pg[slot + 4 * i + 3] = -slope * u * chd;
                }
                if constexpr (SECOND) {                  // slope = be sech^2(u) / de
                    const double cur = 2.0 * th * slope * ide;
                    d2 -= cur;
                    pg2[slot + 4 * i] = 0.0;
                    pg2[slot + 4 * i + 1] = sech2 * ide * chb;
                    pg2[slot + 4 * i + 2] = cur;
                    pg2[slot + 4 * i + 3] = slope * (2.0 * th * u - 1.0) * ide * chd;
                }
            }
            slot += 4 * L.n_steps;
            g = acc;
            if (L.flags & TGP_FLOW_ADD_F0) { g += f; d += 1.0; }
        } else if (L.kind == TGP_FLOW_SAL) {
            const double a = val(0, false, ch0), b = val(1, res, ch1);
            const double r = sqrt(f * f + 1.0);
            const double w = log(f + r);                 // the reference's asinh (flow.py:904-905)
            const double z = b * w - a;
            const double ch = cosh(z);
            g = sinh(z);
            const double dw = (1.0 + f / r) / (f + r);   // derivative of log(f + sqrt(f^2+1)) as autograd forms it
            d = ch * b * dw;
            if (pg) { pg[slot] = -ch; pg[slot + 1] = ch * w * ch1; }
            if constexpr (SECOND) {                      // d = cosh(b w - a) b w',  w' = 1/r,  w'' = -f/r^3
                d2 = g * (b * dw) * (b * dw) - ch * b * f / (r * r * r);
                pg2[slot] = -g * b * dw;
                pg2[slot + 1] = (g * w * b + ch) * dw * ch1;
            }
            slot += 2;
            if (L.flags & TGP_FLOW_ADD_F0) { g += f; d += 1.0; }
        } else if (L.kind == TGP_FLOW_ARCSINH) {
            double chb, chd;
            const double a = val(0, false, ch0), b = val(1, res, chb), c = val(2, false, ch0), de = val(3, res, chd);
            const double u = (f - c) / de;
            const double r = sqrt(u * u + 1.0);
            const double w = log(u + r);                 // the reference's asinh (flow.py:521-522)
            const double dw = (1.0 + u / r) / (u + r);   // its derivative as autograd forms it
            g = a + b * w;
            d = b * dw / de;
            if (pg) { pg[slot] = 1.0; pg[slot + 1] = w * chb; pg[slot + 2] = -d; pg[slot + 3] = -d * u * chd; }
            if constexpr (SECOND) {                      // d = b / (de r),  dr/du = u / r
                const double k3 = b / (de * de * r * r * r);
                d2 = -k3 * u;
                pg2[slot] = 0.0;
                pg2[slot + 1] = dw / de * chb;
                pg2[slot + 2] = k3 * u;
                pg2[slot + 3] = -k3 * chd;
            }
            slot += 4;
            if (L.flags & TGP_FLOW_ADD_F0) { g += f; d += 1.0; }
        } else if (L.kind == TGP_FLOW_BOXCOX) {
            const double lam = val(0, false, ch0);
            const double sg = f > 0.0 ? 1.0 : (f < 0.0 ? -1.0 : 0.0), pos = sg * f;
            const double pw = pow(pos, lam);
            g = (sg * pw - 1.0) / lam;
            d = pos > 0.0 ? pw / pos : (lam == 1.0 ? 1.0 : (lam > 1.0 ? 0.0 : INFINITY));       // |f|^(lam - 1)
            if (pg) pg[slot] = (pos > 0.0 ? sg * pw * log(pos) : 0.0) / lam - (sg * pw - 1.0) / (lam * lam);
            if constexpr (SECOND) {                      // d/df |f|^(lam-1) = (lam - 1) |f|^(lam-1) / f
                d2 = pos > 0.0 ? (lam - 1.0) * d / f : 0.0;
                pg2[slot] = pos > 0.0 ? d * log(pos) : 0.0;
            }
            slot += 1;
            if (L.flags & TGP_FLOW_ADD_F0) { g += f; d += 1.0; }
        } else if (L.kind == TGP_FLOW_INV_BOXCOX) {
            const double lam = val(0, false, ch0);
            const double aux = lam * f + 1.0;
            const double sg = aux > 0.0 ? 1.0 : (aux < 0.0 ? -1.0 : 0.0), pos = sg * aux;
            const double e = 1.0 / lam;
            const double pw = pow(pos, e);
            g = sg * pw;
            const double pwm1 = pos > 0.0 ? pw / pos : (e == 1.0 ? 1.0 : (e > 1.0 ? 0.0 : INFINITY));   // pos^(1/lam - 1)
            d = pwm1;                                     // (1/lam) pos^(1/lam - 1) * lam
            if (pg) pg[slot] = (pos > 0.0 ? -sg * pw * log(pos) * e * e : 0.0) + e * pwm1 * f;
            if constexpr (SECOND) {                      // d = pos^(1/lam - 1):  d' = (1 - lam) d / aux
                d2 = pos > 0.0 ? (1.0 - lam) * d / aux : 0.0;
                pg2[slot] = pos > 0.0 ? d * (-e * e * log(pos) + (e - 1.0) * f / aux) : 0.0;
            }
            slot += 1;
            if (L.flags & TGP_FLOW_ADD_F0) { g += f; d += 1.0; }
        } else {   // identity
            g = f; d = 1.0;
        }
        if (L.flags & TGP_FLOW_SWITCH) {                 // switch_off (flow.py:1130-1149): softplus(scale) * g + bias
            double chs;
            const double sc = val(slot - slot0, true, chs), bi = val(slot - slot0 + 1, false, ch1);
            if (pg) {
                for (int k = slot0; k < slot; ++k) pg[k] *= sc;
                pg[slot] = g * chs; pg[slot + 1] = 1.0;
            }
            if constexpr (SECOND) {
                for (int k = slot0; k < slot; ++k) pg2[k] *= sc;
                pg2[slot] = d * chs; pg2[slot + 1] = 0.0;
                d2 *= sc;
            }
            g = sc * g + bi;
            d *= sc;
            slot += 2;
        }
        if (group_left) {
            group_acc += g; group_d += d;
            if (dl) dl[l] = 1.0;
            if constexpr (SECOND) { group_d2 += d2; d2l[l] = 0.0; }
            if (--group_left == 0) {
                f = group_acc; dtot *= group_d; if (dl) dl[group_l] = group_d;
                if constexpr (SECOND) d2l[group_l] = group_d2;
            }
        } else {
            if (dl) dl[l] = d;
            if constexpr (SECOND) d2l[l] = d2;
            dtot *= d;
            f = g;
        }
    }
    *dG = dtot;
    return f;
}

__device__ __forceinline__ int layer_nparams(const TgpFlowLayer& L) {
    const int sw = (L.flags & TGP_FLOW_SWITCH) ? 2 : 0;
    switch (L.kind) {
        case TGP_FLOW_TANH_STEP: return 4 * L.n_steps + sw;
        case TGP_FLOW_IDENTITY: case TGP_FLOW_STEP_GROUP: return 0;
        case TGP_FLOW_ARCSINH: return 4 + sw;
        case TGP_FLOW_BOXCOX: case TGP_FLOW_INV_BOXCOX: return 1 + sw;
        default: return 2 + sw;
    }
}

// torch.distributions.Normal(0,1).cdf: 0.5 * (1 + erf(x / sqrt(2)))
__device__ __forceinline__ double norm_cdf_ref(double x) { return 0.5 * (1.0 + erf(x / 1.4142135623730951)); }

struct RowQuadArgs {
    int R, likelihood, n_quad, n_theta, n_rowp, want_grad;
    double scale;                       // N / MB_global, applied to every gradient (not to ell_rows)
    const double *mu, *v, *y, *log_var_noise, *theta, *rowp, *qt, *qw;
    double *ell_rows, *g_mu, *g_v;      // per-row outputs (g_* scaled)
    double *ell_sum, *dlogvar, *dtheta; // accumulated with atomics (caller zeroes)
    double *drowp;                      // (R, n_rowp) written
    FlowDesc flow;
};

// Expected log-likelihood per row + gradients w.r.t. (mu, v, log_var_noise, flow parameters).
__global__ void __launch_bounds__(ROW_THREADS) k_row_quad(const RowQuadArgs a) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    __shared__ double prep[FLOW_PREP_DOUBLES];
    flow_prepare(a.flow, a.theta, prep);
    double acc_theta[MAX_THETA];
    double pg[MAX_THETA + MAX_ROWP];
    double dl[TGP_MAX_LAYERS];
    const bool grad = a.want_grad != 0;
    if (grad) for (int k = 0; k < a.n_theta; ++k) acc_theta[k] = 0.0;
    double acc_ell = 0.0, acc_lv = 0.0;

    const double var = a.likelihood == TGP_LIK_BERNOULLI ? 1.0 : exp(a.log_var_noise[0]);
    const double inv = 1.0 / var;
    const double logvar = log(var);

    for (long n = (long)blockIdx.x * wpb + wid; n < a.R; n += (long)gridDim.x * wpb) {
        const double mu = a.mu[n], y = a.y[n];
        double v = a.v[n];
        const double* rowp = a.rowp ? a.rowp + n * a.n_rowp : nullptr;
        double ell = 0.0, gmu = 0.0, gv = 0.0, glv = 0.0;
        double acc_row[MAX_ROWP];
        for (int k = 0; k < a.n_rowp; ++k) acc_row[k] = 0.0;

        if (a.likelihood == TGP_LIK_GAUSS_LINEAR) {
            // closed form: logN(y|mu,var) - 0.5 v/var    (GaussianLinearMean.py:82-86)
            const double q = y * inv * y - 2.0 * (y * inv * mu) + mu * inv * mu;
            ell = -0.5 * (LOG_2PI_F32PI + logvar + q) - 0.5 * inv * v;
            gmu = (y - mu) * inv;
            gv = -0.5 * inv;
            glv = -0.5 + 0.5 * ((y - mu) * (y - mu) + v) * inv;
            if (lane != 0) { ell = gmu = gv = glv = 0.0; }
        } else {
            bool clamped = false;
            if (a.likelihood == TGP_LIK_BERNOULLI && v < 0.0) { v = 0.0; clamped = true; }   // Bernoulli.py:77
            const double sd2 = sqrt(2.0 * v);
            for (int s = lane; s < a.n_quad; s += 32) {
                const double t = a.qt[s], cw = a.qw[s] * INV_SQRT_PI;
                const double f = sd2 * t + mu;
                double dG;
                const double g = flow_forward(a.flow, f, a.theta, rowp, &dG, grad ? pg : nullptr, grad ? dl : nullptr, prep);
                double h, hg;
                if (a.likelihood == TGP_LIK_GAUSS_NONLINEAR) {
                    const double q = y * inv * y - 2.0 * (y * inv * g) + g * inv * g;     // utils.py:191
                    h = -0.5 * (LOG_2PI_F32PI + logvar + q);
                    hg = (y - g) * inv;
                    glv += cw * (-0.5 + 0.5 * (y - g) * (y - g) * inv);
                } else {
                    const double p = norm_cdf_ref(g);
                    const double lp = fmax(log(p), -100.0), lq = fmax(log(1.0 - p), -100.0);   // BCELoss clamp
                    h = y * lp + (1.0 - y) * lq;
                    hg = -(p - y) / fmax(p * (1.0 - p), 1e-12) * INV_SQRT_2PI * exp(-0.5 * g * g);
                }
                ell += cw * h;
                if (grad) {
                    // reverse sweep over the layers: suffix product of layer derivatives
                    double suf = cw * hg;
                    int slot_end = 0;
                    for (int l = 0; l < a.flow.n_layers; ++l) slot_end += layer_nparams(a.flow.layers[l]);
                    for (int l = a.flow.n_layers - 1; l >= 0; --l) {
                        const TgpFlowLayer& L = a.flow.layers[l];
                        const int np = layer_nparams(L);
                        slot_end -= np;
                        if (L.flags & TGP_FLOW_PER_ROW) {
                            for (int k = 0; k < np; ++k) acc_row[L.p0 + k] += suf * pg[slot_end + k];
                        } else {
                            for (int k = 0; k < np; ++k) acc_theta[L.p0 + k] += suf * pg[slot_end + k] * a.scale;
                        }
                        suf *= dl[l];
                    }
                    gmu += suf;
                    gv += suf * t / sd2;
                }
            }
            if (clamped) gv = 0.0;
        }
        ell = warp_sum(ell);
        if (lane == 0) a.ell_rows[n] = ell;
        acc_ell += (lane == 0) ? ell : 0.0;
        if (grad) {
            gmu = warp_sum(gmu); gv = warp_sum(gv);
            if (lane == 0) { a.g_mu[n] = gmu * a.scale; a.g_v[n] = gv * a.scale; }
            acc_lv += glv * a.scale;
            for (int k = 0; k < a.n_rowp; ++k) {
                const double r = warp_sum(acc_row[k]);
                if (lane == 0) a.drowp[n * a.n_rowp + k] = r * a.scale;
            }
        }
    }
    // block-level reduction of the accumulators, one atomic per CTA per slot
    __shared__ double red[ROW_THREADS / 32];
    auto block_add = [&](double val, double* dst) {
        val = warp_sum(val);
        if (lane == 0) red[wid] = val;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < wpb; ++w) t += red[w];
            atomicAdd(dst, t);
        }
        __syncthreads();
    };
    block_add(acc_ell, a.ell_sum);
    if (grad) {
        if (a.likelihood != TGP_LIK_BERNOULLI) block_add(acc_lv, a.dlogvar);
        for (int k = 0; k < a.n_theta; ++k) block_add(acc_theta[k], a.dtheta + k);
    }
}

// Warped Gaussian likelihood (TGP_LIK_GAUSS_WARPED): z = G(y) with the global flow G, z = f + eps, eps ~ N(0, s2).  No
// quadrature: one row per thread.  ell = -0.5 (log 2pi + log s2 + q) - 0.5 v / s2 + log|G'(y)|, q the expanded quadratic form
// of the closed-form branch of k_row_quad at G(y) (an identity warp gives that branch's row).  dell/dtheta = -(G - mu)/s2 dG/dtheta
// + (dG'/dtheta) / G' through the second-order sweep of flow_forward.  Outputs and accumulators as k_row_quad's.
__global__ void __launch_bounds__(ROW_THREADS) k_row_warped(const RowQuadArgs a) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    __shared__ double prep[FLOW_PREP_DOUBLES];
    flow_prepare(a.flow, a.theta, prep);
    double acc_theta[MAX_THETA];
    double pg[MAX_THETA], pg2[MAX_THETA];
    double dl[TGP_MAX_LAYERS], d2l[TGP_MAX_LAYERS], xpl[TGP_MAX_LAYERS];
    const bool grad = a.want_grad != 0;
    if (grad) for (int k = 0; k < a.n_theta; ++k) acc_theta[k] = 0.0;
    double acc_ell = 0.0, acc_lv = 0.0;
    int n_slots = 0;
    for (int l = 0; l < a.flow.n_layers; ++l) n_slots += layer_nparams(a.flow.layers[l]);

    const double var = exp(a.log_var_noise[0]);
    const double inv = 1.0 / var;
    const double logvar = log(var);

    for (long n = (long)blockIdx.x * blockDim.x + threadIdx.x; n < a.R; n += (long)gridDim.x * blockDim.x) {
        const double mu = a.mu[n], v = a.v[n];
        double dG;
        const double z = grad ? flow_forward<true>(a.flow, a.y[n], a.theta, nullptr, &dG, pg, dl, prep, pg2, d2l, xpl)
                              : flow_forward(a.flow, a.y[n], a.theta, nullptr, &dG, nullptr, nullptr, prep);
        const double q = z * inv * z - 2.0 * (z * inv * mu) + mu * inv * mu;
        const double ell = -0.5 * (LOG_2PI_F32PI + logvar + q) - 0.5 * inv * v + log(fabs(dG));
        a.ell_rows[n] = ell;
        acc_ell += ell;
        if (grad) {
            const double gmu = (z - mu) * inv;
            a.g_mu[n] = gmu * a.scale;
            a.g_v[n] = -0.5 * inv * a.scale;
            acc_lv += (-0.5 + 0.5 * ((z - mu) * (z - mu) + v) * inv) * a.scale;
            // reverse sweep: abar = dell/dh, bbar = dell/dh' at the output of each layer
            double abar = -gmu, bbar = 1.0 / dG;
            int slot_end = n_slots;
            for (int l = a.flow.n_layers - 1; l >= 0; --l) {
                const TgpFlowLayer& L = a.flow.layers[l];
                const int np = layer_nparams(L);
                slot_end -= np;
                const double xp = xpl[l];
                for (int k = 0; k < np; ++k)
                    acc_theta[L.p0 + k] += (abar * pg[slot_end + k] + bbar * pg2[slot_end + k] * xp) * a.scale;
                abar = abar * dl[l] + bbar * d2l[l] * xp;
                bbar *= dl[l];
            }
        }
    }
    __shared__ double red[ROW_THREADS / 32];
    auto block_add = [&](double val, double* dst) {
        val = warp_sum(val);
        if (lane == 0) red[wid] = val;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < wpb; ++w) t += red[w];
            atomicAdd(dst, t);
        }
        __syncthreads();
    };
    block_add(acc_ell, a.ell_sum);
    if (grad) {
        block_add(acc_lv, a.dlogvar);
        for (int k = 0; k < a.n_theta; ++k) block_add(acc_theta[k], a.dtheta + k);
    }
}

// G^-1(z) for a global flow by a safeguarded Newton iteration.  Start at h = z; r(h) = s (G(h) - z) with s the sign of G'(z)
// is increasing wherever G is monotone in that orientation.  A bracket with a sign change of r is expanded from the start
// (steps max(1, |z|) doubling, at most 64), then Newton steps that leave the bracket or do not halve the step before last become bisections, until
// |dh| <= 4 eps max(1, |h|) (at most 200 steps).  Returns false — no inverse — when G'(z) = 0, when a point the search
// evaluates has s G' < 0 (G not monotone) or a non-finite G, or when either loop runs out.
__device__ __forceinline__ bool flow_inverse(const FlowDesc& fd, double z, const double* __restrict__ theta, const double* prep,
                                             double* out) {
    constexpr int MAX_EXPAND = 64, MAX_ITER = 200;
    constexpr double TOL = 4.0 * 2.220446049250313e-16;
    double d;
    double h = z;
    const double g0 = flow_forward(fd, h, theta, nullptr, &d, nullptr, nullptr, prep);
    if (!(isfinite(g0) && isfinite(d)) || d == 0.0) return false;
    const double s = d > 0.0 ? 1.0 : -1.0;
    auto eval = [&](double x, double* r, double* dr) -> bool {
        double dx;
        const double gx = flow_forward(fd, x, theta, nullptr, &dx, nullptr, nullptr, prep);
        *r = s * (gx - z);
        *dr = s * dx;
        return isfinite(*r) && *dr >= 0.0;
    };
    double r = s * (g0 - z), dr = s * d;
    if (r == 0.0) { *out = h; return true; }
    // bracket: the last point on the start's side of the root (p) and the first beyond it (t)
    const double dir = r < 0.0 ? 1.0 : -1.0;
    double p = h, rp = r, dp = dr, t = h, rt = r, dt = dr;
    double step = fmax(1.0, fabs(h));
    bool found = false;
    for (int e = 0; e < MAX_EXPAND; ++e, step *= 2.0) {
        t = h + dir * step;
        if (!eval(t, &rt, &dt)) return false;
        if ((rt < 0.0) != (r < 0.0) || rt == 0.0) { found = true; break; }
        p = t; rp = rt; dp = dt;
    }
    if (!found) return false;
    if (rt == 0.0) { *out = t; return true; }
    double lo = fmin(p, t), hi = fmax(p, t);
    if (fabs(rp) <= fabs(rt)) { h = p; r = rp; dr = dp; } else { h = t; r = rt; dr = dt; }
    // a Newton step that would leave the bracket, or that would not at least halve the step before last (steep or flat
    // stretches, e.g. narrow tanh steps), is replaced by a bisection: never slower than bisection
    double dh_old = hi - lo, dh = dh_old;
    for (int it = 0; it < MAX_ITER; ++it) {
        const double hn = h - r / dr;
        if (!(hn > lo && hn < hi) || fabs(2.0 * r) > fabs(dh_old * dr)) {
            dh_old = dh;
            dh = 0.5 * (hi - lo);
            h = lo + dh;
        } else {
            dh_old = dh;
            dh = hn - h;
            h = hn;
        }
        if (!eval(h, &r, &dr)) return false;
        if (r == 0.0 || fabs(dh) <= TOL * fmax(1.0, fabs(h))) { *out = h; return true; }
        if (r < 0.0) lo = h; else hi = h;
    }
    return false;
}

// out[i] = G^-1(z[i]) or NaN; n_fail[0] += number of NaNs (one atomic per warp that has any)
__global__ void __launch_bounds__(ROW_THREADS) k_flow_inverse(const FlowDesc fd, const double* __restrict__ theta,
                                                              const double* __restrict__ z, long R, double* __restrict__ out,
                                                              int* __restrict__ n_fail) {
    __shared__ double prep[FLOW_PREP_DOUBLES];
    flow_prepare(fd, theta, prep);
    int fails = 0;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < R; i += (long)gridDim.x * blockDim.x) {
        double h;
        const bool ok = flow_inverse(fd, z[i], theta, prep, &h);
        out[i] = ok ? h : NAN;
        fails += ok ? 0 : 1;
    }
    for (int o = 16; o > 0; o >>= 1) fails += __shfl_xor_sync(0xffffffffu, fails, o);
    if ((threadIdx.x & 31) == 0 && fails > 0) atomicAdd(n_fail, fails);
}

struct RowTestArgs {
    int R, likelihood, n_quad, n_rowp, n_mc;
    double y_std;
    const double *mu, *v, *y, *log_var_noise, *theta, *rowp, *qt, *qw;   // rowp: (R, n_mc, n_rowp)
    const double* bern_std;             // Bernoulli non-identity flow: batch-wide std of v (reference defect kept)
    double *logp_rows, *m1, *m2;
    FlowDesc flow;
};

// Test log-likelihood per row and predictive moments (sparse_MF_SP.py:705-776, likelihood marginal_moments).
// logp_rows[n] excludes the batch-level constants (-0.5*MB*log(pi_f32)), which the host wrapper applies with the
// reference's float32 arithmetic.
// WARPED (TGP_LIK_GAUSS_WARPED, z = G(y) = f + eps): logp = log N(G(y) | mu, v + s2) + log|G'(y)| - log y_std in the y_std form
// of the closed-form branch; m1 = E[G^-1(z)], m2 = E[G^-1(z)^2] - m1^2 for z ~ N(mu, v + s2) by Gauss-Hermite over the lanes
// with flow_inverse per node, both NaN when an inverse fails.
template <bool WARPED>
__global__ void __launch_bounds__(ROW_THREADS) k_row_test(const RowTestArgs a) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    __shared__ double prep[FLOW_PREP_DOUBLES];
    flow_prepare(a.flow, a.theta, prep);
    const double var = a.likelihood == TGP_LIK_BERNOULLI ? 1.0 : exp(a.log_var_noise[0]);
    const double NEG_INF = -INFINITY;
    for (long n = (long)blockIdx.x * wpb + wid; n < a.R; n += (long)gridDim.x * wpb) {
        const double mu = a.mu[n], v = a.v[n], y = a.y ? a.y[n] : 0.0;
        if constexpr (WARPED) {
            const double ky = var + v;
            if (lane == 0) {
                double dG;
                const double gy = flow_forward(a.flow, y, a.theta, nullptr, &dG, nullptr, nullptr, prep);
                const double C = (a.y_std * sqrt(ky)) * (a.y_std * sqrt(ky));
                const double ic = 1.0 / C, yy = a.y_std * gy, mm = a.y_std * mu;
                a.logp_rows[n] = -0.5 * (LOG_2PI_F32PI + log(C) + (yy * ic * yy - 2.0 * (yy * ic * mm) + mm * ic * mm))
                                 + log(fabs(dG));
            }
            const double sd2 = sqrt(2.0 * ky);
            double e1 = 0.0, e2 = 0.0;
            bool ok = true;
            for (int s = lane; s < a.n_quad; s += 32) {
                const double w = a.qw[s];
                double h = 0.0;
                ok = flow_inverse(a.flow, sd2 * a.qt[s] + mu, a.theta, prep, &h) && ok;
                e1 += INV_SQRT_PI * (h * w);
                e2 += INV_SQRT_PI * (h * h * w);
            }
            e1 = warp_sum(e1); e2 = warp_sum(e2);
            ok = __all_sync(0xffffffffu, ok);
            if (lane == 0) { a.m1[n] = ok ? e1 : NAN; a.m2[n] = ok ? e2 - e1 * e1 : NAN; }
            continue;
        }
        if (a.likelihood == TGP_LIK_GAUSS_LINEAR) {
            if (lane == 0) {
                const double ky = var + v;
                const double C = (a.y_std * sqrt(ky)) * (a.y_std * sqrt(ky));
                const double ic = 1.0 / C, yy = a.y_std * y, mm = a.y_std * mu;
                // per-row share of batched_log_Gaussian over the minibatch dimension (sparse_MF_SP.py:791)
                a.logp_rows[n] = -0.5 * (LOG_2PI_F32PI + log(C) + (yy * ic * yy - 2.0 * (yy * ic * mm) + mm * ic * mm));
                a.m1[n] = mu; a.m2[n] = ky;
            }
            continue;
        }
        if (a.likelihood == TGP_LIK_BERNOULLI) {
            // P(y=1): eq. 3.80 for identity flows, quadrature with the batch-wide std otherwise (Bernoulli.py:98-157)
            double P;
            if (a.flow.n_layers == 0) {
                P = norm_cdf_ref(mu / sqrt(1.0 + v));
            } else {
                const double sd2 = sqrt(2.0 * (a.bern_std[0] * a.bern_std[0]));
                double acc = 0.0;
                for (int s = lane; s < a.n_quad; s += 32) {
                    double dG;
                    const double g = flow_forward(a.flow, sd2 * a.qt[s] + mu, a.theta,
                                                  a.rowp ? a.rowp + n * a.n_rowp : nullptr, &dG, nullptr, nullptr, prep);
                    acc += INV_SQRT_PI * (norm_cdf_ref(g) * a.qw[s]);
                }
                P = fmin(fmax(warp_sum(acc), 0.0), 1.0);
            }
            if (lane == 0) { a.m1[n] = P; a.m2[n] = 0.0; a.logp_rows[n] = 0.0; }
            continue;
        }
        // Gaussian likelihood with non-linear mean
        const double sd2_t = sqrt(2.0 * v);                    // test log-lik uses sqrt(2*cov) directly (:709)
        const double sv = sqrt(v);
        const double sd2_m = sqrt(2.0 * (sv * sv));            // moments go through td.Normal(...).variance
        const double C = (a.y_std * sqrt(var)) * (a.y_std * sqrt(var));
        const double ic = 1.0 / C, logC = log(C), yy = a.y_std * y;
        double out_max = NEG_INF, out_sum = 0.0, m1_acc = 0.0, m2_acc = 0.0;
        for (int mc = 0; mc < a.n_mc; ++mc) {
            const double* rowp = a.rowp ? a.rowp + ((long)n * a.n_mc + mc) * a.n_rowp : nullptr;
            double mx = NEG_INF, sm = 0.0, e1 = 0.0, e2 = 0.0;
            for (int s = lane; s < a.n_quad; s += 32) {
                const double t = a.qt[s], w = a.qw[s];
                double dG;
                const double g = flow_forward(a.flow, sd2_t * t + mu, a.theta, rowp, &dG, nullptr, nullptr, prep);
                const double mm = a.y_std * g;
                const double lp = -0.5 * (LOG_2PI_F32PI + logC + (yy * ic * yy - 2.0 * (yy * ic * mm) + mm * ic * mm));
                const double val = log(w) + lp;
                if (val > mx) { sm = sm * exp(mx - val) + 1.0; mx = val; } else if (val > NEG_INF) { sm += exp(val - mx); }
                const double gm = (sd2_m == sd2_t) ? g
                                                   : flow_forward(a.flow, sd2_m * t + mu, a.theta, rowp, &dG, nullptr, nullptr, prep);
                e1 += INV_SQRT_PI * (gm * w);
                e2 += INV_SQRT_PI * (gm * gm * w);
            }
            const double gmx = warp_max(mx);
            sm = (mx > NEG_INF) ? sm * exp(mx - gmx) : 0.0;
            sm = warp_sum(sm);
            double inner = gmx + log(sm);
            e1 = warp_sum(e1); e2 = warp_sum(e2);
            if (a.n_mc > 1) inner -= 0.5 * 1.1447299718856812;      // -0.5*log(pi) evaluated in float32 (:768)
            if (inner > out_max) { out_sum = out_sum * exp(out_max - inner) + 1.0; out_max = inner; }
            else out_sum += exp(inner - out_max);
            const double m2_mc = var + e2 - e1 * e1;
            m1_acc += e1;
            m2_acc += m2_mc + e1 * e1;
        }
        if (lane == 0) {
            a.logp_rows[n] = a.n_mc > 1 ? out_max + log(out_sum) - log((double)a.n_mc) : out_max + log(out_sum);
            const double m1 = m1_acc / a.n_mc;
            a.m1[n] = m1;
            a.m2[n] = a.n_mc > 1 ? m2_acc / a.n_mc - m1 * m1 : (m2_acc - m1 * m1);
        }
    }
}

}  // namespace tgp
