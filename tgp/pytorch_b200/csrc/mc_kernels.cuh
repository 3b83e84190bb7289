// Monte-Carlo expected log-likelihood of the softmax (multiclass) likelihood — SURVEY.md §8f rank 3.
// Reference: code/dsp/likelihoods/MulticlassCategorical.py:51-105 (expected_log_prob) and :109-151 (marginal_moments).
//
//   F0[s,c,n] = mu[c,n] + sqrt(v[c,n]) eps[s,c,n]            (td.Normal.rsample: loc + eps * scale)
//   FK[s,c,n] = G_c(F0[s,c,n])                               (one flow per class, same architecture, own parameters)
//   ell[n]    = 1/S sum_s ( FK[s,y_n,n] - logsumexp_c FK[s,c,n] )      (-CrossEntropyLoss, mean over the S samples)
//   probs[n,c] = 1/S sum_s softmax_c FK[s,:,n]
//
// The noise eps is an INPUT: the host draws it with the framework's generator exactly as the reference's rsample does, so a
// seeded run sees the reference's stream; the kernel itself is deterministic.  One thread per row (consecutive rows in
// consecutive lanes: every (s, c) slice of mu / v / eps is read coalesced); the softmax couples the classes, so per sample
// all C flows are evaluated first (with their parameter derivatives swept to dFK/dtheta immediately), then weighted by
// w_c = (1[c = y] - softmax_c) / S.  Gradients w.r.t. mu and v go out per row; those of the C x n_theta flow scalars are
// reduced per warp and added with FP64 atomics.
//
// Input-dependent flows (HAS_ROWP): layers flagged TGP_FLOW_PER_ROW read their raw parameters from rowp (C, R, n_rowp), the
// class-stacked outputs of the flow MLPs, fixed per row for the call and shared by all S samples.  Each thread copies its row's
// C x n_rowp values once; the per-row gradient drowp (C, R, n_rowp) = d ell_rows[n] / d rowp[c,n,k] is accumulated over the
// samples in registers / local memory and written once.  HAS_ROWP = false is the global-parameter kernel, unchanged.
#pragma once
#include "row_kernels.cuh"

namespace tgp {

constexpr int MC_MAX_CLASSES = 32;
constexpr int MC_MAX_ACC = 256;          // C * n_theta (and C * n_rowp) of the per-thread gradient accumulators (local memory)
constexpr int MC_THREADS = 128;

struct McSoftmaxArgs {
    int R, C, S, n_theta, want_grad;
    const double *mu, *v, *y, *eps, *theta;        // (C,R), (C,R), (R) labels, (S,C,R), (C,n_theta)
    double *ell_rows, *g_mu, *g_v, *dtheta, *probs;   // (R), (C,R), (C,R), (C,n_theta) accumulated, (R,C) or NULL
    FlowDesc flow;
    int n_rowp;                                        // HAS_ROWP only:
    const double* rowp;                                // (C, R, n_rowp) raw per-row flow parameters
    double* drowp;                                     // (C, R, n_rowp) written when want_grad
};

template <bool HAS_ROWP>
__global__ void __launch_bounds__(MC_THREADS) k_row_mc_softmax(const McSoftmaxArgs a) {
    extern __shared__ double mc_prep[];                 // C tables of 3 * (n_theta + n_rowp) (flow_prepare layout: one slot per
    const int nt = a.n_theta, C = a.C;                  // parameter of every layer, per-row slots left unused)
    const int nr = HAS_ROWP ? a.n_rowp : 0;
    for (int c = 0; c < C; ++c) flow_prepare(a.flow, a.theta + (long)c * nt, mc_prep + (long)c * 3 * (nt + nr));
    const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = n < a.R;
    const bool grad = a.want_grad;
    double acc[MC_MAX_ACC];
    double full[MC_MAX_ACC];                            // dFK_c/dtheta_{c,k} of the current sample
    double rp[HAS_ROWP ? MC_MAX_ACC : 1];               // this row's raw per-row parameters, class-major
    double racc[HAS_ROWP ? MC_MAX_ACC : 1];             // d ell_rows[n] / d rp, summed over the samples
    double rfull[HAS_ROWP ? MC_MAX_ACC : 1];            // dFK_c/drp_{c,k} of the current sample
    double pg[HAS_ROWP ? MAX_THETA + MAX_ROWP : MAX_THETA], dl[TGP_MAX_LAYERS];
    double gk[MC_MAX_CLASSES], dgk[MC_MAX_CLASSES], sd[MC_MAX_CLASSES], m[MC_MAX_CLASSES];
    double gmu[MC_MAX_CLASSES], gv[MC_MAX_CLASSES], pr[MC_MAX_CLASSES];
    if (grad) for (int k = 0; k < C * nt; ++k) acc[k] = 0.0;
    if (live) {
        for (int c = 0; c < C; ++c) {
            m[c] = a.mu[(long)c * a.R + n];
            sd[c] = sqrt(a.v[(long)c * a.R + n]);
            gmu[c] = 0.0; gv[c] = 0.0; pr[c] = 0.0;
        }
        if constexpr (HAS_ROWP) {
            for (int c = 0; c < C; ++c)
                for (int k = 0; k < nr; ++k) rp[c * nr + k] = a.rowp[((long)c * a.R + n) * nr + k];
            if (grad) for (int k = 0; k < C * nr; ++k) racc[k] = 0.0;
        }
        const int y = (int)a.y[n];
        const double inv_s = 1.0 / (double)a.S;
        double ell = 0.0;
        for (int s = 0; s < a.S; ++s) {
            double mx = -INFINITY;
            for (int c = 0; c < C; ++c) {
                const double e = a.eps[((long)s * C + c) * a.R + n];
                const double f = m[c] + e * sd[c];
                const double* th = a.theta + (long)c * nt;
                gk[c] = flow_forward(a.flow, f, th, HAS_ROWP ? rp + c * nr : nullptr, &dgk[c], grad ? pg : nullptr,
                                     grad ? dl : nullptr, mc_prep + (long)c * 3 * (nt + nr));
                if (grad) {                              // reverse sweep: dFK/dtheta_k = pg_k * prod of later layers' slopes
                    double suf = 1.0;
                    int slot_end = nt + nr;              // slots count the parameters of every layer, in descriptor order
                    for (int l = a.flow.n_layers - 1; l >= 0; --l) {
                        const TgpFlowLayer& L = a.flow.layers[l];
                        const int np = layer_nparams(L);
                        slot_end -= np;
                        if constexpr (HAS_ROWP) {        // a layer's parameters start at L.p0 of its own vector
                            if (L.flags & TGP_FLOW_PER_ROW) {
                                for (int k = 0; k < np; ++k) rfull[c * nr + L.p0 + k] = suf * pg[slot_end + k];
                            } else {
                                for (int k = 0; k < np; ++k) full[c * nt + L.p0 + k] = suf * pg[slot_end + k];
                            }
                        } else {                         // all layers global: slot == L.p0
                            for (int k = 0; k < np; ++k) full[c * nt + slot_end + k] = suf * pg[slot_end + k];
                        }
                        suf *= dl[l];
                    }
                }
                mx = fmax(mx, gk[c]);
            }
            double se = 0.0;
            for (int c = 0; c < C; ++c) se += exp(gk[c] - mx);
            const double lse = mx + log(se);
            ell += gk[y] - lse;
            for (int c = 0; c < C; ++c) {
                const double p = exp(gk[c] - lse);
                pr[c] += p;
                if (grad) {
                    const double w = ((c == y ? 1.0 : 0.0) - p) * inv_s;
                    const double wf = w * dgk[c];
                    const double e = a.eps[((long)s * C + c) * a.R + n];
                    gmu[c] += wf;
                    gv[c] += wf * e / (2.0 * sd[c]);
                    for (int k = 0; k < nt; ++k) acc[c * nt + k] += w * full[c * nt + k];
                    if constexpr (HAS_ROWP) for (int k = 0; k < nr; ++k) racc[c * nr + k] += w * rfull[c * nr + k];
                }
            }
        }
        a.ell_rows[n] = ell * inv_s;
        if (a.probs) for (int c = 0; c < C; ++c) a.probs[n * C + c] = pr[c] * inv_s;
        if (grad) for (int c = 0; c < C; ++c) { a.g_mu[(long)c * a.R + n] = gmu[c]; a.g_v[(long)c * a.R + n] = gv[c]; }
        if constexpr (HAS_ROWP) {
            if (grad)
                for (int c = 0; c < C; ++c)
                    for (int k = 0; k < nr; ++k) a.drowp[((long)c * a.R + n) * nr + k] = racc[c * nr + k];
        }
    }
    if (grad) {
        for (int k = 0; k < C * nt; ++k) {
            const double t = warp_sum(acc[k]);
            if ((threadIdx.x & 31) == 0 && t != 0.0) atomicAdd(a.dtheta + k, t);
        }
    }
}

}  // namespace tgp
