/* tgp_b200.h — C-ABI of the B200-native minibatch-ELBO / test-NLL path for SVGP / TGP / ID_TGP.
 *
 * The reference (jmaronas/TGP.pytorch) has no FFI: the path is plain Python method calls.  Each entry point
 * below names the reference method (file:line under /root/reference/code/dsp) whose arithmetic it replaces; the
 * Python host classes in tgp/pytorch_b200/dsp keep the reference's class surface and call these through ctypes
 * (INTEGRATION.md shows the binding a reference maintainer would add).
 *
 * Conventions
 *  - plain C, POD structs, raw DEVICE pointers unless a field says "host"; no torch types;
 *  - every call only ENQUEUES work on `stream` (a cudaStream_t passed as void*) and never synchronises;
 *  - the caller owns every buffer; the library never allocates device memory.  Workspaces are sized by the
 *    *_bytes() queries and carved deterministically, so the same workspace can be reused every step;
 *  - return 0 = ok; < 0 = usage / launch error (text from tgp_last_error());
 *  - one output GP per call (the reference's Dy > 1 case is a loop over outputs); q(u) whitened or not (TgpModel.q_u_form);
 *  - dtype: TGP_F64 is what the reference's main.py runs (set_maximum_precission, config.py:37-46).
 */
#ifndef TGP_B200_H
#define TGP_B200_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

enum { TGP_F64 = 0, TGP_F32 = 1, TGP_F64_I8 = 2 };
enum { TGP_LIK_GAUSS_LINEAR = 0,     /* likelihoods/GaussianLinearMean.py:60-87   (SVGP, closed form)      */
       TGP_LIK_GAUSS_NONLINEAR = 1,  /* likelihoods/GaussianNonLinearMean.py:113-150 (Gauss-Hermite)       */
       TGP_LIK_BERNOULLI = 2 };      /* likelihoods/Bernoulli.py:50-95                                      */
enum { TGP_FLOW_IDENTITY = 0,        /* models/flow.py:296-307                                              */
       TGP_FLOW_AFFINE = 1,          /* models/flow.py:330-340   params [a, b]                              */
       TGP_FLOW_TANH_STEP = 2,       /* models/flow.py:1096-1103 over :755-773   params n_steps x [a,b,c,d] */
       TGP_FLOW_SAL = 3,             /* models/flow.py:904-905, 965-977   params [a, b]                     */
       TGP_FLOW_ARCSINH = 4,         /* models/flow.py:495-557  a + b asinh((f - c) / d)   params [a, b, c, d]
                                      * (RESTRICT: softplus on b and d; asinh(u) = log(u + sqrt(u^2 + 1)))  */
       TGP_FLOW_BOXCOX = 5,          /* models/flow.py:377-421  (sgn(f)|f|^lam - 1) / lam   params [lam] — the
                                      * value AFTER the module's constraint (transform_param, :398-409)     */
       TGP_FLOW_INV_BOXCOX = 6,      /* models/flow.py:423-446  sgn(lam f + 1)|lam f + 1|^(1/lam)  params [lam] */
       TGP_FLOW_STEP_GROUP = 7 };    /* models/flow.py:1039-1103 StepFlow over arbitrary members: header layer, no
                                      * parameters; the next n_steps layers are evaluated at the header's input and
                                      * summed (+ the input with TGP_FLOW_ADD_F0 on the header).  Members: any kind
                                      * except AFFINE / STEP_GROUP (a single tanh is TANH_STEP with n_steps = 1)      */
enum { TGP_FLOW_RESTRICT = 1,        /* set_restrictions: softplus on a (affine) / b (sinh-arcsinh)         */
       TGP_FLOW_ADD_F0 = 2,          /* add_init_f0                                                         */
       TGP_FLOW_PER_ROW = 4,         /* parameters come from the per-row matrix (input-dependent flow)      */
       TGP_FLOW_SWITCH = 8 };        /* step member with a trainable switch_off (models/flow.py:1130-1149): two more
                                      * GLOBAL parameters [s, t] after the layer's own; output softplus(s) g + t.
                                      * Not combinable with TGP_FLOW_PER_ROW                                  */
enum { TGP_KERNEL_RBF = 0,           /* s exp(-r^2 / 2)                       gpytorch ScaleKernel(RBFKernel)        */
       TGP_KERNEL_MATERN12 = 1,      /* s exp(-r)                             gpytorch ScaleKernel(MaternKernel(0.5)) */
       TGP_KERNEL_MATERN32 = 2,      /* s (1 + sqrt3 r) exp(-sqrt3 r)         nu = 1.5                               */
       TGP_KERNEL_MATERN52 = 3 };    /* s (1 + sqrt5 r + 5r^2/3) exp(-sqrt5 r)   nu = 2.5
                                      * r^2 = sum_d ((x_d - z_d) / lengthscale_d)^2, computed by direct differences    */
enum { TGP_QU_WHITENED = 0,          /* u = L v, q(v) = N(m, P P^T), p(v) = N(0, I)    sparse_MF_SP.py:354-382, 406-431  */
       TGP_QU_UNWHITENED = 1 };      /* q(u) = N(m, P P^T), p(u) = N(0, K_zz)         sparse_MF_SP.py:357-360, 386-391, 433-453
                                      * P = tril(L_raw), L = chol(K_zz + jitter I).  Every entry point runs the whitened algebra on
                                      * (L^-1 m, L^-1 P), which gives the same q(f) and KL; tgp_chain_backward maps the gradients back */
#define TGP_MAX_LAYERS 64

typedef struct TgpFlowLayer {
    int kind;      /* TGP_FLOW_*                                                     */
    int flags;     /* TGP_FLOW_RESTRICT | TGP_FLOW_ADD_F0 | TGP_FLOW_PER_ROW         */
    int n_steps;   /* TANH_STEP: number of tanh terms; STEP_GROUP: number of members */
    int p0;        /* first parameter: index into theta, or column of the row matrix */
} TgpFlowLayer;

typedef struct TgpModel {            /* host struct; describes one output GP */
    int dtype;                       /* TGP_F64: all FP64 (DMMA).  TGP_F32: batch contractions as 3xTF32 on
                                      * tcgen05 with FP32 TMEM accumulators.  TGP_F64_I8: batch contractions on the
                                      * tcgen05 INTEGER path (kind::i8, exact s32 accumulation in TMEM) over 15-16
                                      * residue planes, rebuilt by the Chinese remainder theorem — FP64-accurate
                                      * (operands truncated at 52-53 bits below their row maximum).  Per-step
                                      * factorisation, chain and the row epilogue are FP64 in every mode; inputs /
                                      * outputs are FP64 in every mode                                            */
    int M, D;                        /* inducing points, input dimension                                   */
    int likelihood;                  /* TGP_LIK_*                                                          */
    int n_quad;                      /* Gauss-Hermite points (config.py:45,58: 100 in FP64, 50 in FP32)    */
    int n_theta;                     /* global flow scalars                                                */
    int n_rowparams;                 /* per-row flow parameters (ID_TGP), 0 otherwise                      */
    int n_layers;
    TgpFlowLayer layers[TGP_MAX_LAYERS];
    int kernel;                      /* TGP_KERNEL_* (0 = RBF, so a zero-initialised description is unchanged).  Workspace
                                      * sizes do not depend on it                                                   */
    int q_u_form;                    /* TGP_QU_* (0 = whitened, so a zero-initialised description is unchanged).  A non-whitened
                                      * model's step workspace holds one more Mp x Mp matrix (tril(L_raw))                     */
} TgpModel;

typedef struct TgpParams {           /* device pointers to the model parameters (same shapes as the reference's) */
    const void* Z;                   /* (M, D)     sparse_MF_SP.Z[dy]                                      */
    const void* raw_lengthscale;     /* (D,)       covariance_function.base_kernel.raw_lengthscale[dy,0]   */
    const void* raw_outputscale;     /* (1,)       covariance_function.raw_outputscale[dy]                 */
    const void* m;                   /* (M,)       q_U.variational_mean[dy]                                */
    const void* L_raw;               /* (M, M)     q_U.chol_variational_covar[dy] (lower-masked at use)    */
    const void* log_var_noise;       /* (1,)       likelihood.log_var_noise[dy] (unused for Bernoulli)     */
    const void* theta;               /* (n_theta,) flow scalars in descriptor order                        */
} TgpParams;

/* layout (in doubles) of the packed buffer that ranks all-reduce between tgp_qf_backward and tgp_chain_backward */
typedef struct TgpReduceLayout {
    long ell_sum, dlogvar, dos, dls, dtheta, dm, dZ, Gbar, Cbar, total;
    long packed_total;   /* doubles of the tril-packed form that travels in the all-reduce (tgp_reduce_pack) */
} TgpReduceLayout;

const char* tgp_last_error(void);
/* 102: retires library option 1 (tgp_set_option); 101: adds tgp_qf_backward_dx, tgp_flow_mlp_backward_dx and TgpGrads.dX
 * (input gradients); 100: the initial interface */
int tgp_version(void);

size_t tgp_step_workspace_bytes(const TgpModel* model);
size_t tgp_batch_workspace_bytes(const TgpModel* model, long R);
int tgp_reduce_layout(const TgpModel* model, TgpReduceLayout* out);

/* K_zz -> psd-safe Cholesky -> explicit L^-1, C = L_S^T L^-1, KL.
 * Replaces sparse_MF_SP.py:316,330,344-346 and KLD :406-431, utils.py:222-270 (the wrapper drives the jitter
 * ladder: status[0] > 0 is the 1-based index of the first non-positive pivot).  kl_out, status: device.
 * TGP_QU_UNWHITENED: L_S = L^-1 tril(L_raw) and L^-1 m replace tril(L_raw) and m (the whitened pair of the same q(u)), and
 * KL(N(m, P P^T) || N(0, L L^T)) uses the jittered L of the factorisation.  That KL needs L, so it is finished behind the
 * factorisation: kl_out is then ready in the caller's stream order once a consuming entry point (tgp_qf_forward,
 * tgp_qf_backward, tgp_chain_backward, tgp_qf_cov_forward) has been enqueued on it, or once tgp_factor_status() has returned. */
int tgp_prepare(const TgpModel* model, const TgpParams* params, double jitter, void* step_ws, double* kl_out,
                int* status, void* stream);

/* Blocks the HOST until the factorisation enqueued by the last tgp_prepare on the current device has finished (and only that:
 * kernels enqueued after it keep running) and returns its pivot status in *status_out — what the jitter ladder of
 * psd_safe_cholesky (utils.py:241-270) needs to decide.  Not available for a tgp_prepare recorded under graph capture. */
int tgp_factor_status(int* status_out);

/* q(f) marginals of R rows: mu, v (device, length R).  Saves A = K L^-T and B = K C^T in batch_ws for the backward.
 * Replaces sparse_MF_SP.marginal_variational_qf_parameters (sparse_MF_SP.py:274-396, whitened diagonal branch). */
int tgp_qf_forward(const TgpModel* model, const void* step_ws, void* batch_ws, const void* X, long R, void* mu,
                   void* v, void* stream);

/* ---- full covariance of q(f) over a test batch and joint samples (evaluation only, no backward) ---------------------
 * tgp_qf_cov_forward: mu (R) and Sigma = s Phi(X, X) - A A^T + B B^T (R x R, row-major, ld ldc >= R, exactly symmetric) of
 * R rows, A = K_xz L^-T, B = A L_S: the non-diagonal form of sparse_MF_SP.py:376-382.  Reads a step workspace prepared by
 * tgp_prepare in any compute mode and does not touch the batch workspace, so it may run between an ELBO forward and its
 * backward.  FP64 DMMA in every mode.  cov_ws: tgp_qf_cov_workspace_bytes(model, R) bytes, about (3M + 1) R doubles. */
size_t tgp_qf_cov_workspace_bytes(const TgpModel* model, long R);
int tgp_qf_cov_forward(const TgpModel* model, const void* step_ws, void* cov_ws, const void* X, long R, void* mu, void* cov,
                       long ldc, void* stream);

/* L (R x R, ld ldl, lower triangular, upper triangle exactly 0) = chol(cov + jitter I) with the blocked factorisation of
 * tgp_prepare; only the lower triangle of cov is read.  status (device): 0, or the 1-based index of the first pivot that is
 * not above 8 eps * scale_dev[0] (a device scalar, e.g. the outputscale).  chol_ws: tgp_cov_cholesky_workspace_bytes(R)
 * bytes (two Rp x Rp matrices, Rp = R rounded up to 64). */
size_t tgp_cov_cholesky_workspace_bytes(long R);
int tgp_cov_cholesky(long R, const void* cov, long ldc, double jitter, const double* scale_dev, void* chol_ws, void* L, long ldl,
                     int* status, void* stream);

/* out (S x R, row-major) = mu + eps L^T for eps (S x R) drawn by the caller: S joint samples from N(mu, L L^T). */
int tgp_cov_sample(long R, int S, const void* mu, const void* L, long ldl, const void* eps, void* out, void* stream);

/* Expected log-likelihood of R rows given (mu, v): flow o Gauss-Hermite o likelihood, with analytic gradients.
 * Replaces likelihood.expected_log_prob (GaussianNonLinearMean.py:113-150, GaussianLinearMean.py:60-87,
 * Bernoulli.py:50-95) and sparse_MF_SP.ELL's N/MB scaling (sparse_MF_SP.py:601-626; `scale` = N/MB_global).
 * Outputs: ell_rows (R, unscaled), g_mu / g_v (R, scaled), drowparams (R, n_rowparams, scaled) and, ACCUMULATED
 * into the caller-zeroed reduce buffer: ell_sum (unscaled), dlogvar, dtheta (scaled).  want_grad = 0 skips grads. */
int tgp_ell_forward(const TgpModel* model, const TgpParams* params, const void* mu, const void* v, const void* Y,
                    const void* rowparams, long R, double scale, const void* quad_t, const void* quad_w,
                    int want_grad, void* ell_rows, void* g_mu, void* g_v, void* drowparams, double* reduce_buf,
                    void* stream);

/* Backward of tgp_qf_forward for upstream per-row gradients (g_mu, g_v): accumulates the pre-chain quantities
 * (Gbar = dELL/dL^-1, Cbar = dELL/dC, dm, dZ, dlengthscale, doutputscale from the K_xz side) into reduce_buf.
 * Replaces autograd through sparse_MF_SP.py:313-382 (trainer_base.py:341).  Must follow tgp_qf_forward on the SAME
 * batch workspace and rows: it consumes the [A | B] rows the forward left there and K_xz — as stored FP64 values in
 * TGP_F64 / TGP_F32 mode, as the forward's residue planes in TGP_F64_I8 mode, where the FP64 K_xz tiles needed for the
 * kernel-parameter gradients are RECOMPUTED from X and Z (K_xz is never written in FP64 for D <= 32). */
int tgp_qf_backward(const TgpModel* model, const TgpParams* params, const void* step_ws, void* batch_ws,
                    const void* X, long R, const void* g_mu, const void* g_v, double* reduce_buf, void* stream);
/* tgp_qf_backward, and also the gradient w.r.t. the inputs X of sum_n g_mu[n] mu_n + g_v[n] v_n, ACCUMULATED into the
 * caller-zeroed dX (R, D) (D <= 64).  dX = NULL computes nothing more: tgp_qf_backward is this call with dX = NULL.  dX is
 * row-local: under row sharding each rank gets its own rows, and it takes no part in the reduce buffer's all-reduce. */
int tgp_qf_backward_dx(const TgpModel* model, const TgpParams* params, const void* step_ws, void* batch_ws,
                       const void* X, long R, const void* g_mu, const void* g_v, double* reduce_buf, void* dX, void* stream);

/* The replicated O(M^3) chain after the all-reduce: (Gbar, Cbar) -> L_S, L^-1 -> L -> K_zz -> Z, lengthscale,
 * outputscale, plus the KL gradient.  Outputs are d(gE*ELL + gK*KL)/dparam in the raw parameterisation:
 * dZ (M,D), draw_lengthscale (D), draw_outputscale (1), dm (M), dL_raw (M,M; upper triangle exactly 0),
 * dlog_var_noise (1), dtheta (n_theta).  Replaces autograd's cholesky_backward / triangular_solve_backward.
 * g_dev: optional DEVICE pointer to {gE, gK}; when non-NULL it overrides the host scalars (no host sync needed to
 * read autograd's upstream gradients).  TGP_QU_UNWHITENED: dm and dL_raw are the gradients w.r.t. the user's m and L_raw;
 * the chain first forms the adjoints of the whitened pair (L^-1 m, L^-1 P) and maps them back, and the KL term reaches
 * K_zz (and so Z, lengthscale, outputscale) through L.  gE = 0 is valid (the KL alone). */
int tgp_chain_backward(const TgpModel* model, const TgpParams* params, void* step_ws, const double* reduce_buf,
                       double gE, double gK, const double* g_dev, void* dZ, void* draw_lengthscale, void* draw_outputscale, void* dm,
                       void* dL_raw, void* dlog_var_noise, void* dtheta, void* stream);

/* Posterior-predictive samples and 95 % interval coverage per row, from the marginals (mu, v) of the test-NLL pass — replaces
 * sample_from_predictive_distribution (sparse_MF_SP.py:886-992: S x the cost of q(f)) + numpy.quantile + the coverage count of
 * trainers_regression.py:181-224.  Gaussian likelihoods only.  S <= 128 samples per row (Philox stream: seed, *offset_dev, which
 * the call advances); q_lo / q_hi: numpy.quantile-interpolated quantiles at q_lo_p / q_hi_p; covered: 1.0 where q_lo <= y <= q_hi;
 * samples (optional, R x S); count (optional device double): += covered rows.  rowparams: (R, n_mc, n_rowparams), n_mc in {1, S}. */
int tgp_coverage_rows(const TgpModel* model, const TgpParams* params, const void* mu, const void* v, const void* Y,
                      const void* rowparams, long R, int n_mc, int S, unsigned long long seed, unsigned long long* offset_dev,
                      double q_lo_p, double q_hi_p, void* q_lo, void* q_hi, void* covered, void* samples, double* count,
                      void* stream);

/* Monte-Carlo expected log-likelihood of the multiclass softmax likelihood — replaces
 * MulticlassCategorical.expected_log_prob (likelihoods/MulticlassCategorical.py:51-105) and, with probs != NULL,
 * marginal_moments (:109-151).  One GP per class: mu, v are (C, R); eps (S, C, R) is the N(0,1) noise of td.Normal.rsample,
 * drawn by the caller (the reference's generator stream); the C flows share model->layers (global parameters only; per-row
 * flows go through tgp_mc_softmax_rows_rowp) and own
 * one row each of theta (C, n_theta); Y holds the labels 0..C-1 as doubles.
 *   ell_rows[n] = 1/S sum_s log softmax(G(mu + sqrt(v) eps_s))[y_n]
 * want_grad: g_mu, g_v (C, R) = d ell_rows[n] / d mu[c,n], d v[c,n] (unscaled); dtheta (C, n_theta) += d sum_n ell_rows[n] / d theta
 * (caller zeroes).  probs (optional, R x C) = 1/S sum_s softmax.  C <= 32, C * n_theta <= 256. */
int tgp_mc_softmax_rows(const TgpModel* model, int C, int S, long R, const void* mu, const void* v, const void* Y, const void* eps,
                        const void* theta, int want_grad, void* ell_rows, void* g_mu, void* g_v, void* dtheta, void* probs,
                        void* stream);
/* tgp_mc_softmax_rows for input-dependent flows (ID_TGP): the layers flagged TGP_FLOW_PER_ROW take their raw parameters from
 * rowparams (C, R, n_rowparams), row-major: rowparams[(c R + n) n_rowparams + k] is parameter k of class c's flow at row n, the
 * class-stacked MLP outputs evaluated once on X for the call and shared by all S samples.  The C flows share model->layers (one
 * architecture; TgpFlowLayer.p0 indexes theta for global layers and the row vector for per-row ones).  want_grad: drowparams
 * (C, R, n_rowparams) = d ell_rows[n] / d rowparams[c,n,k], WRITTEN (not accumulated) and unscaled like g_mu / g_v; dtheta as in
 * tgp_mc_softmax_rows.  n_rowparams <= 16 and C * n_rowparams <= 256.  With model->n_rowparams = 0 (rowparams, drowparams
 * ignored) this is tgp_mc_softmax_rows, bit for bit. */
int tgp_mc_softmax_rows_rowp(const TgpModel* model, int C, int S, long R, const void* mu, const void* v, const void* Y,
                             const void* eps, const void* theta, int want_grad, void* ell_rows, void* g_mu, void* g_v, void* dtheta,
                             void* probs, const void* rowparams, void* drowparams, void* stream);

/* The exchange format of the one collective per step (SURVEY.md 8e).  The reduce buffer holds two (padded) M x M blocks
 * of which only the lower triangles are populated in TGP_F64 mode (Gbar and dL_S; in TGP_F32 mode the second block, Cbar,
 * is dense): tgp_reduce_pack gathers [small vector | tril(Gbar) | tril or full second block] into `packed`
 * (layout.packed_total doubles: 8.5 MB instead of 16.9 MB at M = 1024), ranks sum `packed`, tgp_reduce_unpack scatters it
 * back for tgp_chain_backward. */
int tgp_reduce_pack(const TgpModel* model, const double* reduce_buf, double* packed, void* stream);
int tgp_reduce_unpack(const TgpModel* model, const double* packed, double* reduce_buf, void* stream);

/* Test log-likelihood rows and predictive moments given (mu, v) (sparse_MF_SP.py:637-825; marginal_moments of the
 * three likelihoods).  rowparams: (R, n_mc, n_rowparams) for MC-dropout flows, n_mc = 1 otherwise.
 * bern_std: device scalar, batch-wide std of v (Bernoulli.py:120 defect, kept for parity). */
int tgp_test_rows(const TgpModel* model, const TgpParams* params, const void* mu, const void* v, const void* Y,
                  const void* rowparams, long R, int n_mc, double y_std, const void* quad_t, const void* quad_w,
                  const double* bern_std, void* logp_rows, void* m1, void* m2, void* stream);

/* ---- input-dependent flow parameters (ID_TGP) ------------------------------------------------------------------------
 * The MLPs theta(x_n) of an input-dependent flow layer (models/flow.py:853-871 builds them, :949-950 evaluates them once
 * per call on X; dropout active in training, sparse_MF_SP.py:133-134).  n_nets independent nets x -> R, each
 * n_hidden_layers x [Linear(.., hidden) -> activation -> Dropout(p)] + Linear(hidden, 1).  Weights are packed per net as
 * [W0 (hidden x n_in), b0 (hidden), W1 (hidden x hidden), b1, ..., w_out (hidden), b_out] (torch Linear.weight order).
 * mask_mode: 0 = no dropout; 1 = Philox-4x32-10 stream (seed, *offset_dev; the forward bumps *offset_dev and EXPORTS the
 * keep-mask to mask_out, which must be non-NULL); 2 = explicit keep-mask mask_in.  Mask layout (n_nets, n_hidden_layers, R,
 * hidden) bytes.  The backward consumes the mask of the forward (NULL for mode 0) and ACCUMULATES into dweights. */
typedef struct TgpMlp {
    int n_nets, n_in, hidden, n_hidden_layers;
    int activation;                  /* 0 relu, 1 tanh, 2 sigmoid, 3 linear */
    int mask_mode;
    double p_drop;
} TgpMlp;
long tgp_flow_mlp_net_doubles(const TgpMlp* mlp);
int tgp_flow_mlp_forward(const TgpMlp* mlp, const void* weights, const void* X, long R, const unsigned char* mask_in,
                         unsigned char* mask_out, unsigned long long seed, unsigned long long* offset_dev, void* out,
                         void* stream);
int tgp_flow_mlp_backward(const TgpMlp* mlp, const void* weights, const void* X, long R, const unsigned char* mask,
                          const void* dout, void* dweights, void* stream);
/* tgp_flow_mlp_backward, and also the gradient w.r.t. X (R, n_in), ACCUMULATED into dX; NULL computes nothing more */
int tgp_flow_mlp_backward_dx(const TgpMlp* mlp, const void* weights, const void* X, long R, const unsigned char* mask,
                             const void* dout, void* dweights, void* dX, void* stream);

/* ---- single-call interface (the entry points SURVEY.md 8b proposes), thin over the stages above -------------------
 * A TgpHandle is a HOST object created once per (model description, device, maximum minibatch rows): it remembers the
 * model, the caller-owned workspace (ONE device allocation of tgp_workspace_bytes(), bound with tgp_bind_workspace and
 * validated against the size the handle needs) and where the per-step / per-batch / reduce / per-row regions live in
 * it.  The library still never allocates device memory.  Reference seam: the body of sparse_MF_SP.ELBO
 * (sparse_MF_SP.py:552-598), its autograd backward (trainer_base.py:341) and test_log_likelihood (:637-825). */
typedef struct TgpHandle TgpHandle;
typedef struct TgpBatch {           /* one minibatch (device pointers) */
    const void* X;                  /* (R, D) */
    const void* Y;                  /* (R,)   */
    const void* rowparams;          /* (R, n_rowparams) input-dependent flow parameters, NULL otherwise */
    long R;
    double scale;                   /* N / MB_global (sparse_MF_SP.py:626) */
    const void* quad_t; const void* quad_w;     /* Gauss-Hermite rule (n_quad,), NULL for the closed-form likelihood */
} TgpBatch;
typedef struct TgpFwdOut {          /* device pointers; any of ell_rows / mu / v may be NULL */
    double* terms;                  /* [0] = scale * sum_n ell_n (this rank's rows), [1] = KL */
    int* status;                    /* 0, or 1-based index of the first non-positive pivot (caller drives the jitter ladder) */
    void* ell_rows; void* mu; void* v;          /* (R,) each */
} TgpFwdOut;
typedef struct TgpGrads {           /* device pointers, raw parameterisation; same meaning as tgp_chain_backward's outputs */
    void* dZ; void* draw_lengthscale; void* draw_outputscale; void* dm; void* dL_raw; void* dlog_var_noise; void* dtheta;
    void* drowparams;               /* (R, n_rowparams), NULL when the flow is not input-dependent */
    void* dX;                       /* (R, D) d(g[0] * ELL)/dX, written; NULL = not computed (tgp_version() >= 101: callers
                                     * built against an older header must rebuild and zero-initialise the struct) */
} TgpGrads;
/* Sum `count` doubles at `buf` over the ranks of the job, enqueued on `stream` (e.g. ncclAllReduce).  NULL = one rank. */
typedef int (*TgpAllReduceFn)(double* buf, long count, void* user, void* stream);

size_t tgp_workspace_bytes(const TgpModel* model, long max_rows);
int tgp_create(const TgpModel* model, long max_rows, TgpHandle** out);
void tgp_destroy(TgpHandle* h);
int tgp_bind_workspace(TgpHandle* h, void* workspace, size_t bytes);
/* forward of one minibatch: prepare (jitter on the K_zz diagonal) + marginals + expected log-likelihood; keeps what the
 * backward needs in the workspace */
int tgp_elbo_fwd(TgpHandle* h, const TgpParams* params, const TgpBatch* batch, double jitter, const TgpFwdOut* out,
                 void* stream);
/* backward of the last tgp_elbo_fwd on this handle: d(g[0] * ELL + g[1] * KL)/dparam with {g[0], g[1]} read from DEVICE
 * memory `g_dev`; `allreduce` (may be NULL) is called once, between the batch pass and the replicated O(M^3) chain, on
 * the tril-packed buffer */
int tgp_elbo_bwd(TgpHandle* h, const TgpParams* params, const TgpBatch* batch, const double* g_dev,
                 const TgpGrads* grads, TgpAllReduceFn allreduce, void* user, void* stream);
/* test log-likelihood rows + predictive moments of one batch (prepare + marginals + tgp_test_rows); refactor = 0 reuses
 * the factorisation already in the workspace (frozen parameters across evaluation batches) */
int tgp_test_nll_fwd(TgpHandle* h, const TgpParams* params, const TgpBatch* batch, int refactor, int n_mc, double y_std,
                     const double* bern_std, void* logp_rows, void* m1, void* m2, void* mu, void* v, int* status,
                     void* stream);

/* ---- optimiser step next to the path (SURVEY.md 8f rank 2) ---------------------------------------------------------------
 * Adam / AdamW-style update of ALL parameter tensors in one launch, with torch.optim.Adam's arithmetic (trainer_base.py:342
 * via optimizers.py:10-22): g += wd p;  m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2;  p -= lr / (1 - b1^t) * m / (sqrt(v) /
 * sqrt(1 - b2^t) + eps).  The step count t lives in DEVICE memory and is incremented by the kernel (graph-replay safe).
 * Tables (device): per tensor the addresses of param / grad / exp_avg / exp_avg_sq (n_tensors x 4 pointers, row-major), its
 * element count, learning rate and weight decay; per 4096-element block its tensor index and element offset.  All FP64. */
int tgp_adam_step(int n_tensors, long n_blocks, const void* const* ptr_table, const long* sizes, const double* lr,
                  const double* weight_decay, const int* block_tensor, const long* block_offset, double beta1, double beta2,
                  double eps, long* step_dev, void* stream);

/* ---- inducing-point initialisation next to the path (SURVEY.md 8f rank 4) -------------------------------------------------
 * One Lloyd iteration of k-means on the device (reference: Z = KMEANS(X_tr, M), utils.py:143-159 / main.py:145, sklearn on the
 * host).  X (N, D) FP64, centroids C (M, D) updated in place when update != 0; assign (N) int32 or NULL; scratch: sums (M, D),
 * counts (M), inertia (1) — zeroed by the call; inertia[0] = sum of squared distances to the nearest OLD centroid.  D <= 32. */
int tgp_kmeans_iteration(const void* X, long N, int D, void* C, int M, int* assign, double* sums, double* counts,
                         double* inertia, int update, void* stream);

/* Library options.  Key 1 (the single-kernel tensor-core forward) is retired: it is an unknown option since tgp_version() 102.
 * TGP_OPT_ROW_CHUNK (FP64 mode): rows per launch of the batch contractions (default 32768; a tuning knob — it changes the
 * workspace size, so set it before asking for tgp_batch_workspace_bytes). */
enum { TGP_OPT_ROW_CHUNK = 2,
       TGP_OPT_OVERLAP_KGEN = 3 };   /* 1 (default): tgp_prepare forks the factorisation onto a library-owned high-priority stream;
                                      * tgp_qf_forward enqueues K_xz generation on the caller's stream and joins afterwards, every
                                      * other consumer of the step workspace joins first; 0: everything on the caller's stream.
                                      * Either way the outputs of each entry point are ready in the order of the caller's stream
                                      * once a consuming entry point has been enqueued on it; kl_out is in stream order for
                                      * whitened models (see tgp_prepare for non-whitened ones), status is read with
                                      * tgp_factor_status() */
int tgp_set_option(int key, int value);

/* Number of kernels this library has launched so far in the process (bench.py's gpu_launches). */
long tgp_launch_count(void);
/* Live per-launch timing of the GEMM kernel with CUDA events on the launching stream (bench.py's roofline).
 * Returns the accumulated milliseconds / launch counts per class ([0] FP64 per-step O(M^3) work, [1] FP64 batch
 * contractions, [2] tcgen05 batch contractions) since the last reset into ms_out[3] / launches_out[3] (host, may be NULL), then enable = 1 / 0 switches the
 * instrumentation on / off and resets the accumulators; enable < 0 only reads.  Synchronises on the recorded events. */
int tgp_gemm_timing(int enable, double* ms_out, long* launches_out);

/* Test hook: the FP64 DMMA GEMM that carries every contraction (C = alpha*Aop*Bop^T + beta*C). */
int tgp_debug_gemm_f64(int M, int N, int K, const double* A, long lda, int a_layout, const double* B, long ldb,
                       int b_layout, double* C, long ldc, double alpha, double beta, int a_tri, int b_tri,
                       int c_lower, void* stream);
/* Test hook: the tcgen05 3xTF32 GEMM of the FP32 mode.  D[m,n] (+)= sum_k A[m,k] B[n,k]; operands are K-major FP32 plane
 * pairs (x, x - tf32_trunc(x)); out_mode 0 stores FP32 into Cf, out_mode 1 atomically adds into FP64 Cd. */
int tgp_debug_gemm_tf32x3(int Mrows, int Ncols, int K, const float* Ahi, const float* Alo, long lda, const float* Bhi,
                          const float* Blo, long ldb, float* Cf, double* Cd, long ldc, int out_mode, int tri_mode,
                          int tri_rows, int lower_rows, int splitk, void* stream);
/* Test hook: C (+)= A B^T (A: M x K, B: N x K, row-major FP64) through the integer-residue pipeline of TGP_F64_I8 with T
 * moduli (9, 12, 15 or 16); tri_mode / tri_rows / lower_rows as in the tf32x3 hook; mn_major bit 0 / 1: A / B is passed transposed ((K x M) /
 * (K x N)) and the tensor core reads it MN-major; scratch: tgp_debug_gemm_crt_bytes() device bytes. */
size_t tgp_debug_gemm_crt_bytes(long M, long N, long K, int T);
int tgp_debug_gemm_crt(long M, long N, long K, const double* A, long lda, const double* B, long ldb, double* C, long ldc,
                       int T, int tri_mode, int tri_rows, int lower_rows, int accumulate, int mn_major, void* scratch,
                       void* stream);
/* Test hook: copies L, L^-1, C (each M x M, row-major, ld = M) out of a prepared step workspace. */
int tgp_debug_export_step(const TgpModel* model, const void* step_ws, double* L, double* Linv, double* C,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif
