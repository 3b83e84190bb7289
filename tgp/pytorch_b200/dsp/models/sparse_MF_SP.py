"""Sparse variational (transformed) GP — host-side mirror of reference code/dsp/models/sparse_MF_SP.py.

Same constructor, attributes and method signatures as the reference class (:47-120, 274, 398, 457, 552, 601, 637,
837-992).  The arithmetic of `ELBO`, `marginal_variational_qf_parameters`, `ELL`, `predictive_distribution` and
`test_log_likelihood` is enqueued on the B200 through libtgp_b200.so (tgp/pytorch_b200/functional.py); this file only
gathers parameters from the unchanged nn.Module tree and shapes the results like the reference does.

Scope of the fused path (anything else raises, nothing falls back to the CPU): whitened or non-whitened q(u), zero mean, (Scale)RBF-ARD or
(Scale)Matern-ARD (nu = 1/2, 3/2, 5/2) kernel, FP64 (what the reference's main.py runs), flows made of affine / tanh-step / sinh-arcsinh
layers (optionally input-dependent with MC-dropout MLPs).  Multi-output models loop over outputs.  Marginals are differentiable;
the full covariance over a batch (`diagonal=False`) and the joint samples drawn from it are evaluation-only (no backward).
"""
import numpy
import torch
import torch.nn as nn
import torch.distributions as td

from .. import config as cg
from ... import functional as Fn
from ...engine import Engine, FlowLayout
from ..kernels import CholeskyVariationalDistribution, ScaleKernel, RBFKernel, MaternKernel
from ..likelihoods.GaussianLinearMean import GaussianLinearMean
from ..likelihoods.GaussianNonLinearMean import GaussianNonLinearMean
from ..likelihoods.Bernoulli import Bernoulli
from ..likelihoods.MulticlassCategorical import MulticlassCategorical
from ..likelihoods import _rows
from ..quadrature import GaussHermiteQuadrature1D
from .config_models import get_init_params
from .flow import instance_flow
from .utils_models import return_mean, enable_eval_dropout

_LIK_KIND = {GaussianLinearMean: 'gauss_linear', GaussianNonLinearMean: 'gauss_nonlinear', Bernoulli: 'bernoulli'}
_INV_SOFTPLUS_ONE = 0.5413248546129181       # softplus^-1(1): outputscale of a bare (unscaled) kernel
_MATERN_KIND = {0.5: 'matern12', 1.5: 'matern32', 2.5: 'matern52'}


class sparse_MF_SP(nn.Module):
    def __init__(self, model_specs, X, init_Z, N, likelihood, num_outputs, is_whiten, K_is_shared, mean_is_shared,
                 Z_is_shared, q_U_is_shared, flow_specs, flow_connection, add_noise_inducing, be_fully_bayesian=False,
                 init_params={}):
        super().__init__()
        assert len(model_specs) == 2, 'Parameter model_specs should be len 2: mean name and kernel instance'
        self.out_dim = int(num_outputs)
        self.inp_dim = int(init_Z.size(1))
        self.kernel_is_shared = K_is_shared
        self.mean_is_shared = mean_is_shared
        self.Z_is_shared = Z_is_shared
        self.q_U_is_shared = q_U_is_shared
        self.N = float(N)
        self.M = init_Z.size(0)
        self.likelihood = likelihood
        self.fully_bayesian = be_fully_bayesian
        self.init_params = get_init_params(init_params)
        self._standard_sampler = None     # built on first use (the reference builds it eagerly, sparse_MF_SP.py:96-97)
        self.is_training = True
        self.quad_points = likelihood.quad_points if isinstance(likelihood, GaussianNonLinearMean) else cg.quad_points
        self.quad = GaussHermiteQuadrature1D(self.quad_points)

        self.initialize_inducing(init_Z, add_noise_inducing)
        self.initialize_variational_distribution(is_whiten)
        self.initialize_mean_function(X, model_specs)
        self.initialize_covariance_function(model_specs)
        self.G_matrix, self.G_flow_connection = self.initialize_flows(flow_connection, flow_specs)
        self.l2_regularize = False
        self.global_batch_rows = None     # row-sharded training: rows of the GLOBAL minibatch (default MB * world)
        self._engines = {}
        self._last = None

    # ---- configuration -------------------------------------------------------------------------------------------
    @property
    def standard_sampler(self):
        """N(0, I_1), the reference's attribute of the same name; scale_tril is given explicitly so that constructing it
        factorises nothing."""
        if self._standard_sampler is None:
            self._standard_sampler = td.MultivariateNormal(torch.zeros(1, device=cg.device), scale_tril=torch.eye(1, device=cg.device))
        return self._standard_sampler

    def be_fully_bayesian(self, mode):
        self.fully_bayesian = mode

    def set_is_training(self, mode):
        self.is_training = mode
        self._invalidate_eval_cache()

    def _invalidate_eval_cache(self):
        """Forget factorisations cached for evaluation batches (see functional._QfMarginals)."""
        for eng in self._engines.values():
            eng.prepared_key = None

    def initialize_inducing(self, init_Z, add_noise_inducing):
        if self.Z_is_shared:
            self.Z = nn.Parameter(init_Z.unsqueeze(dim=0))
            return
        Z = torch.zeros(self.out_dim, self.M, self.inp_dim)
        for l in range(self.out_dim):
            z = init_Z.clone()
            if add_noise_inducing > 0.0:
                power = numpy.random.randn(self.M, self.inp_dim)
                z = init_Z * torch.tensor(add_noise_inducing * power, dtype=cg.dtype).detach()
            Z[l, :] = z
        self.Z = nn.Parameter(Z)

    def initialize_variational_distribution(self, is_whiten):
        o_d = 1 if self.q_U_is_shared else self.out_dim
        q_U = CholeskyVariationalDistribution(self.M, batch_shape=torch.Size([o_d]))
        vd = self.init_params['variational_distribution']
        q_U.chol_variational_covar.data = torch.eye(self.M, self.M).view(1, self.M, self.M).repeat(o_d, 1, 1) * \
            numpy.sqrt(vd['variance_scale'])
        q_U.variational_mean.data = torch.ones(o_d, self.M) * vd['mean_scale']
        self.is_whiten = is_whiten
        self.q_U = q_U

    def initialize_mean_function(self, X, model_specs):
        self.mean_function = return_mean(model_specs[0], self.inp_dim, self.out_dim, None)

    def initialize_covariance_function(self, model_specs):
        kernel = model_specs[1]
        if cg.strict_flag:
            want = torch.Size([1]) if self.kernel_is_shared else torch.Size([self.out_dim])
            assert kernel.batch_shape == want, 'Got a kernel with batch_shape {}, expected {}'.format(kernel.batch_shape, want)
        base = kernel.base_kernel if isinstance(kernel, ScaleKernel) else kernel
        if not isinstance(base, (RBFKernel, MaternKernel)):
            raise NotImplementedError('the fused path covers (Scale)RBF-ARD and (Scale)Matern-ARD kernels')
        self.covariance_function = kernel

    def _kernel_kind(self):
        """Engine kernel name of the covariance function ('rbf', 'matern12', 'matern32', 'matern52')."""
        kern = self.covariance_function
        base = kern.base_kernel if isinstance(kern, ScaleKernel) else kern
        return _MATERN_KIND[base.nu] if isinstance(base, MaternKernel) else 'rbf'

    def initialize_flows(self, flow_connection, flow_specs):
        if flow_connection == 'shared':
            assert len(flow_specs) == 1, 'option shared takes exactly one flow specification'
        elif flow_connection == 'single':
            assert len(flow_specs) == self.out_dim, 'option single takes one flow specification per output'
        else:
            raise ValueError('Invalid value {} for argument flow_connection'.format(flow_connection))
        G = []
        if flow_connection == 'single':
            for fl in flow_specs:
                G.append(instance_flow(fl) if type(fl) == list else fl)
        return nn.ModuleList(G), flow_connection

    # ---- parameter gathering for the kernels ---------------------------------------------------------------------
    def _check_fused_scope(self, X):
        if X.dtype not in (torch.float64, torch.float32):
            raise NotImplementedError('inputs must be float64 (cg.set_maximum_precission(), as main.py does) or float32')
        if not X.is_cuda:
            raise RuntimeError('tgp.pytorch_b200 has no CPU path: move the model and the data to a CUDA device')

    def _gp_params(self, dy):
        """(Z, raw_ls, raw_os, m, L_raw) of output `dy` as contiguous autograd views of the module parameters."""
        zi = 0 if self.Z_is_shared else dy
        ki = 0 if self.kernel_is_shared else dy
        qi = 0 if self.q_U_is_shared else dy
        kern = self.covariance_function
        if isinstance(kern, ScaleKernel):
            raw_ls, raw_os = kern.base_kernel.raw_lengthscale[ki, 0], kern.raw_outputscale[ki:ki + 1]
        else:
            raw_ls = kern.raw_lengthscale[ki, 0]
            raw_os = torch.full((1,), _INV_SOFTPLUS_ONE, dtype=torch.float64, device=raw_ls.device)
        if raw_ls.numel() != self.inp_dim:
            raw_ls = raw_ls.expand(self.inp_dim)
        # float32 models (the reference's import-time default, config.py:53-58) are served by the tensor-core mode:
        # parameters are up-cast here (autograd casts the gradients back), the contractions run as 3xTF32
        d = torch.float64
        return (self.Z[zi].to(d).contiguous(), raw_ls.to(d).contiguous(), raw_os.to(d).contiguous(),
                self.q_U.variational_mean[qi].to(d).contiguous(), self.q_U.chol_variational_covar[qi].to(d).contiguous())

    def _noise(self, dy):
        lik = self.likelihood
        if isinstance(lik, Bernoulli):
            return None
        lv = lik.log_var_noise
        return lv[0 if lik.noise_is_shared else dy].reshape(1).to(torch.float64)

    def _engine(self, dy, layout, device):
        kind = _LIK_KIND[type(self.likelihood)]
        key = (dy, kind, self.quad_points, tuple(tuple(sorted(l.items())) for l in layout.layers), str(device), self._compute(),
               self._kernel_kind(), bool(self.is_whiten))
        if key not in self._engines:
            self._engines[key] = Engine(self.M, self.inp_dim, kind, self.quad_points if kind != 'gauss_linear' else 0,
                                        layout, device, compute=self._compute(), kernel=self._kernel_kind(), whiten=self.is_whiten)
        return self._engines[key]

    def _compute(self):
        return cg.compute if self.Z.dtype == torch.float64 else 'tf32x3'

    def _jitter(self):
        """(constant jitter, ladder base) of psd_safe_cholesky as the reference configures it: cg.constant_jitter is added
        to the K_zz diagonal before every factorisation (utils.py:237), cg.global_jitter is the base of the failure
        ladder (sparse_MF_SP.py:330), defaulting to 1e-8 for float64 and 1e-6 for float32 models (utils.py:258)."""
        base = cg.global_jitter if cg.global_jitter is not None else (1e-8 if self.Z.dtype == torch.float64 else 1e-6)
        return (float(cg.constant_jitter) if cg.constant_jitter is not None else 0.0, float(base))

    def _rows3(self, X):
        if len(X.shape) == 2:
            X = X.unsqueeze(0).expand(self.out_dim, -1, -1)
        assert len(X.shape) == 3, 'Invalid input X.shape'
        return X

    def _global_scale(self, MB):
        from ...dist import global_scale
        dist = Fn._world()
        rows = self.global_batch_rows
        if rows is None:
            rows = MB * (dist.get_world_size() if dist is not None else 1)
        return global_scale(self.N, rows)

    # ---- model computation ---------------------------------------------------------------------------------------
    def _qf_engine(self, dy, device):
        """The engine of the q(f) evaluations of output `dy` (marginals and full covariance share it, and with it the cached
        factorisation); they do not involve the flow / likelihood."""
        key = ('qf', dy, str(device), self._compute(), self._kernel_kind(), bool(self.is_whiten))
        if key not in self._engines:
            self._engines[key] = Engine(self.M, self.inp_dim, 'gauss_linear', 0, FlowLayout([]), device,
                                        compute=self._compute(), kernel=self._kernel_kind(), whiten=self.is_whiten)
        eng = self._engines[key]
        if not cg.cache_factorisation_in_eval:
            eng.prepared_key = None
        return eng

    def _joint_qf(self, X, is_duvenaud):
        """[(engine, mu (MB,), Sigma (MB, MB))] per output, FP64, for rows X (Dy, MB, D): the full covariance of q(f)."""
        if is_duvenaud:
            raise NotImplementedError('is_duvenaud (the deep-GP form) is outside the fused single-layer path')
        self._check_fused_scope(X)
        out = []
        for dy in range(self.out_dim):
            eng = self._qf_engine(dy, X.device)
            mu, cov = Fn.qf_covariance(eng, X[dy].to(torch.float64).contiguous(), *self._gp_params(dy),
                                       cg.check_cholesky_status, self._jitter())
            out.append((eng, mu, cov))
        return out

    def _joint_samples(self, joint, S):
        """f0 (Dy, S, MB) FP64: S joint samples mu + e L^T per output, L = psd_safe_cholesky(Sigma), e ~ N(0, I) (Dy, S, MB)
        drawn here from torch's generator in FP64."""
        MB = joint[0][1].shape[0]
        e = torch.randn(self.out_dim, S, MB, dtype=torch.float64, device=joint[0][1].device)
        constant, base = self._jitter()
        f0 = []
        for dy, (eng, mu, cov) in enumerate(joint):
            L, _ = Fn.cov_cholesky_ladder(eng, cov, base, constant)
            f0.append(eng.cov_sample(mu, L, e[dy].contiguous()))
        return torch.stack(f0)

    def marginal_variational_qf_parameters(self, X, diagonal, is_duvenaud, init_Z=None):
        """q(f) = int p(f|u) q(u) du at the rows of X: mean (Dy,MB,1) and diagonal covariance (Dy,MB,1), or with
        diagonal=False the full covariance over the rows (Dy,MB,MB).  The full covariance has no backward: call it under
        torch.no_grad().  Under row sharding it is the covariance of this rank's rows."""
        X = self._rows3(X)
        if not diagonal:
            joint = self._joint_qf(X, is_duvenaud)
            mean = torch.stack([mu for _, mu, _ in joint]).unsqueeze(2)
            return mean.to(self.Z.dtype), torch.stack([cov for _, _, cov in joint]).to(self.Z.dtype)
        if is_duvenaud:
            raise NotImplementedError('is_duvenaud (the deep-GP form) is outside the fused single-layer path')
        mean, cov, _ = self._marginals(X)
        return mean, cov

    def _marginals(self, X, with_kl=False):
        """q(f) marginals (Dy,MB,1) x 2 at the rows of X (Dy,MB,D), and with_kl=True the KL term of each output (Dy,) from
        the same factorisation (else None)."""
        self._check_fused_scope(X)
        mus, vs, kls = [], [], []
        for dy in range(self.out_dim):
            Z, raw_ls, raw_os, m, L_raw = self._gp_params(dy)
            eng = self._qf_engine(dy, X.device)
            out = Fn.qf_marginals(eng, X[dy].to(torch.float64).contiguous(), Z, raw_ls, raw_os, m, L_raw,
                                  cg.check_cholesky_status, self._jitter(), with_kl=with_kl)
            mus.append(out[0])
            vs.append(out[1])
            if with_kl:
                kls.append(out[2])
        d = self.Z.dtype
        return torch.stack(mus).unsqueeze(2).to(d), torch.stack(vs).unsqueeze(2).to(d), torch.stack(kls) if with_kl else None

    def _kl_engine(self, dy, device):
        """The engine of a stand-alone non-whitened KLD() of output `dy`: a factorisation of its own, so that KLD() leaves the
        workspaces of a pending ELBO or marginals backward alone.  The KL is FP64 in every compute mode: 'f64' suffices."""
        key = ('kl', dy, str(device), self._kernel_kind())
        if key not in self._engines:
            self._engines[key] = Engine(self.M, self.inp_dim, 'gauss_linear', 0, FlowLayout([]), device, compute='f64',
                                        kernel=self._kernel_kind(), whiten=False)
        return self._engines[key]

    def KLD(self):
        """KL[q(u) || p(u)] per output (Dy,).  Whitened: 0.5 (-log|S| + m'm + tr S - M), a few element-wise ops on the
        parameters; `ELBO` takes the same quantity from the fused prepare kernel.  Non-whitened: KL(N(m, S) || N(0, K_zz)),
        which needs the factorisation of K_zz (with the jitter ladder of the marginals): one prepare per output on an engine of
        its own, differentiable through the hand-written chain."""
        if not self.is_whiten:
            self._check_fused_scope(self.Z)
            kls = [Fn.kl_term(self._kl_engine(dy, self.Z.device), *self._gp_params(dy), jitter=self._jitter())
                   for dy in range(self.out_dim)]
            return torch.stack(kls).to(self.Z.dtype)
        m = self.q_U.variational_mean
        L = self.q_U.chol_variational_covar.tril()
        if self.q_U_is_shared:
            m, L = m.repeat(self.out_dim, 1), L.repeat(self.out_dim, 1, 1)
        logdet = torch.log(torch.diagonal(L, dim1=1, dim2=2) ** 2).sum(1)
        return 0.5 * (-logdet + (m * m).sum(1) + (L * L).sum((1, 2)) - float(self.M))

    def ELBO(self, X, Y):
        """(ELBO, ELL, KLD) for a minibatch — the fused forward; `.backward()` runs the fused backward kernels."""
        X = self._rows3(X)
        self._check_fused_scope(X)
        self._invalidate_eval_cache()
        assert self.G_flow_connection == 'single', 'sparse_MF_SP places one independent flow per output'
        MB = Y.size(0)
        scale = self._global_scale(MB)
        if isinstance(self.likelihood, MulticlassCategorical):
            return self._elbo_multiclass(X, Y, scale)
        kind = _LIK_KIND[type(self.likelihood)]
        ELL, KLD = 0.0, 0.0
        for dy in range(self.out_dim):
            Xd = X[dy].to(torch.float64).contiguous()
            Z, raw_ls, raw_os, m, L_raw = self._gp_params(dy)
            if kind == 'gauss_linear':
                layout, theta, rowp = FlowLayout([]), None, None
            else:
                layout, theta, rowp = _rows.flow_pack(self.G_matrix[dy], Xd)
            eng = self._engine(dy, layout, Xd.device)
            y = Y[:, dy].to(torch.float64).contiguous()
            ell, kl, _rows_ll, _mu, _v = Fn.elbo_terms(eng, Xd, y, scale, Z, raw_ls, raw_os, m, L_raw, self._noise(dy),
                                                       theta, rowp, cg.check_cholesky_status, self._jitter(),
                                                       cg.sync_elbo_in_forward)
            self._last = (eng, scale, kl)
            ELL = ELL + ell
            KLD = KLD + kl
        KLD_flow = 0.0
        for flow in self.G_matrix:
            KLD_flow = KLD_flow + flow.KLD()
        ELBO = ELL - KLD - KLD_flow
        out = self.Z.dtype
        return ELBO.to(out), ELL.to(out), (KLD + KLD_flow).to(out)

    def _elbo_multiclass(self, X, Y, scale):
        """One GP per class coupled by the softmax: the q(f) marginals of every class (fused forward, hand-written backward
        through `Fn.qf_marginals`), then ONE Monte-Carlo kernel over all classes (tgp_mc_softmax_rows).  Under row sharding the
        marginals' backward all-reduces its packed buffer (one collective per class) and the flow scalars are summed across
        ranks; the returned ELL is the global one when cg.sync_elbo_in_forward is set, else this rank's share."""
        if self.is_whiten:
            mean, cov = self.marginal_variational_qf_parameters(X, diagonal=True, is_duvenaud=False)
        else:   # each class's KL from the factorisation of its marginals (KLD() would factorise again and void their backward)
            mean, cov, kl_classes = self._marginals(X, with_kl=True)
        ell = self.likelihood.expected_log_prob(Y.t(), mean.squeeze(dim=2), cov.squeeze(dim=2), flow=self.G_matrix, X=X)
        dist = Fn._world()
        if dist is not None and cg.sync_elbo_in_forward:
            tot = ell.detach().clone()
            dist.all_reduce(tot)
            ell = ell + (tot - ell.detach())
        ELL = scale * ell
        KLD = self.KLD().sum() if self.is_whiten else kl_classes.sum()
        KLD_flow = 0.0
        for flow in self.G_matrix:
            KLD_flow = KLD_flow + flow.KLD()
        out = self.Z.dtype
        return (ELL - KLD - KLD_flow).to(out), ELL.to(out), (KLD + KLD_flow).to(out)

    def last_global_elbo(self):
        """Row-sharded training with cg.sync_elbo_in_forward = False: the ELBO over the GLOBAL minibatch of the last step,
        read (after backward()) from slot 0 of the one all-reduced buffer — no extra collective.  Single-output models."""
        eng, scale, kl = self._last
        if eng.last_ell_sum is None:
            raise RuntimeError('last_global_elbo() is valid after backward() of the last ELBO')
        return scale * eng.last_ell_sum - kl.detach()

    def ELL(self, X, Y, mean, cov):
        """(N/MB) * E_q(f)[log p(y|G(f))] per output from given marginals (Dy,MB,1)."""
        assert self.G_flow_connection == 'single', 'sparse_MF_SP places one independent flow per output'
        X = self._rows3(X)
        MB = Y.size(0)
        ell = self.likelihood.expected_log_prob(Y.t(), mean.squeeze(dim=2), cov.squeeze(dim=2), flow=self.G_matrix, X=X)
        return self.N / MB * ell

    # ---- prediction ----------------------------------------------------------------------------------------------
    def _eval_mode(self):
        self.eval()
        if self.fully_bayesian:
            assert enable_eval_dropout(self.modules()), 'fully bayesian mode needs dropout layers in the flow networks'

    def predictive_distribution(self, X, diagonal=True, S_MC_NNet=None):
        """Predictive mean / variance (Dy,MB) plus the q(f) marginals (Dy,MB,1).  diagonal=False (GaussianLinearMean only):
        the predictive covariance Sigma + noise I (Dy,MB,MB) plus q(f)'s mean (Dy,MB,1) and full covariance (Dy,MB,MB)."""
        X = self._rows3(X)
        assert not self.is_training, 'This method only works in eval mode'
        lik = self.likelihood
        if not diagonal and not isinstance(lik, GaussianLinearMean):
            raise NotImplementedError('correlated predictive moments are implemented for the Gaussian likelihood with identity '
                                      'link (GaussianLinearMean); under the other likelihoods the joint predictive is not Gaussian')
        self._eval_mode()
        if self.fully_bayesian:
            assert S_MC_NNet is not None, 'S_MC_NNet is required when the model is fully bayesian'
        n_mc = S_MC_NNet if self.fully_bayesian else 1
        with torch.no_grad():
            mean_q_f, cov_q_f = self.marginal_variational_qf_parameters(X, diagonal=diagonal, is_duvenaud=False)
            if not diagonal:
                m1, m2 = lik.marginal_moments(mean_q_f.squeeze(2), cov_q_f, diagonal=False)
            elif isinstance(lik, GaussianLinearMean):
                m1, m2 = lik.marginal_moments(mean_q_f.squeeze(2), cov_q_f.squeeze(2), diagonal=True)
            elif isinstance(lik, GaussianNonLinearMean):
                m1, m2 = [], []
                for dy in range(self.out_dim):
                    Xr = X[dy].repeat(n_mc, 1) if n_mc > 1 else X[dy]
                    _, a, b = _rows.test_rows('gauss_nonlinear', self.quad_points, None, mean_q_f[dy, :, 0],
                                              cov_q_f[dy, :, 0], self._noise(dy), self.G_matrix[dy], Xr, n_mc=n_mc)
                    m1.append(a)
                    m2.append(b)
                m1, m2 = torch.stack(m1), torch.stack(m2)
            elif isinstance(lik, Bernoulli):
                if n_mc > 1:
                    P = torch.stack([lik.marginal_moments(mean_q_f.squeeze(2), cov_q_f.squeeze(2), self.G_matrix, X)
                                     for _ in range(n_mc)]).mean(0)
                else:
                    P = lik.marginal_moments(mean_q_f.squeeze(2), cov_q_f.squeeze(2), self.G_matrix, X)
                m1, m2 = P, None
            elif isinstance(lik, MulticlassCategorical):
                mq, vq = mean_q_f.squeeze(2), cov_q_f.squeeze(2)
                if n_mc > 1:
                    # the n_mc dropout replicas as repeated rows of one kernel call (each replica draws its own masks and
                    # noise), then the class probabilities averaged over the replicas
                    MB = mq.shape[1]
                    P = lik.marginal_moments(mq.repeat(1, n_mc), vq.repeat(1, n_mc), self.G_matrix, X.repeat(1, n_mc, 1))
                    m1 = P.view(n_mc, MB, -1).mean(0)
                else:
                    m1 = lik.marginal_moments(mq, vq, self.G_matrix, X)
                m2 = None
            else:
                raise ValueError('Unsupported likelihood [{}]'.format(type(lik)))
        self.train()
        return m1, m2, mean_q_f, cov_q_f

    def test_log_likelihood(self, X, Y, return_moments, Y_std, S_MC_NNet=None):
        """log p(Y*|X*) per output (Dy,), and optionally the predictive moments."""
        MB = X.size(0)
        X_run = self._rows3(X)
        assert not self.is_training, 'This method only works in eval mode'
        self._eval_mode()
        if self.fully_bayesian:
            assert S_MC_NNet is not None, 'S_MC_NNet is required when the model is fully bayesian'
        lik = self.likelihood
        predictive_params = None
        with torch.no_grad():
            if isinstance(lik, (GaussianNonLinearMean, GaussianLinearMean)):
                kind = _LIK_KIND[type(lik)]
                n_mc = S_MC_NNet if (self.fully_bayesian and kind == 'gauss_nonlinear') else 1
                mean_q_f, cov_q_f = self.marginal_variational_qf_parameters(X_run, diagonal=True, is_duvenaud=False)
                self._eval_mode()
                logp, m1, m2 = [], [], []
                Y_std = Y_std.reshape(-1).to(torch.float64)
                for dy in range(self.out_dim):
                    Xr = X_run[dy].repeat(n_mc, 1) if n_mc > 1 else X_run[dy]
                    rows, a, b = _rows.test_rows(kind, self.quad_points, Y[:, dy].to(torch.float64), mean_q_f[dy, :, 0],
                                                 cov_q_f[dy, :, 0], self._noise(dy),
                                                 None if kind == 'gauss_linear' else self.G_matrix[dy], Xr,
                                                 y_std=float(Y_std[dy]), n_mc=n_mc)
                    lp = rows.sum()
                    if kind == 'gauss_nonlinear' and n_mc == 1:
                        # the reference evaluates 0.5*MB*log(pi) entirely in float32 (sparse_MF_SP.py:776)
                        lp = lp - (0.5 * MB * torch.log(cg.pi)).to(rows.device)
                    logp.append(lp)
                    m1.append(a)
                    m2.append(b)
                log_p_y = torch.stack(logp)
                if return_moments:
                    predictive_params = [torch.stack(m1), torch.stack(m2)]
            elif isinstance(lik, (Bernoulli, MulticlassCategorical)):
                m_Y, _, _, _ = self.predictive_distribution(X_run, diagonal=True, S_MC_NNet=S_MC_NNet)
                assert torch.isfinite(m_Y).all(), 'Got saturated probabilities'
                if isinstance(lik, Bernoulli):      # as if it came from the categorical likelihood: (MB, 2)
                    m_Y = m_Y.squeeze()
                    m_Y = torch.stack((1.0 - m_Y, m_Y), dim=1)
                # the reference scores classification in float32 (sparse_MF_SP.py:813)
                nll = -torch.log(m_Y.float().gather(1, Y.view(-1, 1).long())).mean()
                log_p_y = -1 * ((nll * MB).sum())
                if return_moments:
                    predictive_params = [m_Y]
            else:
                raise ValueError('Unsupported likelihood [{}]'.format(type(lik)))
        self.train()
        return log_p_y, predictive_params

    def evaluation_bundle(self, X, Y, Y_std, S=100, S_MC_NNet=None, seed=None, want_samples=False):
        """Everything `Trainer_GP_regression.performance_metrics` (reference trainers_regression.py:317-338, 181-224) derives from a
        test batch, from ONE q(f) evaluation: test log-likelihood and predictive moments (`test_log_likelihood`), plus the
        posterior-predictive 95 % interval coverage for which the reference re-runs q(f) on a 100x-repeated X
        (`sample_from_predictive_distribution`, sparse_MF_SP.py:939-992) and calls numpy.quantile on the host.

        Returns a dict: log_p_y (Dy,), m1 / m2 (Dy, MB), sq_err (Dy,) = sum_n (m1 - y)^2, coverage (Dy,) = number of rows whose y
        lies in the [2.5 %, 97.5 %] interval of S predictive samples, q_lo / q_hi (Dy, MB) and optionally samples (Dy, MB, S).
        Gaussian likelihoods; input-dependent flows draw one dropout mask per sample when the model is fully Bayesian."""
        assert not self.is_training, 'This method only works in eval mode'
        lik = self.likelihood
        if isinstance(lik, Bernoulli):
            raise NotImplementedError('interval coverage is defined for the Gaussian likelihoods (regression)')
        kind = _LIK_KIND[type(lik)]
        log_p_y, (m1, m2) = self.test_log_likelihood(X, Y, return_moments=True, Y_std=Y_std, S_MC_NNet=S_MC_NNet)
        X_run = self._rows3(X)
        self._eval_mode()
        out = dict(log_p_y=log_p_y, m1=m1, m2=m2, sq_err=((m1.reshape(self.out_dim, -1) - Y.t()) ** 2).sum(1))
        cov, qlo, qhi, smp = [], [], [], []
        with torch.no_grad():
            mean_q_f, cov_q_f = self.marginal_variational_qf_parameters(X_run, diagonal=True, is_duvenaud=False)   # cached factorisation
            n_mc = S if (self.fully_bayesian and kind == 'gauss_nonlinear') else 1
            for dy in range(self.out_dim):
                Xr = X_run[dy].repeat(n_mc, 1) if n_mc > 1 else X_run[dy]
                a, b, c, s = _rows.coverage_rows(kind, self.quad_points, Y[:, dy].to(torch.float64), mean_q_f[dy, :, 0], cov_q_f[dy, :, 0],
                                                 self._noise(dy), None if kind == 'gauss_linear' else self.G_matrix[dy], Xr, S, n_mc=n_mc,
                                                 seed=cg.config_seed if seed is None else seed, want_samples=want_samples)
                qlo.append(a); qhi.append(b); cov.append(c.sum()); smp.append(s)     # noqa: E702
        self.train()
        out.update(coverage=torch.stack(cov), q_lo=torch.stack(qlo), q_hi=torch.stack(qhi))
        if want_samples:
            out['samples'] = torch.stack(smp)
        return out

    # ---- sampling (caller-side utilities; element-wise torch ops on the kernel outputs) --------------------------
    def sample_from_variational_marginal_base(self, X, diagonal, is_duvenaud, init_Z=None):
        """One sample of q(f) per row (Dy,MB), with the mean (Dy,MB,1) and covariance it was drawn from; diagonal=False draws
        one JOINT sample over the rows of each output from the full covariance (Dy,MB,MB) (no backward: torch.no_grad())."""
        X = self._rows3(X)
        if not diagonal:
            joint = self._joint_qf(X, is_duvenaud)
            f = self._joint_samples(joint, 1)[:, 0, :].to(self.Z.dtype)
            mean = torch.stack([mu for _, mu, _ in joint]).unsqueeze(2).to(self.Z.dtype)
            return f, mean, torch.stack([cov for _, _, cov in joint]).to(self.Z.dtype)
        mean_q_f, cov_q_f = self.marginal_variational_qf_parameters(X, diagonal=True, is_duvenaud=is_duvenaud, init_Z=init_Z)
        e = torch.randn(mean_q_f.shape, dtype=mean_q_f.dtype, device=mean_q_f.device)
        f = (e * cov_q_f.sqrt() + mean_q_f).squeeze(dim=2)
        return f, mean_q_f, cov_q_f

    def sample_from_variational_marginal(self, X, S, diagonal, is_duvenaud, init_Z=None):
        """S warped samples per row.  The reference repeats X S times through the whole q(f) computation
        (sparse_MF_SP.py:911-922), i.e. S x the cost of the marginals; mu and v do not depend on the sample, so they are
        computed ONCE here and repeated (same distribution of samples, 1/S of the work; SURVEY.md §8f rank 1).

        diagonal=False: S joint samples over the rows of each output, f0 = mu + e L^T with L = psd_safe_cholesky(Sigma) and
        e ~ N(0, I) (Dy, S, MB) in FP64.  f0 (Dy, S*MB) keeps the sample-major layout of the diagonal case, and f = G(f0, X)
        goes through the flow modules the same way.  The mean is repeated as (Dy, S*MB, 1); the covariance is returned once,
        (Dy, MB, MB), not repeated.  No backward: call it under torch.no_grad()."""
        X = self._rows3(X)
        if self.is_training:
            self.train()
        else:
            self._eval_mode()
        if not diagonal:
            joint = self._joint_qf(X, is_duvenaud)
            f0 = self._joint_samples(joint, S).reshape(self.out_dim, -1).to(self.Z.dtype)
            mean_q_f0 = torch.stack([mu for _, mu, _ in joint]).unsqueeze(2).repeat(1, S, 1).to(self.Z.dtype)
            cov_q_f = torch.stack([cov for _, _, cov in joint]).to(self.Z.dtype)
            Xr = X.repeat(1, S, 1)
            f = torch.stack([g(f0[idx, :], Xr[idx]) for idx, g in enumerate(self.G_matrix)])
            self.train()
            return f, mean_q_f0, cov_q_f, f0
        mean1, cov1 = self.marginal_variational_qf_parameters(X, diagonal=True, is_duvenaud=is_duvenaud, init_Z=init_Z)
        mean_q_f0, cov_q_f0 = mean1.repeat(1, S, 1), cov1.repeat(1, S, 1)
        e = torch.randn(mean_q_f0.shape, dtype=mean_q_f0.dtype, device=mean_q_f0.device)
        f0 = (e * cov_q_f0.sqrt() + mean_q_f0).squeeze(dim=2)
        Xr = X.repeat(1, S, 1)                      # input-dependent flows see every repeated row (fresh dropout mask each)
        f = torch.stack([g(f0[idx, :], Xr[idx]) for idx, g in enumerate(self.G_matrix)])
        self.train()
        return f, mean_q_f0, cov_q_f0, f0

    def sample_from_predictive_distribution(self, X, S):
        assert not self.is_training, 'This method only works in eval mode'
        assert len(X.shape) == 2, 'Invalid input X.shape'
        self._eval_mode()
        N = X.shape[0]
        samples_arr = []
        with torch.no_grad():
            f_k, _, _, f_0 = self.sample_from_variational_marginal(X, S, diagonal=True, is_duvenaud=False, init_Z=None)
            self._eval_mode()
            for output_idx in range(self.out_dim):
                samples_arr.append(self.likelihood.sample_from_output(f_k, output_idx).view(S, N, 1))
            self.train()
            return torch.stack(samples_arr, dim=0), f_k, f_0
