"""Warped GP: p(y | f) = N(G(y) | f, s2) |G'(y)| with a flow G on the OBSERVATIONS (the identity on f) — the baseline the
transformed GP is defined against (reference code/dsp/likelihoods/WarpedGaussianLinearMean.py:25-168).

The definitions are this project's (DESIGN.md §2): training rows log N(G(y) | mu, s2) - v / (2 s2) + log|G'(y)| in closed form,
test rows log N(G(y*) | mu, v + s2) + log|G'(y*)| - log y_std, predictive moments E[G^-1(z)] and Var[G^-1(z)] for
z ~ N(mu, v + s2) by Gauss-Hermite with a Newton inverse per node, samples G^-1(f + s eps).  All of them run in the fused row
kernels (tgp_ell_forward / tgp_test_rows / tgp_flow_inverse with TGP_LIK_GAUSS_WARPED)."""
import torch
import torch.nn as nn

from .. import config as cg
from ..models.flow import instance_flow
from ..utils import positive_transform, inverse_positive_transform
from . import _rows


class WarpedGaussianLinearMean(nn.Module):
    def __init__(self, out_dim, noise_init, noise_is_shared, flow_specs):
        super().__init__()
        assert len(flow_specs) == out_dim, 'WarpedGaussianLinearMean takes one warp specification per output'
        self.out_dim = out_dim
        self.noise_is_shared = noise_is_shared
        init = inverse_positive_transform(torch.tensor(noise_init, dtype=cg.dtype))
        self.log_var_noise = nn.Parameter(torch.ones(1 if noise_is_shared else out_dim, 1, dtype=cg.dtype) * init)
        # one warp per output: a spec list (StepTanhL, SAL, build_chain, ...) or a flow instance, as sparse_MF_SP.initialize_flows
        self.flow = nn.ModuleList([instance_flow(fl) if type(fl) == list else fl for fl in flow_specs])
        self.quad_points = cg.quad_points

    def _noise(self):
        return self.log_var_noise.expand(self.out_dim, 1) if self.noise_is_shared else self.log_var_noise

    def _check_scope(self):
        if cg.positive_transform != 'exp':
            raise NotImplementedError("the fused epilogue implements positive_transform='exp' (the reference default)")

    def expected_log_prob_rows(self, Y, gauss_mean, gauss_cov, flow=None, X=None):
        """(ELL (Dy,), per-row terms (Dy, MB)) of E_q(f)[log N(G(y) | f, s2)] + log|G'(y)|; `flow` / `X` (the flow on f) are
        not used: the warp is self.flow."""
        self._check_scope()
        noise = self._noise()
        sums, rows = [], []
        for dy in range(self.out_dim):
            s, r = _rows.expected_log_prob_rows('gauss_warped', self.quad_points, Y[dy], gauss_mean[dy], gauss_cov[dy],
                                                noise[dy], self.flow[dy], None)
            sums.append(s)
            rows.append(r)
        return torch.stack(sums), torch.stack(rows)

    def expected_log_prob(self, Y, gauss_mean, gauss_cov, **kwargs):
        """Summed over the minibatch: shape (Dy,)."""
        return self.expected_log_prob_rows(Y, gauss_mean, gauss_cov)[0]

    def marginal_moments(self, gauss_mean, gauss_cov, diagonal=True, **kwargs):
        """(E[G^-1(z)], Var[G^-1(z)]) with z ~ N(mean, cov + s2), shapes (Dy, MB); NaN in the rows whose inverse warp fails."""
        if not diagonal:
            raise NotImplementedError('the joint predictive of the warped likelihood is not Gaussian: diagonal=True only')
        noise = self._noise()
        m1, m2 = [], []
        for dy in range(self.out_dim):
            _, a, b = _rows.test_rows('gauss_warped', self.quad_points, None, gauss_mean[dy], gauss_cov[dy], noise[dy],
                                      self.flow[dy], None)
            m1.append(a)
            m2.append(b)
        return torch.stack(m1), torch.stack(m2)

    def sample_from_output(self, f, i, **kwargs):
        """G_i^-1(f + s eps), eps ~ N(0, 1): samples in the units of y.  `f` holds output i's latent samples, or all outputs
        stacked along the first dimension (how sparse_MF_SP.sample_from_predictive_distribution passes it).  Raises
        ValueError when the inverse warp fails for some samples."""
        if f.dim() >= 2 and f.shape[0] == self.out_dim:
            f = f[i]
        var = positive_transform(self._noise()[i])
        z = f + torch.randn_like(f) * torch.sqrt(var).to(f.dtype)
        h, n_fail = _rows.flow_inverse(self.flow[i], z)
        if n_fail:
            raise ValueError('the inverse warp of output %d failed for %d of %d samples (is G monotone?)' % (i, n_fail, z.numel()))
        return h.to(f.dtype)
