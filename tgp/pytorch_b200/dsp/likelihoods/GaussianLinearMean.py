"""p(y | f) Gaussian, identity link: closed-form expected log-lik of SVGP
(reference code/dsp/likelihoods/GaussianLinearMean.py:20-118; `log_marginal` :121-155 is exact-GP, out of scope)."""
import torch
import torch.nn as nn
import torch.distributions as td

from .. import config as cg
from ..utils import positive_transform, inverse_positive_transform
from . import _rows


class GaussianLinearMean(nn.Module):
    def __init__(self, out_dim, noise_init, noise_is_shared):
        super().__init__()
        self.out_dim = out_dim
        self.noise_is_shared = noise_is_shared
        init = inverse_positive_transform(torch.tensor(noise_init, dtype=cg.dtype))
        self.log_var_noise = nn.Parameter(torch.ones(1 if noise_is_shared else out_dim, 1, dtype=cg.dtype) * init)

    def _noise(self):
        return self.log_var_noise.expand(self.out_dim, 1) if self.noise_is_shared else self.log_var_noise

    def sample_from_output(self, f, i, **kwargs):
        var = positive_transform(self._noise()[i])
        return td.Normal(f, torch.ones_like(f) * torch.sqrt(var)).sample()

    def expected_log_prob_rows(self, Y, gauss_mean, gauss_cov, flow=None, X=None):
        if cg.positive_transform != 'exp':
            raise NotImplementedError("the fused epilogue implements positive_transform='exp' (the reference default)")
        noise = self._noise()
        sums, rows = [], []
        for dy in range(self.out_dim):
            s, r = _rows.expected_log_prob_rows('gauss_linear', 0, Y[dy], gauss_mean[dy], gauss_cov[dy], noise[dy], None, None)
            sums.append(s)
            rows.append(r)
        return torch.stack(sums), torch.stack(rows)

    def expected_log_prob(self, Y, gauss_mean, gauss_cov, **kwargs):
        """log N(y|mu, s2) - 0.5 v / s2 summed over the minibatch: shape (Dy,)."""
        return self.expected_log_prob_rows(Y, gauss_mean, gauss_cov)[0]

    def marginal_moments(self, gauss_mean, gauss_cov, diagonal, **kwargs):
        """(mean, covariance) of p(y*): gauss_cov (Dy,MB) + noise, or with diagonal=False the full (Dy,MB,MB) + noise I."""
        if not diagonal:
            eye = torch.eye(gauss_cov.size(-1), dtype=gauss_cov.dtype, device=gauss_cov.device)
            return gauss_mean.clone(), gauss_cov + positive_transform(self._noise()).view(-1, 1, 1) * eye
        C_Y = positive_transform(self._noise()).expand(-1, gauss_mean.size(1)) + gauss_cov
        return gauss_mean.clone(), C_Y
