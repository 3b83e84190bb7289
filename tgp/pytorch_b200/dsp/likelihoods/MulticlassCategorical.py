"""Categorical likelihood with a softmax link, integrated by Monte Carlo
(reference code/dsp/likelihoods/MulticlassCategorical.py:19-151).

Same constructor and method signatures as the reference.  The S x C x MB noise of `td.Normal(mean, std).rsample([S])` is drawn
here with the framework's generator exactly as rsample draws it (`torch.empty(shape).normal_()`), so a seeded run consumes the
same stream as the reference on the same device; setting `mc_noise` to a (S, C, MB) tensor replaces the draw (parity tests).
Sampling, flows, log-softmax, the mean over samples and all gradients run in ONE kernel (tgp_mc_softmax_rows, or
tgp_mc_softmax_rows_rowp for input-dependent flows, whose MLPs are evaluated on X[c] once per call)."""
import torch
import torch.nn as nn
import torch.distributions as td
from torch.nn.functional import softmax

from .. import config as cg
from . import _rows


class MulticlassCategorical(nn.Module):
    def __init__(self, num_classes):
        super().__init__()
        self.C = num_classes
        self.SMC = cg.quad_points            # number of Monte-Carlo samples
        self.loss = nn.CrossEntropyLoss(reduction='none')
        self.link_function = softmax
        self.mc_noise = None                 # optional explicit N(0,1) noise (S, C, MB) for the next call(s)
        assert num_classes > 2, 'If you have a binary classification problem use the Bernouilli'

    def sample_from_output(self, f, i, **kwargs):
        assert f.size(0) == self.C, 'Bad specified input'
        probs = self.link_function(f.t(), dim=1)
        return td.Categorical(probs=probs).sample().to(cg.dtype)

    def _check(self, gauss_mean, flow, X):
        assert len(flow) == self.C, 'Flow list must be size {} for MultiClass likelihood'.format(self.C)
        assert gauss_mean.size(0) == self.C, 'Multiclass classification requires {} GPs, got {}'.format(self.C, gauss_mean.size(0))
        assert len(X.shape) == 3, 'Bad input X, expected (n_class,MB*S,Dx)'
        assert X.size(0) == self.C, 'Wrong first dimension in X, expected n_classes'

    def _noise(self, gauss_mean):
        if self.mc_noise is not None:
            return self.mc_noise.to(gauss_mean.device)
        # td.Normal.rsample / .sample: _standard_normal(shape) = torch.empty(shape, dtype, device).normal_()
        return torch.empty((self.SMC,) + tuple(gauss_mean.shape), dtype=gauss_mean.dtype, device=gauss_mean.device).normal_()

    def expected_log_prob_rows(self, Y, gauss_mean, gauss_cov, flow, X):
        self._check(gauss_mean, flow, X)
        y = Y.t().squeeze(dim=1).reshape(-1)
        s, rows, _ = _rows.mc_softmax(list(flow), X, y, self._noise(gauss_mean), gauss_mean, gauss_cov)
        return s, rows

    def expected_log_prob(self, Y, gauss_mean, gauss_cov, flow, X, **kwargs):
        """int q(f_0) log p(y | softmax G(f_0)) df_0 by Monte Carlo, summed over the minibatch (a scalar)."""
        return self.expected_log_prob_rows(Y, gauss_mean, gauss_cov, flow, X)[0].to(gauss_mean.dtype)

    def marginal_moments(self, gauss_mean, gauss_cov, flow, X, **kwargs):
        """Class probabilities (MB, C): softmax of the warped samples, averaged over the samples."""
        self._check(gauss_mean, flow, X)
        with torch.no_grad():
            y = torch.zeros(gauss_mean.shape[1], dtype=torch.float64, device=gauss_mean.device)
            _, _, P = _rows.mc_softmax(list(flow), X, y, self._noise(gauss_mean), gauss_mean, gauss_cov, want_probs=True)
        return P.to(gauss_mean.dtype)
