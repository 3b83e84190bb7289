"""ARD-RBF, ARD-Matern and scale kernels carrying the parameter names the reference's gpytorch objects expose
(`raw_lengthscale` (Dy,1,D), `raw_outputscale` (Dy,), `base_kernel`, `batch_shape`, and `nu` for the Matern kernel).

On the hot path only the *parameters* of these modules are read (the fused kernels regenerate K tiles from X, Z and
the raw parameters).  `__call__` exists for API parity (`kernel(x1, x2, diag=...)` with `.evaluate()` on non-diag
results) and evaluates the same closed form with a handful of torch ops; it is not used by ELBO / test-NLL.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F


class _Evaluated:
    def __init__(self, t):
        self._t = t

    def evaluate(self):
        return self._t

    def diag(self):
        return torch.diagonal(self._t, dim1=-2, dim2=-1)


class Kernel(nn.Module):
    def __init__(self, batch_shape=torch.Size([])):
        super().__init__()
        self._batch_shape = torch.Size(batch_shape)

    @property
    def batch_shape(self):
        return self._batch_shape

    def __call__(self, x1, x2=None, diag=False, **params):
        out = self.forward(x1, x1 if x2 is None else x2, diag=diag)
        return out if diag else _Evaluated(out)


class RBFKernel(Kernel):
    def __init__(self, ard_num_dims=None, batch_shape=torch.Size([])):
        super().__init__(batch_shape)
        self.ard_num_dims = ard_num_dims
        self.raw_lengthscale = nn.Parameter(torch.zeros(*batch_shape, 1, 1 if ard_num_dims is None else ard_num_dims))

    @property
    def lengthscale(self):
        return F.softplus(self.raw_lengthscale)

    def forward(self, x1, x2, diag=False):
        a, b = x1 / self.lengthscale, x2 / self.lengthscale
        if diag:
            return torch.exp(-0.5 * (a - b).pow(2).sum(-1))
        d2 = (a.unsqueeze(-2) - b.unsqueeze(-3)).pow(2).sum(-1)
        return torch.exp(-0.5 * d2)


class MaternKernel(Kernel):
    """gpytorch's MaternKernel for nu in {0.5, 1.5, 2.5}.  r = ||(x1 - x2) / lengthscale|| by direct differences (gpytorch
    uses an expanded quadratic form, whose rounding leaves r ~ 1e-8 ||x|| where x1 == x2)."""
    NUS = (0.5, 1.5, 2.5)

    def __init__(self, nu=2.5, ard_num_dims=None, batch_shape=torch.Size([])):
        super().__init__(batch_shape)
        if nu not in self.NUS:
            raise ValueError('nu must be one of 0.5, 1.5, 2.5, got {}'.format(nu))
        self.nu = float(nu)
        self.ard_num_dims = ard_num_dims
        self.raw_lengthscale = nn.Parameter(torch.zeros(*batch_shape, 1, 1 if ard_num_dims is None else ard_num_dims))

    @property
    def lengthscale(self):
        return F.softplus(self.raw_lengthscale)

    def forward(self, x1, x2, diag=False):
        a, b = x1 / self.lengthscale, x2 / self.lengthscale
        d2 = (a - b).pow(2).sum(-1) if diag else (a.unsqueeze(-2) - b.unsqueeze(-3)).pow(2).sum(-1)
        return matern_phi(d2, self.nu)


def matern_phi(d2, nu):
    """phi_nu(r) with r = sqrt(d2); pairs with d2 <= 1e-30 take r = 0 (and no gradient)."""
    r = torch.where(d2 > 1e-30, d2.clamp_min(1e-30).sqrt(), torch.zeros_like(d2))
    if nu == 0.5:
        return torch.exp(-r)
    if nu == 1.5:
        a = r * 3.0 ** 0.5
        return (1.0 + a) * torch.exp(-a)
    a = r * 5.0 ** 0.5
    return (1.0 + a + a * a / 3.0) * torch.exp(-a)


class ScaleKernel(Kernel):
    def __init__(self, base_kernel, batch_shape=torch.Size([])):
        super().__init__(batch_shape)
        self.base_kernel = base_kernel
        self.raw_outputscale = nn.Parameter(torch.zeros(*batch_shape))

    @property
    def outputscale(self):
        return F.softplus(self.raw_outputscale)

    def forward(self, x1, x2, diag=False):
        base = self.base_kernel.forward(x1, x2, diag=diag)
        s = self.outputscale
        return base * (s.unsqueeze(-1) if diag else s.view(*s.shape, 1, 1))


class ZeroMean(nn.Module):
    def forward(self, x):
        return torch.zeros(x.shape[:-1], dtype=x.dtype, device=x.device)


class CholeskyVariationalDistribution(nn.Module):
    """q(u) parameters under the names the reference reads (sparse_MF_SP.py:158-177)."""

    def __init__(self, num_inducing_points, batch_shape=torch.Size([])):
        super().__init__()
        self.variational_mean = nn.Parameter(torch.zeros(*batch_shape, num_inducing_points))
        self.chol_variational_covar = nn.Parameter(torch.eye(num_inducing_points).repeat(*batch_shape, 1, 1))
