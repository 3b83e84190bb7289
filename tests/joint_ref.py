"""CPU reference for the full covariance of q(f) over a batch and joint samples from it.  Test infrastructure, not product.

`qf_joint` is the reference's q(f) algebra (sparse_MF_SP.py:376-382, as O2's `qf_marginals` restates it) without taking
the diagonal: K_xx is the kernel matrix of the rows, and the two quadratic forms become matrix products.  The kernel is
`tests/matern_ref.kernel_ard`, so p['kernel'] selects any of the four covariance functions ('rbf' is O2's own).
"""
import torch
import torch.nn.functional as F

from oracle import tgp_oracle as O
from tests.matern_ref import kernel_ard


def qf_joint(X, p):
    """mu (R,), Sigma (R, R) of q(f) at the rows of X; Sigma is symmetrised (the two products are not exactly symmetric)."""
    Z, m = p['Z'], p['m']
    K_xx = kernel_ard(X, X, p)
    K_zz = kernel_ard(Z, Z, p)
    K_xz = kernel_ard(X, Z, p)
    K_zx = K_xz.t()
    L_zz, _, _ = O.psd_safe_cholesky(K_zz)
    L_S = p['L_raw'] * torch.ones_like(p['L_raw']).tril(0)
    S = L_S @ L_S.t()
    sol_m = torch.linalg.solve_triangular(L_zz.t(), m.view(-1, 1), upper=True)
    mu = (K_xz @ sol_m).view(-1)
    sol = torch.cholesky_solve(K_zx, L_zz, upper=False)
    rhs = torch.linalg.solve_triangular(L_zz, K_zx, upper=False)
    Sigma = K_xx - K_zx.t() @ sol + rhs.t() @ (S @ rhs)
    return mu, 0.5 * (Sigma + Sigma.t())


def outputscale(p):
    return float(F.softplus(torch.as_tensor(p['raw_outputscale'], dtype=torch.float64)))


def joint_samples(mu, Sigma, jitter, eps):
    """mu + eps L^T for eps (S, R), L = chol(Sigma + jitter I) by torch.linalg.cholesky."""
    L = torch.linalg.cholesky(Sigma + jitter * torch.eye(Sigma.shape[0], dtype=Sigma.dtype))
    return mu.view(1, -1) + eps @ L.t()
