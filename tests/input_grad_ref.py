"""CPU reference of the input gradient dELBO/dX: torch.autograd through O2 (oracle/tgp_oracle.py) for the RBF and through
tests/matern_ref.py for the Matern kernels.  Test infrastructure, not product.

The per-row parameters of an input-dependent flow enter as given tensors here: this is the gradient through q(f) alone,
which is what the fused kernels compute (the flow MLP's own share comes from its backward)."""
import torch

from tests import matern_ref as MR


def _leaf(t):
    return t.detach().clone().requires_grad_(True)


def elbo_grads_xz(X, y, p, N, likelihood, n_quad):
    """(ELBO, dELBO/dX, dELBO/dZ) with the kernel p.get('kernel', 'rbf')."""
    X = _leaf(X)
    q = dict(p)
    q['Z'] = _leaf(p['Z'])
    E = MR.elbo(X, y, q, N, likelihood, n_quad)[0]
    gx, gz = torch.autograd.grad(E, [X, q['Z']])
    return E.detach(), gx, gz


def marginals_grad_x(X, p, w_mu, w_v):
    """d(sum_n w_mu[n] mu_n + w_v[n] v_n)/dX."""
    X = _leaf(X)
    mu, v = MR.qf_marginals(X, p)
    return torch.autograd.grad((w_mu * mu).sum() + (w_v * v).sum(), X)[0]


def elbo_value(X, y, p, N, likelihood, n_quad):
    with torch.no_grad():
        return MR.elbo(X, y, p, N, likelihood, n_quad)[0]
