"""CPU reference for the ARD-Matern kernels (nu = 1/2, 3/2, 5/2): the O2 restatement (oracle/tgp_oracle.py) with its
ScaleKernel(RBFKernel) replaced by ScaleKernel(MaternKernel).  Test infrastructure, not product.

Everything but the kernel is O2's own code: `psd_safe_cholesky`, `ell_rows`, `kl_whitened`, the flows and the quadrature.
`p` is an O2 parameter dict with one more key, 'kernel' in {'rbf', 'matern12', 'matern32', 'matern52'}; with 'rbf' the
functions below compute what O2 computes.

The distance is taken by DIRECT differences (gpytorch 1.1.1 uses the expanded quadratic form, which leaves d2 ~ 1e-16
||x||^2 on its K_zz diagonal, so its own nu = 1/2 diagonal is off by ~sqrt(eps) relative).  r = sqrt(clamp_min(d2, 1e-30))
as gpytorch, except that pairs with d2 <= 1e-30 take r = 0: phi(0) = 1 exactly, and such a pair contributes nothing to the
gradients, which is what the clamp yields under autograd.
"""
import math

import torch
import torch.nn.functional as F

from oracle import tgp_oracle as O

MATERN_NU = {'matern12': 0.5, 'matern32': 1.5, 'matern52': 2.5}


def matern_ard(x1, x2, raw_lengthscale, raw_outputscale, nu):
    ls = F.softplus(raw_lengthscale).view(1, -1)
    a, b = x1 / ls, x2 / ls
    d2 = (a.unsqueeze(-2) - b.unsqueeze(-3)).pow(2).sum(-1)
    r = torch.where(d2 > 1e-30, d2.clamp_min(1e-30).sqrt(), torch.zeros_like(d2))
    if nu == 0.5:
        phi = torch.exp(-r)
    elif nu == 1.5:
        c = math.sqrt(3.0) * r
        phi = (1.0 + c) * torch.exp(-c)
    elif nu == 2.5:
        c = math.sqrt(5.0) * r
        phi = (1.0 + c + c * c / 3.0) * torch.exp(-c)
    else:
        raise ValueError('nu must be 0.5, 1.5 or 2.5')
    return phi * F.softplus(raw_outputscale)


def kernel_ard(x1, x2, p):
    """K(x1, x2) of the covariance function p['kernel'] (default 'rbf', O2's rbf_ard)."""
    kind = p.get('kernel', 'rbf')
    if kind == 'rbf':
        return O.rbf_ard(x1, x2, p['raw_lengthscale'], p['raw_outputscale'])
    return matern_ard(x1, x2, p['raw_lengthscale'], p['raw_outputscale'], MATERN_NU[kind])


def qf_marginals(X, p):
    """O.qf_marginals with K_zz and K_xz from `kernel_ard` (K_xx = s for every kind: phi(0) = 1)."""
    Z, m = p['Z'], p['m']
    s = F.softplus(p['raw_outputscale'])
    K_xx = s.expand(X.shape[0])
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
    v = K_xx - torch.sum(K_zx * sol, 0) + torch.sum(rhs * (S @ rhs), 0)
    return mu, v


def elbo(X, y, p, N, likelihood='gauss_nonlinear', n_quad=100):
    """(ELBO, ELL, KLD, rows) as O.elbo."""
    mu, v = qf_marginals(X, p)
    rows = O.ell_rows(mu, v, y, p, likelihood, n_quad)
    ELL = (float(N) / X.shape[0]) * rows.sum()
    KLD = O.kl_whitened(p)
    return ELL - KLD, ELL, KLD, rows


def elbo_and_grads(X, y, p, N, likelihood='gauss_nonlinear', n_quad=100):
    """As O.elbo_and_grads: (ELBO, ELL, KLD, rows, {leaf name: gradient})."""
    leaves = O.leaf_params(p)
    for t in leaves.values():
        t.requires_grad_(True)
        t.grad = None
    E, ELL, KLD, rows = elbo(X, y, p, N, likelihood, n_quad)
    grads = torch.autograd.grad(E, list(leaves.values()), allow_unused=True)
    g = {k: (torch.zeros_like(t) if gi is None else gi) for (k, t), gi in zip(leaves.items(), grads)}
    return E.detach(), ELL.detach(), KLD.detach(), rows.detach(), g


def elbo_multiclass(X, y, plist, N, eps):
    """As O.elbo_multiclass: (ELBO, ELL, KLD, rows, mu (C, MB), v (C, MB))."""
    mv = [qf_marginals(X, p) for p in plist]
    mu, v = torch.stack([a for a, _ in mv]), torch.stack([b for _, b in mv])
    rows = O.ell_rows_mc_softmax(mu, v, y, [p['flow'] for p in plist], eps)
    ELL = (float(N) / X.shape[0]) * rows.sum()
    KLD = torch.stack([O.kl_whitened(p) for p in plist]).sum()
    return ELL - KLD, ELL, KLD, rows, mu, v


def log_likelihood_gauss_nonlinear(X, y, p, y_std, n_quad=100):
    """O.test_log_likelihood, Gaussian non-linear likelihood with global flow parameters: (log p(y), (m1, m2))."""
    with torch.no_grad():
        MB = X.shape[0]
        mu, v = qf_marginals(X, p)
        t, w = O.gauss_hermite(n_quad, mu.dtype)
        var = torch.exp(p['log_var_noise'])
        f = torch.sqrt(2.0 * v).unsqueeze(0) * t.view(-1, 1) + mu.unsqueeze(0)
        g = O.apply_flow(p['flow'], f)
        C = (y_std * torch.sqrt(var)) ** 2
        lp = O._log_gaussian_1d(y_std * y.unsqueeze(0), y_std * g, C)
        log_p = torch.logsumexp(torch.log(w).view(-1, 1) + lp, 0).sum(-1) - 0.5 * MB * torch.log(O.PI_F32)
        return log_p, O.moments_gauss_nonlinear(mu, v, p, n_quad)
