"""Torch restatement of the warped GP (DESIGN.md §2: z = G(y) = f + eps), independent of the kernels.

G is oracle.tgp_oracle.apply_flow applied to y; G'(y) comes from torch.autograd.grad(create_graph=True), so the parameter gradients
of log G'(y) are autograd's double backward.  The GP part is O2's (tests/matern_ref for the kernel, tests/unwhitened_ref for
p['whiten'] = False).  Predictive moments: Gauss-Hermite over z ~ N(mu, v + s2) with scipy's brentq for G^-1.
"""
import math

import numpy as np
import torch
from scipy.optimize import brentq

from oracle import tgp_oracle as O
from tests import matern_ref as MR
from tests import unwhitened_ref as UR


def warp(layers, y):
    """(G(y), G'(y)), both differentiable w.r.t. the flow parameters (and G' w.r.t. y)."""
    with torch.enable_grad():                                    # G' needs a graph even when the caller evaluates without one
        y = y.detach().clone().requires_grad_(True)
        G = O.apply_flow(layers, y)
        dG, = torch.autograd.grad(G.sum(), y, create_graph=True)
    return G, dG


def ell_rows(mu, v, y, p):
    """log N(G(y) | mu, s2) - v / (2 s2) + log|G'(y)| per row (the GaussianLinearMean row at G(y), plus the log-Jacobian)."""
    G, dG = warp(p['flow'], y)
    return O.ell_rows_gauss_linear(mu, v, G, p) + torch.log(torch.abs(dG))


def _gp(p):
    if p.get('whiten', True):
        return MR.qf_marginals, O.kl_whitened
    return UR.qf_marginals, UR.kl


def elbo(X, y, p, N):
    qf, kl = _gp(p)
    mu, v = qf(X, p)
    rows = ell_rows(mu, v, y, p)
    ELL = (float(N) / X.shape[0]) * rows.sum()
    KLD = kl(p)
    return ELL - KLD, ELL, KLD, rows


def elbo_and_grads(X, y, p, N, want_dx=False):
    """(ELBO, ELL, KLD, rows, {leaf name: gradient}) with the leaves of O.leaf_params; want_dx adds 'X'."""
    leaves = O.leaf_params(p)
    for t in leaves.values():
        t.requires_grad_(True)
    if want_dx:
        X = X.detach().clone().requires_grad_(True)
        leaves = dict(leaves, X=X)
    E, ELL, KLD, rows = elbo(X, y, p, N)
    grads = torch.autograd.grad(E, list(leaves.values()), allow_unused=True)
    g = {k: (torch.zeros_like(t) if gi is None else gi) for (k, t), gi in zip(leaves.items(), grads)}
    for t in O.leaf_params(p).values():
        t.requires_grad_(False)
    return E.detach(), ELL.detach(), KLD.detach(), rows.detach(), g


def logp_rows(mu, v, y, p, y_std=1.0):
    """log N(G(y) | mu, v + s2) + log|G'(y)| - log y_std per row (log 2 pi with the float32-rounded pi of the reference)."""
    G, dG = (t.detach() for t in warp(p['flow'], y))
    ky = torch.exp(p['log_var_noise']) + v
    logn = -0.5 * (O.log_2pi_const(torch.float64) + torch.log(ky) + (G - mu) ** 2 / ky)
    return logn + torch.log(torch.abs(dG)) - math.log(y_std)


def inverse(layers, z):
    """G^-1 elementwise by brentq on a bracket grown from z (G increasing or decreasing)."""
    def G(h):
        with torch.no_grad():
            return float(O.apply_flow(layers, torch.tensor([h], dtype=torch.float64))[0])
    out = []
    for zi in np.asarray(z, dtype=np.float64).reshape(-1):
        f = lambda h: G(h) - zi  # noqa: E731
        lo, hi, step = zi, zi, max(1.0, abs(zi))
        while np.sign(f(lo)) == np.sign(f(hi)) and f(lo) != 0.0:
            lo, hi, step = zi - step, zi + step, 2 * step
            if step > 1e12:
                raise ValueError('no bracket for %g' % zi)
        out.append(lo if f(lo) == 0.0 else brentq(f, lo, hi, xtol=1e-15, rtol=4 * np.finfo(float).eps, maxiter=500))
    return torch.tensor(out, dtype=torch.float64).reshape(np.shape(z))


def moments(mu, v, p, n_quad):
    """(E[G^-1(z)], E[G^-1(z)^2] - E[G^-1(z)]^2) for z ~ N(mu, v + s2), Gauss-Hermite with n_quad nodes."""
    t, w = O.gauss_hermite(n_quad, torch.float64)
    ky = torch.exp(p['log_var_noise']).detach() + v.detach()
    z = torch.sqrt(2.0 * ky).unsqueeze(0) * t.view(-1, 1) + mu.detach().unsqueeze(0)
    h = inverse(p['flow'], z.numpy())
    W = w.view(-1, 1) / math.sqrt(math.pi)
    m1 = (W * h).sum(0)
    return m1, (W * h * h).sum(0) - m1 ** 2
