"""CPU reference for the non-whitened q(u) (the reference's is_whiten=False branch, sparse_MF_SP.py:357-360, 386-391, 433-453),
restated in torch FP64 without the whitened formulas.  Test infrastructure, not product.

q(u) = N(m, P P^T) with P = tril(L_raw), p(u) = N(0, K_zz):
  mu = K_xz K^-1 m                                   (cholesky_solve)
  v  = k_xx - diag(K_xz K^-1 K_zx) + diag(K_xz K^-1 S K^-1 K_zx),   S = P P^T
  KL = torch.distributions.kl_divergence(N(m, scale_tril=P), N(0, scale_tril=L)),   L = psd_safe_cholesky(K_zz)
The prior uses the same (possibly jittered) L as the marginals.  Everything else is O2's own code (oracle/tgp_oracle.py): the
Cholesky with its jitter ladder, `ell_rows`, the flows, the Monte-Carlo softmax; the kernel is tests/matern_ref.kernel_ard, so
p['kernel'] selects any of the four covariance functions.
"""
import torch
import torch.distributions as td
import torch.nn.functional as F

from oracle import tgp_oracle as O
from tests.matern_ref import kernel_ard


def _factor(p):
    L_zz, _, _ = O.psd_safe_cholesky(kernel_ard(p['Z'], p['Z'], p))
    return L_zz


def _tril(p):
    return p['L_raw'] * torch.ones_like(p['L_raw']).tril(0)


def qf_marginals(X, p):
    m = p['m']
    K_xx = F.softplus(p['raw_outputscale']).expand(X.shape[0])
    K_zx = kernel_ard(X, p['Z'], p).t()
    L_zz = _factor(p)
    P = _tril(p)
    S = P @ P.t()
    Ki_kzx = torch.cholesky_solve(K_zx, L_zz, upper=False)          # K^-1 K_zx   (M, R)
    mu = Ki_kzx.t() @ m
    v = K_xx - torch.sum(K_zx * Ki_kzx, 0) + torch.sum(Ki_kzx * (S @ Ki_kzx), 0)
    return mu, v


def kl(p):
    """KL(N(m, P P^T) || N(0, L L^T)).  torch's scale_tril wants a positive diagonal; N(m, P P^T) depends on P P^T only, so
    each column of P takes the sign of its diagonal entry."""
    P = _tril(p)
    P = P * torch.sign(torch.diagonal(P)).view(1, -1)
    L_zz = _factor(p)
    q = td.MultivariateNormal(p['m'], scale_tril=P)
    prior = td.MultivariateNormal(torch.zeros_like(p['m']), scale_tril=L_zz)
    return td.kl_divergence(q, prior)


def elbo(X, y, p, N, likelihood='gauss_nonlinear', n_quad=100):
    """(ELBO, ELL, KLD, rows) as O.elbo."""
    mu, v = qf_marginals(X, p)
    rows = O.ell_rows(mu, v, y, p, likelihood, n_quad)
    ELL = (float(N) / X.shape[0]) * rows.sum()
    KLD = kl(p)
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
    KLD = torch.stack([kl(p) for p in plist]).sum()
    return ELL - KLD, ELL, KLD, rows, mu, v


def from_whitened(p):
    """The non-whitened parameters of the same q(f) as the whitened p: (m, L_raw) = (L m_w, L tril(L_raw_w)), L of p's K_zz."""
    L_zz = _factor({k: (v.detach() if torch.is_tensor(v) else v) for k, v in p.items()})
    q = dict(p)
    q['m'] = (L_zz @ p['m'].detach()).detach()
    q['L_raw'] = (L_zz @ _tril(p).detach()).detach()
    return q, L_zz
