"""The CPU reference of the non-whitened q(u) (tests/unwhitened_ref.py) against the fixtures of the unmodified reference (O1):
on every regression and Bernoulli fixture, the non-whitened model built from the fixture's whitened one by
(m, P) = (L m_w, L P_w) gives the fixture's ELBO, ELL, KLD and q(f) marginals, and its m / P gradients map back to the
fixture's whitened ones by the chain rule (L held fixed): d/dm_w = L^T d/dm, d/dP_w = tril(L^T d/dP)."""
import pytest
import torch

from oracle import tgp_oracle as O
from tests import unwhitened_ref as UR
from tests.golden_util import Golden, golden_names, rel_err

TOL = 1e-11


@pytest.mark.parametrize('name', golden_names())
def test_identity_with_the_whitened_fixture(name):
    g = Golden(name)
    p = g.oracle_params('train')
    X, Y = g.t('X'), g.t('Y').view(-1)
    lik, nq = g.meta['likelihood'], g.meta['n_quad']
    q, L = UR.from_whitened(p)
    mu, v = UR.qf_marginals(X, q)
    errs = {'mu': rel_err(mu, g.t('mu')), 'v': rel_err(v, g.t('v'))}
    E, ELL, KLD, _, grads = UR.elbo_and_grads(X, Y, q, g.meta['N'], lik, nq)
    errs.update(ELBO=rel_err(E, g.t('ELBO')), ELL=rel_err(ELL, g.t('ELL')), KLD=rel_err(KLD, g.t('KLD')))
    bad = {k: e for k, e in errs.items() if not e <= TOL}
    assert not bad, (bad, errs)
    gw = {'m': L.t() @ grads['m'], 'L_raw': (L.t() @ grads['L_raw']).tril()}
    gerrs = g.grad_errors(gw)
    assert any(k.startswith('L_raw') for k in gerrs) and 'm' in gerrs
    bad = {k: e for k, e in gerrs.items() if not e < 1e-9}
    assert not bad, (bad, gerrs)


def test_kl_matches_the_closed_form():
    """kl_divergence of the two MultivariateNormals equals 0.5 (tr(K^-1 S) + m' K^-1 m - M + log|K| - log|S|), and is unchanged
    when a column of P changes sign (the distribution depends on P P^T only)."""
    g = torch.Generator().manual_seed(3)
    f64 = torch.float64
    M, D = 9, 3
    p = dict(Z=torch.randn(M, D, generator=g, dtype=f64), raw_lengthscale=O.inv_softplus(torch.tensor([0.9, 1.4, 2.0], dtype=f64)),
             raw_outputscale=O.inv_softplus(torch.tensor(1.2, dtype=f64)), m=torch.randn(M, generator=g, dtype=f64),
             L_raw=0.4 * torch.eye(M, dtype=f64) + 0.1 * torch.randn(M, M, generator=g, dtype=f64), flow=[])
    K = O.rbf_ard(p['Z'], p['Z'], p['raw_lengthscale'], p['raw_outputscale'])
    P = p['L_raw'].tril()
    S = P @ P.t()
    Ki = torch.linalg.inv(K)
    ref = 0.5 * (torch.trace(Ki @ S) + p['m'] @ Ki @ p['m'] - M + torch.logdet(K) - torch.logdet(S))
    assert rel_err(UR.kl(p), ref) < 1e-12
    q = dict(p)
    q['L_raw'] = p['L_raw'].clone()
    q['L_raw'][:, 2] *= -1.0
    assert rel_err(UR.kl(q), UR.kl(p)) < 1e-14
