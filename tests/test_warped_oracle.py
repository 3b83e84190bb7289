"""The torch restatement of the warped GP (tests/warped_ref.py) on the CPU: an identity warp reproduces the GaussianLinearMean
rows of O2, an affine warp adds its analytic log-Jacobian, the flow-parameter gradients of the ELBO (double backward through
log G') match central differences, and the predictive moments of an identity warp are those of the Gaussian predictive."""
import math

import pytest
import torch

from oracle import tgp_oracle as O
from tests import warped_ref as W

f64 = torch.float64


def _t(x):
    return torch.tensor(x, dtype=f64)


def _problem(R=60, M=12, D=3, seed=0, flow=()):
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(R, D, generator=g, dtype=f64)
    y = torch.rand(R, generator=g, dtype=f64) * 2.0 + 0.2          # positive: Box-Cox warps are defined there
    p = dict(Z=X[:M].clone() + 0.01, raw_lengthscale=torch.zeros(D, dtype=f64) + 0.5, raw_outputscale=_t(0.3),
             m=0.3 * torch.randn(M, generator=g, dtype=f64), L_raw=0.5 * torch.eye(M, dtype=f64) + 0.02 * torch.randn(M, M, generator=g, dtype=f64),
             log_var_noise=_t(-1.5), flow=list(flow))
    return X, y, p


WARPS = {
    'steptanh': [('tanh_step', [(_t(0.2), _t(0.3), _t(0.5), _t(-0.2)), (_t(-0.1), _t(0.1), _t(1.5), _t(0.4)),
                                (_t(0.3), _t(-0.2), _t(0.9), _t(0.1))], True), ('affine', _t(1.1), _t(-0.2), False)],
    'sal2': [('sal', _t(0.1), _t(0.9), True, False), ('affine', _t(0.8), _t(0.1), True),
             ('sal', _t(-0.2), _t(1.2), True, False), ('affine', _t(1.3), _t(0.0), True)],
    'arcsinh': [('arcsinh', _t(0.1), _t(0.7), _t(0.3), _t(0.5), True, True)],
    'boxcox': [('boxcox', _t(0.7), False), ('affine', _t(1.2), _t(0.1), False)],
    'invboxcox': [('invboxcox', _t(0.6), True)],
    'stepgroup': [('step_group', [(('sal', _t(0.1), _t(0.3), True, False), (_t(0.2), _t(0.05))),
                                  (('arcsinh', _t(0.0), _t(0.5), _t(0.4), _t(0.2), True, False), None)], True)],
}


def test_identity_warp_is_the_gaussian_linear_row():
    X, y, p = _problem()
    mu, v = O.qf_marginals(X, p)
    assert torch.equal(W.ell_rows(mu, v, y, p).detach(), O.ell_rows_gauss_linear(mu, v, y, p).detach())
    for y_std in (1.0, 2.5):
        ref, (m1, m2) = O.test_log_likelihood(X, y, p, y_std, likelihood='gauss_linear')
        assert float(W.logp_rows(mu, v, y, p, y_std).sum()) == pytest.approx(float(ref), rel=1e-13)
    a, b = W.moments(mu, v, p, 40)
    assert torch.allclose(a, m1, rtol=1e-12, atol=1e-13) and torch.allclose(b, m2, rtol=1e-10)


def test_affine_warp_adds_log_a():
    X, y, p = _problem(flow=[('affine', _t(2.5), _t(-0.4), False)])
    mu, v = O.qf_marginals(X, p)
    ref = O.ell_rows_gauss_linear(mu, v, 2.5 * y - 0.4, p) + math.log(2.5)
    assert torch.allclose(W.ell_rows(mu, v, y, p).detach(), ref.detach(), rtol=1e-14, atol=1e-14)
    ref_t = W.logp_rows(mu, v, 2.5 * y - 0.4, dict(p, flow=[])) + math.log(2.5)
    assert torch.allclose(W.logp_rows(mu, v, y, p), ref_t, rtol=1e-14, atol=1e-14)


@pytest.mark.parametrize('warp', sorted(WARPS))
def test_flow_gradients_match_central_differences(warp):
    X, y, p = _problem(flow=WARPS[warp], seed=len(warp))
    _, _, _, _, g = W.elbo_and_grads(X, y, p, 500.0)
    leaves = {k: t for k, t in O.leaf_params(p).items() if k.startswith('flow')}
    assert leaves
    for name, t in leaves.items():
        h = 1e-6 * max(1.0, abs(float(t)))
        with torch.no_grad():
            t += h
            up = W.elbo(X, y, p, 500.0)[0]
            t -= 2 * h
            dn = W.elbo(X, y, p, 500.0)[0]
            t += h
        fd = float(up - dn) / (2 * h)
        assert float(g[name]) == pytest.approx(fd, rel=1e-6, abs=1e-6), (warp, name)


@pytest.mark.parametrize('warp', sorted(WARPS))
def test_inverse_and_moments(warp):
    X, y, p = _problem(flow=WARPS[warp], R=8, M=4)
    z = O.apply_flow(p['flow'], y).detach()
    assert torch.allclose(W.inverse(p['flow'], z.numpy()), y, rtol=1e-12, atol=1e-12)
    mu, v = O.qf_marginals(X, p)
    m1, m2 = W.moments(mu, v, p, 20)
    assert torch.isfinite(m1).all() and (m2 > 0).all()
