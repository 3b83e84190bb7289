"""Full-size checks at the BASELINE configurations.  Every compute mode against the oracle (O.elbo_and_grads and
O.qf_marginals take seconds at these sizes on a multi-core host): ELBO, per-row terms, mu, v and every gradient.  Then
properties the oracle does not cover: central finite differences of the ELBO against the analytic gradients, row-shard
additivity, agreement of the tensor-core mode with the FP64 mode, finiteness.

cfg4: regression, D = 8, M = 1024, 65536-row minibatch, StepTanhL(1,3), Gaussian likelihood, 100 GH points.
cfg5: binary classification, D = 16, M = 2048, Bernoulli likelihood, SAL(1) flow (32768-row minibatch here).
Both span several of the 16384-row chunks of 'i8crt' and 'tf32x3'.
"""
import functools
import math

import pytest
import torch

from oracle import tgp_oracle as O
from tests.golden_util import rel_err
from tests.test_gpu_matern import _to

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _state(M, D, R, seed, classification):
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    X = torch.randn(R, D, generator=g, dtype=f64)
    w = torch.randn(D, generator=g, dtype=f64)
    if classification:
        pr = 0.5 * (1 + torch.erf((X @ w) / math.sqrt(D) / math.sqrt(2.0)))
        y = (pr > torch.rand(R, generator=g, dtype=f64)).to(f64)
    else:
        y = torch.sinh(0.7 * (X @ w) / math.sqrt(D)) + 0.1 * torch.randn(R, generator=g, dtype=f64)
        y = (y - y.mean()) / y.std()
    p = dict(Z=X[torch.randperm(R, generator=g)[:M]].clone(),
             raw_lengthscale=O.inv_softplus(1.5 + torch.rand(D, generator=g, dtype=f64)),
             raw_outputscale=O.inv_softplus(torch.tensor(1.5, dtype=f64)),
             m=0.5 * torch.randn(M, generator=g, dtype=f64),
             L_raw=0.5 * torch.eye(M, dtype=f64) + 0.02 * torch.randn(M, M, generator=g, dtype=f64),
             log_var_noise=torch.tensor(math.log(0.1), dtype=f64))
    if classification:
        p['flow'] = [('sal', torch.tensor(0.1, dtype=f64), torch.tensor(1.05, dtype=f64), False, False),
                     ('affine', torch.tensor(0.9, dtype=f64), torch.tensor(0.05, dtype=f64), False)]
    else:
        steps = [(torch.tensor(0.1 * i, dtype=f64), torch.tensor(-0.5, dtype=f64), torch.tensor(0.3 * i - 0.3, dtype=f64),
                  torch.tensor(0.2, dtype=f64)) for i in range(3)]
        p['flow'] = [('tanh_step', steps, True), ('affine', torch.tensor(1.05, dtype=f64), torch.tensor(-0.02, dtype=f64), False)]
    return X, y, p


def _elbo(p, X, y, N, lik, compute, grads=True, overrides=None):
    from tests.gpu_util import engine_inputs, make_engine
    from tgp.pytorch_b200 import functional as Fn
    eng, theta, _, names = make_engine(p, lik, 100, DEV, compute=compute)
    ei = engine_inputs(p, DEV)
    if overrides:
        for k, fn in overrides.items():
            ei[k] = fn(ei[k])
    leaves = [ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'], ei['log_var_noise'], theta]
    for t in leaves:
        t.requires_grad_(grads)
    ELL, KLD, rows, mu, v = Fn.elbo_terms(eng, X, y, N / X.shape[0], ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'],
                                          None if lik == 'bernoulli' else ei['log_var_noise'], theta, None)
    E = ELL - KLD
    if grads:
        E.backward()
    return E.detach(), rows, {k: t.grad for k, t in zip(('Z', 'raw_ls', 'raw_os', 'm', 'L_raw', 'noise', 'theta'), leaves)}, mu, v


def _cfg(cfg):
    """(classification, M, D, R, N, likelihood) of a BASELINE configuration."""
    clf = cfg == 'cfg5'
    M, D, R, N = (2048, 16, 32768, 1.0e6) if clf else (1024, 8, 65536, 5.0e6)
    return clf, M, D, R, N, 'bernoulli' if clf else 'gauss_nonlinear'


@functools.lru_cache(maxsize=None)
def _reference(cfg, dtype):
    """The oracle at `cfg` in `dtype` (computed once for the three modes): ELBO, rows, mu, v and every gradient."""
    clf, M, D, R, N, lik = _cfg(cfg)
    X, y, p = _state(M, D, R, seed=2024, classification=clf)
    if dtype != torch.float64:
        X, y, p = X.to(dtype), y.to(dtype), _to(p, dtype)
    E, _, _, rows, gr = O.elbo_and_grads(X, y, p, N, lik, 100)
    with torch.no_grad():
        mu, v = O.qf_marginals(X, p)
    out = dict(ELBO=E, rows=rows, mu=mu, v=v)
    out.update({k: t.detach() for k, t in gr.items() if not (clf and k == 'log_var_noise')})
    return out


@pytest.mark.parametrize('compute', ['f64', 'i8crt', 'tf32x3'])
@pytest.mark.parametrize('cfg', ['cfg4', 'cfg5'])
def test_full_size_every_mode_against_the_oracle(cfg, compute):
    """ELBO, per-row terms, mu, v and every gradient against the oracle.  FP64 modes: the bounds of tests/test_gpu_matern.py
    (1e-10, 1e-9 on v; the Bernoulli bounds of tests/test_gpu_parity.py at cfg5).  'tf32x3': 1e-5 + 4 x (the oracle's own
    float32 evaluation against its float64 one).  At cfg5 that yardstick bounds ELBO, rows, mu and v only: the oracle's float32
    gradients differ from its float64 ones by O(1) there (measured 0.8 on dZ, 1.1 on dm: the Bernoulli ELL is formed by
    cancellation), so they bound nothing; the tensor-core gradient of m stays checked against the FP64 mode at cfg5 by
    test_full_size_finite_differences_and_modes."""
    from tests.conftest import record_residuals
    from tests.test_gpu_matern import _ok
    clf, M, D, R, N, lik = _cfg(cfg)
    X, y, p = _state(M, D, R, seed=2024, classification=clf)
    E, rows, g, mu, v = _elbo(p, X.to(DEV).contiguous(), y.to(DEV).contiguous(), N, lik, compute)
    from tests.gpu_util import flow_layout_and_params
    names = flow_layout_and_params(p['flow'], 'cpu')[3]
    got = dict(ELBO=E, rows=rows, mu=mu, v=v, Z=g['Z'], raw_lengthscale=g['raw_ls'], raw_outputscale=g['raw_os'], m=g['m'],
               L_raw=g['L_raw'])
    if not clf:
        got['log_var_noise'] = g['noise']
    got.update({n: g['theta'][i] for i, n in enumerate(names)})
    ref = _reference(cfg, torch.float64)
    assert set(got) == set(ref)
    errs = {k: rel_err(t.detach().cpu().reshape(-1), ref[k]) for k, t in got.items()}
    record_residuals('full_size[%s,%s]' % (cfg, compute), errs)
    if compute == 'tf32x3':
        ref32 = _reference(cfg, torch.float32)
        keys = ('ELBO', 'rows', 'mu', 'v') if clf else tuple(errs)
        bad = {k: (errs[k], rel_err(ref32[k], ref[k])) for k in keys if not errs[k] < 1e-5 + 4.0 * rel_err(ref32[k], ref[k])}
    else:
        bad = {k: e for k, e in errs.items() if not _ok(k, e, lik)}
    assert not bad, (bad, errs)


@pytest.mark.parametrize('cfg', ['cfg4', 'cfg5'])
def test_full_size_finite_differences_and_modes(cfg):
    clf, M, D, R, N, lik = _cfg(cfg)
    X, y, p = _state(M, D, R, seed=2024, classification=clf)
    Xd, yd = X.to(DEV).contiguous(), y.to(DEV).contiguous()
    E, rows, g, _, _ = _elbo(p, Xd, yd, N, lik, 'f64')
    assert torch.isfinite(E) and torch.isfinite(rows).all()
    for t in g.values():
        assert t is None or torch.isfinite(t).all()
    # central finite differences along three parameter directions (FP64, h chosen for ~1e-7 truncation/round-off balance)
    h = 1e-5
    def fd(key, direction):
        up = _elbo(p, Xd, yd, N, lik, 'f64', grads=False, overrides={key: lambda t: t + h * direction})[0]
        dn = _elbo(p, Xd, yd, N, lik, 'f64', grads=False, overrides={key: lambda t: t - h * direction})[0]
        return float((up - dn) / (2 * h))
    gen = torch.Generator().manual_seed(1)
    d_ls = torch.randn(D, generator=gen, dtype=torch.float64).to(DEV)
    d_m = torch.randn(M, generator=gen, dtype=torch.float64).to(DEV)
    d_Z = torch.randn(M, D, generator=gen, dtype=torch.float64).to(DEV)
    for key, d in (('raw_ls', d_ls), ('m', d_m), ('Z', d_Z)):
        ana = float((g[key] * d).sum())
        num = fd(key, d)
        assert abs(ana - num) < 2e-6 * max(abs(ana), abs(num)), (cfg, key, ana, num)
    # row-shard additivity: two slices with the global scale
    from tests.gpu_util import engine_inputs, make_engine
    eng, theta, _, _ = make_engine(p, lik, 100, DEV)
    ei = engine_inputs(p, DEV)
    eng.set_params(ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'], None if clf else ei['log_var_noise'], theta)
    kl, _ = eng.prepare(0.0)
    tot = 0.0
    for sl in (slice(0, R // 3), slice(R // 3, R)):
        rb = eng.new_reduce_buffer()
        mu, v = eng.qf_forward(Xd[sl].contiguous())
        eng.ell_forward(mu, v, yd[sl].contiguous(), None, N / R, rb, want_grad=False)
        tot = tot + rb[0]
    assert rel_err((N / R * tot - kl[0]).cpu(), E.cpu()) < 1e-12
    # tensor-core mode against the FP64 mode at full size
    E32, rows32, g32, _, _ = _elbo(p, Xd, yd, N, lik, 'tf32x3')
    errs = {'ELBO': rel_err(E32.cpu(), E.cpu()), 'rows': rel_err(rows32.cpu(), rows.cpu()), 'grad m': rel_err(g32['m'].cpu(), g['m'].cpu())}
    from tests.conftest import record_residuals
    record_residuals('tf32x3_full_size:' + cfg, errs)
    # north_star's FP32 tolerance (1e-5 relative) on the ELBO at the BASELINE sizes; the mean is accumulated in FP64 as
    # mu = K_xz (L^-T m) by the K generation — taken from the FP32 rows a = L^-1 k it missed this bound (2.9e-5 at cfg4)
    assert errs['ELBO'] < 1e-5, errs
    assert errs['rows'] < 1e-4, errs
    assert errs['grad m'] < 3e-4, errs
