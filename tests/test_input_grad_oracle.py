"""The CPU reference of dELBO/dX (tests/input_grad_ref.py) pinned two ways on the regression and Bernoulli fixtures, for the RBF
and the three Matern kernels: by central finite differences on single coordinates, and by the translation identity
sum_n dE/dx_n + sum_j dE/dz_j = 0 (K_xz and K_zz, and so the ELBO, are unchanged when X and Z are shifted together)."""
import pytest
import torch

from tests import input_grad_ref as IR
from tests.golden_util import Golden, golden_names

KINDS = ['rbf', 'matern12', 'matern32', 'matern52']
MATERN_FIXTURES = ['synth_reg_d8_m64_p1', 'synth_clf_d16_m48_p1', 'boston_tgp_sal2_p1']


def _cases():
    out = [(n, 'rbf') for n in golden_names(big=False)]
    return out + [(n, k) for n in MATERN_FIXTURES for k in KINDS[1:]]


def _fixture(name, kernel):
    g = Golden(name)
    p = g.oracle_params('train')
    p['kernel'] = kernel
    return g.t('X'), g.t('Y').view(-1), p, g.meta['N'], g.meta['likelihood'], g.meta['n_quad']


@pytest.mark.parametrize('name,kernel', _cases())
def test_translation_identity(name, kernel):
    X, y, p, N, lik, nq = _fixture(name, kernel)
    _, gx, gz = IR.elbo_grads_xz(X, y, p, N, lik, nq)
    assert float(gx.norm()) > 0.0
    resid = gx.sum(0) + gz.sum(0)
    scale = float(gx.abs().sum(0).norm() + gz.abs().sum(0).norm())
    assert float(resid.norm()) <= 1e-12 * scale, (float(resid.norm()), scale)


@pytest.mark.parametrize('name,kernel', [(n, 'rbf') for n in MATERN_FIXTURES] + [(n, k) for n in MATERN_FIXTURES[:2] for k in KINDS[1:]])
def test_central_differences(name, kernel):
    X, y, p, N, lik, nq = _fixture(name, kernel)
    _, gx, _ = IR.elbo_grads_xz(X, y, p, N, lik, nq)
    gen = torch.Generator().manual_seed(11)
    rows = torch.randperm(X.shape[0], generator=gen)[:4].tolist()
    # the row with the largest gradient, so that the check sees a coordinate that matters
    rows.append(int(gx.norm(dim=1).argmax()))
    h = 1e-5
    for n in rows:
        d = int(torch.randint(X.shape[1], (1,), generator=gen))
        Xp, Xm = X.clone(), X.clone()
        Xp[n, d] += h
        Xm[n, d] -= h
        fd = float(IR.elbo_value(Xp, y, p, N, lik, nq) - IR.elbo_value(Xm, y, p, N, lik, nq)) / (2 * h)
        assert abs(fd - float(gx[n, d])) <= 1e-5 * max(1.0, float(gx.abs().max())), (n, d, fd, float(gx[n, d]))
