"""The CPU reference of the full q(f) covariance (tests/joint_ref.py) against the fixture-pinned marginals: on every golden
fixture, for the RBF and each Matern nu, mu and diag(Sigma) equal matern_ref.qf_marginals, and Sigma is symmetric and
positive semi-definite to rounding."""
import pytest
import torch

from tests import joint_ref as JR
from tests import matern_ref as MR
from tests.golden_util import Golden, golden_names, rel_err

KINDS = ['rbf', 'matern12', 'matern32', 'matern52']


@pytest.mark.parametrize('kernel', KINDS)
@pytest.mark.parametrize('name', golden_names())
def test_joint_restatement_matches_the_marginals(name, kernel):
    g = Golden(name)
    p = g.oracle_params('train')
    p['kernel'] = kernel
    X = g.t('X')
    mu, Sigma = JR.qf_joint(X, p)
    mu_m, v_m = MR.qf_marginals(X, p)
    assert rel_err(mu, mu_m) <= 1e-14
    assert rel_err(torch.diagonal(Sigma), v_m) <= 1e-14
    assert torch.equal(Sigma, Sigma.t())
    assert float(torch.linalg.eigvalsh(Sigma).min()) >= -1e-12 * JR.outputscale(p)


def test_joint_samples_have_the_stated_form():
    g = torch.Generator().manual_seed(0)
    A = torch.randn(6, 6, generator=g, dtype=torch.float64)
    Sigma = A @ A.t()
    mu = torch.randn(6, generator=g, dtype=torch.float64)
    eps = torch.randn(4, 6, generator=g, dtype=torch.float64)
    f = JR.joint_samples(mu, Sigma, 1e-9, eps)
    L = torch.linalg.cholesky(Sigma + 1e-9 * torch.eye(6, dtype=torch.float64))
    assert torch.allclose(f, mu + eps @ L.t(), rtol=0, atol=0)
