"""ARD-Matern kernels without a GPU: the closed forms of tests/matern_ref.py against the general Matern formula, its gradients against finite
differences (coincident points included), the kernel modules' parameter surface, and the C-ABI's kernel field."""
import numpy as np
import pytest
import scipy.special as sp
import torch

from oracle import tgp_oracle as O
from tests import matern_ref as MR

NUS = {'matern12': 0.5, 'matern32': 1.5, 'matern52': 2.5}


def _general_matern(r, nu):
    """2^(1-nu) / Gamma(nu) (sqrt(2 nu) r)^nu K_nu(sqrt(2 nu) r), with the limit 1 at r = 0."""
    x = np.sqrt(2.0 * nu) * r
    out = np.ones_like(r)
    pos = x > 0
    out[pos] = 2.0 ** (1.0 - nu) / sp.gamma(nu) * x[pos] ** nu * sp.kv(nu, x[pos])
    return out


@pytest.mark.parametrize('kind', list(NUS))
def test_closed_form_matches_the_general_matern_formula(kind):
    g = torch.Generator().manual_seed(1)
    X = torch.randn(40, 5, generator=g, dtype=torch.float64)
    Z = torch.randn(30, 5, generator=g, dtype=torch.float64)
    raw_ls = O.inv_softplus(0.5 + 2.0 * torch.rand(5, generator=g, dtype=torch.float64))
    raw_os = O.inv_softplus(torch.tensor(1.7, dtype=torch.float64))
    K = MR.matern_ard(X, Z, raw_ls, raw_os, NUS[kind]).numpy()
    ls = torch.nn.functional.softplus(raw_ls).numpy()
    r = np.sqrt((((X.numpy()[:, None, :] - Z.numpy()[None, :, :]) / ls) ** 2).sum(-1))
    ref = 1.7 * _general_matern(r, NUS[kind])
    assert np.max(np.abs(K - ref) / np.abs(ref)) < 1e-12
    Kzz = MR.matern_ard(Z, Z, raw_ls, raw_os, NUS[kind])
    assert torch.equal(torch.diagonal(Kzz), torch.full((30,), float(torch.nn.functional.softplus(raw_os)), dtype=torch.float64))


def _small_problem(kind, seed=4):
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    X = torch.randn(25, 3, generator=g, dtype=f64)
    y = torch.randn(25, generator=g, dtype=f64)
    p = dict(Z=X[:6].clone() + 0.0, raw_lengthscale=O.inv_softplus(torch.tensor([0.8, 1.5, 2.2], dtype=f64)),
             raw_outputscale=O.inv_softplus(torch.tensor(1.3, dtype=f64)), m=torch.randn(6, generator=g, dtype=f64),
             L_raw=0.7 * torch.eye(6, dtype=f64) + 0.05 * torch.randn(6, 6, generator=g, dtype=f64),
             log_var_noise=torch.tensor(-1.0, dtype=f64), flow=[], kernel=kind)
    return X, y, p


@pytest.mark.parametrize('kind', list(NUS))
def test_gradients_match_central_differences_with_coincident_points(kind):
    """Rows 0..5 of X are the inducing points.  For nu = 3/2 and 5/2 the ELBO is smooth there.  For nu = 1/2, |z - x| has a
    kink where z = x: the central quotient averages the two one-sided slopes of each coincident pair, which is the zero
    contribution of the convention, plus the smooth part of every other pair."""
    X, y, p = _small_problem(kind)
    _, _, _, _, g = MR.elbo_and_grads(X, y, p, 100.0, 'gauss_linear', 0)
    for name in ('Z', 'raw_lengthscale', 'raw_outputscale'):
        base = p[name].detach().clone()
        fd = torch.zeros_like(base).reshape(-1)
        for i in range(base.numel()):
            vals = []
            for sgn in (1.0, -1.0):
                q = dict(p)
                t = base.clone().reshape(-1)
                t[i] += sgn * 1e-6
                q[name] = t.reshape(base.shape)
                q = {k: (v.detach() if torch.is_tensor(v) else v) for k, v in q.items()}
                vals.append(float(MR.elbo(X, y, q, 100.0, 'gauss_linear', 0)[0]))
            fd[i] = (vals[0] - vals[1]) / 2e-6
        got = g[name].reshape(-1)
        assert torch.allclose(got, fd, rtol=2e-5, atol=2e-6), (name, got, fd)
        assert torch.isfinite(got).all()


def test_rbf_selection_reproduces_o2():
    """With p['kernel'] = 'rbf' the reference computes exactly what O2 computes (its only change is the kernel)."""
    X, y, p = _small_problem('rbf')
    p['flow'] = []
    E, ELL, KLD, rows, g = MR.elbo_and_grads(X, y, dict(p), 100.0, 'gauss_linear', 0)
    q = {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in p.items() if k != 'kernel'}
    E2, ELL2, KLD2, rows2, g2 = O.elbo_and_grads(X, y, q, 100.0, 'gauss_linear', 0)
    assert torch.equal(E, E2) and torch.equal(rows, rows2) and torch.equal(KLD, KLD2)
    for k in g2:
        assert torch.equal(g[k], g2[k]), k
    assert all(torch.equal(a, b) for a, b in zip(MR.qf_marginals(X, q), O.qf_marginals(X, q)))


def test_instance_kernel_surface_and_values():
    from tgp.pytorch_b200.dsp.models import instance_kernel
    X = torch.randn(7, 4, dtype=torch.float64)
    Z = torch.randn(5, 4, dtype=torch.float64)
    for nu, kind in ((0.5, 'matern12'), (1.5, 'matern32'), (2.5, 'matern52')):
        K = instance_kernel('scale_matern', ard_num_dim=4, num_multioutput=2, kernel_is_shared=False,
                            init_params={'length_scale': 2.0, 'kernel_scale': 1.5, 'nu': nu})
        assert [n for n, _ in K.named_parameters()] == ['raw_outputscale', 'base_kernel.raw_lengthscale']
        assert K.base_kernel.raw_lengthscale.shape == (2, 1, 4) and K.raw_outputscale.shape == (2,)
        assert K.base_kernel.nu == nu
        got = K(X, Z).evaluate()[0]
        ref = MR.matern_ard(X, Z, K.base_kernel.raw_lengthscale[0, 0], K.raw_outputscale[0], nu)
        assert torch.allclose(got, ref, rtol=1e-14, atol=0)
        bare = instance_kernel('matern', ard_num_dim=4, num_multioutput=1, kernel_is_shared=False, init_params={'nu': nu})
        assert [n for n, _ in bare.named_parameters()] == ['raw_lengthscale'] and bare.nu == nu
    assert instance_kernel('matern', ard_num_dim=4, num_multioutput=1, kernel_is_shared=False).nu == 2.5
    with pytest.raises(ValueError):
        instance_kernel('scale_matern', ard_num_dim=4, num_multioutput=1, kernel_is_shared=False, init_params={'nu': 1.0})


def _model(lib_mod, dtype, kernel=0, M=300, D=8):
    m = lib_mod.TgpModel()
    m.dtype, m.M, m.D, m.likelihood, m.n_quad, m.kernel = dtype, M, D, lib_mod.LIK_GAUSS_NONLINEAR, 20, kernel
    return m


def test_c_abi_kernel_field_validation_and_workspace_sizes():
    from tgp.pytorch_b200 import _lib
    import os
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip('libtgp_b200.so not built')
    lib = _lib.load()
    assert lib.tgp_step_workspace_bytes(_model(_lib, _lib.TGP_F64, kernel=4)) == 0
    assert b'kernel' in lib.tgp_last_error()
    assert lib.tgp_step_workspace_bytes(_model(_lib, _lib.TGP_F64, kernel=-1)) == 0
    kinds = (_lib.KERNEL_RBF, _lib.KERNEL_MATERN12, _lib.KERNEL_MATERN32, _lib.KERNEL_MATERN52)
    for dtype in (_lib.TGP_F64, _lib.TGP_F32, _lib.TGP_F64_I8):
        for D in (8, 40):
            sizes = {(lib.tgp_step_workspace_bytes(_model(_lib, dtype, k, D=D)),
                      lib.tgp_batch_workspace_bytes(_model(_lib, dtype, k, D=D), 5000),
                      lib.tgp_workspace_bytes(_model(_lib, dtype, k, D=D), 5000)) for k in kinds}
            assert len(sizes) == 1 and 0 not in next(iter(sizes)), sizes
