"""Full covariance of q(f) over a test batch, its Cholesky factor and joint samples on the GPU (tgp_qf_cov_forward,
tgp_cov_cholesky, tgp_cov_sample and the diagonal=False class API), against the CPU reference of tests/joint_ref.py."""
import warnings

import pytest
import torch

from oracle import tgp_oracle as O
from tests import joint_ref as JR
from tests.golden_util import Golden, rel_err
from tests.gpu_util import engine_inputs
from tests.matern_ref import kernel_ard

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
KINDS = ['rbf', 'matern12', 'matern32', 'matern52']
MODES = ['f64', 'i8crt', 'tf32x3']
EPS = 2.220446049250313e-16


def _problem(M, D, seed, kernel, n=2048):
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    X = torch.randn(n, D, generator=g, dtype=f64)
    Z = X[torch.randperm(n, generator=g)[:M]].clone()
    p = dict(Z=Z, raw_lengthscale=O.inv_softplus(1.0 + 2.0 * torch.rand(D, generator=g, dtype=f64)) * (D / 8.0) ** 0.5,
             raw_outputscale=O.inv_softplus(torch.tensor(1.3, dtype=f64)), m=torch.randn(M, generator=g, dtype=f64),
             L_raw=0.6 * torch.eye(M, dtype=f64) + 0.05 * torch.randn(M, M, generator=g, dtype=f64),
             log_var_noise=torch.tensor(-1.0, dtype=f64), kernel=kernel)
    return X, p


def _fixture_problem(kernel):
    g = Golden('synth_reg_d8_m1024_p1')
    p = g.oracle_params('train')
    p['kernel'] = kernel
    return g.t('X'), p


def _engine(p, compute):
    from tgp.pytorch_b200.engine import Engine, FlowLayout
    return Engine(p['Z'].shape[0], p['Z'].shape[1], 'gauss_linear', 0, FlowLayout([]), DEV, compute=compute,
                  kernel=p['kernel'])


def _gpu_joint(eng, X, p):
    from tgp.pytorch_b200 import functional as Fn
    ei = engine_inputs(p, DEV)
    with torch.no_grad():
        mu, cov = Fn.qf_covariance(eng, X.to(DEV).contiguous(), ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'])
        mu_d, v_d = Fn.qf_marginals(eng, X.to(DEV).contiguous(), ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'])
    return mu, cov, mu_d, v_d


def _check_sigma(X, p, compute, R):
    s = JR.outputscale(p)
    eng = _engine(p, compute)
    mu, cov, mu_d, v_d = _gpu_joint(eng, X[:R], p)
    mu_r, cov_r = JR.qf_joint(X[:R], p)
    cond = float(torch.linalg.cond(kernel_ard(p['Z'], p['Z'], p)))
    bound = max(1e-10, 100 * EPS * cond ** 0.5) * s
    err = float((cov.cpu() - cov_r).abs().max())
    d_err = float((torch.diagonal(cov) - v_d).abs().max())
    from tests.conftest import record_residuals
    record_residuals('joint:%s:%s:M%d' % (compute, p['kernel'], p['Z'].shape[0]),
                     {'sigma_max_abs_over_s': err / s, 'bound_over_s': bound / s, 'mu_rel': rel_err(mu.cpu(), mu_r),
                      'diag_vs_v_over_s': d_err / s, 'mu_vs_diag_path_max_abs': float((mu - mu_d).abs().max())})
    assert err <= bound, (err / s, bound / s)
    assert rel_err(mu.cpu(), mu_r) <= 1e-10
    assert torch.equal(cov, cov.t())
    assert d_err <= (1e-5 if compute == 'tf32x3' else 1e-10) * s, d_err / s
    if compute == 'f64':          # the same K tiles, the same two GEMMs and k_row_stats as the diagonal path
        assert torch.equal(mu, mu_d)


@pytest.mark.parametrize('R', [1, 63, 64, 65, 200, 2048])
@pytest.mark.parametrize('kernel', KINDS)
@pytest.mark.parametrize('compute', MODES)
def test_sigma_against_the_reference(compute, kernel, R):
    X, p = _problem(64, 8, seed=5 + KINDS.index(kernel), kernel=kernel)
    _check_sigma(X, p, compute, R)


@pytest.mark.parametrize('kernel', KINDS)
@pytest.mark.parametrize('compute', MODES)
def test_sigma_on_the_m1024_fixture(compute, kernel):
    X, p = _fixture_problem(kernel)
    _check_sigma(X, p, compute, 2048)


@pytest.mark.parametrize('R', [63, 64, 65, 200, 2048])
def test_cholesky_reconstructs_and_has_a_zero_upper_triangle(R):
    X, p = _problem(64, 8, seed=11, kernel='matern52')
    s = JR.outputscale(p)
    eng = _engine(p, 'f64')
    _, cov, _, _ = _gpu_joint(eng, X[:R], p)
    j = 1e-6 * s
    L, status = eng.cov_cholesky(cov, j)
    assert int(status.item()) == 0
    Lc, Sc = L.cpu(), cov.cpu() + j * torch.eye(R, dtype=torch.float64)
    rec = float((Lc @ Lc.t() - Sc).abs().max())
    L2, st2 = eng.cov_cholesky(cov, 0.5 * s)
    ref = torch.linalg.cholesky(cov.cpu() + 0.5 * s * torch.eye(R, dtype=torch.float64))
    from tests.conftest import record_residuals
    record_residuals('joint_cholesky', {'reconstruction_over_s': rec / s,
                                        'vs_lapack_over_sqrt_s': float((L2.cpu() - ref).abs().max()) / s ** 0.5})
    assert rec <= 1e-12 * s
    assert torch.equal(torch.triu(Lc, 1), torch.zeros(R, R, dtype=torch.float64))
    # well conditioned: the factor itself against LAPACK's on the same matrix
    assert int(st2.item()) == 0
    assert float((L2.cpu() - ref).abs().max()) <= 1e-10 * s ** 0.5


def test_duplicated_rows_take_the_jitter_ladder():
    from tgp.pytorch_b200 import functional as Fn
    X, p = _problem(64, 8, seed=13, kernel='rbf')
    Xd = torch.cat([X[:100], X[10:20], X[:3]])             # 13 rows repeated: Sigma is singular
    eng = _engine(p, 'f64')
    _, cov, _, _ = _gpu_joint(eng, Xd, p)
    _, status = eng.cov_cholesky(cov, 0.0)
    assert int(status.item()) != 0
    with pytest.warns(Fn.NumericalWarning):
        L, j = Fn.cov_cholesky_ladder(eng, cov, 1e-8, 0.0)
    assert j > 0
    s = JR.outputscale(p)
    Lc = L.cpu()
    assert float((Lc @ Lc.t() - cov.cpu() - j * torch.eye(cov.shape[0], dtype=torch.float64)).abs().max()) <= 1e-12 * s


def test_nan_parameter_raises_nan_error():
    from tgp.pytorch_b200 import functional as Fn
    X, p = _problem(64, 8, seed=17, kernel='rbf')
    eng = _engine(p, 'f64')
    _, cov, _, _ = _gpu_joint(eng, X[:100], p)
    bad = cov.clone()
    bad[5, 3] = bad[3, 5] = float('nan')
    with pytest.raises(Fn.NanError):
        Fn.cov_cholesky_ladder(eng, bad, 1e-8, 0.0)
    p['raw_lengthscale'] = p['raw_lengthscale'].clone()
    p['raw_lengthscale'][2] = float('nan')
    with pytest.raises(Fn.NanError):
        _gpu_joint(_engine(p, 'f64'), X[:100], p)


def test_seeded_samples_equal_the_cpu_formula():
    X, p = _problem(64, 8, seed=19, kernel='matern32')
    eng = _engine(p, 'f64')
    mu, cov, _, _ = _gpu_joint(eng, X[:200], p)
    L, status = eng.cov_cholesky(cov, 1e-6)
    assert int(status.item()) == 0
    eps = torch.randn(37, 200, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    f0 = eng.cov_sample(mu, L, eps.to(DEV))
    ref = mu.cpu().view(1, -1) + eps @ L.cpu().t()
    from tests.conftest import record_residuals
    record_residuals('joint_samples', {'vs_cpu_rel': rel_err(f0.cpu(), ref)})
    assert rel_err(f0.cpu(), ref) <= 1e-12
    assert rel_err(f0.cpu(), JR.joint_samples(mu.cpu(), cov.cpu(), 1e-6, eps)) <= 1e-8


def test_sample_mean_and_covariance_within_monte_carlo_error():
    from tgp.pytorch_b200 import functional as Fn
    X, p = _problem(64, 8, seed=23, kernel='matern52')
    eng = _engine(p, 'f64')
    mu, cov, _, _ = _gpu_joint(eng, X[:64], p)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        L, j = Fn.cov_cholesky_ladder(eng, cov, 1e-8, 0.0)
    S = 20000
    eps = torch.randn(S, 64, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    f0 = eng.cov_sample(mu, L, eps.to(DEV)).cpu()
    Sig = cov.cpu() + j * torch.eye(64, dtype=torch.float64)
    d = torch.diagonal(Sig)
    assert bool(((f0.mean(0) - mu.cpu()).abs() <= 5 * (d / S).sqrt()).all())
    C = torch.cov(f0.t())
    sd = ((d.view(-1, 1) * d.view(1, -1) + Sig ** 2) / S).sqrt()
    assert bool(((C - Sig).abs() <= 5 * sd + 1e-15).all())


# ---- class API ------------------------------------------------------------------------------------------------------
def _golden_model(name):
    from tests.model_util import build_from_golden
    g = Golden(name)
    return g, build_from_golden(g, DEV)


def _params_of(model, dy, kernel='rbf'):
    kern = model.covariance_function
    ki = 0 if model.kernel_is_shared else dy
    return dict(Z=model.Z[0 if model.Z_is_shared else dy].detach().cpu().double(),
                raw_lengthscale=kern.base_kernel.raw_lengthscale[ki, 0].detach().cpu().double(),
                raw_outputscale=kern.raw_outputscale[ki].detach().cpu().double(),
                m=model.q_U.variational_mean[0 if model.q_U_is_shared else dy].detach().cpu().double(),
                L_raw=model.q_U.chol_variational_covar[0 if model.q_U_is_shared else dy].detach().cpu().double(),
                kernel=kernel)


@pytest.mark.parametrize('name', ['boston_tgp_steptanh13_p1', 'boston_tgp_sal2_p1'])
def test_tgp_joint_samples_go_through_the_flow(name):
    g, model = _golden_model(name)
    model.set_is_training(False)
    Xt = g.t('Xte').to(DEV)
    MB, S = Xt.shape[0], 5
    torch.manual_seed(0)
    with torch.no_grad():
        f, mean, cov, f0 = model.sample_from_variational_marginal(Xt, S, diagonal=False, is_duvenaud=False)
        assert f.shape == (1, S * MB) and f0.shape == (1, S * MB)
        assert mean.shape == (1, S * MB, 1) and cov.shape == (1, MB, MB)
        model._eval_mode()
        ref = model.G_matrix[0](f0[0], Xt.repeat(S, 1))
        model.train()
    assert torch.equal(f[0], ref)
    mu_r, cov_r = JR.qf_joint(g.t('Xte'), _params_of(model, 0))
    assert rel_err(cov[0].cpu(), cov_r) < 1e-9 and rel_err(mean[0, :MB, 0].cpu(), mu_r) < 1e-10
    with torch.no_grad():
        fb, mb, cb = model.sample_from_variational_marginal_base(Xt, diagonal=False, is_duvenaud=False)
    assert fb.shape == (1, MB) and mb.shape == (1, MB, 1) and cb.shape == (1, MB, MB)


def test_svgp_joint_samples_take_the_identity_flow():
    from tgp.pytorch_b200.dsp.models import sparse_MF_SP
    g, model = _golden_model('boston_svgp_p1')
    Xt = g.t('Xte').to(DEV)
    with torch.no_grad():
        f, _, _, f0 = sparse_MF_SP.sample_from_variational_marginal(model, Xt, 3, diagonal=False, is_duvenaud=False)
    assert torch.equal(f, f0)


@pytest.mark.parametrize('shared', [True, False])
def test_two_outputs_shapes_and_values(shared):
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    cg.device = DEV
    from tgp.pytorch_b200.dsp.models import instance_kernel, sparse_MF_GP
    from tgp.pytorch_b200.dsp.likelihoods import GaussianLinearMean
    K = instance_kernel('scale_matern', ard_num_dim=8, num_multioutput=2, kernel_is_shared=shared,
                        init_params={'length_scale': 2.0, 'kernel_scale': 1.5, 'nu': 2.5})
    X, p = _problem(64, 8, seed=29, kernel='matern52', n=600)
    lik = GaussianLinearMean(out_dim=2, noise_init=0.3, noise_is_shared=False)
    ip = {'variational_distribution': {'variance_scale': 0.5, 'mean_scale': 0.3}}
    model = sparse_MF_GP(['zero', K], X, p['Z'], 6000, lik, 2, True, shared, False, False, False, 0.0, ip).to(DEV)
    with torch.no_grad():
        if not shared:
            K.base_kernel.raw_lengthscale[1].add_(0.3)
        model.q_U.variational_mean[1].mul_(-0.7)
    Xd = X.to(DEV)
    with torch.no_grad():
        mean, cov = model.marginal_variational_qf_parameters(Xd, diagonal=False, is_duvenaud=False)
    assert mean.shape == (2, 600, 1) and cov.shape == (2, 600, 600) and cov.dtype == torch.float64
    for dy in range(2):
        mu_r, cov_r = JR.qf_joint(X, _params_of(model, dy, 'matern52'))
        assert rel_err(mean[dy, :, 0].cpu(), mu_r) < 1e-10
        assert float((cov[dy].cpu() - cov_r).abs().max()) < 1e-9
    model.set_is_training(False)
    m1, m2, mq, cq = model.predictive_distribution(Xd, diagonal=False)
    noise = torch.exp(lik.log_var_noise.detach()).view(2, 1, 1)
    assert rel_err(m2.cpu(), (cq + noise * torch.eye(600, dtype=torch.float64, device=DEV)).cpu()) <= 1e-15
    assert m2.shape == (2, 600, 600) and torch.equal(m1, mq.squeeze(2))
    with pytest.raises(NotImplementedError, match='no_grad'):
        model.marginal_variational_qf_parameters(Xd, diagonal=False, is_duvenaud=False)


def test_float32_model_returns_float32_within_fp32_error():
    g, model = _golden_model('boston_svgp_p1')
    model = model.float()
    Xt = g.t('Xte', torch.float32).to(DEV)
    with torch.no_grad():
        mean, cov = model.marginal_variational_qf_parameters(Xt, diagonal=False, is_duvenaud=False)
        _, v = model.marginal_variational_qf_parameters(Xt, diagonal=True, is_duvenaud=False)
    assert mean.dtype == torch.float32 and cov.dtype == torch.float32
    s = float(torch.nn.functional.softplus(model.covariance_function.raw_outputscale.double()))
    assert float((torch.diagonal(cov[0]).double() - v[0, :, 0].double()).abs().max()) <= 1e-5 * s


def test_bernoulli_and_multiclass_shapes_and_predictive_refusal():
    from tgp.pytorch_b200.dsp import config as cg
    g, model = _golden_model('synth_clf_d16_m48_p1')
    model.set_is_training(False)
    Xt = g.t('Xte').to(DEV)
    with torch.no_grad():
        mean, cov = model.marginal_variational_qf_parameters(Xt, diagonal=False, is_duvenaud=False)
    assert mean.shape == (1, Xt.shape[0], 1) and cov.shape == (1, Xt.shape[0], Xt.shape[0])
    with pytest.raises(NotImplementedError, match='GaussianLinearMean'):
        model.predictive_distribution(Xt, diagonal=False)
    from tests.golden_util import MulticlassGolden
    from tgp.pytorch_b200.dsp import flows as F
    from tgp.pytorch_b200.dsp.models import instance_kernel, sparse_MF_SP
    from tgp.pytorch_b200.dsp.models.flow import instance_flow
    from tgp.pytorch_b200.dsp.likelihoods import MulticlassCategorical
    mg = MulticlassGolden('mc_synth_c3_sal1_p1')
    Cn, M = mg.meta['C'], mg.meta['M']
    X = mg.t('X')
    cg.set_maximum_precission()
    K = instance_kernel('scale_rbf', ard_num_dim=X.shape[1], num_multioutput=Cn, kernel_is_shared=False)
    mc = sparse_MF_SP(['zero', K], X, X[:M].clone(), mg.meta['N'], MulticlassCategorical(Cn), Cn, True, False, False, False,
                      False, [instance_flow(F.SAL(1)) for _ in range(Cn)], 'single', 0.0, False).to(DEV)
    with torch.no_grad():
        mean, cov = mc.marginal_variational_qf_parameters(X.to(DEV), diagonal=False, is_duvenaud=False)
    assert mean.shape == (Cn, X.shape[0], 1) and cov.shape == (Cn, X.shape[0], X.shape[0])
    mc.set_is_training(False)
    with pytest.raises(NotImplementedError, match='GaussianLinearMean'):
        mc.predictive_distribution(X.to(DEV), diagonal=False)


def test_frozen_parameters_reuse_the_cached_factorisation():
    from tgp.pytorch_b200 import _lib
    lib = _lib.load()
    g, model = _golden_model('boston_tgp_sal2_p1')
    Xt = g.t('Xte').to(DEV)
    with torch.no_grad():
        n0 = lib.tgp_launch_count()
        mean1, cov1 = model.marginal_variational_qf_parameters(Xt, diagonal=False, is_duvenaud=False)
        n1 = lib.tgp_launch_count()
        mean2, cov2 = model.marginal_variational_qf_parameters(Xt, diagonal=False, is_duvenaud=False)
        n2 = lib.tgp_launch_count()
        eng = [e for k, e in model._engines.items() if k[0] == 'qf'][0]
        eng.qf_cov(Xt.double().contiguous())
        n3 = lib.tgp_launch_count()
    assert torch.equal(cov1, cov2) and torch.equal(mean1, mean2)
    assert n2 - n1 == n3 - n2 < n1 - n0          # the second call launches the covariance kernels only: no tgp_prepare


def _elbo_run(X, y, p, Xc=None):
    from tgp.pytorch_b200 import functional as Fn
    from tgp.pytorch_b200.engine import Engine, FlowLayout
    eng = Engine(p['Z'].shape[0], p['Z'].shape[1], 'gauss_linear', 0, FlowLayout([]), DEV, compute='f64', kernel=p['kernel'])
    ei = engine_inputs(p, DEV)
    leaves = [ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'], ei['log_var_noise']]
    for t in leaves:
        t.requires_grad_(True)
    ELL, KLD, _, mu, v = Fn.elbo_terms(eng, X.to(DEV).contiguous(), y.to(DEV).contiguous(), 3.0, *leaves, None)
    if Xc is not None:
        for _ in range(2):
            eng.qf_cov(Xc.to(DEV).contiguous())
    (ELL - KLD).backward()
    return [(ELL - KLD).detach().reshape(1), mu, v] + [t.grad.detach().reshape(-1) for t in leaves]


def test_covariance_calls_between_forward_and_backward_change_nothing():
    X, p = _problem(64, 8, seed=31, kernel='matern32')
    y = torch.randn(2048, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    a1 = _elbo_run(X, y, p)
    a2 = _elbo_run(X, y, p)
    b = _elbo_run(X, y, p, Xc=X[:300])
    assert torch.equal(b[1], a1[1]) and torch.equal(b[2], a1[2])          # mu, v: no atomics on the forward
    for x, y1, y2 in zip(b, a1, a2):
        spread = float((y1 - y2).abs().max())
        assert float((x - y1).abs().max()) <= max(4 * spread, 1e-14 * float(y1.abs().max())), (x, y1, spread)
