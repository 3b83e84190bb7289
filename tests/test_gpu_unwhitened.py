"""The non-whitened q(u) (is_whiten=False, TGP_QU_UNWHITENED) on the GPU, in the three compute modes and for the four kernels,
against the CPU reference of tests/unwhitened_ref.py (the reference's non-whitened branch in torch FP64).

Problems are built as the non-whitened form of a whitened q(u): (m, P) = (L m_w, L P_w) with L of the CPU factorisation, so
that q(u) has the scale of a trained model; every quantity is then computed from (m, P) alone.
"""
import warnings

import numpy as np
import pytest
import torch

from oracle import tgp_oracle as O
from tests import joint_ref as JR
from tests import unwhitened_ref as UR
from tests.golden_util import Golden, MulticlassGolden, rel_err
from tests.gpu_util import engine_inputs, flow_layout_and_params

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
KINDS = ['rbf', 'matern12', 'matern32', 'matern52']
GRAD_KEYS = ('Z', 'raw_lengthscale', 'raw_outputscale', 'm', 'L_raw', 'log_var_noise')


def _problem(R, M, D, seed, kernel, lik='gauss_nonlinear'):
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    X = torch.randn(R, D, generator=g, dtype=f64)
    y = torch.randn(R, generator=g, dtype=f64)
    if lik == 'bernoulli':
        y = (y > 0).to(f64)
    Z = X[torch.randperm(R, generator=g)[:M]].clone()
    p = dict(Z=Z, raw_lengthscale=O.inv_softplus(1.0 + 2.0 * torch.rand(D, generator=g, dtype=f64)) * (D / 8.0) ** 0.5,
             raw_outputscale=O.inv_softplus(torch.tensor(1.3, dtype=f64)),
             m=torch.randn(M, generator=g, dtype=f64),
             L_raw=0.6 * torch.eye(M, dtype=f64) + 0.05 * torch.randn(M, M, generator=g, dtype=f64),
             log_var_noise=torch.tensor(-1.2, dtype=f64), kernel=kernel)
    if lik == 'gauss_nonlinear':
        steps = [tuple(0.3 * torch.randn((), generator=g, dtype=f64) for _ in range(4)) for _ in range(2)]
        p['flow'] = [('tanh_step', steps, True)]
    elif lik == 'bernoulli':
        p['flow'] = [('sal', torch.tensor(0.2, dtype=f64), torch.tensor(1.1, dtype=f64), False, False)]
    else:
        p['flow'] = []
    q, _ = UR.from_whitened(p)
    return X, y, q


def _engine(p, lik, nq, compute, whiten=False):
    from tgp.pytorch_b200.engine import Engine, FlowLayout
    fl, theta, _, names = flow_layout_and_params(p['flow'], DEV)
    if lik == 'gauss_linear':
        fl, theta = FlowLayout([]), torch.zeros(0, dtype=torch.float64, device=DEV)
    eng = Engine(p['Z'].shape[0], p['Z'].shape[1], lik, nq, fl, DEV, compute=compute, kernel=p.get('kernel', 'rbf'),
                 whiten=whiten)
    return eng, theta, names


def _cuda(X, y, p, N, lik, nq, compute, whiten=False, jitter=(0.0, None)):
    from tgp.pytorch_b200 import functional as Fn
    eng, theta, names = _engine(p, lik, nq, compute, whiten)
    ei = engine_inputs(p, DEV)
    leaves = [ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'], ei['log_var_noise'], theta]
    for t in leaves:
        t.requires_grad_(True)
    ELL, KLD, rows, mu, v = Fn.elbo_terms(eng, X.to(DEV).contiguous(), y.to(DEV).contiguous(), N / X.shape[0], *leaves[:6],
                                          theta, None, jitter=jitter)
    (ELL - KLD).backward()
    out = dict(ELBO=(ELL - KLD).detach().cpu(), ELL=ELL.detach().cpu(), KLD=KLD.detach().cpu(), rows=rows.cpu(), mu=mu.cpu(),
               v=v.cpu())
    for k, t in zip(GRAD_KEYS, leaves):
        out[k] = (t.grad if t.grad is not None else torch.zeros_like(t)).detach().cpu().reshape(-1)
    for i, n in enumerate(names):
        out[n] = theta.grad[i].detach().cpu()
    if lik == 'bernoulli':
        out.pop('log_var_noise')
    return out, eng


def _oracle(X, y, p, N, lik, nq):
    p = {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in p.items()}
    E, ELL, KLD, rows, gr = UR.elbo_and_grads(X, y, p, N, lik, nq)
    mu, v = UR.qf_marginals(X, p)
    out = dict(ELBO=E, ELL=ELL, KLD=KLD, rows=rows, mu=mu.detach(), v=v.detach())
    for k, t in gr.items():
        out[k] = t.detach().reshape(-1)
    return out


def _to(p, dt):
    return {k: (v.to(dt) if torch.is_tensor(v) else
                [tuple(x.to(dt) if torch.is_tensor(x) else (list(map(lambda s: tuple(t.to(dt) for t in s), x))
                                                            if isinstance(x, list) else x) for x in lay) for lay in v]
                if k == 'flow' else v) for k, v in p.items()}


def _ok(k, e, lik):
    """The FP64 bounds of the whitened path (tests/test_gpu_parity.py, tests/test_gpu_matern.py), Bernoulli's included."""
    if lik == 'bernoulli':
        if k in ('ELBO', 'ELL', 'rows'):
            return e < dict(ELBO=5e-6, ELL=5e-6, rows=1e-4)[k]
        if k not in ('KLD', 'mu', 'v'):
            return e < 2e-6
    return e < dict(v=1e-9, KLD=1e-12).get(k, 1e-10)


def _whitened_of(p):
    """The whitened parameters of the same q(f): (m_w, P_w) = (L^-1 m, L^-1 P), L of the CPU factorisation."""
    L = UR._factor(p)
    return dict(p, m=torch.linalg.solve_triangular(L, p['m'].view(-1, 1), upper=False).view(-1),
                L_raw=torch.linalg.solve_triangular(L, UR._tril(p), upper=False))


# 'tf32x3', gradient of m: dm = L^-T dm~ carries the FP32-grade error of dELL/dm~ (accumulated from the FP32 A planes) times
# the conditioning of L^-1.  Measured 2.4e-5 on the RBF / Gauss-Hermite problem below, against a yardstick of 1.9e-5
# (1e-5 + 4 x 2.3e-6); DESIGN.md section 5 reports it.  Every other quantity of every problem holds the yardstick.
TF32_DM_BOUND = 1e-4


@pytest.mark.parametrize('lik', ['gauss_nonlinear', 'gauss_linear', 'bernoulli'])
@pytest.mark.parametrize('kernel', KINDS)
@pytest.mark.parametrize('compute', ['f64', 'i8crt', 'tf32x3'])
def test_elbo_and_every_gradient_against_the_reference(compute, kernel, lik):
    X, y, p = _problem(1000, 64, 8, seed=31 + KINDS.index(kernel), kernel=kernel, lik=lik)
    nq = 30 if lik != 'gauss_linear' else 0
    got, _ = _cuda(X, y, p, 5000.0, lik, nq, compute)
    if lik == 'bernoulli' and compute != 'tf32x3':
        white, _ = _cuda(X, y, _whitened_of(p), 5000.0, lik, nq, compute, whiten=True)
    ref = _oracle(X, y, p, 5000.0, lik, nq)
    errs = {k: rel_err(got[k], ref[k]) for k in got}
    if compute == 'tf32x3':      # the yardstick of tests/test_gpu_tensorcore.py: the reference's FP32 evaluation against FP64
        ref32 = _oracle(X.float(), y.float(), _to(p, torch.float32), 5000.0, lik, nq)
        bound = {k: 1e-5 + 4.0 * rel_err(ref32[k], ref[k]) for k in errs}
        bound['m'] = max(bound['m'], TF32_DM_BOUND)
        bad = {k: (e, bound[k]) for k, e in errs.items() if not e < bound[k]}
    else:
        if lik == 'bernoulli':
            # ELL, ELBO and rows: where p = Phi(G(f)) rounds to 1 at a quadrature node, the reference's BCELoss takes
            # max(log(1 - p), -100), a step that two FP64 evaluations of the same q(f) need not take at the same nodes
            # (DESIGN.md section 5 (iii)).  For these three the whitened device path on the same q(f) is the yardstick;
            # mu, v, KLD and every gradient are held to the reference.
            for k in ('ELBO', 'ELL', 'rows'):
                errs[k + '_vs_whitened'] = rel_err(got[k], white[k])
                errs.pop(k)
        bad = {k: e for k, e in errs.items() if not (e < 1e-10 if k.endswith('_vs_whitened') else _ok(k, e, lik))}
    assert not bad, (bad, errs)


@pytest.mark.parametrize('kernel', KINDS)
@pytest.mark.parametrize('compute', ['f64', 'i8crt'])
def test_full_size(compute, kernel):
    """M = 1024: the full M x M gradient of L_raw through the non-whitened chain."""
    X, y, p = _problem(4096, 1024, 8, seed=5 + KINDS.index(kernel), kernel=kernel)
    got, _ = _cuda(X, y, p, 40960.0, 'gauss_nonlinear', 20, compute)
    ref = _oracle(X, y, p, 40960.0, 'gauss_nonlinear', 20)
    errs = {k: rel_err(got[k], ref[k]) for k in got}
    bad = {k: e for k, e in errs.items() if not _ok(k, e, 'gauss_nonlinear')}
    assert not bad, (bad, errs)


@pytest.mark.parametrize('compute', ['f64', 'i8crt'])
def test_identity_with_the_whitened_model_on_the_device(compute):
    """A non-whitened model built from a whitened one with the device's own L (export_step): same ELBO, mu and v, and
    d/dm_w = L^T d/dm, d/dP_w = tril(L^T d/dP)."""
    X, y, pw = _problem(1000, 64, 8, seed=41, kernel='matern52')
    pw = dict(pw)
    g = torch.Generator().manual_seed(2)
    pw['m'] = torch.randn(64, generator=g, dtype=torch.float64)
    pw['L_raw'] = 0.6 * torch.eye(64, dtype=torch.float64) + 0.05 * torch.randn(64, 64, generator=g, dtype=torch.float64).tril()
    w, eng = _cuda(X, y, pw, 5000.0, 'gauss_nonlinear', 30, compute, whiten=True)
    L = eng.export_step()[0].cpu()
    pu = dict(pw)
    pu['m'] = L @ pw['m']
    pu['L_raw'] = L @ pw['L_raw'].tril()
    u, _ = _cuda(X, y, pu, 5000.0, 'gauss_nonlinear', 30, compute)
    errs = {k: rel_err(u[k], w[k]) for k in ('ELBO', 'ELL', 'KLD', 'mu', 'v')}
    errs['dm'] = rel_err(L.t() @ u['m'], w['m'])
    errs['dL_raw'] = rel_err((L.t() @ u['L_raw'].reshape(64, 64)).tril(), w['L_raw'].reshape(64, 64))
    bad = {k: e for k, e in errs.items() if not e <= dict(dm=1e-10, dL_raw=1e-10).get(k, 1e-12)}
    assert not bad, (bad, errs)


def test_jitter_ladder_fixture():
    """The singular-K_zz fixture: the ladder's jittered L is the prior's L as well."""
    g = Golden('boston_svgp_jitter')
    p = g.oracle_params('train')
    p['kernel'] = 'rbf'
    q, _ = UR.from_whitened(p)
    X, y = g.t('X'), g.t('Y').view(-1)
    lik, nq = g.meta['likelihood'], g.meta['n_quad']
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter('always')
        got, _ = _cuda(X, y, q, g.meta['N'], lik, nq, 'f64')
    assert any('jitter' in str(w.message) for w in rec)
    ref = _oracle(X, y, q, g.meta['N'], lik, nq)
    errs = {k: rel_err(got[k], ref[k]) for k in got}
    # K_zz is singular to working precision: the whitened path's bound for this fixture (tests/test_gpu_parity.py)
    bad = {k: e for k, e in errs.items() if not e < 1e-7}
    assert not bad, (bad, errs)


def test_handle_api_matches_the_staged_entry_points():
    from tgp.pytorch_b200.session import ElboSession
    X, y, p = _problem(1000, 64, 8, seed=23, kernel='matern12')
    staged, _ = _cuda(X, y, p, 5000.0, 'gauss_nonlinear', 30, 'f64')
    eng, theta, _ = _engine(p, 'gauss_nonlinear', 30, 'f64')
    ei = engine_inputs(p, DEV)
    ses = ElboSession(eng, 1000)
    args = (ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'], ei['log_var_noise'], theta)
    out = ses.forward(X.to(DEV).contiguous(), y.to(DEV).contiguous(), 5.0, *args)
    assert int(out['status'].item()) == 0
    assert rel_err((out['terms'][0] - out['terms'][1]).cpu(), staged['ELBO']) < 1e-12
    assert rel_err(out['terms'][1].cpu(), staged['KLD']) < 1e-12
    grads = ses.backward(torch.tensor([1.0, -1.0], dtype=torch.float64, device=DEV))
    for k, n in (('Z', 'Z'), ('raw_ls', 'raw_lengthscale'), ('raw_os', 'raw_outputscale'), ('m', 'm'), ('L_raw', 'L_raw')):
        assert rel_err(grads[k].cpu().reshape(-1), staged[n]) < 1e-12, k
    ses.close()


def _svgp(Dy, X, p, kernel='scale_rbf', nu=None):
    """sparse_MF_GP with is_whiten=False, Dy outputs (own Z, kernel and q(u) each), parameters of p (output 0) and of p with
    a scaled m / L_raw (the other outputs)."""
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    cg.device = DEV
    from tgp.pytorch_b200.dsp.models import instance_kernel, sparse_MF_GP
    from tgp.pytorch_b200.dsp.likelihoods import GaussianLinearMean
    K = instance_kernel(kernel, ard_num_dim=X.shape[1], num_multioutput=Dy, kernel_is_shared=False,
                        init_params={} if nu is None else {'nu': nu})
    lik = GaussianLinearMean(out_dim=Dy, noise_init=0.3, noise_is_shared=False)
    model = sparse_MF_GP(['zero', K], X, p['Z'], 6000, lik, Dy, False, False, False, False, False, 0.0, {})
    assert not model.is_whiten
    with torch.no_grad():
        K.base_kernel.raw_lengthscale.copy_(p['raw_lengthscale'].view(1, 1, -1).expand_as(K.base_kernel.raw_lengthscale))
        K.raw_outputscale.fill_(float(p['raw_outputscale']))
        for dy in range(Dy):
            model.q_U.variational_mean[dy].copy_(p['m'] * (1.0 + 0.5 * dy))
            model.q_U.chol_variational_covar[dy].copy_(p['L_raw'] * (1.0 - 0.2 * dy))
    return model.to(DEV)


def _params_of(model, dy, kernel='rbf'):
    K = model.covariance_function
    return dict(Z=model.Z[dy].detach().cpu().double(), raw_lengthscale=K.base_kernel.raw_lengthscale[dy, 0].detach().cpu().double(),
                raw_outputscale=K.raw_outputscale[dy].detach().cpu().double(), m=model.q_U.variational_mean[dy].detach().cpu().double(),
                L_raw=model.q_U.chol_variational_covar[dy].detach().cpu().double(), kernel=kernel, flow=[])


def test_two_outputs_marginals_elbo_and_kld():
    """Dy = 2 through the class API: marginals, the ELBO's KL and KLD() against the reference for each output."""
    X, y, p = _problem(600, 64, 8, seed=9, kernel='rbf', lik='gauss_linear')
    model = _svgp(2, X, p)
    Xd = X.to(DEV)
    mean, cov = model.marginal_variational_qf_parameters(Xd, True, False)
    kld = model.KLD()
    assert kld.shape == (2,)
    for dy in range(2):
        po = _params_of(model, dy)
        mu_o, v_o = UR.qf_marginals(X, po)
        assert rel_err(mean[dy, :, 0].detach().cpu(), mu_o) < 1e-10
        assert rel_err(cov[dy, :, 0].detach().cpu(), v_o) < 1e-9
        assert rel_err(kld[dy].detach().cpu(), UR.kl(po)) < 1e-12
    Y = torch.randn(600, 2, dtype=torch.float64, device=DEV)
    ELBO, ELL, KLD = model.ELBO(Xd, Y)
    assert rel_err(KLD.detach().cpu(), kld.sum().detach().cpu()) < 1e-12
    (-ELBO).backward()
    for n, t in model.named_parameters():
        assert t.grad is not None and torch.isfinite(t.grad).all(), n


def test_kld_alone_and_between_an_elbo_and_its_backward():
    """KLD() has a backward of its own (the chain with gE = 0) and a factorisation of its own: evaluated between a forward and
    its backward, it leaves the pending ELBO and marginals backward intact."""
    X, y, p = _problem(600, 64, 8, seed=13, kernel='matern32', lik='gauss_linear')
    model = _svgp(1, X, p, kernel='scale_matern', nu=1.5)
    po = _params_of(model, 0, 'matern32')
    po.update(log_var_noise=model.likelihood.log_var_noise[0].detach().cpu().double().reshape(()))
    leaves = {k: po[k].clone().requires_grad_(True) for k in ('Z', 'raw_lengthscale', 'raw_outputscale', 'm', 'L_raw')}
    names = {'Z': 'Z', 'raw_lengthscale': 'covariance_function.base_kernel.raw_lengthscale',
             'raw_outputscale': 'covariance_function.raw_outputscale', 'm': 'q_U.variational_mean',
             'L_raw': 'q_U.chol_variational_covar'}
    own = dict(model.named_parameters())

    def check(loss_ref, tag):
        ref = torch.autograd.grad(loss_ref, list(leaves.values()))
        for (k, n), r in zip(names.items(), ref):
            assert rel_err(own[n].grad[0].detach().cpu().reshape(-1), r.reshape(-1)) < 1e-10, (tag, k)
        model.zero_grad()

    # alone
    kld = model.KLD()
    kld.sum().backward()
    check(UR.kl(dict(po, **leaves)), 'KLD alone')
    # between an ELBO and its backward: d(ELBO + KLD) = d(ELL)
    Xd, Yd = X.to(DEV), y.view(-1, 1).to(DEV)
    ELBO, _, _ = model.ELBO(Xd, Yd)
    kld = model.KLD()
    (ELBO + kld.sum()).backward()
    q = dict(po, **leaves)
    E_ref, _, K_ref, _ = UR.elbo(X, y, q, 6000.0, 'gauss_linear', 0)
    check(E_ref + K_ref, 'ELBO + KLD')
    # between the marginals and their backward
    mean, cov = model.marginal_variational_qf_parameters(Xd, True, False)
    kld = model.KLD()
    (mean.sum() + cov.sum() - kld.sum()).backward()
    mu_r, v_r = UR.qf_marginals(X, dict(po, **leaves))
    check(mu_r.sum() + v_r.sum() - UR.kl(dict(po, **leaves)), 'marginals - KLD')


@pytest.mark.parametrize('kernel', KINDS)
@pytest.mark.parametrize('compute', ['f64', 'i8crt', 'tf32x3'])
def test_full_covariance_and_joint_samples(compute, kernel):
    """diagonal=False: mu and Sigma of q(f) over a test batch against the reference's non-whitened algebra
    (K_xx - K_xz K^-1 K_zx + K_xz K^-1 S K^-1 K_zx), and joint samples mu + eps chol(Sigma)^T."""
    from tgp.pytorch_b200 import functional as Fn
    X, _, p = _problem(200, 128, 8, seed=51 + KINDS.index(kernel), kernel=kernel, lik='gauss_linear')
    eng, _, _ = _engine(p, 'gauss_linear', 0, compute)
    ei = engine_inputs(p, DEV)
    with torch.no_grad():
        mu, Sigma = Fn.qf_covariance(eng, X.to(DEV).contiguous(), ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'])
    K_zz = UR.kernel_ard(p['Z'], p['Z'], p)
    L_zz, _, _ = O.psd_safe_cholesky(K_zz)
    K_zx = UR.kernel_ard(X, p['Z'], p).t()
    P = p['L_raw'].tril()
    A = torch.cholesky_solve(K_zx, L_zz)
    ref = UR.kernel_ard(X, X, p) - K_zx.t() @ A + A.t() @ (P @ (P.t() @ A))
    ref = 0.5 * (ref + ref.t())
    assert rel_err(mu.cpu(), A.t() @ p['m']) < 1e-10
    assert rel_err(Sigma.cpu(), ref) < 1e-9
    assert rel_err(torch.diagonal(Sigma).cpu(), UR.qf_marginals(X, p)[1]) < 1e-9
    L, status = eng.cov_cholesky(Sigma, 1e-6)
    assert int(status.item()) == 0
    eps = torch.randn(5, 200, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    f = eng.cov_sample(mu, L, eps.to(DEV).contiguous())
    assert rel_err(f.cpu(), JR.joint_samples(mu.cpu(), Sigma.cpu(), 1e-6, eps)) <= 1e-8


def test_class_api_joint_posterior():
    """sparse_MF_GP(is_whiten=False): marginal_variational_qf_parameters and sample_from_variational_marginal with
    diagonal=False agree with the diagonal path."""
    X, _, p = _problem(300, 64, 8, seed=61, kernel='rbf', lik='gauss_linear')
    model = _svgp(1, X, p)
    model.eval()
    Xd = X.to(DEV)
    with torch.no_grad():
        mean_d, var_d = model.marginal_variational_qf_parameters(Xd, True, False)
        mean, cov = model.marginal_variational_qf_parameters(Xd, False, False)
        f, mean_s, cov_s, f0 = model.sample_from_variational_marginal(Xd, 4, False, False)
    assert cov.shape == (1, 300, 300) and f0.shape == (1, 4 * 300)
    assert rel_err(mean.cpu(), mean_d.cpu()) < 1e-12
    assert rel_err(torch.diagonal(cov[0]).cpu(), var_d[0, :, 0].cpu()) < 1e-10
    assert rel_err(cov_s.cpu(), cov.cpu()) < 1e-12 and torch.isfinite(f).all()


@pytest.mark.parametrize('compute', ['f64', 'i8crt'])
def test_multiclass_model_against_the_reference(compute):
    """C = 3 GPs (is_whiten=False) coupled by the Monte-Carlo softmax likelihood, through sparse_MF_SP with the parameters and
    noise draws of a multiclass fixture (its variational parameters read as non-whitened ones), against UR.elbo_multiclass.
    Each class's KL comes from the factorisation of its marginals."""
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    cg.device = DEV
    from tgp.pytorch_b200.dsp import flows as F
    from tgp.pytorch_b200.dsp.models import instance_kernel, sparse_MF_SP
    from tgp.pytorch_b200.dsp.models.flow import instance_flow
    from tgp.pytorch_b200.dsp.likelihoods import MulticlassCategorical
    g = MulticlassGolden('mc_synth_c3_sal1_p1')
    meta = g.meta
    Cn, M = meta['C'], meta['M']
    X = g.t('X')
    cg.quad_points = meta['S']
    K = instance_kernel('scale_rbf', ard_num_dim=X.shape[1], num_multioutput=Cn, kernel_is_shared=False)
    flows = [instance_flow(F.SAL(1)) for _ in range(Cn)]
    model = sparse_MF_SP(['zero', K], X, X[:M].clone(), meta['N'], MulticlassCategorical(Cn), Cn, False, False, False, False,
                         False, flows, 'single', 0.0, False)
    own = dict(model.named_parameters())
    with torch.no_grad():
        for n in meta['param_names']:
            own[n].copy_(torch.tensor(np.asarray(g.z['param:' + n]), dtype=torch.float64).reshape(own[n].shape))
    model = model.to(DEV)
    old = cg.compute
    cg.compute = compute
    try:
        model.likelihood.mc_noise = g.t('eps').to(DEV)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            ELBO, ELL, KLD = model.ELBO(X.to(DEV), torch.tensor(np.asarray(g.z['Y'])).to(DEV))
            (-ELBO).backward()
    finally:
        cg.compute = old
        model.likelihood.mc_noise = None
    plist = g.plist()
    for p in plist:
        for k in ('Z', 'raw_lengthscale', 'raw_outputscale', 'm', 'L_raw'):
            p[k].requires_grad_(True)
    E, ELL_o, KLD_o, _, _, _ = UR.elbo_multiclass(X, g.t('Y').reshape(-1), plist, meta['N'], g.t('eps'))
    E.backward()
    errs = {'ELBO': rel_err(ELBO.detach().cpu(), E.detach()), 'ELL': rel_err(ELL.detach().cpu(), ELL_o.detach()),
            'KLD': rel_err(KLD.detach().cpu(), KLD_o.detach())}
    names = {'Z': 'Z', 'raw_lengthscale': 'covariance_function.base_kernel.raw_lengthscale',
             'raw_outputscale': 'covariance_function.raw_outputscale', 'm': 'q_U.variational_mean',
             'L_raw': 'q_U.chol_variational_covar'}
    for k, n in names.items():
        got = -own[n].grad.detach().cpu()
        ref = torch.stack([p[k].grad.reshape(got[c].shape) for c, p in enumerate(plist)])
        errs[k] = rel_err(got, ref)
    bad = {k: e for k, e in errs.items() if not e < 1e-10}
    assert not bad, (bad, errs)
