"""ARD-Matern kernels (nu = 1/2, 3/2, 5/2) on the GPU against the CPU reference of tests/matern_ref.py (O2 with the kernel
selected by p['kernel']).

Every problem draws Z from rows of X, so that minibatch rows coincide with inducing points: the K_xz entries there are s,
and for nu = 1/2 such pairs follow the zero-contribution convention of the kernel gradients (DESIGN section 5).
"""
import pytest
import torch

from oracle import tgp_oracle as O
from tests import matern_ref as MR
from tests.golden_util import rel_err
from tests.gpu_util import engine_inputs, flow_layout_and_params

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
KINDS = ['matern12', 'matern32', 'matern52']
GRAD_KEYS = ('Z', 'raw_lengthscale', 'raw_outputscale', 'm', 'L_raw', 'log_var_noise')


def _problem(R, M, D, seed, kernel, lik='gauss_nonlinear'):
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    X = torch.randn(R, D, generator=g, dtype=f64)
    y = torch.randn(R, generator=g, dtype=f64)
    if lik == 'bernoulli':
        y = (y > 0).to(f64)
    Z = X[torch.randperm(R, generator=g)[:M]].clone()                 # coincident points by construction
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
    return X, y, p


def _engine(p, lik, nq, compute):
    from tgp.pytorch_b200.engine import Engine, FlowLayout
    fl, theta, _, names = flow_layout_and_params(p['flow'], DEV)
    if lik == 'gauss_linear':
        fl, theta = FlowLayout([]), torch.zeros(0, dtype=torch.float64, device=DEV)
    eng = Engine(p['Z'].shape[0], p['Z'].shape[1], lik, nq, fl, DEV, compute=compute, kernel=p['kernel'])
    return eng, theta, names


def _cuda(X, y, p, N, lik, nq, compute, want_dx=False):
    """ELBO terms, rows, mu, v and every parameter gradient; with want_dx also out['X'] = dELBO/dX."""
    from tgp.pytorch_b200 import functional as Fn
    eng, theta, names = _engine(p, lik, nq, compute)
    ei = engine_inputs(p, DEV)
    leaves = [ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'], ei['log_var_noise'], theta]
    for t in leaves:
        t.requires_grad_(True)
    Xd = X.to(DEV).contiguous().requires_grad_(want_dx)
    ELL, KLD, rows, mu, v = Fn.elbo_terms(eng, Xd, y.to(DEV).contiguous(), N / X.shape[0], *leaves[:6], theta, None)
    (ELL - KLD).backward()
    out = dict(ELBO=(ELL - KLD).detach().cpu(), ELL=ELL.detach().cpu(), KLD=KLD.detach().cpu(), rows=rows.cpu(), mu=mu.cpu(),
               v=v.cpu())
    if want_dx:
        out['X'] = Xd.grad.detach().cpu()
    for k, t in zip(GRAD_KEYS, leaves):
        out[k] = (t.grad if t.grad is not None else torch.zeros_like(t)).detach().cpu().reshape(-1)
    for i, n in enumerate(names):
        out[n] = theta.grad[i].detach().cpu()
    if lik == 'bernoulli':
        out.pop('log_var_noise')
    return out, names


def _oracle(X, y, p, N, lik, nq):
    E, ELL, KLD, rows, gr = MR.elbo_and_grads(X, y, p, N, lik, nq)
    mu, v = MR.qf_marginals(X, p)
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
    """The FP64 parity bounds of the RBF path (tests/test_gpu_parity.py), including its Bernoulli bounds: the reference's
    Bernoulli ELL is formed by cancellation, which two faithful FP64 evaluations do not reproduce to 1e-10."""
    if lik == 'bernoulli':
        if k in ('ELBO', 'ELL', 'rows'):
            return e < dict(ELBO=5e-6, ELL=5e-6, rows=1e-4)[k]
        if k not in ('KLD', 'mu', 'v'):
            return e < 2e-6
    return e < dict(v=1e-9, KLD=1e-12).get(k, 1e-10)


@pytest.mark.parametrize('lik', ['gauss_nonlinear', 'gauss_linear', 'bernoulli'])
@pytest.mark.parametrize('kernel', KINDS)
@pytest.mark.parametrize('compute', ['f64', 'i8crt', 'tf32x3'])
def test_elbo_and_every_gradient_against_the_oracle(compute, kernel, lik):
    X, y, p = _problem(1000, 64, 8, seed=17 + KINDS.index(kernel), kernel=kernel, lik=lik)
    nq = 30 if lik != 'gauss_linear' else 0
    got, _ = _cuda(X, y, p, 5000.0, lik, nq, compute)
    ref = _oracle(X, y, p, 5000.0, lik, nq)
    errs = {k: rel_err(got[k], ref[k]) for k in got}
    if compute == 'tf32x3':      # yardstick of tests/test_gpu_tensorcore.py: O2's own FP32 evaluation against its FP64 one
        ref32 = _oracle(X.float(), y.float(), _to(p, torch.float32), 5000.0, lik, nq)
        bad = {k: (e, rel_err(ref32[k], ref[k])) for k, e in errs.items() if not e < 1e-5 + 4.0 * rel_err(ref32[k], ref[k])}
    else:
        bad = {k: e for k, e in errs.items() if not _ok(k, e, lik)}
    assert not bad, (bad, errs)


@pytest.mark.parametrize('R,M,D', [(4096, 1024, 8), (1000, 64, 40)])
@pytest.mark.parametrize('kernel', KINDS)
@pytest.mark.parametrize('compute', ['f64', 'i8crt'])
def test_full_size_and_wide_inputs(compute, kernel, R, M, D):
    """M = 1024 (the full M x M gradient of L_raw) and D = 40 ('i8crt' stages K_xz through FP64 for D > 32)."""
    X, y, p = _problem(R, M, D, seed=R + M + D, kernel=kernel)
    got, _ = _cuda(X, y, p, 10.0 * R, 'gauss_nonlinear', 20, compute)
    ref = _oracle(X, y, p, 10.0 * R, 'gauss_nonlinear', 20)
    errs = {k: rel_err(got[k], ref[k]) for k in got}
    bad = {k: e for k, e in errs.items() if not _ok(k, e, 'gauss_nonlinear')}
    assert not bad, (bad, errs)


@pytest.mark.parametrize('kernel', KINDS)
def test_test_log_likelihood_and_predictive_moments(kernel):
    from tgp.pytorch_b200 import functional as Fn
    X, y, p = _problem(700, 64, 8, seed=3, kernel=kernel)
    eng, theta, _ = _engine(p, 'gauss_nonlinear', 30, 'f64')
    ei = engine_inputs(p, DEV)
    Xd, yd = X.to(DEV).contiguous(), y.to(DEV).contiguous()
    with torch.no_grad():
        mu, v = Fn.qf_marginals(eng, Xd, ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'])
    eng.set_params(ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'], ei['log_var_noise'], theta)
    logp_rows, m1, m2 = eng.test_rows(mu, v, yd, None, 1, 1.7)
    lp, (m1_o, m2_o) = MR.log_likelihood_gauss_nonlinear(X, y, p, torch.tensor(1.7, dtype=torch.float64), 30)
    assert rel_err(logp_rows.sum().cpu() - 0.5 * X.shape[0] * torch.log(O.PI_F32), lp) < 1e-10
    assert rel_err(m1.cpu(), m1_o.detach()) < 1e-10
    assert rel_err(m2.cpu(), m2_o.detach()) < 1e-9


def test_model_api_with_a_shared_kernel_over_two_outputs():
    """instance_kernel('scale_matern') through an SVGP model with Dy = 2 and kernel_is_shared=True: the q(f) marginals of
    both outputs against O2, and a fused ELBO whose backward reaches the shared kernel's parameters."""
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    cg.device = DEV
    from tgp.pytorch_b200.dsp.models import instance_kernel, sparse_MF_GP
    from tgp.pytorch_b200.dsp.likelihoods import GaussianLinearMean
    K = instance_kernel('scale_matern', ard_num_dim=8, num_multioutput=2, kernel_is_shared=True,
                        init_params={'length_scale': 2.0, 'kernel_scale': 1.5, 'nu': 1.5})
    assert K.base_kernel.nu == 1.5 and K.batch_shape == torch.Size([1])
    X, _, p = _problem(600, 64, 8, seed=9, kernel='matern32', lik='gauss_linear')
    lik = GaussianLinearMean(out_dim=2, noise_init=0.3, noise_is_shared=False)
    ip = {'variational_distribution': {'variance_scale': 0.5, 'mean_scale': 0.3}}
    model = sparse_MF_GP(['zero', K], X, p['Z'], 6000, lik, 2, True, True, False, False, False, 0.0, ip).to(DEV)
    Xd = X.to(DEV)
    mean, cov = model.marginal_variational_qf_parameters(Xd, True, False)
    for dy in range(2):
        po = dict(Z=model.Z[0 if model.Z_is_shared else dy].detach().cpu().double(),
                  raw_lengthscale=K.base_kernel.raw_lengthscale[0, 0].detach().cpu().double(),
                  raw_outputscale=K.raw_outputscale[0].detach().cpu().double(),
                  m=model.q_U.variational_mean[dy].detach().cpu().double(),
                  L_raw=model.q_U.chol_variational_covar[dy].detach().cpu().double(), kernel='matern32')
        mu_o, v_o = MR.qf_marginals(X, po)
        assert rel_err(mean[dy, :, 0].detach().cpu().double(), mu_o) < 1e-10
        assert rel_err(cov[dy, :, 0].detach().cpu().double(), v_o) < 1e-9
    ELBO, _, _ = model.ELBO(Xd, torch.randn(600, 2, dtype=torch.float64, device=DEV))
    (-ELBO).backward()
    assert torch.isfinite(ELBO)
    for n in ('base_kernel.raw_lengthscale', 'raw_outputscale'):
        g = dict(K.named_parameters())[n].grad
        assert g is not None and torch.isfinite(g).all() and float(g.abs().max()) > 0, n


@pytest.mark.parametrize('compute', ['f64', 'i8crt'])
def test_multiclass_model_against_the_reference(compute):
    """C = 3 GPs with ScaleKernel(MaternKernel(nu = 3/2)) coupled by the Monte-Carlo softmax likelihood, through
    sparse_MF_SP with the parameters and noise draws of a multiclass fixture, against MR.elbo_multiclass."""
    import warnings
    import numpy as np
    from tests.golden_util import MulticlassGolden
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
    K = instance_kernel('scale_matern', ard_num_dim=X.shape[1], num_multioutput=Cn, kernel_is_shared=False,
                        init_params={'nu': 1.5})
    flows = [instance_flow(F.SAL(1)) for _ in range(Cn)]
    model = sparse_MF_SP(['zero', K], X, X[:M].clone(), meta['N'], MulticlassCategorical(Cn), Cn, True, False, False, False,
                         False, flows, 'single', 0.0, False)
    own = dict(model.named_parameters())
    assert list(own) == list(meta['param_names'])
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
        p['kernel'] = 'matern32'
        for k in ('Z', 'raw_lengthscale', 'raw_outputscale', 'm', 'L_raw'):
            p[k].requires_grad_(True)
    E, ELL_o, KLD_o, _, _, _ = MR.elbo_multiclass(X, g.t('Y').reshape(-1), plist, meta['N'], g.t('eps'))
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


def test_handle_api_matches_the_staged_entry_points():
    from tgp.pytorch_b200.session import ElboSession
    X, y, p = _problem(1000, 64, 8, seed=23, kernel='matern12')
    staged, names = _cuda(X, y, p, 5000.0, 'gauss_nonlinear', 30, 'f64')
    eng, theta, _ = _engine(p, 'gauss_nonlinear', 30, 'f64')
    ei = engine_inputs(p, DEV)
    ses = ElboSession(eng, 1000)
    args = (ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'], ei['log_var_noise'], theta)
    out = ses.forward(X.to(DEV).contiguous(), y.to(DEV).contiguous(), 5.0, *args)
    assert int(out['status'].item()) == 0
    assert rel_err((out['terms'][0] - out['terms'][1]).cpu(), staged['ELBO']) < 1e-12
    grads = ses.backward(torch.tensor([1.0, -1.0], dtype=torch.float64, device=DEV))
    for k, n in (('Z', 'Z'), ('raw_ls', 'raw_lengthscale'), ('raw_os', 'raw_outputscale'), ('m', 'm'), ('L_raw', 'L_raw')):
        assert rel_err(grads[k].cpu().reshape(-1), staged[n]) < 1e-12, k
    ses.close()
