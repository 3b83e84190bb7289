"""Input gradients dX on the GPU (k_input_grads, k_flow_mlp<true, true>) against the CPU reference of tests/input_grad_ref.py, and the
properties a caller relies on: the translation identity at M = 1024 / 2048, row-sharded halves, the handle API, the flow
MLPs of ID_TGP, several outputs and classes, float32 models, and that asking for dX changes no other gradient."""
import warnings

import numpy as np
import pytest
import torch

from tests import input_grad_ref as IR
from tests import unwhitened_ref as UR
from tests.golden_util import Golden, MulticlassGolden, rel_err
from tests.gpu_util import engine_inputs
from tests.model_util import build_from_golden, set_dropout_mode
from tests.test_gpu_matern import _engine, _ok, _problem, _to

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
KINDS = ['rbf', 'matern12', 'matern32', 'matern52']
PARAMS = ('Z', 'raw_ls', 'raw_os', 'm', 'L_raw', 'log_var_noise')


def _leaves(p, whiten):
    ei = engine_inputs(p, DEV)
    if not whiten:      # the non-whitened q(u) of the same q(f): same dX
        q, _ = UR.from_whitened(p)
        ei['m'], ei['L_raw'] = q['m'].to(DEV).contiguous(), q['L_raw'].to(DEV).contiguous()
    return ei


def _elbo_dx(X, y, p, N, lik, nq, compute, whiten=True, want_dx=True):
    """(X.grad or None, {param: grad}) of ELL - KLD through Fn.elbo_terms."""
    from tgp.pytorch_b200 import functional as Fn
    from tgp.pytorch_b200.engine import Engine
    eng0, theta, _ = _engine(p, lik, nq, compute)
    eng = Engine(eng0.M, eng0.D, lik, nq, eng0.flow, DEV, compute=compute, kernel=p['kernel'], whiten=whiten)
    ei = _leaves(p, whiten)
    leaves = [ei[k].requires_grad_(True) for k in PARAMS] + [theta.requires_grad_(True)]
    Xd = X.to(DEV).contiguous().requires_grad_(want_dx)
    ELL, KLD, _, _, _ = Fn.elbo_terms(eng, Xd, y.to(DEV).contiguous(), N / X.shape[0], *leaves, None)
    (ELL - KLD).backward()
    grads = {k: (t.grad.detach().clone() if t.grad is not None else None) for k, t in zip(PARAMS + ('theta',), leaves)}
    return (Xd.grad.detach().cpu() if want_dx else None), grads


@pytest.mark.parametrize('whiten', [True, False])
@pytest.mark.parametrize('lik', ['gauss_nonlinear', 'gauss_linear', 'bernoulli'])
@pytest.mark.parametrize('kernel', KINDS)
@pytest.mark.parametrize('compute', ['f64', 'i8crt', 'tf32x3'])
def test_elbo_dx_against_the_reference(compute, kernel, lik, whiten):
    X, y, p = _problem(1000, 64, 8, seed=31 + KINDS.index(kernel), kernel=kernel, lik=lik)
    nq = 30 if lik != 'gauss_linear' else 0
    got, _ = _elbo_dx(X, y, p, 5000.0, lik, nq, compute, whiten)
    _, ref, _ = IR.elbo_grads_xz(X, y, p, 5000.0, lik, nq)
    e = rel_err(got, ref)
    if compute == 'tf32x3':      # the bar of tests/test_gpu_matern.py: O2's own FP32 evaluation against its FP64 one
        _, ref32, _ = IR.elbo_grads_xz(X.float(), y.float(), _to(p, torch.float32), 5000.0, lik, nq)
        assert e < 1e-5 + 4.0 * rel_err(ref32, ref), (e, rel_err(ref32, ref))
    else:
        assert _ok('X', e, lik), e


@pytest.mark.parametrize('whiten', [True, False])
@pytest.mark.parametrize('kernel', KINDS)
@pytest.mark.parametrize('compute', ['f64', 'i8crt', 'tf32x3'])
def test_marginals_dx_against_the_reference(compute, kernel, whiten):
    from tgp.pytorch_b200 import functional as Fn
    from tgp.pytorch_b200.engine import Engine, FlowLayout
    X, _, p = _problem(900, 64, 8, seed=5 + KINDS.index(kernel), kernel=kernel)
    g = torch.Generator().manual_seed(7)
    w_mu, w_v = torch.randn(900, generator=g, dtype=torch.float64), torch.randn(900, generator=g, dtype=torch.float64)
    eng = Engine(64, 8, 'gauss_linear', 0, FlowLayout([]), DEV, compute=compute, kernel=kernel, whiten=whiten)
    ei = _leaves(p, whiten)
    Xd = X.to(DEV).contiguous().requires_grad_(True)
    mu, v = Fn.qf_marginals(eng, Xd, ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'])
    ((mu * w_mu.to(DEV)).sum() + (v * w_v.to(DEV)).sum()).backward()
    ref = IR.marginals_grad_x(X, p, w_mu, w_v)
    e = rel_err(Xd.grad.cpu(), ref)
    if compute == 'tf32x3':
        ref32 = IR.marginals_grad_x(X.float(), _to(p, torch.float32), w_mu.float(), w_v.float())
        assert e < 1e-5 + 4.0 * rel_err(ref32, ref), (e, rel_err(ref32, ref))
    else:
        assert e < 1e-10, e


def _model_grads(g, compute, X=None, Y=None):
    """(model, X.grad, {name: grad}) of -ELBO through the class API on fixture g."""
    from tgp.pytorch_b200.dsp import config as cg
    old = cg.compute
    cg.compute = compute
    try:
        model = build_from_golden(g, DEV)
        set_dropout_mode(model, g)
        Xd = (g.t('X') if X is None else X).to(DEV).requires_grad_(True)
        Yd = (g.t('Y') if Y is None else Y).to(DEV)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            ELBO, _, _ = model.ELBO(Xd, Yd)
            (-ELBO).backward()
    finally:
        cg.compute = old
    return model, Xd.grad.detach().cpu(), {n: t.grad.detach().cpu() for n, t in model.named_parameters() if t.grad is not None}


@pytest.mark.parametrize('compute', ['f64', 'i8crt', 'tf32x3'])
@pytest.mark.parametrize('name', ['synth_reg_d8_m1024_p1', 'synth_clf_d16_m2048_p1'])
def test_translation_identity_on_the_device(name, compute):
    """sum_n dE/dx_n + sum_j dE/dz_j = 0: no reference needed.  'f64' / 'i8crt' hold it to FP64 rounding; 'tf32x3' forms the
    Z gradient's K_xz share in FP32."""
    _, gx, gr = _model_grads(Golden(name), compute)
    gz = gr['Z'].reshape(-1, gx.shape[1])
    resid = float((gx.sum(0) + gz.sum(0)).norm())
    scale = float(gx.abs().sum(0).norm() + gz.abs().sum(0).norm())
    assert resid <= (1e-11 if compute != 'tf32x3' else 1e-5) * scale, (resid, scale)


@pytest.mark.parametrize('name', ['boston_idtgp_nodrop_p1', 'power_idtgp_nodrop_p1'])
def test_flow_mlp_dx_matches_the_torch_modules(name):
    """ID_TGP: the MLPs in the fused kernel (k_flow_mlp<true, true>) and as torch modules give the same dX.  (The module path draws
    its own dropout masks, so the recorded-mask case is checked on the MLPs alone, test_flow_mlp_dx_against_autograd.)"""
    from tgp.pytorch_b200.dsp import config as cg
    g = Golden(name)
    _, gx_kernel, _ = _model_grads(g, 'f64')
    old = cg.flow_mlp_in_kernel
    cg.flow_mlp_in_kernel = False
    try:
        _, gx_modules, _ = _model_grads(g, 'f64')
    finally:
        cg.flow_mlp_in_kernel = old
    assert float(gx_kernel.norm()) > 0.0
    assert rel_err(gx_kernel, gx_modules) < 1e-11


@pytest.mark.parametrize('name', ['boston_idtgp_drop_p1', 'power_idtgp_drop_p1'])
def test_idtgp_dx_with_recorded_masks_against_the_oracle(name):
    """ID_TGP through the class API with the reference's recorded dropout masks: X.grad against autograd of O2 in which every
    per-row flow parameter is the oracle MLP (O.flow_mlp with the same weights and masks) evaluated at X."""
    from oracle import tgp_oracle as O
    from tgp.pytorch_b200 import functional as Fn
    g = Golden(name)
    model, gx, _ = _model_grads(g, 'f64')
    p = g.oracle_params('train')
    X = g.t('X').requires_grad_(True)
    acts = {v: k.lower() for k, v in Fn._ACT_CODE.items()}
    n_row = 0
    for li, lay in enumerate(p['flow']):
        if lay[0] != 'sal' or lay[1].dim() == 0:
            continue
        layer = model.G_matrix[0].flow_arr[li]
        nets = layer._nets()
        spec = Fn.mlp_spec(nets)
        masks = layer.dropout_masks
        outs = []
        for ni, net in enumerate(nets):
            ws = [(b.forward_lin[0].weight.detach().cpu(), b.forward_lin[0].bias.detach().cpu()) for b in net]
            outs.append(O.flow_mlp(X, ws, acts[spec['act']], spec['p'], [masks[ni, l] for l in range(spec['L'])]))
        assert rel_err(outs[0].detach(), lay[1]) < 1e-12 and rel_err(outs[1].detach(), lay[2]) < 1e-12
        p['flow'][li] = (lay[0], outs[0], outs[1]) + tuple(lay[3:])
        n_row += 1
    assert n_row > 0
    E = O.elbo(X, g.t('Y').view(-1), p, g.meta['N'], g.meta['likelihood'], g.meta['n_quad'])[0]
    ref = torch.autograd.grad(E, X)[0]
    assert rel_err(-gx, ref) < 1e-10


def test_flow_mlp_dx_against_autograd():
    from tgp.pytorch_b200 import functional as Fn
    from tests.test_gpu_flow_mlp import _nets
    nets = _nets(3, 13, 40, 2, 'tanh', 0.25, seed=8)
    spec = Fn.mlp_spec(nets)
    g = torch.Generator().manual_seed(4)
    R = 333
    X = torch.randn(R, 13, generator=g, dtype=torch.float64).to(DEV)
    w = torch.randn(R, 3, generator=g, dtype=torch.float64).to(DEV)
    masks = (torch.rand(3, 2, R, 40, generator=g) > 0.25).to(torch.uint8)
    Xa = X.clone().requires_grad_(True)
    (Fn.flow_mlp(None, nets, spec, Xa, masks) * w).sum().backward()
    gw = [p.grad.clone() for net in nets for p in net.parameters()]
    for net in nets:
        net.zero_grad()
    (Fn.flow_mlp(None, nets, spec, X, masks) * w).sum().backward()      # without dX: the weights' gradients are unchanged
    for a, p in zip(gw, [p for net in nets for p in net.parameters()]):
        assert rel_err(a.cpu(), p.grad.cpu()) < 1e-12
    from oracle import tgp_oracle as O
    Xc = X.cpu().requires_grad_(True)
    ref = 0.0
    for ni, net in enumerate(nets):
        ws = [(b.forward_lin[0].weight.detach().cpu(), b.forward_lin[0].bias.detach().cpu()) for b in net]
        ref = ref + (O.flow_mlp(Xc, ws, 'tanh', 0.25, [masks[ni, l] for l in range(2)]) * w[:, ni].cpu()).sum()
    ref.backward()
    assert rel_err(Xa.grad.cpu(), Xc.grad) < 1e-12


def test_row_halves_give_the_rows_of_the_whole_batch():
    g = Golden('synth_reg_d8_m64_p1')
    X, Y = g.t('X'), g.t('Y')
    R = X.shape[0]
    h = R // 2
    model, gx, _ = _model_grads(g, 'f64')
    parts = []
    for sl in (slice(0, h), slice(h, R)):
        from tgp.pytorch_b200.dsp import config as cg
        m = build_from_golden(g, DEV)
        m.global_batch_rows = R
        Xd = X[sl].to(DEV).requires_grad_(True)
        old = cg.compute
        cg.compute = 'f64'
        try:
            ELBO, _, _ = m.ELBO(Xd, Y[sl].to(DEV))
            (-ELBO).backward()
        finally:
            cg.compute = old
        parts.append(Xd.grad.cpu())
    assert rel_err(torch.cat(parts), gx) < 1e-13


def test_handle_api_dx_equals_the_class_api():
    from tgp.pytorch_b200.session import ElboSession
    X, y, p = _problem(1000, 64, 8, seed=41, kernel='matern52')
    gx, _ = _elbo_dx(X, y, p, 5000.0, 'gauss_nonlinear', 30, 'i8crt')
    eng, theta, _ = _engine(p, 'gauss_nonlinear', 30, 'i8crt')
    ei = engine_inputs(p, DEV)
    ses = ElboSession(eng, 1000)
    ses.forward(X.to(DEV).contiguous(), y.to(DEV).contiguous(), 5.0, *[ei[k] for k in PARAMS], theta)
    out = ses.backward(torch.tensor([1.0, -1.0], dtype=torch.float64, device=DEV), input_grad=True)
    assert rel_err(out['X'].cpu(), gx) < 1e-13
    ses.close()


@pytest.mark.parametrize('compute', ['f64', 'i8crt', 'tf32x3'])
def test_other_gradients_do_not_change(compute):
    X, y, p = _problem(3000, 256, 8, seed=2, kernel='rbf')
    _, with_dx = _elbo_dx(X, y, p, 1e4, 'gauss_nonlinear', 20, compute, want_dx=True)
    _, without = _elbo_dx(X, y, p, 1e4, 'gauss_nonlinear', 20, compute, want_dx=False)
    errs = {k: rel_err(with_dx[k].cpu(), without[k].cpu()) for k in with_dx if with_dx[k] is not None}
    bad = {k: e for k, e in errs.items() if not e <= 1e-13}
    assert not bad, errs


def test_two_outputs_shared_x_and_a_float32_model():
    """Dy = 2 (each output its own GP) on one X: dX sums both outputs; a float32 model returns a float32 X.grad."""
    from tests.test_gpu_unwhitened import _params_of, _svgp
    X, _, p = _problem(600, 64, 8, seed=9, kernel='rbf', lik='gauss_linear')
    Y = torch.randn(600, 2, dtype=torch.float64)
    model = _svgp(2, X, p)
    Xd = X.to(DEV).requires_grad_(True)
    ELBO, _, _ = model.ELBO(Xd, Y.to(DEV))
    ELBO.backward()
    ref = 0.0
    for dy in range(2):
        po = _params_of(model, dy)
        lv = model.likelihood.log_var_noise[dy].detach().cpu().double().reshape(())
        po['log_var_noise'] = lv
        Xc = X.clone().requires_grad_(True)
        E = UR.elbo(Xc, Y[:, dy], po, 6000, 'gauss_linear', 0)[0]
        ref = ref + torch.autograd.grad(E, Xc)[0]
    assert rel_err(Xd.grad.cpu(), ref) < 1e-10
    # float32 model: the FP64 path runs on the float32 values, and X.grad comes back as float32
    model32 = model.float()
    X32 = X.float().to(DEV).requires_grad_(True)
    ELBO32, _, _ = model32.ELBO(X32, Y.float().to(DEV))
    ELBO32.backward()
    assert X32.grad.dtype == torch.float32
    ref32 = 0.0
    for dy in range(2):
        po = _params_of(model32, dy)
        po['log_var_noise'] = model32.likelihood.log_var_noise[dy].detach().cpu().double().reshape(())
        Xc = X.float().double().requires_grad_(True)
        E = UR.elbo(Xc, Y.float().double()[:, dy], po, 6000, 'gauss_linear', 0)[0]
        ref32 = ref32 + torch.autograd.grad(E, Xc)[0]
    assert rel_err(X32.grad.double().cpu(), ref32) < 1e-5      # the model's float32 outputs feed the backward


def test_multiclass_dx_against_the_reference():
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
    Xd = X.to(DEV).requires_grad_(True)
    try:
        model.likelihood.mc_noise = g.t('eps').to(DEV)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            ELBO, _, _ = model.ELBO(Xd, torch.tensor(np.asarray(g.z['Y'])).to(DEV))
            ELBO.backward()
    finally:
        model.likelihood.mc_noise = None
    Xc = X.clone().requires_grad_(True)
    E = UR.elbo_multiclass(Xc, g.t('Y').reshape(-1), g.plist(), meta['N'], g.t('eps'))[0]
    ref = torch.autograd.grad(E, Xc)[0]
    assert rel_err(Xd.grad.cpu(), ref) < 1e-10
