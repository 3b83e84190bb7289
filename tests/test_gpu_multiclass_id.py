"""Input-dependent flows under the Monte-Carlo softmax likelihood (multiclass ID-TGP) on the device: tgp_mc_softmax_rows_rowp
against tgp_mc_softmax_rows and against tests/mc_id_ref.py, and `sparse_MF_SP` with `MulticlassCategorical` and input-dependent
flows through the class API (ELBO, every named gradient, dX, the fully Bayesian predictive) against the same reference."""
import ctypes as C
import warnings

import numpy as np
import pytest
import torch

from oracle import tgp_oracle as O
from tests import mc_id_ref as R
from tests.golden_util import MulticlassGolden, multiclass_names, rel_err
from tests.gpu_util import flow_layout_and_params

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
TOL = 1e-10


# ---- kernel level --------------------------------------------------------------------------------------------------------
def _pack(flows):
    """C O2 layer lists whose parameters are () (global) or (R,) (per row) -> (FlowLayout, theta (C, n_theta) or None,
    rowp (C, R, n_rowp) or None, per class the global leaves and the per-row leaves in kernel order)."""
    from tgp.pytorch_b200.engine import FlowLayout
    desc, glob, rows = [], [[] for _ in flows], [[] for _ in flows]
    for i, lay in enumerate(flows[0]):
        if lay[0] in ('sal', 'affine'):
            per_row = lay[1].dim() > 0
            pars = [[f[i][1], f[i][2]] for f in flows]
            desc.append(dict(kind='sal', restrict=lay[3], add_f0=lay[4], per_row=per_row) if lay[0] == 'sal'
                        else dict(kind='affine', restrict=lay[3]))
        else:
            per_row = lay[1][0][0].dim() > 0
            pars = [[t for st in f[i][1] for t in st] for f in flows]
            desc.append(dict(kind='tanh_step', n_steps=len(lay[1]), add_f0=lay[2], per_row=per_row))
        for c in range(len(flows)):
            (rows if per_row else glob)[c].extend(pars[c])
    layout = FlowLayout(desc)
    theta = torch.stack([torch.stack([t.detach().reshape(()) for t in g]) for g in glob]) if glob[0] else None
    rowp = torch.stack([torch.stack([t.detach() for t in r], dim=-1) for r in rows]) if rows[0] else None
    return layout, theta, rowp, glob, rows


def _run(layout, mu, v, y, eps, theta, rowp, entry='rowp'):
    """One kernel call: rows, g_mu, g_v, dtheta, drowp, probs (CPU)."""
    from tgp.pytorch_b200 import _lib
    from tgp.pytorch_b200.dsp.likelihoods._rows import _mc_model
    lib = _lib.load()
    Cn, Rn = mu.shape
    d = dict(dtype=torch.float64, device=DEV)
    dev = lambda t: None if t is None else t.to(DEV).double().contiguous()        # noqa: E731
    mu_d, v_d, y_d, e_d, th, rp = dev(mu), dev(v), dev(y), dev(eps), dev(theta), dev(rowp)
    rows, g_mu, g_v, probs = torch.empty(Rn, **d), torch.empty(Cn, Rn, **d), torch.empty(Cn, Rn, **d), torch.empty(Rn, Cn, **d)
    dth = None if th is None else torch.zeros_like(th)
    drp = None if rp is None else torch.full_like(rp, float('nan'))              # written, not accumulated
    ptr = lambda t: None if t is None else t.data_ptr()                          # noqa: E731
    args = (_mc_model(layout), Cn, eps.shape[0], Rn, ptr(mu_d), ptr(v_d), ptr(y_d), ptr(e_d), ptr(th), 1, ptr(rows), ptr(g_mu),
            ptr(g_v), ptr(dth), ptr(probs))
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    if entry == 'rowp':
        _lib.check(lib.tgp_mc_softmax_rows_rowp(*args, ptr(rp), ptr(drp), st), 'tgp_mc_softmax_rows_rowp')
    else:
        _lib.check(lib.tgp_mc_softmax_rows(*args, st), 'tgp_mc_softmax_rows')
    torch.cuda.synchronize()
    cpu = lambda t: None if t is None else t.cpu()                               # noqa: E731
    return rows.cpu(), g_mu.cpu(), g_v.cpu(), cpu(dth), cpu(drp), probs.cpu()


@pytest.mark.parametrize('name', multiclass_names())
def test_rowp_entry_point_without_per_row_flows_equals_the_global_one(name):
    g = MulticlassGolden(name)
    packs = [flow_layout_and_params(p['flow'], DEV) for p in g.plist()]
    theta = torch.stack([p[1] for p in packs])
    args = (packs[0][0], g.t('mu'), g.t('v'), g.t('Y').reshape(-1), g.t('eps'), theta, None)
    new, old = _run(*args, entry='rowp'), _run(*args, entry='global')
    for i, what in enumerate(('rows', 'g_mu', 'g_v')):
        assert torch.equal(new[i], old[i]), what
    assert torch.equal(new[5], old[5]), 'probs'
    # dtheta: per-warp sums added with FP64 atomics, so the order of the additions (not the code) may differ between calls
    assert rel_err(new[3], old[3]) < 1e-14 and new[4] is None


def _rand_layers(kind, Rn, gen):
    """One class's flow with random per-row (Rn,) and global () raw parameters."""
    def pr(scale=0.5, shift=0.0):
        return shift + scale * torch.randn(Rn, generator=gen, dtype=torch.float64)

    def gl(scale=0.3, shift=0.0):
        return shift + scale * torch.randn((), generator=gen, dtype=torch.float64)
    aff = lambda: ('affine', gl(0.2, 1.0), gl(0.2), False)                          # noqa: E731
    sal_r = lambda res, f0: ('sal', pr(0.4), pr(0.3, 0.8 if not res else 0.5), res, f0)   # noqa: E731
    tanh_r = lambda n, f0: ('tanh_step', [(pr(0.5), pr(0.5), pr(0.8), pr(0.5)) for _ in range(n)], f0)   # noqa: E731
    if kind == 'id_sal1':
        return [sal_r(False, False), aff()]
    if kind == 'id_sal2':
        return [sal_r(False, False), aff(), sal_r(True, True), aff()]
    if kind == 'id_steptanh13':
        return [tanh_r(3, True), aff()]
    if kind == 'mixed':               # global layers before, between and after per-row ones: both accumulators, both p0 ranges
        return [('sal', gl(0.3), gl(0.2, 0.5), True, False), aff(), sal_r(True, True), tanh_r(2, True),
                ('tanh_step', [(gl(), gl(), gl(0.5), gl())], True), aff()]
    raise ValueError(kind)


@pytest.mark.parametrize('Rn', [1, 127, 128, 129, 4099])
@pytest.mark.parametrize('Cn', [3, 4])
@pytest.mark.parametrize('kind', ['id_sal1', 'id_sal2', 'id_steptanh13', 'mixed'])
def test_kernel_against_the_reference_with_random_per_row_parameters(kind, Cn, Rn):
    gen = torch.Generator().manual_seed(1000 * Cn + Rn)
    S = 12
    flows = [_rand_layers(kind, Rn, gen) for _ in range(Cn)]
    layout, theta, rowp, glob, rows_l = _pack(flows)
    assert layout.n_rowparams > 0 and layout.n_theta > 0
    mu = (0.7 * torch.randn(Cn, Rn, generator=gen, dtype=torch.float64)).requires_grad_(True)
    v = (0.05 + torch.rand(Cn, Rn, generator=gen, dtype=torch.float64)).requires_grad_(True)
    y = torch.randint(0, Cn, (Rn,), generator=gen).double()
    eps = torch.randn(S, Cn, Rn, generator=gen, dtype=torch.float64)
    leaves = [t for c in range(Cn) for t in glob[c] + rows_l[c]]
    for t in leaves:
        t.requires_grad_(True)
    ref_rows = O.ell_rows_mc_softmax(mu, v, y, flows, eps)
    gr = torch.autograd.grad(ref_rows.sum(), [mu, v] + leaves)
    rows, g_mu, g_v, dth, drp, probs = _run(layout, mu.detach(), v.detach(), y, eps, theta, rowp)
    k = 2
    ref_dth, ref_drp = [], []
    for c in range(Cn):
        ref_dth.append(torch.stack([t.reshape(()) for t in gr[k:k + len(glob[c])]]))
        k += len(glob[c])
        ref_drp.append(torch.stack(gr[k:k + len(rows_l[c])], dim=-1))
        k += len(rows_l[c])
    with torch.no_grad():
        ref_probs = O.probs_mc_softmax(mu, v, flows, eps)
    errs = {'rows': rel_err(rows, ref_rows.detach()), 'g_mu': rel_err(g_mu, gr[0]), 'g_v': rel_err(g_v, gr[1]),
            'dtheta': rel_err(dth, torch.stack(ref_dth)), 'drowp': rel_err(drp, torch.stack(ref_drp)),
            'probs': rel_err(probs, ref_probs)}
    assert all(e < TOL for e in errs.values()), errs


# ---- class API -------------------------------------------------------------------------------------------------------------
D, M, MB, S, H, NH = 5, 16, 300, 16, 8, 2


def _model(Cn, act, p_drop, flow='sal', whiten=True, seed=0, X=None, n_ind=M, N=4000):
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    cg.device = DEV
    from tgp.pytorch_b200.dsp import flows as F
    from tgp.pytorch_b200.dsp.models import instance_kernel, sparse_MF_SP
    from tgp.pytorch_b200.dsp.models.flow import instance_flow
    from tgp.pytorch_b200.dsp.likelihoods import MulticlassCategorical
    torch.manual_seed(seed)
    gen = torch.Generator().manual_seed(seed)
    if X is None:
        X = torch.randn(MB, D, generator=gen, dtype=torch.float64)
    Y = torch.randint(0, Cn, (X.shape[0], 1), generator=gen).double()
    K = instance_kernel('scale_rbf', ard_num_dim=X.shape[1], num_multioutput=Cn, kernel_is_shared=False,
                        init_params={'length_scale': 2.0, 'kernel_scale': 2.0, 'noisy_variance': 1e-6})
    idc = dict(input_dependent=True, input_dim=X.shape[1], hidden_dim=H, num_hidden_layers=NH, hidden_activation=act, dropout=p_drop,
               inference='MC_dropout', batch_norm=0)
    flows = []
    for _ in range(Cn):
        spec = F.SAL(1, **idc) if flow == 'sal' else F.StepTanhL(1, 2, add_f0=True, **idc)
        fl = instance_flow(spec)
        fl.turn_off_initializer_parameters()
        flows.append(fl)
    ip = {'variational_distribution': {'variance_scale': 1e-5, 'mean_scale': 0.0}}
    model = sparse_MF_SP(['zero', K], X, X[:n_ind].clone(), N, MulticlassCategorical(Cn), Cn, whiten, False, False, False, False,
                         flows, 'single', 0.0, False, ip)
    with torch.no_grad():
        model.q_U.variational_mean.copy_(0.5 * torch.randn(Cn, n_ind, generator=gen, dtype=torch.float64))
        L = 0.1 * torch.randn(Cn, n_ind, n_ind, generator=gen, dtype=torch.float64).tril(-1) + 0.6 * torch.eye(n_ind, dtype=torch.float64)
        model.q_U.chol_variational_covar.copy_(L)
        for c in range(Cn):
            model.G_matrix[c].flow_arr[-1].a.fill_(1.0 + 0.1 * c)
            model.G_matrix[c].flow_arr[-1].b.fill_(0.05 * c)
    return model.to(DEV), X, Y


def _net_weights(leaf, prefix):
    return [(leaf['%s.%d.forward_lin.0.weight' % (prefix, l)], leaf['%s.%d.forward_lin.0.bias' % (prefix, l)]) for l in range(NH + 1)]


def _split(masks, n):
    return None if masks is None else [[masks[k, l].cpu() for l in range(NH)] for k in range(n)]


def _ref_flows(model, leaf, masks_of):
    """The mc_id_ref layer lists of the model's class flows on the reference leaves (name -> CPU tensor)."""
    from tgp.pytorch_b200.dsp.models.flow import AffineFlow, Sinh_ArcsinhFlow, StepFlow
    out = []
    for c, G in enumerate(model.G_matrix):
        layers = []
        for i, fl in enumerate(G.flow_arr):
            pre = 'G_matrix.%d.flow_arr.%d' % (c, i)
            if isinstance(fl, AffineFlow):
                layers.append(('affine', leaf[pre + '.a'], leaf[pre + '.b'], fl.set_restrictions))
            elif isinstance(fl, Sinh_ArcsinhFlow):
                mk = _split(masks_of(fl), 2) or [None, None]
                a, b = (R.Net(_net_weights(leaf, pre + '.NNets_' + x), mk[k]) for k, x in enumerate('ab'))
                layers.append(('sal', a, b, fl.set_restrictions, fl.add_init_f0))
            elif isinstance(fl, StepFlow):
                steps = []
                for j, t in enumerate(fl.flow_arr):
                    mk = _split(masks_of(t), 4) or [None] * 4
                    steps.append(tuple(R.Net(_net_weights(leaf, '%s.flow_arr.%d.NNets_%s' % (pre, j, x)), mk[k])
                                       for k, x in enumerate('abcd')))
                layers.append(('tanh_step', steps, fl.add_init_f0))
        out.append(layers)
    return out


def _ref_plist(model, leaf, masks_of):
    flows = _ref_flows(model, leaf, masks_of)
    return [{'Z': leaf['Z'][c], 'raw_lengthscale': leaf['covariance_function.base_kernel.raw_lengthscale'][c].reshape(-1),
             'raw_outputscale': leaf['covariance_function.raw_outputscale'][c].reshape(()), 'm': leaf['q_U.variational_mean'][c],
             'L_raw': leaf['q_U.chol_variational_covar'][c], 'flow': flows[c]} for c in range(len(flows))]


def _leaves(model):
    return {n: p.detach().cpu().clone().requires_grad_(True) for n, p in model.named_parameters()}


def _id_layers(model):
    from tgp.pytorch_b200.dsp.models.flow import Sinh_ArcsinhFlow, TanhFlow
    return [m for m in model.modules() if isinstance(m, (Sinh_ArcsinhFlow, TanhFlow)) and m.input_dependent]


def _elbo(model, X, Y, eps):
    model.likelihood.mc_noise = eps.to(DEV)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        ELBO, ELL, KLD = model.ELBO(X, Y)
        (-ELBO).backward()
    return ELBO.detach().cpu()


@pytest.mark.parametrize('whiten', [True, False])
@pytest.mark.parametrize('dropout', ['off', 'explicit', 'philox'])
@pytest.mark.parametrize('act', ['tanh', 'relu'])
@pytest.mark.parametrize('Cn', [3, 4])
@pytest.mark.parametrize('compute', ['f64', 'i8crt'])
def test_model_elbo_and_every_named_gradient(compute, Cn, act, dropout, whiten):
    if not whiten and (compute, Cn, act, dropout) != ('f64', 3, 'tanh', 'explicit'):
        pytest.skip('the non-whitened q(u) runs once')
    from tgp.pytorch_b200.dsp import config as cg
    p_drop = 0.0 if dropout == 'off' else 0.3
    model, X, Y = _model(Cn, act, p_drop, whiten=whiten, seed=Cn)
    gen = torch.Generator().manual_seed(5)
    eps = torch.randn(S, Cn, MB, generator=gen, dtype=torch.float64)
    if dropout == 'explicit':
        for lay in _id_layers(model):
            lay.dropout_masks = (torch.rand(2, NH, MB, H, generator=gen) > p_drop).to(torch.uint8)
    old = cg.compute
    cg.compute = compute
    try:
        E = _elbo(model, X.to(DEV), Y.to(DEV), eps)
    finally:
        cg.compute = old
        model.likelihood.mc_noise = None
    masks_of = {'off': lambda fl: None, 'explicit': lambda fl: fl.dropout_masks, 'philox': lambda fl: fl.last_dropout_masks}[dropout]
    if dropout == 'philox':
        assert all(lay.last_dropout_masks is not None for lay in _id_layers(model))
    leaf = _leaves(model)
    E0 = R.elbo_multiclass(X, Y.reshape(-1), _ref_plist(model, leaf, masks_of), 4000, eps, act, p_drop, whiten=whiten)[0]
    grads = dict(zip(leaf, torch.autograd.grad(E0, list(leaf.values()))))
    errs = {'ELBO': rel_err(E, E0.detach())}
    for n, prm in model.named_parameters():
        errs[n] = rel_err(-prm.grad.cpu(), grads[n])
    assert any('NNets_a' in n for n in errs) and any('forward_lin.0.weight' in n for n in errs)
    bad = {k: e for k, e in errs.items() if not e < TOL}
    assert not bad, bad


ZERO_READOUT = ['mc_synth_c3_sal1_p1', 'mc_synth_c4_steptanh12_p1']


@pytest.mark.parametrize('compute', ['f64', 'i8crt'])
@pytest.mark.parametrize('name', ZERO_READOUT)
def test_zero_readout_model_reproduces_the_global_flow_fixture(name, compute):
    """Input-dependent flows whose read-out layers have zero weights and the fixture's flow scalars as biases: the fixture's
    ELBO, its GP gradients and, through the read-out biases, its flow-scalar gradients — with dropout on."""
    from tgp.pytorch_b200.dsp import config as cg
    g = MulticlassGolden(name)
    Cn = g.meta['C']
    X = g.t('X')
    model, _, _ = _model(Cn, 'tanh', 0.25, flow='sal' if 'sal' in name else 'steptanh', seed=3, X=X, n_ind=g.meta['M'],
                         N=g.meta['N'])
    own = dict(model.named_parameters())
    readout = {}
    with torch.no_grad():
        for n in g.meta['param_names']:
            val = torch.tensor(np.asarray(g.z['param:' + n]), dtype=torch.float64)
            if n in own:
                own[n].copy_(val.reshape(own[n].shape))
                continue
            head, x = n.rsplit('.', 1)                      # a flow scalar now computed by a net
            net = '%s.NNets_%s.%d.forward_lin.0' % (head, x, NH)
            own[net + '.weight'].zero_()
            own[net + '.bias'].copy_(val.reshape(1))
            readout[net + '.bias'] = n
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
    errs = {'ELBO': rel_err(ELBO.detach().cpu(), g.t('ELBO')), 'ELL': rel_err(ELL.detach().cpu(), g.t('ELL')),
            'KLD': rel_err(KLD.detach().cpu(), g.t('KLD'))}
    for n in g.meta['param_names']:
        if n in own:
            errs[n] = rel_err(-own[n].grad.cpu().reshape(-1), g.t('grad:' + n).reshape(-1))
    for b, n in readout.items():
        errs[n] = rel_err(-own[b].grad.cpu().reshape(-1), g.t('grad:' + n).reshape(-1))
    assert len(readout) > 0
    bad = {k: e for k, e in errs.items() if not e < TOL}
    assert not bad, bad


@pytest.mark.parametrize('flow', ['sal', 'steptanh'])
@pytest.mark.parametrize('compute', ['f64', 'i8crt'])
def test_input_gradient_through_the_marginals_and_the_mlps(compute, flow):
    from tgp.pytorch_b200.dsp import config as cg
    Cn = 3
    model, X, Y = _model(Cn, 'tanh', 0.3, flow=flow, seed=7)
    gen = torch.Generator().manual_seed(8)
    eps = torch.randn(S, Cn, MB, generator=gen, dtype=torch.float64)
    for lay in _id_layers(model):
        lay.dropout_masks = (torch.rand(2 if flow == 'sal' else 4, NH, MB, H, generator=gen) > 0.3).to(torch.uint8)
    Xd = X.to(DEV).clone().requires_grad_(True)
    old = cg.compute
    cg.compute = compute
    try:
        _elbo(model, Xd, Y.to(DEV), eps)
    finally:
        cg.compute = old
        model.likelihood.mc_noise = None
    leaf = _leaves(model)
    Xr = X.clone().requires_grad_(True)
    E0 = R.elbo_multiclass(Xr, Y.reshape(-1), _ref_plist(model, leaf, lambda fl: fl.dropout_masks), 4000, eps, 'tanh', 0.3)[0]
    gx, = torch.autograd.grad(E0, [Xr])
    assert rel_err(-Xd.grad.cpu(), gx) < TOL


@pytest.mark.parametrize('Cn', [3, 4])
def test_fully_bayesian_predictive_averages_the_dropout_replicas(Cn):
    k, MBte = 5, 64
    model, _, _ = _model(Cn, 'relu', 0.25, seed=11)
    gen = torch.Generator().manual_seed(12)
    Xte = torch.randn(MBte, D, generator=gen, dtype=torch.float64)
    Yte = torch.randint(0, Cn, (MBte,), generator=gen)
    eps = torch.randn(S, Cn, k * MBte, generator=gen, dtype=torch.float64)
    model.be_fully_bayesian(True)
    model.set_is_training(False)
    model.likelihood.mc_noise = eps.to(DEV)
    try:
        lp, (m_Y,) = model.test_log_likelihood(Xte.to(DEV), Yte.to(DEV), return_moments=True, Y_std=torch.ones(1, device=DEV),
                                               S_MC_NNet=k)
    finally:
        model.likelihood.mc_noise = None
    masks = [lay.last_dropout_masks for lay in _id_layers(model)]
    assert all(m is not None and m.shape[2] == k * MBte for m in masks)
    leaf = _leaves(model)
    plist = _ref_plist(model, leaf, lambda fl: fl.last_dropout_masks)
    with torch.no_grad():
        mv = [O.qf_marginals(Xte, p) for p in plist]
        mu, v = torch.stack([a for a, _ in mv]), torch.stack([b for _, b in mv])
        P = R.probs(mu.repeat(1, k), v.repeat(1, k), [p['flow'] for p in plist], Xte.repeat(k, 1), eps, 'relu', 0.25)
        P = P.view(k, MBte, Cn).mean(0)
    assert rel_err(m_Y.cpu().double(), P) < TOL
    nll = -torch.log(P.float().gather(1, Yte.view(-1, 1))).mean()
    assert abs(float(lp) + float(nll * MBte)) < 1e-5 * abs(float(nll * MBte))
