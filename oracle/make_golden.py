"""Generate `tests/golden/*.npz` by running the UNMODIFIED reference under `oracle/ref_shims` (O1).

Run where the original project is checked out (`TGP_REFERENCE_ROOT=<checkout> python oracle/make_golden.py`).
Each fixture stores the inputs, every parameter, a JSON description of the flow, and the reference's outputs:
ELBO / ELL / KLD, q(f) marginals, every gradient of ELBO, test log-likelihood and predictive moments.
`tests/test_oracle_golden.py` replays them through `oracle/tgp_oracle.py` (O2); `tests/test_gpu_parity.py`
replays them through the CUDA path.
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle.ref_loader import REFERENCE_ROOT, load_reference  # noqa: E402
from tests.golden_util import variational_grid  # noqa: E402

dsp = load_reference()
import dsp.config as cg  # noqa: E402
from dsp.models import instance_kernel, sparse_MF_SP, sparse_MF_GP  # noqa: E402
from dsp.models.flow import (instance_flow, AffineFlow, StepFlow, TanhFlow, Sinh_ArcsinhFlow,  # noqa: E402
                             IdentityFlow, CompositeFlow, ArcsinhFlow, BoxCoxFlow, InverseBoxCoxFlow)
from dsp.likelihoods import GaussianNonLinearMean, GaussianLinearMean, Bernoulli, MulticlassCategorical  # noqa: E402
from dsp.flows import (SAL, StepTanhL, ArcSL, BoxCoxL, InverseBoxCoxL, build_chain,  # noqa: E402
                       StepSAL, StepArcSL, StepBoxCoxL, StepInverseBoxCoxL, StepAllL)

OUT = os.path.join(os.path.dirname(HERE), 'tests', 'golden')
UCI = os.path.join(REFERENCE_ROOT or '', 'code', 'datasets', 'regression', 'uci')


def load_uci(name, seed=1):
    """Same preprocessing as reference data path (uci_datasets.py:72-97, data.py:260-299): split pickle,
    standardise X and Y with training statistics."""
    import pandas as pd
    import pickle
    arr = pd.read_csv(os.path.join(UCI, name + '.csv'), header=None).values.astype(np.float64)
    with open(os.path.join(UCI, 'splits_idx_%s.pkl' % name), 'rb') as fh:
        sp = pickle.load(fh)['seed_%d' % seed]
    tr, te = np.asarray(sp['train']), np.asarray(sp['test'])
    X, Y = arr[:, :-1], arr[:, -1:]
    Xtr, Ytr, Xte, Yte = X[tr], Y[tr], X[te], Y[te]
    xm, xs = Xtr.mean(0), Xtr.std(0)
    xs[xs == 0] = 1.0
    ym, ys = Ytr.mean(0), Ytr.std(0)
    f = lambda a: torch.tensor(a, dtype=torch.float64)  # noqa: E731
    return f((Xtr - xm) / xs), f((Ytr - ym) / ys), f((Xte - xm) / xs), f((Yte - ym) / ys), float(ys[0])


def build(kind, X, M, N, flow=None, likelihood=None, seed=0):
    torch.manual_seed(seed)
    np.random.seed(seed)
    Dx = X.shape[1]
    K = instance_kernel('scale_rbf', ard_num_dim=Dx, num_multioutput=1, kernel_is_shared=False,
                        init_params={'length_scale': 2.0, 'kernel_scale': 2.0, 'noisy_variance': 1e-6})
    Z = X[torch.randperm(X.shape[0])[:M]].clone()
    ip = {'variational_distribution': {'variance_scale': 1e-5, 'mean_scale': 0.0}}
    if kind == 'SVGP':
        lik = GaussianLinearMean(out_dim=1, noise_init=0.05, noise_is_shared=False)
        return sparse_MF_GP(['zero', K], X, Z, N, lik, 1, True, False, False, False, False, 0.0, ip)
    lik = likelihood or GaussianNonLinearMean(out_dim=1, noise_init=0.05, noise_is_shared=False,
                                              quadrature_points=cg.quad_points)
    return sparse_MF_SP(['zero', K], X, Z, N, lik, 1, True, False, False, False, False, [flow], 'single', 0.0,
                        False, ip)


def randomise(model, seed, nnet_scale=0.2):
    """P1 'mid-training' state (SURVEY.md §8d): nothing at its trivial initial value."""
    g = torch.Generator().manual_seed(seed)
    M = model.M
    with torch.no_grad():
        for n, prm in model.named_parameters():
            if n == 'Z':
                prm.add_(0.05 * torch.randn(prm.shape, generator=g))
            elif n.endswith('raw_lengthscale'):
                ls = 0.5 + 2.5 * torch.rand(prm.shape, generator=g)
                prm.copy_(ls + torch.log(-torch.expm1(-ls)))
            elif n.endswith('raw_outputscale'):
                s = torch.full(prm.shape, 1.5)
                prm.copy_(s + torch.log(-torch.expm1(-s)))
            elif n.endswith('variational_mean'):
                prm.copy_(torch.randn(prm.shape, generator=g))
            elif n.endswith('chol_variational_covar'):
                prm.copy_(0.5 * torch.eye(M).unsqueeze(0) + 0.05 * torch.randn(prm.shape, generator=g))
            elif n.endswith('log_var_noise'):
                prm.copy_(torch.log(torch.full(prm.shape, 0.2)))
            elif 'G_matrix' in n and 'NNets' not in n:
                prm.add_(0.3 * torch.randn(prm.shape, generator=g))
            elif 'NNets' in n:
                prm.add_(nnet_scale * torch.randn(prm.shape, generator=g))


def randomise_big(model, seed):
    """P1 state for the BASELINE-size fixtures.  Same distributions as `randomise`, except that the M x M variational
    factor is drawn from a 17-level grid (0.5 I + 0.05 * k/8, k in -8..8, strictly lower part only; the upper triangle,
    which the reference masks away at use, is zero); the fixture stores the grid's seed instead of the M x M parameter.
    Returns that seed."""
    randomise(model, seed)
    with torch.no_grad():
        model.q_U.chol_variational_covar.copy_(torch.from_numpy(variational_grid(model.M, seed + 1000)))
    return seed + 1000


def flow_to_spec(flow, store, X=None, prefix='fl'):
    """Walk a reference CompositeFlow and emit the oracle layer list (JSON-able; arrays go to `store`)."""
    spec = []
    idx = [0]

    def put(t):
        k = '%s_%d' % (prefix, idx[0])
        idx[0] += 1
        store[k] = t.detach().cpu().numpy().astype(np.float64)
        return k

    def member(sub):
        if isinstance(sub, TanhFlow):
            assert sub.set_restrictions and not sub.input_dependent
            assert not sub.add_init_f0
            return ['tanh_step', [[put(sub.a), put(sub.b), put(sub.c), put(sub.d)]], False]
        if isinstance(sub, ArcsinhFlow):
            return ['arcsinh', put(sub.a), put(sub.b), put(sub.c), put(sub.d), bool(sub.set_restrictions), bool(sub.add_init_f0)]
        if isinstance(sub, BoxCoxFlow):
            return ['invboxcox' if isinstance(sub, InverseBoxCoxFlow) else 'boxcox', put(sub.transform_param()),
                    bool(sub.add_init_f0)]
        if isinstance(sub, Sinh_ArcsinhFlow):
            assert not sub.input_dependent
            return ['sal', put(sub.a), put(sub.b), bool(sub.set_restrictions), bool(sub.add_init_f0)]
        raise NotImplementedError(type(sub))

    for fl in flow.flow_arr:
        if isinstance(fl, IdentityFlow):
            spec.append(['identity'])
        elif isinstance(fl, AffineFlow):
            spec.append(['affine', put(fl.a), put(fl.b), bool(fl.set_restrictions)])
        elif isinstance(fl, StepFlow) and all(isinstance(s, TanhFlow) for s in fl.flow_arr):
            steps = []
            for sw, sub in zip(fl.switch_off, fl.flow_arr):
                assert isinstance(sub, TanhFlow) and not sw.is_trainable and sub.set_restrictions
                assert not sub.add_init_f0 and not sub.input_dependent
                steps.append([put(sub.a), put(sub.b), put(sub.c), put(sub.d)])
            spec.append(['tanh_step', steps, bool(fl.add_init_f0)])
        elif isinstance(fl, StepFlow):               # general linear combination, members behind their switch_off
            members = [[member(sub), [put(sw.a), put(sw.b)] if sw.is_trainable else None]
                       for sw, sub in zip(fl.switch_off, fl.flow_arr)]
            spec.append(['step_group', members, bool(fl.add_init_f0)])
        elif isinstance(fl, ArcsinhFlow):
            spec.append(['arcsinh', put(fl.a), put(fl.b), put(fl.c), put(fl.d), bool(fl.set_restrictions), bool(fl.add_init_f0)])
        elif isinstance(fl, BoxCoxFlow):             # InverseBoxCoxFlow derives from it
            kind = 'invboxcox' if isinstance(fl, InverseBoxCoxFlow) else 'boxcox'
            spec.append([kind, put(fl.transform_param()), bool(fl.add_init_f0)])      # lam AFTER the constraint
        elif isinstance(fl, Sinh_ArcsinhFlow):
            if fl.input_dependent:
                a = fl.NNets_a(X).squeeze(-1)
                b = fl.NNets_b(X).squeeze(-1)
                spec.append(['sal', put(a), put(b), bool(fl.set_restrictions), bool(fl.add_init_f0)])
            else:
                spec.append(['sal', put(fl.a), put(fl.b), bool(fl.set_restrictions), bool(fl.add_init_f0)])
        else:
            raise NotImplementedError(type(fl))
    return spec


def dropout_off(model):
    for m in model.modules():
        if 'Dropout' in type(m).__name__:
            m.eval()


class DropoutTape:
    """MC-dropout with RECORDED masks.  While active, nn.Dropout.forward draws its keep-mask with torch.bernoulli from the
    global RNG (the distribution nn.Dropout uses: keep with probability 1 - p, scale by 1 / (1 - p)) and stores it
    ('record'), or re-applies the stored masks in call order ('replay').  The reference's code path is untouched: the
    dropout layers live in the pytorchlib stand-in (oracle/ref_shims/pytorchlib), whose source is unavailable offline."""

    def __init__(self):
        self.masks, self.mode, self.i = [], 'record', 0

    def __enter__(self):
        tape = self
        self._orig = torch.nn.Dropout.forward

        def fwd(mod, x):
            if not mod.training:
                return x
            if tape.mode == 'record':
                mask = torch.bernoulli(torch.full_like(x, 1.0 - mod.p))
                tape.masks.append(mask.to(torch.uint8))
            else:
                mask = tape.masks[tape.i].to(x.dtype)
                tape.i += 1
            return x * mask / (1.0 - mod.p)
        torch.nn.Dropout.forward = fwd
        return self

    def __exit__(self, *exc):
        torch.nn.Dropout.forward = self._orig

    def replay(self):
        self.mode, self.i = 'replay', 0


ONLY = set(sys.argv[1:])      # optional fixture names: write only these (the others are left untouched on disk)


def projection_basis(M, k=6):
    """Deterministic (M, k) matrix of exact dyadic rationals (integer hash / 1024 - 0.5): bit-identical on every host."""
    i = np.arange(M, dtype=np.int64)[:, None]
    c = np.arange(k, dtype=np.int64)[None, :]
    return (((i * 2654435761 + (c + 1) * 40503 + i * c * 97) % 1024).astype(np.float64) / 1024.0) - 0.5


def record(name, model, X, Y, Xte, Yte, y_std, likelihood, id_flow=False, extra=None, big=False, tape=None, grid_seed=None):
    """big=True (fixtures at the BASELINE sizes M = 1024 / 2048): the M x M gradient of chol_variational_covar is stored
    as checksums — G R, G^T R for the fixed basis R above, its diagonal and Frobenius norm — instead of 8-32 MB of
    incompressible doubles, and the parameter itself as the seed `grid_seed` of randomise_big plus its SHA-256
    (tests/golden_util regenerates it)."""
    if ONLY and name not in ONLY:
        return
    store = {}
    model.set_is_training(True)
    for prm in model.parameters():
        prm.grad = None
    E, ELL, KLD = model.ELBO(X, Y)
    E.backward()
    store['X'], store['Y'] = X.numpy(), Y.numpy()
    store['Xte'], store['Yte'] = Xte.numpy(), Yte.numpy()
    store['ELBO'], store['ELL'], store['KLD'] = E.item(), ELL.item(), KLD.item()
    names = []
    for n, prm in model.named_parameters():
        if big and n.endswith('chol_variational_covar'):
            p = prm.detach().numpy()
            assert np.array_equal(p, variational_grid(p.shape[1], grid_seed))
            store['paramgrid:' + n] = np.array([grid_seed, p.shape[1]], dtype=np.int64)
            store['paramsha256:' + n] = np.array(hashlib.sha256(np.ascontiguousarray(p).tobytes()).hexdigest())
        else:
            store['param:' + n] = prm.detach().numpy().copy()
        gr = (torch.zeros_like(prm) if prm.grad is None else prm.grad).numpy().copy()
        if big and n.endswith('chol_variational_covar'):
            G = gr[0]
            R = projection_basis(G.shape[0])
            store['gradproj:' + n] = np.stack([G @ R, G.T @ R])
            store['graddiag:' + n] = np.diag(G).copy()
            store['gradnorm:' + n] = np.linalg.norm(G)
        else:
            store['grad:' + n] = gr
        names.append(n)
    with torch.no_grad():
        mu, v = model.marginal_variational_qf_parameters(X, diagonal=True, is_duvenaud=False)
        store['mu'], store['v'] = mu.view(-1).numpy(), v.view(-1).numpy()
        flow = model.G_matrix[0]
        comp = flow if isinstance(flow, CompositeFlow) else CompositeFlow([flow])
        if tape is not None:
            # dropout ON: the per-row flow parameters of the training batch are those of the recorded masks (replayed);
            # masks are stored per input-dependent layer as (n_nets, n_hidden_layers, rows, hidden) in evaluation order
            # (reference flow.py:949-950: NNets_a then NNets_b, hidden layers front to back)
            tape.replay()
            spec_tr = flow_to_spec(comp, store, X, 'fl')
            assert tape.i == len(tape.masks)
            id_layers = [i for i, fl in enumerate(comp.flow_arr) if isinstance(fl, Sinh_ArcsinhFlow) and fl.input_dependent]
            per = len(tape.masks) // len(id_layers)
            for j, li in enumerate(id_layers):
                mk = torch.stack(tape.masks[j * per:(j + 1) * per])              # (2 * L, rows, hidden)
                store['dropmask:%d' % li] = mk.view(2, per // 2, mk.shape[1], mk.shape[2]).numpy()
            dropout_off(model)                # the test side of the fixture is the point-estimate (dropout off) path
        else:
            spec_tr = flow_to_spec(comp, store, X, 'fl')
        spec_te = flow_to_spec(comp, store, Xte, 'flte')
    model.set_is_training(False)
    lp, mom = model.test_log_likelihood(Xte, Yte if likelihood != 'bernoulli' else Yte.long(),
                                        return_moments=True, Y_std=torch.ones(1) * y_std, S_MC_NNet=None)
    store['test_logp'] = float(lp.sum())
    for i, mm in enumerate(mom):
        if mm is not None:
            store['test_moment%d' % i] = mm.detach().double().numpy().reshape(-1) if likelihood != 'bernoulli' \
                else mm.detach().double().numpy()
    model.set_is_training(True)
    meta = {'name': name, 'likelihood': likelihood, 'N': float(model.N), 'M': int(model.M), 'y_std': y_std,
            'n_quad': int(cg.quad_points), 'flow_train': spec_tr, 'flow_test': spec_te, 'param_names': names,
            'id_flow': id_flow, 'dtype': 'float64', 'big': bool(big), 'dropout': tape is not None}
    if extra:
        meta.update(extra)
    store['meta'] = np.array(json.dumps(meta))
    np.savez_compressed(os.path.join(OUT, name + '.npz'), **store)
    print('%-34s ELBO % .12e  ELL % .12e  KLD % .12e  test_logp % .12e' % (name, store['ELBO'], store['ELL'],
                                                                          store['KLD'], store['test_logp']))


def synthetic_regression(n, d, seed):
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(n, d, generator=g)
    w = torch.randn(d, generator=g)
    y = torch.sinh(0.7 * (X @ w) / d ** 0.5) + 0.1 * torch.randn(n, generator=g)
    y = (y - y.mean()) / y.std()
    return X, y.view(-1, 1)


def synthetic_classification(n, d, seed):
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(n, d, generator=g)
    w = torch.randn(d, generator=g)
    pr = 0.5 * (1 + torch.erf((X @ w) / d ** 0.5 / 2 ** 0.5))
    y = (pr > torch.rand(n, generator=g)).double()
    return X, y.view(-1, 1)


def main():
    os.makedirs(OUT, exist_ok=True)
    Xb, Yb, Xbt, Ybt, ysb = load_uci('boston')
    Xp, Yp, Xpt, Ypt, ysp = load_uci('power')
    print('boston', tuple(Xb.shape), tuple(Xbt.shape), 'power', tuple(Xp.shape), tuple(Xpt.shape))
    Nb, Np = Xb.shape[0], Xp.shape[0]

    # cfg1: SVGP boston, init (P0) and mid-training (P1)
    m = build('SVGP', Xb, 100, Nb)
    record('boston_svgp_p0', m, Xb, Yb, Xbt, Ybt, ysb, 'gauss_linear')
    randomise(m, 11)
    record('boston_svgp_p1', m, Xb, Yb, Xbt, Ybt, ysb, 'gauss_linear')

    # identity-flow KAT: TGP with SAL(2) at init == SVGP closed form (SURVEY.md §4)
    m = build('TGP', Xb, 100, Nb, SAL(2))
    record('boston_tgp_sal2_p0', m, Xb, Yb, Xbt, Ybt, ysb, 'gauss_nonlinear')
    randomise(m, 12)
    record('boston_tgp_sal2_p1', m, Xb, Yb, Xbt, Ybt, ysb, 'gauss_nonlinear')

    # cfg2: TGP StepTanhL(1,3); and the shipped boston architecture StepTanhL(10,2) (exp_config.py:31-41)
    torch.manual_seed(3); np.random.seed(3)  # noqa: E702
    m = build('TGP', Xb, 100, Nb, StepTanhL(1, 3, add_f0=True), seed=3)
    randomise(m, 13)
    record('boston_tgp_steptanh13_p1', m, Xb, Yb, Xbt, Ybt, ysb, 'gauss_nonlinear')
    m = build('TGP', Xb, 100, Nb, StepTanhL(10, 2, add_f0=True), seed=4)
    randomise(m, 14)
    record('boston_tgp_steptanh102_p1', m, Xb, Yb, Xbt, Ybt, ysb, 'gauss_nonlinear')

    # power: shipped TGP architecture SAL(2) (exp_config.py:45-55), first 2048 training rows as the minibatch
    m = build('TGP', Xp, 100, Np, SAL(2), seed=5)
    randomise(m, 15)
    record('power_tgp_sal2_p1', m, Xp[:2048], Yp[:2048], Xpt[:256], Ypt[:256], ysp, 'gauss_nonlinear')

    # cfg3: ID_TGP.  boston SAL(1)+MLP(13->25->1,tanh,p=.5); power SAL(3)+MLP(4->50->50->1,relu,p=.25)
    for tag, (X, Y, Xt, Yt, ys), nb, cfgd, sd in (
            ('boston', (Xb, Yb, Xbt, Ybt, ysb), 1,
             dict(hidden_activation='tanh', num_hidden_layers=1, dropout=0.5, batch_norm=0, hidden_dim=25), 6),
            ('power', (Xp[:1024], Yp[:1024], Xpt[:128], Ypt[:128], ysp), 3,
             dict(hidden_activation='relu', num_hidden_layers=2, dropout=0.25, batch_norm=0, hidden_dim=50), 7)):
        spec = SAL(nb, input_dependent=True, input_dim=X.shape[1], inference='MC_dropout', **cfgd)
        torch.manual_seed(sd); np.random.seed(sd)  # noqa: E702
        fl = instance_flow(spec)
        fl.turn_off_initializer_parameters()
        m = build('TGP', X, 100, float(X.shape[0]), fl, seed=sd)
        randomise(m, 20 + sd)
        dropout_off(m)     # deterministic MLP (dropout masks come from the global RNG; see SURVEY.md §7.7)
        record('%s_idtgp_nodrop_p1' % tag, m, X, Y, Xt, Yt, ys, 'gauss_nonlinear', id_flow=True)

    # cfg4-like, small: D=8, M=64, StepTanhL(1,3)
    Xs, Ys = synthetic_regression(768, 8, 1234)
    m = build('TGP', Xs[:512], 64, 5000.0, StepTanhL(1, 3, add_f0=True), seed=8)
    randomise(m, 18)
    record('synth_reg_d8_m64_p1', m, Xs[:512], Ys[:512], Xs[512:], Ys[512:], 1.7, 'gauss_nonlinear')

    # cfg5-like, small: Bernoulli, D=16, M=48, SAL(1)
    Xc, Yc = synthetic_classification(640, 16, 4321)
    cg.quad_points = 100
    m = build('TGP', Xc[:512], 48, 3000.0, SAL(1), likelihood=Bernoulli(), seed=9)
    randomise(m, 19)
    record('synth_clf_d16_m48_p1', m, Xc[:512], Yc[:512], Xc[512:], Yc[512:], 1.0, 'bernoulli')

    # jitter ladder: duplicated inducing rows make K_zz singular -> reference adds 1e-8 (utils.py:256-268)
    m = build('SVGP', Xb, 40, Nb, seed=10)
    randomise(m, 21)
    with torch.no_grad():
        m.Z[0, 1] = m.Z[0, 0]
        m.Z[0, 3] = m.Z[0, 2]
    record('boston_svgp_jitter', m, Xb[:128], Yb[:128], Xbt, Ybt, ysb, 'gauss_linear', extra={'expects_jitter': True})

    # the largest StepTanhL architecture of the reference's launch scripts (bash_scripts/launch_test_uci_medium-small_
    # regression.sh, 'energy': 15 blocks x 4 steps = 270 flow scalars), on the boston split
    m = build('TGP', Xb, 100, Nb, StepTanhL(15, 4, add_f0=True), seed=22)
    randomise(m, 32)
    record('boston_tgp_steptanh154_p1', m, Xb, Yb, Xbt, Ybt, ysb, 'gauss_nonlinear')


def main_dropout():
    """cfg3 in TRAINING mode: ID_TGP with MC-dropout ACTIVE (nn.Module.training stays True in the reference's training loop,
    sparse_MF_SP.py:133-134), masks recorded so that another implementation can be fed the same ones."""
    Xb, Yb, Xbt, Ybt, ysb = load_uci('boston')
    Xp, Yp, Xpt, Ypt, ysp = load_uci('power')
    for tag, (X, Y, Xt, Yt, ys), nb, cfgd, sd in (
            ('boston', (Xb, Yb, Xbt, Ybt, ysb), 1,
             dict(hidden_activation='tanh', num_hidden_layers=1, dropout=0.5, batch_norm=0, hidden_dim=25), 6),
            ('power', (Xp[:1024], Yp[:1024], Xpt[:128], Ypt[:128], ysp), 3,
             dict(hidden_activation='relu', num_hidden_layers=2, dropout=0.25, batch_norm=0, hidden_dim=50), 7)):
        spec = SAL(nb, input_dependent=True, input_dim=X.shape[1], inference='MC_dropout', **cfgd)
        torch.manual_seed(sd); np.random.seed(sd)  # noqa: E702
        fl = instance_flow(spec)
        fl.turn_off_initializer_parameters()
        m = build('TGP', X, 100, float(X.shape[0]), fl, seed=sd)
        # three composed sinh-arcsinh blocks with 1 / (1 - p)-scaled hidden units overflow to ~1e21 with the 0.2 weight
        # noise of the dropout-off fixtures; 0.05 keeps the ELBO at the magnitude of a training run
        randomise(m, 20 + sd, nnet_scale=0.2 if tag == 'boston' else 0.05)
        torch.manual_seed(100 + sd)
        with DropoutTape() as tape:
            record('%s_idtgp_drop_p1' % tag, m, X, Y, Xt, Yt, ys, 'gauss_nonlinear', id_flow=True, tape=tape)


def boxcox_constraint(lam):
    """The constraint of the reference's own Box-Cox chains (flows.py:542, n = 2): lam in (0.01, 2.01)."""
    return 2.0 * torch.sigmoid(lam) + 0.01


def main_flows():
    """SURVEY.md §8f rank 3: the remaining flow families of the reference's launch scripts — arcsinh, Box-Cox and inverse
    Box-Cox layers and the build_chain combinations (flows.py:71-109, 140-214; flow.py:377-446, 495-557)."""
    Xb, Yb, Xbt, Ybt, ysb = load_uci('boston')
    Nb = Xb.shape[0]
    cases = (('boston_tgp_arcsl2_p1', 'ArcSL:2', lambda: ArcSL(2), False, 50),
             ('boston_tgp_bcl1_p1', 'BoxCoxL:1:random', lambda: BoxCoxL(1, init_random=True), False, 51),
             ('boston_tgp_bcl_al_p1', 'build_chain:BCL_AL:1', lambda: build_chain('BCL_AL', 1, constraint=boxcox_constraint), True, 52),
             ('boston_tgp_sal_invbcl_p1', 'build_chain:SAL_InvBCL:1', lambda: build_chain('SAL_InvBCL', 1, constraint=boxcox_constraint), True, 53),
             ('boston_tgp_sal_al2_p1', 'build_chain:SAL_AL:2', lambda: build_chain('SAL_AL', 2), False, 54))
    for name, builder, make, constrained, sd in cases:
        torch.manual_seed(sd); np.random.seed(sd)  # noqa: E702
        m = build('TGP', Xb, 100, Nb, make(), seed=sd)
        g = torch.Generator().manual_seed(sd + 100)
        randomise(m, sd + 10)
        with torch.no_grad():
            # keep the Box-Cox exponents in their well-behaved range and the composed map gentle
            for n, prm in m.named_parameters():
                if n.endswith('.lam'):
                    prm.copy_((0.3 * torch.randn((), generator=g)).reshape(prm.shape) if constrained
                              else (1.0 + 0.15 * torch.randn((), generator=g)).reshape(prm.shape))
        record(name, m, Xb, Yb, Xbt, Ybt, ysb, 'gauss_nonlinear',
               extra={'flow_builder': builder, 'boxcox_constraint': constrained})


def main_steps():
    """The general step flows (flows.py:284-491): linear combinations of sinh-arcsinh / arcsinh / Box-Cox / inverse Box-Cox
    members, most of them behind a trainable switch_off (flow.py:1039-1149)."""
    Xb, Yb, Xbt, Ybt, ysb = load_uci('boston')
    Nb = Xb.shape[0]
    cases = (('boston_tgp_stepsal_p1', 'StepSAL:1:3', lambda: StepSAL(1, 3, add_f0=True), 60),
             ('boston_tgp_steparcsl_p1', 'StepArcSL:2:2', lambda: StepArcSL(2, 2), 61),
             ('boston_tgp_stepbcl_p1', 'StepBoxCoxL:1:2', lambda: StepBoxCoxL(1, 2), 62),
             ('boston_tgp_stepinvbcl_p1', 'StepInverseBoxCoxL:1:2', lambda: StepInverseBoxCoxL(1, 2, add_f0=True), 63),
             ('boston_tgp_stepall_p1', 'StepAllL:1', lambda: StepAllL(1), 64))
    for name, builder, make, sd in cases:
        torch.manual_seed(sd); np.random.seed(sd)  # noqa: E702
        m = build('TGP', Xb, 100, Nb, make(), seed=sd)
        g = torch.Generator().manual_seed(sd + 100)
        randomise(m, sd + 10)
        with torch.no_grad():
            for n, prm in m.named_parameters():
                if n.endswith('.lam'):               # unconstrained exponents near 1: the composed map stays gentle
                    prm.copy_((1.0 + 0.15 * torch.randn((), generator=g)).reshape(prm.shape))
        record(name, m, Xb, Yb, Xbt, Ybt, ysb, 'gauss_nonlinear', extra={'flow_builder': builder, 'boxcox_constraint': False})


def main_multiclass():
    """Softmax likelihood integrated by Monte Carlo, one GP per class (likelihoods/MulticlassCategorical.py:51-151,
    sparse_MF_SP.py:552-626 with out_dim = C).  The N(0,1) draws of td.Normal.rsample / .sample are reproduced from the seed set
    immediately before the call (both are `empty(shape).normal_()` on the default generator); tests/test_oracle_golden.py
    confirms them by re-evaluating the reference's numbers from these draws."""
    cases = (('mc_synth_c3_sal1_p1', 3, 5, 20, 96, 30, 'SAL:1', lambda: SAL(1), 70),
             ('mc_synth_c4_steptanh12_p1', 4, 6, 24, 80, 20, 'StepTanhL:1:2', lambda: StepTanhL(1, 2, add_f0=True), 71),
             ('mc_synth_c3_stepsal_p1', 3, 4, 16, 64, 16, 'StepSAL:1:2', lambda: StepSAL(1, 2, add_f0=True), 72))
    for name, C, D, M, MB, S, builder, make, sd in cases:
        if ONLY and name not in ONLY:
            continue
        torch.manual_seed(sd); np.random.seed(sd)  # noqa: E702
        g = torch.Generator().manual_seed(sd)
        X = torch.randn(MB + 32, D, generator=g, dtype=torch.float64)
        W = torch.randn(D, C, generator=g, dtype=torch.float64)
        Y = torch.argmax(X @ W + 0.5 * torch.randn(MB + 32, C, generator=g, dtype=torch.float64), dim=1, keepdim=True)
        cg.quad_points = S
        K = instance_kernel('scale_rbf', ard_num_dim=D, num_multioutput=C, kernel_is_shared=False,
                            init_params={'length_scale': 2.0, 'kernel_scale': 2.0, 'noisy_variance': 1e-6})
        ip = {'variational_distribution': {'variance_scale': 1e-5, 'mean_scale': 0.0}}
        flows = [instance_flow(make()) for _ in range(C)]
        m = sparse_MF_SP(['zero', K], X, X[:M].clone(), 5000., MulticlassCategorical(C), C, True, False, False, False, False,
                         flows, 'single', 0.0, False, ip)
        randomise(m, sd + 10)
        Xtr, Ytr, Xte, Yte = X[:MB], Y[:MB], X[MB:], Y[MB:]
        store = {'X': Xtr.numpy(), 'Y': Ytr.numpy(), 'Xte': Xte.numpy(), 'Yte': Yte.numpy()}
        m.set_is_training(True)
        torch.manual_seed(sd + 1)
        E, ELL, KLD = m.ELBO(Xtr, Ytr)
        E.backward()
        torch.manual_seed(sd + 1)
        store['eps'] = torch.empty(S, C, MB, dtype=torch.float64).normal_().numpy()
        store['ELBO'], store['ELL'], store['KLD'] = E.item(), ELL.item(), KLD.item()
        names = []
        for n, prm in m.named_parameters():
            store['param:' + n] = prm.detach().numpy().copy()
            store['grad:' + n] = (torch.zeros_like(prm) if prm.grad is None else prm.grad).numpy().copy()
            names.append(n)
        specs = []
        with torch.no_grad():
            mu, v = m.marginal_variational_qf_parameters(Xtr.repeat(C, 1, 1), diagonal=True, is_duvenaud=False)
            store['mu'], store['v'] = mu.squeeze(2).numpy(), v.squeeze(2).numpy()
            for c in range(C):
                specs.append(flow_to_spec(m.G_matrix[c], store, Xtr, 'fl%d' % c))
        m.set_is_training(False)
        torch.manual_seed(sd + 2)
        lp, mom = m.test_log_likelihood(Xte, Yte, return_moments=True, Y_std=torch.ones(1), S_MC_NNet=None)
        torch.manual_seed(sd + 2)
        store['eps_te'] = torch.empty(S, C, Xte.shape[0], dtype=torch.float64).normal_().numpy()
        store['test_logp'] = float(lp)
        store['test_probs'] = mom[0].detach().double().numpy()
        meta = {'name': name, 'likelihood': 'multiclass', 'C': C, 'S': S, 'N': float(m.N), 'M': M, 'flows': specs,
                'flow_builder': builder, 'param_names': names, 'dtype': 'float64'}
        store['meta'] = np.array(json.dumps(meta))
        np.savez_compressed(os.path.join(OUT, name + '.npz'), **store)
        print('%-34s ELBO % .12e  ELL % .12e  KLD % .12e  test_logp % .12e' % (name, store['ELBO'], store['ELL'], store['KLD'],
                                                                              store['test_logp']))


def main_big():
    """Fixtures at the BASELINE.json sizes (configs[3]: D=8, M=1024, StepTanhL(1,3); configs[4]: Bernoulli, D=16, M=2048,
    SAL(1)); row counts the CPU oracle replays in seconds.  Z = distinct data rows, as in bench.py."""
    Xs, Ys = synthetic_regression(2048 + 256, 8, 1234)
    m = build('TGP', Xs, 1024, 5.0e6, StepTanhL(1, 3, add_f0=True), seed=40)
    s = randomise_big(m, 41)
    record('synth_reg_d8_m1024_p1', m, Xs[:2048], Ys[:2048], Xs[2048:], Ys[2048:], 1.3, 'gauss_nonlinear', big=True,
           grid_seed=s)
    Xc, Yc = synthetic_classification(4096, 16, 4321)
    cg.quad_points = 100
    m = build('TGP', Xc, 2048, 1.0e6, SAL(1), likelihood=Bernoulli(), seed=42)
    s = randomise_big(m, 43)
    record('synth_clf_d16_m2048_p1', m, Xc[:1024], Yc[:1024], Xc[1024:1152], Yc[1024:1152], 1.0, 'bernoulli', big=True,
           grid_seed=s)


if __name__ == '__main__':
    if 'BIG' in ONLY:
        ONLY.discard('BIG')
        main_big()
    elif 'MULTICLASS' in ONLY:
        ONLY.discard('MULTICLASS')
        main_multiclass()
    elif 'STEPS' in ONLY:
        ONLY.discard('STEPS')
        main_steps()
    elif 'FLOWS' in ONLY:
        ONLY.discard('FLOWS')
        main_flows()
    elif 'DROPOUT' in ONLY:
        ONLY.discard('DROPOUT')
        main_dropout()
    else:
        main()
