"""Drop-in checks against the UNMODIFIED reference (needs TGP_REFERENCE_ROOT = a checkout of the original TGP.pytorch).

1. Every name the reference's main.py / exp_utils.py import from the hot-path modules (main.py:26-37, exp_utils.py:7-8) exists
   in tgp.pytorch_b200.dsp with the same call signature; so do the methods the reference's trainer calls on the model.
2. INTEGRATION.md path A in practice: the reference's OWN initialisers (dsp/initializers/initializers.py:29-182, unchanged
   code) are run on OUR flow modules — same seeds, CPU — and must follow the loss trajectory they produce on the
   reference's flow modules.  (The ELBO itself cannot run here: the product has no CPU path and this container no GPU.)
"""
import inspect

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.needs_reference


def _ref():
    from oracle.ref_loader import load_reference
    return load_reference()


def _sig(fn):
    return [(p.name, p.kind, p.default if p.default is inspect._empty or isinstance(p.default, (int, float, bool, str, type(None))) else 'obj')
            for p in inspect.signature(fn).parameters.values()]


def test_public_names_and_signatures_match_the_reference():
    _ref()
    import dsp.models as rm, dsp.models.flow as rf, dsp.likelihoods as rl, dsp.flows as rfl, dsp.utils as ru   # noqa: E401
    from tgp.pytorch_b200.dsp import models as om, likelihoods as ol, flows as ofl, utils as ou
    from tgp.pytorch_b200.dsp.models import flow as of
    pairs = [(rm.instance_kernel, om.instance_kernel), (rm.sparse_MF_SP.__init__, om.sparse_MF_SP.__init__),
             (rm.sparse_MF_GP.__init__, om.sparse_MF_GP.__init__), (rf.instance_flow, of.instance_flow),
             (rl.GaussianNonLinearMean.__init__, ol.GaussianNonLinearMean.__init__),
             (rl.GaussianLinearMean.__init__, ol.GaussianLinearMean.__init__), (rl.Bernoulli.__init__, ol.Bernoulli.__init__),
             (rl.MulticlassCategorical.__init__, ol.MulticlassCategorical.__init__),
             (rfl.SAL, ofl.SAL), (rfl.StepTanhL, ofl.StepTanhL), (ru.KMEANS, ou.KMEANS),
             (rfl.BoxCoxL, ofl.BoxCoxL), (rfl.InverseBoxCoxL, ofl.InverseBoxCoxL), (rfl.ArcSL, ofl.ArcSL),
             (rfl.build_chain, ofl.build_chain), (rfl.StepSAL, ofl.StepSAL), (rfl.StepArcSL, ofl.StepArcSL),
             (rfl.StepBoxCoxL, ofl.StepBoxCoxL), (rfl.StepInverseBoxCoxL, ofl.StepInverseBoxCoxL), (rfl.StepAllL, ofl.StepAllL)]
    for meth in ('ELBO', 'KLD', 'ELL', 'marginal_variational_qf_parameters', 'predictive_distribution', 'test_log_likelihood',
                 'sample_from_predictive_distribution', 'sample_from_variational_marginal', 'be_fully_bayesian', 'set_is_training'):
        pairs.append((getattr(rm.sparse_MF_SP, meth), getattr(om.sparse_MF_SP, meth)))
    for cls in ('AffineFlow', 'TanhFlow', 'Sinh_ArcsinhFlow', 'StepFlow', 'CompositeFlow', 'IdentityFlow', 'ArcsinhFlow', 'BoxCoxFlow',
                'InverseBoxCoxFlow'):
        pairs.append((getattr(rf, cls).__init__, getattr(of, cls).__init__))
        pairs.append((getattr(rf, cls).forward, getattr(of, cls).forward))
    for lik in ('GaussianNonLinearMean', 'GaussianLinearMean', 'Bernoulli', 'MulticlassCategorical'):
        pairs.append((getattr(rl, lik).expected_log_prob, getattr(ol, lik).expected_log_prob))
        pairs.append((getattr(rl, lik).marginal_moments, getattr(ol, lik).marginal_moments))
    bad = [(r.__qualname__, _sig(r), _sig(o)) for r, o in pairs if _sig(r) != _sig(o)]
    assert not bad, bad


def _plain(x):
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    if isinstance(x, dict):
        return {k: _plain(v) for k, v in x.items()}
    if isinstance(x, np.ndarray):
        return ('array', x.shape, x.tolist())
    return x


@pytest.mark.parametrize('gen,args,kw', [('StepSAL', (2, 3), {}), ('StepSAL', (1, 2), {'init_random': True, 'add_f0': True}),
                                         ('StepArcSL', (2, 2), {}), ('StepBoxCoxL', (1, 3), {'add_f0': True}),
                                         ('StepInverseBoxCoxL', (2, 2), {'init_random': True}), ('StepAllL', (3,), {}),
                                         ('StepTanhL', (2, 3), {'add_f0': True}), ('ArcSL', (2,), {}), ('BoxCoxL', (1,), {})])
def test_flow_generators_draw_the_reference_specification(gen, args, kw):
    """Same numpy seed -> the same (name, init dict) list as the reference's generator (flows.py:115-491): schema, values,
    RNG draw order; and the modules built from it carry the reference's parameter names in the reference's order."""
    _ref()
    import dsp.flows as rfl, dsp.models.flow as rf           # noqa: E401
    from tgp.pytorch_b200.dsp import flows as ofl
    from tgp.pytorch_b200.dsp.models import flow as of
    np.random.seed(11)
    ref = getattr(rfl, gen)(*args, **kw)
    np.random.seed(11)
    own = getattr(ofl, gen)(*args, **kw)
    drop = lambda spec: [(n, {k: v for k, v in d.items() if not k.startswith('input_dep') and k != 'input_dim'}) for n, d in spec]  # noqa: E731
    assert _plain(drop(ref)) == _plain(drop(own))
    names_ref = [(n, tuple(p.shape)) for n, p in rf.instance_flow(ref).named_parameters()]
    names_own = [(n, tuple(p.shape)) for n, p in of.instance_flow(own).named_parameters()]
    assert names_ref == names_own


def test_reference_initialiser_drives_our_flow_modules():
    """find_forward_params (reference initializers.py:29-109) fits G ~ identity on linspace(Y.min - 1, Y.max + 1) before training
    (main.py:168-190).  Run the reference's function on the reference's StepTanhL flow and on ours: same loss trajectory."""
    _ref()
    import dsp.config as rcg
    from dsp.initializers import find_forward_params
    import dsp.models.flow as rf, dsp.flows as rfl           # noqa: E401
    from tgp.pytorch_b200.dsp import config as ocg
    ocg.set_maximum_precission()
    rcg.set_maximum_precission()
    from tgp.pytorch_b200.dsp.models import flow as of
    from tgp.pytorch_b200.dsp import flows as ofl
    x = np.linspace(-3.0, 3.0, 500)
    import warnings
    losses = []
    for inst, gen in ((rf.instance_flow, rfl.StepTanhL), (of.instance_flow, ofl.StepTanhL)):
        torch.manual_seed(0)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            flow, loss = find_forward_params(x, x.copy(), lambda: inst(gen(1, 3, add_f0=True)), num_restarts=1, num_epochs=40, seed=3)
        losses.append(np.asarray(loss, dtype=np.float64))
        want = ['flow_arr.0.flow_arr.%d.%s' % (i, c) for i in range(3) for c in 'abcd'] + ['flow_arr.1.a', 'flow_arr.1.b']
        assert [n for n, _ in flow.named_parameters()] == want
    assert np.allclose(losses[0], losses[1], rtol=1e-12, atol=0.0), np.abs(losses[0] / losses[1] - 1).max()


def test_reference_input_dependent_initialiser_drives_our_flow_modules():
    """find_forward_params_input_dependent_flow (reference initializers.py:111-182, main.py:193-208): fits the flow MLPs to the
    constant initial parameters through `forward_initializer`, then calls `turn_off_initializer_parameters`."""
    _ref()
    from dsp.initializers import find_forward_params_input_dependent_flow
    import dsp.models.flow as rf, dsp.flows as rfl           # noqa: E401
    from tgp.pytorch_b200.dsp.models import flow as of
    from tgp.pytorch_b200.dsp import flows as ofl
    g = torch.Generator().manual_seed(1)
    X = torch.randn(64, 4, generator=g, dtype=torch.float64)
    loader = [(X[:32], X[:32, :1]), (X[32:], X[32:, :1])]
    cfg = dict(input_dependent=True, input_dim=4, inference='MC_dropout', hidden_activation='relu', num_hidden_layers=2, dropout=0.25,
               batch_norm=0, hidden_dim=16)
    out = []
    import contextlib, io, warnings
    for inst, gen in ((rf.instance_flow, rfl.SAL), (of.instance_flow, ofl.SAL)):
        torch.manual_seed(5)
        np.random.seed(5)
        flow = inst(gen(2, **cfg))
        with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
            warnings.simplefilter('ignore')
            torch.manual_seed(6)
            flow, loss = find_forward_params_input_dependent_flow(loader, FLOW=flow, num_epochs=5, noise_var=0.0)
        out.append(loss)
        assert all(fl.parameters_are_turn_off for fl in flow.flow_arr if hasattr(fl, 'parameters_are_turn_off'))
        assert not [n for n, _ in flow.named_parameters() if n.endswith('.0.a') and 'NNets' not in n]     # scalars detached from the model
    assert abs(out[0] - out[1]) <= 1e-12 * abs(out[0]), out
