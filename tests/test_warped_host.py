"""The warped likelihood without a GPU: the constant and the new entry point in the header and the binding, descriptor packing of
WarpedGaussianLinearMean.flow, the scope refusals of the model class, and C-ABI validation that fails before any launch."""
import ctypes as C
import os

import pytest
import torch

from tgp.pytorch_b200 import _lib

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'tgp_b200.h')
FAKE = C.c_void_p(4096)          # never dereferenced: validation returns before anything is enqueued


def _lib_or_skip():
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip('libtgp_b200.so not built')
    return _lib.load()


def _model(layers=(), n_theta=0, n_quad=20, likelihood=None):
    m = _lib.TgpModel()
    m.dtype, m.M, m.D, m.n_quad = _lib.TGP_F64, 64, 8, n_quad
    m.likelihood = _lib.LIK_GAUSS_WARPED if likelihood is None else likelihood
    m.n_layers, m.n_theta = len(layers), n_theta
    for i, (kind, flags, p0) in enumerate(layers):
        m.layers[i].kind, m.layers[i].flags, m.layers[i].n_steps, m.layers[i].p0 = kind, flags, 1, p0
    return m


def _fp64():
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    cg.device = 'cpu'


def test_constant_entry_point_and_binding():
    text = open(HEADER).read()
    assert 'TGP_LIK_GAUSS_WARPED = 3' in text and _lib.LIK_GAUSS_WARPED == 3
    assert 'int tgp_flow_inverse(' in text and 'tgp_flow_inverse' in _lib.SIGNATURES
    from tgp.pytorch_b200.engine import _LIK
    assert _LIK['gauss_warped'] == _lib.LIK_GAUSS_WARPED
    lib = _lib_or_skip()
    assert lib.tgp_flow_inverse.argtypes == _lib.SIGNATURES['tgp_flow_inverse'][1]


def test_validation_of_the_warped_likelihood():
    lib = _lib_or_skip()
    sal = (_lib.FLOW_SAL, _lib.FLOW_RESTRICT, 0)
    assert lib.tgp_step_workspace_bytes(_model([sal], 2)) > 0
    assert lib.tgp_step_workspace_bytes(_model([sal], 2, n_quad=0)) == 0            # the moments need a rule
    assert b'n_quad' in lib.tgp_last_error()
    assert lib.tgp_step_workspace_bytes(_model([sal], 2, likelihood=4)) == 0
    assert b'unknown likelihood' in lib.tgp_last_error()
    per_row = _model([(_lib.FLOW_SAL, _lib.FLOW_PER_ROW, 0)])
    per_row.n_rowparams = 2
    assert lib.tgp_step_workspace_bytes(per_row) == 0
    assert b'global parameters' in lib.tgp_last_error()
    per_row.n_rowparams = 0
    assert lib.tgp_step_workspace_bytes(per_row) == 0
    assert b'input-dependent warps' in lib.tgp_last_error()
    p = _lib.TgpParams()
    rc = lib.tgp_ell_forward(per_row, p, FAKE, FAKE, FAKE, None, 10, 1.0, None, None, 1, FAKE, FAKE, FAKE, None, FAKE, None)
    assert rc == -1 and b'input-dependent warps' in lib.tgp_last_error()
    # a warp with parameters needs theta (quadrature pointers may be NULL)
    rc = lib.tgp_ell_forward(_model([sal], 2), p, FAKE, FAKE, FAKE, None, 10, 1.0, None, None, 1, FAKE, FAKE, FAKE, None, FAKE, None)
    assert rc == -1 and b'theta required' in lib.tgp_last_error()
    # the test rows need the rule for the moments, and one dropout sample
    rc = lib.tgp_test_rows(_model([sal], 2), p, FAKE, FAKE, FAKE, None, 10, 1, 1.0, None, None, None, FAKE, FAKE, FAKE, None)
    assert rc == -1 and b'quadrature rule' in lib.tgp_last_error()
    rc = lib.tgp_test_rows(_model([sal], 2), p, FAKE, FAKE, FAKE, None, 10, 2, 1.0, FAKE, FAKE, None, FAKE, FAKE, FAKE, None)
    assert rc == -1 and b'n_mc = 1' in lib.tgp_last_error()
    p.log_var_noise = FAKE
    rc = lib.tgp_coverage_rows(_model([sal], 2), p, FAKE, FAKE, FAKE, None, 10, 1, 8, 0, None, 0.025, 0.975, FAKE, FAKE, FAKE,
                               None, None, None)
    assert rc == -1 and b'warped likelihood' in lib.tgp_last_error()


def test_flow_inverse_validation():
    lib = _lib_or_skip()
    sal = (_lib.FLOW_SAL, _lib.FLOW_RESTRICT, 0)
    n_fail = C.c_void_p(8192)
    assert lib.tgp_flow_inverse(_model([sal], 2), None, FAKE, 10, FAKE, n_fail, None) == -1
    assert b'NULL argument' in lib.tgp_last_error()
    assert lib.tgp_flow_inverse(_model([sal], 2), FAKE, FAKE, 10, FAKE, None, None) == -1
    per_row = _model([(_lib.FLOW_SAL, _lib.FLOW_PER_ROW, 0)], likelihood=_lib.LIK_GAUSS_NONLINEAR)
    per_row.n_rowparams = 2
    assert lib.tgp_flow_inverse(per_row, None, FAKE, 10, FAKE, n_fail, None) == -1
    assert b'global parameters' in lib.tgp_last_error()
    assert lib.tgp_flow_inverse(_model([sal], 2), None, None, 0, None, None, None) == 0


def test_descriptor_packing_of_the_warps():
    _fp64()
    import numpy
    from tgp.pytorch_b200.dsp.flows import SAL, StepTanhL
    from tgp.pytorch_b200.dsp.likelihoods import WarpedGaussianLinearMean
    from tgp.pytorch_b200.dsp.likelihoods import _rows
    from tgp.pytorch_b200.dsp.models.flow import instance_flow
    numpy.random.seed(0)
    inst = instance_flow(SAL(1))
    lik = WarpedGaussianLinearMean(2, 0.05, False, [StepTanhL(1, 3, add_f0=True), inst])
    assert isinstance(lik.flow, torch.nn.ModuleList) and lik.flow[1] is inst
    assert lik.log_var_noise.shape == (2, 1)
    layout, theta, rowp = _rows.flow_pack(lik.flow[0], None)
    assert rowp is None and layout.n_theta == 14 and theta.shape == (14,)
    assert [(l['kind'], l['n_steps'], l['add_f0'], l['p0']) for l in layout.layers] == [('tanh_step', 3, True, 0), ('affine', 0, False, 12)]
    step, aff = lik.flow[0].flow_arr
    want = [t for s in step.flow_arr for t in (s.a, s.b, s.c, s.d)] + [aff.a, aff.b]
    assert torch.equal(theta, torch.stack([t.detach() for t in want]))
    md = _lib.TgpModel()
    layout.fill(md)
    assert (md.n_layers, md.n_theta, md.layers[0].kind, md.layers[0].flags) == (2, 14, _lib.FLOW_TANH_STEP, _lib.FLOW_ADD_F0)
    layout, theta, _ = _rows.flow_pack(lik.flow[1], None)
    assert [l['kind'] for l in layout.layers] == ['sal', 'affine'] and layout.n_theta == 4
    shared = WarpedGaussianLinearMean(2, 0.05, True, [StepTanhL(1, 1), StepTanhL(1, 1)])
    assert shared.log_var_noise.shape == (1, 1) and len(shared.flow) == 2


def _cpu_model(lik, flow_on_f=None):
    from tgp.pytorch_b200.dsp.models import instance_kernel, sparse_MF_GP, sparse_MF_SP
    X = torch.randn(40, 3, dtype=torch.float64)
    K = instance_kernel('scale_rbf', ard_num_dim=3, num_multioutput=1, kernel_is_shared=False)
    ip = {'variational_distribution': {'variance_scale': 1e-2, 'mean_scale': 0.0}}
    if flow_on_f is None:
        return sparse_MF_GP(['zero', K], X, X[:8].clone(), 100, lik, 1, True, False, False, False, False, 0.0, ip), X
    return sparse_MF_SP(['zero', K], X, X[:8].clone(), 100, lik, 1, True, False, False, False, False, [flow_on_f], 'single',
                        0.0, False, ip), X


def test_scope_refusals_of_the_model_class():
    _fp64()
    from tgp.pytorch_b200.dsp.flows import SAL, StepTanhL
    from tgp.pytorch_b200.dsp.likelihoods import WarpedGaussianLinearMean
    from tgp.pytorch_b200.dsp.models.flow import instance_flow
    lik = WarpedGaussianLinearMean(1, 0.05, False, [StepTanhL(1, 2, add_f0=True)])
    model, X = _cpu_model(lik)
    assert model.quad_points == lik.quad_points
    layout, theta = model._warp_pack(0, X)
    assert layout.n_theta == 10 and theta.shape == (10,)
    with pytest.raises(NotImplementedError, match='joint predictive'):
        lik.marginal_moments(torch.zeros(1, 5), torch.ones(1, 5, 5), diagonal=False)
    model.set_is_training(False)
    with pytest.raises(NotImplementedError, match='not Gaussian'):
        model.predictive_distribution(X, diagonal=False)
    with pytest.raises(NotImplementedError, match='warped likelihood'):
        model.evaluation_bundle(X, torch.zeros(40, 1, dtype=torch.float64), torch.ones(1, dtype=torch.float64))
    # a flow on f as well as the warp
    model2, X = _cpu_model(WarpedGaussianLinearMean(1, 0.05, False, [StepTanhL(1, 2, add_f0=True)]), instance_flow(SAL(1)))
    with pytest.raises(NotImplementedError, match='flow on f'):
        model2._warp_pack(0, X)
    # an input-dependent warp
    idw = instance_flow(SAL(1, input_dependent=True, input_dim=3, hidden_dim=4, num_hidden_layers=1))
    idw.turn_off_initializer_parameters()
    model3, X = _cpu_model(WarpedGaussianLinearMean(1, 0.05, False, [idw]))
    with pytest.raises(NotImplementedError, match='input-dependent warps'):
        model3._warp_pack(0, X)
