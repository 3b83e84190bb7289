"""Input gradients in the C-ABI without a GPU: the new exports, the TgpGrads layout (dX appended, no earlier field moved) and
argument validation through tgp_last_error()."""
import ctypes as C
import os

import pytest

from tgp.pytorch_b200 import _lib

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'tgp_b200.h')
NEW = ('tgp_qf_backward_dx', 'tgp_flow_mlp_backward_dx')
FAKE = C.c_void_p(4096)          # never dereferenced: validation returns before anything is enqueued


def _lib_or_skip():
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip('libtgp_b200.so not built')
    return _lib.load()


def _model(D=8):
    m = _lib.TgpModel()
    m.dtype, m.M, m.D, m.likelihood, m.n_quad = _lib.TGP_F64, 64, D, _lib.LIK_GAUSS_NONLINEAR, 20
    return m


def _mlp(n_in=4):
    m = _lib.TgpMlp()
    m.n_nets, m.n_in, m.hidden, m.n_hidden_layers, m.activation, m.mask_mode = 2, n_in, 16, 2, 0, 0
    return m


def test_exports_and_interface_version_102():
    text = open(HEADER).read()
    for name in NEW:
        assert name + '(' in text and name in _lib.SIGNATURES
    lib = _lib_or_skip()
    for name in NEW:
        assert hasattr(lib, name)
    assert lib.tgp_version() == 102


def test_grads_struct_layout():
    names = [f for f, _ in _lib.TgpGrads._fields_]
    assert names == ['dZ', 'draw_lengthscale', 'draw_outputscale', 'dm', 'dL_raw', 'dlog_var_noise', 'dtheta', 'drowparams', 'dX']
    ptr = C.sizeof(C.c_void_p)
    for i, n in enumerate(names):
        assert getattr(_lib.TgpGrads, n).offset == i * ptr
    assert _lib.TgpGrads().dX is None
    text = open(HEADER).read()
    body = text[text.index('typedef struct TgpGrads'):text.index('} TgpGrads;')]
    assert body.index('void* drowparams;') < body.index('void* dX;')


def test_qf_backward_dx_validation():
    lib = _lib_or_skip()
    p = _lib.TgpParams()
    # NULL inputs are refused whether or not dX is asked for
    assert lib.tgp_qf_backward_dx(_model(), p, None, FAKE, FAKE, 10, FAKE, FAKE, FAKE, FAKE, None) == -1
    assert b'NULL argument' in lib.tgp_last_error()
    assert lib.tgp_qf_backward_dx(_model(), p, FAKE, FAKE, FAKE, 10, None, FAKE, FAKE, None, None) == -1
    # input gradients cover D <= 64, as the kernel-parameter gradients do
    assert lib.tgp_qf_backward_dx(_model(65), p, FAKE, FAKE, FAKE, 10, FAKE, FAKE, FAKE, FAKE, None) == -2
    assert b'D <= 64' in lib.tgp_last_error()
    # an invalid model is refused before anything else
    bad = _model()
    bad.dtype = 9
    assert lib.tgp_qf_backward_dx(bad, p, FAKE, FAKE, FAKE, 10, FAKE, FAKE, FAKE, FAKE, None) == -1
    assert b'dtype' in lib.tgp_last_error()
    # no rows: nothing to do
    assert lib.tgp_qf_backward_dx(_model(), p, None, None, None, 0, None, None, None, None, None) == 0


def test_flow_mlp_backward_dx_validation():
    lib = _lib_or_skip()
    assert lib.tgp_flow_mlp_backward_dx(_mlp(), FAKE, FAKE, 10, None, None, FAKE, FAKE, None) == -1
    assert b'NULL argument' in lib.tgp_last_error()
    assert lib.tgp_flow_mlp_backward_dx(_mlp(65), FAKE, FAKE, 10, None, FAKE, FAKE, FAKE, None) == -1
    assert b'n_in' in lib.tgp_last_error()
    m = _mlp()
    m.mask_mode, m.p_drop = 2, 0.25
    assert lib.tgp_flow_mlp_backward_dx(m, FAKE, FAKE, 10, None, FAKE, FAKE, FAKE, None) == -1
    assert b'keep-mask' in lib.tgp_last_error()
