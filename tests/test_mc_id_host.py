"""tgp_mc_softmax_rows_rowp without a GPU: the export and its binding, and the argument checks that return before anything is
enqueued.  tgp_mc_softmax_rows keeps refusing per-row flows."""
import ctypes as C
import os

import pytest

from tgp.pytorch_b200 import _lib
from tgp.pytorch_b200.engine import FlowLayout

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'tgp_b200.h')
FAKE = C.c_void_p(4096)          # never dereferenced: validation returns before anything is enqueued


def _lib_or_skip():
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip('libtgp_b200.so not built')
    return _lib.load()


def _model(layers):
    from tgp.pytorch_b200.dsp.likelihoods._rows import _mc_model
    return _mc_model(FlowLayout(layers))


ID_SAL = [dict(kind='sal', per_row=True), dict(kind='affine')]                   # 2 per-row, 2 global
ID_TANH3 = [dict(kind='tanh_step', n_steps=3, add_f0=True, per_row=True), dict(kind='affine')]   # 12 per-row


def _call(lib, md, C_, rowp, want_grad, drowp, R=10, S=4):
    return lib.tgp_mc_softmax_rows_rowp(md, C_, S, R, FAKE, FAKE, FAKE, FAKE, FAKE, want_grad, FAKE, FAKE, FAKE, FAKE, None,
                                        rowp, drowp, None)


def test_export_and_binding():
    text = open(HEADER).read()
    assert 'tgp_mc_softmax_rows_rowp(' in text and 'tgp_mc_softmax_rows_rowp' in _lib.SIGNATURES
    res, args = _lib.SIGNATURES['tgp_mc_softmax_rows_rowp']
    assert args[:-3] == _lib.SIGNATURES['tgp_mc_softmax_rows'][1][:-1] and len(args) == 18
    lib = _lib_or_skip()
    assert lib.tgp_mc_softmax_rows_rowp.argtypes == args
    assert lib.tgp_version() == 102


def test_rowp_argument_checks():
    lib = _lib_or_skip()
    md = _model(ID_SAL)
    assert md.n_rowparams == 2 and md.n_theta == 2
    assert _call(lib, md, 3, None, 0, None) == -1
    assert b'rowparams required' in lib.tgp_last_error()
    assert _call(lib, md, 3, FAKE, 1, None) == -1
    assert b'drowparams required' in lib.tgp_last_error()
    # 3 x 12 per-row parameters fit the accumulator, 32 x 12 do not
    big = _model(ID_TANH3)
    assert big.n_rowparams == 12
    assert _call(lib, big, 32, FAKE, 1, FAKE) == -1
    assert b'C * n_rowparams' in lib.tgp_last_error()
    # the checks shared with tgp_mc_softmax_rows
    assert _call(lib, md, 33, FAKE, 1, FAKE) == -1
    assert b'number of classes' in lib.tgp_last_error()
    assert _call(lib, md, 3, FAKE, 1, FAKE, S=0) == -1
    assert b'S must be positive' in lib.tgp_last_error()
    bad = _model(ID_SAL)
    bad.n_rowparams = 17
    assert _call(lib, bad, 3, FAKE, 1, FAKE) == -1
    assert b'per-row flow parameters' in lib.tgp_last_error()
    # no rows: nothing to do
    assert _call(lib, md, 3, None, 1, None, R=0) == 0


def test_global_entry_point_still_refuses_per_row_flows():
    lib = _lib_or_skip()
    md = _model(ID_SAL)
    rc = lib.tgp_mc_softmax_rows(md, 3, 4, 10, FAKE, FAKE, FAKE, FAKE, FAKE, 1, FAKE, FAKE, FAKE, FAKE, None, None)
    assert rc == -1
    assert b'the Monte-Carlo softmax likelihood takes flows with global parameters' in lib.tgp_last_error()
