"""The non-whitened q(u) form in the C-ABI without a GPU: exported constants and struct layout, validation of q_u_form, and
workspace sizes (whitened sizes as before the form existed; a non-whitened step workspace adds exactly its Mp x Mp region)."""
import os

import pytest

from tgp.pytorch_b200 import _lib

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'tgp_b200.h')

# (dtype, M, D) -> (tgp_step_workspace_bytes, tgp_workspace_bytes(model, 5000)) of whitened models, recorded with the
# library as it was before TgpModel.q_u_form existed
WHITENED_SIZES = {
    (0, 64, 8): (333312, 13443392), (0, 300, 8): (18929920, 84091712), (0, 1024, 8): (75604992, 305928512),
    (0, 2048, 16): (302302208, 813340992), (1, 64, 8): (464896, 19991104), (1, 300, 8): (21812832, 117334336),
    (1, 1024, 8): (109167616, 446081344), (1, 2048, 16): (436536320, 1169144128), (2, 64, 8): (661508, 39520064),
    (2, 300, 8): (26209284, 216572736), (2, 1024, 8): (159499268, 837180224), (2, 2048, 16): (637862916, 2119113536),
}


def _lib_or_skip():
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip('libtgp_b200.so not built')
    return _lib.load()


def _model(dtype, M, D, q_u_form=0):
    m = _lib.TgpModel()
    m.dtype, m.M, m.D, m.likelihood, m.n_quad, m.q_u_form = dtype, M, D, _lib.LIK_GAUSS_NONLINEAR, 20, q_u_form
    return m


def _pad(M):
    mp = 64
    while mp < M:
        mp *= 2
    return mp


def test_constants_and_struct_layout():
    assert (_lib.QU_WHITENED, _lib.QU_UNWHITENED) == (0, 1)
    text = open(HEADER).read()
    assert 'TGP_QU_WHITENED = 0' in text and 'TGP_QU_UNWHITENED = 1' in text
    # appended after `kernel`: no earlier field moves, and a zero-initialised description is whitened
    assert _lib.TgpModel._fields_[-1][0] == 'q_u_form' and _lib.TgpModel._fields_[-2][0] == 'kernel'
    assert _lib.TgpModel.q_u_form.offset == _lib.TgpModel.kernel.offset + 4
    assert _lib.TgpModel().q_u_form == _lib.QU_WHITENED
    assert text.index('int kernel;') < text.index('int q_u_form;') < text.index('} TgpModel;')


def test_validation_rejects_unknown_forms():
    lib = _lib_or_skip()
    for bad in (2, -1, 7):
        assert lib.tgp_step_workspace_bytes(_model(_lib.TGP_F64, 64, 8, bad)) == 0
        assert b'q_u_form' in lib.tgp_last_error()
        assert lib.tgp_workspace_bytes(_model(_lib.TGP_F64_I8, 64, 8, bad), 100) == 0


@pytest.mark.parametrize('key', sorted(WHITENED_SIZES))
def test_workspace_sizes(key):
    lib = _lib_or_skip()
    dtype, M, D = key
    step_w, handle_w = WHITENED_SIZES[key]
    assert lib.tgp_step_workspace_bytes(_model(dtype, M, D)) == step_w
    assert lib.tgp_workspace_bytes(_model(dtype, M, D), 5000) == handle_w
    # step_layout carves tril(L_raw) last, on the next 256-byte boundary (common.cuh Carve)
    step_u = lib.tgp_step_workspace_bytes(_model(dtype, M, D, _lib.QU_UNWHITENED))
    assert step_u == (step_w + 255) // 256 * 256 + 8 * _pad(M) ** 2
    assert lib.tgp_batch_workspace_bytes(_model(dtype, M, D, 1), 5000) == lib.tgp_batch_workspace_bytes(_model(dtype, M, D), 5000)
    ceil = lambda n: (n + 255) // 256 * 256  # noqa: E731
    assert lib.tgp_workspace_bytes(_model(dtype, M, D, 1), 5000) - handle_w == ceil(step_u) - ceil(step_w)
    rw, ru = _lib.TgpReduceLayout(), _lib.TgpReduceLayout()
    assert lib.tgp_reduce_layout(_model(dtype, M, D), rw) == 0 and lib.tgp_reduce_layout(_model(dtype, M, D, 1), ru) == 0
    assert [getattr(rw, f) for f, _ in rw._fields_] == [getattr(ru, f) for f, _ in ru._fields_]
