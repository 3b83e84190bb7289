"""Host side of the full-covariance entry points, without a GPU: the symbols are exported, the workspace sizes behave, and
argument validation fails with a message before anything reaches the device."""
import ctypes as C
import os

import pytest

NEW = ('tgp_qf_cov_workspace_bytes', 'tgp_qf_cov_forward', 'tgp_cov_cholesky_workspace_bytes', 'tgp_cov_cholesky',
       'tgp_cov_sample')


def _lib():
    from tgp.pytorch_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip('libtgp_b200.so not built')
    return _lib, _lib.load()


def _model(L, dtype, kernel=0, M=300, D=8):
    m = L.TgpModel()
    m.dtype, m.M, m.D, m.likelihood, m.n_quad, m.kernel = dtype, M, D, L.LIK_GAUSS_LINEAR, 0, kernel
    return m


def test_new_symbols_are_exported_and_bound():
    L, lib = _lib()
    for name in NEW:
        assert hasattr(lib, name) and name in L.SIGNATURES, name


def test_workspace_sizes_grow_with_R_and_ignore_mode_and_kernel():
    L, lib = _lib()
    Rs = (1, 2, 63, 64, 65, 200, 2048, 4097, 16384)
    dtypes = (L.TGP_F64, L.TGP_F32, L.TGP_F64_I8)
    kinds = (L.KERNEL_RBF, L.KERNEL_MATERN12, L.KERNEL_MATERN32, L.KERNEL_MATERN52)
    for M, D in ((64, 8), (1024, 8), (300, 40)):
        prev = 0
        for R in Rs:
            sizes = {lib.tgp_qf_cov_workspace_bytes(_model(L, dt, k, M, D), R) for dt in dtypes for k in kinds}
            assert len(sizes) == 1, (M, D, R, sizes)
            size = sizes.pop()
            assert size >= prev and size >= (3 * M + 1) * R * 8
            prev = size
    prev = 0
    for R in Rs:
        size = lib.tgp_cov_cholesky_workspace_bytes(R)
        Rp = -(-R // 64) * 64
        assert size >= prev and size >= (2 * Rp + 64) * Rp * 8
        prev = size
    assert lib.tgp_qf_cov_workspace_bytes(_model(L, L.TGP_F64), 0) == 0
    assert lib.tgp_cov_cholesky_workspace_bytes(0) == 0


def _err(lib):
    return lib.tgp_last_error().decode()


def test_argument_validation_happens_before_any_device_call():
    """Host pointers that are never dereferenced stand in for device buffers: every call below must be refused first."""
    L, lib = _lib()
    buf = C.create_string_buffer(64)
    p = C.cast(buf, C.c_void_p)
    md = _model(L, L.TGP_F64)
    assert lib.tgp_qf_cov_forward(md, p, p, p, 0, p, p, 1, None) < 0 and 'R' in _err(lib)
    assert lib.tgp_qf_cov_forward(md, p, p, p, 10, p, p, 9, None) < 0 and 'ldc' in _err(lib)
    assert lib.tgp_qf_cov_forward(md, None, p, p, 10, p, p, 10, None) < 0 and 'NULL' in _err(lib)
    assert lib.tgp_qf_cov_forward(md, p, p, p, 10, p, None, 10, None) < 0 and 'NULL' in _err(lib)
    bad = _model(L, L.TGP_F64, kernel=4)
    assert lib.tgp_qf_cov_forward(bad, p, p, p, 10, p, p, 10, None) < 0 and 'kernel' in _err(lib)
    assert lib.tgp_qf_cov_workspace_bytes(bad, 10) == 0

    assert lib.tgp_cov_cholesky(0, p, 1, 0.0, p, p, p, 1, p, None) < 0 and 'R' in _err(lib)
    assert lib.tgp_cov_cholesky(10, p, 9, 0.0, p, p, p, 10, p, None) < 0 and 'ld' in _err(lib)
    assert lib.tgp_cov_cholesky(10, p, 10, 0.0, p, p, p, 9, p, None) < 0 and 'ld' in _err(lib)
    assert lib.tgp_cov_cholesky(10, p, 10, -1e-9, p, p, p, 10, p, None) < 0 and 'jitter' in _err(lib)
    assert lib.tgp_cov_cholesky(10, p, 10, float('nan'), p, p, p, 10, p, None) < 0 and 'jitter' in _err(lib)
    assert lib.tgp_cov_cholesky(10, p, 10, 0.0, None, p, p, 10, p, None) < 0 and 'NULL' in _err(lib)
    assert lib.tgp_cov_cholesky(10, p, 10, 0.0, p, p, p, 10, None, None) < 0 and 'NULL' in _err(lib)

    assert lib.tgp_cov_sample(0, 1, p, p, 1, p, p, None) < 0 and 'R' in _err(lib)
    assert lib.tgp_cov_sample(10, 0, p, p, 10, p, p, None) < 0 and 'S' in _err(lib)
    assert lib.tgp_cov_sample(10, 3, p, p, 9, p, p, None) < 0 and 'ldl' in _err(lib)
    assert lib.tgp_cov_sample(10, 3, p, p, 10, None, p, None) < 0 and 'NULL' in _err(lib)


def test_joint_calls_under_autograd_are_refused_without_a_gpu():
    """qf_covariance has no backward: with grad enabled and a parameter that requires grad it raises before touching the
    engine (a stand-in object here)."""
    import torch
    from tgp.pytorch_b200 import functional as Fn
    t = torch.zeros(3, dtype=torch.float64, requires_grad=True)
    with pytest.raises(NotImplementedError, match='no_grad'):
        Fn.qf_covariance(object(), torch.zeros(2, 1, dtype=torch.float64), t, t, t, t, t)
