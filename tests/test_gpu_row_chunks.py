"""The row-chunk loops of the batch contractions against the CPU references, at row counts that cross the chunk boundaries.

'i8crt' and 'tf32x3' split a minibatch into chunks of 16384 rows (CRT_ROW_CHUNK in crt_driver.cuh, TC_ROW_CHUNK in
tc_driver.cuh: compile-time constants), 'f64' into chunks of TGP_OPT_ROW_CHUNK = 32768 rows.  R = 16384 is one full chunk,
R = 16385 adds a one-row chunk, R = 32845 = 2 * 16384 + 77 also crosses the 'f64' chunk and leaves a ragged last chunk of 77
rows.  Per chunk, the 'i8crt' backward rebuilds the column exponents of [Abar | Bbar] and the W~ planes, and reads its slice of
the K residue planes (and, for D > 32, of the FP64 K_xz); 'tf32x3' keeps one set of K^T planes per chunk and picks its split-K
from the chunk's row count; both accumulate Gbar / Cbar across chunks, and every mode offsets X, dX, mu and the row gradients
by the chunk's first row.

Three checks: the references (tests/matern_ref.py, tests/input_grad_ref.py) at these row counts; chunk invariance (the gradients
of the whole batch equal the sum of the gradients of its chunk-sized slices to FP64 rounding, in every mode, so a wrong chunk
offset shows up as an O(1) error even where the FP32 bound of 'tf32x3' is loose); the backward of the q(f) marginals.  Last, a
float32 model with D = 64, which the tensor-core mode serves with more than 48 KiB of shared memory in its K generation.
"""
import warnings

import pytest
import torch

from tests import input_grad_ref as IR
from tests import matern_ref as MR
from tests.conftest import record_residuals
from tests.golden_util import rel_err
from tests.gpu_util import engine_inputs
from tests.test_gpu_matern import _cuda, _engine, _ok, _oracle, _problem, _to

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
CHUNK = 16384                        # CRT_ROW_CHUNK and TC_ROW_CHUNK
RAGGED = 2 * CHUNK + 77
MODES = ['f64', 'i8crt', 'tf32x3']
LIK, NQ = 'gauss_nonlinear', 20
# (M, D, kernel): the Matern-1/2 backward recomputes K from the chunk's rows of X, and its coincident rows (Z is drawn from X)
# take the r = 0 convention; D = 40 > 32 makes 'i8crt' stage K_xz in FP64, whose chunk slice the RBF's kernel gradients read
SHAPES = [(201, 8, 'matern12'), (96, 40, 'rbf')]
PARAMS = ('Z', 'raw_ls', 'raw_os', 'm', 'L_raw', 'log_var_noise')


def _yardstick(errs, ref, ref32):
    """'tf32x3' bound: 1e-5 + 4 x (O2's own float32 evaluation against its float64 one), as in tests/test_gpu_matern.py."""
    return {k: (e, rel_err(ref32[k], ref[k])) for k, e in errs.items() if not e < 1e-5 + 4.0 * rel_err(ref32[k], ref[k])}


@pytest.mark.parametrize('M,D,kernel', SHAPES)
@pytest.mark.parametrize('R', [CHUNK, CHUNK + 1, RAGGED])
@pytest.mark.parametrize('compute', MODES)
def test_elbo_and_every_gradient_across_row_chunks(compute, R, M, D, kernel):
    X, y, p = _problem(R, M, D, seed=R + M + D, kernel=kernel)
    N = 10.0 * R
    got, _ = _cuda(X, y, p, N, LIK, NQ, compute, want_dx=True)
    ref = _oracle(X, y, p, N, LIK, NQ)
    ref['X'] = IR.elbo_grads_xz(X, y, p, N, LIK, NQ)[1]
    errs = {k: rel_err(got[k], ref[k]) for k in got}
    record_residuals('row_chunks[%s,%s,D=%d]' % (compute, kernel, D), errs)
    if compute == 'tf32x3':
        X32, y32, p32 = X.float(), y.float(), _to(p, torch.float32)
        ref32 = _oracle(X32, y32, p32, N, LIK, NQ)
        ref32['X'] = IR.elbo_grads_xz(X32, y32, p32, N, LIK, NQ)[1]
        bad = _yardstick(errs, ref, ref32)
    else:
        bad = {k: e for k, e in errs.items() if not _ok(k, e, LIK)}
    assert not bad, (bad, errs)


def _sliced_grads(X, y, p, N, compute, slices):
    """{parameter: gradient, 'X': dX} of ELL - KLD over the rows of X, accumulated over one call per row slice with the global
    scale N / R and the KL counted in the first call only: what row-sharded evaluation computes across ranks."""
    from tgp.pytorch_b200 import functional as Fn
    eng, theta, names = _engine(p, LIK, NQ, compute)
    ei = engine_inputs(p, DEV)
    leaves = [ei[k].requires_grad_(True) for k in PARAMS] + [theta.requires_grad_(True)]
    Xd = X.to(DEV).contiguous().requires_grad_(True)
    yd = y.to(DEV).contiguous()
    for i, sl in enumerate(slices):
        ELL, KLD, _, _, _ = Fn.elbo_terms(eng, Xd[sl].contiguous(), yd[sl].contiguous(), N / X.shape[0], *leaves, None)
        (ELL - KLD if i == 0 else ELL).backward()
    out = {k: t.grad.detach().cpu().reshape(-1) for k, t in zip(PARAMS, leaves)}
    out.update({n: theta.grad[i].detach().cpu() for i, n in enumerate(names)})
    out['X'] = Xd.grad.detach().cpu()
    return out


@pytest.mark.parametrize('M,D,kernel', SHAPES)
@pytest.mark.parametrize('compute', MODES)
def test_gradients_do_not_depend_on_the_row_chunking(compute, M, D, kernel):
    """One call over R = 32845 rows against three calls over the chunk-sized slices [0, 16384), [16384, 32768), [32768, R).  In
    'i8crt' and 'tf32x3' each slice is what the one call computes as its chunk (same rows, same column exponents, same split-K),
    so only the order of the FP64 accumulation across chunks differs; 'f64' runs its one call as chunks of 32768 + 77 rows."""
    X, y, p = _problem(RAGGED, M, D, seed=7 + M + D, kernel=kernel)
    N = 10.0 * RAGGED
    whole = _sliced_grads(X, y, p, N, compute, [slice(0, RAGGED)])
    parts = _sliced_grads(X, y, p, N, compute, [slice(0, CHUNK), slice(CHUNK, 2 * CHUNK), slice(2 * CHUNK, RAGGED)])
    errs = {k: rel_err(parts[k], whole[k]) for k in whole}
    record_residuals('row_chunk_invariance[%s,%s,D=%d]' % (compute, kernel, D), errs)
    bad = {k: e for k, e in errs.items() if not e < 1e-12}
    assert not bad, (bad, errs)


@pytest.mark.parametrize('M,D,kernel', SHAPES)
@pytest.mark.parametrize('compute', MODES)
def test_marginals_dx_across_row_chunks(compute, M, D, kernel):
    """Fn.qf_marginals with X.requires_grad at R = 32845 against the autograd reference of tests/input_grad_ref.py."""
    from tgp.pytorch_b200 import functional as Fn
    from tgp.pytorch_b200.engine import Engine, FlowLayout
    X, _, p = _problem(RAGGED, M, D, seed=3 + M + D, kernel=kernel)
    g = torch.Generator().manual_seed(11)
    w_mu = torch.randn(RAGGED, generator=g, dtype=torch.float64)
    w_v = torch.randn(RAGGED, generator=g, dtype=torch.float64)
    eng = Engine(M, D, 'gauss_linear', 0, FlowLayout([]), DEV, compute=compute, kernel=kernel)
    ei = engine_inputs(p, DEV)
    Xd = X.to(DEV).contiguous().requires_grad_(True)
    mu, v = Fn.qf_marginals(eng, Xd, ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'])
    ((mu * w_mu.to(DEV)).sum() + (v * w_v.to(DEV)).sum()).backward()
    ref = IR.marginals_grad_x(X, p, w_mu, w_v)
    e = rel_err(Xd.grad.cpu(), ref)
    record_residuals('row_chunks_marginals_dx[%s,%s,D=%d]' % (compute, kernel, D), {'X': e})
    if compute == 'tf32x3':
        ref32 = IR.marginals_grad_x(X.float(), _to(p, torch.float32), w_mu.float(), w_v.float())
        assert e < 1e-5 + 4.0 * rel_err(ref32, ref), (e, rel_err(ref32, ref))
    else:
        assert e < 1e-10, e


def test_float32_model_with_64_input_dimensions():
    """A float32 SVGP (served by 'tf32x3') with D = 64 over 16385 rows: ELBO, every parameter gradient and X.grad against the
    reference evaluated on the model's float32 values, within the FP32 bound of the tests above."""
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    cg.device = DEV
    from tgp.pytorch_b200.dsp.models import instance_kernel, sparse_MF_GP
    from tgp.pytorch_b200.dsp.likelihoods import GaussianLinearMean
    R, M, D, N = CHUNK + 1, 64, 64, 1.0e5
    X, y, p = _problem(R, M, D, seed=64, kernel='rbf', lik='gauss_linear')
    K = instance_kernel('scale_rbf', ard_num_dim=D, num_multioutput=1, kernel_is_shared=False)
    lik = GaussianLinearMean(out_dim=1, noise_init=0.3, noise_is_shared=True)
    model = sparse_MF_GP(['zero', K], X, p['Z'], N, lik, 1, True, False, False, False, False, 0.0, {})
    with torch.no_grad():
        K.base_kernel.raw_lengthscale.copy_(p['raw_lengthscale'].view(1, 1, -1))
        K.raw_outputscale.fill_(float(p['raw_outputscale']))
        model.q_U.variational_mean[0].copy_(p['m'])
        model.q_U.chol_variational_covar[0].copy_(p['L_raw'])
        lik.log_var_noise.fill_(float(p['log_var_noise']))
    model = model.float().to(DEV)
    X32, y32 = X.float(), y.float()
    Xd = X32.to(DEV).requires_grad_(True)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        ELBO, _, _ = model.ELBO(Xd, y32.view(-1, 1).to(DEV))
        ELBO.backward()
    assert any(e.compute == 'tf32x3' for e in model._engines.values())
    assert ELBO.dtype == torch.float32 and Xd.grad.dtype == torch.float32
    prm = dict(model.named_parameters())
    got = {'ELBO': ELBO.detach().cpu(), 'X': Xd.grad.cpu(), 'Z': prm['Z'].grad, 'm': prm['q_U.variational_mean'].grad,
           'L_raw': prm['q_U.chol_variational_covar'].grad, 'log_var_noise': prm['likelihood.log_var_noise'].grad,
           'raw_outputscale': prm['covariance_function.raw_outputscale'].grad,
           'raw_lengthscale': prm['covariance_function.base_kernel.raw_lengthscale'].grad}
    # the reference on the model's own (float32) parameter values, in float64 and in float32
    q = dict(Z=prm['Z'][0], raw_lengthscale=prm['covariance_function.base_kernel.raw_lengthscale'].view(-1),
             raw_outputscale=prm['covariance_function.raw_outputscale'].view(()), m=prm['q_U.variational_mean'][0],
             L_raw=prm['q_U.chol_variational_covar'][0], log_var_noise=prm['likelihood.log_var_noise'].view(()), flow=[],
             kernel='rbf')
    q = {k: (v.detach().cpu().double() if torch.is_tensor(v) else v) for k, v in q.items()}

    def reference(dt):
        qd = _to(q, dt)
        E, _, _, _, gr = MR.elbo_and_grads(X32.to(dt), y32.to(dt), qd, N, 'gauss_linear', 0)
        out = {k: gr[k] for k in ('Z', 'm', 'L_raw', 'log_var_noise', 'raw_outputscale', 'raw_lengthscale')}
        out.update(ELBO=E, X=IR.elbo_grads_xz(X32.to(dt), y32.to(dt), qd, N, 'gauss_linear', 0)[1])
        return out
    ref, ref32 = reference(torch.float64), reference(torch.float32)
    errs = {k: rel_err(t.detach().double().cpu(), ref[k]) for k, t in got.items()}
    record_residuals('row_chunks_float32_model_d64', errs)
    bad = _yardstick(errs, ref, ref32)
    assert not bad, (bad, errs)
