"""Edge cases of the CUDA path against the oracle on seeded random problems: ragged / tiny batches, inducing-point
counts around the 64-row Cholesky blocks and 128-wide GEMM tiles, input dimensions across the kernel-gradient
specialisations, multi-output models with shared / per-output parameters."""
import pytest
import torch

from oracle import tgp_oracle as O
from tests.golden_util import rel_err
from tests.test_gpu_matern import _to

pytestmark = pytest.mark.gpu
EDGE_TOL = 1e-10      # north_star's FP64 tolerance, values and gradients alike (measured: see profiles/r02_parity_residuals.json)


def _tol(p):
    """1e-10, widened only where the problem itself cannot carry it: a = L^-1 k and the gradients through L^-T carry
    ~eps * cond(L) = eps * sqrt(cond(K_zz)) of forward error in ANY FP64 evaluation; one of the random tiny problems
    below (D = 1, five inducing points on a line) has cond(K_zz) = 2e12."""
    return max(EDGE_TOL, 100.0 * 2.2e-16 * _cond(p) ** 0.5)


def _cond(p):
    with torch.no_grad():
        return float(torch.linalg.cond(O.rbf_ard(p['Z'], p['Z'], p['raw_lengthscale'], p['raw_outputscale'])))


def _tol32(p, e32):
    """'tf32x3': the FP32 bound of tests/test_gpu_matern.py, 1e-5 + 4 x e32 (e32: the oracle's own float32 evaluation against
    its float64 one), widened as _tol where the problem cannot carry it.  The FP32 planes of L^-1 leave ~eps32 * sqrt(cond(K_zz))
    of error in a = L^-1 k; at cond(K_zz) = 2e12 (the D = 1 problem) that is 0.17, and K_zz is singular in float32, so the
    oracle's float32 run adds jitter and no longer evaluates the same problem (measured: 5.5e-2 on dm against e32 = 6e-5)."""
    return max(1e-5 + 4.0 * e32, 1.19e-7 * _cond(p) ** 0.5)
DEV = 'cuda:0'


def _problem(R, M, D, seed, flow=True):
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    X = torch.randn(R, D, generator=g, dtype=f64)
    y = torch.randn(R, generator=g, dtype=f64)
    p = dict(Z=torch.randn(M, D, generator=g, dtype=f64),
             raw_lengthscale=O.inv_softplus(1.0 + 2.0 * torch.rand(D, generator=g, dtype=f64)) ,
             raw_outputscale=O.inv_softplus(torch.tensor(1.3, dtype=f64)),
             m=torch.randn(M, generator=g, dtype=f64),
             L_raw=0.6 * torch.eye(M, dtype=f64) + 0.05 * torch.randn(M, M, generator=g, dtype=f64),
             log_var_noise=torch.tensor(-1.2, dtype=f64))
    if flow:
        steps = [tuple(0.3 * torch.randn((), generator=g, dtype=f64) for _ in range(4)) for _ in range(2)]
        p['flow'] = [('tanh_step', steps, True), ('affine', torch.tensor(0.9, dtype=f64), torch.tensor(0.1, dtype=f64), False),
                     ('sal', torch.tensor(0.2, dtype=f64), torch.tensor(1.1, dtype=f64), False, False)]
    else:
        p['flow'] = []
    return X, y, p


def _cuda(X, y, p, N, lik, nq, compute):
    """(ELBO, rows and every gradient of the CUDA path, flow-parameter names)."""
    from tests.gpu_util import engine_inputs, make_engine
    from tgp.pytorch_b200 import functional as Fn
    eng, theta, rowp, names = make_engine(p, lik, nq, DEV, compute=compute)
    ei = engine_inputs(p, DEV)
    leaves = [ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'], ei['log_var_noise'], theta]
    for t in leaves:
        t.requires_grad_(True)
    scale = N / X.shape[0]
    ELL, KLD, rows, mu, v = Fn.elbo_terms(eng, X.to(DEV).contiguous(), y.to(DEV).contiguous(), scale, *leaves[:6], theta, None)
    (ELL - KLD).backward()
    out = {'ELBO': (ELL - KLD).detach().cpu(), 'rows': rows.cpu(), 'Z': ei['Z'].grad.cpu(), 'ls': ei['raw_ls'].grad.cpu(),
           'os': ei['raw_os'].grad.cpu().view(()), 'm': ei['m'].grad.cpu(), 'L': ei['L_raw'].grad.cpu(),
           'noise': ei['log_var_noise'].grad.cpu().view(())}
    if theta.numel():
        out['theta'] = theta.grad.cpu()
    return out, names


def _oracle(X, y, p, N, lik, nq, names):
    """The oracle's values under the keys of _cuda (in the dtype of X and p)."""
    E, _, _, rows_o, gr = O.elbo_and_grads(X, y, p, N, lik, nq)
    out = {'ELBO': E, 'rows': rows_o, 'Z': gr['Z'], 'ls': gr['raw_lengthscale'], 'os': gr['raw_outputscale'], 'm': gr['m'],
           'L': gr['L_raw'], 'noise': gr['log_var_noise']}
    if names:
        out['theta'] = torch.stack([gr[n].reshape(()) for n in names])
    return out


def _cuda_vs_oracle(X, y, p, N, lik='gauss_nonlinear', nq=30, compute='f64'):
    got, names = _cuda(X, y, p, N, lik, nq, compute)
    ref = _oracle(X, y, p, N, lik, nq, names)
    return {k: rel_err(got[k], ref[k]) for k in got}


@pytest.mark.parametrize('R,M,D', [(1, 5, 1), (3, 1, 2), (130, 63, 3), (257, 65, 4), (64, 128, 8), (300, 129, 5),
                                     (1000, 200, 13), (77, 257, 16), (50, 40, 33), (40, 30, 64)])
@pytest.mark.parametrize('compute', ['f64', 'i8crt', 'tf32x3'])
def test_shapes_around_tile_and_block_boundaries(R, M, D, compute):
    """Every mode: ragged row counts, M around the 64 / 128 / 256 tile and block sizes, D beyond the register-resident K
    generators (D > 32: 'i8crt' falls back to staged K generation and keeps an FP64 K_xz for the kernel gradients; D >= 53:
    the K generation of 'tf32x3' needs more than 48 KiB of shared memory).  'tf32x3' is held to the FP32 bound _tol32."""
    X, y, p = _problem(R, M, D, seed=R * 7 + M * 3 + D)
    got, names = _cuda(X, y, p, 10.0 * R, 'gauss_nonlinear', 30, compute)
    ref = _oracle(X, y, p, 10.0 * R, 'gauss_nonlinear', 30, names)
    err = {k: rel_err(got[k], ref[k]) for k in got}
    from tests.conftest import record_residuals
    record_residuals('edge_shapes[%s]' % compute, err)
    if compute == 'tf32x3':
        ref32 = _oracle(X.float(), y.float(), _to(p, torch.float32), 10.0 * R, 'gauss_nonlinear', 30, names)
        bad = {k: (e, rel_err(ref32[k], ref[k])) for k, e in err.items() if not e < _tol32(p, rel_err(ref32[k], ref[k]))}
    else:
        bad = {k: e for k, e in err.items() if not e < _tol(p)}
    assert not bad, (bad, err)


def test_input_dimension_beyond_kernel_gradient_specialisations_is_refused():
    X, y, p = _problem(20, 10, 65, seed=5)
    with pytest.raises(ValueError, match='dimension'):
        _cuda_vs_oracle(X, y, p, N=100.0)


def test_svgp_closed_form_ragged():
    X, y, p = _problem(333, 70, 6, seed=9, flow=False)
    err = _cuda_vs_oracle(X, y, p, N=5000.0, lik='gauss_linear', nq=0)
    assert all(e < 1e-9 for e in err.values()), err


@pytest.mark.parametrize('shared', [False, True])
def test_two_output_model_matches_sum_of_single_output_oracles(shared):
    """Dy = 2 (the reference's batched multi-output path, sparse_MF_SP.py:292-345): independent GPs per output, with
    either per-output or shared Z / kernel / q(u)."""
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    cg.device = DEV
    from tgp.pytorch_b200.dsp.models import instance_kernel, sparse_MF_SP
    from tgp.pytorch_b200.dsp.likelihoods import GaussianNonLinearMean
    from tgp.pytorch_b200.dsp.flows import SAL
    g = torch.Generator().manual_seed(3)
    R, M, D, Dy = 150, 24, 3, 2
    X = torch.randn(R, D, generator=g, dtype=torch.float64)
    Y = torch.randn(R, Dy, generator=g, dtype=torch.float64)
    K = instance_kernel('scale_rbf', ard_num_dim=D, num_multioutput=Dy, kernel_is_shared=shared,
                        init_params={'length_scale': 1.5, 'kernel_scale': 1.2})
    lik = GaussianNonLinearMean(out_dim=Dy, noise_init=0.3, noise_is_shared=False, quadrature_points=40)
    torch.manual_seed(0)
    model = sparse_MF_SP(['zero', K], X, X[:M].clone(), 1000.0, lik, Dy, True, shared, False, shared, shared,
                         [SAL(1, init_random=True), SAL(1, init_random=True)], 'single', 0.0, False,
                         {'variational_distribution': {'variance_scale': 0.3, 'mean_scale': 0.2}}).to(DEV)
    with torch.no_grad():
        model.Z.add_(0.1 * torch.randn(model.Z.shape, generator=g, dtype=torch.float64).to(DEV))
        model.q_U.variational_mean.add_(torch.randn(model.q_U.variational_mean.shape, generator=g, dtype=torch.float64).to(DEV))
    ELBO, ELL, KLD = model.ELBO(X.to(DEV), Y.to(DEV))
    ELBO.backward()
    total, gZ = 0.0, []
    for dy in range(Dy):
        zi = 0 if shared else dy
        fl = model.G_matrix[dy].flow_arr
        p = dict(Z=model.Z[zi].detach().cpu().clone(),
                 raw_lengthscale=model.covariance_function.base_kernel.raw_lengthscale[zi, 0].detach().cpu().clone(),
                 raw_outputscale=model.covariance_function.raw_outputscale[zi].detach().cpu().clone(),
                 m=model.q_U.variational_mean[zi].detach().cpu().clone(),
                 L_raw=model.q_U.chol_variational_covar[zi].detach().cpu().clone(),
                 log_var_noise=lik.log_var_noise[dy, 0].detach().cpu().clone(),
                 flow=[('sal', fl[0].a.detach().cpu().clone(), fl[0].b.detach().cpu().clone(), False, False),
                       ('affine', fl[1].a.detach().cpu().clone(), fl[1].b.detach().cpu().clone(), False)])
        E, _, _, _, gr = O.elbo_and_grads(X, Y[:, dy].contiguous(), p, 1000.0, 'gauss_nonlinear', 40)
        total = total + E
        gZ.append(gr['Z'])
    assert rel_err(ELBO.detach().cpu(), total) < 1e-10
    ref_gZ = (gZ[0] + gZ[1]).unsqueeze(0) if shared else torch.stack(gZ)
    assert rel_err(model.Z.grad.cpu(), ref_gZ) < EDGE_TOL


@pytest.mark.parametrize('chunk', [128, 384])
def test_batch_contractions_in_several_ragged_row_chunks(chunk):
    """The FP64 batch contractions run in launches of `TGP_OPT_ROW_CHUNK` rows (32768 by default, i.e. a single launch for
    every small fixture).  Force several launches with a ragged last one: forward, kept K_xz, backward staging and the
    accumulation over chunks must reproduce the oracle."""
    from tgp.pytorch_b200 import _lib
    lib = _lib.load()
    X, y, p = _problem(1000, 96, 5, seed=11)
    try:
        _lib.check(lib.tgp_set_option(_lib.OPT_ROW_CHUNK, chunk), 'tgp_set_option')
        err = _cuda_vs_oracle(X, y, p, N=25000.0)
    finally:
        _lib.check(lib.tgp_set_option(_lib.OPT_ROW_CHUNK, 32768), 'tgp_set_option')
    from tests.conftest import record_residuals
    record_residuals('edge_row_chunks', err)
    bad = {k: e for k, e in err.items() if not e < _tol(p)}
    assert not bad, (bad, err)
    assert lib.tgp_set_option(_lib.OPT_ROW_CHUNK, 1) != 0            # refused: below one GEMM tile
