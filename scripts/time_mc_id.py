"""Cost of input-dependent flows under the Monte-Carlo softmax likelihood (multiclass ID-TGP) against global flows.

  - kernel: CUDA-event time of one Monte-Carlo softmax call with gradients (k_row_mc_softmax) at R rows and S samples, for
    SAL(1) flows with global parameters (tgp_mc_softmax_rows) and with per-row sinh-arcsinh parameters
    (tgp_mc_softmax_rows_rowp, its <true> instantiation), at C = 3 and 10;
  - step: one ELBO forward + backward of `sparse_MF_SP` with `MulticlassCategorical` and SAL(1) flows per class, input-dependent
    (MLPs with MC dropout through the fused MLP kernels) against the same model with global flows, noise drawn every step.
Medians over --reps timed calls after --warmup, the two variants alternated --rounds times in one process.  Device name and
power limit are read in the same run.  Writes <out>.json and <out>.txt.

    python scripts/time_mc_id.py --out profiles/r07_mc_id
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import warnings

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # reported, not hidden: a number without its power limit is incomplete
        q = 'unavailable (%s)' % e
    return dict(device=name, power_limit_and_max_sm_clock=q)


def timed(fn, reps):
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return out


def kernel_calls(Cn, R, S, dev):
    """{variant: zero-argument launcher} for the global and the per-row SAL(1) flow on the same inputs."""
    import ctypes as C
    from tgp.pytorch_b200 import _lib
    from tgp.pytorch_b200.engine import FlowLayout
    from tgp.pytorch_b200.dsp.likelihoods._rows import _mc_model
    lib = _lib.load()
    g = torch.Generator(device=dev).manual_seed(Cn)
    d = dict(dtype=torch.float64, device=dev)
    mu, v = 0.5 * torch.randn(Cn, R, generator=g, **d), 0.1 + torch.rand(Cn, R, generator=g, **d)
    y = torch.randint(0, Cn, (R,), generator=g, device=dev).double()
    eps = torch.randn(S, Cn, R, generator=g, **d)
    rows, g_mu, g_v = torch.empty(R, **d), torch.empty(Cn, R, **d), torch.empty(Cn, R, **d)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    glob = FlowLayout([dict(kind='sal'), dict(kind='affine')])
    perrow = FlowLayout([dict(kind='sal', per_row=True), dict(kind='affine')])
    th4 = torch.tensor([0.1, 0.9, 1.1, 0.05], **d).repeat(Cn, 1).contiguous()
    th2 = th4[:, 2:].contiguous()
    rowp = torch.stack([0.1 + 0.2 * torch.randn(Cn, R, generator=g, **d), 0.9 + 0.1 * torch.randn(Cn, R, generator=g, **d)], -1)
    drowp = torch.empty_like(rowp)
    dth4, dth2 = torch.zeros_like(th4), torch.zeros_like(th2)
    md_g, md_r = _mc_model(glob), _mc_model(perrow)
    common = (mu.data_ptr(), v.data_ptr(), y.data_ptr(), eps.data_ptr())

    def run_global():
        _lib.check(lib.tgp_mc_softmax_rows(md_g, Cn, S, R, *common, th4.data_ptr(), 1, rows.data_ptr(), g_mu.data_ptr(),
                                           g_v.data_ptr(), dth4.data_ptr(), None, st), 'tgp_mc_softmax_rows')

    def run_per_row():
        _lib.check(lib.tgp_mc_softmax_rows_rowp(md_r, Cn, S, R, *common, th2.data_ptr(), 1, rows.data_ptr(), g_mu.data_ptr(),
                                                g_v.data_ptr(), dth2.data_ptr(), None, rowp.data_ptr(), drowp.data_ptr(), st),
                   'tgp_mc_softmax_rows_rowp')
    return {'global': run_global, 'per_row': run_per_row}


def model_steps(Cn, MB, M, D, S, H, dev):
    """{variant: one ELBO forward + backward} for SAL(1) flows with global and with input-dependent parameters."""
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    cg.device = dev
    cg.quad_points = S
    from tgp.pytorch_b200.dsp import flows as F
    from tgp.pytorch_b200.dsp.models import instance_kernel, sparse_MF_SP
    from tgp.pytorch_b200.dsp.models.flow import instance_flow
    from tgp.pytorch_b200.dsp.likelihoods import MulticlassCategorical
    g = torch.Generator().manual_seed(7)
    X = torch.randn(MB, D, generator=g, dtype=torch.float64)
    Y = torch.randint(0, Cn, (MB, 1), generator=g).double()
    steps = {}
    for variant in ('global', 'per_row'):
        torch.manual_seed(1)
        K = instance_kernel('scale_rbf', ard_num_dim=D, num_multioutput=Cn, kernel_is_shared=False,
                            init_params={'length_scale': 2.0, 'kernel_scale': 2.0, 'noisy_variance': 1e-6})
        flows = []
        for _ in range(Cn):
            if variant == 'global':
                fl = instance_flow(F.SAL(1))
            else:
                fl = instance_flow(F.SAL(1, input_dependent=True, input_dim=D, hidden_dim=H, num_hidden_layers=1,
                                         hidden_activation='relu', dropout=0.25, inference='MC_dropout', batch_norm=0))
                fl.turn_off_initializer_parameters()
            flows.append(fl)
        ip = {'variational_distribution': {'variance_scale': 1e-2, 'mean_scale': 0.0}}
        model = sparse_MF_SP(['zero', K], X, X[:M].clone(), 10 * MB, MulticlassCategorical(Cn), Cn, True, False, False, False,
                             False, flows, 'single', 0.0, False, ip).to(dev)
        Xd, Yd = X.to(dev), Y.to(dev)

        def step(model=model, Xd=Xd, Yd=Yd):
            model.zero_grad(set_to_none=True)
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                (-model.ELBO(Xd, Yd)[0]).backward()
        steps[variant] = step
    return steps


def alternate(fns, warmup, reps, rounds):
    times = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            for _ in range(warmup):
                fn()
            torch.cuda.synchronize()
            times[k].extend(timed(fn, reps))
    return {k: dict(ms_median=statistics.median(t), ms_min=min(t), ms_max=max(t), n=len(t)) for k, t in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rows', type=int, default=65536)
    ap.add_argument('--samples', type=int, default=100)
    ap.add_argument('--classes', default='3,10')
    ap.add_argument('--step-classes', type=int, default=10)
    ap.add_argument('--step-rows', type=int, default=8192)
    ap.add_argument('--step-M', type=int, default=256)
    ap.add_argument('--step-D', type=int, default=8)
    ap.add_argument('--step-hidden', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', required=True, help='path without extension: writes .json and .txt')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this script measures GPU time only')
    dev = torch.device('cuda', 0)
    from tgp.pytorch_b200.dsp import config as cg
    result = dict(info=device_info(), kernel=[], step=None)
    lines = []
    for Cn in [int(c) for c in args.classes.split(',')]:
        t = alternate(kernel_calls(Cn, args.rows, args.samples, dev), args.warmup, args.reps, args.rounds)
        result['kernel'].append(dict(C=Cn, R=args.rows, S=args.samples, flow='SAL(1)', **{k: v for k, v in t.items()}))
        lines.append('kernel C=%d R=%d S=%d SAL(1): global %.3f ms, per-row %.3f ms (x%.2f)' % (
            Cn, args.rows, args.samples, t['global']['ms_median'], t['per_row']['ms_median'],
            t['per_row']['ms_median'] / t['global']['ms_median']))
        print(lines[-1], flush=True)
        torch.cuda.empty_cache()
    t = alternate(model_steps(args.step_classes, args.step_rows, args.step_M, args.step_D, args.samples, args.step_hidden, dev),
                  args.warmup, args.reps, args.rounds)
    result['step'] = dict(C=args.step_classes, MB=args.step_rows, M=args.step_M, D=args.step_D, S=args.samples,
                          mlp='1 x %d relu, dropout 0.25' % args.step_hidden, compute=cg.compute, **t)
    lines.append('step C=%d MB=%d M=%d D=%d S=%d (%s): global %.3f ms, ID %.3f ms (x%.2f)' % (
        args.step_classes, args.step_rows, args.step_M, args.step_D, args.samples, cg.compute, t['global']['ms_median'],
        t['per_row']['ms_median'], t['per_row']['ms_median'] / t['global']['ms_median']))
    print(lines[-1])
    lines.append('device: %(device)s, power limit / max SM clock: %(power_limit_and_max_sm_clock)s' % result['info'])
    print(lines[-1])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out + '.json', 'w') as f:
        json.dump(result, f, indent=1)
    with open(args.out + '.txt', 'w') as f:
        f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
