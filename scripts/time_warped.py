"""Cost of the warped GP (TGP_LIK_GAUSS_WARPED) against SVGP and TGP on bench.py's cfg4 problem (65536 rows, M = 1024, D = 8).

In each compute mode three models are timed alternately in one process on the same seeded minibatch and GP parameters:
  - svgp:   GaussianLinearMean (closed form, no flow);
  - warped: the warped likelihood with bench.py's StepTanhL(1,3) flow as the warp G(y) (closed form + second-order flow sweep);
  - tgp:    bench.py's workload, StepTanhL(1,3) on f under 100-point Gauss-Hermite.
step = one ELBO forward + backward, median over --steps CUDA-event-timed steps after --warmup, per round.  On the warped and TGP
engines the row epilogue alone (k_row_warped / k_row_quad: tgp_ell_forward with gradients) and the test rows with predictive
moments (k_row_test, 100 Gauss-Hermite nodes with a Newton inverse each for the warped model) are timed over --stage-reps calls.
Device name and power limit are read in the same run.  Writes one JSON file (--out) and prints a table.

    python scripts/time_warped.py --out profiles/r07_warped.json
"""
import argparse
import importlib.util
import json
import os
import statistics
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

MODELS = [('svgp', 'gauss_linear'), ('warped', 'gauss_warped'), ('tgp', 'gauss_nonlinear')]


def load_bench():
    spec = importlib.util.spec_from_file_location('tgp_bench', os.path.join(ROOT, 'bench.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--modes', default='i8crt,f64,tf32x3')
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--rounds', type=int, default=3, help='alternations of the three models')
    ap.add_argument('--stage-reps', type=int, default=20)
    ap.add_argument('--out', required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this script measures GPU time only')
    bench = load_bench()
    from tgp.pytorch_b200 import functional as Fn
    from tgp.pytorch_b200.engine import Engine, FlowLayout
    dev = torch.device('cuda', 0)
    wl = bench.WORKLOADS['cfg4']
    gen = torch.Generator().manual_seed(1234)
    X, Y = bench.synth(wl, 4 * wl['batch'], gen)
    p = bench.param_state(wl, X, gen)
    xb, yb = X[:wl['batch']].to(dev).contiguous(), Y.view(-1)[:wl['batch']].to(dev).contiguous()
    scale = wl['N'] / float(wl['batch'])
    result = dict(info=device_info(), workload='cfg4', rows=wl['batch'], M=wl['M'], D=wl['D'], n_quad=bench.N_QUAD, results=[])
    for mode in args.modes.split(','):
        runs = {}
        for name, lik in MODELS:
            eng0, t = bench.build_engine(p, wl, dev, mode)
            flow = FlowLayout([]) if lik == 'gauss_linear' else eng0.flow
            eng = Engine(wl['M'], wl['D'], lik, 0 if lik == 'gauss_linear' else bench.N_QUAD, flow, dev, compute=mode)
            theta = None if lik == 'gauss_linear' else t['theta']
            leaves = [t['Z'], t['raw_ls'], t['raw_os'], t['m'], t['L_raw'], t['log_var_noise'], theta]
            for x in leaves:
                if x is not None:
                    x.requires_grad_(True)

            def step(eng=eng, leaves=leaves):
                for x in leaves:
                    if x is not None:
                        x.grad = None
                terms = Fn.elbo_terms(eng, xb, yb, scale, *leaves, None, check_status=True)
                (-(terms[0] - terms[1])).backward()
            runs[name] = (eng, step, [], leaves)
        for _ in range(args.rounds):
            for name, _ in MODELS:
                eng, step, times, _ = runs[name]
                for _ in range(args.warmup):
                    step()
                torch.cuda.synchronize()
                times.append(statistics.median(timed(step, args.steps)))
        for name, lik in MODELS:
            eng, step, times, leaves = runs[name]
            row = dict(mode=mode, model=name, likelihood=lik, step_ms_round_medians=times, step_ms_median=statistics.median(times))
            if lik != 'gauss_linear':
                eng.set_params(*[x.detach() for x in leaves])
                with torch.no_grad():
                    eng.prepare(0.0)
                    mu, v = eng.qf_forward(xb)
                    rb = eng.new_reduce_buffer()
                    for _ in range(3):
                        eng.ell_forward(mu, v, yb, None, scale, rb)
                        eng.test_rows(mu, v, yb, None, 1, 1.0)
                    torch.cuda.synchronize()
                    row['ell_rows_ms_median'] = statistics.median(timed(lambda: eng.ell_forward(mu, v, yb, None, scale, rb),
                                                                        args.stage_reps))
                    row['test_rows_with_moments_ms_median'] = statistics.median(
                        timed(lambda: eng.test_rows(mu, v, yb, None, 1, 1.0), args.stage_reps))
                    row['test_rows_nan_moments'] = int(torch.isnan(eng.test_rows(mu, v, yb, None, 1, 1.0)[1]).sum())
            result['results'].append(row)
            print('%-6s %-6s step %.3f ms (round medians %s)%s' % (
                mode, name, row['step_ms_median'], ' '.join('%.3f' % x for x in times),
                '' if lik == 'gauss_linear' else '  ell rows %.4f ms  test rows + moments %.4f ms (NaN rows %d)' % (
                    row['ell_rows_ms_median'], row['test_rows_with_moments_ms_median'], row['test_rows_nan_moments'])),
                flush=True)
    print(json.dumps(result['info']))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
