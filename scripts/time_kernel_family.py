"""Cost of the covariance function: RBF against ARD-Matern (nu = 1/2, 3/2, 5/2) on bench.py's cfg4 / cfg5 problems.

For each workload and compute mode, the four kernels are timed alternately in one process on the same seeded minibatch:
  - step: one ELBO forward + backward (the step of bench.py), median over --steps CUDA-event-timed steps after --warmup;
  - K generation and kernel gradients: device time per row chunk of the kernels that generate K_xz tiles
    (k_rbf_tile_reg / k_rbf_planes / k_rbf_residues) and of k_kernel_grads (K_xz and K_zz), from torch.profiler over
    --prof-steps further steps, divided by the number of launches.
Device name and power limit are read in the same run.  Writes one JSON file (--out) and prints a table.

    python scripts/time_kernel_family.py --out profiles/r03_kernel_family.json
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

KINDS = ['rbf', 'matern12', 'matern32', 'matern52']
KGEN = ('k_rbf_tile_reg', 'k_rbf_planes', 'k_rbf_residues', 'k_rbf_tile')


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workloads', default='cfg4,cfg5')
    ap.add_argument('--modes', default='i8crt,f64,tf32x3')
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--rounds', type=int, default=2, help='alternations of the four kernels')
    ap.add_argument('--prof-steps', type=int, default=2)
    ap.add_argument('--out', required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this script measures GPU time only')
    bench = load_bench()
    from tgp.pytorch_b200 import functional as Fn
    from tgp.pytorch_b200.engine import Engine
    dev = torch.device('cuda', 0)
    result = dict(info=device_info(), results=[])
    for wname in args.workloads.split(','):
        wl = bench.WORKLOADS[wname]
        gen = torch.Generator().manual_seed(1234)
        n = 4 * wl['batch']
        X, Y = bench.synth(wl, n, gen)
        p = bench.param_state(wl, X, gen)
        xb, yb = X[:wl['batch']].to(dev).contiguous(), Y.view(-1)[:wl['batch']].to(dev).contiguous()
        scale = wl['N'] / float(wl['batch'])
        for mode in args.modes.split(','):
            steps = {}
            for kind in KINDS:
                eng0, t = bench.build_engine(p, wl, dev, mode)
                eng = Engine(wl['M'], wl['D'], wl['likelihood'], eng0.n_quad, eng0.flow, dev, compute=mode, kernel=kind)
                leaves = [t['Z'], t['raw_ls'], t['raw_os'], t['m'], t['L_raw'], t['log_var_noise'], t['theta']]
                for x in leaves:
                    if x is not None:
                        x.requires_grad_(True)

                def step(eng=eng, leaves=leaves):
                    for x in leaves:
                        if x is not None:
                            x.grad = None
                    terms = Fn.elbo_terms(eng, xb, yb, scale, *leaves, None, check_status=True)
                    (-(terms[0] - terms[1])).backward()
                steps[kind] = (step, [])
            for _ in range(args.rounds):
                for kind in KINDS:
                    step, times = steps[kind]
                    for _ in range(args.warmup):
                        step()
                    torch.cuda.synchronize()
                    for _ in range(args.steps):
                        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a.record()
                        step()
                        b.record()
                        b.synchronize()
                        times.append(a.elapsed_time(b))
            for kind in KINDS:
                step, times = steps[kind]
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(args.prof_steps):
                        step()
                    torch.cuda.synchronize()
                kg = dict(ms=0.0, n=0)
                gr = dict(ms=0.0, n=0)
                for ev in prof.key_averages():
                    name = ev.key
                    dt = getattr(ev, 'device_time_total', None)
                    if dt is None:
                        dt = ev.cuda_time_total
                    if any(k in name for k in KGEN):
                        kg['ms'] += dt / 1000.0
                        kg['n'] += ev.count
                    elif 'k_kernel_grads' in name:
                        gr['ms'] += dt / 1000.0
                        gr['n'] += ev.count
                row = dict(workload=wname, mode=mode, kernel=kind, step_ms_median=statistics.median(times),
                           step_ms_min=min(times), step_ms_max=max(times), n_steps=len(times),
                           kgen_ms_per_launch=kg['ms'] / max(kg['n'], 1), kgen_launches_per_step=kg['n'] / args.prof_steps,
                           kgrad_ms_per_launch=gr['ms'] / max(gr['n'], 1), kgrad_launches_per_step=gr['n'] / args.prof_steps)
                result['results'].append(row)
                print('%s %-6s %-8s step %.3f ms (min %.3f max %.3f)  K-gen %.3f ms x %.0f  k_kernel_grads %.3f ms x %.0f' % (
                    wname, mode, kind, row['step_ms_median'], row['step_ms_min'], row['step_ms_max'], row['kgen_ms_per_launch'],
                    row['kgen_launches_per_step'], row['kgrad_ms_per_launch'], row['kgrad_launches_per_step']), flush=True)
    print(json.dumps(result['info']))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
