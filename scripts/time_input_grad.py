"""Cost of the input gradients (dX) on bench.py's cfg4 / cfg5 problems: the backward of one ELBO step with and without
X.requires_grad, in the three compute modes.

For each workload and mode the two arms are timed alternately (--rounds) in one process on the same seeded minibatch and
parameters.  Each timed call is the backward alone: the forward is enqueued and synchronised first, then CUDA events wrap
`.backward()`; medians over --steps calls after --warmup.  The 'dx' arm's backward adds k_input_grads (one pass over each
row chunk's Kbar) and the multiplication by the ELL weight; the other arm launches exactly what a run without input
gradients launches.  Device name and power limit are read in the same run.  Writes one JSON file (--out), prints a table.

    python scripts/time_input_grad.py --out profiles/r06_input_grad.json
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

ARMS = [('no_dx', False), ('dx', True)]


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
    ap.add_argument('--workloads', default='cfg4,cfg5')
    ap.add_argument('--modes', default='i8crt,f64,tf32x3')
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--rounds', type=int, default=2, help='alternations of the two arms')
    ap.add_argument('--out', required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this script measures GPU time only')
    bench = load_bench()
    from tgp.pytorch_b200 import functional as Fn
    dev = torch.device('cuda', 0)
    result = dict(info=device_info(), results=[])
    for wname in args.workloads.split(','):
        wl = bench.WORKLOADS[wname]
        gen = torch.Generator().manual_seed(1234)
        X, Y = bench.synth(wl, 4 * wl['batch'], gen)
        p = bench.param_state(wl, X, gen)
        xb, yb = X[:wl['batch']].to(dev).contiguous(), Y.view(-1)[:wl['batch']].to(dev).contiguous()
        scale = wl['N'] / float(wl['batch'])
        for mode in args.modes.split(','):
            eng, t = bench.build_engine(p, wl, dev, mode)
            leaves = [t['Z'], t['raw_ls'], t['raw_os'], t['m'], t['L_raw'], t['log_var_noise'], t['theta']]
            for x in leaves:
                if x is not None:
                    x.requires_grad_(True)
            times = {arm: [] for arm, _ in ARMS}

            def backward_ms(want_dx):
                Xa = xb.clone().requires_grad_(want_dx)
                for x in leaves:
                    if x is not None:
                        x.grad = None
                terms = Fn.elbo_terms(eng, Xa, yb, scale, *leaves, None, check_status=True)
                loss = -(terms[0] - terms[1])
                torch.cuda.synchronize()
                return timed(loss.backward, 1)[0]
            for _ in range(args.rounds):
                for arm, want_dx in ARMS:
                    for _ in range(args.warmup):
                        backward_ms(want_dx)
                    times[arm].extend(backward_ms(want_dx) for _ in range(args.steps))
            for arm, _ in ARMS:
                ts = times[arm]
                row = dict(workload=wname, mode=mode, arm=arm, M=wl['M'], D=wl['D'], rows=wl['batch'],
                           backward_ms_median=statistics.median(ts), backward_ms_min=min(ts), backward_ms_max=max(ts), n=len(ts))
                result['results'].append(row)
                print('%s %-6s %-5s backward %.3f ms (min %.3f max %.3f)' % (wname, mode, arm, row['backward_ms_median'],
                                                                          row['backward_ms_min'], row['backward_ms_max']), flush=True)
            d = statistics.median(times['dx']) - statistics.median(times['no_dx'])
            print('%s %-6s dX adds %.3f ms to the backward' % (wname, mode, d), flush=True)
    print(json.dumps(result['info']))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
