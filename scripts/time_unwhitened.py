"""Cost of the non-whitened q(u) (TGP_QU_UNWHITENED) against the whitened one on bench.py's cfg4 / cfg5 problems.

For each workload and compute mode the two forms are timed alternately in one process on the same seeded minibatch and
parameters (the non-whitened model reads bench.py's m and L_raw as its own):
  - step: one ELBO forward + backward (the step of bench.py), median over --steps CUDA-event-timed steps after --warmup;
  - prepare / chain: CUDA-event time of tgp_prepare and of tgp_chain_backward alone (medians over --stage-reps calls), with
    TGP_OPT_OVERLAP_KGEN off for these calls so that the whole factorisation runs on the timed stream.
Device name and power limit are read in the same run.  Writes one JSON file (--out) and prints a table.

    python scripts/time_unwhitened.py --out profiles/r05_unwhitened.json
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

FORMS = [('whitened', True), ('unwhitened', False)]


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
    ap.add_argument('--rounds', type=int, default=2, help='alternations of the two forms')
    ap.add_argument('--stage-reps', type=int, default=10)
    ap.add_argument('--out', required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this script measures GPU time only')
    bench = load_bench()
    from tgp.pytorch_b200 import _lib
    from tgp.pytorch_b200 import functional as Fn
    from tgp.pytorch_b200.engine import Engine
    lib = _lib.load()
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
            runs = {}
            for form, whiten in FORMS:
                eng0, t = bench.build_engine(p, wl, dev, mode)
                eng = Engine(wl['M'], wl['D'], wl['likelihood'], eng0.n_quad, eng0.flow, dev, compute=mode, whiten=whiten)
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
                runs[form] = (eng, step, [])
            for _ in range(args.rounds):
                for form, _ in FORMS:
                    eng, step, times = runs[form]
                    for _ in range(args.warmup):
                        step()
                    torch.cuda.synchronize()
                    times.extend(timed(step, args.steps))
            for form, _ in FORMS:
                eng, step, times = runs[form]
                step()                       # leaves a prepared step workspace and the reduce buffer of its backward
                torch.cuda.synchronize()
                lib.tgp_set_option(_lib.OPT_OVERLAP_KGEN, 0)
                try:
                    prep = timed(lambda: eng.prepare(0.0), args.stage_reps)
                    chain = timed(lambda: eng.chain_backward(eng._rb, 1.0, -1.0), args.stage_reps)
                finally:
                    lib.tgp_set_option(_lib.OPT_OVERLAP_KGEN, 1)
                row = dict(workload=wname, mode=mode, form=form, M=wl['M'], rows=wl['batch'],
                           step_ms_median=statistics.median(times), step_ms_min=min(times), step_ms_max=max(times),
                           n_steps=len(times), prepare_ms_median=statistics.median(prep), chain_ms_median=statistics.median(chain))
                result['results'].append(row)
                print('%s %-6s %-10s step %.3f ms (min %.3f max %.3f)  prepare %.3f ms  chain %.3f ms' % (
                    wname, mode, form, row['step_ms_median'], row['step_ms_min'], row['step_ms_max'], row['prepare_ms_median'],
                    row['chain_ms_median']), flush=True)
    print(json.dumps(result['info']))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
