"""Cost of the full q(f) covariance over a test batch, its Cholesky factor and joint samples (DESIGN section 5, README).

For each configuration (M, D, kernel) and batch size R, one engine in compute mode 'f64' is prepared once, then CUDA events
after --warmup calls time, as the median over --reps calls:
  - qf_cov   tgp_qf_cov_forward: K_xz, [A | B], mu, the lower half of -A A^T + B B^T, k_cov_assemble;
  - chol     tgp_cov_cholesky of Sigma + 1e-6 s I;
  - sample   tgp_cov_sample with S = 100.
Achieved FP64 rates use shape-derived operation counts: R (R + 1) 2M for the Sigma product (lower half), R^3 / 3 for the
factor and S R (R + 1) for the samples.  In the same process torch does the same three steps on the GPU as a yardstick:
B B^T - A A^T with matmul (full product), torch.linalg.cholesky, mu + eps L^T.  Device name and power limit are read in
the same run.  Writes <out>.json and <out>.txt.

    python scripts/time_joint_posterior.py --out profiles/r04_joint_posterior
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

CONFIGS = [(1024, 8, 'rbf'), (1024, 8, 'matern52'), (2048, 16, 'rbf')]
S_SAMPLES = 100


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # reported, not hidden: a number without its power limit is incomplete
        q = 'unavailable (%s)' % e
    return dict(device=name, power_limit_and_max_sm_clock=q)


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return statistics.median(ms)


def problem(M, D, kernel, R, seed=7):
    from tgp.pytorch_b200.engine import Engine, FlowLayout
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    X = torch.randn(R, D, generator=g, dtype=f64)
    Z = torch.randn(M, D, generator=g, dtype=f64)
    dev = 'cuda:0'
    raw_ls = torch.full((D,), float(torch.log(torch.expm1(torch.tensor(1.5 * (D / 8.0) ** 0.5)))), dtype=f64)
    raw_os = torch.tensor([0.5], dtype=f64)
    m = torch.randn(M, generator=g, dtype=f64)
    L_raw = 0.3 * torch.eye(M, dtype=f64) + 0.01 * torch.randn(M, M, generator=g, dtype=f64)
    eng = Engine(M, D, 'gauss_linear', 0, FlowLayout([]), dev, compute='f64', kernel=kernel)
    params = [t.to(dev).contiguous() for t in (Z, raw_ls, raw_os, m, L_raw)]
    return eng, X.to(dev).contiguous(), params


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rows', default='1024,4096,16384')
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', required=True, help='output path without extension')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this script measures GPU time only')
    from tgp.pytorch_b200 import functional as Fn
    info = device_info()
    rows = []
    for M, D, kernel in CONFIGS:
        for R in [int(r) for r in args.rows.split(',')]:
            eng, X, params = problem(M, D, kernel, R)
            with torch.no_grad():
                mu, cov = Fn.qf_covariance(eng, X, *params)
            s = float(torch.nn.functional.softplus(params[2]))
            jit = 1e-6 * s
            L, status = eng.cov_cholesky(cov, jit)
            assert int(status.item()) == 0, 'the timed factorisation must succeed'
            eps = torch.randn(S_SAMPLES, R, dtype=torch.float64, device='cuda:0')
            t_cov = timed(lambda: eng.qf_cov(X), args.warmup, args.reps)
            t_chol = timed(lambda: eng.cov_cholesky(cov, jit), args.warmup, args.reps)
            t_smp = timed(lambda: eng.cov_sample(mu, L, eps), args.warmup, args.reps)
            # torch yardstick on the same device: the same products / factorisation / samples
            A = torch.randn(R, M, dtype=torch.float64, device='cuda:0')
            B = torch.randn(R, M, dtype=torch.float64, device='cuda:0')
            Sj = cov + jit * torch.eye(R, dtype=torch.float64, device='cuda:0')
            tt_prod = timed(lambda: B @ B.t() - A @ A.t(), args.warmup, args.reps)
            tt_chol = timed(lambda: torch.linalg.cholesky(Sj), args.warmup, args.reps)
            tt_smp = timed(lambda: mu.view(1, -1) + eps @ L.t(), args.warmup, args.reps)
            f_prod, f_chol, f_smp = R * (R + 1) * 2.0 * M, R ** 3 / 3.0, S_SAMPLES * R * (R + 1.0)
            row = dict(M=M, D=D, kernel=kernel, R=R, S=S_SAMPLES, qf_cov_ms=t_cov, cov_cholesky_ms=t_chol, cov_sample_ms=t_smp,
                       torch_product_ms=tt_prod, torch_cholesky_ms=tt_chol, torch_sample_ms=tt_smp,
                       qf_cov_product_tflops=f_prod / t_cov * 1e-9, cov_cholesky_tflops=f_chol / t_chol * 1e-9,
                       cov_sample_tflops=f_smp / t_smp * 1e-9, torch_cholesky_tflops=f_chol / tt_chol * 1e-9)
            rows.append(row)
            print(json.dumps(row), flush=True)
            del eng, cov, L, Sj, A, B
            torch.cuda.empty_cache()
    out = dict(info, warmup=args.warmup, reps=args.reps, statistic='median of CUDA-event-timed calls', rows=rows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out + '.json', 'w') as f:
        json.dump(out, f, indent=1)
    lines = ['# full q(f) covariance, Cholesky and joint samples (FP64), %s, %s' % (info['device'], info['power_limit_and_max_sm_clock']),
             '# median of %d CUDA-event-timed calls after %d warm-up calls; TF/s from shape-derived counts (lower-half Sigma '
             'product R(R+1)2M, factor R^3/3, samples S R(R+1))' % (args.reps, args.warmup),
             '%5s %3s %-9s %6s | %9s %7s | %9s %7s | %9s | %9s %9s %9s' % ('M', 'D', 'kernel', 'R', 'qf_cov ms', 'TF/s', 'chol ms',
                                                                       'TF/s', 'sample ms', 'torch AAT', 'torch chol', 'torch smp')]
    for r in rows:
        lines.append('%5d %3d %-9s %6d | %9.3f %7.2f | %9.3f %7.2f | %9.3f | %9.3f %9.3f %9.3f' % (
            r['M'], r['D'], r['kernel'], r['R'], r['qf_cov_ms'], r['qf_cov_product_tflops'], r['cov_cholesky_ms'],
            r['cov_cholesky_tflops'], r['cov_sample_ms'], r['torch_product_ms'], r['torch_cholesky_ms'], r['torch_sample_ms']))
    with open(args.out + '.txt', 'w') as f:
        f.write('\n'.join(lines) + '\n')
    print('\n'.join(lines))


if __name__ == '__main__':
    main()
