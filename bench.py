#!/usr/bin/env python
"""bench.py — minibatch ELBO forward+backward throughput of the B200 path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our CUDA path, one process per GPU under torchrun
  python bench.py --impl reference --gpus N ...            # the reference's algorithm on the host CPU cores (oracle port)
  options: --workload cfg4|cfg5   --scaling weak|strong   --compute i8crt|f64|tf32x3

Workloads (SURVEY.md §8d):
  cfg4 (default; BASELINE.json configs[3], the configuration the metric is quoted on): TGP regression, synthetic
       N = 5 M rows, D = 8, M = 1024 inducing points, StepTanhL(1,3) flow, Gaussian likelihood, 100 Gauss-Hermite points;
  cfg5 (configs[4]): TGP binary classification, N = 1 M, D = 16, M = 2048, SAL(1) flow, Bernoulli likelihood, 100 points.
Both with FP64 results (what the reference's main.py runs): the default compute mode `i8crt` evaluates the batch contractions on
the tcgen05 integer tensor pipe through CRT residues (FP64-accurate, parity-tested at 1e-10 like `f64`, the DMMA mode).  One step = ELBO forward + backward over one minibatch:
  weak scaling  (default): 65536 rows PER GPU, global minibatch 65536 * N;
  strong scaling          : 65536 rows in total, 65536 / N per GPU.
The N/MB scale uses the global size; ranks exchange ONE all-reduce of the tril-packed pre-chain gradient buffer per step.

One JSON line on stdout (rank 0).  Keys per the driver contract plus `roofline`, `cpu_baseline`, `dist_parity` (N > 1).
"""
import argparse
import hashlib
import json
import math
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True        # the benchmark writes nothing into the tree it runs from (it may be read-only)

SEED = 1234
N_QUAD = 100
METRIC = 'elbo_fwd_bwd_rows_per_s'
WORKLOADS = {
    'cfg4': dict(N=5_000_000, D=8, M=1024, batch=65536, likelihood='gauss_nonlinear', flow='StepTanhL(1,3)',
                 text='TGP regression synthetic N=5M D=8 M=1024, StepTanhL(1,3), Gaussian lik, 100 GH points (BASELINE configs[3])'),
    'cfg5': dict(N=1_000_000, D=16, M=2048, batch=65536, likelihood='bernoulli', flow='SAL(1)',
                 text='TGP binary classification synthetic N=1M D=16 M=2048, SAL(1), Bernoulli lik, 100 GH points (BASELINE configs[4])'),
}


def synth(wl, n, gen):
    """SURVEY.md §8d synthetic data: regression y = sinh(0.7 Xw / sqrt D) + 0.1 eps (standardised); classification
    y = 1[Phi(Xw / sqrt D) > u]."""
    d = wl['D']
    X = torch.randn(n, d, generator=gen, dtype=torch.float64)
    w = torch.randn(d, generator=gen, dtype=torch.float64)
    if wl['likelihood'] == 'bernoulli':
        pr = 0.5 * (1 + torch.erf((X @ w) / math.sqrt(d) / math.sqrt(2.0)))
        y = (pr > torch.rand(n, generator=gen, dtype=torch.float64)).double()
    else:
        y = torch.sinh(0.7 * (X @ w) / math.sqrt(d)) + 0.1 * torch.randn(n, generator=gen, dtype=torch.float64)
        y = (y - y.mean()) / y.std()
    return X, y.view(-1, 1)


def param_state(wl, X, gen):
    """'Mid-training' state P1 (SURVEY.md §8d): nothing at a trivial value; K_zz stays well conditioned.  Oracle-style
    dict (oracle/tgp_oracle.py), also consumed by `build_engine` below."""
    M, D = wl['M'], wl['D']
    idx = torch.randperm(X.shape[0], generator=gen)[:M]
    inv_sp = lambda t: t + torch.log(-torch.expm1(-t))  # noqa: E731
    f64 = torch.float64
    p = dict(Z=X[idx].clone(),
             raw_lengthscale=inv_sp(1.5 + 1.0 * torch.rand(D, generator=gen, dtype=f64)),
             raw_outputscale=inv_sp(torch.tensor(1.5, dtype=f64)),
             m=torch.randn(M, generator=gen, dtype=f64),
             L_raw=0.5 * torch.eye(M, dtype=f64) + 0.05 * torch.randn(M, M, generator=gen, dtype=f64),
             log_var_noise=torch.log(torch.tensor(0.05, dtype=f64)))
    if wl['flow'] == 'StepTanhL(1,3)':
        steps = []
        for _ in range(3):
            e = torch.randn(4, generator=gen, dtype=f64)
            steps.append((e[0].clone(), inv_sp(torch.abs((e[1] + 1.0) / 3.0) + 1e-3), e[2].clone(),
                          inv_sp(torch.abs((e[3] + 1.0) / 3.0) + 1e-3)))
        p['flow'] = [('tanh_step', steps, True), ('affine', torch.tensor(1.1, dtype=f64), torch.tensor(-0.05, dtype=f64), False)]
    else:   # SAL(1): sinh-arcsinh then affine (reference flows.py:115-136)
        e = torch.randn(2, generator=gen, dtype=f64)
        p['flow'] = [('sal', 0.3 * e[0].clone(), 1.0 + 0.2 * torch.tanh(e[1]), False, False),
                     ('affine', torch.tensor(0.9, dtype=f64), torch.tensor(0.1, dtype=f64), False)]
    return p


def build_engine(p, wl, dev, compute):
    """Oracle-style parameter dict -> (Engine, device parameter tensors in C-ABI order, theta)."""
    from tgp.pytorch_b200.engine import Engine, FlowLayout
    desc, theta = [], []
    for lay in p['flow']:
        if lay[0] == 'affine':
            desc.append(dict(kind='affine', restrict=lay[3]))
            theta += [lay[1], lay[2]]
        elif lay[0] == 'tanh_step':
            desc.append(dict(kind='tanh_step', n_steps=len(lay[1]), add_f0=lay[2]))
            for st in lay[1]:
                theta += list(st)
        elif lay[0] == 'sal':
            desc.append(dict(kind='sal', restrict=lay[3], add_f0=lay[4]))
            theta += [lay[1], lay[2]]
    f = lambda t: t.detach().to(dev).double().contiguous()  # noqa: E731
    eng = Engine(wl['M'], wl['D'], wl['likelihood'], N_QUAD, FlowLayout(desc), dev, compute=compute)
    t = dict(Z=f(p['Z']), raw_ls=f(p['raw_lengthscale'].reshape(-1)), raw_os=f(p['raw_outputscale'].reshape(1)), m=f(p['m']),
             L_raw=f(p['L_raw']), log_var_noise=None if wl['likelihood'] == 'bernoulli' else f(p['log_var_noise'].reshape(1)),
             theta=f(torch.stack([x.reshape(()) for x in theta])))
    return eng, t


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML from a background thread every 100 ms;
    the same fields as the nvidia-smi query of the profiling recipe, without forking nvidia-smi under the load)."""

    def __init__(self, gpu_index):
        self.gpu, self.rows, self._stop, self._thr, self._nvml = gpu_index, [], False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(vis.split(',')[self.gpu]) if vis and vis.split(',')[self.gpu].isdigit() else self.gpu
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._nvml = pynvml
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        except Exception:
            self._nvml = None

    def _loop(self):
        nv = self._nvml
        while not self._stop:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h) if hasattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons') \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                self.rows.append((sm, mx, rs))
            except Exception:
                pass
            time.sleep(0.1)

    def stop(self):
        if self._nvml is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvml unavailable']}
        self._stop = True
        self._thr.join(timeout=1.0)
        nv = self._nvml
        names = {'hw_slowdown': getattr(nv, 'nvmlClocksThrottleReasonHwSlowdown', 0x8),
                 'hw_thermal_slowdown': getattr(nv, 'nvmlClocksThrottleReasonHwThermalSlowdown', 0x40),
                 'sw_thermal_slowdown': getattr(nv, 'nvmlClocksThrottleReasonSwThermalSlowdown', 0x20),
                 'sw_power_cap': getattr(nv, 'nvmlClocksThrottleReasonSwPowerCap', 0x4)}
        reasons = set()
        for _, _, rs in self.rows:
            for n, bit in names.items():
                if rs & bit:
                    reasons.add(n)
        sm = [r[0] for r in self.rows]
        mx = [r[1] for r in self.rows]
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': float(max(mx)) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def measure_gemm_peak(dev, dtype, tf32=False, n=8192, reps=5):
    """cuBLAS GEMM n^3 via torch.matmul, best of `reps` (the method of MEASURED_PEAKS.json, which holds no FP64 / TF32 figure)."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = tf32
    a = torch.randn(n, n, dtype=dtype, device=dev)
    b = torch.randn(n, n, dtype=dtype, device=dev)
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record()  # noqa: E702
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.backends.cuda.matmul.allow_tf32 = old
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def measure_int8_peak(dev, n=8192, reps=5):
    """cuBLASLt INT8 GEMM n^3 via torch._int_mm (s8 x s8 -> s32), best of `reps`, in TOP/s."""
    try:
        a = torch.randint(-64, 64, (n, n), dtype=torch.int8, device=dev)
        b = torch.randint(-64, 64, (n, n), dtype=torch.int8, device=dev)
        torch._int_mm(a, b)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch._int_mm(a, b); e1.record()  # noqa: E702
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    except Exception:          # noqa: BLE001
        return None


def i8crt_executed_ops(M, rows, chunk=16384):
    """Integer operations (2 x MAC) the three residue GEMMs of compute mode i8crt EXECUTE per step: 128 x 256 tiles over their
    clipped k-ranges (csrc/gemm_i8.cuh decode), times the modulus count of each contraction (csrc/crt_driver.cuh)."""
    log2P = {15: 117.82, 16: 125.41}
    bits_other = lambda T, k, fixed: min(53, int(math.floor(log2P[T] - 1.0 - math.log2(max(k, 1)) - fixed - 1e-6)))  # noqa: E731
    Tf = 15 if bits_other(15, M, 53) >= 52 else 16
    Tb = 15 if min(53, int(math.floor((log2P[15] - 1.0 - math.log2(2 * M)) / 2.0))) >= 52 else 16
    cdiv = lambda a, b: (a + b - 1) // b  # noqa: E731
    total = 0.0
    for r0 in range(0, rows, chunk):
        rc = min(chunk, rows - r0)
        mt = cdiv(rc, 128) * 128
        fwd = sum(min(M, n0 + 256) if n0 < M else M for n0 in range(0, 2 * M, 256))                   # k-length per n-tile
        bwd = sum(2 * M - (n0 // 128) * 128 for n0 in range(0, M, 256))
        wgt = 0
        for mp in range(cdiv(cdiv(2 * M, 128), 2)):
            for n0 in range(0, M, 256):
                m_hi = (2 * mp + 1) * 128
                if m_hi < M and n0 > m_hi + 127:
                    continue
                wgt += 2 * 128 * 256 * cdiv(rc, 128) * 128
        total += 2.0 * (Tf * mt * 256 * fwd + Tb * mt * 256 * bwd + 16 * wgt)
    return total


LEAF_NAMES = ('Z', 'raw_lengthscale', 'raw_outputscale', 'm', 'L_raw', 'log_var_noise', 'theta')
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, outputs):
    """Writes out_dir/<name>.npy (float64) for each array, so that two builds can be compared output for output."""
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError('--dump-outputs: %d bytes exceed the %d-byte limit' % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def load_json(path):
    try:
        return json.load(open(path))
    except Exception:
        return {}


def lib_hash():
    """Hash of the library SOURCES (csrc/ + include/): ties a profile to a build.  (The .so itself is not byte-reproducible: two
    nvcc runs over identical sources differ, so a hash of the binary would change with every rebuild.)"""
    h = hashlib.sha1()
    base = os.path.join(ROOT, 'tgp', 'pytorch_b200', 'csrc')
    files = sorted(os.path.join(base, f) for f in os.listdir(base) if f.endswith(('.cu', '.cuh')))
    files.append(os.path.join(ROOT, 'include', 'tgp_b200.h'))
    for f in files:
        with open(f, 'rb') as fh:
            h.update(fh.read())
    return h.hexdigest()[:12]


# ---------------------------------------------------------------------------------------------------------------
def cpu_reference_steps(wl, p, X, Y, rows, steps, warmup):
    """ELBO + backward of the reference's algorithm (oracle port O2, pinned to the unmodified reference by tests/golden:
    /root/reference does not exist on the GPU box) on the host cores; each step is a `rows`-row minibatch."""
    from oracle import tgp_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    times = []
    for s in range(warmup + steps):
        lo = (s * rows) % max(X.shape[0] - rows, 1)
        xb, yb = X[lo:lo + rows], Y[lo:lo + rows].view(-1)
        t0 = time.perf_counter()
        O.elbo_and_grads(xb, yb, p, float(wl['N']), wl['likelihood'], N_QUAD)
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
    return rows / float(np.median(times)), float(np.median(times))


def run_reference(args):
    """The reference's CPU implementation of the path (kind 'port': the oracle restatement — the reference itself needs
    /root/reference, absent on the GPU box), all host threads, at the SAME minibatch size as our arm."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    rows = wl['batch']                                  # the arm's own minibatch size: 65536 rows per step
    gen = torch.Generator().manual_seed(SEED)
    X, Y = synth(wl, rows * 2, gen)
    p = param_state(wl, X, gen)
    rows_s, sec = cpu_reference_steps(wl, p, X, Y, rows, args.steps, args.warmup)
    cores = torch.get_num_threads()
    line = {'impl': 'reference', 'metric': METRIC, 'value': rows_s, 'unit': 'rows/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': sec * 1e3, 'higher_is_better': True,
            'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': dict(workload_config(wl, args, 1), cpu_rows_per_step=rows,
                           cpu_arm='oracle port O2 (torch CPU, all host threads); one host, independent of --gpus'),
            'cpu_baseline': {'value': rows_s, 'unit': 'rows/s', 'cores': cores, 'kind': 'port',
                             'sample': '%d-row minibatch per step (the arm\'s own batch size; M=%d, D=%d, %d GH points, FP64), '
                                       'torch CPU with %d threads, median of %d steps' % (rows, wl['M'], wl['D'], N_QUAD, cores, args.steps)},
            'e2e': {'value': rows_s, 'unit': 'rows/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    emit(line)


def workload_config(wl, args, world):
    rows = wl['batch'] if args.scaling == 'weak' else wl['batch'] // world
    return {'workload': wl['text'], 'name': args.workload, 'N': wl['N'], 'D': wl['D'], 'M': wl['M'],
            'rows_per_gpu_per_step': rows, 'global_batch': rows * world, 'parallelism': 'rows x%d' % world,
            'l2': 'per-step working set (A|B workspace %.2f GB) >> 126 MB L2, plus an explicit 256 MiB L2 flush between steps'
                  % (rows * 2 * wl['M'] * 8 / 1e9)}


# ---------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import ctypes as C
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py needs a CUDA device: the product has no CPU path')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    from tgp.pytorch_b200 import _lib, functional as Fn
    from tgp.pytorch_b200.dist import local_slice
    lib = _lib.load()
    if args.no_overlap:
        lib.tgp_set_option(_lib.OPT_OVERLAP_KGEN, 0)
    wl = WORKLOADS[args.workload]
    N_DATA, D, M = wl['N'], wl['D'], wl['M']
    BATCH = wl['batch'] if args.scaling == 'weak' else wl['batch'] // world      # rows per GPU per step
    global_batch = BATCH * world

    gen = torch.Generator().manual_seed(SEED)
    X, Y = synth(wl, N_DATA, gen)                     # identical on every rank (same seed)
    p = param_state(wl, X, gen)
    perm = torch.randperm(N_DATA, generator=gen)
    steps_total = args.warmup + args.steps
    scale = float(N_DATA) / global_batch

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    # the dataset lives in HBM for the device arm; minibatches are gathered by index on the device
    Xd, Yd = X.to(dev), Y.view(-1).to(dev)
    perm_d = perm.to(dev)

    def dev_batch(step):
        lo = ((step * global_batch) + rank * BATCH) % (N_DATA - global_batch)
        idx = perm_d[lo:lo + BATCH]
        return Xd.index_select(0, idx), Yd.index_select(0, idx)

    def make_step(compute):
        eng, t = build_engine(p, wl, dev, compute)
        leaves = [t['Z'], t['raw_ls'], t['raw_os'], t['m'], t['L_raw'], t['log_var_noise'], t['theta']]
        for x in leaves:
            if x is not None:
                x.requires_grad_(True)

        def step_fn(xb, yb, sc=scale):
            for x in leaves:
                if x is not None:
                    x.grad = None
            # sync_ell=False: ONE collective per step (the global ELL rides in the packed all-reduce of the backward)
            terms = Fn.elbo_terms(eng, xb, yb, sc, *leaves, None, check_status=True, sync_ell=False)
            loss = -(terms[0] - terms[1])
            loss.backward()
            return loss, terms
        return eng, leaves, step_fn

    def dist_parity():
        """N > 1: the all-reduced gradients of a row-sharded global minibatch against ONE rank evaluating the whole
        minibatch alone (same kernels, no collective).  Max L2-relative error over tensors and ranks."""
        eng, leaves, step_fn = make_step('f64')
        G = 2048 * world
        idx = perm_d[:G]
        xg, yg = Xd.index_select(0, idx), Yd.index_select(0, idx)
        sl = local_slice(G, rank, world)
        sc = float(N_DATA) / G
        step_fn(xg[sl].contiguous(), yg[sl].contiguous(), sc)
        got = [None if x is None else x.grad.clone() for x in leaves]
        ell_global = float((sc * eng.last_ell_sum).item())
        with Fn.local_only():
            loss, _ = step_fn(xg, yg, sc)
        errs = [float((a - x.grad).norm() / x.grad.norm()) for a, x in zip(got, leaves) if x is not None]
        kl = float(eng.kl.item())
        errs.append(abs((-(ell_global - kl)) - float(loss.item())) / abs(float(loss.item())))
        w = torch.tensor([max(errs)], dtype=torch.float64, device=dev)
        dist.all_reduce(w, op=dist.ReduceOp.MAX)
        return {'max_rel_err': float(w.item()), 'global_rows': G, 'ok': bool(w.item() < 1e-10),
                'what': 'all-reduced ELBO and gradients (Z, lengthscale, outputscale, m, L_S, noise, flow) of a row-sharded '
                        'global minibatch vs one rank evaluating it alone; max L2-relative error over tensors and ranks'}

    def measure(compute, sample_clocks, keep_outputs=False):
        """W warm-up + K timed ELBO fwd+bwd steps of the device arm in one compute mode.  keep_outputs: also return, as
        float64 host arrays, what the last timed step gave its caller (loss, the elbo_terms outputs, every gradient)."""
        eng, leaves, step_fn = make_step(compute)
        clocks = ClockSampler(local)
        if sample_clocks and rank == 0 and not args.no_clocks:
            clocks.start()                              # sampler runs through warm-up + timed region (same load)
        timing_on = 0 if args.no_gemm_timing else 1
        lib.tgp_gemm_timing(timing_on, None, None)      # events get created during warm-up, not in the timed region
        # pre-warm until the step time is steady (a fresh box starts with cold clocks / lazily loaded modules):
        # stop when three consecutive steps agree within 3 %, or after 8 s
        t_pre, recent = time.perf_counter(), []
        while True:
            t0 = time.perf_counter()
            step_fn(*dev_batch(0))
            torch.cuda.synchronize()
            recent = (recent + [time.perf_counter() - t0])[-3:]
            el = time.perf_counter() - t_pre
            done = el > 8.0 or (len(recent) == 3 and el > 2.0 and max(recent) < 1.03 * min(recent))
            if world > 1:                               # every rank must leave the loop in the same iteration
                flag = torch.tensor([1.0 if done else 0.0], device=dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                done = bool(flag.item() > 0.5)
            if done:
                break
        for s in range(args.warmup):
            step_fn(*dev_batch(s))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        lib.tgp_gemm_timing(timing_on, None, None)      # reset the accumulators
        launches0 = lib.tgp_launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for s in range(args.warmup, steps_total):
            flush.fill_(s & 0xFF)                       # L2 flush between timed iterations
            loss, terms = step_fn(*dev_batch(s))
        ev1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        outputs = None
        if keep_outputs:
            outputs = dict(zip(('loss', 'ell', 'kld', 'ell_rows', 'mu', 'v'), (loss,) + tuple(terms)))
            outputs.update(('grad_' + n, x.grad) for n, x in zip(LEAF_NAMES, leaves) if x is not None)
            outputs = {k: t.detach().double().cpu().numpy() for k, t in outputs.items()}
        gemm_ms, gemm_n = (C.c_double * 3)(), (C.c_long * 3)()
        lib.tgp_gemm_timing(0, gemm_ms, gemm_n)
        launches = lib.tgp_launch_count() - launches0
        clk = clocks.stop() if (sample_clocks and rank == 0) else None
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        loss_global = float((-(scale * eng.last_ell_sum - eng.kl[0])).item())      # global ELBO from the packed all-reduce
        # test-NLL forward (no gradients): marginals + quadrature log-lik + moments on the same batches
        with torch.no_grad():
            eng.set_params(*[None if x is None else x.detach() for x in leaves])
            eng.prepare(0.0)
            bstd = torch.ones(1, dtype=torch.float64, device=dev) if wl['likelihood'] == 'bernoulli' else None

            def nll_pass(refactor):
                for s in range(args.steps):
                    xb, yb = dev_batch(args.warmup + s)
                    if refactor:
                        eng.prepare(0.0)
                    mu, v = eng.qf_forward(xb)
                    eng.test_rows(mu, v, yb, None, 1, 1.0, v.std().reshape(1) if bstd is not None else None)
            nll_pass(True)
            torch.cuda.synchronize()
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
            nll_pass(True)
            e1.record()
            nll_pass(False)                            # same pass with the factorisation reused (frozen parameters)
            e2.record()
            torch.cuda.synchronize()
            tn = torch.tensor([e0.elapsed_time(e1), e1.elapsed_time(e2)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tn, op=dist.ReduceOp.MAX)
        return dict(ms_total=ms, value=global_batch * args.steps / (ms * 1e-3), loss=loss_global, outputs=outputs,
                    gemm_ms=list(gemm_ms), gemm_n=list(gemm_n), launches=int(launches), clocks=clk,
                    test_nll_rows_per_s=global_batch * args.steps / (float(tn[0].item()) * 1e-3),
                    test_nll_cached_rows_per_s=global_batch * args.steps / (float(tn[1].item()) * 1e-3))

    parity = dist_parity() if world > 1 else None
    # the secondary mode runs first: on a fresh box the first seconds of a process are not steady (cold clocks, lazy
    # module loads), and the headline should not absorb that
    second = args.other or ('f64' if args.compute != 'f64' else 'tf32x3')
    other = None
    if not args.no_other_mode:
        measure(second, False)                      # discarded: absorbs the cold start of a fresh box
    head = measure(args.compute, True, keep_outputs=bool(args.dump_outputs))
    if not args.no_other_mode:
        other = measure(second, False)
    ms_total, value, final_loss, launches, clk = head['ms_total'], head['value'], head['loss'], head['launches'], head['clocks']
    gemm_ms, gemm_n = head['gemm_ms'], head['gemm_n']

    # ---- end-to-end arm: host (pinned) minibatches through the public class API, loss read back every step -----
    e2e = run_e2e(args, wl, p, X, Y, perm, rank, world, dev, BATCH)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, head['outputs'])
    # ---- roofline of the dominant kernel -----------------------------------------------------------------------------
    peaks = load_json(os.path.join(ROOT, 'MEASURED_PEAKS.json'))
    extra = load_json(os.path.join(ROOT, 'profiles', 'r02_measured_peaks_extra.json'))     # scripts/measure_peaks.py on this pool
    peak64 = measure_gemm_peak(dev, torch.float64)
    peak_tf32 = measure_gemm_peak(dev, torch.float32, tf32=True)
    peak_i8 = measure_int8_peak(dev)
    alg_flop_step = 6.0 * M * M * BATCH                         # SURVEY.md §8d: 6*M^2 FLOP per row, fwd+bwd (per GPU)

    def with_traffic(r, mode):
        prof = load_json(os.path.join(ROOT, 'profiles', 'r02_roofline_traffic.json')).get(args.workload + ':' + mode)
        if prof and prof.get('lib_hash') == lib_hash():
            r['traffic'] = prof.get('traffic')                  # dram bytes per launch from ncu --set full of THIS build
            r['traffic_source'] = prof.get('source')
        elif prof:
            r['traffic_note'] = 'profiles/r02_roofline_traffic.json was captured from a different build (%s); not reported' % prof.get('lib_hash')
        return r

    def roofline_of(mode, g_ms, g_n, step_ms):
        tag = 1 if mode == 'f64' else 2
        k_ms, k_n = g_ms[tag] / args.steps, g_n[tag] / args.steps
        ach = alg_flop_step / (k_ms * 1e-3) / 1e12 if k_ms > 0 else 0.0
        if mode == 'i8crt':
            # the bounding pipe is the INTEGER tensor pipe: executed u8 x u8 operations against the measured INT8 GEMM rate;
            # the algorithmic FP64 rate (6 M^2 FLOP per row) is reported beside it, with the cuBLAS DGEMM rate for scale
            ops = i8crt_executed_ops(M, BATCH)
            ex = ops / (k_ms * 1e-3) / 1e12 if k_ms > 0 else 0.0
            r = {'bound': 'tensor', 'kernel': 'gemm_i8_mod_kernel (tcgen05 kind::i8, u8 x u8 -> s32 in TMEM, 15-16 residue planes, '
                                                 '2-CTA clusters with TMA multicast), the three batch contractions',
                    'achieved': ex, 'peak': peak_i8, 'unit': 'TOP/s', 'frac': ex / peak_i8 if peak_i8 else None,
                    'peak_source': 'cuBLASLt INT8 GEMM 8192^3 via torch._int_mm, best of 5, measured in this run (tcgen05 kind::i8 issue '
                                   'rate measured by scripts/microbench/mma_rate.cu: 4556 TOP/s); MEASURED_PEAKS.json holds bf16 %.0f TF/s '
                                   'and HBM %.0f GB/s only' % (peaks.get('bf16_tflops', 0.0), peaks.get('hbm_gbs', 0.0)),
                    'executed_int8_ops_per_step': ops, 'algorithmic_fp64_tflops': ach, 'cublas_dgemm_tflops': peak64,
                    'algorithmic_vs_cublas_dgemm': ach / peak64 if peak64 else None,
                    'algorithmic_flop_per_launch': alg_flop_step / max(k_n, 1), 'avg_launch_ms': k_ms / max(k_n, 1),
                    'launches_per_step': k_n, 'kernel_share_of_step': k_ms / step_ms, 'traffic': None,
                    'per_step_o_m3_gemm_ms': g_ms[0] / args.steps,
                    'note': 'FP64-accurate results (operands truncated at 52-53 bits below their row maximum, integer product exact); '
                            'the residue conversion and CRT reconstruction kernels around the GEMMs are counted in ms_per_step, not here'}
            return with_traffic(r, mode)
        if mode == 'f64':
            peak, src, kern = peak64, 'cuBLAS DGEMM 8192^3 via torch.matmul, best of 5, measured in this run', \
                'gemm_f64_kernel (FP64 DMMA mma.sync.m8n8k4), the six batch contractions'
        else:
            peak, src, kern = peak_tf32, 'cuBLAS TF32 GEMM 8192^3 via torch.matmul (allow_tf32), best of 5, measured in this run', \
                'gemm_tf32x3_kernel (tcgen05 kind::tf32, TMEM accumulators), the three batch contractions'
        r = {'bound': 'tensor', 'kernel': kern, 'achieved': ach, 'peak': peak, 'unit': 'TFLOP/s', 'frac': ach / peak if peak else None,
             'peak_source': src + '; MEASURED_PEAKS.json holds bf16 %.0f TF/s and HBM %.0f GB/s only'
                            % (peaks.get('bf16_tflops', 0.0), peaks.get('hbm_gbs', 0.0)),
             'pool_peaks': {k: extra.get(k) for k in ('fp64_tflops', 'fp64_tflops_sustained', 'tf32_tflops', 'tf32_tflops_sustained',
                                                      'int8_tops')} if extra else None,
             'algorithmic_flop_per_launch': alg_flop_step / max(k_n, 1), 'avg_launch_ms': k_ms / max(k_n, 1),
             'launches_per_step': k_n, 'kernel_share_of_step': k_ms / step_ms, 'traffic': None,
             'per_step_o_m3_gemm_ms': g_ms[0] / args.steps}
        if mode == 'tf32x3':
            # executed: three TF32 MMAs per product, dense 128x256 tiles incl. the dense C half: (2 + 2 + 2) M^2 MACs * 3
            r['executed_tflops'] = 3.0 * 2.0 * (1.5 + 1.5 + 1.5) * M * M * BATCH / (k_ms * 1e-3) / 1e12 if k_ms > 0 else 0.0
            r['executed_frac_of_peak'] = r['executed_tflops'] / peak if peak else None
        return with_traffic(r, mode)

    roofline = roofline_of(args.compute, gemm_ms, gemm_n, ms_total / args.steps)
    # ---- CPU baseline (rank 0, N = 1 only): the oracle port on the host cores, bounded sample ----------------------
    cpu = None
    if world == 1 and not args.no_cpu:
        rows = wl['batch']
        rows_s, sec = cpu_reference_steps(wl, p, X[:rows * 2], Y[:rows * 2], rows, 3, 1)
        cpu = {'value': rows_s, 'unit': 'rows/s', 'cores': torch.get_num_threads(), 'kind': 'port',
               'sample': '3 steps of a %d-row minibatch of the same workload after 1 warm-up (median %.2f s/step); oracle '
                         'port O2, torch CPU' % (rows, sec)}
    line = {'metric': METRIC, 'value': value, 'unit': 'rows/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_total / args.steps, 'higher_is_better': True, 'scaling': args.scaling,
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'config': workload_config(wl, args, world),
            'clocks': clk, 'e2e': e2e, 'gpu_launches': int(launches), 'roofline': roofline, 'cpu_baseline': cpu,
            'final_loss': final_loss, 'compute': args.compute, 'collectives_per_step': 1 if world > 1 else 0,
            'test_nll': {'value': head['test_nll_rows_per_s'], 'unit': 'rows/s',
                         'what': 'test log-lik + predictive moments forward (prepare + marginals + quadrature), device-resident',
                         'with_factorisation_reused_across_batches': head['test_nll_cached_rows_per_s']}}
    if parity is not None:
        line['dist_parity'] = parity
    if other is not None:
        line['other_mode'] = {'compute': second, 'value': other['value'], 'unit': 'rows/s',
                              'ms_per_step': other['ms_total'] / args.steps, 'final_loss': other['loss'],
                              'loss_rel_diff_vs_headline': abs(other['loss'] - final_loss) / abs(final_loss),
                              'test_nll_rows_per_s': other['test_nll_rows_per_s'],
                              'roofline': roofline_of(second, other['gemm_ms'], other['gemm_n'], other['ms_total'] / args.steps),
                              'note': 'f64 = every contraction on the FP64 DMMA pipe (mma.sync.m8n8k4.f64); i8crt = batch contractions on '
                                      'the tcgen05 integer pipe through CRT residues (FP64-accurate); tf32x3 = tcgen05 3xTF32 (FP32 '
                                      'accuracy); per-step factorisation, backward chain and the row epilogue are FP64 in every mode'}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_e2e(args, wl, p, X, Y, perm, rank, world, dev, BATCH):
    """Same metric through the public API (`sparse_MF_SP.ELBO` + backward) with HOST buffers: every step gathers its
    minibatch into pinned memory, copies it to the device, and reads the loss back."""
    import torch.distributed as dist
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    cg.device = str(dev)
    cg.sync_elbo_in_forward = False            # one collective per step; the global ELBO is read after backward
    cg.compute = args.compute                  # the class API runs the headline compute mode
    from tgp.pytorch_b200.dsp.models import instance_kernel, sparse_MF_SP
    from tgp.pytorch_b200.dsp.models.flow import instance_flow
    from tgp.pytorch_b200.dsp.likelihoods import GaussianNonLinearMean, Bernoulli
    from tgp.pytorch_b200.dsp.flows import StepTanhL, SAL
    N_DATA, D, M = wl['N'], wl['D'], wl['M']
    K = instance_kernel('scale_rbf', ard_num_dim=D, num_multioutput=1, kernel_is_shared=False,
                        init_params={'length_scale': 2.0, 'kernel_scale': 2.0})
    np.random.seed(0)
    if wl['likelihood'] == 'bernoulli':
        lik, flow = Bernoulli(), instance_flow(SAL(1))
    else:
        lik = GaussianNonLinearMean(out_dim=1, noise_init=0.05, noise_is_shared=False, quadrature_points=N_QUAD)
        flow = instance_flow(StepTanhL(1, 3, add_f0=True))
    model = sparse_MF_SP(['zero', K], X[:1024], p['Z'], float(N_DATA), lik, 1, True, False, False, False, False,
                         [flow], 'single', 0.0, False,
                         {'variational_distribution': {'variance_scale': 1e-5, 'mean_scale': 0.0}})
    with torch.no_grad():
        model.q_U.variational_mean.copy_(p['m'].view(1, -1))
        model.q_U.chol_variational_covar.copy_(p['L_raw'].view(1, M, M))
        model.covariance_function.base_kernel.raw_lengthscale.copy_(p['raw_lengthscale'].view(1, 1, D))
    model.to(dev)
    model.global_batch_rows = BATCH * world
    from tgp.pytorch_b200.data import PinnedMinibatchStager
    global_batch = BATCH * world
    stager = PinnedMinibatchStager(X, Y, BATCH, dev)

    def batch_index(step):
        lo = ((step * global_batch) + rank * BATCH) % (N_DATA - global_batch)
        return perm[lo:lo + BATCH]

    def one(step):
        """One step of the user-level loop: the step's inputs come from HOST memory (gathered into pinned buffers and
        copied to the device by the stager — for step+1 while step computes), the loss is read back to the host."""
        xb, yb = stager.get()
        model.zero_grad(set_to_none=True)
        ELBO, _, _ = model.ELBO(xb, yb)
        (-ELBO).backward()
        stager.stage(batch_index(step + 1))             # host gather + H2D of the next step under this step's backward
        return float(model.last_global_elbo().item())   # device -> host read of the step's result (global ELBO)

    stager.stage(batch_index(0))
    for s in range(min(args.warmup, 3)):
        one(s)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for s in range(args.steps):
        one(args.warmup + s)
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    return {'value': BATCH * world * args.steps / float(dt.item()), 'unit': 'rows/s',
            'h2d_bytes_per_step': stager.bytes_per_step, 'd2h_bytes_per_step': 8,
            'note': 'sparse_MF_SP.ELBO + backward per step through the class API; every step gathers its minibatch from host '
                    'memory into pinned buffers and copies it to the device (PinnedMinibatchStager: the gather + H2D of step '
                    's+1 overlap the kernels of step s), and reads the (global) ELBO back'}


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else any library prints to fd 1 (e.g. NCCL's version
    banner) was diverted to stderr at start-up."""
    os.write(_REAL_STDOUT, (json.dumps(line) + '\n').encode())


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='cfg4', choices=sorted(WORKLOADS))
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='weak: 65536 rows per GPU per step; strong: 65536 rows per step in total')
    ap.add_argument('--no-cpu', action='store_true', help='skip the CPU baseline leg')
    ap.add_argument('--compute', default='i8crt', choices=['f64', 'tf32x3', 'i8crt'],
                    help='f64: FP64 DMMA; i8crt: FP64-accurate on the tcgen05 integer path (CRT residues); tf32x3: tcgen05 3xTF32')
    ap.add_argument('--other', default=None, choices=['f64', 'tf32x3', 'i8crt'], help='secondary mode reported as other_mode')
    ap.add_argument('--no-other-mode', action='store_true', help='measure only the headline compute mode')
    ap.add_argument('--no-gemm-timing', action='store_true', help='(diagnostic) do not instrument GEMM launches with events')
    ap.add_argument('--no-clocks', action='store_true', help='(diagnostic) do not sample nvidia-smi during the timed region')
    ap.add_argument('--no-overlap', action='store_true', help='(diagnostic) K_xz generation on the main stream (TGP_OPT_OVERLAP_KGEN = 0)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step of the headline mode returned (loss, ELL, KLD, per-row ell, mu, v '
                         'and every gradient) as DIR/<name>.npy, float64; inputs are seeded, so runs with the same '
                         'arguments can be compared')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
