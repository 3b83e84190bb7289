"""Per-stage device time of one cfg4 step (CUDA events on the current stream, median of 10)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
from tests.gpu_util import engine_inputs, make_engine
dev = 'cuda:0'
WL = bench.WORKLOADS[os.environ.get('TGP_WORKLOAD', 'cfg4')]
gen = torch.Generator().manual_seed(bench.SEED)
X, Y = bench.synth(WL, 200000, gen)
p = bench.param_state(WL, X, gen)
xb, yb = X[:65536].to(dev), Y[:65536].view(-1).to(dev)
scale = WL['N'] / 65536


def timed(fn, n=10):
    ts = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record(); out = fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2], out


from tgp.pytorch_b200 import _lib
if os.environ.get('TGP_ROW_CHUNK'):
    _lib.load().tgp_set_option(_lib.OPT_ROW_CHUNK, int(os.environ['TGP_ROW_CHUNK']))
for compute in sys.argv[1:] or ['f64', 'i8crt', 'tf32x3']:
    eng, theta, _, _ = make_engine(p, WL['likelihood'], 100, dev, compute=compute)
    ei = engine_inputs(p, dev)
    eng.set_params(ei['Z'], ei['raw_ls'], ei['raw_os'], ei['m'], ei['L_raw'], ei['log_var_noise'], theta)
    for _ in range(3):
        eng.prepare(0.0); mu, v = eng.qf_forward(xb)
    t_prep, _ = timed(lambda: eng.prepare(0.0))
    t_fwd, (mu, v) = timed(lambda: eng.qf_forward(xb))
    rb = eng.new_reduce_buffer()
    t_ell, (rows, g_mu, g_v, _) = timed(lambda: eng.ell_forward(mu, v, yb, None, scale, rb))
    def bwd():
        eng.qf_forward(xb)      # qf_backward consumes the saved [A|B]; re-create it (time subtracted below)
        eng.qf_backward(xb, g_mu, g_v, rb)
    t_fb, _ = timed(bwd)
    t_chain, _ = timed(lambda: eng.chain_backward(rb, 1.0, -1.0))
    bstd = v.std().reshape(1) if WL['likelihood'] == 'bernoulli' else None
    t_test, _ = timed(lambda: eng.test_rows(mu, v, yb, None, 1, 1.0, bstd))
    print('%-13s prepare %.3f  qf_forward %.3f  ell %.3f  qf_backward %.3f  chain %.3f  test_rows %.3f  | sum %.3f ms'
          % (compute, t_prep, t_fwd, t_ell, t_fb - t_fwd, t_chain, t_test, t_prep + t_fwd + t_ell + (t_fb - t_fwd) + t_chain))
