"""Single-call interface of the C-ABI (include/tgp_b200.h: tgp_create / tgp_bind_workspace / tgp_elbo_fwd / tgp_elbo_bwd /
tgp_test_nll_fwd) — what a binding that does not want to sequence the stages itself uses.

One `ElboSession` = one TgpHandle + ONE caller-owned device allocation of `tgp_workspace_bytes()`.  The class-level API
(`dsp.models.sparse_MF_SP`) drives the staged entry points through `engine.Engine` instead, because autograd sits between
the forward and the backward there; both run the same kernels.
"""
import ctypes as C

import torch

from . import _lib
from .engine import Engine, _ptr, _stream


class ElboSession:
    def __init__(self, engine: Engine, max_rows: int):
        self.lib = engine.lib
        self.eng = engine                       # source of the model description, the quadrature rule and the device
        self.device = engine.device
        self.max_rows = int(max_rows)
        self.handle = C.c_void_p()
        _lib.check(self.lib.tgp_create(engine.model, self.max_rows, C.byref(self.handle)), 'tgp_create')
        nbytes = self.lib.tgp_workspace_bytes(engine.model, self.max_rows)
        self.workspace = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.tgp_bind_workspace(self.handle, _ptr(self.workspace), nbytes), 'tgp_bind_workspace')
        self._batch = None
        self._keep = None

    def close(self):
        if self.handle:
            self.lib.tgp_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:      # noqa: BLE001 — interpreter shutdown
            pass

    def _params(self, Z, raw_ls, raw_os, m, L_raw, log_var_noise, theta):
        self.eng.set_params(Z, raw_ls, raw_os, m, L_raw, log_var_noise, theta)      # validates shapes / dtypes / device
        return self.eng._params

    def _make_batch(self, X, Y, scale, rowparams=None):
        b = _lib.TgpBatch()
        b.X, b.Y = X.data_ptr(), (Y.data_ptr() if Y is not None else None)
        b.rowparams = rowparams.data_ptr() if rowparams is not None else None
        b.R, b.scale = X.shape[0], float(scale)
        b.quad_t = self.eng.qt.data_ptr() if self.eng.qt is not None else None
        b.quad_w = self.eng.qw.data_ptr() if self.eng.qw is not None else None
        return b

    def forward(self, X, Y, scale, Z, raw_ls, raw_os, m, L_raw, log_var_noise, theta, jitter=0.0):
        """-> dict(terms=(2,) [scale * sum ell, KL], status=(1,) int32, ell_rows, mu, v); all device tensors."""
        with torch.cuda.device(self.device):
            p = self._params(Z, raw_ls, raw_os, m, L_raw, log_var_noise, theta)
            R = X.shape[0]
            f64 = torch.float64
            out = dict(terms=torch.empty(2, dtype=f64, device=self.device), status=torch.zeros(1, dtype=torch.int32, device=self.device),
                       ell_rows=torch.empty(R, dtype=f64, device=self.device), mu=torch.empty(R, dtype=f64, device=self.device),
                       v=torch.empty(R, dtype=f64, device=self.device))
            fo = _lib.TgpFwdOut()
            fo.terms, fo.status, fo.ell_rows, fo.mu, fo.v = (out[k].data_ptr() for k in ('terms', 'status', 'ell_rows', 'mu', 'v'))
            self._batch = self._make_batch(X, Y, scale)
            self._keep = (X, Y, p)
            _lib.check(self.lib.tgp_elbo_fwd(self.handle, p, self._batch, float(jitter), fo, _stream(self.device)), 'tgp_elbo_fwd')
        return out

    def backward(self, g_dev, allreduce=None, input_grad=False):
        """Gradients of g_dev[0] * ELL + g_dev[1] * KL (g_dev: device tensor of 2 doubles).  `allreduce(tensor)` — called
        once on the tril-packed exchange buffer — makes the step row-sharded (e.g. torch.distributed.all_reduce).
        input_grad=True also returns out['X'], the gradient w.r.t. the rows of X of the last forward (this rank's rows)."""
        eng, dev, f64 = self.eng, self.device, torch.float64
        M, D = eng.M, eng.D
        out = dict(Z=torch.empty(M, D, dtype=f64, device=dev), raw_ls=torch.empty(D, dtype=f64, device=dev),
                   raw_os=torch.empty(1, dtype=f64, device=dev), m=torch.empty(M, dtype=f64, device=dev),
                   L_raw=torch.empty(M, M, dtype=f64, device=dev), log_var_noise=torch.zeros(1, dtype=f64, device=dev),
                   theta=torch.zeros(eng.flow.n_theta, dtype=f64, device=dev))
        g = _lib.TgpGrads()
        g.dZ, g.draw_lengthscale, g.draw_outputscale = out['Z'].data_ptr(), out['raw_ls'].data_ptr(), out['raw_os'].data_ptr()
        g.dm, g.dL_raw, g.dlog_var_noise = out['m'].data_ptr(), out['L_raw'].data_ptr(), out['log_var_noise'].data_ptr()
        g.dtheta = out['theta'].data_ptr() if eng.flow.n_theta else None
        if input_grad:
            out['X'] = torch.empty(self._batch.R, D, dtype=f64, device=dev)
            g.dX = out['X'].data_ptr()
        cb = _lib.ALLREDUCE_FN(0)
        if allreduce is not None:
            n_packed = eng.layout.packed_total

            def _cb(buf, count, _user, _stream_):
                try:
                    # the exchange buffer lives inside our workspace tensor: view it without copying
                    off = buf - self.workspace.data_ptr()
                    view = self.workspace[off:off + 8 * count].view(torch.float64)
                    assert count == n_packed
                    allreduce(view)
                    return 0
                except Exception:      # noqa: BLE001 — must not unwind through C
                    return 1
            cb = _lib.ALLREDUCE_FN(_cb)
        with torch.cuda.device(dev):
            _lib.check(self.lib.tgp_elbo_bwd(self.handle, self._keep[2], self._batch, _ptr(g_dev), g, cb, None,
                                             _stream(dev)), 'tgp_elbo_bwd')
        return out

    def test_nll(self, X, Y, Z, raw_ls, raw_os, m, L_raw, log_var_noise, theta, y_std=1.0, refactor=True, bern_std=None):
        """-> (logp_rows, m1, m2, mu, v, status)."""
        dev, f64 = self.device, torch.float64
        with torch.cuda.device(dev):
            p = self._params(Z, raw_ls, raw_os, m, L_raw, log_var_noise, theta)
            R = X.shape[0]
            logp, m1, m2, mu, v = (torch.empty(R, dtype=f64, device=dev) for _ in range(5))
            status = torch.zeros(1, dtype=torch.int32, device=dev)
            b = self._make_batch(X, Y, 1.0)
            _lib.check(self.lib.tgp_test_nll_fwd(self.handle, p, b, 1 if refactor else 0, 1, float(y_std), _ptr(bern_std),
                                                 _ptr(logp), _ptr(m1), _ptr(m2), _ptr(mu), _ptr(v), _ptr(status), _stream(dev)),
                       'tgp_test_nll_fwd')
        return logp, m1, m2, mu, v, status
