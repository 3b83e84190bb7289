"""Thin torch-facing wrapper over the C-ABI: owns workspaces, passes raw device pointers and the current stream.

One `Engine` per (output GP, device).  Nothing here computes: every method enqueues kernels of
`libtgp_b200.so` on `torch.cuda.current_stream()` and returns device tensors.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib

_KIND = {'identity': _lib.FLOW_IDENTITY, 'affine': _lib.FLOW_AFFINE, 'tanh_step': _lib.FLOW_TANH_STEP,
         'sal': _lib.FLOW_SAL, 'arcsinh': _lib.FLOW_ARCSINH, 'boxcox': _lib.FLOW_BOXCOX, 'invboxcox': _lib.FLOW_INV_BOXCOX,
         'step_group': _lib.FLOW_STEP_GROUP}
_NPAR = {'affine': 2, 'sal': 2, 'arcsinh': 4, 'boxcox': 1, 'invboxcox': 1, 'step_group': 0}
_LIK = {'gauss_linear': _lib.LIK_GAUSS_LINEAR, 'gauss_nonlinear': _lib.LIK_GAUSS_NONLINEAR,
        'bernoulli': _lib.LIK_BERNOULLI, 'gauss_warped': _lib.LIK_GAUSS_WARPED}


class FlowLayout:
    """Flat description of a composed flow G for the kernels.

    `layers`: list of dicts {kind, restrict, add_f0, n_steps, per_row, switch}.  Global parameters of all layers are packed
    in descriptor order into `theta`; per-row (input-dependent) parameters into the columns of a (R, n_rowparams)
    matrix.  Parameter order inside a layer: affine [a, b]; tanh_step n_steps x [a, b, c, d]; sal [a, b]; arcsinh
    [a, b, c, d]; boxcox / invboxcox [lam after the module's constraint]; a `step_group` header (n_steps members follow,
    all evaluated at the header's input and summed) has none; a member with `switch` appends its switch_off [s, t]
    (reference code/dsp/models/flow.py:330-340, 377-446, 495-557, 755-773, 965-977, 1039-1149).
    """

    def __init__(self, layers):
        self.layers = []
        self.n_theta = 0
        self.n_rowparams = 0
        for lay in layers:
            kind = lay['kind']
            if kind == 'identity':
                continue
            npar = 4 * lay.get('n_steps', 0) if kind == 'tanh_step' else _NPAR[kind]
            switch = bool(lay.get('switch', False))                 # step member with a trainable switch_off: + [s, t]
            npar += 2 if switch else 0
            per_row = bool(lay.get('per_row', False))
            if switch and per_row:
                raise NotImplementedError('input-dependent step members with a trainable switch_off')
            p0 = self.n_rowparams if per_row else self.n_theta
            if per_row:
                self.n_rowparams += npar
            else:
                self.n_theta += npar
            self.layers.append(dict(kind=kind, restrict=bool(lay.get('restrict', False)),
                                    add_f0=bool(lay.get('add_f0', False)), n_steps=int(lay.get('n_steps', 0)),
                                    per_row=per_row, p0=p0, npar=npar, switch=switch))
        if len(self.layers) > _lib.MAX_LAYERS:
            raise ValueError('flow has %d layers; the fused epilogue supports %d' % (len(self.layers), _lib.MAX_LAYERS))

    def fill(self, model):
        model.n_layers = len(self.layers)
        model.n_theta = self.n_theta
        model.n_rowparams = self.n_rowparams
        for i, lay in enumerate(self.layers):
            L = model.layers[i]
            L.kind = _KIND[lay['kind']]
            L.flags = (_lib.FLOW_RESTRICT if lay['restrict'] else 0) | (_lib.FLOW_ADD_F0 if lay['add_f0'] else 0) | \
                      (_lib.FLOW_PER_ROW if lay['per_row'] else 0) | (_lib.FLOW_SWITCH if lay['switch'] else 0)
            L.n_steps = lay['n_steps']
            L.p0 = lay['p0']


_GH_CACHE = {}


def gauss_hermite(n, device):
    """numpy hermgauss(n), as gpytorch's GaussHermiteQuadrature1D builds its rule (FP64 build)."""
    key = (n, str(device))
    if key not in _GH_CACHE:
        t, w = np.polynomial.hermite.hermgauss(n)
        _GH_CACHE[key] = (torch.tensor(t, dtype=torch.float64, device=device),
                          torch.tensor(w, dtype=torch.float64, device=device))
    return _GH_CACHE[key]


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _on_device(fn):
    """Engine methods enqueue on the ENGINE's device: make it current for the call (kernel launches, per-device function
    attributes and the stream lookup all depend on the current device)."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *a, **k):
        if torch.cuda.current_device() == self.device.index:
            return fn(self, *a, **k)
        with torch.cuda.device(self.device):
            return fn(self, *a, **k)
    return wrapped


def _chk(t, name, shape=None):
    if t is None:
        return
    if not t.is_cuda:
        raise ValueError('%s must be a CUDA tensor (there is no CPU path)' % name)
    if t.dtype != torch.float64:
        raise ValueError('%s must be float64, got %s' % (name, t.dtype))
    if not t.is_contiguous():
        raise ValueError('%s must be contiguous' % name)
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise ValueError('%s has shape %s, expected %s' % (name, tuple(t.shape), tuple(shape)))


# covariance function of the engine -> TgpModel.kernel
KERNELS = {'rbf': _lib.KERNEL_RBF, 'matern12': _lib.KERNEL_MATERN12, 'matern32': _lib.KERNEL_MATERN32,
           'matern52': _lib.KERNEL_MATERN52}


class Engine:
    def __init__(self, M, D, likelihood, n_quad, flow_layout, device, compute='f64', kernel='rbf', whiten=True):
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise RuntimeError('tgp.pytorch_b200 runs on CUDA devices only (no CPU fallback)')
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        self.M, self.D = int(M), int(D)
        self.likelihood = likelihood
        self.flow = flow_layout
        self.model = _lib.TgpModel()
        if compute not in ('f64', 'tf32x3', 'i8crt'):
            raise ValueError("compute must be 'f64', 'tf32x3' or 'i8crt'")
        self.compute = compute
        self.model.dtype = {'f64': _lib.TGP_F64, 'tf32x3': _lib.TGP_F32, 'i8crt': _lib.TGP_F64_I8}[compute]
        self.model.M, self.model.D = self.M, self.D
        if kernel not in KERNELS:
            raise ValueError('kernel must be one of %s' % (', '.join(repr(k) for k in KERNELS),))
        self.kernel = kernel
        self.model.kernel = KERNELS[kernel]
        # q(u) = N(m, P P^T) of the whitened variable (True) or of u itself (False, the reference's is_whiten=False)
        self.whiten = bool(whiten)
        self.model.q_u_form = _lib.QU_WHITENED if self.whiten else _lib.QU_UNWHITENED
        self.model.likelihood = _LIK[likelihood]
        self.model.n_quad = int(n_quad)
        flow_layout.fill(self.model)
        self.n_quad = int(n_quad)
        nbytes = self.lib.tgp_step_workspace_bytes(self.model)
        if nbytes == 0:
            raise ValueError('invalid model description: ' + self.lib.tgp_last_error().decode())
        self.step_ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        self.layout = _lib.TgpReduceLayout()
        _lib.check(self.lib.tgp_reduce_layout(self.model, self.layout), 'tgp_reduce_layout')
        self.kl = torch.zeros(1, dtype=torch.float64, device=self.device)
        self.status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._batch_ws = None
        self._cov_ws = None
        self._chol_ws = None
        self._rb = None
        self._packed = None
        self.last_ell_sum = None
        self._params = None
        self._keep = None
        self.generation = 0          # bumped by every prepare(); backward passes check it
        self.prepared_key = None     # parameter identity/version of the factorisation held in step_ws (eval cache)
        self.qt, self.qw = gauss_hermite(self.n_quad, self.device) if likelihood != 'gauss_linear' else (None, None)

    # -- helpers ------------------------------------------------------------------------------------------------
    def batch_ws(self, R):
        # the size is asked for on every call: it depends on library options (TGP_OPT_ROW_CHUNK) as well as on R
        nbytes = self.lib.tgp_batch_workspace_bytes(self.model, R)
        if self._batch_ws is None or self._batch_ws.numel() < nbytes:
            self._batch_ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        return self._batch_ws

    def new_reduce_buffer(self, fresh=True):
        """The packed pre-chain accumulator, zeroed.  fresh=False re-uses one persistent buffer per engine (the training
        step: its previous contents are dead once the previous backward has been enqueued)."""
        if fresh:
            return torch.zeros(self.layout.total, dtype=torch.float64, device=self.device)
        if self._rb is None:
            self._rb = torch.empty(self.layout.total, dtype=torch.float64, device=self.device)
        return self._rb.zero_()

    @_on_device
    def pack_reduce(self, rb):
        if self._packed is None:
            self._packed = torch.empty(self.layout.packed_total, dtype=torch.float64, device=self.device)
        _lib.check(self.lib.tgp_reduce_pack(self.model, _ptr(rb), _ptr(self._packed), _stream(self.device)), 'tgp_reduce_pack')
        return self._packed

    @_on_device
    def unpack_reduce(self, packed, rb):
        _lib.check(self.lib.tgp_reduce_unpack(self.model, _ptr(packed), _ptr(rb), _stream(self.device)), 'tgp_reduce_unpack')
        return rb

    def set_params(self, Z, raw_ls, raw_os, m, L_raw, log_var_noise, theta):
        M, D = self.M, self.D
        _chk(Z, 'Z', (M, D)); _chk(raw_ls, 'raw_lengthscale', (D,)); _chk(raw_os, 'raw_outputscale', (1,))
        _chk(m, 'm', (M,)); _chk(L_raw, 'L_raw', (M, M)); _chk(log_var_noise, 'log_var_noise', (1,))
        _chk(theta, 'theta', (self.flow.n_theta,))
        p = _lib.TgpParams()
        p.Z, p.raw_lengthscale, p.raw_outputscale = Z.data_ptr(), raw_ls.data_ptr(), raw_os.data_ptr()
        p.m, p.L_raw = m.data_ptr(), L_raw.data_ptr()
        p.log_var_noise = log_var_noise.data_ptr() if log_var_noise is not None else None
        p.theta = theta.data_ptr() if theta is not None and theta.numel() > 0 else None
        self._params = p
        self._keep = (Z, raw_ls, raw_os, m, L_raw, log_var_noise, theta)     # keep the storage alive

    # -- the C-ABI stages ---------------------------------------------------------------------------------------
    @_on_device
    def prepare(self, jitter=0.0):
        self.generation += 1
        _lib.check(self.lib.tgp_prepare(self.model, self._params, float(jitter), _ptr(self.step_ws), _ptr(self.kl),
                                        _ptr(self.status), _stream(self.device)), 'tgp_prepare')
        return self.kl, self.status

    def status_reader(self):
        """Returns a function that blocks the host until the factorisation of the last prepare() has finished — and only the
        factorisation: the library copies the 4-byte pivot status to pinned host memory right behind it (on its own
        high-priority stream when TGP_OPT_OVERLAP_KGEN forks it there) — and yields the status.  Call it after the kernels
        that consume the factorisation have been enqueued: the check then costs no pipeline bubble."""
        dev = self.device

        def read():
            out = C.c_int(0)
            with torch.cuda.device(dev):
                _lib.check(self.lib.tgp_factor_status(C.byref(out)), 'tgp_factor_status')
            return int(out.value)
        return read

    @_on_device
    def qf_forward(self, X):
        R = X.shape[0]
        _chk(X, 'X', (R, self.D))
        mu = torch.empty(R, dtype=torch.float64, device=self.device)
        v = torch.empty(R, dtype=torch.float64, device=self.device)
        _lib.check(self.lib.tgp_qf_forward(self.model, _ptr(self.step_ws), _ptr(self.batch_ws(R)), _ptr(X), R, _ptr(mu),
                                           _ptr(v), _stream(self.device)), 'tgp_qf_forward')
        return mu, v

    # -- full covariance over a test batch (evaluation only: no backward) ----------------------------------------------
    @_on_device
    def qf_cov(self, X):
        """(mu (R,), Sigma (R, R)) of q(f) at the rows of X from the factorisation in the step workspace (prepare() first).
        Leaves the batch workspace alone, so it may run between an ELBO forward and its backward."""
        R = X.shape[0]
        _chk(X, 'X', (R, self.D))
        nbytes = self.lib.tgp_qf_cov_workspace_bytes(self.model, R)
        if self._cov_ws is None or self._cov_ws.numel() < nbytes:
            self._cov_ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        mu = torch.empty(R, dtype=torch.float64, device=self.device)
        cov = torch.empty(R, R, dtype=torch.float64, device=self.device)
        _lib.check(self.lib.tgp_qf_cov_forward(self.model, _ptr(self.step_ws), _ptr(self._cov_ws), _ptr(X), R, _ptr(mu),
                                               _ptr(cov), R, _stream(self.device)), 'tgp_qf_cov_forward')
        return mu, cov

    @_on_device
    def cov_cholesky(self, cov, jitter=0.0, scale=None):
        """(L, status): L = chol(cov + jitter I), lower with an exactly zero upper triangle; status (device int32) is 0 or the
        1-based index of the first pivot not above 8 eps * scale.  scale: device scalar, default the outputscale of the
        parameters last set (the prior variance, which bounds every diagonal entry of a posterior covariance)."""
        R = cov.shape[0]
        _chk(cov, 'cov', (R, R))
        if scale is None:
            scale = torch.nn.functional.softplus(self._keep[2]).reshape(1)
        _chk(scale, 'scale', (1,))
        nbytes = self.lib.tgp_cov_cholesky_workspace_bytes(R)
        if self._chol_ws is None or self._chol_ws.numel() < nbytes:
            self._chol_ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        L = torch.empty(R, R, dtype=torch.float64, device=self.device)
        status = torch.zeros(1, dtype=torch.int32, device=self.device)
        _lib.check(self.lib.tgp_cov_cholesky(R, _ptr(cov), R, float(jitter), _ptr(scale), _ptr(self._chol_ws), _ptr(L), R,
                                             _ptr(status), _stream(self.device)), 'tgp_cov_cholesky')
        return L, status

    @_on_device
    def cov_sample(self, mu, L, eps):
        """mu + eps L^T (S, R) for eps (S, R) drawn by the caller."""
        S, R = eps.shape
        _chk(mu, 'mu', (R,)); _chk(L, 'L', (R, R)); _chk(eps, 'eps', (S, R))
        out = torch.empty(S, R, dtype=torch.float64, device=self.device)
        _lib.check(self.lib.tgp_cov_sample(R, S, _ptr(mu), _ptr(L), R, _ptr(eps), _ptr(out), _stream(self.device)),
                   'tgp_cov_sample')
        return out

    @_on_device
    def ell_forward(self, mu, v, Y, rowparams, scale, reduce_buf, want_grad=True):
        R = mu.shape[0]
        _chk(mu, 'mu', (R,)); _chk(v, 'v', (R,)); _chk(Y, 'Y', (R,))
        nrp = self.flow.n_rowparams
        if nrp:
            _chk(rowparams, 'rowparams', (R, nrp))
        ell_rows = torch.empty(R, dtype=torch.float64, device=self.device)
        g_mu = torch.empty(R, dtype=torch.float64, device=self.device) if want_grad else None
        g_v = torch.empty(R, dtype=torch.float64, device=self.device) if want_grad else None
        drow = torch.empty(R, nrp, dtype=torch.float64, device=self.device) if (want_grad and nrp) else None
        _lib.check(self.lib.tgp_ell_forward(self.model, self._params, _ptr(mu), _ptr(v), _ptr(Y),
                                            _ptr(rowparams) if nrp else None, R, float(scale), _ptr(self.qt),
                                            _ptr(self.qw), 1 if want_grad else 0, _ptr(ell_rows), _ptr(g_mu), _ptr(g_v),
                                            _ptr(drow), _ptr(reduce_buf), _stream(self.device)), 'tgp_ell_forward')
        return ell_rows, g_mu, g_v, drow

    @_on_device
    def qf_backward(self, X, g_mu, g_v, reduce_buf, dX=None):
        """Accumulates the pre-chain sums into reduce_buf; with dX (R, D), zeroed by the caller, also accumulates there the
        gradient of sum_n g_mu[n] mu_n + g_v[n] v_n w.r.t. the rows of X."""
        R = X.shape[0]
        _chk(g_mu, 'g_mu', (R,)); _chk(g_v, 'g_v', (R,))
        if dX is None:
            _lib.check(self.lib.tgp_qf_backward(self.model, self._params, _ptr(self.step_ws), _ptr(self.batch_ws(R)),
                                                _ptr(X), R, _ptr(g_mu), _ptr(g_v), _ptr(reduce_buf), _stream(self.device)),
                       'tgp_qf_backward')
            return
        _chk(dX, 'dX', (R, self.D))
        _lib.check(self.lib.tgp_qf_backward_dx(self.model, self._params, _ptr(self.step_ws), _ptr(self.batch_ws(R)),
                                               _ptr(X), R, _ptr(g_mu), _ptr(g_v), _ptr(reduce_buf), _ptr(dX),
                                               _stream(self.device)), 'tgp_qf_backward_dx')

    @_on_device
    def chain_backward(self, reduce_buf, gE=1.0, gK=-1.0, g_dev=None):
        M, D, dev = self.M, self.D, self.device
        f64 = torch.float64
        out = dict(Z=torch.empty(M, D, dtype=f64, device=dev), raw_ls=torch.empty(D, dtype=f64, device=dev),
                   raw_os=torch.empty(1, dtype=f64, device=dev), m=torch.empty(M, dtype=f64, device=dev),
                   L_raw=torch.empty(M, M, dtype=f64, device=dev), log_var_noise=torch.zeros(1, dtype=f64, device=dev),
                   theta=torch.zeros(self.flow.n_theta, dtype=f64, device=dev))
        _lib.check(self.lib.tgp_chain_backward(self.model, self._params, _ptr(self.step_ws), _ptr(reduce_buf), float(gE),
                                               float(gK), _ptr(g_dev), _ptr(out['Z']), _ptr(out['raw_ls']), _ptr(out['raw_os']),
                                               _ptr(out['m']), _ptr(out['L_raw']), _ptr(out['log_var_noise']),
                                               _ptr(out['theta']) if self.flow.n_theta else None, _stream(self.device)),
                   'tgp_chain_backward')
        return out

    @_on_device
    def test_rows(self, mu, v, Y, rowparams, n_mc, y_std, bern_std=None):
        R = mu.shape[0]
        _chk(mu, 'mu', (R,)); _chk(v, 'v', (R,)); _chk(Y, 'Y', (R,))
        nrp = self.flow.n_rowparams
        if nrp:
            _chk(rowparams, 'rowparams', (R, n_mc, nrp))
        f64 = torch.float64
        logp = torch.empty(R, dtype=f64, device=self.device)
        m1 = torch.empty(R, dtype=f64, device=self.device)
        m2 = torch.empty(R, dtype=f64, device=self.device)
        _lib.check(self.lib.tgp_test_rows(self.model, self._params, _ptr(mu), _ptr(v), _ptr(Y),
                                          _ptr(rowparams) if nrp else None, R, int(n_mc), float(y_std), _ptr(self.qt),
                                          _ptr(self.qw), _ptr(bern_std), _ptr(logp), _ptr(m1), _ptr(m2), _stream(self.device)),
                   'tgp_test_rows')
        return logp, m1, m2

    @_on_device
    def flow_inverse(self, theta, z):
        """(G^-1(z) elementwise, NaN where the Newton inverse fails; device int32 count of the failures) for the engine's
        flow with global parameters theta (n_theta,).  Forward only."""
        _chk(theta, 'theta', (self.flow.n_theta,))
        R = z.numel()
        _chk(z, 'z', (R,))
        out = torch.empty(R, dtype=torch.float64, device=self.device)
        n_fail = torch.zeros(1, dtype=torch.int32, device=self.device)
        _lib.check(self.lib.tgp_flow_inverse(self.model, _ptr(theta) if self.flow.n_theta else None, _ptr(z), R, _ptr(out),
                                             _ptr(n_fail), _stream(self.device)), 'tgp_flow_inverse')
        return out, n_fail

    @_on_device
    def coverage_rows(self, mu, v, Y, rowparams, n_mc, S, seed=0, q=(0.025, 0.975), want_samples=False):
        """Posterior-predictive samples + interval coverage from given marginals (tgp_coverage_rows).
        -> (q_lo, q_hi, covered, samples or None)."""
        R = mu.shape[0]
        _chk(mu, 'mu', (R,)); _chk(v, 'v', (R,)); _chk(Y, 'Y', (R,))
        nrp = self.flow.n_rowparams
        if nrp:
            _chk(rowparams, 'rowparams', (R, n_mc, nrp))
        f64 = torch.float64
        qlo, qhi, cov = (torch.empty(R, dtype=f64, device=self.device) for _ in range(3))
        smp = torch.empty(R, S, dtype=f64, device=self.device) if want_samples else None
        if getattr(self, '_cov_offset', None) is None:
            self._cov_offset = torch.zeros(1, dtype=torch.int64, device=self.device)
        _lib.check(self.lib.tgp_coverage_rows(self.model, self._params, _ptr(mu), _ptr(v), _ptr(Y), _ptr(rowparams) if nrp else None, R,
                                              int(n_mc), int(S), int(seed) % (1 << 64), _ptr(self._cov_offset), float(q[0]), float(q[1]),
                                              _ptr(qlo), _ptr(qhi), _ptr(cov), _ptr(smp), None, _stream(self.device)), 'tgp_coverage_rows')
        return qlo, qhi, cov, smp

    @_on_device
    def export_step(self):
        M = self.M
        L, Li, Cm = (torch.empty(M, M, dtype=torch.float64, device=self.device) for _ in range(3))
        _lib.check(self.lib.tgp_debug_export_step(self.model, _ptr(self.step_ws), _ptr(L), _ptr(Li), _ptr(Cm), _stream(self.device)),
                   'tgp_debug_export_step')
        return L, Li, Cm


def debug_gemm(A, B, C_out, M, N, K, lda, ldb, ldc, a_layout, b_layout, alpha=1.0, beta=0.0, a_tri=0, b_tri=0,
               c_lower=0):
    lib = _lib.load()
    _lib.check(lib.tgp_debug_gemm_f64(M, N, K, _ptr(A), lda, a_layout, _ptr(B), ldb, b_layout, _ptr(C_out), ldc,
                                      float(alpha), float(beta), a_tri, b_tri, c_lower, _stream()), 'tgp_debug_gemm_f64')


def tf32_planes(x):
    """(rn_tf32(x), x - rn_tf32(x)) for an FP32 tensor — the operand format of the tcgen05 3xTF32 GEMM."""
    if x.dtype != torch.float32:
        raise ValueError('tf32_planes expects a float32 tensor, got %s' % x.dtype)
    bits = x.contiguous().view(torch.int32)
    half = torch.tensor(0x1000, dtype=torch.int32, device=x.device)
    mask = torch.tensor(-8192, dtype=torch.int32, device=x.device)
    hi = torch.bitwise_and(bits + half, mask).view(torch.float32)        # round-to-nearest TF32 (cvt.rna)
    assert hi.shape == x.shape
    return hi, x - hi


def debug_gemm_tf32x3(A, B, out, out_mode=0, tri_mode=0, tri_rows=0, lower_rows=0, splitk=1):
    """out (+)= A @ B.T with A (Mrows, K), B (Ncols, K) FP32 row-major; out FP32 (mode 0) or FP64 accumulated (mode 1)."""
    lib = _lib.load()
    Ah, Al = tf32_planes(A.contiguous())
    Bh, Bl = tf32_planes(B.contiguous())
    Mrows, K = A.shape
    Ncols = B.shape[0]
    _lib.check(lib.tgp_debug_gemm_tf32x3(Mrows, Ncols, K, _ptr(Ah), _ptr(Al), A.stride(0), _ptr(Bh), _ptr(Bl), B.stride(0),
                                         _ptr(out) if out_mode == 0 else None, _ptr(out) if out_mode == 1 else None,
                                         out.stride(0), out_mode, tri_mode, tri_rows, lower_rows, splitk, _stream()),
               'tgp_debug_gemm_tf32x3')
    return Ah, Al, Bh, Bl


def debug_gemm_crt(A, B, out, T=16, tri_mode=0, tri_rows=0, lower_rows=0, accumulate=False, mn_major=0):
    """out (+)= A @ B.T through the integer-residue (CRT) pipeline of compute mode 'i8crt'; A (M, K), B (N, K), out (M, N) FP64.
    mn_major bit 0 / 1: A / B is given transposed ((K, M) / (K, N)) and read MN-major by the tensor core."""
    lib = _lib.load()
    Mr, K = (A.shape[1], A.shape[0]) if mn_major & 1 else A.shape
    N = B.shape[1] if mn_major & 2 else B.shape[0]
    scratch = torch.empty(lib.tgp_debug_gemm_crt_bytes(Mr, N, K, T), dtype=torch.uint8, device=A.device)
    _lib.check(lib.tgp_debug_gemm_crt(Mr, N, K, _ptr(A), A.stride(0), _ptr(B), B.stride(0), _ptr(out), out.stride(0), T, tri_mode,
                                      tri_rows, lower_rows, 1 if accumulate else 0, mn_major, _ptr(scratch), _stream()),
               'tgp_debug_gemm_crt')
    return out
