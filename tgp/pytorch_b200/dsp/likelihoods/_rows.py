"""Shared launcher for the likelihood classes: (mu, v) rows -> fused epilogue kernels.

`expected_log_prob` of every likelihood is differentiable w.r.t. (gauss_mean, gauss_cov, noise, flow parameters)
through the analytic gradients the kernel emits (tgp_ell_forward), with no autograd graph over the S x MB
quadrature grid the reference materialises.
"""
import torch

from ...engine import Engine, FlowLayout

_ENGINES = {}


def flow_pack(flow, X, n_mc=1):
    """flow module -> (FlowLayout, theta tensor or None, rowparams (R, n_rowparams) or None)."""
    layers, glob, rows = flow.describe(X, n_mc) if flow is not None else ([], [], [])
    layout = FlowLayout(layers)
    theta = torch.stack([g.reshape(()) for g in glob]).to(torch.float64) if glob else None
    rowp = torch.stack(rows, dim=-1).to(torch.float64) if rows else None
    return layout, theta, rowp


def row_engine(likelihood, n_quad, layout, device):
    """An Engine used only for its per-row kernels (M and D are irrelevant there)."""
    key = (likelihood, n_quad, tuple((l['kind'], l['restrict'], l['add_f0'], l['n_steps'], l['per_row'], l['p0'])
                                     for l in layout.layers), str(device))
    if key not in _ENGINES:
        _ENGINES[key] = Engine(1, 1, likelihood, n_quad, layout, device)
    return _ENGINES[key]


class _EllRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, eng, y, mu, v, log_var_noise, theta, rowp):
        dev = mu.device
        z = torch.zeros(1, dtype=torch.float64, device=dev)
        eng.set_params(torch.zeros(1, 1, dtype=torch.float64, device=dev), z, z, z, torch.ones(1, 1, dtype=torch.float64, device=dev),
                       None if log_var_noise is None else log_var_noise.detach().reshape(1).contiguous(),
                       None if theta is None else theta.detach().contiguous())
        rb = eng.new_reduce_buffer()
        rows, g_mu, g_v, drow = eng.ell_forward(mu.detach().double().contiguous(), v.detach().double().contiguous(),
                                                y.double().contiguous(),
                                                None if rowp is None else rowp.detach().contiguous(), 1.0, rb)
        ctx.save_for_backward(g_mu, g_v, drow if drow is not None else z)
        ctx.rb, ctx.layout, ctx.has = rb, eng.layout, (log_var_noise is not None, theta is not None, rowp is not None)
        ctx.n_theta, ctx.lv_shape = eng.flow.n_theta, None if log_var_noise is None else log_var_noise.shape
        ctx.io_dtype = mu.dtype
        ctx.mark_non_differentiable(rows)
        return rb[eng.layout.ell_sum].clone(), rows

    @staticmethod
    def backward(ctx, g_sum, _g_rows):
        g_mu, g_v, drow = ctx.saved_tensors
        lay, rb = ctx.layout, ctx.rb
        has_noise, has_theta, has_rowp = ctx.has
        d_lv = (rb[lay.dlogvar] * g_sum).reshape(ctx.lv_shape) if has_noise else None
        d_th = rb[lay.dtheta:lay.dtheta + ctx.n_theta] * g_sum if has_theta else None
        return (None, None, (g_mu * g_sum).to(ctx.io_dtype), (g_v * g_sum).to(ctx.io_dtype), d_lv, d_th,
                drow * g_sum if has_rowp else None)


def expected_log_prob_rows(likelihood, n_quad, y, mu, v, log_var_noise, flow, X):
    """Sum over the rows of E_q(f)[log p(y | G(f))] for ONE output GP, and the per-row terms."""
    layout, theta, rowp = flow_pack(flow, X) if likelihood != 'gauss_linear' else (FlowLayout([]), None, None)
    eng = row_engine(likelihood, n_quad, layout, mu.device)
    lv = None if log_var_noise is None else log_var_noise.to(torch.float64)
    return _EllRows.apply(eng, y, mu, v, lv, theta, rowp)


def test_rows(likelihood, n_quad, y, mu, v, log_var_noise, flow, X, y_std=1.0, n_mc=1, bern_std=None):
    """Per-row test log-likelihood and predictive moments (forward only)."""
    with torch.no_grad():
        layout, theta, rowp = flow_pack(flow, X, n_mc) if likelihood != 'gauss_linear' else (FlowLayout([]), None, None)
        eng = row_engine(likelihood, n_quad, layout, mu.device)
        dev = mu.device
        z = torch.zeros(1, dtype=torch.float64, device=dev)
        eng.set_params(torch.zeros(1, 1, dtype=torch.float64, device=dev), z, z, z, torch.ones(1, 1, dtype=torch.float64, device=dev),
                       None if log_var_noise is None else log_var_noise.detach().reshape(1).contiguous(),
                       None if theta is None else theta.detach().contiguous())
        R = mu.shape[0]
        if rowp is not None:
            # rows of X were laid out as (n_mc, R): the kernel wants (R, n_mc, n_rowparams)
            rowp = rowp.reshape(n_mc, R, -1).permute(1, 0, 2).contiguous()
        if y is None:
            y = torch.zeros(R, dtype=torch.float64, device=dev)
        return eng.test_rows(mu.double().contiguous(), v.double().contiguous(), y.double().contiguous(), rowp, n_mc, y_std,
                             None if bern_std is None else bern_std.double())


def coverage_rows(likelihood, n_quad, y, mu, v, log_var_noise, flow, X, S, n_mc=1, seed=0, want_samples=False):
    """S posterior-predictive samples per row, their 2.5 % / 97.5 % quantiles and the coverage indicator of y (forward only)."""
    with torch.no_grad():
        layout, theta, rowp = flow_pack(flow, X, n_mc) if likelihood != 'gauss_linear' else (FlowLayout([]), None, None)
        eng = row_engine(likelihood, n_quad, layout, mu.device)
        dev = mu.device
        z = torch.zeros(1, dtype=torch.float64, device=dev)
        eng.set_params(torch.zeros(1, 1, dtype=torch.float64, device=dev), z, z, z, torch.ones(1, 1, dtype=torch.float64, device=dev),
                       log_var_noise.detach().reshape(1).to(torch.float64).contiguous(), None if theta is None else theta.detach().contiguous())
        R = mu.shape[0]
        if rowp is not None:
            rowp = rowp.reshape(n_mc, R, -1).permute(1, 0, 2).contiguous()
        return eng.coverage_rows(mu.double().contiguous(), v.double().contiguous(), y.double().contiguous(), rowp, n_mc, S, seed,
                                 want_samples=want_samples)


# ---- Monte-Carlo softmax likelihood (tgp_mc_softmax_rows) -------------------------------------------------------------
def _mc_model(layout):
    """TgpModel carrying only the flow architecture (the MC kernel ignores the GP / likelihood fields)."""
    from ... import _lib
    md = _lib.TgpModel()
    md.dtype, md.M, md.D = _lib.TGP_F64, 1, 1
    md.likelihood, md.n_quad = _lib.LIK_GAUSS_NONLINEAR, 1
    layout.fill(md)
    return md


def mc_flow_pack(flows, X):
    """C flow modules of one architecture -> (FlowLayout, theta (C, n_theta) or None, rowp (C, R, n_rowparams) or None).
    Input-dependent layers evaluate each class's MLPs on X[c]; their outputs are stacked class-major."""
    packs = [flow_pack(fl, X[c] if X is not None else None) for c, fl in enumerate(flows)]
    first = packs[0][0]
    for lay, _th, _rp in packs:
        if lay.layers != first.layers:          # kinds, flags, per_row and p0 of every layer
            raise NotImplementedError('the Monte-Carlo softmax kernel takes one flow architecture for all classes')
    theta = torch.stack([p[1] for p in packs]) if first.n_theta > 0 else None
    rowp = torch.stack([p[2] for p in packs]) if first.n_rowparams > 0 else None
    return first, theta, rowp


class _McSoftmax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, layout, y, eps, want_probs, mu, v, theta, rowp):
        import ctypes as C
        from ... import _lib
        lib = _lib.load()
        if not mu.is_cuda:
            raise RuntimeError('tgp.pytorch_b200 has no CPU path: move the model and the data to a CUDA device')
        dev = mu.device
        Cn, R = mu.shape
        S = eps.shape[0]
        assert tuple(eps.shape) == (S, Cn, R), 'eps must be (S, C, R)'
        d = torch.float64
        mu_d, v_d = mu.detach().to(d).contiguous(), v.detach().to(d).contiguous()
        th = None if theta is None else theta.detach().to(d).contiguous()
        rp = None if rowp is None else rowp.detach().to(d).contiguous()
        assert rp is None or tuple(rp.shape) == (Cn, R, layout.n_rowparams), 'rowp must be (C, R, n_rowparams)'
        grad = any(ctx.needs_input_grad)
        rows = torch.empty(R, dtype=d, device=dev)
        g_mu = torch.empty(Cn, R, dtype=d, device=dev) if grad else None
        g_v = torch.empty(Cn, R, dtype=d, device=dev) if grad else None
        dth = torch.zeros_like(th) if (grad and th is not None) else None
        drp = torch.empty_like(rp) if (grad and rp is not None) else None
        probs = torch.empty(R, Cn, dtype=d, device=dev) if want_probs else None
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        args = (_mc_model(layout), Cn, S, R, ptr(mu_d), ptr(v_d), ptr(y.to(d).contiguous()), ptr(eps.to(d).contiguous()), ptr(th),
                1 if grad else 0, ptr(rows), ptr(g_mu), ptr(g_v), ptr(dth), ptr(probs))
        with torch.cuda.device(dev):
            st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            if rp is None:
                _lib.check(lib.tgp_mc_softmax_rows(*args, st), 'tgp_mc_softmax_rows')
            else:
                _lib.check(lib.tgp_mc_softmax_rows_rowp(*args, ptr(rp), ptr(drp), st), 'tgp_mc_softmax_rows_rowp')
        if grad:
            ctx.save_for_backward(g_mu, g_v, dth if dth is not None else rows.new_zeros(1),
                                  drp if drp is not None else rows.new_zeros(1))
        ctx.has_theta, ctx.has_rowp, ctx.io_dtype = th is not None, rp is not None, mu.dtype
        out_p = probs if want_probs else rows.new_zeros(0)
        ctx.mark_non_differentiable(rows, out_p)
        return rows.sum(), rows, out_p

    @staticmethod
    def backward(ctx, g_sum, _g_rows, _g_probs):
        g_mu, g_v, dth, drp = ctx.saved_tensors
        return (None, None, None, None, (g_mu * g_sum).to(ctx.io_dtype), (g_v * g_sum).to(ctx.io_dtype),
                dth * g_sum if ctx.has_theta else None, drp * g_sum if ctx.has_rowp else None)


def mc_softmax(flows, X, y, eps, mu, v, want_probs=False):
    """(sum over rows of the MC expected log-likelihood, per-row terms, class probabilities or empty)."""
    from ... import functional as Fn
    layout, theta, rowp = mc_flow_pack(flows, X)
    if theta is not None and theta.requires_grad and Fn._world() is not None:
        theta = Fn._SumGradAcrossRanks.apply(theta)          # the flow scalars see rank-local rows only
    # rowp is row-local; the MLP weights behind it are summed across ranks by the fused MLP backward / synced_module_call
    return _McSoftmax.apply(layout, y, eps, bool(want_probs), mu, v, theta, rowp)
