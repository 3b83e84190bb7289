"""The seam between the reference-shaped host classes and the C-ABI kernels.

`elbo_terms` is what `sparse_MF_SP.ELBO` calls (reference code/dsp/models/sparse_MF_SP.py:552-598): it returns the
(N/MB)-scaled expected log-likelihood, the whitened KL and the per-row expected log-likelihoods, differentiable
w.r.t. every parameter through hand-written backward kernels (no autograd graph over the batch).

Row sharding (SURVEY.md §8e): when `torch.distributed` is initialised each rank passes its contiguous row slice of
the global minibatch and the GLOBAL scale N/MB_global; the packed pre-chain buffer is all-reduced once per backward
(NCCL over NVLink), the O(M^3) chain runs replicated.
"""
import warnings

import torch

from . import _lib  # noqa: F401  (fails loudly when the library has not been built)


class NanError(RuntimeError):
    """Stand-in for gpytorch.utils.errors.NanError (raised by the reference at code/dsp/utils.py:241-254)."""


class NumericalWarning(RuntimeWarning):
    """Stand-in for gpytorch.utils.warnings.NumericalWarning (code/dsp/utils.py:266)."""


_LOCAL_ONLY = [False]


class local_only:
    """Context manager: inside it the path behaves as a single rank even when torch.distributed is initialised (no
    collective is issued) — e.g. to evaluate a whole global minibatch on one rank as the yardstick of a parity check."""

    def __enter__(self):
        self._old = _LOCAL_ONLY[0]
        _LOCAL_ONLY[0] = True

    def __exit__(self, *exc):
        _LOCAL_ONLY[0] = self._old


def _world():
    import torch.distributed as dist
    if not _LOCAL_ONLY[0] and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist
    return None


def global_std(v):
    """`v.std()` (unbiased, as torch) over the rows of ALL ranks: under row sharding the reference's Bernoulli `marginal_moments`
    needs the batch-wide standard deviation of the variances (`Bernoulli.py:120,141`, a defect kept for parity; SURVEY.md §8e
    "Exception").  Two tiny all-reduces (count + sum, then the centred sum of squares); one rank: plain `v.std()`."""
    dist = _world()
    if dist is None:
        return v.std()
    acc = torch.stack([torch.tensor(float(v.numel()), dtype=torch.float64, device=v.device), v.double().sum()])
    dist.all_reduce(acc)
    mean = acc[1] / acc[0]
    ss = ((v.double() - mean) ** 2).sum().reshape(1)
    dist.all_reduce(ss)
    return torch.sqrt(ss[0] / (acc[0] - 1.0)).to(v.dtype)


def _jitter_ladder(engine, fail, base_jitter=None, constant_jitter=0.0):
    """The failure branch of psd_safe_cholesky (code/dsp/utils.py:241-270): NaN check, then jitter base * 10^i on top of
    the constant jitter; base = cg.global_jitter (sparse_MF_SP.py:330) or 1e-8 (1e-6 for float32 models)."""
    Z = engine._keep[0]
    if torch.isnan(Z).any() or torch.isnan(engine._keep[1]).any() or torch.isnan(engine._keep[2]).any():
        raise NanError('cholesky: the kernel matrix has NaN entries')
    jitter = 1e-8 if base_jitter is None else base_jitter
    for i in range(3):
        j = jitter * (10 ** i)
        kl, _ = engine.prepare(constant_jitter + j)
        if engine.status_reader()() == 0:        # blocks on the factorisation alone (it may run on the library's own stream)
            warnings.warn('A not p.d., added jitter of %g to the diagonal' % j, NumericalWarning)
            return kl, j
    raise RuntimeError('cholesky: matrix not positive definite after 3 jitter escalations (first bad pivot %d)' % fail)


def prepare_then(engine, work, check=True, base_jitter=None, constant_jitter=0.0):
    """Reference semantics of psd_safe_cholesky (code/dsp/utils.py:222-270): factorise with cg.constant_jitter only (None =
    0, :237); on failure add base * 10^i, i = 0..2, warning each time; raise after the third failure.

    `work()` enqueues everything that consumes the factorisation.  The 4-byte pivot status is copied to the host on a
    side stream that waits for the factorisation only, and is read AFTER `work()` has been enqueued: the host blocks
    ~1 ms (until the factorisation is done) while the compute stream still holds the whole forward, so the (almost
    always successful) check costs no pipeline bubble; on failure the ladder runs and `work()` is enqueued again on the
    jittered factor.  `check=False` skips the read-back altogether."""
    engine.prepared_key = None
    kl, status = engine.prepare(constant_jitter)
    if not check:
        return kl, work()
    read_status = engine.status_reader()        # D2H of the status on a side stream, ordered after prepare only
    out = work()
    fail = read_status()
    if fail == 0:
        return kl, out
    kl, _ = _jitter_ladder(engine, fail, base_jitter, constant_jitter)
    return kl, work()


def _param_key(tensors):
    """Identity + in-place version of every parameter tensor: unchanged key <=> unchanged factorisation inputs."""
    return tuple((t.data_ptr(), t._version, tuple(t.shape)) for t in tensors)


def _check_generation(ctx):
    if ctx.generation != ctx.engine.generation:
        raise RuntimeError('the model was evaluated again before backward(): the saved per-step workspace (L^-1, A, B) '
                           'has been overwritten; call backward() before the next ELBO / marginal evaluation')


def allreduce_packed(engine, rb):
    """THE collective of a training step (SURVEY.md §8e): sum over ranks of the pre-chain reduce buffer.  The two
    lower-triangular M x M blocks travel tril-packed (tgp_reduce_pack / tgp_reduce_unpack: 2 M^2 -> M (M + 1) doubles,
    16.9 -> 8.5 MB at M = 1024); slot 0 carries the ELL sum, so no second collective is needed for the loss value."""
    dist = _world()
    if dist is None:
        return rb
    packed = engine.pack_reduce(rb)
    dist.all_reduce(packed)
    engine.unpack_reduce(packed, rb)
    return rb


class _SumGradAcrossRanks(torch.autograd.Function):
    """Identity whose backward all-reduces (sum) the gradient: wraps parameters that are used on rank-local rows only."""

    @staticmethod
    def forward(ctx, p):
        return p.view_as(p)

    @staticmethod
    def backward(ctx, g):
        dist = _world()
        if dist is not None:
            g = g.contiguous().clone()
            dist.all_reduce(g)
        return g


def synced_module_call(module, X):
    """module(X), such that under row sharding every parameter of `module` receives the gradient summed over ranks.
    Used for the input-dependent flow MLPs (ID_TGP): they see only this rank's rows, and their gradients do not travel
    in the packed reduce buffer."""
    if _world() is None:
        return module(X)
    params = {n: _SumGradAcrossRanks.apply(p) for n, p in module.named_parameters()}
    return torch.func.functional_call(module, params, (X,))


class _ElboTerms(torch.autograd.Function):
    @staticmethod
    def forward(ctx, engine, X, Y, scale, check_status, jitter, sync_ell, Z, raw_ls, raw_os, m, L_raw, log_var_noise, theta,
                rowparams):
        need_grad = ctx.needs_input_grad[1] or any(ctx.needs_input_grad[7:])
        engine.set_params(Z.detach(), raw_ls.detach(), raw_os.detach(), m.detach(), L_raw.detach(),
                          None if log_var_noise is None else log_var_noise.detach(),
                          None if theta is None else theta.detach())
        rp = None if rowparams is None else rowparams.detach().contiguous()

        def work():
            mu, v = engine.qf_forward(X)
            rb = engine.new_reduce_buffer(fresh=False)
            return (mu, v, rb) + tuple(engine.ell_forward(mu, v, Y, rp, scale, rb, want_grad=need_grad))

        kl, (mu, v, rb, ell_rows, g_mu, g_v, drow) = prepare_then(engine, work, check=check_status,
                                                                  base_jitter=jitter[1], constant_jitter=jitter[0])
        ell = rb[engine.layout.ell_sum:engine.layout.ell_sum + 1].clone()
        dist = _world()
        if dist is not None and sync_ell:
            dist.all_reduce(ell)                   # every rank returns the GLOBAL ELL (cg.sync_elbo_in_forward)
        ctx.engine, ctx.X, ctx.rb, ctx.g = engine, X, rb, (g_mu, g_v, drow)
        ctx.generation = engine.generation
        ctx.has = (log_var_noise is not None, theta is not None, rowparams is not None)
        ctx.mark_non_differentiable(ell_rows, mu, v)
        return (ell * scale).reshape(()), kl.clone().reshape(()), ell_rows, mu, v

    @staticmethod
    def backward(ctx, g_ell, g_kl, _g_rows, _g_mu, _g_v):
        engine, X, rb = ctx.engine, ctx.X, ctx.rb
        g_mu, g_v, drow = ctx.g
        if g_mu is None:
            raise RuntimeError('backward called on an ELBO evaluated without gradients')
        _check_generation(ctx)
        dX = torch.zeros_like(X) if ctx.needs_input_grad[1] else None
        engine.qf_backward(X, g_mu, g_v, rb, dX)
        allreduce_packed(engine, rb)               # the one collective of the step (SURVEY.md §8e); dX is row-local
        engine.last_ell_sum = rb[engine.layout.ell_sum]        # global sum_n ell_n (unscaled), valid after backward
        zero = torch.zeros((), dtype=torch.float64, device=rb.device)
        g_dev = torch.stack([g_ell if g_ell is not None else zero, g_kl if g_kl is not None else zero]).contiguous()
        out = engine.chain_backward(rb, 0.0, 0.0, g_dev=g_dev)
        has_noise, has_theta, has_rowp = ctx.has
        g_rowp = drow * g_dev[0] if (has_rowp and drow is not None) else None
        g_X = dX * g_dev[0] if dX is not None else None            # the KL does not depend on X
        return (None, g_X, None, None, None, None, None, out['Z'], out['raw_ls'], out['raw_os'], out['m'], out['L_raw'],
                out['log_var_noise'] if has_noise else None, out['theta'] if has_theta else None, g_rowp)


def elbo_terms(engine, X, Y, scale, Z, raw_ls, raw_os, m, L_raw, log_var_noise, theta, rowparams=None,
               check_status=True, jitter=(0.0, None), sync_ell=True):
    """Returns (ELL, KLD, ell_rows, mu, v): ELL = scale * sum_n ell_n.

    Row-sharded (torch.distributed initialised): `sync_ell=True` sums ELL over ranks in the forward (every rank returns
    the global value, a second small collective per step); `sync_ell=False` returns the rank-local share — the global
    sum then rides in slot 0 of the one packed all-reduce of the backward (`engine.last_ell_sum`).  Gradients are the
    global ones in both cases.  `jitter` = (constant jitter, ladder base or None) — cg.constant_jitter / cg.global_jitter."""
    return _ElboTerms.apply(engine, X, Y, float(scale), bool(check_status), tuple(jitter), bool(sync_ell), Z, raw_ls,
                            raw_os, m, L_raw, log_var_noise, theta, rowparams)


def _on_factorisation(engine, params, frozen, work, check_status, jitter):
    """`work()` on the factorisation of `params` = (Z, raw_ls, raw_os, m, L_raw).  With frozen parameters (no gradient
    wanted) whose identity and version match the factorisation already in the step workspace, that factorisation is
    reused (evaluation over many batches; the reference refactorises K_zz for every batch, sparse_MF_SP.py:330);
    otherwise prepare_then factorises first."""
    key = _param_key(params) + (tuple(jitter),)
    if frozen and engine.prepared_key == key:
        engine.generation += 1
        return work()
    _, out = prepare_then(engine, work, check=check_status, base_jitter=jitter[1], constant_jitter=jitter[0])
    engine.prepared_key = key if check_status else None
    return out


class _QfMarginals(torch.autograd.Function):
    """mu, v of q(f) with a hand-written backward (used by marginal_variational_qf_parameters when called alone), and the
    KL term of the same factorisation: a model that needs both (the multiclass ELBO) cannot factorise twice, because the
    second factorisation would overwrite what the marginals' backward reads."""

    @staticmethod
    def forward(ctx, engine, X, check_status, jitter, Z, raw_ls, raw_os, m, L_raw):
        engine.set_params(Z.detach(), raw_ls.detach(), raw_os.detach(), m.detach(), L_raw.detach(), None, None)
        mu, v = _on_factorisation(engine, (Z, raw_ls, raw_os, m, L_raw), not any(ctx.needs_input_grad),
                                  lambda: engine.qf_forward(X), check_status, jitter)
        ctx.engine, ctx.X = engine, X
        ctx.generation = engine.generation
        return mu, v, engine.kl.clone().reshape(())        # the KL is in stream order once qf_forward has been enqueued

    @staticmethod
    def backward(ctx, g_mu, g_v, g_kl):
        engine, X = ctx.engine, ctx.X
        _check_generation(ctx)
        rb = engine.new_reduce_buffer()
        zeros = torch.zeros(X.shape[0], dtype=torch.float64, device=X.device)
        dX = torch.zeros_like(X) if ctx.needs_input_grad[1] else None
        engine.qf_backward(X, zeros if g_mu is None else g_mu.contiguous(), zeros if g_v is None else g_v.contiguous(), rb, dX)
        allreduce_packed(engine, rb)               # row-sharded callers (multiclass ELBO): sum over ranks before the chain
        if g_kl is None:
            out = engine.chain_backward(rb, 1.0, 0.0)
        else:
            g_dev = torch.stack([torch.ones((), dtype=torch.float64, device=X.device), g_kl.reshape(()).to(torch.float64)])
            out = engine.chain_backward(rb, g_dev=g_dev.contiguous())
        return None, dX, None, None, out['Z'], out['raw_ls'], out['raw_os'], out['m'], out['L_raw']


def qf_marginals(engine, X, Z, raw_ls, raw_os, m, L_raw, check_status=True, jitter=(0.0, None), with_kl=False):
    """(mu, v) of q(f) at the rows of X; with_kl=True: (mu, v, KL) with the KL term of the same factorisation."""
    mu, v, kl = _QfMarginals.apply(engine, X, bool(check_status), tuple(jitter), Z, raw_ls, raw_os, m, L_raw)
    return (mu, v, kl) if with_kl else (mu, v)


class _KlTerm(torch.autograd.Function):
    """KL[q(u) || p(u)] of one output GP from its own factorisation (sparse_MF_SP.KLD of a non-whitened model, whose KL
    depends on K_zz).  The backward is the chain with a zero reduce buffer and gE = 0."""

    @staticmethod
    def forward(ctx, engine, jitter, Z, raw_ls, raw_os, m, L_raw):
        engine.set_params(Z.detach(), raw_ls.detach(), raw_os.detach(), m.detach(), L_raw.detach(), None, None)
        # the status read blocks the host until the factorisation, and the KL behind it, is done (no entry point consumes
        # the factorisation in this forward): it is also the psd_safe_cholesky check of the reference's KLD
        kl, _ = prepare_then(engine, lambda: None, check=True, base_jitter=jitter[1], constant_jitter=jitter[0])
        ctx.engine = engine
        ctx.generation = engine.generation
        return kl.clone().reshape(())

    @staticmethod
    def backward(ctx, g_kl):
        engine = ctx.engine
        _check_generation(ctx)
        g_dev = torch.stack([torch.zeros((), dtype=torch.float64, device=g_kl.device), g_kl.reshape(()).to(torch.float64)])
        out = engine.chain_backward(engine.new_reduce_buffer(), g_dev=g_dev.contiguous())
        return None, None, out['Z'], out['raw_ls'], out['raw_os'], out['m'], out['L_raw']


def kl_term(engine, Z, raw_ls, raw_os, m, L_raw, jitter=(0.0, None)):
    return _KlTerm.apply(engine, tuple(jitter), Z, raw_ls, raw_os, m, L_raw)


def qf_covariance(engine, X, Z, raw_ls, raw_os, m, L_raw, check_status=True, jitter=(0.0, None)):
    """(mu (R,), Sigma (R, R)) of q(f) at the rows of X: the full covariance over the batch (tgp_qf_cov_forward), FP64 in
    every compute mode.  Evaluation only: there is no backward, so a call that would need one raises instead of returning
    a silently detached result.  Under row sharding each rank gets the covariance of its own rows."""
    params = (Z, raw_ls, raw_os, m, L_raw)
    if torch.is_grad_enabled() and any(t.requires_grad for t in params + (X,)):
        raise NotImplementedError('the full covariance of q(f) has no backward: call it under torch.no_grad()')
    engine.set_params(Z.detach(), raw_ls.detach(), raw_os.detach(), m.detach(), L_raw.detach(), None, None)
    return _on_factorisation(engine, params, True, lambda: engine.qf_cov(X), check_status, jitter)


def cov_cholesky_ladder(engine, cov, base_jitter=None, constant_jitter=0.0):
    """L with L L^T = cov + jitter I, with the semantics of psd_safe_cholesky (code/dsp/utils.py:222-270) as in
    _jitter_ladder: factorise with the constant jitter only; on failure check for NaN (NanError), then add base * 10^i,
    i = 0..2, warning each time; raise after the third failure.  base: as sparse_MF_SP._jitter() (default 1e-8).
    Returns (L, jitter added on top of the constant one)."""
    L, status = engine.cov_cholesky(cov, constant_jitter)
    fail = int(status.item())
    if fail == 0:
        return L, 0.0
    if torch.isnan(cov).any():
        raise NanError('cholesky: the covariance matrix has NaN entries')
    jitter = 1e-8 if base_jitter is None else base_jitter
    for i in range(3):
        j = jitter * (10 ** i)
        L, status = engine.cov_cholesky(cov, constant_jitter + j)
        if int(status.item()) == 0:
            warnings.warn('A not p.d., added jitter of %g to the diagonal' % j, NumericalWarning)
            return L, j
    raise RuntimeError('cholesky: matrix not positive definite after 3 jitter escalations (first bad pivot %d)' % fail)


# ---- input-dependent flow MLPs on the device (tgp_flow_mlp_forward / _backward) ---------------------------------------
_ACT_CODE = {'ReLU': 0, 'Tanh': 1, 'Sigmoid': 2, 'Identity': 3}
_PHILOX_OFFSET = {}


def mlp_spec(nets):
    """Architecture of a list of flow MLPs if the fused kernel covers it, else None: every net =
    num_H x [Linear -> activation -> (Dropout)] + [Linear(H, 1)], identical shapes, no batch-norm, H <= 64, n_in <= 64."""
    import torch.nn as nn
    spec = None
    for net in nets:
        blocks = [list(b.forward_lin) if hasattr(b, 'forward_lin') else None for b in net]
        if any(b is None for b in blocks) or len(blocks) < 2:
            return None
        hidden, last = blocks[:-1], blocks[-1]
        if not (isinstance(last[0], nn.Linear) and last[0].out_features == 1 and all(isinstance(m, nn.Identity) for m in last[1:])):
            return None
        p, act, drops = 0.0, None, []
        for b in hidden:
            if not isinstance(b[0], nn.Linear) or len(b) < 2 or type(b[1]).__name__ not in _ACT_CODE:
                return None
            rest = b[2:]
            if len(rest) > 1 or (rest and 'Dropout' not in type(rest[0]).__name__):
                return None
            if rest:
                p = float(rest[0].p)
                drops.append(rest[0])
            act = type(b[1]).__name__ if act is None else act
            if type(b[1]).__name__ != act:
                return None
        H, n_in = hidden[0][0].out_features, hidden[0][0].in_features
        if any(b[0].out_features != H for b in hidden) or H > 64 or n_in > 64 or len(hidden) > 4 or last[0].in_features != H:
            return None
        if drops and len(drops) != len(hidden):
            return None
        cur = dict(n_in=n_in, H=H, L=len(hidden), act=_ACT_CODE[act], p=p, training=bool(drops) and any(d.training for d in drops))
        if spec is None:
            spec = cur
        elif spec != cur:
            return None
    return spec


def _mlp_weights(nets):
    ws = []
    for net in nets:
        for b in net:
            lin = b.forward_lin[0]
            ws += [lin.weight, lin.bias]
    return ws


class _FlowMlp(torch.autograd.Function):
    @staticmethod
    def forward(ctx, X, spec, mask_in, owner, n_nets, *weights):
        import ctypes as C
        lib = _lib.load()
        dev = X.device
        m = _lib.TgpMlp()
        m.n_nets, m.n_in, m.hidden, m.n_hidden_layers, m.activation = n_nets, spec['n_in'], spec['H'], spec['L'], spec['act']
        drop = spec['training'] and spec['p'] > 0.0
        m.mask_mode = 0 if not drop else (2 if mask_in is not None else 1)
        m.p_drop = spec['p'] if drop else 0.0
        Xc = X.detach().to(torch.float64).contiguous()
        R = Xc.shape[0]
        Wp = torch.cat([w.detach().reshape(-1).to(torch.float64) for w in weights]).contiguous()
        assert Wp.numel() == n_nets * lib.tgp_flow_mlp_net_doubles(m), 'flow MLP weight packing does not match the kernel layout'
        out = torch.empty(R, n_nets, dtype=torch.float64, device=dev)
        mask = None
        if m.mask_mode == 2:
            mask = mask_in.to(device=dev, dtype=torch.uint8).contiguous()
            if tuple(mask.shape) != (n_nets, spec['L'], R, spec['H']):
                raise ValueError('dropout mask must have shape (n_nets, n_hidden_layers, rows, hidden) = %s, got %s'
                                 % ((n_nets, spec['L'], R, spec['H']), tuple(mask.shape)))
        mask_out = torch.empty(n_nets, spec['L'], R, spec['H'], dtype=torch.uint8, device=dev) if m.mask_mode == 1 else None
        off = None
        if m.mask_mode == 1:
            key = str(dev)
            if key not in _PHILOX_OFFSET:
                _PHILOX_OFFSET[key] = torch.zeros(1, dtype=torch.int64, device=dev)
            off = _PHILOX_OFFSET[key]
        from .dsp import config as cg
        dist = _world()
        seed = (int(cg.config_seed) * 0x9E3779B97F4A7C15 + (dist.get_rank() if dist is not None else 0) * 0xD1B54A32D192ED03 + 0x1234567) % (1 << 64)
        with torch.cuda.device(dev):
            st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            _lib.check(lib.tgp_flow_mlp_forward(m, Wp.data_ptr(), Xc.data_ptr(), R, None if mask is None else mask.data_ptr(),
                                                None if mask_out is None else mask_out.data_ptr(), seed,
                                                None if off is None else off.data_ptr(), out.data_ptr(), st), 'tgp_flow_mlp_forward')
        used = mask if m.mask_mode == 2 else mask_out
        if owner is not None:
            owner.last_dropout_masks = used                  # exported keep-mask of this call (None when dropout is off)
        ctx.m, ctx.Xc, ctx.Wp, ctx.mask, ctx.shapes, ctx.dtypes = m, Xc, Wp, used, [w.shape for w in weights], [w.dtype for w in weights]
        ctx.x_dtype = X.dtype
        return out

    @staticmethod
    def backward(ctx, dout):
        import ctypes as C
        lib = _lib.load()
        dev = ctx.Xc.device
        dW = torch.zeros_like(ctx.Wp)
        dX = torch.zeros_like(ctx.Xc) if ctx.needs_input_grad[0] else None
        d = dout.to(torch.float64).contiguous()
        with torch.cuda.device(dev):
            st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            mask = None if ctx.mask is None else ctx.mask.data_ptr()
            if dX is None:
                _lib.check(lib.tgp_flow_mlp_backward(ctx.m, ctx.Wp.data_ptr(), ctx.Xc.data_ptr(), ctx.Xc.shape[0], mask, d.data_ptr(),
                                                     dW.data_ptr(), st), 'tgp_flow_mlp_backward')
            else:
                _lib.check(lib.tgp_flow_mlp_backward_dx(ctx.m, ctx.Wp.data_ptr(), ctx.Xc.data_ptr(), ctx.Xc.shape[0], mask,
                                                        d.data_ptr(), dW.data_ptr(), dX.data_ptr(), st), 'tgp_flow_mlp_backward_dx')
        dist = _world()
        if dist is not None:
            dist.all_reduce(dW)          # each rank saw its own rows only: ONE collective for all MLP weights of the layer
        grads, o = [], 0
        for shp, dt in zip(ctx.shapes, ctx.dtypes):
            n = 1
            for k in shp:
                n *= k
            grads.append(dW[o:o + n].reshape(shp).to(dt))
            o += n
        return (None if dX is None else dX.to(ctx.x_dtype), None, None, None, None) + tuple(grads)


def flow_mlp(owner, nets, spec, X, mask_in=None):
    """theta(x_n) of `len(nets)` flow MLPs in one kernel: (R, n_nets).  Differentiable w.r.t. the MLP weights and X."""
    return _FlowMlp.apply(X, spec, mask_in, owner, len(nets), *_mlp_weights(nets))
