"""CPU reference for input-dependent flows under the Monte-Carlo softmax likelihood (multiclass ID-TGP).  Test infrastructure,
not product.

Every class c has its own flow, all of one architecture.  An input-dependent layer holds, in place of each of its scalar
parameters, one MLP: theta_c(x) = O.flow_mlp(X, weights, act, p, masks), the net of reference models/flow.py:853-871 evaluated
on the rows once per call (:949-950).  The per-row tensors (MB,) then go into O2's own layer lists, whose `apply_flow`
broadcasts them over the (S, MB) samples, and from there into `O.ell_rows_mc_softmax` / `O.probs_mc_softmax` unchanged.

A per-row parameter is written `Net(weights, masks)`: weights [(W_0, b_0), ..., (W_out, b_out)] as torch Linear stores them,
masks a list of keep-masks (rows, H), one per hidden layer, or None (dropout off).  Global parameters stay tensors of shape ().
Supported layers: ('sal', a, b, restrict, add_f0), ('tanh_step', [(a, b, c, d), ...], add_f0) with per-row or global
parameters (one kind per layer) and O2's global layers.

The reference itself cannot be run on this combination offline: its own path is pinned through the identity of
`zero_readout`, which turns a global-flow fixture into an input-dependent model computing exactly the same numbers.
"""
from collections import namedtuple

import torch

from oracle import tgp_oracle as O

Net = namedtuple('Net', 'weights masks')


def _value(par, X, act, p_drop):
    return O.flow_mlp(X, par.weights, act, p_drop, par.masks) if isinstance(par, Net) else par


def evaluate(layers, X, act, p_drop=0.0):
    """One class's layer list with its MLPs evaluated at the rows of X (R, D): an O2 layer list with (R,) parameters."""
    out = []
    for lay in layers:
        if lay[0] == 'sal':
            out.append(('sal', _value(lay[1], X, act, p_drop), _value(lay[2], X, act, p_drop), lay[3], lay[4]))
        elif lay[0] == 'tanh_step':
            out.append(('tanh_step', [tuple(_value(t, X, act, p_drop) for t in st) for st in lay[1]], lay[2]))
        else:
            out.append(lay)
    return out


def class_flows(flows, X, act, p_drop=0.0):
    """C layer lists -> C O2 layer lists at the rows of X (R, D) or (C, R, D)."""
    return [evaluate(f, X[c] if X.dim() == 3 else X, act, p_drop) for c, f in enumerate(flows)]


def ell_rows(mu, v, y, flows, X, eps, act, p_drop=0.0):
    return O.ell_rows_mc_softmax(mu, v, y, class_flows(flows, X, act, p_drop), eps)


def probs(mu, v, flows, X, eps, act, p_drop=0.0):
    return O.probs_mc_softmax(mu, v, class_flows(flows, X, act, p_drop), eps)


def elbo_multiclass(X, y, plist, N, eps, act, p_drop=0.0, whiten=True):
    """As O.elbo_multiclass, with plist[c]['flow'] an input-dependent layer list: (ELBO, ELL, KLD, rows, mu (C, MB), v (C, MB)).
    whiten=False: the non-whitened q(u) of tests/unwhitened_ref.py."""
    if whiten:
        qf, kl = O.qf_marginals, O.kl_whitened
    else:
        from tests import unwhitened_ref as U
        qf, kl = U.qf_marginals, U.kl
    mv = [qf(X, p) for p in plist]
    mu, v = torch.stack([a for a, _ in mv]), torch.stack([b for _, b in mv])
    rows = ell_rows(mu, v, y, [p['flow'] for p in plist], X, eps, act, p_drop)
    ELL = (float(N) / X.shape[0]) * rows.sum()
    KLD = torch.stack([kl(p) for p in plist]).sum()
    return ELL - KLD, ELL, KLD, rows, mu, v


def random_net(D, H, L, gen, scale=0.5, dtype=torch.float64):
    """A net of L hidden layers of width H on D inputs, with N(0, scale^2) weights drawn from `gen`."""
    dims = [D] + [H] * L
    w = [(scale * torch.randn(dims[i + 1], dims[i], generator=gen, dtype=dtype), scale * torch.randn(dims[i + 1], generator=gen, dtype=dtype))
         for i in range(L)]
    w.append((scale * torch.randn(1, H, generator=gen, dtype=dtype), scale * torch.randn(1, generator=gen, dtype=dtype)))
    return Net(w, None)


def zero_readout(layers, D, H, L, gen, rows=None, p_drop=0.0):
    """The input-dependent restatement of a global-flow layer list: every parameter of its sal / tanh_step layers becomes a net
    with random hidden layers, a read-out of zero weights and the raw scalar as its bias.  Such a net outputs exactly that
    scalar at every row, whatever its hidden layers and dropout masks, so the model computes the global-flow one.  With
    p_drop > 0 every net also gets random keep-masks for `rows` rows."""
    def net(scalar):
        n = random_net(D, H, L, gen)
        masks = None if p_drop == 0.0 else [(torch.rand(rows, H, generator=gen) > p_drop).to(torch.uint8) for _ in range(L)]
        return Net(n.weights[:-1] + [(torch.zeros(1, H, dtype=scalar.dtype), scalar.detach().clone().reshape(1))], masks)
    out = []
    for lay in layers:
        if lay[0] == 'sal':
            out.append(('sal', net(lay[1]), net(lay[2]), lay[3], lay[4]))
        elif lay[0] == 'tanh_step':
            out.append(('tanh_step', [tuple(net(t) for t in st) for st in lay[1]], lay[2]))
        else:
            out.append(lay)
    return out
