"""Pins tests/mc_id_ref.py, the reference for input-dependent flows under the Monte-Carlo softmax likelihood, to the fixtures of
the unmodified reference.  No fixture of that combination exists, so the pin is an identity: an input-dependent model whose
read-out layers have zero weights and the fixture's raw flow scalars as biases outputs those scalars at every row, and so
computes the fixture's global-flow model.  The read-out bias enters theta_c(x_n) with slope 1 at every row, so its gradient is
sum_n d/d rowp[c, n], which must equal the fixture's d/d theta."""
import pytest
import torch

from oracle import tgp_oracle as O
from tests import mc_id_ref as R
from tests.golden_util import MulticlassGolden, rel_err

# the fixtures whose flows have input-dependent forms (StepSAL's members carry a trainable switch_off, which stays global-only)
NAMES = ['mc_synth_c3_sal1_p1', 'mc_synth_c4_steptanh12_p1']
GP = ('Z', 'raw_lengthscale', 'raw_outputscale', 'm', 'L_raw')
FIX_TOL = 1e-11


def _readout_biases(flow):
    """(O.layer_leaves name of the scalar each per-row net replaces, read-out bias tensor) of one input-dependent layer list."""
    out = []
    for i, lay in enumerate(flow):
        if lay[0] == 'sal' and isinstance(lay[1], R.Net):
            out += [('flow%d.a' % i, lay[1].weights[-1][1]), ('flow%d.b' % i, lay[2].weights[-1][1])]
        elif lay[0] == 'tanh_step' and isinstance(lay[1][0][0], R.Net):
            for j, st in enumerate(lay[1]):
                out += [('flow%d.%d.%s' % (i, j, c), net.weights[-1][1]) for c, net in zip('abcd', st)]
    return out


@pytest.mark.parametrize('act', ['tanh', 'relu'])
@pytest.mark.parametrize('name', NAMES)
def test_zero_readout_restatement_reproduces_the_fixture(name, act):
    g = MulticlassGolden(name)
    X, y, eps, N = g.t('X'), g.t('Y').reshape(-1), g.t('eps'), g.meta['N']
    gen = torch.Generator().manual_seed(11)
    plist = g.plist()
    # dropout masks change nothing behind a zero read-out
    id_plist = [dict(p, flow=R.zero_readout(p['flow'], X.shape[1], 7, 2, gen, rows=X.shape[0], p_drop=0.3)) for p in plist]
    biases = [dict(_readout_biases(p['flow'])) for p in id_plist]
    assert all(len(b) > 0 for b in biases)
    leaves = []
    for c, p in enumerate(id_plist):
        lv = {k: p[k] for k in GP}
        lv.update(biases[c])
        for i, lay in enumerate(p['flow']):                 # global layers kept from the fixture (the affine read-out)
            if lay[0] == 'affine':
                lv.update(O.layer_leaves(lay, 'flow%d' % i))
        for t in lv.values():
            t.requires_grad_(True)
        leaves.append(lv)
    E, ELL, KLD, rows, mu, v = R.elbo_multiclass(X, y, id_plist, N, eps, act, 0.3)
    grads = torch.autograd.grad(E, [t for lv in leaves for t in lv.values()])
    it = iter(grads)
    got = [{k: next(it) for k in lv} for lv in leaves]

    # O2 on the global-flow fixture itself
    plist_o = g.plist()
    o_leaves = [O.leaf_params(p) for p in plist_o]
    for lv in o_leaves:
        lv.pop('log_var_noise')
        for t in lv.values():
            t.requires_grad_(True)
    E0, ELL0, KLD0, rows0, _, _ = O.elbo_multiclass(X, y, plist_o, N, eps)
    grads0 = torch.autograd.grad(E0, [t for lv in o_leaves for t in lv.values()])
    it = iter(grads0)
    ref = [{k: next(it) for k in lv} for lv in o_leaves]

    for a, b in ((E, E0), (ELL, ELL0), (KLD, KLD0), (rows, rows0)):
        assert rel_err(a.detach(), b.detach()) < 1e-11
    for a, key in ((E, 'ELBO'), (ELL, 'ELL'), (KLD, 'KLD')):
        assert rel_err(a.detach(), g.t(key)) < 1e-11, key
    for c in range(g.meta['C']):
        fix = g.ref_grads_of_class(c)
        for k in got[c]:
            assert rel_err(got[c][k], ref[c][k]) < 1e-11, (c, k)
            assert rel_err(got[c][k], fix[k]) < FIX_TOL, (c, k)
        # every flow scalar of the fixture is accounted for: the per-row ones through their read-out biases
        assert set(got[c]) - set(GP) == set(fix) - set(GP)


def test_per_row_parameters_broadcast_like_global_ones():
    """A per-row parameter equal at every row gives the rows of the global flow, and the sum of its per-row gradients is the
    global gradient: the property the kernel's per-row accumulator relies on."""
    g = MulticlassGolden(NAMES[0])
    plist = g.plist()
    mu, v, y, eps = g.t('mu'), g.t('v'), g.t('Y').reshape(-1), g.t('eps')
    R_ = mu.shape[1]
    flows = [p['flow'] for p in plist]
    a = [f[0][1].clone().requires_grad_(True) for f in flows]
    ar = [t.detach().expand(R_).clone().requires_grad_(True) for t in a]
    rows_g = O.ell_rows_mc_softmax(mu, v, y, [[('sal', a[c], f[0][2], f[0][3], f[0][4])] + f[1:] for c, f in enumerate(flows)], eps)
    rows_r = O.ell_rows_mc_softmax(mu, v, y, [[('sal', ar[c], f[0][2], f[0][3], f[0][4])] + f[1:] for c, f in enumerate(flows)], eps)
    assert torch.equal(rows_g, rows_r)
    ga = torch.autograd.grad(rows_g.sum(), a)
    gr = torch.autograd.grad(rows_r.sum(), ar)
    for c in range(len(flows)):
        assert rel_err(gr[c].sum(), ga[c]) < 1e-13
