"""Load `tests/golden/*.npz` (written by oracle/make_golden.py) into oracle-style parameter dicts."""
import glob
import hashlib
import json
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def golden_names(big=None):
    """Fixture names; big=False / True selects the small fixtures / the two at the BASELINE.json sizes (M = 1024, 2048)."""
    names = sorted(os.path.basename(f)[:-4] for f in glob.glob(os.path.join(GOLDEN_DIR, '*.npz'))
                   if not os.path.basename(f).startswith(('traj_', 'mc_')))
    if big is None:
        return names
    return [n for n in names if (('_m1024_' in n or '_m2048_' in n) == big)]


def multiclass_names():
    """Fixtures of the Monte-Carlo softmax likelihood (one GP per class; oracle/make_golden.py main_multiclass)."""
    return sorted(os.path.basename(f)[:-4] for f in glob.glob(os.path.join(GOLDEN_DIR, 'mc_*.npz')))


def trajectory_names():
    return sorted(os.path.basename(f)[:-4] for f in glob.glob(os.path.join(GOLDEN_DIR, 'traj_*.npz')))


def flow_grad_keys(spec, constrained=False):
    """Leaf names (oracle.leaf_params keys) of a fixture's flow scalars in the REFERENCE's module order — the order in which
    `named_parameters()` lists them; None where the stored gradient is not comparable."""
    keys = []
    for i, lay in enumerate(spec):
        if lay[0] == 'affine':
            keys += ['flow%d.a' % i, 'flow%d.b' % i]
        elif lay[0] == 'tanh_step':
            for j in range(len(lay[1])):
                keys += ['flow%d.%d.%s' % (i, j, c) for c in 'abcd']
        elif lay[0] == 'sal':
            keys += ['flow%d.a' % i, 'flow%d.b' % i]
        elif lay[0] == 'arcsinh':
            keys += ['flow%d.%s' % (i, c) for c in 'abcd']
        elif lay[0] in ('boxcox', 'invboxcox'):
            # the layer's leaf is lam AFTER the module's constraint; the reference's gradient is w.r.t. the raw
            # parameter: comparable only when there is no constraint (the class-API tests cover the chain)
            keys += ['flow%d.lam' % i if not constrained else None]
        elif lay[0] == 'step_group':
            # module order of the reference's StepFlow: every trainable switch_off first, then the members
            own = {'tanh_step': 'abcd', 'sal': 'ab', 'arcsinh': 'abcd'}
            for j, (m, sw) in enumerate(lay[1]):
                if sw is not None:
                    keys += ['flow%d.m%d.sw_a' % (i, j), 'flow%d.m%d.sw_b' % (i, j)]
            for j, (m, sw) in enumerate(lay[1]):
                if m[0] == 'tanh_step':
                    keys += ['flow%d.m%d.0.%s' % (i, j, c) for c in 'abcd']
                elif m[0] in ('boxcox', 'invboxcox'):
                    keys += ['flow%d.m%d.lam' % (i, j) if not constrained else None]
                else:
                    keys += ['flow%d.m%d.%s' % (i, j, c) for c in own[m[0]]]
    return keys


def variational_grid(M, seed):
    """(1, M, M) variational factor of the BASELINE-size fixtures (oracle/make_golden.randomise_big): 0.5 I + 0.05 k / 8 on
    the lower triangle, k drawn uniformly from -8..8 by a torch CPU generator seeded with `seed`."""
    g = torch.Generator().manual_seed(int(seed))
    q = torch.randint(-8, 9, (1, M, M), generator=g).double() / 8.0
    return (0.5 * torch.eye(M, dtype=torch.float64).unsqueeze(0) + 0.05 * q).tril().numpy()


class _Arrays(dict):
    """The arrays of one fixture; `.files` lists the keys, as on the NpzFile they were read from."""

    @property
    def files(self):
        return list(self)


def _load_fixture(path):
    """Reads a fixture; a parameter stored as `paramgrid:<name>` = (seed, M) is regenerated with `variational_grid` and
    checked against the SHA-256 of the parameter the reference was run with (`paramsha256:<name>`)."""
    with np.load(path, allow_pickle=False) as z:
        arrays = _Arrays((k, z[k]) for k in z.files)
    for key in [k for k in arrays if k.startswith('paramgrid:')]:
        name = key[len('paramgrid:'):]
        seed, M = (int(x) for x in arrays.pop(key))
        a = variational_grid(M, seed)
        want = str(arrays.pop('paramsha256:' + name))
        if hashlib.sha256(a.tobytes()).hexdigest() != want:
            raise RuntimeError('%s: %s regenerated from seed %d differs from the stored SHA-256 (torch CPU generator changed?)'
                               % (os.path.basename(path), name, seed))
        arrays['param:' + name] = a
    return arrays


class Golden:
    def __init__(self, name):
        self.name = name
        self.z = _load_fixture(os.path.join(GOLDEN_DIR, name + '.npz'))
        self.meta = json.loads(str(self.z['meta']))

    def t(self, key, dtype=torch.float64):
        return torch.tensor(np.asarray(self.z[key]), dtype=dtype)

    def _flow(self, spec, dtype, leaf_cache):
        def get(k):
            if k not in leaf_cache:
                leaf_cache[k] = self.t(k, dtype)
            return leaf_cache[k]
        layers = []
        for lay in spec:
            if lay[0] == 'step_group':
                members = [(self._flow([m], dtype, leaf_cache)[0], None if sw is None else (get(sw[0]), get(sw[1])))
                           for m, sw in lay[1]]
                layers.append(('step_group', members, lay[2]))
            elif lay[0] == 'identity':
                layers.append(('identity',))
            elif lay[0] == 'affine':
                layers.append(('affine', get(lay[1]), get(lay[2]), lay[3]))
            elif lay[0] == 'tanh_step':
                layers.append(('tanh_step', [tuple(get(k) for k in st) for st in lay[1]], lay[2]))
            elif lay[0] == 'sal':
                layers.append(('sal', get(lay[1]), get(lay[2]), lay[3], lay[4]))
            elif lay[0] == 'arcsinh':
                layers.append(('arcsinh', get(lay[1]), get(lay[2]), get(lay[3]), get(lay[4]), lay[5], lay[6]))
            elif lay[0] in ('boxcox', 'invboxcox'):
                layers.append((lay[0], get(lay[1]), lay[2]))
        return layers

    def oracle_params(self, which='train', dtype=torch.float64):
        p = {}
        for n in self.meta['param_names']:
            a = self.t('param:' + n, dtype)
            if n == 'Z':
                p['Z'] = a[0]
            elif n.endswith('raw_lengthscale'):
                p['raw_lengthscale'] = a.view(-1)
            elif n.endswith('raw_outputscale'):
                p['raw_outputscale'] = a.view(())
            elif n.endswith('variational_mean'):
                p['m'] = a[0]
            elif n.endswith('chol_variational_covar'):
                p['L_raw'] = a[0]
            elif n.endswith('log_var_noise'):
                p['log_var_noise'] = a.view(())
        if 'log_var_noise' not in p:       # Bernoulli has no noise parameter
            p['log_var_noise'] = torch.zeros((), dtype=dtype)
        self._leaf = {}
        p['flow'] = self._flow(self.meta['flow_train' if which == 'train' else 'flow_test'], dtype, self._leaf)
        return p

    def ref_grads(self):
        """name -> reference gradient, keyed like oracle.leaf_params (global scalars only)."""
        g = {}
        names = self.meta['param_names']
        for n in names:
            if 'grad:' + n not in self.z.files:      # BASELINE-size fixtures keep the M x M gradient as checksums
                continue
            a = self.t('grad:' + n)
            if n == 'Z':
                g['Z'] = a[0]
            elif n.endswith('raw_lengthscale'):
                g['raw_lengthscale'] = a.view(-1)
            elif n.endswith('raw_outputscale'):
                g['raw_outputscale'] = a.view(())
            elif n.endswith('variational_mean'):
                g['m'] = a[0]
            elif n.endswith('chol_variational_covar'):
                g['L_raw'] = a[0]
            elif n.endswith('log_var_noise'):
                g['log_var_noise'] = a.view(())
        # flow scalars, in module order == oracle layer order
        if not self.meta['id_flow']:
            flow_names = [n for n in names if n.startswith('G_matrix')]
            vals = [self.t('grad:' + n).view(()) for n in flow_names]
            keys = flow_grad_keys(self.meta['flow_train'], self.meta.get('boxcox_constraint'))
            assert len(keys) == len(vals), (keys, flow_names)
            g.update({k: v for k, v in zip(keys, vals) if k is not None})
        return g


    def grad_errors(self, grads):
        """L2-relative error of every gradient in `grads` (keyed like `ref_grads`) against the reference's.  For the
        BASELINE-size fixtures the M x M gradient of chol_variational_covar is checked through the stored checksums
        (G R, G^T R for oracle/make_golden.projection_basis, the diagonal and the Frobenius norm)."""
        errs = {k: rel_err(torch.as_tensor(grads[k]).detach().cpu(), gr) for k, gr in self.ref_grads().items() if k in grads}
        key = [n for n in self.meta['param_names'] if n.endswith('chol_variational_covar')][0]
        if 'gradproj:' + key in self.z.files:
            G = torch.as_tensor(grads['L_raw']).detach().cpu().double()
            R = torch.tensor(projection_basis(G.shape[0]))
            proj = self.t('gradproj:' + key)
            errs['L_raw.GR'] = rel_err(G @ R, proj[0])
            errs['L_raw.GtR'] = rel_err(G.t() @ R, proj[1])
            errs['L_raw.diag'] = rel_err(torch.diagonal(G), self.t('graddiag:' + key))
            errs['L_raw.norm'] = rel_err(G.norm(), self.t('gradnorm:' + key))
        return errs


def projection_basis(M, k=6):
    """Same matrix as oracle/make_golden.projection_basis (exact dyadic rationals, identical on every host)."""
    i = np.arange(M, dtype=np.int64)[:, None]
    c = np.arange(k, dtype=np.int64)[None, :]
    return (((i * 2654435761 + (c + 1) * 40503 + i * c * 97) % 1024).astype(np.float64) / 1024.0) - 0.5


def rel_err(a, b):
    a = torch.as_tensor(a, dtype=torch.float64).reshape(-1)
    b = torch.as_tensor(b, dtype=torch.float64).reshape(-1)
    den = float(b.norm())
    return float((a - b).norm()) / (den if den > 0 else 1.0)


class MulticlassGolden(Golden):
    """Fixture of the Monte-Carlo softmax likelihood: C GPs, one flow each (same architecture), recorded noise draws."""

    def plist(self, dtype=torch.float64):
        """One oracle parameter dict per class."""
        C = self.meta['C']
        out = []
        for c in range(C):
            p = {'Z': self.t('param:Z', dtype)[c].clone(),
                 'raw_lengthscale': self.t('param:covariance_function.base_kernel.raw_lengthscale', dtype)[c].reshape(-1).clone(),
                 'raw_outputscale': self.t('param:covariance_function.raw_outputscale', dtype)[c].reshape(()).clone(),
                 'm': self.t('param:q_U.variational_mean', dtype)[c].clone(),
                 'L_raw': self.t('param:q_U.chol_variational_covar', dtype)[c].clone(),
                 'log_var_noise': torch.zeros((), dtype=dtype)}
            p['flow'] = self._flow(self.meta['flows'][c], dtype, {})
            out.append(p)
        return out

    def ref_grads_of_class(self, c):
        g = {'Z': self.t('grad:Z')[c],
             'raw_lengthscale': self.t('grad:covariance_function.base_kernel.raw_lengthscale')[c].reshape(-1),
             'raw_outputscale': self.t('grad:covariance_function.raw_outputscale')[c].reshape(()),
             'm': self.t('grad:q_U.variational_mean')[c],
             'L_raw': self.t('grad:q_U.chol_variational_covar')[c]}
        names = [n for n in self.meta['param_names'] if n.startswith('G_matrix.%d.' % c)]
        keys = flow_grad_keys(self.meta['flows'][c])
        assert len(keys) == len(names), (keys, names)
        g.update({k: self.t('grad:' + n).reshape(()) for k, n in zip(keys, names)})
        return g
