"""CPU tests of the host side: the dsp mirror builds reference-shaped modules (same parameter names), flow
descriptors pack as the kernels expect, the C-ABI library loads and exports every declared symbol, and the product
refuses to run without a GPU instead of falling back."""
import os
import re

import pytest
import torch

from tests.golden_util import Golden, golden_names
from tests.model_util import build_from_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_exports_every_declared_symbol():
    from tgp.pytorch_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, 'include', 'tgp_b200.h')).read()
    declared = set(re.findall(r'\b(tgp_[a-z0-9_]+)\s*\(', header))
    assert declared, 'no declarations found'
    for name in declared:
        assert hasattr(lib, name), 'library does not export %s' % name
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))
    assert lib.tgp_version() >= 100


def test_cabi_rejects_bad_descriptions_without_a_gpu():
    from tgp.pytorch_b200 import _lib
    lib = _lib.load()
    m = _lib.TgpModel()
    m.M, m.D, m.likelihood, m.n_quad = 0, 3, 1, 100
    assert lib.tgp_step_workspace_bytes(m) == 0
    assert b'positive' in lib.tgp_last_error()
    m.M = 16
    m.dtype = 7
    assert lib.tgp_step_workspace_bytes(m) == 0
    m.dtype = _lib.TGP_F32
    assert lib.tgp_step_workspace_bytes(m) > 0
    m.dtype = _lib.TGP_F64
    assert lib.tgp_step_workspace_bytes(m) > 0
    lay = _lib.TgpReduceLayout()
    assert lib.tgp_reduce_layout(m, lay) == 0
    assert lay.total == lay.Cbar + 64 * 64 and lay.Gbar % 2 == 0


@pytest.mark.parametrize('name', golden_names())
def test_models_reproduce_reference_parameter_names(name):
    g = Golden(name)
    model = build_from_golden(g, 'cpu')          # asserts the name sets are identical
    assert model.M == g.meta['M'] and model.out_dim == 1


def test_flow_descriptor_packing():
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    from tgp.pytorch_b200.dsp.flows import StepTanhL, SAL
    from tgp.pytorch_b200.dsp.models.flow import instance_flow
    from tgp.pytorch_b200.engine import FlowLayout
    fl = instance_flow(StepTanhL(2, 3, add_f0=True))
    layers, glob, rows = fl.describe()
    lay = FlowLayout(layers)
    assert [l['kind'] for l in lay.layers] == ['tanh_step', 'affine', 'tanh_step', 'affine']
    assert lay.n_theta == len(glob) == 2 * (3 * 4 + 2) and lay.n_rowparams == 0 and not rows
    assert [l['p0'] for l in lay.layers] == [0, 12, 14, 26]
    idf = instance_flow(SAL(2, input_dependent=True, input_dim=4, hidden_dim=5, dropout=0.25, num_hidden_layers=2))
    idf.turn_off_initializer_parameters()
    layers, glob, rows = idf.describe(torch.randn(7, 4, dtype=torch.float64))
    lay = FlowLayout(layers)
    assert lay.n_rowparams == 4 and lay.n_theta == 4 and len(rows) == 4 and rows[0].shape == (7,)
    assert [(l['per_row'], l['p0']) for l in lay.layers] == [(True, 0), (False, 0), (True, 2), (False, 2)]


def test_flow_modules_match_oracle_forward():
    """The torch `forward` of the flow modules (used by initialisers / sampling) agrees with the oracle's flows."""
    from oracle import tgp_oracle as O
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    from tgp.pytorch_b200.dsp.flows import StepTanhL, SAL
    from tgp.pytorch_b200.dsp.models.flow import instance_flow
    f = torch.linspace(-3, 3, 41, dtype=torch.float64)
    for spec in (StepTanhL(2, 3, add_f0=True), SAL(2, init_random=True)):
        fl = instance_flow(spec)
        layers = []
        for sub in fl.flow_arr:
            kind = type(sub).__name__
            if kind == 'AffineFlow':
                layers.append(('affine', sub.a, sub.b, sub.set_restrictions))
            elif kind == 'StepFlow':
                layers.append(('tanh_step', [(s.a, s.b, s.c, s.d) for s in sub.flow_arr], sub.add_init_f0))
            else:
                layers.append(('sal', sub.a, sub.b, sub.set_restrictions, sub.add_init_f0))
        assert torch.allclose(fl(f), O.apply_flow(layers, f), rtol=1e-14, atol=1e-14)


def test_step_group_packing_and_module_forward():
    """General step flows (flows.py:284-491): the descriptor of a StepFlow over arbitrary members — group header, one layer per
    member, switch_off pairs appended to the members that have a trainable one — and the torch `forward` of the modules against
    the oracle's `step_group` layer."""
    import numpy as np
    from oracle import tgp_oracle as O
    from tgp.pytorch_b200.dsp import config as cg
    cg.set_maximum_precission()
    from tgp.pytorch_b200.dsp.flows import StepAllL, StepSAL
    from tgp.pytorch_b200.dsp.models.flow import instance_flow
    from tgp.pytorch_b200.engine import FlowLayout
    np.random.seed(3)
    fl = instance_flow(StepAllL(1, init_random=True))
    with torch.no_grad():
        for n, prm in fl.named_parameters():
            if n.endswith('.lam'):
                prm.fill_(1.2)
    layers, glob, rows = fl.describe()
    lay = FlowLayout(layers)
    assert [l['kind'] for l in lay.layers] == ['step_group', 'invboxcox', 'boxcox', 'arcsinh', 'sal', 'tanh_step', 'affine']
    assert lay.layers[0]['n_steps'] == 5 and lay.layers[0]['npar'] == 0
    assert [l['switch'] for l in lay.layers] == [False, True, True, False, True, False, False]      # boxcox, inverse boxcox, sinh-arcsinh
    assert [l['npar'] for l in lay.layers] == [0, 3, 3, 4, 4, 4, 2] and lay.n_theta == len(glob) == 20 and not rows
    step = fl.flow_arr[0]
    members = []
    for sw, sub in zip(step.switch_off, step.flow_arr):
        kind = type(sub).__name__
        if kind == 'TanhFlow':
            m = ('tanh_step', [(sub.a, sub.b, sub.c, sub.d)], False)
        elif kind == 'ArcsinhFlow':
            m = ('arcsinh', sub.a, sub.b, sub.c, sub.d, sub.set_restrictions, sub.add_init_f0)
        elif kind == 'Sinh_ArcsinhFlow':
            m = ('sal', sub.a, sub.b, sub.set_restrictions, sub.add_init_f0)
        else:
            m = ('invboxcox' if kind == 'InverseBoxCoxFlow' else 'boxcox', sub.transform_param().reshape(()), sub.add_init_f0)
        members.append((m, (sw.a, sw.b) if sw.is_trainable else None))
    aff = fl.flow_arr[1]
    ol = [('step_group', members, step.add_init_f0), ('affine', aff.a, aff.b, aff.set_restrictions)]
    f = torch.linspace(0.2, 3, 29, dtype=torch.float64)           # positive: the inverse Box-Cox member with lam > 1
    assert torch.allclose(fl(f), O.apply_flow(ol, f), rtol=1e-13, atol=1e-13)
    # a switch_off on an input-dependent member is refused, not silently mis-packed
    with pytest.raises(NotImplementedError):
        FlowLayout([dict(kind='step_group', n_steps=1), dict(kind='sal', per_row=True, switch=True)])
    fl2 = instance_flow(StepSAL(2, 3, add_f0=True))
    lay2 = FlowLayout(fl2.describe()[0])
    assert [l['kind'] for l in lay2.layers] == ['step_group', 'sal', 'sal', 'sal', 'affine'] * 2 and lay2.n_theta == 2 * (3 * 4 + 2)


def test_cabi_validates_step_groups_without_a_gpu():
    from tgp.pytorch_b200 import _lib
    lib = _lib.load()
    m = _lib.TgpModel()
    m.dtype, m.M, m.D, m.likelihood, m.n_quad = _lib.TGP_F64, 16, 2, _lib.LIK_GAUSS_NONLINEAR, 20

    def layers(*spec):
        m.n_layers = len(spec)
        for i, (kind, flags, n) in enumerate(spec):
            m.layers[i].kind, m.layers[i].flags, m.layers[i].n_steps, m.layers[i].p0 = kind, flags, n, 0
        return lib.tgp_step_workspace_bytes(m)
    assert layers((_lib.FLOW_STEP_GROUP, 0, 2), (_lib.FLOW_SAL, _lib.FLOW_SWITCH, 0), (_lib.FLOW_ARCSINH, 0, 0), (_lib.FLOW_AFFINE, 0, 0)) > 0
    assert layers((_lib.FLOW_STEP_GROUP, 0, 3), (_lib.FLOW_SAL, 0, 0), (_lib.FLOW_AFFINE, 0, 0)) == 0          # runs past the end
    assert b'step group' in lib.tgp_last_error()
    assert layers((_lib.FLOW_STEP_GROUP, 0, 1), (_lib.FLOW_AFFINE, 0, 0)) == 0                                 # affine member
    assert layers((_lib.FLOW_SAL, _lib.FLOW_SWITCH, 0),) == 0                                                  # switch outside a group
    assert layers((_lib.FLOW_STEP_GROUP, 0, 1), (_lib.FLOW_SAL, _lib.FLOW_SWITCH | _lib.FLOW_PER_ROW, 0)) == 0
    assert layers((_lib.FLOW_STEP_GROUP, 0, 1), (_lib.FLOW_STEP_GROUP, 0, 1), (_lib.FLOW_SAL, 0, 0)) == 0      # nesting


def test_no_cpu_fallback():
    g = Golden('boston_svgp_p1')
    model = build_from_golden(g, 'cpu')
    with pytest.raises(RuntimeError, match='no CPU path'):
        model.ELBO(g.t('X'), g.t('Y'))


def test_minibatch_stager_has_no_cpu_path():
    """The pinned-host stager copies into CUDA memory; asking it for a CPU device must fail loudly, not degrade."""
    import pytest
    from tgp.pytorch_b200.data import PinnedMinibatchStager
    X, Y = torch.zeros(8, 2, dtype=torch.float64), torch.zeros(8, 1, dtype=torch.float64)
    with pytest.raises(RuntimeError):
        PinnedMinibatchStager(X, Y, 4, 'cpu')


def test_library_options_retired_key_and_workspace_sizing_without_a_gpu():
    """Option ids in the ctypes binding equal the header's enum and the retired key 1 is rejected as unknown; the row-chunk
    option is validated and changes the batch workspace size it documents (pure host code: no kernel is launched)."""
    from tgp.pytorch_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, 'include', 'tgp_b200.h')).read()
    enum = dict(re.findall(r'(TGP_OPT_[A-Z_]+)\s*=\s*(\d+)', header))
    assert '1' not in enum.values()                      # key 1 (the retired single-kernel tensor-core forward) is unknown
    assert int(enum['TGP_OPT_ROW_CHUNK']) == _lib.OPT_ROW_CHUNK
    m = _lib.TgpModel()
    m.dtype, m.M, m.D, m.likelihood, m.n_quad = _lib.TGP_F64, 256, 4, 1, 30
    R = 100000
    try:
        assert lib.tgp_set_option(_lib.OPT_ROW_CHUNK, 8192) == 0
        small = lib.tgp_batch_workspace_bytes(m, R)
        assert lib.tgp_set_option(_lib.OPT_ROW_CHUNK, 65536) == 0
        large = lib.tgp_batch_workspace_bytes(m, R)
        # [A|B] (2M) and K_xz (M) are per row; the two staging buffers (M each) are per chunk
        assert small >= 8 * (3 * 256 * R + 2 * 256 * 8192) and large - small == 8 * 2 * 256 * (65536 - 8192)
        assert lib.tgp_set_option(_lib.OPT_ROW_CHUNK, 64) != 0 and b'row chunk' in lib.tgp_last_error()
        assert lib.tgp_set_option(1, 1) != 0 and b'unknown option' in lib.tgp_last_error()
        assert lib.tgp_set_option(99, 1) != 0
    finally:
        assert lib.tgp_set_option(_lib.OPT_ROW_CHUNK, 32768) == 0


def test_workspace_sizes_follow_the_compute_mode_without_a_gpu():
    """The step workspace holds the FP64 region plus the planes of the active mode only, so the FP64 mode's is the smallest
    and each tensor-core mode adds an amount that depends on M alone; batch sizes grow with R across the row-chunk edges
    (16384 rows for the tensor-core modes, 32768 for FP64); the single-call workspace holds all the regions."""
    from tgp.pytorch_b200 import _lib
    lib = _lib.load()
    modes = (_lib.TGP_F64, _lib.TGP_F32, _lib.TGP_F64_I8)
    m = _lib.TgpModel()
    m.likelihood, m.n_quad = 1, 30
    for M in (1, 100, 1024, 2048):
        extra = set()
        for D in (1, 8, 33):
            m.M, m.D = M, D
            step = {}
            for dt in modes:
                m.dtype = dt
                step[dt] = lib.tgp_step_workspace_bytes(m)
                batch = [lib.tgp_batch_workspace_bytes(m, R) for R in (1, 16383, 16384, 16385, 32768, 32769, 100000)]
                assert batch[0] > 0 and batch == sorted(batch), (M, D, dt, batch)
                lay = _lib.TgpReduceLayout()
                assert lib.tgp_reduce_layout(m, lay) == 0
                for R in (1, 4096):
                    need = step[dt] + lib.tgp_batch_workspace_bytes(m, R) + 8 * (lay.total + lay.packed_total)
                    assert lib.tgp_workspace_bytes(m, R) >= need, (M, D, dt, R)
            assert 0 < step[_lib.TGP_F64] < step[_lib.TGP_F32] and step[_lib.TGP_F64] < step[_lib.TGP_F64_I8], (M, D, step)
            extra.add((step[_lib.TGP_F32] - step[_lib.TGP_F64], step[_lib.TGP_F64_I8] - step[_lib.TGP_F64]))
        assert len(extra) == 1, (M, extra)


def test_split_csv_reader_standardises_like_the_reference(tmp_path):
    """data.load_split_csv: the airline-style on-disk format (header-less CSV + splits_idx pickle,
    regression_datasets.py:95-192) with the training-statistics standardisation of data.py:260-299."""
    import pickle
    import numpy as np
    from tgp.pytorch_b200.data import load_split_csv
    rng = np.random.default_rng(0)
    data = rng.normal(size=(200, 6)) * np.array([1, 10, 0.1, 5, 2, 3]) + np.array([0, 5, -1, 2, 0, 7])
    csv = tmp_path / 'airline.csv'
    np.savetxt(csv, data, delimiter=',')
    perm = rng.permutation(200)
    with open(tmp_path / 'splits_idx_airline.pkl', 'wb') as fh:
        pickle.dump({'seed_3': {'train': perm[:150], 'test': perm[150:]}}, fh)
    X_tr, Y_tr, X_te, Y_te, Y_std = load_split_csv(str(csv), str(tmp_path / 'splits_idx_airline.pkl'), 3)
    raw = np.loadtxt(csv, delimiter=',')
    tr, te = raw[perm[:150]], raw[perm[150:]]
    xm, xs = tr[:, :-1].mean(0), tr[:, :-1].std(0) + 1e-15
    ym, ys = tr[:, -1].mean(), tr[:, -1].std() + 1e-15
    assert np.allclose(X_tr.numpy(), (tr[:, :-1] - xm) / xs, rtol=0, atol=1e-14)
    assert np.allclose(X_te.numpy(), (te[:, :-1] - xm) / xs, rtol=0, atol=1e-14)
    assert np.allclose(Y_te.numpy()[:, 0], (te[:, -1] - ym) / ys, rtol=0, atol=1e-14)
    assert abs(float(Y_std) - ys) < 1e-15 and Y_tr.shape == (150, 1)
    with pytest.raises(ValueError, match='md5'):
        load_split_csv(str(csv), str(tmp_path / 'splits_idx_airline.pkl'), 3, md5sum='0' * 32)
