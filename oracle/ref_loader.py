"""Import the UNMODIFIED reference (`$TGP_REFERENCE_ROOT/code/dsp`) under `oracle/ref_shims` ("O1").

TEST INFRASTRUCTURE ONLY.  Works only where TGP_REFERENCE_ROOT names a checkout of the original TGP.pytorch project,
which this repository does not contain; it is used by `oracle/make_golden.py` to generate `tests/golden/*.npz` and by
the `needs_reference` CPU tests.  Never imported by the product, the GPU tests, `smoke()` or `bench.py`.

What is patched, and nothing else (SURVEY.md §8c):
  * `sys.path`: shims first, then the reference's `code/` directory;
  * `scipy.integrate.cumtrapz` alias (removed from scipy; imported at reference `dsp/utils.py:26`);
  * `torch.__version__` reads '1.5.0' only while `dsp.config` runs its version gate (`dsp/config.py:18-25,74`).
"""
import os
import sys
import warnings

REFERENCE_ROOT = os.environ.get('TGP_REFERENCE_ROOT')
_SHIMS = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'ref_shims')


def reference_available():
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, 'code', 'dsp'))


def load_reference():
    """Returns the reference's `dsp` package (module object), CPU device, FP64 + 100 quadrature points."""
    if not reference_available():
        raise RuntimeError('reference tree not found: set TGP_REFERENCE_ROOT to a checkout of the original TGP.pytorch '
                           '(got %r)' % REFERENCE_ROOT)
    warnings.filterwarnings('ignore')
    for p in (os.path.join(REFERENCE_ROOT, 'code'), _SHIMS):
        if p in sys.path:
            sys.path.remove(p)
        sys.path.insert(0, p)
    import scipy.integrate
    if not hasattr(scipy.integrate, 'cumtrapz'):
        scipy.integrate.cumtrapz = scipy.integrate.cumulative_trapezoid
    import torch
    if 'dsp' not in sys.modules:
        real = torch.__version__
        torch.__version__ = '1.5.0'
        try:
            import dsp.config  # noqa: F401
        finally:
            torch.__version__ = real
    import dsp
    import dsp.config as cg
    import dsp.models  # noqa: F401
    import dsp.likelihoods  # noqa: F401
    import dsp.flows  # noqa: F401
    cg.device = 'cpu'
    cg.set_maximum_precission()   # what the reference's main.py always does (main.py:124)
    return dsp
