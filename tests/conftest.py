import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run with -m gpu on the B200 box)')
    config.addinivalue_line('markers', 'needs_reference: needs a checkout of the original TGP.pytorch named by TGP_REFERENCE_ROOT')


def pytest_collection_modifyitems(config, items):
    import torch
    from oracle.ref_loader import reference_available
    has_gpu = torch.cuda.is_available()
    has_ref = reference_available()
    for item in items:
        if 'gpu' in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason='no CUDA device'))
        if 'needs_reference' in item.keywords and not has_ref:
            item.add_marker(pytest.mark.skip(reason='TGP_REFERENCE_ROOT does not name a TGP.pytorch checkout'))


# ---- measured residuals -----------------------------------------------------------------------------------------
# Parity tests call record_residuals(test, {quantity: L2-relative error}); the session writes the worst value per
# (test, quantity) to gpurun_out/parity_residuals.json so that the tolerances in the tests can be read against what
# was actually measured (copied to profiles/ per round).
_RESIDUALS = {}


def record_residuals(test, errs):
    slot = _RESIDUALS.setdefault(test, {})
    for k, e in errs.items():
        e = float(e)
        if not (slot.get(k, -1.0) >= e):
            slot[k] = e


def pytest_sessionfinish(session, exitstatus):
    if not _RESIDUALS:
        return
    import json
    out = os.path.join(ROOT, 'gpurun_out')
    try:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, 'parity_residuals.json'), 'w') as fh:
            json.dump(_RESIDUALS, fh, indent=1, sort_keys=True)
    except OSError:
        pass
