"""Model layer of the host-side mirror.

Re-exports the names the reference's `code/main.py:26-37` imports from `dsp.models`:

* `instance_kernel`  — factory of the (Scale)RBF-ARD and (Scale)Matern-ARD kernel parameter holders,
* `sparse_MF_SP`     — sparse variational transformed GP (TGP / ID_TGP) whose ELBO, marginals and test log-likelihood run
                       in the sm_100a kernels of libtgp_b200.so,
* `sparse_MF_GP`     — SVGP, the same model with identity flows,
* `return_mean`, `enable_eval_dropout` — small helpers used by the model and by MC-dropout evaluation.
"""
from .sparse_MF_GP import sparse_MF_GP
from .sparse_MF_SP import sparse_MF_SP
from .utils_models import enable_eval_dropout, instance_kernel, return_mean

__all__ = ['enable_eval_dropout', 'instance_kernel', 'return_mean', 'sparse_MF_GP', 'sparse_MF_SP']
