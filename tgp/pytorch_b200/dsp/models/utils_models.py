"""Kernel / mean factories and the MC-dropout switch (reference code/dsp/models/utils_models.py:145-193, 285-294,
358-364).  Kernels: 'scale_rbf' and 'rbf' (what the reference's main.py builds), and 'scale_matern' / 'matern' with
init_params['nu'] in {0.5, 1.5, 2.5} (default 2.5, gpytorch's default)."""
import torch

from .. import config as cg
from ..kernels import MaternKernel, RBFKernel, ScaleKernel, ZeroMean
from ..utils import inv_softplus


def instance_kernel(name, ard_num_dim, num_multioutput, kernel_is_shared, init_params={}, kernels=None):
    if ard_num_dim is not None and not isinstance(ard_num_dim, int):
        raise ValueError('ard_num_dim must be None or int, got {}'.format(type(ard_num_dim)))
    ls = init_params.get('length_scale', 1.0)
    ks = init_params.get('kernel_scale', 1.0)
    if kernel_is_shared:
        num_multioutput = 1
    batch = torch.Size([num_multioutput])
    if name in ('rbf', 'scale_rbf', 'matern', 'scale_matern'):
        if name in ('rbf', 'scale_rbf'):
            base = RBFKernel(ard_num_dims=ard_num_dim, batch_shape=batch)
        else:
            base = MaternKernel(nu=init_params.get('nu', 2.5), ard_num_dims=ard_num_dim, batch_shape=batch)
        base.raw_lengthscale.data = inv_softplus(torch.ones(num_multioutput, 1, base.raw_lengthscale.size(-1), dtype=cg.dtype) * ls)
        if not name.startswith('scale_'):
            return base
        K = ScaleKernel(base, batch_shape=batch)
        K.raw_outputscale.data = inv_softplus(torch.ones(num_multioutput, dtype=cg.dtype) * ks)
        return K
    raise NotImplementedError("kernel %r is outside the fused hot-path scope ('rbf', 'scale_rbf', 'matern', "
                              "'scale_matern')" % (name,))


def return_mean(name, input_dim, output_dim, W):
    if name == 'zero':
        return ZeroMean()
    raise NotImplementedError("mean %r is outside the hot-path scope (main.py uses 'zero')" % (name,))


def enable_eval_dropout(modules):
    found = False
    for module in modules:
        if 'Dropout' in type(module).__name__:
            module.train()
            found = True
    return found
