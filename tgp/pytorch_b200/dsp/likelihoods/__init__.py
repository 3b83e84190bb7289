"""Observation models of the hot path.  Each class keeps the reference's constructor and method signatures
(`expected_log_prob`, `marginal_moments`, `sample_from_output`) and launches the fused row epilogue
(`_rows.py` -> tgp_ell_forward / tgp_test_rows) instead of materialising the S x MB quadrature grid.

`MulticlassCategorical` integrates by Monte Carlo in its own kernel (tgp_mc_softmax_rows).  `WarpedGaussianLinearMean` (the warped
GP: a flow on the observations) runs in the same row kernels with its own closed-form rows (TGP_LIK_GAUSS_WARPED)."""
from .Bernoulli import Bernoulli
from .GaussianLinearMean import GaussianLinearMean
from .GaussianNonLinearMean import GaussianNonLinearMean
from .MulticlassCategorical import MulticlassCategorical
from .WarpedGaussianLinearMean import WarpedGaussianLinearMean

__all__ = ['Bernoulli', 'GaussianLinearMean', 'GaussianNonLinearMean', 'MulticlassCategorical', 'WarpedGaussianLinearMean']
