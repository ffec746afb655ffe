"""bmm-mcmc_b200: B200-native allocation-sampling path of the bmm-mcmc R package.

`gibbs_full`, `gibbs_collapsed`, `gibbs_dp`, `gibbs_stickbreaking` mirror R/utils.R:23-107; the
sampling itself runs in hand-written sm_100a CUDA behind the C ABI of include/bmm_capi.h.
"""
from .api import gibbs_full, gibbs_collapsed, gibbs_dp, gibbs_stickbreaking, predictive, waic, loo, loglik_matrix, Plan, PackedX  # noqa: F401
from .rcompat import RRng, load_dataset, DATASET_NAMES  # noqa: F401
from .plot import plot_gibbs, plot_alpha  # noqa: F401
