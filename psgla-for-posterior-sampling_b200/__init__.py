"""psgla_b200 -- B200-native (sm_100a) PSGLA / PnP-ULA proximal Langevin sampling.

Drop-in for the hot path of Marien-RENAUD/PSGLA-for-posterior-sampling: same entry points
(``psgla``, ``pnpula`` / ``pnp_ula``, ``PnP_ULA``, ``SnoPnP_ULA``, ``Theorical_MMSE``), hand-written CUDA behind a
C ABI (include/psgla_b200.h), no CPU fallback.  Import as ``psgla_b200`` (see psgla_b200.py at the repo root; the
directory name carries the reference's name and is not a Python identifier).
"""
from . import _lib  # noqa: F401
from . import dist  # noqa: F401
from . import metrics  # noqa: F401
from . import image_set  # noqa: F401
from .image_set import load_image, run_image_set  # noqa: F401
from .diagnostics import mcmc_diagnostics, mcmc_diagnostics_large, mcmc_summary  # noqa: F401
from .metrics import posterior_summary, psnr_ssim  # noqa: F401
from .denoisers import (DRUNET_KEYS, GSDRUNET_KEYS, DRUNet, DnCNN, GSDRUNet, TVDenoiser, lipschitz_dncnn_state_dict,  # noqa: F401
                        random_dncnn_state_dict, random_drunet_state_dict, random_gsdrunet_state_dict,  # noqa: F401
                        smoothing_dncnn_state_dict)  # noqa: F401
from .operators import (DeblurDataGrad, InpaintingDataGrad, PriorGrad, blur_taps, make_deblurring,  # noqa: F401
                        make_inpainting)
from .params import as_pnpula_kwargs, as_psgla_kwargs, sampler_params  # noqa: F401
from .restoration_algorithms import pnp, pnp_ula, pnpula, pnpula_run, psgla, psgla_run, red  # noqa: F401
from .sampling_2D import GMMChains, PnP_ULA, SnoPnP_ULA, run_chains  # noqa: F401
from .utils_2D import (GMMDenoiser, Theorical_MMSE, Wasserstein_distance, constantes_conditionnal_prob,  # noqa: F401
                       gaussian_mixt_example, sample_gaussian, sample_posterior, sliced_wasserstein_distance)

__version__ = "0.1.0"
