"""pd_unet_b200 -- the PD-UNet measurement operators (CT Radon / FBP, radial-MRI NUFFT, fused
primal-dual updates) as hand-written sm_100a CUDA behind the torch_radon / torchkbnufft call shapes.
See DESIGN.md.  Importing the package does not load the CUDA library; the first operator call does,
and raises if it is missing (there is no CPU fallback)."""
from ._lib import PduError, launch_count, set_option  # noqa: F401
from .radon import Radon, RadonFanbeam  # noqa: F401
from .nufft import (KbInterp, KbInterpAdjoint, KbNufft, KbNufftAdjoint, ToepNufft,  # noqa: F401
                    calc_density_compensation_function, calc_toeplitz_kernel, toep_cg)
from . import updates, parallel  # noqa: F401

__version__ = "0.1.0"
