"""nestfit_b200 -- B200-native likelihood hot path of NestFit.

Same public names as ``nestfit`` for the path it replaces (reference
nestfit/__init__.py:8-62); everything numerical runs in hand-written sm_100a
CUDA kernels behind the C ABI of ``include/nestfit_b200.h``.
"""
from .core import (  # noqa: F401
    Distribution, Prior, ConstantPrior, DuplicatePrior, OrderedPrior, SpacedPrior, CenSepPrior,
    ResolvedCenSepPrior, ResolvedPlacementPrior, PriorTransformer, Spectrum, Runner,
)
from .pixels import PixelBlock  # noqa: F401
from .models.ammonia import amm_predict, AmmoniaSpectrum, AmmoniaRunner  # noqa: F401
from .models.gaussian import gauss_predict, GaussianRunner  # noqa: F401
from .models.diazenylium import nnhp_predict, DiazenyliumSpectrum, DiazenyliumRunner  # noqa: F401
from .prior_constructors import get_irdc_priors, get_synth_priors  # noqa: F401
from .sampler import NestedSamplingBatch, Dumper, run_multinest, run_multinest_batch  # noqa: F401
from .store import HdfStore, MemGroup  # noqa: F401
from .main import (  # noqa: F401
    NoiseMap, NoiseMapUniform, DataCube, CubeStack, CubeFitter, get_multiproc_indices, get_block_indices,
)
from . import postprocess  # noqa: F401
from .postprocess import (  # noqa: F401
    take_by_components, apply_circular_mask, get_indep_info_kernel, aggregate_run_attributes, convolve_evidence,
    extended_masked_evidence, aggregate_run_products, aggregate_intensity_marginals, aggregate_run_pdfs,
    convolve_post_pdfs,
    quantize_conv_marginals, deblend_hf_intensity, generate_predicted_profiles, postprocess_run,
)
