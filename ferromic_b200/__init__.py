"""ferromic_b200 -- B200 (sm_100a) implementation of ferromic's per-site population-genetics
estimators (segregating sites, pi, Watterson theta, per-site pi/theta tracks, Hudson FST/Dxy,
Weir & Cockerham FST, pairwise sample differences) behind the reference's own Python surface (`import ferromic_b200 as fm`).

All estimator arithmetic runs in hand-written CUDA kernels through the C-ABI library
`libferromic_gpu.so` (include/ferromic_gpu.h); there is no CPU fallback."""
from ._lib import FerromicGpuError, SO_PATH, lib  # noqa: F401
from .api import (  # noqa: F401
    DiversitySite,
    FstEstimate,
    HudsonDxyResult,
    HudsonFstResult,
    HudsonFstSite,
    Population,
    WcFstResult,
    WcFstSite,
    adjusted_sequence_length,
    hudson_dxy,
    hudson_fst,
    hudson_fst_sites,
    hudson_fst_with_sites,
    inversion_allele_frequency,
    pairwise_difference_arrays,
    pairwise_differences,
    nucleotide_diversity,
    per_site_diversity,
    per_site_diversity_arrays,
    segregating_sites,
    watterson_theta,
    wc_fst,
    wc_fst_components,
    wc_fst_from_membership,
)

__version__ = "0.1.0"
