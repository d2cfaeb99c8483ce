"""b4d — B200-native BM4D denoise path for ExaSPIM uint16 volumes.

Drop-in for the one call the reference makes into the closed ``bm4d`` wheel
(data_handling.py:332, :926; evaluate.py:202) plus the offset / quantize /
statistics steps around it.  See DESIGN.md and INTEGRATION.md at the repo root.
"""
from .api import (  # noqa: F401
    BM4DProfile,
    BM4DStages,
    Denoiser,
    bm4d,
    bm4d_batch,
    get_denoiser,
    make_foreground_mask,
    noise_scaled_step,
    precompute_targets,
    quantize,
    noise_model_from_psd,
    patch_has_incoherent_segment,
    denoise_quantized,
    tile_stats,
    noise_sigma,
    noise_sigma_from_hist,
)
from .cache import load_patch_cache, write_patch_cache  # noqa: F401
from .codec import chunk_grid, chunk_shuffle, compute_cratio, entropy_bytes, estimate_cratio  # noqa: F401
from .sharding import (  # noqa: F401
    bind_to_gpu_numa,
    denoise_slab_exchange,
    denoise_volume_sharded,
    exchange_halo,
    exchange_planes,
    merge_histograms,
    slab_plan,
    stats_from_hist,
)

__all__ = [
    "BM4DProfile",
    "BM4DStages",
    "Denoiser",
    "bm4d",
    "bm4d_batch",
    "get_denoiser",
    "make_foreground_mask",
    "noise_scaled_step",
    "precompute_targets",
    "quantize",
    "noise_model_from_psd",
    "patch_has_incoherent_segment",
    "denoise_quantized",
    "tile_stats",
    "noise_sigma",
    "noise_sigma_from_hist",
    "slab_plan",
    "bind_to_gpu_numa",
    "denoise_volume_sharded",
    "merge_histograms",
    "denoise_slab_exchange",
    "exchange_halo",
    "exchange_planes",
    "stats_from_hist",
    "write_patch_cache",
    "chunk_grid",
    "chunk_shuffle",
    "compute_cratio",
    "entropy_bytes",
    "estimate_cratio",
    "load_patch_cache",
]
