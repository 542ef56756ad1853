"""Mirror of the sampling part of terrain_diffusion.inference / terrain_diffusion.training.evaluation."""
from .canvas import BlendCanvas  # noqa: F401
from .samplers import (process_base_cond_img, sample_base_diffusion,  # noqa: F401
                       sample_decoder_consistency_tiled, sample_decoder_diffusion_sharded,
                       sample_decoder_diffusion_tiled)
from .sharded import ShardedCanvas  # noqa: F401
from .solve import DiffusionSolve  # noqa: F401
from .tiling import linear_weight_window, padded_batch_size, shard_rows, tile_starts, window_range  # noqa: F401
from .stages import coarse_stage_tile, decoder_stage_tile, latent_stage_tiles, process_latent_conditioning  # noqa: F401
from .lazy_canvas import LazyCanvas, TensorWindow  # noqa: F401
from .pipeline import TerrainPipeline, WorldPipeline  # noqa: F401
from .multiphase import (build_timestep_ranges, infinite_diffusion_canvases, phase_step_ranges,  # noqa: F401
                         sample_infinite_diffusion)
