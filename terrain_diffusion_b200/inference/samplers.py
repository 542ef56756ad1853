"""Bounded-canvas tiled samplers -- drop-ins for terrain_diffusion.training.evaluation.sample_diffusion_decoder
(reference sample_diffusion_decoder.py:44-211) and sample_diffusion_base.sample_base_diffusion (sample_diffusion_base.py
:51-168), running tile solves as fused CUDA graphs and the overlap blend on a device-resident canvas.

Tile order, tile origins (`tile_starts`, last tile clamped) and the blend window are the reference's, integer for
integer.  Unlike the reference function as shipped, the multi-tile diffusion sampler resets the solver state per tile
(the reference raises IndexError on tile #2 because its stateful scheduler is never reset -- SURVEY.md section 0
item 7); the per-tile reset is the behaviour of the reference's own working samplers (sample_diffusion_base.py:147,
world_pipeline.py:934).  Independent tiles may be solved `tile_batch` at a time; the blend is still applied in
row-major order so the canvas is bit-identical to a sequential run.

Both diffusion samplers take the reference's two-model guidance (a guide U-Net evaluated on the same input every step,
mo = mo_g + s*(mo_m - mo_g), recorded into the same graph) and the decoder sampler its score_scaling (folded into the
update coefficients); see inference/solve.py.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn.functional as F

from .canvas import BlendCanvas
from .solve import DiffusionSolve, check_guide
from .tiling import linear_weight_window, tile_starts


MAX_CACHED_SOLVES = 12      # every cached solve owns an activation arena and a CUDA graph


class _LruDict(dict):
    """dict that keeps at most MAX_CACHED_SOLVES entries, dropping the least recently inserted / fetched."""

    def __getitem__(self, k):
        v = super().pop(k)
        super().__setitem__(k, v)
        return v

    def __setitem__(self, k, v):
        super().__setitem__(k, v)
        while len(self) > MAX_CACHED_SOLVES:
            super().pop(next(iter(self)))


def _solve_cache(model):
    if not hasattr(model, "_solve_cache"):
        model._solve_cache = _LruDict()
    return model._solve_cache


def get_diffusion_solve(model, scheduler, n, h, w, num_steps, step_range=None, guide=None, guidance_scale: float = 1.0,
                        score_scaling: float = 1.0) -> DiffusionSolve:
    """Cached fused N-step solve (or one phase of it: step_range).  The key is everything the solve bakes in: the
    sigma table and the per-step order schedule (they cover sigma_min/max/rho/schedule, scaling_p/scaling_t,
    lower_order_final, euler_at_final, ...) plus the options that change the update formula.  The caller's scheduler
    is put in the state the reference leaves it in (`set_timesteps(num_steps)`) on a cache hit too.
    Guided (a guide and guidance_scale != 1): the guide's folded weights join the key, the scale does not -- it lives
    in the solve's device table and is rewritten on a hit, so a sweep over guidance_scale reuses one program.
    score_scaling != 1 changes the coefficient rows and joins the key."""
    guided = guide is not None and float(guidance_scale) != 1.0
    if guided:
        check_guide(model, guide)
    scheduler.set_timesteps(num_steps)
    c = scheduler.config
    key = (n, h, w, num_steps, None if step_range is None else tuple(int(v) for v in step_range),
           tuple(float(v) for v in scheduler.sigmas), tuple(scheduler.order_schedule()),
           float(c.sigma_data), c.prediction_type, c.final_sigmas_type, c.solver_order, c.algorithm_type, c.solver_type,
           id(model.folded()))
    if guided:
        key += (("guide", id(guide.folded())),)
    if float(score_scaling) != 1.0:
        key += (("score_scaling", float(score_scaling)),)
    cache = _solve_cache(model)
    if key not in cache:
        cache[key] = DiffusionSolve(model, scheduler, n, h, w, num_steps, step_range=step_range,
                                    guide=guide if guided else None, guidance_scale=guidance_scale,
                                    score_scaling=score_scaling)
    solve = cache[key]
    if guided:
        solve.set_guidance_scale(guidance_scale)
    return solve


def get_consistency_solve(model, n, h, w, t: float, sigma_data: float = 0.5, from_unit_noise: bool = False,
                          out_scale: float = 1.0) -> DiffusionSolve:
    """Cached one-step TrigFlow consistency program (solve.consistency_rows) for `n` tiles of h x w."""
    from .solve import consistency_rows
    key = ("cm", n, h, w, float(t), float(sigma_data), bool(from_unit_noise), float(out_scale), id(model.folded()))
    cache = _solve_cache(model)
    if key not in cache:
        cache[key] = DiffusionSolve(model, None, n, h, w, 1,
                                    coef_rows=consistency_rows(t, sigma_data, from_unit_noise, out_scale))
    return cache[key]


@torch.no_grad()
def sample_decoder_diffusion_tiled(model, scheduler, cond_img: torch.Tensor, noise: torch.Tensor,
                                   tile_size: Optional[int] = None, tile_stride: Optional[int] = None, *,
                                   num_steps: Optional[int] = None, guidance_model=None, guidance_scale: float = 1.0,
                                   score_scaling: float = 1.0, weight_window_fn=None, tile_batch: int = 1):
    """Tiled DPM-Solver++ sampling of a decoder canvas (sample_diffusion_decoder.py:44-125); noise is the initial
    sample already scaled by sigma_0.  guidance_model / guidance_scale: two-model guidance in every step;
    score_scaling: the reference's _scale_score alpha (1 disables)."""
    if guidance_model is not None and float(guidance_scale) != 1.0:
        check_guide(model, guidance_model)
    if num_steps is None:
        num_steps = scheduler.num_inference_steps
        if num_steps is None:
            raise ValueError("num_steps is None and scheduler.set_timesteps was never called")
    b, c, h, w = noise.shape
    device, dtype = noise.device, noise.dtype
    cond_img = cond_img.to(device=device, dtype=dtype)
    if cond_img.shape[-2:] != (h, w):
        cond_img = F.interpolate(cond_img, size=(h, w), mode="nearest")
    tile_size = tile_size or min(h, w)
    tile_stride = tile_stride or tile_size
    window = (weight_window_fn(tile_size, device, torch.float32)[0, 0] if weight_window_fn is not None
              else linear_weight_window(tile_size, device)).contiguous()
    tiles = [(i0, j0) for i0 in tile_starts(h, tile_size, tile_stride) for j0 in tile_starts(w, tile_size, tile_stride)]
    canvases = [BlendCanvas(c, h, w, device) for _ in range(b)]
    noise32, cond32 = noise.float(), cond_img.float()
    group = max(1, int(tile_batch))
    for g0 in range(0, len(tiles), group):
        chunk = tiles[g0:g0 + group]
        n = b * len(chunk)
        solve = get_diffusion_solve(model, scheduler, n, tile_size, tile_size, num_steps, guide=guidance_model,
                                    guidance_scale=guidance_scale, score_scaling=score_scaling)
        x = torch.cat([noise32[..., i0:i0 + tile_size, j0:j0 + tile_size] for (i0, j0) in chunk], dim=0)
        cd = torch.cat([cond32[..., i0:i0 + tile_size, j0:j0 + tile_size] for (i0, j0) in chunk], dim=0)
        out = solve.run(x, cd)
        for t, (i0, j0) in enumerate(chunk):
            for bi in range(b):
                canvases[bi].accumulate(out[t * b + bi], i0, j0, window)
    return torch.stack([cv.normalized() for cv in canvases]).to(dtype)


@torch.no_grad()
def process_base_cond_img(cond_img: torch.Tensor, histogram_raw, cond_means, cond_stds, noise_level) -> torch.Tensor:
    """The base model's 58-dim condition of a batch of 4 x 4 condition windows, with the semantics of the reference's
    _process_cond_img (sample_diffusion_base.py:11-48): standardise; NaNs of batch ROW 0 become cond_means[0] and
    those of row 1 cond_means[1] (the reference indexes the batch there, not the channel); centre-2 x 2 climate means;
    a climate mean that is still NaN is replaced by torch.randn_like (global generator); mp_concat of the six parts
    [means 16 | p5 16 | climate 4 | mask 16 | histogram | noise-level term].  Small torch ops on cond_img's device."""
    from .stages import _concat_scales, _const_on          # (stages imports this module)
    dev = cond_img.device
    means_h = torch.as_tensor(cond_means).detach().cpu().float().flatten()
    x = (cond_img.float() - _const_on(dev, means_h).view(1, -1, 1, 1)) / \
        _const_on(dev, torch.as_tensor(cond_stds).detach().cpu()).view(1, -1, 1, 1)
    x[0:1] = x[0:1].nan_to_num(float(means_h[0]))
    x[1:2] = x[1:2].nan_to_num(float(means_h[1]))
    level = (torch.as_tensor(noise_level, dtype=torch.float32).to(dev) - 0.5) * math.sqrt(12)
    clim = x[:, 2:6, 1:3, 1:3].mean(dim=(2, 3))
    nan = torch.isnan(clim)
    clim[nan] = torch.randn_like(clim[nan])
    parts = [x[:, 0].flatten(1), x[:, 1].flatten(1), clim, x[:, 6].flatten(1),
             torch.as_tensor(histogram_raw).to(device=dev, dtype=torch.float32), level.reshape(-1, 1)]
    return torch.cat(parts, dim=1) * _concat_scales([p.shape[1] for p in parts], dev)


@torch.no_grad()
def sample_base_diffusion(model, scheduler, shape, cond_inputs, *, cond_means=None, cond_stds=None, noise_level=0.0,
                          histogram_raw=None, dtype: torch.dtype = torch.float32, steps: int = 15, guide_model=None,
                          guidance_scale: float = 1.0, generator: Optional[torch.Generator] = None,
                          tile_size: Optional[int] = None, weight_window_fn=None, noise: Optional[torch.Tensor] = None,
                          tile_batch: Optional[int] = None):
    """Base-model (latent) diffusion sampling, optionally tiled and guided (sample_diffusion_base.py:51-168).

    sigma_0 is the scheduler's sigmas[0] as it stands on entry (before set_timesteps), the initial sample
    torch.randn(shape, generator, model device, dtype) * sigma_0 -- the reference's call, so the same generator state
    on the same device gives the same noise.  `noise` (optional) replaces that draw with a given unit-variance tensor.
    Untiled (tile_size None): cond_inputs is the list of conditional inputs as given; returns the samples (not divided
    by sigma_data).  Tiled: stride tile_size // 2, cond_inputs a [B, 7, len(h_starts)+3, len(w_starts)+3] grid whose
    4 x 4 window [ic:ic+4, jc:jc+4] becomes the condition of tile (ic, jc) (process_base_cond_img); every tile is a
    fresh solve; returns blend / weights / sigma_data.  The tiles of the canvas are solved together, `tile_batch`
    tiles per solve (None: all of them), and blended in row-major order."""
    device = model.device
    sigma0 = scheduler.sigmas[0].to(device)
    if noise is None:
        noise = torch.randn(shape, generator=generator, device=device, dtype=dtype)
    x_init = noise.to(device=device, dtype=dtype) * sigma0
    kw = dict(guide=guide_model, guidance_scale=guidance_scale)
    if tile_size is None:
        b, c, h, w = shape
        solve = get_diffusion_solve(model, scheduler, b, h, w, steps, **kw)
        ci = list(cond_inputs) if cond_inputs is not None else []
        return solve.run(x_init.float(), None, conditional_inputs=ci).to(dtype, copy=True)
    b, c, h, w = shape
    stride = tile_size // 2
    hs, ws = tile_starts(h, tile_size, stride), tile_starts(w, tile_size, stride)
    if cond_inputs.ndim == 1 and len(hs) * len(ws) > 1:
        raise ValueError(f"cond_inputs must be a tensor image for tiled sampling. Cond inputs must have width "
                         f"{len(ws) + 3} and height {len(hs) + 3}.")
    if cond_inputs.ndim == 4 and tuple(cond_inputs.shape[-2:]) != (len(hs) + 3, len(ws) + 3):
        raise ValueError(f"cond_inputs grid is {tuple(cond_inputs.shape[-2:])}, tiling needs "
                         f"{(len(hs) + 3, len(ws) + 3)}")
    window = (weight_window_fn(tile_size, device, torch.float32)[0, 0] if weight_window_fn is not None
              else linear_weight_window(tile_size, device)).contiguous()
    tiles = [(ic, i0, jc, j0) for ic, i0 in enumerate(hs) for jc, j0 in enumerate(ws)]
    conds = []
    for ic, _i0, jc, _j0 in tiles:             # the reference's per-tile order (its NaN fill draws from the generator)
        if cond_inputs.ndim == 4:
            conds.append(process_base_cond_img(cond_inputs[..., ic:ic + 4, jc:jc + 4].clone(), histogram_raw,
                                               cond_means, cond_stds, noise_level).to(device))
        else:
            conds.append(cond_inputs.to(device).float().reshape(1, -1).expand(b, -1))
    canvases = [BlendCanvas(c, h, w, device) for _ in range(b)]
    x32 = x_init.float()
    group = len(tiles) if tile_batch is None else max(1, int(tile_batch))
    for g0 in range(0, len(tiles), group):
        chunk = tiles[g0:g0 + group]
        solve = get_diffusion_solve(model, scheduler, b * len(chunk), tile_size, tile_size, steps, **kw)
        x = torch.cat([x32[..., i0:i0 + tile_size, j0:j0 + tile_size] for (_ic, i0, _jc, j0) in chunk], dim=0)
        cv = torch.cat(conds[g0:g0 + len(chunk)], dim=0)
        out = solve.run(x, None, conditional_inputs=[cv])
        for t, (_ic, i0, _jc, j0) in enumerate(chunk):
            for bi in range(b):
                canvases[bi].accumulate(out[t * b + bi], i0, j0, window)
    sigma_data = float(scheduler.config.sigma_data)
    return torch.stack([cv.normalized(sigma_data) for cv in canvases]).to(dtype)


@torch.no_grad()
def sample_decoder_consistency_tiled(model, scheduler, cond_img: torch.Tensor, noise: torch.Tensor,
                                     tile_size: Optional[int] = None, tile_stride: Optional[int] = None, *,
                                     intermediate_t=None, weight_window_fn=None):
    """n-step TrigFlow consistency sampling per tile (sample_diffusion_decoder.py:129-211): x_t = cos t*s + sin t*z,
    pred = -model(x_t/sigma_d, t), s' = cos t*x_t - sin t*sigma_d*pred; blend; / sigma_d."""
    b, c, h, w = noise.shape
    device, dtype = noise.device, noise.dtype
    cond_img = cond_img.to(device=device, dtype=dtype)
    if cond_img.shape[-2:] != (h, w):
        cond_img = F.interpolate(cond_img, size=(h, w), mode="nearest")
    tile_size = tile_size or min(h, w)
    tile_stride = tile_stride or tile_size
    window = (weight_window_fn(tile_size, device, torch.float32)[0, 0] if weight_window_fn is not None
              else linear_weight_window(tile_size, device)).contiguous()
    sigma_data = float(scheduler.config.sigma_data)
    ts = [math.atan(float(scheduler.sigmas[0]) / sigma_data)]
    if intermediate_t is not None:
        if torch.is_tensor(intermediate_t):
            ts += [float(v) for v in intermediate_t.flatten()]
        elif isinstance(intermediate_t, (list, tuple)):
            ts += [float(v) for v in intermediate_t]
        else:
            ts.append(float(intermediate_t))
    canvases = [BlendCanvas(c, h, w, device) for _ in range(b)]
    for i0 in tile_starts(h, tile_size, tile_stride):
        for j0 in tile_starts(w, tile_size, tile_stride):
            samples = torch.zeros((b, c, tile_size, tile_size), device=device, dtype=torch.float32)
            tile_cond = cond_img[..., i0:i0 + tile_size, j0:j0 + tile_size].float()
            z = noise[..., i0:i0 + tile_size, j0:j0 + tile_size].float() * sigma_data
            for t in ts:
                x_t = math.cos(t) * samples + math.sin(t) * z
                tt = torch.full((b,), t, device=device, dtype=torch.float32)
                pred = -model(torch.cat([x_t / sigma_data, tile_cond], dim=1), tt, [])
                samples = math.cos(t) * x_t - math.sin(t) * sigma_data * pred
            for bi in range(b):
                canvases[bi].accumulate(samples[bi].contiguous(), i0, j0, window)
    return torch.stack([cv.normalized(sigma_data) for cv in canvases]).to(dtype)


@torch.no_grad()
def sample_decoder_diffusion_sharded(model, scheduler, cond_img: torch.Tensor, noise: torch.Tensor, tile_size: int,
                                     tile_stride: int, *, num_steps: int, tile_batch: int = 1, group=None):
    """Multi-GPU form of sample_decoder_diffusion_tiled for ONE canvas (batch 1): every rank holds the full noise /
    conditioning canvas (they are inputs), solves only its stripe of tile rows, and the overlap strips are exchanged
    with the neighbours (inference/sharded.py).  Returns this rank's owned rows [C, rows, W] and their (lo, hi)."""
    from .sharded import ShardedCanvas
    b, c, h, w = noise.shape
    assert b == 1, "one canvas per call"
    device = noise.device
    canvas = ShardedCanvas(c, h, w, tile_size, tile_stride, device, group=group)
    tiles = canvas.my_tiles()
    noise32, cond32 = noise.float(), cond_img.to(device).float()
    group_n = max(1, int(tile_batch))
    for g0 in range(0, len(tiles), group_n):
        chunk = tiles[g0:g0 + group_n]
        solve = get_diffusion_solve(model, scheduler, len(chunk), tile_size, tile_size, num_steps)
        x = torch.cat([noise32[..., i0:i0 + tile_size, j0:j0 + tile_size] for (i0, j0) in chunk], dim=0)
        cd = torch.cat([cond32[..., i0:i0 + tile_size, j0:j0 + tile_size] for (i0, j0) in chunk], dim=0)
        out = solve.run(x, cd)
        for t, (i0, j0) in enumerate(chunk):
            canvas.add_tile(out[t].clone(), i0, j0)
        if g0 + len(chunk) >= canvas.n_boundary_tiles():
            canvas.start_exchange()          # boundary rows are done: their strip travels during the interior solves
    canvas.finalize()
    return canvas.normalized_owned(), (canvas.own_lo, canvas.own_hi)
