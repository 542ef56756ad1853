"""ORACLE (test infrastructure, not product): CPU restatement of two-model guidance, score scaling and the base-model
diffusion sampler of xandergos/terrain-diffusion @ 82a0431:

  guided output  mo = mo_g + s*(mo_m - mo_g)        training/evaluation/sample_diffusion_base.py:105-110,
                                                    sample_diffusion_decoder.py:112-117
  _scale_score                                      sample_diffusion_decoder.py:7-40
  _process_cond_img                                 sample_diffusion_base.py:11-48
  sample_base_diffusion (noise passed explicitly)   sample_diffusion_base.py:51-168

Parity pinned by tests against outputs of the unmodified reference recorded by tests/golden/make_golden_guided.py.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import tiling as otile
from .unet import mp_concat

BASE_CFG = dict(image_size=512, in_channels=5, out_channels=5, model_channels=192, model_channel_mults=[1, 2, 3, 4],
                layers_per_block=3, attn_resolutions=[8, 16], midblock_attention=True, concat_balance=0.5,
                conditional_inputs=[["tensor", 58, 1.0]], fourier_scale="pos", block_kwargs={"dropout": 0.1})
"""configs/diffusion_base/diffusion_192-3.cfg [model] (Diffusion-Base-192x3)."""
GUIDE_CFG = dict(BASE_CFG, model_channels=128, block_kwargs=None)
"""configs/diffusion_base/diffusion_128-3.cfg [model] (Diffusion-Base-128x3, the shipped guide of the base model)."""

COND_MEANS = [14.99, 11.65, 15.87, 619.26, 833.12, 69.40, 0.66]     # diffusion_192-3.cfg [sweep_dataset]
COND_STDS = [21.72, 21.78, 10.40, 452.29, 738.09, 34.59, 0.47]
COND_IMG_SEED = 1234


def guided_output(mo_m: torch.Tensor, mo_g: torch.Tensor, s: float) -> torch.Tensor:
    """mo_g + s * (mo_m - mo_g) in the tensors' dtype, operation by operation."""
    return mo_g + s * (mo_m - mo_g)


def scale_score(mo, sample, sigma, sigma_data: float, alpha: float = 1.0):
    """_scale_score: v = -sigma_d mo; x0 = x cos t - v sin t; eps = x sin t + v cos t; x0_a = x + alpha (x0 - x);
    returns (eps cos t - x0_a sin t) / -sigma_d with t = atan(sigma / sigma_d)."""
    if alpha == 1.0:
        return mo
    sigma = torch.as_tensor(sigma, dtype=sample.dtype)
    sd = torch.as_tensor(sigma_data, dtype=sample.dtype)
    v = -sd * mo
    t = torch.atan(sigma / sd)
    c, s = torch.cos(t), torch.sin(t)
    x0 = sample * c - v * s
    eps = sample * s + v * c
    x0a = sample + alpha * (x0 - sample)
    return (eps * c - x0a * s) / -sd


def scale_score_linear(sigma: float, sigma_data: float, alpha: float) -> tuple[float, float]:
    """(a, b) with scale_score(mo, x) = a x + b mo, evaluated in fp64 from the trig form above (x = 1, mo = 0 and
    x = 0, mo = 1)."""
    f = lambda x, mo: float(scale_score(torch.tensor(mo, dtype=torch.float64), torch.tensor(x, dtype=torch.float64),
                                        sigma, sigma_data, alpha))
    return f(1.0, 0.0), f(0.0, 1.0)


def process_cond_img(cond_img, histogram_raw, cond_means, cond_stds, noise_level):
    """_process_cond_img: standardise; NaNs of batch ROW 0 -> cond_means[0] and of row 1 -> cond_means[1] (the
    reference indexes the batch, not the channel); centre 2 x 2 climate means; remaining NaN climate means ->
    randn_like (global generator); mp_concat of the six parts with equal weights."""
    means = torch.as_tensor(cond_means).view(1, -1, 1, 1)
    stds = torch.as_tensor(cond_stds).view(1, -1, 1, 1)
    x = (cond_img - means) / stds
    x[0:1] = x[0:1].nan_to_num(float(cond_means[0]))
    x[1:2] = x[1:2].nan_to_num(float(cond_means[1]))
    level = (noise_level - 0.5) * np.sqrt(12)
    clim = x[:, 2:6, 1:3, 1:3].mean(dim=(2, 3))
    nan = torch.isnan(clim)
    clim[nan] = torch.randn_like(clim[nan])
    parts = [x[:, 0:1].flatten(1), x[:, 1:2].flatten(1), clim.flatten(1), x[:, 6:7].flatten(1), histogram_raw,
             level.view(-1, 1)]
    return mp_concat(parts, [1 / len(parts)] * len(parts), dim=1).float()


def sample_base_diffusion(model_fn, guide_fn, make_scheduler, noise, cond_inputs, *, steps, guidance_scale=1.0,
                          tile_size=None, cond_means=None, cond_stds=None, noise_level=None, histogram_raw=None):
    """sample_base_diffusion with the unit-variance initial noise given (the reference draws it with torch.randn from
    its generator).  model_fn / guide_fn(x, t, cond_list) -> model output.  Untiled: returns the samples (no
    division by sigma_data); tiled (stride tile_size // 2, 4 x 4 condition windows, per-tile scheduler reset):
    returns blend / weights / sigma_data."""
    sched = make_scheduler()
    sigma0 = sched.sigmas[0] if getattr(sched, "sigmas", None) is not None else None
    if sigma0 is None:
        sched.set_timesteps(1000)
        sigma0 = sched.sigmas[0]

    def solve(x, cond):
        sched.set_timesteps(steps)
        for t, sigma in zip(sched.timesteps, sched.sigmas):
            xin = sched.precondition_inputs(x, sigma)
            cn = sched.trigflow_precondition_noise(sigma.view(-1).expand(x.shape[0]))
            mo = model_fn(xin, cn, cond)
            if guide_fn is not None and guidance_scale != 1.0:
                mo = guided_output(mo, guide_fn(xin, cn, cond), guidance_scale)
            x = sched.step(mo, t, x)
        return x

    x = noise * sigma0
    if tile_size is None:
        return solve(x, cond_inputs)
    n, c, h, w = x.shape
    hs, ws = otile.tile_starts(h, tile_size, tile_size // 2), otile.tile_starts(w, tile_size, tile_size // 2)
    weights = otile.linear_weight_window(tile_size)
    acc, acc_w = torch.zeros_like(x), torch.zeros_like(x)
    for ic, i0 in enumerate(hs):
        for jc, j0 in enumerate(ws):
            cond = [process_cond_img(cond_inputs[..., ic:ic + 4, jc:jc + 4].clone(), histogram_raw, cond_means,
                                     cond_stds, noise_level)]
            tile = solve(x[..., i0:i0 + tile_size, j0:j0 + tile_size], cond)
            otile.accumulate(acc, acc_w, tile, weights, i0, j0)
    return acc / acc_w / sched.sigma_data


# ---------------------------------------------------------------------------------------------- fixture inputs
def tiled_inputs() -> dict:
    """Inputs of the tiled base-sampler golden: 2 canvases of 96 x 96 (4 tiles of 64, stride 32), a 5 x 5 grid of the
    seven raw condition channels with NaNs in batch rows 0 and 1 (replaced before the climate crop is taken)."""
    g = torch.Generator().manual_seed(62)
    means, stds = torch.tensor(COND_MEANS), torch.tensor(COND_STDS)
    img = torch.randn(2, 7, 5, 5, generator=g) * stds.view(1, -1, 1, 1) + means.view(1, -1, 1, 1)
    img[:, 6] = (img[:, 6] > means[6]).float()
    img[0, 0, 1, 2] = float("nan")
    img[1, 3, 2, 2] = float("nan")
    return dict(cond_img=img, cond_means=means, cond_stds=stds, noise_level=torch.tensor([[0.0], [0.05]]),
                histogram_raw=torch.randn(2, 5, generator=g))


def cond_img_inputs() -> dict:
    """Inputs of the _process_cond_img golden: 3 images; row 2 has a NaN inside the centre 2 x 2 of channel 4."""
    g = torch.Generator().manual_seed(63)
    means, stds = torch.tensor(COND_MEANS), torch.tensor(COND_STDS)
    img = torch.randn(3, 7, 4, 4, generator=g) * stds.view(1, -1, 1, 1) + means.view(1, -1, 1, 1)
    img[0, 1, 0, 0] = float("nan")
    img[1, 2, 1, 1] = float("nan")
    img[2, 4, 2, 1] = float("nan")
    return dict(cond_img=img, cond_means=means, cond_stds=stds, noise_level=torch.tensor([[0.0], [0.1], [0.02]]),
                histogram_raw=torch.randn(3, 5, generator=g))
