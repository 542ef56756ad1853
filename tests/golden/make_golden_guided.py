"""Golden fixtures of two-model guidance (tests/golden/guided_golden.npz), generated from the UNMODIFIED reference
xandergos/terrain-diffusion @ 82a0431 on the CPU through the diffusers stand-in under oracle/_stub, with procedural
weights (oracle.unet.procedural_state_dict):

  guide_fwd.*        one forward of the Diffusion-Base-128x3 architecture (the shipped guide of the base model) at
                     64 x 64, batch 2, 58-dim tensor condition (inputs: the seed-41 stream below)
  base_untiled.*     sample_base_diffusion (training/evaluation/sample_diffusion_base.py:51-113), untiled, 192x3 main +
                     128x3 guide, guidance scale 2.15, 4 steps, batch 2; the initial noise is a seeded CPU stream and is
                     stored next to the result
  base_tiled.*       the same function's tiled branch (:115-168) on a 96 x 96 canvas: tile 64 / stride 32 = 4 tiles,
                     a 5 x 5 condition grid (oracle.guided.tiled_inputs; noise: the seed-61 stream) processed per
                     tile by _process_cond_img (with NaNs in batch rows 0 and 1, which the reference replaces before
                     the climate crop), 2 steps, guidance scale 2.15
  decoder.*          sample_decoder_diffusion_tiled (sample_diffusion_decoder.py:44-125) on one 64 x 64 tile, decoder
                     64x3 main + a 64x3 guide with other weights, guidance scale 2, score_scaling 1.3, 4 steps
  cond_img.*         _process_cond_img on a 3-image batch whose third row has a NaN climate mean (filled with
                     randn_like from the global generator, seeded below)

Every sampler case is run twice: in fp32, and with both U-Nets in the reference's own bf16 mode (model.to(bfloat16),
bf16 inputs, as WorldPipeline does for dtype='bf16') around the same fp32 sampler; `*.ref_bf16_err` is the rel-RMS of
the bf16 result against the fp32 one -- the second clause of the DESIGN section 2 tolerance.

    python tests/golden/make_golden_guided.py
"""
from __future__ import annotations

import sys
import time
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
REF = Path("/root/reference")
sys.path[:0] = [str(ROOT / "oracle" / "_stub"), str(REF), str(ROOT)]

from terrain_diffusion.models.edm_unet import EDMUnet2D  # noqa: E402
from terrain_diffusion.scheduler.dpmsolver import EDMDPMSolverMultistepScheduler  # noqa: E402
from terrain_diffusion.training.evaluation.sample_diffusion_base import (  # noqa: E402
    _process_cond_img, sample_base_diffusion)
from terrain_diffusion.training.evaluation.sample_diffusion_decoder import sample_decoder_diffusion_tiled  # noqa: E402

from oracle import guided as OG  # noqa: E402
from oracle import unet as O  # noqa: E402

torch.set_grad_enabled(False)


class Bf16(torch.nn.Module):
    """The reference U-Net in its own bf16 mode: bf16 weights and inputs, output returned in fp32."""

    def __init__(self, m):
        super().__init__()
        self.m = m.to(torch.bfloat16)

    def forward(self, x, noise_labels, conditional_inputs):
        ci = [c.to(torch.bfloat16) if c.is_floating_point() else c for c in conditional_inputs]
        return self.m(x.to(torch.bfloat16), noise_labels.to(torch.bfloat16), ci).float()


def build_ref(cfg, seed):
    m = EDMUnet2D(**cfg).eval()
    m.load_state_dict(O.procedural_state_dict(cfg, seed=seed))
    return m


def rel_rms(a, b):
    return float((a.float() - b.float()).square().mean().sqrt() / b.float().square().mean().sqrt())


def both(out, key, fn, main_cfg, main_seed, guide_cfg, guide_seed):
    """fn(main, guide) -> fp32 tensor, once with fp32 models and once with bf16 models."""
    t0 = time.time()
    y = fn(build_ref(main_cfg, main_seed), build_ref(guide_cfg, guide_seed))
    yb = fn(Bf16(build_ref(main_cfg, main_seed)), Bf16(build_ref(guide_cfg, guide_seed)))
    out[key + ".y"] = y.float().contiguous().numpy()
    out[key + ".ref_bf16_err"] = np.float64(rel_rms(yb, y))
    print(key, tuple(y.shape), f"bf16 err {out[key + '.ref_bf16_err']:.3e}", f"{time.time() - t0:.0f}s", flush=True)


def main():
    out = {}
    base, guide = OG.BASE_CFG, OG.GUIDE_CFG

    # ---- one guide forward
    g = torch.Generator().manual_seed(41)
    x = torch.randn(2, 5, 64, 64, generator=g)
    t = torch.atan(torch.exp(torch.randn(2, generator=g) * 1.5) / 0.5)
    c = torch.randn(2, 58, generator=g)
    m = build_ref(guide, 1)
    y = m(x, t, [c])
    yb = Bf16(build_ref(guide, 1))(x, t, [c])
    out.update({"guide_fwd.y": y.numpy(), "guide_fwd.ref_bf16_err": np.float64(rel_rms(yb, y))})
    print("guide_fwd", float(out["guide_fwd.ref_bf16_err"]), flush=True)

    # ---- untiled guided base sampler
    cvec = torch.randn(2, 58, generator=torch.Generator().manual_seed(52))
    out["base_untiled.noise"] = torch.randn((2, 5, 64, 64), generator=torch.Generator().manual_seed(51)).numpy()
    out["base_untiled.cond"] = cvec.numpy()

    def untiled(mm, gm):
        return sample_base_diffusion(mm, EDMDPMSolverMultistepScheduler(sigma_min=0.002, sigma_max=80, sigma_data=0.5),
                                     (2, 5, 64, 64), [cvec], cond_means=None, cond_stds=None, histogram_raw=None,
                                     steps=4, guide_model=gm, guidance_scale=2.15,
                                     generator=torch.Generator().manual_seed(51))
    both(out, "base_untiled", untiled, base, 0, guide, 1)

    # ---- tiled guided base sampler: 96^2 canvas, 4 tiles, 5 x 5 condition grid
    ti = OG.tiled_inputs()
    out.update({"base_tiled." + k: v.numpy() for k, v in ti.items()})

    def tiled(mm, gm):
        return sample_base_diffusion(mm, EDMDPMSolverMultistepScheduler(sigma_min=0.002, sigma_max=80, sigma_data=0.5),
                                     (2, 5, 96, 96), ti["cond_img"].clone(), cond_means=ti["cond_means"],
                                     cond_stds=ti["cond_stds"], noise_level=ti["noise_level"],
                                     histogram_raw=ti["histogram_raw"], steps=2, guide_model=gm, guidance_scale=2.15,
                                     generator=torch.Generator().manual_seed(61), tile_size=64)
    both(out, "base_tiled", tiled, base, 0, guide, 1)

    # ---- guided, score-scaled decoder tile
    g = torch.Generator().manual_seed(71)
    sched = EDMDPMSolverMultistepScheduler(sigma_min=0.002, sigma_max=80, sigma_data=0.5)
    sched.set_timesteps(4)
    noise = torch.randn(1, 1, 64, 64, generator=g) * sched.sigmas[0]
    cond = torch.randn(1, 4, 64, 64, generator=g)
    out["decoder.noise"], out["decoder.cond"] = noise.numpy(), cond.numpy()

    def decoder(mm, gm):
        s = EDMDPMSolverMultistepScheduler(sigma_min=0.002, sigma_max=80, sigma_data=0.5)
        return sample_decoder_diffusion_tiled(mm, s, cond, noise, 64, 64, num_steps=4, guidance_model=gm,
                                              guidance_scale=2.0, score_scaling=1.3)
    both(out, "decoder", decoder, O.DECODER_CFG, 0, O.DECODER_CFG, 2)

    # ---- _process_cond_img, including the randn_like fill of a NaN climate mean (batch row 2)
    ci = OG.cond_img_inputs()
    out.update({"cond_img." + k: v.numpy() for k, v in ci.items()})
    torch.manual_seed(OG.COND_IMG_SEED)
    out["cond_img.y"] = _process_cond_img(ci["cond_img"].clone(), ci["histogram_raw"], ci["cond_means"],
                                          ci["cond_stds"], ci["noise_level"]).numpy()

    np.savez_compressed(HERE / "guided_golden.npz", **out)
    print({k: getattr(v, "shape", ()) for k, v in out.items()})


if __name__ == "__main__":
    main()
