"""CPU checks of two-model guidance and score scaling (run with -m "not gpu"): the score-scaling fold against the
reference's _scale_score formula, the guided descriptor's ABI, the solve-cache key, the base model's condition
processing and the oracle restatements against tests/golden/guided_golden.npz."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import guided as OG
from oracle import scheduler as osched
from oracle import tiling as otile
from oracle import unet as ounet
from terrain_diffusion_b200 import _lib as L
from terrain_diffusion_b200.inference import process_base_cond_img
from terrain_diffusion_b200.inference import samplers as S
from terrain_diffusion_b200.inference.solve import check_guide, score_scaling_fold
from terrain_diffusion_b200.scheduler import EDMDPMSolverMultistepScheduler

ROOT = Path(__file__).resolve().parent.parent
GG = np.load(ROOT / "tests" / "golden" / "guided_golden.npz")


def rel_rms(a, b):
    return float((a - b).square().mean().sqrt() / b.square().mean().sqrt())


def _rows(steps=12):
    sch = EDMDPMSolverMultistepScheduler()
    sch.set_timesteps(steps)
    order = sch.order_schedule()
    return [sch.step_coefficients(i, order[i]) for i in range(steps)]


@pytest.mark.parametrize("alpha", [0.5, 0.9, 1.3, 2.0])
def test_score_scaling_fold_equals_reference_formula_fp64(alpha):
    for row in _rows():
        sigma = 0.5 * np.tan(row["t"])
        a, b = OG.scale_score_linear(sigma, 0.5, alpha)
        got = score_scaling_fold(row, 0.5, alpha)
        assert got["c_skip"] == pytest.approx(row["c_skip"] + row["c_out"] * a, rel=1e-12, abs=1e-15)
        assert got["c_out"] == pytest.approx(row["c_out"] * b, rel=1e-12)
        assert {k: got[k] for k in ("c_in", "t", "r", "k")} == {k: row[k] for k in ("c_in", "t", "r", "k")}


def test_score_scaling_alpha_one_gives_identical_rows():
    for row in _rows():
        assert score_scaling_fold(row, 0.5, 1.0) == row


def test_score_scaling_fold_applied_to_a_sample():
    """x0 from the folded row == x0 from the unfolded row applied to _scale_score(mo) (fp64 element-wise)."""
    g = torch.Generator().manual_seed(3)
    x, mo = torch.randn(64, generator=g, dtype=torch.float64), torch.randn(64, generator=g, dtype=torch.float64)
    for row in _rows(6):
        sigma = 0.5 * np.tan(row["t"])
        f = score_scaling_fold(row, 0.5, 1.4)
        want = row["c_skip"] * x + row["c_out"] * OG.scale_score(mo, x, sigma, 0.5, 1.4)
        torch.testing.assert_close(f["c_skip"] * x + f["c_out"] * mo, want, rtol=1e-12, atol=1e-12)


def test_guided_descriptor_abi():
    lib = L.lib()
    assert L.ABI_STRUCTS[8] is L.TdxConvOutGuidedDesc
    assert lib.tdx_abi_sizeof(8) == C.sizeof(L.TdxConvOutGuidedDesc) == C.sizeof(L.TdxConvOutDesc) + 8
    assert lib.tdx_abi_sizeof(3) == C.sizeof(L.TdxConvOutDesc) == 72        # the plain descriptor is unchanged
    assert L.TdxConvOutGuidedDesc.guide_out.offset == C.sizeof(L.TdxConvOutDesc)
    d = L.TdxConvOutGuidedDesc()
    assert lib.tdx_conv_out_guided_run(C.byref(d), None) == -1                # validation runs without a GPU
    assert lib.tdx_conv_out_guided_run(None, None) == -1


# ------------------------------------------------------------------------------------------------ solve cache key
class _FakeModel:
    def __init__(self, cfg, device="cuda:0"):
        self.config, self.device, self._fw = dict(cfg), torch.device(device), object()

    def folded(self):
        return self._fw


class _FakeSolve:
    made = []

    def __init__(self, model, scheduler, n, h, w, num_steps, step_range=None, guide=None, guidance_scale=1.0,
                 score_scaling=1.0):
        self.guide, self.scale, self.score_scaling = guide, guidance_scale, score_scaling
        _FakeSolve.made.append(self)

    def set_guidance_scale(self, s):
        self.scale = s


def test_cache_key_guide_changes_it_scale_does_not(monkeypatch):
    monkeypatch.setattr(S, "DiffusionSolve", _FakeSolve)
    m, g = _FakeModel(ounet.DECODER_CFG), _FakeModel(ounet.DECODER_CFG)
    sch = EDMDPMSolverMultistepScheduler()
    plain = S.get_diffusion_solve(m, sch, 1, 64, 64, 4)
    assert S.get_diffusion_solve(m, sch, 1, 64, 64, 4, guide=g, guidance_scale=1.0) is plain   # s == 1: unguided
    assert S.get_diffusion_solve(m, sch, 1, 64, 64, 4, guide=None, guidance_scale=2.0) is plain
    s2 = S.get_diffusion_solve(m, sch, 1, 64, 64, 4, guide=g, guidance_scale=2.0)
    assert s2 is not plain and s2.guide is g and s2.scale == 2.0
    s3 = S.get_diffusion_solve(m, sch, 1, 64, 64, 4, guide=g, guidance_scale=3.0)
    assert s3 is s2 and s3.scale == 3.0                                   # same program, table rewritten
    other = S.get_diffusion_solve(m, sch, 1, 64, 64, 4, guide=_FakeModel(ounet.DECODER_CFG), guidance_scale=3.0)
    assert other is not s2
    a = S.get_diffusion_solve(m, sch, 1, 64, 64, 4, guide=g, guidance_scale=2.0, score_scaling=1.3)
    assert a is not s2 and a.score_scaling == 1.3
    assert S.get_diffusion_solve(m, sch, 1, 64, 64, 4, score_scaling=1.3) not in (plain, a)
    assert len(_FakeSolve.made) == 5


def test_mismatched_guide_raises_before_planning(monkeypatch):
    monkeypatch.setattr(S, "DiffusionSolve", _FakeSolve)
    m = _FakeModel(ounet.DECODER_CFG)
    sch = EDMDPMSolverMultistepScheduler()
    for bad in (_FakeModel(dict(ounet.DECODER_CFG, out_channels=2)), _FakeModel(dict(ounet.DECODER_CFG, in_channels=6)),
                _FakeModel(dict(ounet.DECODER_CFG, conditional_inputs=[["tensor", 58, 1.0]])),
                _FakeModel(ounet.DECODER_CFG, device="cuda:1")):
        with pytest.raises(ValueError):
            check_guide(m, bad)
        with pytest.raises(ValueError):
            S.get_diffusion_solve(m, sch, 1, 64, 64, 4, guide=bad, guidance_scale=2.0)
    check_guide(_FakeModel(OG.BASE_CFG), _FakeModel(OG.GUIDE_CFG))        # the shipped pair is compatible


# ------------------------------------------------------------------------------------------------ condition vector
def _cond_img_case():
    return {k: torch.from_numpy(GG["cond_img." + k]) for k in ("cond_img", "cond_means", "cond_stds", "noise_level",
                                                                "histogram_raw")}


def test_process_base_cond_img_matches_reference_golden():
    ci = _cond_img_case()
    torch.manual_seed(OG.COND_IMG_SEED)       # the reference's NaN climate fill draws from the global generator
    got = process_base_cond_img(ci["cond_img"].clone(), ci["histogram_raw"], ci["cond_means"], ci["cond_stds"],
                                ci["noise_level"])
    want = torch.from_numpy(GG["cond_img.y"])
    assert got.shape == (3, 58) and not torch.isnan(want).any()
    torch.testing.assert_close(got, want, rtol=1e-5, atol=1e-5)


def test_oracle_process_cond_img_matches_reference_golden():
    ci = _cond_img_case()
    torch.manual_seed(OG.COND_IMG_SEED)
    got = OG.process_cond_img(ci["cond_img"].clone(), ci["histogram_raw"], ci["cond_means"], ci["cond_stds"],
                              ci["noise_level"])
    torch.testing.assert_close(got, torch.from_numpy(GG["cond_img.y"]), rtol=0, atol=0)


# ------------------------------------------------------------------------------------------------ oracle restatements
def test_oracle_guided_score_scaled_decoder_matches_reference_golden():
    cfg = ounet.DECODER_CFG
    sd_m, sd_g = ounet.procedural_state_dict(cfg, seed=0), ounet.procedural_state_dict(cfg, seed=2)
    noise, cond = torch.from_numpy(GG["decoder.noise"]), torch.from_numpy(GG["decoder.cond"])
    sch = osched.OracleScheduler()
    sch.set_timesteps(4)
    x = noise.clone()
    for t, sigma in zip(sch.timesteps, sch.sigmas):
        xin = torch.cat([sch.precondition_inputs(x, sigma), cond], dim=1)
        cn = sch.trigflow_precondition_noise(sigma.view(-1))
        mo = OG.guided_output(ounet.unet_forward(sd_m, cfg, xin, cn, []), ounet.unet_forward(sd_g, cfg, xin, cn, []), 2.0)
        x = sch.step(OG.scale_score(mo, x, sigma, 0.5, 1.3), t, x)
    assert rel_rms(x, torch.from_numpy(GG["decoder.y"])) < 1e-5


@pytest.mark.slow
def test_oracle_base_sampler_tiled_matches_reference_golden():
    sd_m, sd_g = ounet.procedural_state_dict(OG.BASE_CFG, seed=0), ounet.procedural_state_dict(OG.GUIDE_CFG, seed=1)
    ti = OG.tiled_inputs()
    noise = torch.randn((2, 5, 96, 96), generator=torch.Generator().manual_seed(61))
    got = OG.sample_base_diffusion(lambda x, t, c: ounet.unet_forward(sd_m, OG.BASE_CFG, x, t, c),
                                   lambda x, t, c: ounet.unet_forward(sd_g, OG.GUIDE_CFG, x, t, c),
                                   osched.OracleScheduler, noise, ti["cond_img"], steps=2, guidance_scale=2.15,
                                   tile_size=64, cond_means=ti["cond_means"], cond_stds=ti["cond_stds"],
                                   noise_level=ti["noise_level"], histogram_raw=ti["histogram_raw"])
    assert otile.tile_starts(96, 64, 32) == [0, 32]
    assert rel_rms(got, torch.from_numpy(GG["base_tiled.y"])) < 1e-4
