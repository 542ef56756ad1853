"""Two-model guidance and score scaling on the GPU: the guided last convolution bit for bit against a torch fp32
restatement, the guide and the guided samplers against the unmodified reference (tests/golden/make_golden_guided.py),
and the properties of the guided program (no guide == today's program, the guidance scale in the device table,
tile batching against the oracle)."""
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
from terrain_diffusion_b200.inference import DiffusionSolve, sample_base_diffusion, sample_decoder_diffusion_tiled
from terrain_diffusion_b200.inference.samplers import get_diffusion_solve
from terrain_diffusion_b200.layout import to_nc8hw8
from terrain_diffusion_b200.models import EDMUnet2D
from terrain_diffusion_b200.scheduler import EDMDPMSolverMultistepScheduler

pytestmark = pytest.mark.gpu
GG = np.load(Path(__file__).resolve().parent / "golden" / "guided_golden.npz")
TOL = 1.0e-2


def rel_rms(a, b):
    return float((a - b).square().mean().sqrt() / (b.square().mean().sqrt() + 1e-30))


def _model(cfg, seed):
    m = EDMUnet2D(**cfg).eval()
    m.load_state_dict(ounet.procedural_state_dict(cfg, seed=seed))
    return m.cuda()


@pytest.fixture(scope="module")
def base_pair():
    return _model(OG.BASE_CFG, 0), _model(OG.GUIDE_CFG, 1)


@pytest.fixture(scope="module")
def decoder_pair():
    return _model(ounet.DECODER_CFG, 0), _model(ounet.DECODER_CFG, 2)


def _sched():
    return EDMDPMSolverMultistepScheduler(sigma_min=0.002, sigma_max=80, sigma_data=0.5)


def _check(err, key):
    """DESIGN section 2: err <= 1e-2 and <= 1.25 x the reference's own bf16 error; where that bf16 error itself exceeds
    1e-2 (guidance amplifies bf16 rounding), the relative clause alone."""
    ref_bf16 = float(GG[key + ".ref_bf16_err"])
    assert err <= 1.25 * ref_bf16, (err, ref_bf16)
    if ref_bf16 <= TOL:
        assert err < TOL, (err, ref_bf16)


# ------------------------------------------------------------------------------------------------ the kernel
@pytest.mark.parametrize("c_in,c_out", [(64, 1), (128, 1), (192, 5), (128, 8)])
def test_guided_conv_out_is_bit_exact(c_in, c_out):
    """F = F_g + s*(F_m - F_g) with F_m the kernel's own unguided model_out, then the update, op for op in fp32."""
    g = torch.Generator(device="cuda").manual_seed(c_in + c_out)
    n, h, w = 2, 24, 40
    dev = "cuda"
    x = to_nc8hw8(torch.randn(n, c_in, h, w, device=dev, generator=g)).contiguous()
    wpad = 1 if c_out == 1 else 8
    weight = torch.zeros(9, c_in, wpad, device=dev)
    weight[..., :c_out] = torch.randn(9, c_in, c_out, device=dev, generator=g) / (3 * c_in ** 0.5)
    f_m = torch.empty(n, c_out, h, w, device=dev)
    d = L.TdxConvOutDesc()
    d.x, d.c_in, d.weight, d.c_out = x.data_ptr(), c_in, weight.data_ptr(), c_out
    d.n_img, d.height, d.width = n, h, w
    d.model_out = f_m.data_ptr()
    L.call(L.lib().tdx_conv_out_run, dev, C.byref(d))
    f_g = torch.randn(n, c_out, h, w, device=dev, generator=g)
    sample = torch.randn(n, c_out, h, w, device=dev, generator=g) * 3
    x0p = torch.randn(n, c_out, h, w, device=dev, generator=g)
    coef = torch.tensor([0.3, -0.7, 0.55, 0.12, 2.15], device=dev)
    s0, p0 = sample.clone(), x0p.clone()
    f = torch.empty_like(f_m)
    gd = L.TdxConvOutGuidedDesc()
    gd.base = d
    gd.base.model_out = f.data_ptr()
    gd.base.sched_coef, gd.base.sample, gd.base.x0_prev = coef.data_ptr(), sample.data_ptr(), x0p.data_ptr()
    gd.guide_out = f_g.data_ptr()
    L.call(L.lib().tdx_conv_out_guided_run, dev, C.byref(gd))
    torch.cuda.synchronize()
    cs, co, r, k, s = (coef[i] for i in range(5))
    want_f = torch.add(f_g, torch.mul(s, torch.sub(f_m, f_g)))
    x0 = torch.add(torch.mul(cs, s0), torch.mul(co, want_f))
    want_x = torch.add(torch.add(torch.mul(r, s0), torch.mul(1.0 - r, x0)), torch.mul(k, torch.sub(x0, p0)))
    assert torch.equal(f, want_f)
    assert torch.equal(x0p, x0)
    assert torch.equal(sample, want_x)


# ------------------------------------------------------------------------------------------------ against the reference
def test_guide_128x3_forward_matches_reference_golden(base_pair):
    _, guide = base_pair
    g = torch.Generator().manual_seed(41)
    x = torch.randn(2, 5, 64, 64, generator=g)
    t = torch.atan(torch.exp(torch.randn(2, generator=g) * 1.5) / 0.5)
    c = torch.randn(2, 58, generator=g)
    y = guide(x.cuda(), t.cuda(), [c.cuda()]).cpu()
    _check(rel_rms(y, torch.from_numpy(GG["guide_fwd.y"])), "guide_fwd")


def test_guided_base_sampler_untiled_matches_reference_golden(base_pair):
    m, guide = base_pair
    noise = torch.from_numpy(GG["base_untiled.noise"]).cuda()
    got = sample_base_diffusion(m, _sched(), (2, 5, 64, 64), [torch.from_numpy(GG["base_untiled.cond"]).cuda()],
                                steps=4, guide_model=guide, guidance_scale=2.15, noise=noise).cpu()
    _check(rel_rms(got, torch.from_numpy(GG["base_untiled.y"])), "base_untiled")


def test_guided_base_sampler_tiled_matches_reference_golden(base_pair):
    m, guide = base_pair
    ti = {k: torch.from_numpy(GG["base_tiled." + k]) for k in ("cond_img", "cond_means", "cond_stds", "noise_level",
                                                                 "histogram_raw")}
    noise = torch.randn((2, 5, 96, 96), generator=torch.Generator().manual_seed(61))
    got = sample_base_diffusion(m, _sched(), (2, 5, 96, 96), ti["cond_img"].cuda(), cond_means=ti["cond_means"],
                                cond_stds=ti["cond_stds"], noise_level=ti["noise_level"],
                                histogram_raw=ti["histogram_raw"], steps=2, guide_model=guide, guidance_scale=2.15,
                                tile_size=64, noise=noise.cuda()).cpu()
    assert got.shape == (2, 5, 96, 96)
    _check(rel_rms(got, torch.from_numpy(GG["base_tiled.y"])), "base_tiled")


def test_guided_score_scaled_decoder_tile_matches_reference_golden(decoder_pair):
    m, guide = decoder_pair
    got = sample_decoder_diffusion_tiled(m, _sched(), torch.from_numpy(GG["decoder.cond"]).cuda(),
                                         torch.from_numpy(GG["decoder.noise"]).cuda(), 64, 64, num_steps=4,
                                         guidance_model=guide, guidance_scale=2.0, score_scaling=1.3).cpu()
    _check(rel_rms(got, torch.from_numpy(GG["decoder.y"])), "decoder")


# ------------------------------------------------------------------------------------------------ program properties
@pytest.mark.parametrize("guide_kind", ["none", "scale_one"])
def test_no_guide_or_scale_one_is_todays_program(decoder_pair, guide_kind):
    m, guide = decoder_pair
    g = torch.Generator().manual_seed(5)
    x, cond = (torch.randn(2, 1, 64, 64, generator=g) * 80).cuda(), torch.randn(2, 4, 64, 64, generator=g).cuda()
    plain = DiffusionSolve(m, _sched(), 2, 64, 64, 4)
    kw = dict(guide=None, guidance_scale=2.0) if guide_kind == "none" else dict(guide=guide, guidance_scale=1.0)
    other = DiffusionSolve(m, _sched(), 2, 64, 64, 4, **kw)
    assert other.guide is None and other.launches_per_solve == plain.launches_per_solve
    assert L.lib().tdx_program_num_launches(other.prog.handle) == L.lib().tdx_program_num_launches(plain.prog.handle)
    assert torch.equal(other.coef, plain.coef)
    assert torch.equal(plain.run(x, cond).clone(), other.run(x, cond).clone())


def test_guided_program_adds_exactly_the_guide_forward(decoder_pair):
    m, guide = decoder_pair
    plain = DiffusionSolve(m, _sched(), 1, 64, 64, 3)
    guided = DiffusionSolve(m, _sched(), 1, 64, 64, 3, guide=guide, guidance_scale=2.0)
    per_fwd = (plain.launches_per_solve - 1) // 3
    assert guided.launches_per_solve == plain.launches_per_solve + 1 + 3 * per_fwd
    assert guided.coef.shape == (3, 5) and torch.all(guided.coef[:, 4] == 2.0)
    assert guided.guide_igemm_flops == guided.igemm_flops == plain.igemm_flops     # same architecture


def test_changing_the_scale_reuses_the_program_and_matches_a_fresh_solve(decoder_pair):
    m, guide = decoder_pair
    g = torch.Generator().manual_seed(6)
    x, cond = (torch.randn(1, 1, 64, 64, generator=g) * 80).cuda(), torch.randn(1, 4, 64, 64, generator=g).cuda()
    a = get_diffusion_solve(m, _sched(), 1, 64, 64, 4, guide=guide, guidance_scale=2.0)
    out_a = a.run(x, cond).clone()
    handle = a.prog.handle.value
    b = get_diffusion_solve(m, _sched(), 1, 64, 64, 4, guide=guide, guidance_scale=2.6)
    assert b is a and b.prog.handle.value == handle
    out_b = b.run(x, cond).clone()
    fresh = DiffusionSolve(m, _sched(), 1, 64, 64, 4, guide=guide, guidance_scale=2.6)
    assert torch.equal(out_b, fresh.run(x, cond).clone())
    assert not torch.equal(out_a, out_b)


def test_guided_multi_tile_batching_matches_oracle_per_tile_reset(decoder_pair):
    """4 tiles of 64 @ 32 on a 96 x 96 canvas, solved one by one and all four in one guided program.  The blend is
    applied in row-major order either way, but a batch of 4 runs other igemm work-item shapes than a batch of 1 (fp32
    summation order, see test_parity_r2_gpu.py::test_batch16_rows_equal_single_tile_rows), so the two canvases agree to
    bf16-pipeline precision, not bit for bit; both match the oracle with a per-tile solver reset."""
    m, guide = decoder_pair
    g = torch.Generator().manual_seed(8)
    sch = _sched()
    sch.set_timesteps(2)
    noise = torch.randn(1, 1, 96, 96, generator=g) * float(sch.sigmas[0])
    cond = torch.randn(1, 4, 96, 96, generator=g)
    outs = [sample_decoder_diffusion_tiled(m, _sched(), cond.cuda(), noise.cuda(), 64, 32, num_steps=2,
                                           guidance_model=guide, guidance_scale=2.0, tile_batch=tb).cpu()
            for tb in (1, 4)]
    assert rel_rms(outs[1], outs[0]) < 6e-3
    cfg = ounet.DECODER_CFG
    sd_m, sd_g = ounet.procedural_state_dict(cfg, seed=0), ounet.procedural_state_dict(cfg, seed=2)
    fn = lambda x, t: OG.guided_output(ounet.unet_forward(sd_m, cfg, x, t, []), ounet.unet_forward(sd_g, cfg, x, t, []),
                                       2.0)
    ref = otile.sample_decoder_diffusion_tiled(fn, osched.OracleScheduler, cond, noise, 64, 32, num_steps=2)
    for out in outs:
        assert rel_rms(out, ref) < TOL


def test_mismatched_guide_raises_value_error(base_pair, decoder_pair):
    m, _ = decoder_pair
    base, _ = base_pair
    with pytest.raises(ValueError):
        DiffusionSolve(m, _sched(), 1, 64, 64, 2, guide=base, guidance_scale=2.0)
    with pytest.raises(ValueError):
        sample_decoder_diffusion_tiled(m, _sched(), torch.zeros(1, 4, 64, 64, device="cuda"),
                                       torch.zeros(1, 1, 64, 64, device="cuda"), num_steps=2, guidance_model=base,
                                       guidance_scale=2.0)


def test_cpu_guide_raises():
    cpu = EDMUnet2D(**ounet.DECODER_CFG).eval()
    gpu = _model(ounet.DECODER_CFG, 0)
    with pytest.raises(ValueError):
        DiffusionSolve(gpu, _sched(), 1, 64, 64, 2, guide=cpu, guidance_scale=2.0)
    with pytest.raises(L.TdxError):
        DiffusionSolve(cpu, _sched(), 1, 64, 64, 2)
