"""Throughput of two-model guided solves (one JSON line per workload).

    python tools/bench_guided.py [--reps 5] [--ref-steps 4] [--no-reference]

Workloads (procedural weights, synthetic inputs):
  base-guided     Diffusion-Base-192x3 + Diffusion-Base-128x3 guide, 64 x 64 latent tiles, 32 steps, s = 2.15
                  (the reference evaluation CLI's defaults, evaluation/base_diffusion.py), batch 40 and batch 1
  decoder-guided  decoder 64x3 + a same-architecture guide, 256 x 256 tiles, 20 steps, s = 2, 1 and 16 tiles

Per line: guided and unguided tile-steps/s measured in the same call (alternating, median of --reps), the time ratio
against the FLOP ratio 1 + G_guide / G_main (sums of 2*M*N*K over the igemm launches of the two recorded forwards), the
igemm share of the sustained bf16 peak (bench.py's roofline method and MEASURED_PEAKS.json), the card name and power
limit read in the same call, and a reference-GPU arm: the same guided solve through the oracle U-Nets in bf16 eager and
under torch.compile.  Needs a CUDA device; exits with an error otherwise.
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def card_info(index: int) -> dict:
    info = {"name": torch.cuda.get_device_name(index), "power_limit_w": None}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        info["power_limit_w"] = pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
    except Exception as e:  # pragma: no cover
        info["power_limit_error"] = repr(e)[:120]
    return info


def peak_tflops():
    try:
        p = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()).get("bf16_tflops_sustained")
        if p:
            return float(p), "MEASURED_PEAKS.json bf16_tflops_sustained"
    except Exception:
        pass
    return 1400.0, "fallback (B200 sustained ~1.4 PFLOP/s)"


def time_ms(fn) -> float:
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def reference_arm(cfg_m, cfg_g, n, size, steps, s, x0, cond_img, cond_vec, ref_steps):
    """The guided solve through the oracle U-Nets (PyTorch library kernels) in bf16, eager and torch.compile."""
    from oracle import scheduler as osched
    from oracle import unet as ounet
    from oracle.guided import guided_output
    dev = x0.device
    sd_m = {k: v.to(dev) for k, v in ounet.procedural_state_dict(cfg_m, seed=0).items()}
    sd_g = {k: v.to(dev) for k, v in ounet.procedural_state_dict(cfg_g, seed=1 if cond_vec is not None else 2).items()}
    ci = [cond_vec.bfloat16()] if cond_vec is not None else []

    def fwd(x, t):
        return guided_output(ounet.unet_forward(sd_m, cfg_m, x, t, ci).float(),
                             ounet.unet_forward(sd_g, cfg_g, x, t, ci).float(), s)

    out = {}
    variants = [("eager_bf16", fwd)]
    try:
        variants.append(("compile_bf16", torch.compile(fwd)))
    except Exception as e:  # pragma: no cover
        out["compile_bf16"] = {"unavailable": repr(e)[:200]}
    for name, f in variants:
        try:
            def solve(k):
                sch = osched.OracleScheduler()
                sch.set_timesteps(steps)
                sch.sigmas, sch.timesteps = sch.sigmas.to(dev), sch.timesteps.to(dev)
                x = x0.clone()
                for i, (t, sigma) in enumerate(zip(sch.timesteps, sch.sigmas)):
                    if i >= k:
                        break
                    xin = sch.precondition_inputs(x, sigma)
                    if cond_img is not None:
                        xin = torch.cat([xin, cond_img], dim=1)
                    lab = sch.trigflow_precondition_noise(sigma.view(-1)).expand(n)
                    mo = f(xin.bfloat16(), lab.bfloat16())
                    sch.step_index = i
                    x = sch.step(mo, t, x)
                return x
            with torch.no_grad():
                solve(min(3, steps))
                torch.cuda.synchronize()
                ms = time_ms(lambda: solve(ref_steps))
            out[name] = {"tile_steps_per_s": n * ref_steps / (ms / 1e3), "ms_per_step": ms / ref_steps,
                         "steps_timed": ref_steps}
        except Exception as e:  # pragma: no cover
            out[name] = {"unavailable": repr(e)[:300]}
    return out


def run(workload, n, args):
    from oracle import guided as OG
    from oracle import unet as ounet
    from terrain_diffusion_b200.inference.samplers import get_diffusion_solve
    from terrain_diffusion_b200.models import EDMUnet2D
    from terrain_diffusion_b200.scheduler import EDMDPMSolverMultistepScheduler
    dev = torch.device("cuda", 0)
    if workload == "base-guided":
        cfg_m, cfg_g, size, steps, s, gseed = OG.BASE_CFG, OG.GUIDE_CFG, 64, 32, 2.15, 1
    else:
        cfg_m, cfg_g, size, steps, s, gseed = ounet.DECODER_CFG, ounet.DECODER_CFG, 256, 20, 2.0, 2

    def model(cfg, seed):
        m = EDMUnet2D(**cfg).eval()
        m.load_state_dict(ounet.procedural_state_dict(cfg, seed=seed))
        return m.to(dev)

    main, guide = model(cfg_m, 0), model(cfg_g, gseed)
    sched = EDMDPMSolverMultistepScheduler()
    g = torch.Generator().manual_seed(7)
    cs = cfg_m["out_channels"]
    x0 = (torch.randn(n, cs, size, size, generator=g) * float(sched.sigmas[0])).to(dev)
    cond_img = torch.randn(n, cfg_m["in_channels"] - cs, size, size, generator=g).to(dev) if cfg_m["in_channels"] > cs \
        else None
    cond_vec = torch.randn(n, 58, generator=g).to(dev) if cfg_m["conditional_inputs"] else None
    ci = [cond_vec] if cond_vec is not None else None
    guided = get_diffusion_solve(main, sched, n, size, size, steps, guide=guide, guidance_scale=s)
    plain = get_diffusion_solve(main, sched, n, size, size, steps)
    for sv in (guided, plain):
        sv.prog.instantiate()
        for _ in range(args.warmup):
            sv.run(x0, cond_img, conditional_inputs=ci)
    torch.cuda.synchronize()
    ms_g, ms_p = [], []
    for _ in range(args.reps):                       # alternating, so clock drift hits both arms alike
        ms_g.append(time_ms(lambda: guided.run(x0, cond_img, conditional_inputs=ci)))
        ms_p.append(time_ms(lambda: plain.run(x0, cond_img, conditional_inputs=ci)))
    med = lambda v: sorted(v)[len(v) // 2]
    tg, tp = med(ms_g), med(ms_p)
    flops = guided.igemm_flops + guided.guide_igemm_flops
    flop_ratio = 1.0 + guided.guide_igemm_flops / guided.igemm_flops
    # igemm share: per-launch events of an eager run give the kernel's share of a solve; its time inside the graph
    # replay is that share of the replayed solve (bench.py's roofline method)
    guided.sample.copy_(x0)
    guided.x0_prev.zero_()
    guided.prog.profile()
    guided.sample.copy_(x0)
    guided.x0_prev.zero_()
    msl, kinds = guided.prog.profile()
    share = sum(m for m, k in zip(msl, kinds) if k == 1) / sum(msl)
    achieved = flops / (tg * share / 1e3) / 1e12
    peak, peak_src = peak_tflops()
    line = {"workload": workload, "tiles": n, "tile": size, "steps": steps, "guidance_scale": s,
            "main": f"{cfg_m['model_channels']}x{cfg_m['layers_per_block']}",
            "guide": f"{cfg_g['model_channels']}x{cfg_g['layers_per_block']}",
            "guided_tile_steps_per_s": n * steps / (tg / 1e3), "unguided_tile_steps_per_s": n * steps / (tp / 1e3),
            "guided_ms_per_solve": tg, "unguided_ms_per_solve": tp, "reps": args.reps,
            "time_ratio": tg / tp, "flop_ratio": flop_ratio,
            "igemm_gflop_main": guided.igemm_flops / 1e9, "igemm_gflop_guide": guided.guide_igemm_flops / 1e9,
            "launches_guided": guided.launches_per_solve, "launches_unguided": plain.launches_per_solve,
            "roofline": {"kernel": "tdx::igemm_kernel", "achieved_tflops": achieved, "peak_tflops": peak,
                         "frac": achieved / peak, "igemm_share_of_solve": share, "peak_source": peak_src},
            "card": card_info(0)}
    if not args.no_reference:
        line["reference_gpu"] = reference_arm(cfg_m, cfg_g, n, size, steps, s, x0, cond_img, cond_vec,
                                              min(args.ref_steps, steps))
        best = max((v["tile_steps_per_s"] for v in line["reference_gpu"].values() if "tile_steps_per_s" in v),
                   default=None)
        line["speedup_vs_reference_gpu"] = line["guided_tile_steps_per_s"] / best if best else None
    print(json.dumps(line), flush=True)
    del guided, plain
    main._solve_cache.clear()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--ref-steps", type=int, default=4, help="solver steps timed in the reference-GPU arm")
    ap.add_argument("--no-reference", action="store_true", help="skip the reference-GPU arm")
    ap.add_argument("--only", choices=["base-guided", "decoder-guided"], default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tools/bench_guided.py needs a CUDA device (B200); there is no CPU fallback")
    for workload, n in (("base-guided", 40), ("base-guided", 1), ("decoder-guided", 1), ("decoder-guided", 16)):
        if args.only in (None, workload):
            with torch.no_grad():
                run(workload, n, args)


if __name__ == "__main__":
    main()
