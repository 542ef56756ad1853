#!/usr/bin/env python
"""bench.py -- denoising steps/sec on 256x256 tiles of the 30m decoder U-Net (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-gpu] [--tiles B] [--size S]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One *step* = one decoder U-Net forward + one DPM-Solver++ update on the batch of tiles a GPU holds (default: ONE
256x256 tile per GPU = BASELINE configs[1]).  Steps come in 20-step solves (each solve starts from fresh noise, the
steps inside a solve are data-dependent).  `value` = tile-steps/s over all ranks with inputs resident in HBM;
`e2e` = the same through the public API (sample_decoder_diffusion_tiled) with pinned-host inputs and a D2H read of
every solve's result.  Weights are seeded synthetic (no checkpoints offline); data is synthetic.

--impl reference times the reference's own algorithm on the host CPU cores (the oracle port, fp32, all threads) --
rank 0 only, bounded number of steps.  --impl reference-gpu: the same algorithm through PyTorch library kernels on the
GPU (bf16 eager and torch.compile), the stated kernel to beat.

Other workloads (not the driver's line): --workload canvas|export strong-scales ONE blended canvas over the ranks
(BASELINE configs[2] / configs[3]-shaped); --workload latent = the latent consistency stage (253 M base U-Net, batches of
64^2 tiles; SURVEY 8(f) rank 1); --workload world = the reference's TTFT / TTST latency harness (evaluation/latency.py)
through the drop-in WorldPipeline.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

METRIC = "denoising steps/sec, 256^2 latent tiles, 30m U-Net"
UNIT = "tile-steps/s"
SOLVE_STEPS = 20
GFLOP_PER_STEP_256 = 343.94  # dense conv + linear FLOPs of one decoder forward at 256x256 (BASELINE.md section 2)


def igemm_gflop(size: int) -> float:
    """FLOPs executed by the tcgen05 implicit-GEMM launches in one forward (everything except first/last conv, linears)."""
    # BASELINE.md Appendix F: 6->64 first conv 0.453, 64->1 last conv 0.075, linears 0.003 at 256^2
    return (GFLOP_PER_STEP_256 - 0.453 - 0.075 - 0.003) * (size / 256.0) ** 2


DUMP_LIMIT_BYTES = 60 << 20     # all arrays of one dump, so the files (with their .npy headers) stay under 64 MB


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each tensor as <out_dir>/<name>.npy in float32, so two builds run with the same arguments (hence the same
    seeded inputs) can be compared output for output.  A tensor larger than its share of DUMP_LIMIT_BYTES is stored as
    every k-th element of its flattened form, the smallest k that fits: the same elements on every run."""
    import numpy as np
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    limit = DUMP_LIMIT_BYTES // len(arrays)
    for name, t in arrays.items():
        t = t.detach().float()
        stride = -(-t.numel() * 4 // limit)
        if stride > 1:
            t = t.reshape(-1)[::stride]
        np.save(d / f"{name}.npy", t.cpu().numpy())


# ----------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Polls NVML during the timed region (SM clock, throttle reasons)."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz, self.ok = [], set(), None, False
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        if self.ok:
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.ok:
            self.t.join(timeout=1.0)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ----------------------------------------------------------------------------------------------------- CPU arm
def usable_cores() -> int:
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:  # cgroup v2 CPU quota
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return n


_BEST_THREADS = None


def best_cpu_threads() -> int:
    """Give the CPU arm its best shot: time one 64x64 forward at several thread counts (all usable cores included)
    and keep the fastest -- torch's CPU convolutions do not scale to every core of a many-core host."""
    global _BEST_THREADS
    if _BEST_THREADS is None:
        from oracle import unet as ounet
        cfg = ounet.DECODER_CFG
        sd = ounet.procedural_state_dict(cfg, seed=0)
        x = torch.randn(1, 5, 64, 64)
        t = torch.tensor([1.0])
        cores = usable_cores()
        cands = sorted({c for c in (4, 8, 16, 32, 64, cores) if c <= cores})
        best, best_t = cands[0], float("inf")
        for c in cands:
            torch.set_num_threads(c)
            with torch.no_grad():
                ounet.unet_forward(sd, cfg, x, t, [])
                t0 = time.perf_counter()
                ounet.unet_forward(sd, cfg, x, t, [])
                dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = c, dt
        _BEST_THREADS = best
    return _BEST_THREADS


def cpu_steps(size: int, n_steps: int, budget_s: float):
    """The reference's algorithm (oracle port, fp32, best thread count): forward + scheduler.step per step.
    Returns (executed_steps, seconds)."""
    from oracle import scheduler as osched
    from oracle import unet as ounet
    torch.set_num_threads(best_cpu_threads())
    cfg = ounet.DECODER_CFG
    sd = ounet.procedural_state_dict(cfg, seed=0)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 1, size, size, generator=g) * 80
    cond = torch.randn(1, 4, size, size, generator=g)
    sch = osched.OracleScheduler()
    sch.set_timesteps(SOLVE_STEPS)
    done, t0 = 0, time.perf_counter()
    with torch.no_grad():
        for t, sigma in zip(sch.timesteps, sch.sigmas):
            if done >= n_steps or (done >= 1 and time.perf_counter() - t0 > budget_s):
                break
            scaled = sch.precondition_inputs(x, sigma)
            mo = ounet.unet_forward(sd, cfg, torch.cat([scaled, cond], dim=1),
                                    sch.trigflow_precondition_noise(sigma.view(-1)), [])
            x = sch.step(mo, t, x)
            done += 1
    return done, time.perf_counter() - t0


def run_reference_arm(args, rank):
    if rank != 0:
        return
    cores = best_cpu_threads()
    cpu_steps(args.size, min(args.warmup, 2), 30.0)  # warm-up (thread pools, allocator)
    want = args.steps
    done, secs = cpu_steps(args.size, min(want, SOLVE_STEPS), 90.0)
    value = done / secs
    sample = f"{done} of {want} requested steps of one {args.size}x{args.size} tile (20-step schedule), fp32, {cores} threads (best of a sweep up to {usable_cores()} usable cores)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 / value, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"configs[1]: 30m decoder U-Net, one {args.size}x{args.size} tile, 20-step DPM-Solver++ "
                               "(reference algorithm, oracle port on host CPU)", "tile": args.size,
                   "solve_steps": SOLVE_STEPS},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------- GPU reference
def run_reference_gpu_arm(args, rank):
    """The stated "kernel to beat" (SURVEY 8(d), BASELINE.md section 4): the reference algorithm itself on the same B200
    through PyTorch library kernels -- bf16 eager (cuDNN / cuBLAS / ATen elementwise, weight re-normalisation every
    forward, like WorldPipeline with dtype='bf16') and under torch.compile (Inductor, world_pipeline.py:421-430).  The
    reference tree cannot travel to the GPU box, so the model is its oracle restatement (bit-compatible in fp32 with the
    reference, tests/test_oracle_golden.py) moved to the device; comparison arm only, never the default."""
    if rank != 0:
        return
    from oracle import scheduler as osched
    from oracle import unet as ounet
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    cfg = ounet.DECODER_CFG
    B, S = args.tiles, args.size
    sd = {k: v.to(dev) for k, v in ounet.procedural_state_dict(cfg, seed=0).items()}
    g = torch.Generator().manual_seed(1)
    noise = (torch.randn(B, 1, S, S, generator=g) * 80).to(dev)
    cond = torch.randn(B, 4, S, S, generator=g).to(dev).bfloat16()

    def fwd(x, t):
        return ounet.unet_forward(sd, cfg, x, t, [])

    results = {}
    variants = [("eager_bf16", fwd)]
    try:
        variants.append(("compile_bf16", torch.compile(fwd)))
    except Exception as e:  # pragma: no cover
        results["compile_bf16"] = {"unavailable": repr(e)[:200]}
    for name, f in variants:
        try:
            def solve(n_steps):
                sch = osched.OracleScheduler()
                sch.set_timesteps(SOLVE_STEPS)
                sch.sigmas, sch.timesteps = sch.sigmas.to(dev), sch.timesteps.to(dev)
                x = noise.clone()
                for i, (t, sigma) in enumerate(zip(sch.timesteps, sch.sigmas)):
                    if i >= n_steps:
                        break
                    scaled = sch.precondition_inputs(x, sigma).bfloat16()
                    lab = sch.trigflow_precondition_noise(sigma.view(-1)).expand(B).bfloat16()
                    mo = f(torch.cat([scaled, cond], dim=1), lab).float()
                    sch.step_index = i                      # no .item() sync inside the timed loop
                    x = sch.step(mo, t, x)
                return x
            with torch.no_grad():
                solve(max(args.warmup, 3))
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                done = 0
                e0.record()
                while done < args.steps:
                    n = min(SOLVE_STEPS, args.steps - done)
                    solve(n)
                    done += n
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            results[name] = {"value": B * args.steps / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / args.steps}
        except Exception as e:  # pragma: no cover
            results[name] = {"unavailable": repr(e)[:300]}
    best = max((r["value"] for r in results.values() if "value" in r), default=None)
    line = {"impl": "reference-gpu", "metric": METRIC, "value": best, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": (1e3 * B / best) if best else None, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"configs[1]: 30m decoder U-Net, {B} x {S}x{S} tile, 20-step DPM-Solver++ -- the "
                                   "reference algorithm (oracle restatement) through PyTorch library kernels on the GPU",
                       "tiles_per_gpu": B, "tile": S, "solve_steps": SOLVE_STEPS},
            "variants": results, "gpu_launches": 0,
            "note": "comparison arm (the stated kernel to beat), PyTorch/cuDNN/Inductor kernels; not the product"}
    print(json.dumps(line), flush=True)


def run_reference_gpu_latent(args, rank):
    """--impl reference-gpu --workload latent: the latent consistency stage's arithmetic (base U-Net forward on a batch of
    64^2 tiles + TrigFlow update, world_pipeline.py:1097-1128) through PyTorch library kernels, bf16 eager and
    torch.compile -- the kernel to beat for SURVEY 8(f)-1."""
    if rank != 0:
        return
    import math
    from oracle import unet as ounet
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    B = args.tiles if args.tiles > 1 else 16
    T, sdat = 64, 0.5
    t0 = math.atan(80.0 / sdat)
    sd = {k: v.to(dev) for k, v in ounet.procedural_state_dict(BASE_CFG, seed=0).items()}
    g = torch.Generator().manual_seed(3)
    z = torch.randn(B, 5, T, T, generator=g).to(dev)
    cvec = torch.randn(B, 58, generator=g).to(dev).bfloat16()
    lab = torch.full((B,), t0, device=dev).bfloat16()

    def fwd(x, t, c):
        return ounet.unet_forward(sd, BASE_CFG, x, t, [c])

    results = {}
    variants = [("eager_bf16", fwd)]
    try:
        variants.append(("compile_bf16", torch.compile(fwd)))
    except Exception as e:  # pragma: no cover
        results["compile_bf16"] = {"unavailable": repr(e)[:200]}
    for name, f in variants:
        try:
            def phase():
                x_t = math.sin(t0) * sdat * z                       # first phase: s = 0
                pred = -f((x_t / sdat).bfloat16(), lab, cvec).float()
                return (math.cos(t0) * x_t - math.sin(t0) * sdat * pred) / sdat
            with torch.no_grad():
                for _ in range(max(args.warmup, 3)):
                    phase()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    phase()
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            results[name] = {"value": B * args.steps / (ms / 1e3), "unit": "tile-phases/s", "ms_per_step": ms / args.steps}
        except Exception as e:  # pragma: no cover
            results[name] = {"unavailable": repr(e)[:300]}
    best = max((r["value"] for r in results.values() if "value" in r), default=None)
    print(json.dumps({"impl": "reference-gpu", "metric": "latent-stage tile-phases/sec, 64^2 latent tiles, base 253M U-Net",
                      "value": best, "unit": "tile-phases/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                      "higher_is_better": True, "dtype": "bf16", "data": "synthetic",
                      "config": {"workload": f"base U-Net, {B} x 64x64 latent tiles, one consistency phase per step -- the "
                                             "reference algorithm (oracle restatement) through PyTorch library kernels"},
                      "variants": results, "gpu_launches": 0,
                      "note": "comparison arm (the kernel to beat), not the product"}), flush=True)


# ----------------------------------------------------------------------------------------------------- canvas arm
CANVASES = {
    # BASELINE configs[2]: 4 x 4 = 16 overlapping 512-px tiles at stride 384 (training/evaluation/__init__.py:16-22 gives
    # starts [0, 384, 768, 1152] for 1664 px; "2048 px" in BASELINE.json is not reachable with the reference's strides)
    "canvas": dict(size=1664, tile=512, stride=384, name="configs[2]: 1664^2 canvas, 4x4 tiles of 512 @ stride 384"),
    # configs[3]-shaped export canvas: 24 x 24 = 576 tiles (9344^2 px); 8192^2 itself gives 21 (bounded) or 23 (window
    # indexing) tile rows, neither of which stripes evenly over 8 GPUs
    "export": dict(size=9344, tile=512, stride=384, name="configs[3]-shaped: 9344^2 canvas, 24x24 tiles of 512 @ stride 384"),
}


def run_canvas_arm(args, rank, local_rank, world):
    """Strong scaling of ONE canvas: tile rows striped over the ranks, overlap strips exchanged with the neighbours
    while the interior tiles are solved (inference/sharded.py), result bit-identical to the single-GPU canvas."""
    import torch.distributed as dist
    from terrain_diffusion_b200.inference import sample_decoder_diffusion_sharded
    from terrain_diffusion_b200.inference.sharded import ShardedCanvas
    from terrain_diffusion_b200.models import EDMUnet2D
    from terrain_diffusion_b200.scheduler import EDMDPMSolverMultistepScheduler
    from oracle import unet as ounet
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29533")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    else:
        dist.init_process_group("gloo", rank=0, world_size=1)      # ShardedCanvas speaks torch.distributed
    cv = CANVASES[args.workload]
    H, T, S_ = cv["size"], cv["tile"], cv["stride"]
    cfg = ounet.DECODER_CFG
    model = EDMUnet2D(**cfg).eval()
    model.load_state_dict(ounet.procedural_state_dict(cfg, seed=0))
    model = model.to(dev)
    sched = EDMDPMSolverMultistepScheduler()
    g = torch.Generator().manual_seed(5)                            # every rank holds the same input canvas
    noise = (torch.randn(1, 1, H, H, generator=g) * 80).to(dev)
    cond = torch.randn(1, 4, H, H, generator=g).to(dev)
    steps = args.solve_steps
    probe = ShardedCanvas(1, H, H, T, S_, dev)
    n_tiles = len(probe.row_starts) * len(probe.col_starts)
    halo = (probe._strip_rows() + probe._upper_rows()) * H * 2 * 4
    del probe

    def solve():
        return sample_decoder_diffusion_sharded(model, sched, cond, noise, T, S_, num_steps=steps,
                                                tile_batch=args.tile_batch)
    solve()                                                         # warm-up: plans, graphs, NCCL connections
    torch.cuda.synchronize()
    reps = max(1, -(-args.steps // steps))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    with ClockSampler(local_rank) as clk:
        e0.record()
        for _ in range(reps):
            own, (lo, hi) = solve()
        e1.record()
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms = float(t_ms.item())
    value = n_tiles * steps * reps / (ms / 1e3)
    if rank == 0:
        line = {"metric": METRIC.replace("256^2", f"{T}^2"), "value": value, "unit": UNIT, "n_gpus": world,
                "steps": reps * steps, "warmup": steps, "ms_per_step": ms / (reps * steps), "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"{cv['name']}, {steps}-step solves per tile, blended; rows striped over "
                                       f"{world} GPU(s) with neighbour strip exchange", "canvas": H, "tile": T,
                           "stride": S_, "tiles": n_tiles, "solve_steps": steps, "tile_batch": args.tile_batch,
                           "halo_bytes_per_rank_per_solve": halo, "parallelism": f"tile-row stripes x{world}",
                           "l2": "every tile solve streams > 1 GB of activations (> 126 MB L2)"},
                "clocks": clk.summary(), "tflops": value * GFLOP_PER_STEP_256 * (T / 256.0) ** 2 / 1e3,
                "owned_rows": [lo, hi]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
    dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------- latent arm
BASE_CFG = dict(image_size=512, in_channels=5, out_channels=5, model_channels=192, model_channel_mults=[1, 2, 3, 4],
                layers_per_block=3, attn_resolutions=[8, 16], midblock_attention=True, concat_balance=0.5,
                conditional_inputs=[["tensor", 58, 1.0]], fourier_scale="pos", block_kwargs={"dropout": 0.1})
"""configs/diffusion_base/diffusion_192-3.cfg:54-69 (253.7 M parameters; self-attention at 8^2 / 16^2)."""
GFLOP_PER_LATENT_PHASE = 193.65   # one base-model forward on a 64^2 latent tile (SURVEY.md 8(d))


def run_latent_arm(args, rank, local_rank, world):
    """SURVEY 8(f) rank 1: the latent consistency stage (world_pipeline.py:1052-1131) -- one TrigFlow phase of the 253 M
    base U-Net (58-dim conditioning vector, self-attention) on batches of 64^2 latent tiles.  A step = one phase of one
    tile; `value` with the batch resident, `e2e` through `latent_stage_tiles` (host coarse windows in, packed tiles back
    to the host, tile noise generated on the device), which is what the pipeline's stage callback runs."""
    import math
    import torch.distributed as dist
    from terrain_diffusion_b200.inference.samplers import get_consistency_solve
    from terrain_diffusion_b200.inference.stages import latent_stage_tiles
    from terrain_diffusion_b200.inference.tiling import linear_weight_window
    from terrain_diffusion_b200.models import EDMUnet2D
    from oracle import unet as ounet
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    model = EDMUnet2D(**BASE_CFG).eval()
    model.load_state_dict(ounet.procedural_state_dict(BASE_CFG, seed=0))
    model = model.to(dev)
    B = args.tiles if args.tiles > 1 else 16                       # the product batches 16 windows (latents_batch_size)
    T, sd = 64, 0.5
    t_init = math.atan(80.0 / sd)
    g = torch.Generator().manual_seed(3 + rank)
    z = torch.randn(B, 5, T, T, generator=g).to(dev)
    cvec = torch.randn(B, 58, generator=g).to(dev)
    solve = get_consistency_solve(model, B, T, T, t_init, sd, from_unit_noise=True, out_scale=1.0 / sd)
    solve.prog.instantiate()
    for _ in range(max(3, args.warmup)):
        solve.run(z, None, conditional_inputs=[cvec])
    torch.cuda.synchronize()
    flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device=dev)
    flush.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    with ClockSampler(local_rank) as clk:
        e0.record()
        for _ in range(args.steps):
            solve.run(z, None, conditional_inputs=[cvec])
        e1.record()
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms = float(t_ms.item())
    value = world * B * args.steps / (ms / 1e3)
    # e2e: the stage callback with host inputs / host outputs
    ww = linear_weight_window(T, dev)
    ctxs = [(0, i // 4, i % 4) for i in range(B)]
    coarse_h = [torch.cat([torch.randn(6, 4, 4, generator=g), torch.ones(1, 4, 4)]).pin_memory() for _ in range(B)]
    hist = torch.zeros(1, 5)
    means, stds = torch.zeros(7), torch.ones(7)
    out_h = torch.empty(B, 6, T, T).pin_memory()

    def stage():
        tiles = latent_stage_tiles(model, 1234, ctxs, None, coarse_h, t_init, ww, hist, means, stds, pad_batch_to=16)
        out_h.copy_(torch.stack(tiles), non_blocking=True)
        torch.cuda.synchronize()
    e2e_value, e2e_err = None, None
    try:
        stage()
        n_e = 5
        t0 = time.perf_counter()
        for _ in range(n_e):
            stage()
        e2e_value = world * B * n_e / (time.perf_counter() - t0)
    except Exception as exc:                                       # the kernel-only number stands on its own
        e2e_err = repr(exc)
    roof = None
    if rank == 0:
        solve.run(z, None, conditional_inputs=[cvec])
        solve.prog.profile()
        msl, kinds = solve.prog.profile()
        ig_ms = sum(m for m, k in zip(msl, kinds) if k == 1)
        n_ig = sum(1 for k in kinds if k == 1)
        share = ig_ms / sum(msl)
        step_ms = ms / args.steps
        flops = GFLOP_PER_LATENT_PHASE * 1e9 * B
        achieved = flops / (step_ms * share / 1e3) / 1e12
        peak = 1400.0
        try:
            peak = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()).get("bf16_tflops_sustained") or peak
        except Exception:
            pass
        roof = {"bound": "tensor", "kernel": "tdx::igemm_kernel (tcgen05 implicit-GEMM conv)", "achieved": achieved,
                "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None, "launches": n_ig,
                "kernel_share_of_step": share, "avg_launch_us": step_ms * share / n_ig * 1e3,
                "method": "as the default arm: per-launch CUDA events give the share, x graph-replayed step time"}
        line = {"metric": "latent-stage tile-phases/sec, 64^2 latent tiles, base 253M U-Net", "value": value,
                "unit": "tile-phases/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"SURVEY 8(f)-1: base U-Net (253.7M params, self-attention, 58-dim conditioning), "
                                       f"{B} x 64x64 latent tiles per launch, one TrigFlow consistency phase per step",
                           "tiles_per_gpu": B, "tile": T, "parallelism": f"tiles x{world}",
                           "l2": "L2 flushed before the timed region; 507 MB of bf16 weights + the activation arena "
                                 "stream through L2 every phase",
                           "gflop_per_tile_phase": GFLOP_PER_LATENT_PHASE},
                "clocks": clk.summary(),
                "e2e": {"value": e2e_value, "unit": "tile-phases/s", "h2d_bytes_per_step": 7 * 16 * 4,
                        "d2h_bytes_per_step": 6 * T * T * 4, "error": e2e_err,
                        "api": "terrain_diffusion_b200.inference.stages.latent_stage_tiles"},
                "gpu_launches": solve.launches_per_solve * args.steps, "roofline": roof,
                "tflops": value * GFLOP_PER_LATENT_PHASE / 1e3}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------- world arm
COARSE_CFG = dict(image_size=16, in_channels=11, out_channels=6, model_channels=128, model_channel_mults=[1],
                  layers_per_block=2, attn_resolutions=[], midblock_attention=False, concat_balance=0.5,
                  conditional_inputs=[["float", 64, 0.2]] * 5, fourier_scale="pos", block_kwargs={})
"""configs/diffusion_coarse/diffusion_coarse.cfg:50-62."""


def run_world_arm(args, rank, local_rank, world):
    """The reference's own latency harness (evaluation/latency.py:19-127) through the drop-in `WorldPipeline`: TTFT = the
    first `get(i, j, i + 512, j + 512)` at a location far from everything computed before (coarse 20-step windows, two
    latent phases in batches of up to 16, 1-step decoder windows 512 @ stride 384, read-out, D2H); TTST = the adjacent
    tile.  Synthetic conditioning (no rasters), seeded random weights; plans / graphs are built by the warm-up get as in
    the reference (its torch.compile warm-up).  Runs on rank 0 only (a latency, not a throughput)."""
    import random
    from terrain_diffusion_b200.inference import WorldPipeline
    from terrain_diffusion_b200.models import EDMUnet2D
    from oracle import unet as ounet
    if rank != 0:
        return
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    def build(cfg):
        m = EDMUnet2D(**cfg).eval()
        m.load_state_dict(ounet.procedural_state_dict(cfg, seed=0))
        return m

    def cond_fn(i1, i2, j1, j2):
        gg = torch.Generator().manual_seed((i1 * 7919 + j1 + 12345) & 0x7FFFFFFF)
        return torch.randn(5, i2 - i1, j2 - j1, generator=gg)

    tile = args.size if args.size != 256 else 512
    pipe = WorldPipeline.from_local_models(build(COARSE_CFG), build(BASE_CFG), build(ounet.DECODER_CFG), seed=42,
                                           latents_batch_size=[1, 2, 4, 8, 16], torch_compile=True, dtype="bf16",
                                           caching_strategy="direct", cache_limit=None, decoder_tile_size=512,
                                           decoder_tile_stride=384, conditioning_fn=cond_fn)
    pipe.to(dev)
    pipe.bind("TEMP")
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    pipe.get(0, 0, tile, tile, with_climate=False)                 # warm-up: plans, graphs, folded weights
    torch.cuda.synchronize()
    warm_s = time.perf_counter() - t0
    sep = 100_000
    rnd = random.Random(7)
    for k in range(max(0, args.warmup)):                           # further untimed gets: the other padded batch sizes
        wi, wj = -(k + 1) * sep + rnd.randint(0, sep // 10), rnd.randint(0, sep)
        pipe.get(wi, wj, wi + tile, wj + tile, with_climate=False)
        pipe.empty_cache()
    torch.cuda.synchronize()
    ttft, ttst = [], []
    runs = max(1, args.steps)
    with ClockSampler(local_rank) as clk:
        for run in range(runs):
            bi = (run + 1) * sep + rnd.randint(0, sep // 10)
            bj = rnd.randint(0, sep)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pipe.get(bi, bj, bi + tile, bj + tile, with_climate=False)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            pipe.get(bi, bj + tile, bi + tile, bj + 2 * tile, with_climate=False)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            ttft.append(t1 - t0)
            ttst.append(t2 - t1)
            pipe.empty_cache()

    def pct(v, q):
        s_ = sorted(v)
        return s_[int((len(s_) - 1) * q / 100 + 0.5)]
    mean = sum(ttft) / len(ttft)
    line = {"metric": "TTFT: seconds to the first 512^2 WorldPipeline.get() at a cold location", "value": mean,
            "unit": "s", "n_gpus": 1, "steps": runs, "warmup": 1 + max(0, args.warmup), "ms_per_step": mean * 1e3, "higher_is_better": False,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "evaluation/latency.py harness: WorldPipeline (coarse 2.8M / base 253M / decoder 27.9M, "
                                   "seeded random weights, synthetic conditioning), get() of one 512^2 tile far from "
                                   "the cache (TTFT) and of its neighbour (TTST), decoder windows 512 @ 384, latent "
                                   "batches <= 16", "tile": tile, "runs": runs},
            "ttft": {"mean": mean, "p5": pct(ttft, 5), "p50": pct(ttft, 50), "p95": pct(ttft, 95)},
            "ttst": {"mean": sum(ttst) / len(ttst), "p5": pct(ttst, 5), "p50": pct(ttst, 50), "p95": pct(ttst, 95)},
            "first_get_with_plan_building_s": warm_s,
            "peak_vram_mb": torch.cuda.max_memory_allocated() / 2 ** 20,
            "clocks": clk.summary(),
            "e2e": {"value": mean, "unit": "s", "h2d_bytes_per_step": None, "d2h_bytes_per_step": tile * tile * 4,
                    "api": "terrain_diffusion_b200.inference.WorldPipeline.get"}}
    print(json.dumps(line), flush=True)
    pipe.close()


# ----------------------------------------------------------------------------------------------------- our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--tiles", type=int, default=1, help="independent tiles solved together per GPU")
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="tiles", choices=["tiles", "canvas", "export", "latent", "world"],
                    help="tiles (default, the BASELINE metric: independent 256^2 tiles per GPU, weak scaling) | canvas "
                         "(configs[2]: one 1664^2 canvas, strong scaling) | export (configs[3]-shaped 9344^2 canvas)")
    ap.add_argument("--solve-steps", type=int, default=SOLVE_STEPS, help="denoising steps per tile (canvas workloads)")
    ap.add_argument("--tile-batch", type=int, default=4, help="tiles solved together per launch (canvas workloads)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the denoised tiles of the last timed step (rank 0) as "
                         "DIR/sample.npy, float32 [tiles, 1, size, size]; a strided sample if above 60 MiB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "tiles"):
        ap.error("--dump-outputs is implemented for the default arm (--impl ours --workload tiles)")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if args.impl == "reference-gpu":
        if args.workload == "latent":
            run_reference_gpu_latent(args, rank)
        else:
            run_reference_gpu_arm(args, rank)
        return
    if args.workload == "latent":
        run_latent_arm(args, rank, local_rank, world)
        return
    if args.workload == "world":
        run_world_arm(args, rank, local_rank, world)
        return
    if args.workload != "tiles":
        run_canvas_arm(args, rank, local_rank, world)
        return

    import torch.distributed as dist
    from terrain_diffusion_b200.inference import sample_decoder_diffusion_tiled
    from terrain_diffusion_b200.inference.samplers import get_diffusion_solve
    from terrain_diffusion_b200.models import EDMUnet2D
    from terrain_diffusion_b200.scheduler import EDMDPMSolverMultistepScheduler
    from oracle import unet as ounet  # only for the config dict / seeded synthetic weights and the cpu_baseline leg

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    cfg = ounet.DECODER_CFG
    model = EDMUnet2D(**cfg).eval()
    model.load_state_dict(ounet.procedural_state_dict(cfg, seed=0))
    model = model.to(dev)
    sched = EDMDPMSolverMultistepScheduler()
    B, S = args.tiles, args.size

    g = torch.Generator().manual_seed(1 + rank)
    noise_h = (torch.randn(B, 1, S, S, generator=g) * 80).pin_memory()
    cond_h = torch.randn(B, 4, S, S, generator=g).pin_memory()
    noise_d, cond_d = noise_h.to(dev), cond_h.to(dev)

    def make_solves(k):
        full, rem = divmod(k, SOLVE_STEPS)
        plan = [SOLVE_STEPS] * full + ([rem] if rem else [])
        solves = {n: get_diffusion_solve(model, sched, B, S, S, n) for n in set(plan)}
        for s in solves.values():
            s.prog.instantiate()
        return plan, solves

    def run_plan(plan, solves):
        out = None
        for n in plan:
            out = solves[n].run(noise_d, cond_d)
        return out

    wplan, wsolves = make_solves(args.warmup)
    plan, solves = make_solves(args.steps)
    run_plan(wplan, wsolves)          # W untimed warm-up steps
    torch.cuda.synchronize()

    flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device=dev)
    flush.zero_()                      # evict L2 once; every step's working set then exceeds L2 by itself
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    with ClockSampler(local_rank) as clk:
        e0.record()
        last = run_plan(plan, solves)  # exactly K timed steps
        e1.record()
        torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        # `last` is the solver's state buffer: the e2e and roofline passes below overwrite it
        dump_outputs(args.dump_outputs, {"sample": last})
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    value = world * B * args.steps / (ms_max / 1e3)
    launches = sum(solves[n].launches_per_solve for n in plan)

    # ---------------- e2e: public API, pinned-host inputs, D2H result every solve
    n_solves = max(5, min(len(plan), 10))
    out_h = torch.empty(B, 1, S, S).pin_memory()
    sample_decoder_diffusion_tiled(model, sched, cond_d, noise_d, S, S, num_steps=SOLVE_STEPS)  # warm
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    per_solve = []
    for _ in range(n_solves):
        t0 = time.perf_counter()
        nz = noise_h.to(dev, non_blocking=True)
        cd = cond_h.to(dev, non_blocking=True)
        y = sample_decoder_diffusion_tiled(model, sched, cd, nz, S, S, num_steps=SOLVE_STEPS)
        out_h.copy_(y, non_blocking=True)
        torch.cuda.synchronize()
        per_solve.append(time.perf_counter() - t0)
    # the MEDIAN solve (host jitter of a shared box moves the mean by up to 10 %; the mean is reported beside it)
    e2e_s = sorted(per_solve)[len(per_solve) // 2]
    e2e_mean_s = sum(per_solve) / len(per_solve)
    t_e = torch.tensor([e2e_s, e2e_mean_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = world * B * SOLVE_STEPS / float(t_e[0].item())
    e2e_mean_value = world * B * SOLVE_STEPS / float(t_e[1].item())
    h2d = (noise_h.numel() + cond_h.numel()) * 4 / SOLVE_STEPS
    d2h = out_h.numel() * 4 / SOLVE_STEPS

    # ---------------- roofline of the dominant kernel (tcgen05 implicit GEMM): live per-launch CUDA events
    roof, cpu_base = None, None
    if rank == 0:
        s20 = get_diffusion_solve(model, sched, B, S, S, SOLVE_STEPS)
        s20.sample.copy_(noise_d)
        s20.x0_prev.zero_()
        s20.prog.profile()  # warm (eager)
        s20.sample.copy_(noise_d)
        s20.x0_prev.zero_()
        msl, kinds = s20.prog.profile()
        ig_ms = sum(m for m, k in zip(msl, kinds) if k == 1)
        n_ig = sum(1 for k in kinds if k == 1)
        tot_ms = sum(msl)
        flops = igemm_gflop(S) * 1e9 * B * SOLVE_STEPS
        share = ig_ms / tot_ms
        # Eager per-launch events include the host launch gap of every kernel (sum of parts > the graph replay), so the
        # kernel's duration inside the timed region = its SHARE of the step x the graph-replayed step time.
        step_ms = ms_max / args.steps
        ig_ms_in_graph = step_ms * SOLVE_STEPS * share
        achieved = flops / (ig_ms_in_graph / 1e3) / 1e12
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        peak = peaks.get("bf16_tflops_sustained")
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"
        if not peak:
            peak, peak_src = 1400.0, "fallback (B200_PROFILING.md sustained ~1.4 PFLOP/s)"
        traffic = None
        try:
            tj = json.loads((ROOT / "profiles" / "igemm_traffic.json").read_text())
            if tj.get("workload_tiles", 1) == args.tiles:   # the ncu capture is of the default (1-tile) workload
                traffic = tj.get("dram_bytes_per_launch")
        except Exception:
            pass
        roof = {"bound": "tensor", "kernel": "tdx::igemm_kernel (tcgen05 implicit-GEMM conv)", "achieved": achieved,
                "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "launches": n_ig,
                "avg_launch_us": ig_ms_in_graph / n_ig * 1e3,
                "avg_launch_us_eager_events": ig_ms / n_ig * 1e3,
                "kernel_share_of_step": share,
                "algorithmic_gflop_per_launch": flops / n_ig / 1e9,
                "method": "per-launch CUDA events (tdx_program_profile, eager) give the kernel's share of a step; "
                          "duration in the timed region = share x graph-replayed step time"}
        if world == 1 and not args.no_cpu_baseline:
            cores = best_cpu_threads()
            cpu_steps(S, 1, 60.0)
            done, secs = cpu_steps(S, 8, 25.0)
            cpu_base = {"value": done / secs, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"{done} steps of one {S}x{S} tile (oracle port of the reference algorithm, fp32, "
                                  f"{cores} threads = best of a sweep up to {usable_cores()} usable cores)"}

    if rank == 0:
        arena_mb = sum(t.numel() * t.element_size() for t in solves[plan[0]].prog.arena.values()) / 2 ** 20
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"configs[1]: 30m decoder U-Net (27.9M params), {B} x {S}x{S} tile per GPU, "
                                   f"{SOLVE_STEPS}-step DPM-Solver++ solves, bf16 tcgen05 / fp32 accumulate",
                       "tiles_per_gpu": B, "tile": S, "solve_steps": SOLVE_STEPS, "parallelism": f"tiles x{world}",
                       "l2": f"L2 flushed before the timed region; each step streams a {arena_mb:.0f} MiB activation "
                             "arena + 56 MiB weights (> 126 MB L2), steps are data-dependent so no flush between them",
                       "gflop_per_tile_step": GFLOP_PER_STEP_256 * (S / 256.0) ** 2},
            "clocks": clk.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "solves": n_solves, "stat": "median solve (each solve timed from H2D to the synchronised D2H)",
                    "value_from_mean": e2e_mean_value,
                    "api": "terrain_diffusion_b200.inference.sample_decoder_diffusion_tiled"},
            "gpu_launches": launches,
            "roofline": roof,
            "cpu_baseline": cpu_base,
            "tflops": value * GFLOP_PER_STEP_256 * (S / 256.0) ** 2 / 1e3,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
