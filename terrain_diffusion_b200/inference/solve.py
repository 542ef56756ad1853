"""Whole N-step tile solves as ONE CUDA graph.

The reference's per-tile loop (training/evaluation/sample_diffusion_decoder.py:105-120; world_pipeline.py:934-949)
runs, per step: precondition_inputs, trigflow_precondition_noise, cat, the U-Net, scheduler.step -- thousands of
launches and host-side scalar math.  Here the step sequence is planned once: the scaled-sample/cond concat is folded
into the first convolution, scheduler.step into the last one, and the per-step scalars (c_in, t, c_skip, c_out, r, k)
sit in a small device table, so a K-step solve of a batch of tiles is a single graph launch of ~80*K kernels.

Two-model autoguidance (EDM2; training/evaluation/sample_diffusion_base.py:105-110) records the guide's forward before
the main one in every step of the same graph: the guide's last convolution writes F_g, the main one combines
F = F_g + s*(F_m - F_g) before the update, with s read from the coefficient table.  Score scaling
(sample_diffusion_decoder.py:7-40) is linear in (x, F) and folds into c_skip / c_out (score_scaling_fold).
"""
from __future__ import annotations

import math

import torch

from ..models.plan import UNetEmitter, UNetProgram


def score_scaling_fold(row: dict, sigma_data: float, alpha: float) -> dict:
    """A coefficient row with the reference's _scale_score folded in.  _scale_score maps the model output to
    mo' = a*x + b*mo with, for t = atan(sigma / sigma_d) (the row's noise label), c = cos t, s = sin t:
        a = s*(1 - alpha)*(1 - c) / sigma_d ,  b = c^2 + alpha*s^2
    so x0 = c_skip*x + c_out*mo' = (c_skip + c_out*a)*x + (c_out*b)*mo.  fp64, like the row; alpha == 1 returns the
    row unchanged."""
    alpha = float(alpha)
    if alpha == 1.0:
        return dict(row)
    c, s = math.cos(row["t"]), math.sin(row["t"])
    a = s * (1.0 - alpha) * (1.0 - c) / sigma_data
    b = c * c + alpha * s * s
    return dict(row, c_skip=row["c_skip"] + row["c_out"] * a, c_out=row["c_out"] * b)


def check_guide(model, guide) -> None:
    """A guide must read and write what the model does: same in / out channels, same conditional inputs, same
    device.  Raises ValueError (before anything is planned or launched)."""
    mc, gc = model.config, guide.config
    io = lambda c: (int(c["in_channels"]), int(c.get("out_channels") or c["in_channels"]))
    if io(mc) != io(gc):
        raise ValueError(f"guide model has (in, out) channels {io(gc)}, the model {io(mc)}")
    kinds = lambda c: [(str(k), int(d)) for k, d, _w in (c.get("conditional_inputs") or [])]
    if kinds(mc) != kinds(gc):
        raise ValueError(f"guide model conditional inputs {kinds(gc)} differ from the model's {kinds(mc)}")
    if guide.device != model.device:
        raise ValueError(f"guide model is on {guide.device}, the model on {model.device}")


class DiffusionSolve:
    """K-step EDM DPM-Solver++ solve of `n` independent tiles: sample[n, Cs, h, w] (<- noise*sigma0), cond[n, Cc, h, w]."""

    def __init__(self, model, scheduler, n: int, h: int, w: int, num_steps: int, step_range=None, coef_rows=None,
                 guide=None, guidance_scale: float = 1.0, score_scaling: float = 1.0):
        """coef_rows: explicit per-step tables [dict(c_in, t, c_skip, c_out, r, k)] instead of a scheduler's (the
        TrigFlow consistency step is the same fused program with other numbers: consistency_rows()).
        step_range = (i0, i1): only steps i0 .. i1-1 of the `num_steps` schedule (one PHASE of a multi-phase
        InfiniteDiffusion solve, inference/multiphase.py).  A range that starts in the middle of the schedule starts
        from a blended canvas, so the multistep history is empty there: its first step is first order, exactly like
        a scheduler whose state was reset and positioned at step i0.
        guide, guidance_scale: two-model guidance mo = mo_g + s*(mo_m - mo_g), the guide evaluated on the same input
        in every step.  Without a guide or with s == 1 the program is the unguided one (the reference does not
        evaluate the guide then).  s sits in the coefficient table: set_guidance_scale() changes it without
        re-recording.  score_scaling: the reference's _scale_score alpha, folded into the coefficients (applied
        after guidance, as in the reference)."""
        self.guide = guide if (guide is not None and float(guidance_scale) != 1.0) else None
        if self.guide is not None:
            check_guide(model, self.guide)
        if float(score_scaling) != 1.0 and scheduler is None:
            raise ValueError("score_scaling needs the scheduler's sigma_data")
        fw = model.folded()
        dev = fw.device
        if coef_rows is not None:
            co = [dict(r) for r in coef_rows]
            self.schedule_steps, self.step_range = len(co), (0, len(co))
            num_steps = len(co)
        else:
            scheduler.set_timesteps(num_steps)
            order = scheduler.order_schedule()
            i0, i1 = (0, num_steps) if step_range is None else (int(step_range[0]), int(step_range[1]))
            if not (0 <= i0 < i1 <= num_steps):
                raise ValueError(f"step_range {step_range} is not inside the {num_steps}-step schedule")
            self.schedule_steps, self.step_range = num_steps, (i0, i1)
            co = [scheduler.step_coefficients(i, order[i] and not (i == i0 and i0 > 0)) for i in range(i0, i1)]
            num_steps = i1 - i0                  # from here on: the number of steps this solve runs
        if float(score_scaling) != 1.0:
            co = [score_scaling_fold(c, float(scheduler.config.sigma_data), score_scaling) for c in co]
        self.model, self.n, self.h, self.w, self.num_steps = model, n, h, w, num_steps
        cs = fw.out_channels
        cc = fw.in_channels - cs
        # {c_skip, c_out, r, k} per step, plus the guidance scale s as a 5th column when guided
        extra = [float(guidance_scale)] if self.guide is not None else []
        self.coef = torch.tensor([[c["c_skip"], c["c_out"], c["r"], c["k"]] + extra for c in co],
                                 dtype=torch.float64).to(torch.float32).to(dev).contiguous()
        self.c_in = torch.tensor([c["c_in"] for c in co], dtype=torch.float64).to(torch.float32).to(dev).contiguous()
        self.labels = torch.tensor([[c["t"]] * n for c in co], dtype=torch.float64).to(torch.float32).to(
            dev).contiguous()
        self.sample = torch.zeros((n, cs, h, w), dtype=torch.float32, device=dev)
        self.cond = torch.zeros((n, max(cc, 1), h, w), dtype=torch.float32, device=dev)
        self.x0_prev = torch.zeros_like(self.sample)
        self.prog = UNetProgram(fw.device)
        # the noise labels of all steps are known up front: ONE embed launch produces every step's modulation vectors
        em = UNetEmitter(fw, n, h, w, cvec_sets=num_steps)
        self.host_emb = len(model.conditional_layers) > 0 or not fw.pos_emb
        if self.host_emb:
            # conditional models (coarse: five float conditions): the 256-wide embeddings of all steps are computed
            # by host torch ops per run() and handed to the embed launch
            self.emb_all = torch.zeros((num_steps * n, fw.emb_channels), dtype=torch.float32, device=dev)
            em.emit_embed(self.prog, emb_in=self.emb_all)
        else:
            em.emit_embed(self.prog, labels=self.labels.reshape(-1))
        gem, self.guide_out, self.guide_host_emb = None, None, False
        if self.guide is not None:
            # the guide: its own arena and modulation vectors; its last convolution writes F_g (plain model_out mode)
            gw = self.guide.folded()
            gem = UNetEmitter(gw, n, h, w, cvec_sets=num_steps)
            self.guide_out = torch.zeros_like(self.sample)
            self.guide_host_emb = len(self.guide.conditional_layers) > 0 or not gw.pos_emb
            if self.guide_host_emb:
                self.guide_emb_all = torch.zeros((num_steps * n, gw.emb_channels), dtype=torch.float32, device=dev)
                gem.emit_embed(self.prog, emb_in=self.guide_emb_all)
            else:
                gem.emit_embed(self.prog, labels=self.labels.reshape(-1))
        for i in range(num_steps):
            srcs = [(self.sample, cs, self.c_in[i:i + 1])]
            if cc > 0:
                srcs.append((self.cond, cc, None))
            sched = dict(coef=self.coef[i], sample=self.sample, x0_prev=self.x0_prev)
            if gem is not None:
                # before the main forward: the main last convolution updates `sample` in place
                gem.emit(self.prog, srcs, model_out=self.guide_out, cvec_set=i)
                sched["guide_out"] = self.guide_out
            em.emit(self.prog, srcs, model_out=None, sched=sched, cvec_set=i)
        self.launches_per_solve = self.prog.n_launch
        # sum of 2*M*N*K over the tensor-core launches of one solve, per model (the guide's share is its cost)
        self.igemm_flops = em.igemm_flops
        self.guide_igemm_flops = gem.igemm_flops if gem is not None else 0

    def set_guidance_scale(self, s: float) -> None:
        """Rewrite the guidance scale in the device table (stream-ordered; no re-recording of the program)."""
        if self.guide is None:
            raise ValueError("this solve was recorded without a guide (guide None or guidance_scale == 1)")
        self.coef[:, 4].fill_(float(s))

    @torch.no_grad()
    def run(self, noise: torch.Tensor, cond: torch.Tensor | None, use_graph: bool = True,
            conditional_inputs=None) -> torch.Tensor:
        """noise: [n, Cs, h, w] initial sample (already scaled by sigma_0); returns the denoised sample (a view of the
        solver's state buffer -- copy it before the next run)."""
        if self.host_emb or self.guide_host_emb:
            # conditional models: ONE batched evaluation of compute_embeddings for the labels of all steps (per model;
            # the guide gets the same conditional inputs)
            ci = [c.to(self.labels.device).repeat(self.num_steps, *([1] * (c.dim() - 1)))
                  for c in (conditional_inputs or [])]
            if self.host_emb:
                self.emb_all.copy_(self.model._host_embedding(self.labels.reshape(-1), ci))
            if self.guide_host_emb:
                self.guide_emb_all.copy_(self.guide._host_embedding(self.labels.reshape(-1), ci))
        self.sample.copy_(noise)
        if cond is not None:
            self.cond.copy_(cond)
        self.x0_prev.zero_()
        self.prog.run(use_graph)
        return self.sample


def consistency_rows(t: float, sigma_data: float = 0.5, from_unit_noise: bool = False, out_scale: float = 1.0):
    """Coefficient row that makes the fused step program a TrigFlow consistency step
    (world_pipeline.py:1097-1128,1235-1239):   model_in = x_t / sigma_d ;  s' = cos t * x_t + sin t * sigma_d * F
    (pred = -F).  from_unit_noise: the sample buffer holds the unit-variance noise z of a FIRST phase (s = 0, so
    x_t = sin t * sigma_d * z): the re-noising folds into the scalars and no mixing launch is needed.  out_scale
    multiplies the result (1 / sigma_d for a final phase)."""
    import math
    ct, st = math.cos(t), math.sin(t)
    s = st * sigma_data if from_unit_noise else 1.0
    return [dict(c_in=s / sigma_data, t=float(t), c_skip=ct * s * out_scale, c_out=st * sigma_data * out_scale, r=0.0,
                 k=0.0)]
