"""Checkers for the text-to-image loop — TEST INFRASTRUCTURE ONLY, next to oracle/unet_oracle.py and oracle/unet_emul.py.

* `DPMSolverMultistepSchedulerOracle`: diffusers 0.9 DPMSolverMultistepScheduler (dpmsolver++, midpoint, order 2,
  lower_order_final) restated from SURVEY Appendix C [memory, unpinned], with the update in float64.
* `txt2img_loop`: StableDiffusionPipeline 0.9 `__call__`'s denoising loop with the initial latents injected, any
  scheduler with a diffusers `step(eps, t, x)` (this one or oracle.unet_oracle.PNDMSchedulerOracle).
* `txt2img_loop_emul`: the same loop with fp16 storage at the points where the B200 path stores fp16 (the UNet through
  oracle.unet_emul.unet_forward, each fp16 tensor op of the fused scheduler kernels rounded once).
"""
from __future__ import annotations

import typing as T

import numpy as np
import torch

from oracle import unet_emul as ue


def r16(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.float16).to(torch.float32)


class DPMSolverMultistepSchedulerOracle:
    def __init__(self, num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012):
        betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
        self.alphas_cumprod = torch.cumprod(1.0 - betas, dim=0)              # the model's fp32 table
        ac = self.alphas_cumprod.double()
        self.alpha_t, self.sigma_t = ac.sqrt(), (1 - ac).sqrt()
        self.lambda_t = self.alpha_t.log() - self.sigma_t.log()
        self.num_train_timesteps = num_train_timesteps
        self.timesteps: T.Optional[torch.Tensor] = None

    def set_timesteps(self, n: int):
        ts = np.linspace(0, self.num_train_timesteps - 1, n + 1).round()[::-1][:-1].copy().astype(np.int64)
        self.timesteps = torch.from_numpy(ts)
        self.model_outputs: T.List[T.Optional[torch.Tensor]] = [None, None]
        self.lower_order_nums = 0

    def step(self, model_output, timestep: int, sample):
        ts = self.timesteps.tolist()
        i = ts.index(int(timestep))
        t, s0 = (ts[i + 1] if i + 1 < len(ts) else 0), ts[i]
        dt = sample.dtype
        x = sample.double()
        m0 = (x - self.sigma_t[s0] * model_output.double()) / self.alpha_t[s0]
        self.model_outputs = [self.model_outputs[1], m0]
        lower_order_final = i == len(ts) - 1 and len(ts) < 15
        h = self.lambda_t[t] - self.lambda_t[s0]
        c0 = self.alpha_t[t] * (torch.exp(-h) - 1.0)
        x_t = (self.sigma_t[t] / self.sigma_t[s0]) * x - c0 * m0
        if not (self.lower_order_nums < 1 or lower_order_final):
            r0 = (self.lambda_t[s0] - self.lambda_t[ts[i - 1]]) / h
            x_t = x_t - 0.5 * c0 * (1.0 / r0) * (m0 - self.model_outputs[0])
        self.lower_order_nums = min(self.lower_order_nums + 1, 2)
        return x_t.to(dt)


def txt2img_loop(unet, scheduler, text, uncond, latents, steps: int, guidance: float):
    """diffusers 0.9 StableDiffusionPipeline.__call__ (CFG) from injected latents.  Returns (latents, UNet evaluations)."""
    scheduler.set_timesteps(steps)
    ctx = torch.cat([uncond.expand(text.shape[0], -1, -1), text])
    x, n = latents, 0
    for t in scheduler.timesteps:
        eps = unet(torch.cat([x, x]), int(t), ctx)
        n += 1
        eu, et = eps.chunk(2)
        x = scheduler.step(eu + guidance * (et - eu), int(t), x)
    return x, n


@torch.no_grad()
def txt2img_loop_emul(unet_module, scheduler: str, text, uncond, latents, steps: int, guidance: float):
    """`txt2img_loop` with fp16 storage where the B200 path stores fp16.  scheduler: "DPMSolverMultistepScheduler"
    (rf_cfg_dpmpp_step_f16: every fp16 tensor op of the reference's step rounded once, fp32 scalars computed as the
    reference computes them) or "PNDMScheduler" (rf_cfg_pndm_step_f16, as oracle.unet_emul.img2img_loop_emul)."""
    from riffusion.scheduler_b200 import get_scheduler

    s = get_scheduler(scheduler)            # host tables / scalars only; no device op is called
    s.set_timesteps(steps)
    ctx = torch.cat([uncond.expand(text.shape[0], -1, -1), text]).float()
    x = r16(latents.float())
    n, m1, ets, counter, cur_sample = 0, None, [], 0, None
    ratio = s.num_train_timesteps // steps
    for t in s.timesteps.tolist():
        eps = ue.unet_forward(unet_module, torch.cat([x, x]), t, ctx)
        n += 1
        eu, et = eps.chunk(2)
        e0 = r16(eu + r16(r16(et - eu) * guidance))
        if scheduler == "DPMSolverMultistepScheduler":
            c = s.coefficients(t)
            m0 = r16(r16(x - r16(c["sigma_s"] * e0)) * float(np.float32(1.0) / np.float32(c["alpha_s"])))
            xt = r16(r16(c["c_x"] * x) - r16(c["c_0"] * m0))
            if c["second"]:
                xt = r16(xt - r16(c["c_d1"] * r16(c["inv_r0"] * r16(m0 - m1))))
            s.lower_order_nums = min(s.lower_order_nums + 1, 2)
            x, m1 = xt, m0
            continue
        prev_t, cur_t = t - ratio, t
        if counter != 1:
            ets = ets[-3:] + [e0]
        else:
            prev_t, cur_t = t, t + ratio
        sample = x
        if len(ets) == 1 and counter == 0:
            e, cur_sample = e0, x
        elif len(ets) == 1 and counter == 1:
            e, sample, cur_sample = 0.5 * e0 + 0.5 * ets[-1], cur_sample, None
        elif len(ets) == 2:
            e = 1.5 * ets[-1] - 0.5 * ets[-2]
        elif len(ets) == 3:
            e = (23 / 12) * ets[-1] - (16 / 12) * ets[-2] + (5 / 12) * ets[-3]
        else:
            e = (55 / 24) * ets[-1] - (59 / 24) * ets[-2] + (37 / 24) * ets[-3] - (9 / 24) * ets[-4]
        ca, cb = s.coefficients(cur_t, prev_t)
        x = r16(ca * sample - cb * e)
        counter += 1
    return x, n
