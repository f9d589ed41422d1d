"""Checkers for the img2img loop — TEST INFRASTRUCTURE ONLY, next to tests/txt2img_oracle.py.

* `img2img_loop`: StableDiffusionImg2ImgPipeline 0.9 `__call__`'s denoising loop from injected noisy latents over
  timesteps[t_start:] (SURVEY Appendix D), any scheduler with a diffusers `step(eps, t, x)`.
* `img2img_loop_emul`: the same loop with fp16 storage where the B200 path stores fp16 (the UNet through
  oracle.unet_emul.unet_forward, each fp16 tensor op of the fused scheduler kernels rounded once), as
  txt2img_oracle.txt2img_loop_emul does for the whole timestep list.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import unet_emul as ue
from txt2img_oracle import r16


def img2img_loop(unet, scheduler, text, uncond, latents, steps: int, t_start: int, guidance: float):
    """Returns (latents, UNet evaluations).  The scheduler's multistep history starts empty at t_start."""
    scheduler.set_timesteps(steps)
    ctx = torch.cat([uncond.expand(text.shape[0], -1, -1), text])
    x, n = latents, 0
    for t in scheduler.timesteps[t_start:]:
        eps = unet(torch.cat([x, x]), int(t), ctx)
        n += 1
        eu, et = eps.chunk(2)
        x = scheduler.step(eu + guidance * (et - eu), int(t), x)
    return x, n


@torch.no_grad()
def img2img_loop_emul(unet_module, scheduler: str, text, uncond, latents, steps: int, t_start: int, guidance: float):
    from riffusion.scheduler_b200 import get_scheduler

    s = get_scheduler(scheduler)            # host tables / scalars only; no device op is called
    s.set_timesteps(steps)
    ctx = torch.cat([uncond.expand(text.shape[0], -1, -1), text]).float()
    x = r16(latents.float())
    n, m1, ets, counter, cur_sample = 0, None, [], 0, None
    ratio = s.num_train_timesteps // steps
    for t in s.timesteps.tolist()[t_start:]:
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
