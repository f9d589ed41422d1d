"""PNDM (PLMS) and DPM-Solver++ schedulers for the denoising loop — host-side tables + one fused device step.

Restates diffusers 0.9 `PNDMScheduler(skip_prk_steps=True, steps_offset=1, beta_schedule="scaled_linear",
beta_start=0.00085, beta_end=0.012, set_alpha_to_one=False)` [memory; SURVEY Appendix B], i.e. the scheduler
`RiffusionPipeline.interpolate_img2img` drives at riffusion/riffusion_pipeline.py:314,361-365,379,392-396,403,418.
The scalar recurrences (alphas, timestep table, multistep weights) run on the host in fp32; the tensor update
runs in one kernel fused with the classifier-free-guidance combine (`rf_cfg_pndm_step_f16`).
"""
from __future__ import annotations

import types
import typing as T

import numpy as np
import torch

from riffusion import tc_ops as ops


class _Img2ImgMixin:
    """What diffusers 0.9 `StableDiffusionImg2ImgPipeline` asks of its scheduler [memory; SURVEY Appendix D]: the
    strength -> timestep arithmetic of `get_timesteps` and `add_noise` on fp16 latents.  Shared by both schedulers
    (`alphas_cumprod`, `timesteps`, `config` and `set_timesteps` come from the class)."""

    def img2img_timesteps(self, num_inference_steps: int, strength: float) -> T.Tuple[int, torch.Tensor, int]:
        """`set_timesteps(n)`, then `init_timestep = min(int(n * strength) + offset, n)`,
        `t_start = max(n - init_timestep + offset, 0)` with offset = config["steps_offset"].  Returns (t_start,
        timesteps[t_start:], the noise timestep timesteps[t_start]).  The multistep history starts empty at t_start."""
        if not 0.0 <= strength <= 1.0:
            raise ValueError(f"The value of strength should in [0.0, 1.0] but is {strength}")
        self.set_timesteps(num_inference_steps)
        offset = self.config.get("steps_offset", 0)
        init_timestep = min(int(num_inference_steps * strength) + offset, num_inference_steps)
        t_start = max(num_inference_steps - init_timestep + offset, 0)
        timesteps = self.timesteps[t_start:]
        if len(timesteps) == 0:
            raise ValueError(f"strength {strength} with {num_inference_steps} inference steps leaves no denoising step")
        return t_start, timesteps, int(timesteps[0])

    def add_noise_scalars(self, timestep: int) -> T.Tuple[float, float]:
        """(sqrt(a[t]), sqrt(1 - a[t])) as fp16 values: alphas_cumprod is cast to the sample dtype before the index, and
        `1 - a` and `** 0.5` are fp16 tensor ops (computed in fp32, rounded to fp16 once each)."""
        a = np.float16(self.alphas_cumprod[int(timestep)].item())
        s = np.float16(np.sqrt(np.float32(a)))
        s1 = np.float16(np.sqrt(np.float32(np.float16(np.float32(1.0) - np.float32(a)))))
        return float(s), float(s1)

    def add_noise_fp16(self, original: torch.Tensor, noise: torch.Tensor, timestep: int) -> torch.Tensor:
        """img2img's `add_noise` on fp16 latents: fp16(fp16(s x) + fp16(s1 noise)), every op rounded as torch rounds
        it (rf_add_noise_f16_seq).  `add_noise` above, which riffuse uses, rounds once and stays as it is."""
        s, s1 = self.add_noise_scalars(timestep)
        return ops.add_noise_f16_seq(original, noise, s, s1)


class PNDMSchedulerB200(_Img2ImgMixin):
    order = 1

    def __init__(self, num_train_timesteps: int = 1000, beta_start: float = 0.00085, beta_end: float = 0.012,
                 steps_offset: int = 1):
        betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
        self.alphas_cumprod = torch.cumprod(1.0 - betas, dim=0)
        self.final_alpha_cumprod = self.alphas_cumprod[0]
        self.num_train_timesteps = num_train_timesteps
        self.config = {"steps_offset": steps_offset, "num_train_timesteps": num_train_timesteps}
        self.init_noise_sigma = 1.0
        self.timesteps: T.Optional[torch.Tensor] = None
        self.set_timesteps(50)

    # -- schedule -------------------------------------------------------------------------------
    def set_timesteps(self, num_inference_steps: int, device=None) -> None:
        self.num_inference_steps = num_inference_steps
        ratio = self.num_train_timesteps // num_inference_steps
        base = (np.arange(0, num_inference_steps) * ratio).round() + self.config["steps_offset"]
        plms = np.concatenate([base[:-1], base[-2:-1], base[-1:]])[::-1].copy()      # 961 duplicated
        self.timesteps = torch.from_numpy(plms.astype(np.int64))
        self.ets: T.List[torch.Tensor] = []
        self.counter = 0
        self.cur_sample: T.Optional[torch.Tensor] = None

    def scale_model_input(self, sample: torch.Tensor, timestep=None) -> torch.Tensor:
        return sample

    def _alpha(self, t: int) -> float:
        return float(self.alphas_cumprod[t]) if t >= 0 else float(self.final_alpha_cumprod)

    def coefficients(self, timestep: int, prev_timestep: int) -> T.Tuple[float, float]:
        a_t, a_p = self._alpha(timestep), self._alpha(prev_timestep)
        b_t, b_p = 1.0 - a_t, 1.0 - a_p
        denom = a_t * b_p ** 0.5 + (a_t * b_t * a_p) ** 0.5
        return (a_p / a_t) ** 0.5, (a_p - a_t) / denom

    def add_noise(self, original: torch.Tensor, noise: torch.Tensor, timestep, mask=None, blend_with=None) -> torch.Tensor:
        a = float(self.alphas_cumprod[int(timestep)])
        return ops.axpby(original.contiguous(), noise.contiguous(), a ** 0.5, (1.0 - a) ** 0.5, mask, blend_with)

    # -- one multistep update ------------------------------------------------------------------------
    def plan(self, timestep: int):
        """Host bookkeeping of one PLMS step: returns (coef4, history tensors, sample_override, push, ca, cb)."""
        timestep = int(timestep)
        prev = timestep - self.num_train_timesteps // self.num_inference_steps
        push = self.counter != 1
        if not push:                                   # 2nd call: redo the first step from the saved sample
            prev, timestep = timestep, timestep + self.num_train_timesteps // self.num_inference_steps
        n_hist = len(self.ets[-3:]) + 1 if push else len(self.ets)
        override = None
        if n_hist == 1 and self.counter == 0:
            coef, hist = (1.0, 0.0, 0.0, 0.0), []
        elif n_hist == 1 and self.counter == 1:
            coef, hist, override = (0.5, 0.5, 0.0, 0.0), [self.ets[-1]], self.cur_sample
        elif n_hist == 2:
            coef, hist = (1.5, -0.5, 0.0, 0.0), [self.ets[-1]]
        elif n_hist == 3:
            coef, hist = (23 / 12, -16 / 12, 5 / 12, 0.0), [self.ets[-1], self.ets[-2]]
        else:
            coef, hist = (55 / 24, -59 / 24, 37 / 24, -9 / 24), [self.ets[-1], self.ets[-2], self.ets[-3]]
        ca, cb = self.coefficients(timestep, prev)
        return coef, hist, override, push, ca, cb

    def step_cfg(self, eps_pair: torch.Tensor, guidance: float, timestep: int, sample: torch.Tensor) -> torch.Tensor:
        """Guidance combine (riffusion_pipeline.py:411-415) + scheduler.step (:418) in one kernel.
        eps_pair = UNet output for [uncond | text]."""
        coef, hist, override, push, ca, cb = self.plan(timestep)
        if self.counter == 0:
            self.cur_sample = sample
        base = sample if override is None else override
        eps, prev = ops.cfg_pndm_step(eps_pair.contiguous(), guidance, hist, coef, base.contiguous(), ca, cb, want_eps=push)
        if push:
            self.ets = self.ets[-3:] + [eps]
        elif override is not None:
            self.cur_sample = None
        self.counter += 1
        return prev

    def step(self, model_output: torch.Tensor, timestep, sample: torch.Tensor, **kwargs):
        """diffusers-compatible signature: the model output is already guided."""
        pair = torch.cat([model_output, model_output]).contiguous()     # eps_u == eps_t  =>  guided eps == eps
        return types.SimpleNamespace(prev_sample=self.step_cfg(pair, 0.0, int(timestep), sample))


class DPMSolverMultistepSchedulerB200(_Img2ImgMixin):
    """DPM-Solver++(2M): diffusers 0.9 `DPMSolverMultistepScheduler.from_config(<the PNDM config above>)`, i.e.
    algorithm_type="dpmsolver++", solver_type="midpoint", solver_order=2, lower_order_final=True, epsilon prediction, no
    thresholding [memory; SURVEY Appendix C].  The reference's default txt2img scheduler (streamlit/util.py:26-33).

    The tables and per-step scalars are computed on the host with fp32 torch ops, as the reference computes them; the
    tensor update runs in one kernel fused with the guidance combine (`rf_cfg_dpmpp_step_f16`).  The x0 history lives
    in two ping-pong buffers: step i reads the buffer step i-1 wrote and writes the other one."""
    order = 1

    def __init__(self, num_train_timesteps: int = 1000, beta_start: float = 0.00085, beta_end: float = 0.012,
                 steps_offset: int = 1):
        betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
        self.alphas_cumprod = torch.cumprod(1.0 - betas, dim=0)
        self.alpha_t = torch.sqrt(self.alphas_cumprod)
        self.sigma_t = torch.sqrt(1 - self.alphas_cumprod)
        self.lambda_t = torch.log(self.alpha_t) - torch.log(self.sigma_t)
        self.num_train_timesteps = num_train_timesteps
        # `from_config(<PNDM config>)` keeps the PNDM config's steps_offset = 1 as a hidden entry of the DPM config
        # [memory; SURVEY Appendix D]; only img2img reads it, and only strength 1.0 depends on it
        self.config = {"num_train_timesteps": num_train_timesteps, "solver_order": 2, "lower_order_final": True,
                       "steps_offset": steps_offset}
        self.init_noise_sigma = 1.0
        self.timesteps: T.Optional[torch.Tensor] = None
        self.set_timesteps(50)

    def set_timesteps(self, num_inference_steps: int, device=None) -> None:
        """`linspace(0, 999, n + 1).round()[::-1][:-1]`: n timesteps from 999 down, `steps_offset` is not used."""
        self.num_inference_steps = num_inference_steps
        ts = np.linspace(0, self.num_train_timesteps - 1, num_inference_steps + 1).round()[::-1][:-1].copy()
        self.timesteps = torch.from_numpy(ts.astype(np.int64))
        self.lower_order_nums = 0
        self._x0_bufs: T.Optional[T.List[torch.Tensor]] = None
        self._x0_prev: T.Optional[torch.Tensor] = None
        self._slot = 0

    def scale_model_input(self, sample: torch.Tensor, timestep=None) -> torch.Tensor:
        return sample

    def coefficients(self, timestep: int) -> T.Dict[str, T.Any]:
        """Scalars of the step at `timestep`, each a 0-dim fp32 torch result as in the reference, returned as floats."""
        ts = self.timesteps.tolist()
        i = ts.index(int(timestep))
        t = ts[i + 1] if i + 1 < len(ts) else 0
        s0 = ts[i]
        lower_order_final = i == len(ts) - 1 and self.config["lower_order_final"] and len(ts) < 15
        second = not (self.lower_order_nums < 1 or lower_order_final)
        h = self.lambda_t[t] - self.lambda_t[s0]
        c_0 = self.alpha_t[t] * (torch.exp(-h) - 1.0)
        co = dict(second=second, sigma_s=float(self.sigma_t[s0]), alpha_s=float(self.alpha_t[s0]),
                  c_x=float(self.sigma_t[t] / self.sigma_t[s0]), c_0=float(c_0), inv_r0=0.0, c_d1=0.0)
        if second:
            h_0 = self.lambda_t[s0] - self.lambda_t[ts[i - 1]]
            r0 = h_0 / h
            co.update(inv_r0=float(1.0 / r0), c_d1=float(0.5 * c_0))
        return co

    def step_cfg(self, eps_pair: torch.Tensor, guidance: float, timestep: int, sample: torch.Tensor) -> torch.Tensor:
        """Guidance combine + scheduler.step in one kernel.  eps_pair = UNet output for [uncond | text]."""
        co = self.coefficients(timestep)
        sample = sample.contiguous()
        if self._x0_bufs is None or self._x0_bufs[0].shape != sample.shape or self._x0_bufs[0].device != sample.device:
            self._x0_bufs = [torch.empty_like(sample), torch.empty_like(sample)]
        x0_out = self._x0_bufs[self._slot]
        _, prev = ops.cfg_dpmpp_step(eps_pair.contiguous(), guidance, sample, self._x0_prev if co["second"] else None,
                                     co["sigma_s"], co["alpha_s"], co["c_x"], co["c_0"], co["inv_r0"], co["c_d1"],
                                     x0_out=x0_out)
        self._x0_prev, self._slot = x0_out, self._slot ^ 1
        self.lower_order_nums = min(self.lower_order_nums + 1, self.config["solver_order"])
        return prev

    def step(self, model_output: torch.Tensor, timestep, sample: torch.Tensor, **kwargs):
        """diffusers-compatible signature: the model output is already guided."""
        pair = torch.cat([model_output, model_output]).contiguous()     # eps_u == eps_t  =>  guided eps == eps
        return types.SimpleNamespace(prev_sample=self.step_cfg(pair, 0.0, int(timestep), sample))


# the reference's scheduler menu (streamlit/util.py:26-33); index 0 is its default
SCHEDULER_OPTIONS = [
    "DPMSolverMultistepScheduler",
    "PNDMScheduler",
    "DDIMScheduler",
    "LMSDiscreteScheduler",
    "EulerDiscreteScheduler",
    "EulerAncestralDiscreteScheduler",
]


def get_scheduler(name: str):
    """A fresh scheduler for `name` (streamlit/util.py:80-109), configured from SD-1.5's PNDM config."""
    if name == "DPMSolverMultistepScheduler":
        return DPMSolverMultistepSchedulerB200()
    if name == "PNDMScheduler":
        return PNDMSchedulerB200()
    if name in SCHEDULER_OPTIONS:
        raise NotImplementedError(f"{name} has no B200 implementation; use DPMSolverMultistepScheduler or PNDMScheduler")
    raise ValueError(f"Unknown scheduler {name}")
