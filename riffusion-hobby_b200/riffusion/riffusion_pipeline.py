"""RiffusionPipeline — B200-native drop-in for riffusion/riffusion_pipeline.py.

Same public surface as the reference class (`load_checkpoint`, `riffuse`, `interpolate_img2img`, `embed_text`,
`embed_text_weighted`, `device`, module-level `preprocess_image` / `preprocess_mask`) and the same control flow
around the inner seams (`self.unet(...)`, `self.scheduler.*`, `self.vae.*`), but those seams are the tcgen05
implementations of this package (UNetB200, PNDMSchedulerB200, VaeB200) instead of diffusers modules.

What is NOT here: diffusers (`DiffusionPipeline.from_pretrained`, hub download, traced-UNet download) — none of
it is installable in this image.  Checkpoints are loaded from diffusers-format state dicts on disk
(`load_checkpoint` on a local directory holding `unet/`, `vae/` weights as .safetensors/.bin), or created with
random-init SD-1.5 weights (`random_init`, BASELINE config 4).  The CLIP text encoder is outside the hot path
(runs once per prompt, lru-cached in the reference); it is used through `transformers` when a tokenizer / text
encoder is supplied, otherwise callers pass text embeddings directly.
"""
from __future__ import annotations

import functools
import inspect
import typing as T
from pathlib import Path

import numpy as np
import torch
from PIL import Image

from riffusion import tc_ops as ops
from riffusion.datatypes import InferenceInput
from riffusion.scheduler_b200 import PNDMSchedulerB200
from riffusion.unet_b200 import UNetB200
from riffusion.util import torch_util
from riffusion.vae_b200 import VaeB200

VAE_SCALE = 0.18215


class RiffusionPipeline:
    """Prompt / seed interpolation on spectrogram images (img2img), running on one B200."""

    def __init__(self, vae: VaeB200, unet: UNetB200, scheduler: T.Optional[PNDMSchedulerB200] = None,
                 text_encoder=None, tokenizer=None, device: str = "cuda"):
        self.vae, self.unet = vae, unet
        self.scheduler = scheduler or PNDMSchedulerB200()
        self.text_encoder, self.tokenizer = text_encoder, tokenizer
        self._device = torch.device(device)
        self._moment_cache: T.Dict[int, T.Tuple[torch.Tensor, torch.Tensor]] = {}
        self.device_slerp = True        # rf_slerp_f16 instead of the reference's host-numpy round trip
        self.use_cuda_graph = True      # replay each CFG UNet evaluation as one CUDA graph
        self._graphs: T.Dict[T.Tuple, T.Any] = {}

    # ------------------------------------------------------------------------------ construction
    @classmethod
    def random_init(cls, seed: int = 0, device: str = "cuda", with_vae: bool = True) -> "RiffusionPipeline":
        """Random-init SD-1.5 architecture (N(0, 0.02^2) weights), BASELINE config 4 — there is no network to
        fetch riffusion/riffusion-model-v1."""
        from riffusion.sd15_spec import random_state_dicts

        unet_sd, vae_sd = random_state_dicts(seed, with_vae=with_vae)
        vae = VaeB200(vae_sd, device=device) if with_vae else None
        return cls(vae=vae, unet=UNetB200(unet_sd, device=device), device=device)

    @classmethod
    def load_checkpoint(cls, checkpoint: str, use_traced_unet: bool = True, channels_last: bool = False,
                        dtype: torch.dtype = torch.float16, device: str = "cuda", local_files_only: bool = False,
                        low_cpu_mem_usage: bool = False, cache_dir: T.Optional[str] = None) -> "RiffusionPipeline":
        """Load a diffusers-layout checkpoint directory (`unet/diffusion_pytorch_model.{safetensors,bin}`,
        `vae/...`, optional `text_encoder/`, `tokenizer/`).  Signature kept from riffusion_pipeline.py:63-125;
        `use_traced_unet` / `channels_last` are accepted and ignored (the tcgen05 UNet already is the fast path,
        activations are always channels-last)."""
        device = torch_util.check_device(device)
        if dtype != torch.float16:
            raise ValueError("the B200-native pipeline computes in fp16 (the reference forces fp32 only on CPU/MPS)")
        root = Path(checkpoint)
        if not root.is_dir():
            raise FileNotFoundError(
                f"{checkpoint!r} is not a local diffusers checkpoint directory; hub download is not available "
                "(no diffusers / network in this build)")
        unet_sd = _load_weights(root / "unet")
        vae_sd = _load_weights(root / "vae")
        text_encoder = tokenizer = None
        if (root / "text_encoder").is_dir() and (root / "tokenizer").is_dir():
            from transformers import CLIPTextModel, CLIPTokenizer

            tokenizer = CLIPTokenizer.from_pretrained(root / "tokenizer")
            text_encoder = CLIPTextModel.from_pretrained(root / "text_encoder", torch_dtype=torch.float16).to(device)
        return cls(vae=VaeB200(vae_sd, device=device), unet=UNetB200(unet_sd, device=device),
                   text_encoder=text_encoder, tokenizer=tokenizer, device=device)

    @property
    def device(self) -> str:
        return str(self._device)

    # ------------------------------------------------------------------------------ text
    @functools.lru_cache()
    def embed_text(self, text) -> torch.Tensor:
        """CLIP embedding of a prompt, (1, 77, 768) fp16 (riffusion_pipeline.py:177-191)."""
        if self.tokenizer is None or self.text_encoder is None:
            raise RuntimeError("no text encoder loaded: pass text embeddings to interpolate_img2img directly")
        ids = self.tokenizer(text, padding="max_length", max_length=self.tokenizer.model_max_length, truncation=True,
                             return_tensors="pt").input_ids
        with torch.no_grad():
            return self.text_encoder(ids.to(self.device))[0].to(torch.float16)

    @functools.lru_cache()
    def embed_text_weighted(self, text) -> torch.Tensor:
        """CLIP embedding with "(word:1.2)" / "[word]" attention weights (riffusion_pipeline.py:193-206 ->
        external/prompt_weighting.py:236-372): parse, encode in chunks of 75 tokens, scale token rows by their weights,
        restore the mean."""
        from riffusion.external.prompt_weighting import get_weighted_text_embeddings

        if self.tokenizer is None or self.text_encoder is None:
            raise RuntimeError("no text encoder loaded: pass text embeddings to interpolate_img2img directly")
        with torch.no_grad():
            return get_weighted_text_embeddings(pipe=self, prompt=text, uncond_prompt=None, max_embeddings_multiples=3,
                                                no_boseos_middle=False, skip_parsing=False, skip_weighting=False)[0]

    # ------------------------------------------------------------------------------ riffuse
    @torch.no_grad()
    def riffuse(self, inputs: InferenceInput, init_image: Image.Image, mask_image: T.Optional[Image.Image] = None,
                use_reweighting: bool = True) -> Image.Image:
        """Interpolate between the two prompts / seeds of `inputs` on `init_image` (riffusion_pipeline.py:208-287)."""
        alpha = inputs.alpha
        start, end = inputs.start, inputs.end
        guidance_scale = start.guidance * (1.0 - alpha) + end.guidance * alpha
        generator_start = torch.Generator(device=self.device).manual_seed(start.seed)
        generator_end = torch.Generator(device=self.device).manual_seed(end.seed)
        embed = self.embed_text_weighted if use_reweighting else self.embed_text
        embed_start, embed_end = embed(start.prompt), embed(end.prompt)
        text_embedding = embed_start + alpha * (embed_end - embed_start)          # linear, not slerp (:249)

        init_latents = self.encode_image(init_image, torch.Generator(device=self.device).manual_seed(start.seed))
        mask = None
        if mask_image:
            vae_scale_factor = 2 ** (len(self.vae.config.block_out_channels) - 1)
            mask = preprocess_mask(mask_image, scale_factor=vae_scale_factor).to(device=self.device, dtype=embed_start.dtype)
        outputs = self.interpolate_img2img(
            text_embeddings=text_embedding, init_latents=init_latents, mask=mask, generator_a=generator_start,
            generator_b=generator_end, interpolate_alpha=alpha, strength_a=start.denoising, strength_b=end.denoising,
            num_inference_steps=inputs.num_inference_steps, guidance_scale=guidance_scale)
        return outputs["images"][0]

    @torch.no_grad()
    def riffuse_batch(self, inputs: T.Sequence[InferenceInput], init_images: T.Union[Image.Image, T.Sequence[Image.Image]],
                      mask_image: T.Optional[Image.Image] = None, use_reweighting: bool = True) -> T.List[Image.Image]:
        """`riffuse` for a list of requests in one batched denoising loop (SURVEY 8(f)-2) — what
        streamlit/tasks/interpolation.py:146-164 does one request at a time.  Every request draws exactly what `riffuse`
        draws for it (posterior noise and noise_a from generator(start.seed), noise_b from generator(end.seed), per-request
        alpha for the slerp and the prompt interpolation), so result i equals `riffuse(inputs[i], ...)` up to the batch-size
        dependent accumulation order of the kernels.  Requests are grouped by (strength, guidance, steps): the PNDM state
        and the guidance scalar are shared inside a group."""
        images = [init_images] * len(inputs) if isinstance(init_images, Image.Image) else list(init_images)
        assert len(images) == len(inputs)
        embed = self.embed_text_weighted if use_reweighting else self.embed_text
        groups: T.Dict[T.Tuple, T.List[int]] = {}
        for i, inp in enumerate(inputs):
            a = inp.alpha
            strength = (1 - a) * inp.start.denoising + a * inp.end.denoising
            guidance = inp.start.guidance * (1.0 - a) + inp.end.guidance * a
            # exact floats, not rounded: `int(num_inference_steps * strength)` (:361) depends on the last bit of the
            # reference's own lerp (alpha 0.3, denoising 0.75 -> 0.7499999999999999 -> one evaluation fewer)
            groups.setdefault((strength, guidance, inp.num_inference_steps), []).append(i)
        mask = None
        if mask_image:
            vae_scale_factor = 2 ** (len(self.vae.config.block_out_channels) - 1)
            mask = preprocess_mask(mask_image, scale_factor=vae_scale_factor).to(device=self.device, dtype=torch.float16)
        results: T.List[T.Optional[Image.Image]] = [None] * len(inputs)
        for (strength, guidance, steps), idx in groups.items():
            texts, lats, nas, nbs, alphas = [], [], [], [], []
            for i in idx:
                inp = inputs[i]
                e0, e1 = embed(inp.start.prompt), embed(inp.end.prompt)
                texts.append(e0 + inp.alpha * (e1 - e0))
                lats.append(self.encode_image(images[i], torch.Generator(device=self.device).manual_seed(inp.start.seed)))
                ga = torch.Generator(device=self.device).manual_seed(inp.start.seed)
                gb = torch.Generator(device=self.device).manual_seed(inp.end.seed)
                shape = lats[-1].shape
                nas.append(torch.randn(shape, generator=ga, device=self.device, dtype=torch.float16))
                nbs.append(torch.randn(shape, generator=gb, device=self.device, dtype=torch.float16))
                alphas.append(float(inp.alpha))
            na, nb = torch.cat(nas), torch.cat(nbs)
            if self.device_slerp:
                noise = ops.slerp(alphas, na, nb)
            else:
                noise = torch.cat([torch_util.slerp(al, na[j:j + 1], nb[j:j + 1]) for j, al in enumerate(alphas)])
            out = self.interpolate_img2img(
                text_embeddings=torch.cat(texts), init_latents=torch.cat(lats), mask=mask, generator_a=None, generator_b=None,
                interpolate_alpha=0.0, strength_a=strength, strength_b=strength, num_inference_steps=steps,
                guidance_scale=guidance, noise=noise)
            for j, i in enumerate(idx):
                results[i] = out["images"][j]
        return results  # type: ignore[return-value]

    def encode_image(self, init_image: Image.Image, generator: torch.Generator) -> torch.Tensor:
        """preprocess + VAE posterior sample * 0.18215 (:252-264).  The (mean, logvar) moments only depend on the
        image and are cached; the posterior noise is drawn from `generator` like the reference."""
        key = hash(init_image.tobytes()) ^ hash(init_image.size)
        if key not in self._moment_cache:
            img = preprocess_image(init_image).to(device=self.device, dtype=torch.float16)
            self._moment_cache[key] = self.vae.encode_moments(img)
        mean, logvar = self._moment_cache[key]
        from riffusion.vae_b200 import _Posterior

        return VAE_SCALE * _Posterior(mean, logvar).sample(generator=generator)

    # ------------------------------------------------------------------------------ denoising loop
    @torch.no_grad()
    def interpolate_img2img(self, text_embeddings: torch.Tensor, init_latents: torch.Tensor,
                            generator_a: torch.Generator, generator_b: torch.Generator, interpolate_alpha: float,
                            mask: T.Optional[torch.Tensor] = None, strength_a: float = 0.8, strength_b: float = 0.8,
                            num_inference_steps: int = 50, guidance_scale: float = 7.5,
                            negative_prompt: T.Optional[T.Union[str, T.List[str]]] = None,
                            num_images_per_prompt: int = 1, eta: T.Optional[float] = 0.0,
                            output_type: T.Optional[str] = "pil", uncond_embeddings: T.Optional[torch.Tensor] = None,
                            noise_a: T.Optional[torch.Tensor] = None, noise_b: T.Optional[torch.Tensor] = None,
                            noise: T.Optional[torch.Tensor] = None, **kwargs) -> T.Dict[str, T.Any]:
        """riffusion_pipeline.py:289-436.  Extra keyword-only inputs (`uncond_embeddings`, `noise_a`, `noise_b`)
        let callers inject what the reference computes internally (CLIP("") and the generator draws) — used by
        the parity tests and by runs without a text encoder."""
        batch_size = text_embeddings.shape[0]
        self.scheduler.set_timesteps(num_inference_steps)
        dev = self._device
        text_embeddings = text_embeddings.to(device=dev, dtype=torch.float16)
        bs_embed, seq_len, _ = text_embeddings.shape
        text_embeddings = text_embeddings.repeat(1, num_images_per_prompt, 1).view(bs_embed * num_images_per_prompt, seq_len, -1)

        do_cfg = guidance_scale > 1.0
        if do_cfg:
            if uncond_embeddings is None:
                if negative_prompt is None:                                    # :328-335
                    uncond_tokens = [""]
                elif isinstance(negative_prompt, str):
                    uncond_tokens = [negative_prompt]
                elif batch_size != len(negative_prompt):
                    raise ValueError("The length of `negative_prompt` should be equal to batch_size.")
                else:
                    uncond_tokens = list(negative_prompt)
                if self.tokenizer is None:
                    raise RuntimeError("classifier-free guidance needs the CLIP embedding of ''; pass uncond_embeddings")
                ids = self.tokenizer(uncond_tokens, padding="max_length", max_length=self.tokenizer.model_max_length,
                                     truncation=True, return_tensors="pt").input_ids
                uncond_embeddings = self.text_encoder(ids.to(self.device))[0]
            uncond_embeddings = uncond_embeddings.to(device=dev, dtype=torch.float16)
            uncond_embeddings = uncond_embeddings.repeat_interleave(batch_size * num_images_per_prompt // uncond_embeddings.shape[0], dim=0)
            context = torch.cat([uncond_embeddings, text_embeddings]).contiguous()              # :354
        else:
            context = text_embeddings.contiguous()

        latents_dtype = torch.float16
        strength = (1 - interpolate_alpha) * strength_a + interpolate_alpha * strength_b          # :358
        offset = self.scheduler.config.get("steps_offset", 0)
        init_timestep = min(int(num_inference_steps * strength) + offset, num_inference_steps)    # :361-363
        t_noise = int(self.scheduler.timesteps[-init_timestep])                                   # :365
        init_latents = init_latents.to(device=dev, dtype=latents_dtype).contiguous()
        if noise is None:
            if noise_a is None:
                noise_a = torch.randn(init_latents.shape, generator=generator_a, device=self.device, dtype=latents_dtype)
            if noise_b is None:
                noise_b = torch.randn(init_latents.shape, generator=generator_b, device=self.device, dtype=latents_dtype)
            if self.device_slerp:      # fp32 reductions on the GPU, no device->host->device round trip
                noise = ops.slerp(interpolate_alpha, noise_a.to(dev, latents_dtype), noise_b.to(dev, latents_dtype))
            else:                      # the reference's host-numpy slerp in fp16 (bit-compatible)
                noise = torch_util.slerp(interpolate_alpha, noise_a.to(dev, latents_dtype), noise_b.to(dev, latents_dtype))
        noise = noise.to(dev, latents_dtype).contiguous()
        init_latents_orig = init_latents
        latents = self.scheduler.add_noise(init_latents, noise, t_noise)                           # :379

        accepts_eta = "eta" in set(inspect.signature(self.scheduler.step).parameters.keys())       # PNDM ignores eta
        del accepts_eta
        t_start = max(num_inference_steps - init_timestep + offset, 0)                             # :392
        timesteps = self.scheduler.timesteps[t_start:]
        mask_blend = None
        if mask is not None:                                                                       # :420-425
            def mask_blend(x: torch.Tensor, t_int: int) -> torch.Tensor:
                m = mask.to(device=dev, dtype=latents_dtype).expand_as(x).contiguous()
                return self.scheduler.add_noise(init_latents_orig, noise, t_int, mask=m, blend_with=x)
        latents, n_evals = self._denoise(self.scheduler, latents, context, timesteps, guidance_scale,  # :398-418
                                         mask_blend)

        # :427 — the reference rescales in fp16 (`1.0 / 0.18215 * latents`) and returns THAT tensor under "latents"; the
        # un-scaled loop state and the evaluation count are extra keys of this implementation
        scaled = (1.0 / VAE_SCALE) * latents
        out: T.Dict[str, T.Any] = dict(latents=scaled, nsfw_content_detected=False, latents_unscaled=latents,
                                       n_unet_evals=n_evals)
        if output_type == "latent" or self.vae is None:
            out["images"] = None
            return out
        image = self.vae.decode(scaled).sample                                                       # :428
        if output_type == "pil":
            # :430-434 `(image / 2 + 0.5).clamp(0, 1)` -> numpy_to_pil, in the fp16 arithmetic of the reference's CUDA path
            u8 = ops.vae_image_to_u8(image).cpu().numpy()
            out["images"] = [Image.fromarray(im) for im in u8]
        else:
            out["images"] = (image / 2 + 0.5).clamp(0, 1).cpu().permute(0, 2, 3, 1).numpy()         # float16 array, like the reference
        return out

    def _graphed_unet(self, latent_shape, context: torch.Tensor):
        """One captured CFG evaluation per (latent shape, context shape); a new request only refreshes the
        cross-attention K / V^T that the graph reads (capture costs two eager evaluations + instantiation)."""
        from riffusion.graphed import GraphedUNet

        gkey = (tuple(latent_shape), tuple(context.shape))
        graphed = self._graphs.get(gkey)
        if graphed is None:
            graphed = self._graphs[gkey] = GraphedUNet(self.unet, latent_shape, context)
        else:
            graphed.set_context(context)
        return graphed

    def _denoise(self, sched, latents: torch.Tensor, context: torch.Tensor, timesteps, guidance_scale: float,
                 after_step: T.Optional[T.Callable[[torch.Tensor, int], torch.Tensor]] = None
                 ) -> T.Tuple[torch.Tensor, int]:
        """The denoising loop of interpolate_img2img, txt2img and img2img: one CFG UNet evaluation per timestep (a CUDA
        graph replay when enabled, [uncond | text] doubled batch; text only when guidance <= 1), then the fused guidance +
        scheduler step.  `after_step(latents, t)` runs after each step (riffuse's mask blend).  Returns (latents,
        number of UNet evaluations)."""
        do_cfg = guidance_scale > 1.0
        graphed = self._graphed_unet(latents.shape, context) if self.use_cuda_graph and do_cfg else None
        ctx_cache: T.Dict[str, T.Any] = {}
        n_evals = 0
        for t in timesteps:
            t_int = int(t)
            if graphed is not None:
                eps_pair = graphed(latents, t_int)
            else:
                model_in = torch.cat([latents] * 2) if do_cfg else latents
                eps_pair = self.unet(model_in, t_int, encoder_hidden_states=context, ctx_cache=ctx_cache).sample
            n_evals += 1
            if not do_cfg:
                eps_pair = torch.cat([eps_pair, eps_pair])
            latents = sched.step_cfg(eps_pair, guidance_scale if do_cfg else 0.0, t_int, latents)
            if after_step is not None:
                latents = after_step(latents, t_int)
        return latents, n_evals

    # ------------------------------------------------------------------------------ txt2img
    @torch.no_grad()
    def txt2img(self, prompt: T.Union[str, T.Sequence[str], None] = None, *,
                negative_prompt: T.Union[str, T.Sequence[T.Optional[str]], None] = None,
                seed: T.Union[int, T.Sequence[int]] = 42, num_inference_steps: int = 50, guidance_scale: float = 7.5,
                width: int = 512, height: int = 512, scheduler: str = "DPMSolverMultistepScheduler",
                text_embeddings: T.Optional[torch.Tensor] = None, uncond_embeddings: T.Optional[torch.Tensor] = None,
                latents: T.Optional[torch.Tensor] = None, output_type: str = "pil") -> T.Dict[str, T.Any]:
        """Text to image from pure noise: diffusers 0.9 `StableDiffusionPipeline.__call__` as the reference's text-to-audio
        tasks run it (streamlit/util.py run_txt2img; SURVEY Appendix C).

        `prompt`, `negative_prompt` and `seed` may be lists (a scalar is used for every clip): the clips run as one
        batched CFG loop with per-clip text and unconditional embeddings and one generator per clip, so clip i equals a
        single call with `seed[i]` up to the batch-size dependent accumulation order of the kernels.  Prompts are encoded
        with the plain tokenizer + text encoder (`embed_text`, 77 tokens), the unconditional embedding is that of
        `negative_prompt or ""`.  `text_embeddings` / `uncond_embeddings` / `latents` inject what would otherwise be
        computed (B, 77, D) / (1 or B, 77, D) / (B, 4, height/8, width/8) fp16.  A fresh scheduler is built per call;
        `self.scheduler`, which riffuse uses, is not touched.

        Returns images (PIL list, or None for output_type="latent", or a float32 (B, H, W, 3) array for "np"),
        latents (1/0.18215-scaled, what the VAE decodes), latents_unscaled and n_unet_evals."""
        from riffusion.scheduler_b200 import get_scheduler

        if height % 8 or width % 8:
            raise ValueError(f"`height` and `width` have to be divisible by 8 but are {height} and {width}.")
        if height % 64 or width % 64:
            raise NotImplementedError(
                f"height {height} / width {width}: sizes that are not multiples of 64 need up-sampling to odd sizes "
                "(diffusers' upsample_size), which UNetB200 does not implement")
        sched = get_scheduler(scheduler)
        dev = self._device
        B, per_clip, context = self._batch_context(prompt, negative_prompt, seed, text_embeddings, uncond_embeddings,
                                                   guidance_scale, latents=None if latents is None else latents.shape[0])

        shape = (B, 4, height // 8, width // 8)
        if latents is None:
            latents = torch.cat([torch.randn((1,) + shape[1:], generator=torch.Generator(device=self.device).manual_seed(int(s)),
                                             device=self.device, dtype=torch.float16) for s in per_clip(seed)])
        latents = latents.to(device=dev, dtype=torch.float16).contiguous()
        if tuple(latents.shape) != shape:
            raise ValueError(f"latents must have shape {shape}, got {tuple(latents.shape)}")
        # `latents * init_noise_sigma` is the identity: both schedulers have init_noise_sigma = 1

        sched.set_timesteps(num_inference_steps)
        latents, n_evals = self._denoise(sched, latents, context, sched.timesteps, guidance_scale)
        return self._decode_output(latents, n_evals, output_type)

    def _batch_context(self, prompt, negative_prompt, seed, text_embeddings, uncond_embeddings, guidance_scale: float,
                       **batch_sizes: T.Optional[int]):
        """Batch size, per-clip broadcast and CFG context of txt2img / img2img.  `prompt`, `negative_prompt` and `seed`
        may be lists; the batch size is their common length, which the first dimension of `text_embeddings` and the
        `batch_sizes` given (None entries are ignored) must equal.  Returns (B, per_clip, context) with context = [uncond | text]
        (text only when guidance <= 1)."""
        dev = self._device
        as_list = lambda v: list(v) if isinstance(v, (list, tuple)) else None   # noqa: E731
        lists = [v for v in (as_list(prompt), as_list(negative_prompt), as_list(seed)) if v is not None]
        if text_embeddings is not None:
            lists.append(list(range(text_embeddings.shape[0])))
        for n in batch_sizes.values():
            if n is not None:
                lists.append(list(range(n)))
        B = len(lists[0]) if lists else 1
        if any(len(v) != B for v in lists):
            raise ValueError(f"prompt, negative_prompt, seed, text_embeddings and {', '.join(batch_sizes)} must agree on the "
                             "batch size")
        per_clip = lambda v: as_list(v) if as_list(v) is not None else [v] * B   # noqa: E731

        if text_embeddings is None:
            if prompt is None:
                raise ValueError("pass a prompt or text_embeddings")
            text_embeddings = torch.cat([self.embed_text(p) for p in per_clip(prompt)])
        text_embeddings = text_embeddings.to(device=dev, dtype=torch.float16)
        if guidance_scale > 1.0:
            if uncond_embeddings is None:
                uncond_embeddings = torch.cat([self.embed_text(n or "") for n in per_clip(negative_prompt)])
            uncond_embeddings = uncond_embeddings.to(device=dev, dtype=torch.float16)
            uncond_embeddings = uncond_embeddings.expand(B, -1, -1) if uncond_embeddings.shape[0] == 1 else uncond_embeddings
            context = torch.cat([uncond_embeddings, text_embeddings]).contiguous()
        else:
            context = text_embeddings.contiguous()
        return B, per_clip, context

    def _decode_output(self, latents: torch.Tensor, n_evals: int, output_type: str) -> T.Dict[str, T.Any]:
        """decode_latents of txt2img / img2img: 1 / 0.18215 * latents, VAE decode, (image / 2 + 0.5).clamp(0, 1) in fp16,
        then `.float()`, so numpy_to_pil's (x * 255).round() runs in fp32."""
        scaled = (1.0 / VAE_SCALE) * latents
        out: T.Dict[str, T.Any] = dict(latents=scaled, latents_unscaled=latents, n_unet_evals=n_evals, images=None)
        if output_type == "latent" or self.vae is None:
            return out
        image = self.vae.decode(scaled).sample
        if output_type == "pil":
            u8 = ops.vae_image_to_u8(image, fp32_scale=True).cpu().numpy()
            out["images"] = [Image.fromarray(im) for im in u8]
        else:
            out["images"] = (image / 2 + 0.5).clamp(0, 1).cpu().permute(0, 2, 3, 1).float().numpy()
        return out

    # ------------------------------------------------------------------------------ img2img
    @torch.no_grad()
    def img2img(self, prompt: T.Union[str, T.Sequence[str], None] = None, *,
                init_image: T.Union[Image.Image, T.Sequence[Image.Image], None] = None,
                init_images_u8: T.Optional[torch.Tensor] = None, strength: float = 0.8, num_inference_steps: int = 50,
                guidance_scale: float = 7.5, negative_prompt: T.Union[str, T.Sequence[T.Optional[str]], None] = None,
                seed: T.Union[int, T.Sequence[int]] = 42, scheduler: str = "DPMSolverMultistepScheduler",
                text_embeddings: T.Optional[torch.Tensor] = None, uncond_embeddings: T.Optional[torch.Tensor] = None,
                noise: T.Optional[torch.Tensor] = None, output_type: str = "pil") -> T.Dict[str, T.Any]:
        """Image to image: diffusers 0.9 `StableDiffusionImg2ImgPipeline.__call__` as the reference's audio-to-audio task
        runs it (streamlit/util.py run_img2img; SURVEY Appendix D).

        The init image is a PIL image (or one per clip), preprocessed on the host as `preprocess_image` does, or
        `init_images_u8`, a (1 or B, H, W, 3) uint8 tensor whose sides are multiples of 32, converted on the device with
        the same arithmetic.  Each clip draws from one generator seeded with its seed: the VAE posterior sample first,
        then the noise.  The noise is added at timesteps[t_start] with the fp16 op sequence of `add_noise`, and the loop
        runs timesteps[t_start:] with a fresh scheduler (`self.scheduler`, which riffuse uses, is not touched).
        `prompt`, `negative_prompt` and `seed` may be lists, batched as in `txt2img`; `text_embeddings`,
        `uncond_embeddings` and `noise` ((B, 4, H/8, W/8) fp16, replacing the second draw) inject what would otherwise
        be computed.

        Returns images (PIL list, None for output_type="latent", or a float32 (B, H, W, 3) array for "np"), latents
        (1/0.18215-scaled), latents_unscaled and n_unet_evals."""
        from riffusion.scheduler_b200 import get_scheduler
        from riffusion.vae_b200 import _Posterior

        if (init_image is None) == (init_images_u8 is None):
            raise ValueError("pass exactly one of init_image and init_images_u8")
        dev = self._device
        if init_images_u8 is not None:
            if init_images_u8.dim() != 4 or init_images_u8.shape[-1] != 3 or init_images_u8.dtype != torch.uint8:
                raise ValueError(f"init_images_u8 must be a (B, H, W, 3) uint8 tensor, got {tuple(init_images_u8.shape)} "
                                 f"{init_images_u8.dtype}")
            if init_images_u8.shape[1] % 32 or init_images_u8.shape[2] % 32:
                raise ValueError(f"init_images_u8 sides must be multiples of 32, got {tuple(init_images_u8.shape[1:3])}")
            height, width = int(init_images_u8.shape[1]), int(init_images_u8.shape[2])
        else:
            imgs = [init_image] if isinstance(init_image, Image.Image) else list(init_image)
            width, height = (x - x % 32 for x in imgs[0].size)
        if height % 64 or width % 64:
            raise NotImplementedError(
                f"height {height} / width {width}: sizes that are not multiples of 64 need up-sampling to odd sizes "
                "(diffusers' upsample_size), which UNetB200 does not implement")
        sched = get_scheduler(scheduler)
        _, timesteps, t_noise = sched.img2img_timesteps(num_inference_steps, strength)
        n_img = init_images_u8.shape[0] if init_images_u8 is not None else len(imgs)
        B, per_clip, context = self._batch_context(prompt, negative_prompt, seed, text_embeddings, uncond_embeddings,
                                                   guidance_scale, noise=None if noise is None else noise.shape[0],
                                                   init_images=None if n_img == 1 else n_img)

        if init_images_u8 is not None:
            image = ops.image_u8_to_f16(init_images_u8.to(dev))
        else:
            image = torch.cat([preprocess_image(im) for im in imgs]).to(device=dev, dtype=torch.float16)
        mean, logvar = self.vae.encode_moments(image)                       # one batched encoder pass
        lats, noises = [], []
        for i, s in enumerate(per_clip(seed)):
            g = torch.Generator(device=self.device).manual_seed(int(s))
            j = i if n_img > 1 else 0
            lats.append(VAE_SCALE * _Posterior(mean[j:j + 1], logvar[j:j + 1]).sample(generator=g))
            if noise is None:
                noises.append(torch.randn(lats[-1].shape, generator=g, device=self.device, dtype=torch.float16))
        init_latents = torch.cat(lats).contiguous()
        noise = torch.cat(noises) if noise is None else noise.to(device=dev, dtype=torch.float16).contiguous()
        if noise.shape != init_latents.shape:
            raise ValueError(f"noise must have shape {tuple(init_latents.shape)}, got {tuple(noise.shape)}")
        latents = sched.add_noise_fp16(init_latents, noise, t_noise)
        latents, n_evals = self._denoise(sched, latents, context, timesteps, guidance_scale)
        return self._decode_output(latents, n_evals, output_type)

    @torch.no_grad()
    def audio_to_audio_clips(self, waveforms: torch.Tensor, *, converter, prompt: T.Union[str, T.Sequence[str], None] = None,
                             init_angles: T.Optional[torch.Tensor] = None, **img2img_kwargs) -> T.Dict[str, T.Any]:
        """img2img on a batch of equally long mono clips without leaving the device, what the reference's audio-to-audio
        task does one clip at a time: waveform -> mel amplitudes (rf_stft_mel) -> spectrogram image (rf_mel_to_image) ->
        Pillow-exact BICUBIC resize to the next multiples of 32 (rf_resample_u8) -> `img2img` -> uint8 image (fp32
        rounding) -> BICUBIC resize back -> mel amplitudes (mono = R plane, max_value 30e6) -> inverse mel + Griffin-Lim.

        `waveforms`: (B, L) float32 samples at the converter's rate, int16-valued as `spectrogram_from_audio` reads them.
        `converter` is a mono SpectrogramConverter.  The img2img keywords (strength, seed, num_inference_steps, ...) pass
        through.  Returns device tensors: source_images and images (B, H, W, 3) uint8, waveform (B, hop (W - 1)) fp32,
        latents, latents_unscaled, and n_unet_evals."""
        from riffusion import _native

        p = converter.p
        if p.stereo:
            raise NotImplementedError("audio_to_audio_clips is mono only (no 20 kHz stereo on the device path); use "
                                      "img2img with SpectrogramImageConverter images for stereo")
        L = int(waveforms.shape[-1])
        H, W = p.num_frequencies, 1 + L // p.hop_length
        H32, W32 = (-(-v // 32) * 32 for v in (H, W))
        if H32 % 64 or W32 % 64:
            raise NotImplementedError(
                f"clips of {L} samples give {H} x {W} images, {H32} x {W32} after the 32-stride resize: sizes that are "
                "not multiples of 64 need up-sampling to odd sizes (diffusers' upsample_size), which UNetB200 does not "
                "implement")
        wave = _native.require_cuda(waveforms, "waveforms", torch.float32)
        wave = wave[None] if wave.dim() == 1 else wave
        B = wave.shape[0]
        mel = converter.mel_amplitudes_from_waveform(wave)
        src = torch.empty((B, H, W, 3), dtype=torch.uint8, device=wave.device)
        mx = torch.empty((B,), dtype=torch.float32, device=wave.device)
        lib = _native.lib()
        for i in range(B):
            _native.check(lib.rf_mel_to_image(mel[i].data_ptr(), 1, H, W, float(p.power_for_image), src[i].data_ptr(),
                                              mx[i:i + 1].data_ptr(), _native.stream_ptr(wave.device)))
        out = self.img2img(prompt, init_images_u8=ops.resample_u8(src, H32, W32), output_type="latent",
                           **img2img_kwargs)
        riffed = ops.resample_u8(ops.vae_image_to_u8(self.vae.decode(out["latents"]).sample, fp32_scale=True), H, W)
        return dict(source_images=src, images=riffed, waveform=self._waveform_from_u8(riffed, converter, init_angles),
                    latents=out["latents"], latents_unscaled=out["latents_unscaled"], n_unet_evals=out["n_unet_evals"])

    @torch.no_grad()
    def text_to_audio_clips(self, prompt: T.Union[str, T.Sequence[str], None] = None, *, converter,
                            init_angles: T.Optional[torch.Tensor] = None, height: T.Optional[int] = None,
                            **txt2img_kwargs) -> T.Dict[str, torch.Tensor]:
        """`txt2img` followed by the audio conversion without leaving the device: latents -> VAE decode -> uint8 image
        (fp32 rounding, as txt2img's PIL images) -> mel amplitudes (mono = R plane) -> inverse mel + Griffin-Lim.  What
        the reference's text-to-audio task does per clip (run_txt2img, then audio_segment_from_spectrogram_image) minus the
        host round trip and `apply_filters`.  `converter` is a SpectrogramConverter; mono only, and `height` must be its
        number of mel bins.  Returns device tensors: images (B, H, W, 3) uint8, waveform (B, 441 (W - 1)) fp32, latents,
        latents_unscaled, n_unet_evals."""
        p = converter.p
        if p.stereo:
            raise NotImplementedError("text_to_audio_clips is mono only; use txt2img + SpectrogramImageConverter for stereo")
        height = p.num_frequencies if height is None else height
        if height != p.num_frequencies:
            raise ValueError(f"height {height} must equal the number of mel bins {p.num_frequencies}")
        out = self.txt2img(prompt, height=height, output_type="latent", **txt2img_kwargs)
        image = self.vae.decode(out["latents"]).sample
        u8 = ops.vae_image_to_u8(image, fp32_scale=True)
        return dict(images=u8, waveform=self._waveform_from_u8(u8, converter, init_angles), latents=out["latents"],
                    latents_unscaled=out["latents_unscaled"], n_unet_evals=out["n_unet_evals"])

    def _waveform_from_u8(self, u8: torch.Tensor, converter, init_angles: T.Optional[torch.Tensor]) -> torch.Tensor:
        """(B, H, W, 3) uint8 spectrogram images on the device -> (B, hop (W - 1)) waveforms: image_util
        spectrogram_from_image semantics (mono = R plane, max_value 30e6) + inverse mel + Griffin-Lim."""
        from riffusion import _native

        B, H, W, _ = u8.shape
        mel = torch.empty((B, H, W), dtype=torch.float32, device=u8.device)
        lib = _native.lib()
        p = converter.p
        for i in range(B):
            _native.check(lib.rf_image_to_mel(u8[i].data_ptr(), H, W, 0, float(p.power_for_image), 30e6, mel[i].data_ptr(),
                                              _native.stream_ptr(u8.device)))
        return converter.waveform_from_mel_amplitudes(mel, init_angles)

    # ------------------------------------------------------------------------------ batched request -> audio
    @torch.no_grad()
    def generate_clips(self, text_embeddings: torch.Tensor, uncond_embeddings: torch.Tensor, init_latents: torch.Tensor,
                       noise: torch.Tensor, strength: float, num_inference_steps: int, guidance_scale: float,
                       converter, init_angles: T.Optional[torch.Tensor] = None) -> T.Dict[str, torch.Tensor]:
        """B independent requests end to end on the device (SURVEY 8(f)-1/2): denoise -> VAE decode -> uint8 image ->
        mel amplitudes (image_util.spectrogram_from_image semantics, mono = R plane) -> inverse mel + Griffin-Lim.
        This is what `server.compute_request` does per request (riffuse, then audio_from_spectrogram_image,
        server.py:145-164) without leaving the GPU in between.  Returns device tensors:
        images (B,512,512,3) uint8, waveform (B, L) fp32, latents."""
        out = self.interpolate_img2img(
            text_embeddings=text_embeddings, init_latents=init_latents, generator_a=None, generator_b=None,
            interpolate_alpha=0.0, strength_a=strength, strength_b=strength, num_inference_steps=num_inference_steps,
            guidance_scale=guidance_scale, uncond_embeddings=uncond_embeddings, noise=noise, output_type="latent")
        latents = out["latents_unscaled"]
        image = self.vae.decode(out["latents"]).sample
        u8 = ops.vae_image_to_u8(image)
        wave = self._waveform_from_u8(u8, converter, init_angles)
        return dict(images=u8, waveform=wave, latents=out["latents"], latents_unscaled=latents,
                    n_unet_evals=out["n_unet_evals"])

    @staticmethod
    def numpy_to_pil(images: np.ndarray) -> T.List[Image.Image]:
        """diffusers DiffusionPipeline.numpy_to_pil: (x * 255).round().astype(uint8)"""
        if images.ndim == 3:
            images = images[None, ...]
        images = (images * 255).round().astype("uint8")
        return [Image.fromarray(im) for im in images]

    def progress_bar(self, iterable):
        return iterable


def _load_weights(folder: Path) -> T.Dict[str, torch.Tensor]:
    for name in ("diffusion_pytorch_model.safetensors", "model.safetensors"):
        f = folder / name
        if f.exists():
            from safetensors.torch import load_file

            return load_file(str(f))
    for name in ("diffusion_pytorch_model.bin", "pytorch_model.bin"):
        f = folder / name
        if f.exists():
            return torch.load(str(f), map_location="cpu", weights_only=True)
    raise FileNotFoundError(f"no diffusers weight file under {folder}")


def preprocess_image(image: Image.Image) -> torch.Tensor:
    """PIL RGB -> (1, 3, H, W) float in [-1, 1], size rounded down to multiples of 32 with LANCZOS
    (riffusion_pipeline.py:439-452)."""
    w, h = image.size
    w, h = (x - x % 32 for x in (w, h))
    image = image.resize((w, h), resample=Image.LANCZOS)
    arr = np.array(image).astype(np.float32) / 255.0
    arr = arr[None].transpose(0, 3, 1, 2)
    return 2.0 * torch.from_numpy(arr) - 1.0


def preprocess_mask(mask: Image.Image, scale_factor: int = 8) -> torch.Tensor:
    """PIL mask -> (1, 4, h/8, w/8) with white = repaint (riffusion_pipeline.py:455-477)."""
    mask = mask.convert("L")
    w, h = mask.size
    w, h = (x - x % 32 for x in (w, h))
    mask = mask.resize((w // scale_factor, h // scale_factor), resample=Image.NEAREST)
    arr = np.array(mask).astype(np.float32) / 255.0
    arr = np.tile(arr, (4, 1, 1))[None]          # the reference's transpose(0,1,2,3) is a no-op
    return torch.from_numpy(1 - arr)
