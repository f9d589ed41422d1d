"""Text to image on the host: the DPM-Solver++ tables and scalars (SURVEY Appendix C self-checks), the solver's algebra,
the txt2img control flow against the oracle loop with the device ops replaced by torch stand-ins, argument errors, and
the `riffusion.text_to_audio` front end with the pipeline faked.  No GPU, no kernels."""
import json
import types

import numpy as np
import pytest
import torch
from PIL import Image

from riffusion.riffusion_pipeline import RiffusionPipeline
from riffusion.scheduler_b200 import DPMSolverMultistepSchedulerB200, SCHEDULER_OPTIONS, get_scheduler


def _close(got, want, rel=2e-7):
    assert abs(got - want) <= rel * abs(want), (got, want)


# ------------------------------------------------------------------------------------------------ scheduler tables
def test_dpm_timesteps_and_self_check_scalars():
    s = DPMSolverMultistepSchedulerB200()
    s.set_timesteps(10)
    assert s.timesteps.tolist() == [999, 899, 799, 699, 599, 500, 400, 300, 200, 100]
    s.set_timesteps(30)
    ts = s.timesteps.tolist()
    assert ts == [999, 966, 932, 899, 866, 832, 799, 766, 733, 699, 666, 633, 599, 566, 533, 499, 466, 433, 400, 366,
                  333, 300, 266, 233, 200, 166, 133, 100, 67, 33]
    assert s.timesteps.dtype == torch.int64 and s.init_noise_sigma == 1.0
    c = s.coefficients(999)                                   # step 0, 999 -> 966: first order
    assert not c["second"]
    _close(c["c_x"], 0.998885989)
    _close(c["c_0"], -0.0147348447)
    s.lower_order_nums = 1                                    # step 1, 966 -> 932: second order
    c = s.coefficients(966)
    assert c["second"]
    _close(c["c_x"], 0.998393178)
    _close(c["c_0"], -0.0175359584)
    _close(c["inv_r0"], 0.981989384)
    _close(c["c_d1"], -0.00876797922)
    s.lower_order_nums = 2                                    # last step, 33 -> 0: second order (30 >= 15 steps)
    c = s.coefficients(33)
    assert c["second"]
    _close(c["c_x"], 0.165234849)
    _close(c["c_0"], -0.836932540)
    _close(c["inv_r0"], 4.52971792)
    _close(c["c_d1"], -0.418466270)
    s.set_timesteps(10)                                       # fewer than 15 steps: lower_order_final
    s.lower_order_nums = 2
    assert not s.coefficients(100)["second"] and s.coefficients(200)["second"]


def test_dpm_tables_are_fp32_torch():
    s = DPMSolverMultistepSchedulerB200()
    ac = torch.cumprod(1.0 - torch.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000, dtype=torch.float32) ** 2, dim=0)
    assert torch.equal(s.alphas_cumprod, ac)
    assert torch.equal(s.alpha_t, torch.sqrt(ac)) and torch.equal(s.sigma_t, torch.sqrt(1 - ac))
    assert torch.equal(s.lambda_t, torch.log(torch.sqrt(ac)) - torch.log(torch.sqrt(1 - ac)))
    assert all(t.dtype == torch.float32 for t in (s.alpha_t, s.sigma_t, s.lambda_t))


def test_dpm_first_order_equals_ddim_eta0():
    """x_t = (s_t/s_s) x - a_t (e^-h - 1) x0  ==  a_t x0 + s_t eps  with  x0 = (x - s_s eps) / a_s  (DDIM, eta = 0)"""
    s = DPMSolverMultistepSchedulerB200()
    a, sg = s.alpha_t.double(), s.sigma_t.double()
    lam = a.log() - sg.log()                                  # float64 throughout: an identity, not a rounding check
    rng = np.random.default_rng(0)
    x, eps = torch.from_numpy(rng.standard_normal(64)), torch.from_numpy(rng.standard_normal(64))
    for _ in range(200):
        t, src = sorted(rng.choice(1000, size=2, replace=False).tolist())
        x0 = (x - sg[src] * eps) / a[src]
        dpm = (sg[t] / sg[src]) * x - a[t] * (torch.exp(-(lam[t] - lam[src])) - 1.0) * x0
        ddim = a[t] * x0 + sg[t] * (x - a[src] * x0) / sg[src]
        assert torch.allclose(dpm, ddim, rtol=1e-12, atol=1e-12), (src, t)


def _dpm_stand_in(eps_pair, guidance, sample, x0_prev, sigma_s, alpha_s, c_x, c_0, inv_r0=0.0, c_d1=0.0, x0_out=None,
                  out=None):
    """torch definition of rf_cfg_dpmpp_step_f16 (math in the tensors' own precision, float64 here)"""
    n = sample.shape[0]
    eu, et = eps_pair[:n], eps_pair[n:]
    e = eu + guidance * (et - eu)
    m0 = (sample - sigma_s * e) / alpha_s
    xt = c_x * sample - c_0 * m0
    if x0_prev is not None:
        xt = xt - c_d1 * (inv_r0 * (m0 - x0_prev))
    x0_out = torch.empty_like(sample) if x0_out is None else x0_out
    x0_out.copy_(m0)
    return x0_out, xt


@pytest.mark.parametrize("steps", [10, 30])
def test_dpm_exact_denoiser_stays_on_trajectory(monkeypatch, steps):
    """A model that returns the true eps of x = a_s x0* + s_s eps* makes every x0 prediction x0*, so D1 = 0 and every
    step lands on a_t x0* + s_t eps*; 10 steps exercise lower_order_final, 30 the second-order last step."""
    from riffusion import tc_ops

    monkeypatch.setattr(tc_ops, "cfg_dpmpp_step", _dpm_stand_in)
    s = DPMSolverMultistepSchedulerB200()
    s.set_timesteps(steps)
    a, sg = s.alpha_t.double(), s.sigma_t.double()
    g = torch.Generator().manual_seed(steps)
    x0s, epss = torch.randn(2, 4, 8, 8, generator=g, dtype=torch.float64), torch.randn(2, 4, 8, 8, generator=g, dtype=torch.float64)
    ts = s.timesteps.tolist()
    x = a[ts[0]] * x0s + sg[ts[0]] * epss
    for i, t in enumerate(ts):
        eps = (x - a[t] * x0s) / sg[t]
        pair = torch.cat([eps - 0.5, eps - 0.25])            # guided: eu + 2 (et - eu) = eps
        x = s.step_cfg(pair, 2.0, t, x)
        t_next = ts[i + 1] if i + 1 < len(ts) else 0
        want = a[t_next] * x0s + sg[t_next] * epss
        err = float((x - want).abs().max())
        assert err < 2e-5, (i, t, err)
    assert s.lower_order_nums == 2


def test_get_scheduler_and_options():
    from riffusion.scheduler_b200 import PNDMSchedulerB200

    assert SCHEDULER_OPTIONS[0] == "DPMSolverMultistepScheduler" and len(SCHEDULER_OPTIONS) == 6
    assert isinstance(get_scheduler("DPMSolverMultistepScheduler"), DPMSolverMultistepSchedulerB200)
    assert isinstance(get_scheduler("PNDMScheduler"), PNDMSchedulerB200)
    assert get_scheduler("PNDMScheduler") is not get_scheduler("PNDMScheduler")
    for name in SCHEDULER_OPTIONS[2:]:
        with pytest.raises(NotImplementedError, match=name):
            get_scheduler(name)
    with pytest.raises(ValueError):
        get_scheduler("Bogus")


# ------------------------------------------------------------------------------------------------ txt2img control flow
def _fake_ops(monkeypatch):
    """torch definitions of the two fused scheduler kernels on fp16 tensors (math in fp32, one rounding per output)"""
    from riffusion import tc_ops

    def dpm(eps_pair, guidance, sample, x0_prev, *co, x0_out=None, out=None):
        x0, xt = _dpm_stand_in(eps_pair.float(), guidance, sample.float(), None if x0_prev is None else x0_prev.float(), *co)
        x0_out = torch.empty_like(sample) if x0_out is None else x0_out
        x0_out.copy_(x0)
        return x0_out, xt.to(sample.dtype)

    def pndm(eps_pair, guidance, hist, coef, sample, ca, cb, want_eps=True):
        n = sample.shape[0]
        eu, et = eps_pair[:n].float(), eps_pair[n:].float()
        eps = eu + guidance * (et - eu)
        e = coef[0] * eps
        for c, h in zip(coef[1:], hist):
            e = e + c * h.float()
        return (eps.to(sample.dtype) if want_eps else None), (ca * sample.float() - cb * e).to(sample.dtype)

    monkeypatch.setattr(tc_ops, "cfg_dpmpp_step", dpm)
    monkeypatch.setattr(tc_ops, "cfg_pndm_step", pndm)


def _model(x, t, ctx):
    return 0.3 * torch.tanh(x.float()) + 0.002 * (t / 1000.0) + 0.05 * ctx.float().mean(dim=(1, 2))[:, None, None, None]


class _FakeUNet:
    def __init__(self):
        self.calls = []

    def __call__(self, x, t, encoder_hidden_states=None, **kw):
        self.calls.append((tuple(x.shape), int(t)))
        return types.SimpleNamespace(sample=_model(x, int(t), encoder_hidden_states).to(torch.float16))


def _cpu_pipe():
    pipe = RiffusionPipeline(vae=None, unet=_FakeUNet(), device="cpu")
    pipe.use_cuda_graph = False
    return pipe


def test_txt2img_control_flow_matches_oracle_loop(monkeypatch):
    """pure-noise start, CFG doubling, one evaluation per DPM timestep (n + 1 for PNDM), scheduler stepping and the
    1/0.18215 rescale of txt2img against txt2img_loop with the fp64 DPM oracle / the PNDM oracle"""
    from oracle import unet_oracle as uo
    from txt2img_oracle import DPMSolverMultistepSchedulerOracle, txt2img_loop

    _fake_ops(monkeypatch)
    torch.manual_seed(7)
    lat = torch.randn(2, 4, 8, 16).half()
    text, uncond = torch.randn(2, 77, 16).half(), torch.randn(1, 77, 16).half()
    for scheduler, steps, n_want in (("DPMSolverMultistepScheduler", 10, 10), ("DPMSolverMultistepScheduler", 20, 20),
                                     ("DPMSolverMultistepScheduler", 30, 30), ("PNDMScheduler", 50, 51)):
        pipe = _cpu_pipe()
        before = pipe.scheduler
        out = pipe.txt2img(text_embeddings=text, uncond_embeddings=uncond, latents=lat, num_inference_steps=steps,
                           guidance_scale=7.0, width=128, height=64, scheduler=scheduler, output_type="latent")
        assert pipe.scheduler is before and out["images"] is None
        oracle = DPMSolverMultistepSchedulerOracle() if scheduler.startswith("DPM") else uo.PNDMSchedulerOracle()
        ref, n_ref = txt2img_loop(_model, oracle, text.float(), uncond.float(), lat.float(), steps, 7.0)
        assert out["n_unet_evals"] == n_ref == n_want == len(pipe.unet.calls)
        assert all(shape == (4, 4, 8, 16) for shape, _ in pipe.unet.calls)
        if scheduler.startswith("DPM"):
            assert pipe.unet.calls[0][1] == 999 and [t for _, t in pipe.unet.calls] == oracle.timesteps.tolist()
        err = float((out["latents_unscaled"].float() - ref).norm() / ref.norm())
        print(f"txt2img {scheduler} {steps} steps: fp16 stand-ins vs oracle loop rel L2 {err:.2e}")
        assert err < 2e-2, (scheduler, steps, err)
        assert torch.equal(out["latents"], (1.0 / 0.18215) * out["latents_unscaled"])


def test_txt2img_seeds_prompts_and_embeddings(monkeypatch):
    """per-clip generators (seed list), per-clip text / negative prompts through embed_text, scalar broadcast, and the
    no-guidance path (guidance <= 1: text context only)"""
    _fake_ops(monkeypatch)
    pipe = _cpu_pipe()
    seen = []

    def embed(text):
        seen.append(text)
        return torch.full((1, 77, 16), float(len(text)), dtype=torch.float16)

    pipe.embed_text = embed
    out = pipe.txt2img(["a", "bb"], negative_prompt=[None, "ccc"], seed=[3, 4], num_inference_steps=4, width=64,
                       height=64, output_type="latent")
    assert seen == ["a", "bb", "", "ccc"]
    ref = _cpu_pipe()
    ref.embed_text = embed
    lat = torch.cat([torch.randn((1, 4, 8, 8), generator=torch.Generator().manual_seed(s), dtype=torch.float16)
                     for s in (3, 4)])
    out2 = ref.txt2img(["a", "bb"], negative_prompt=[None, "ccc"], latents=lat, num_inference_steps=4, width=64,
                       height=64, output_type="latent")
    assert torch.equal(out["latents_unscaled"], out2["latents_unscaled"])
    seen.clear()
    pipe.txt2img("x", negative_prompt="nn", seed=[1, 2, 3], num_inference_steps=2, width=64, height=64, output_type="latent")
    assert seen == ["x"] * 3 + ["nn"] * 3
    seen.clear()
    pipe.unet.calls.clear()
    out = pipe.txt2img("x", seed=1, guidance_scale=1.0, num_inference_steps=3, width=64, height=64, output_type="latent")
    assert seen == ["x"] and [s for s, _ in pipe.unet.calls] == [(1, 4, 8, 8)] * 3 and out["n_unet_evals"] == 3
    with pytest.raises(ValueError):
        pipe.txt2img(["a", "b"], seed=[1, 2, 3], width=64, height=64)


def test_txt2img_argument_errors():
    pipe = _cpu_pipe()
    for w, h in ((500, 512), (512, 516)):
        with pytest.raises(ValueError, match="divisible by 8"):
            pipe.txt2img("a", width=w, height=h)
    for w, h in ((520, 512), (512, 584)):
        with pytest.raises(NotImplementedError, match="multiples of 64"):
            pipe.txt2img("a", width=w, height=h)
    for name in SCHEDULER_OPTIONS[2:]:
        with pytest.raises(NotImplementedError, match=name):
            pipe.txt2img("a", scheduler=name)
    with pytest.raises(ValueError, match="shape"):
        pipe.txt2img(text_embeddings=torch.zeros(1, 77, 16).half(), uncond_embeddings=torch.zeros(1, 77, 16).half(),
                     latents=torch.zeros(1, 4, 8, 8).half(), width=128, height=64)


# ------------------------------------------------------------------------------------------------ front end
def test_text_to_audio_parser():
    from riffusion import cli, text_to_audio

    parser = cli.build_parser(text_to_audio.COMMANDS, prog="riffusion.text_to_audio")
    sub = next(a for a in parser._actions if a.dest == "command")
    assert set(sub.choices) == {"text-to-audio", "text-to-audio-batch"}
    flags = {o for act in sub.choices["text-to-audio"]._actions for o in act.option_strings}
    assert {"--prompt", "--checkpoint", "--output-dir", "--negative-prompt", "--seed", "--num-clips",
            "--num-inference-steps", "--guidance", "--width", "--scheduler", "--use-20k", "--device"} <= flags
    ns = parser.parse_args(["text-to-audio", "--prompt", "church bells", "--checkpoint", "ck", "--output-dir", "o"])
    assert (ns.negative_prompt, ns.seed, ns.num_clips, ns.num_inference_steps, ns.guidance, ns.width, ns.scheduler,
            ns.use_20k, ns.device) == ("", 42, 1, 30, 7.0, 512, "DPMSolverMultistepScheduler", False, "cuda")
    ns = parser.parse_args(["text-to-audio", "--prompt", "p", "--checkpoint", "ck", "--output-dir", "o", "--use-20k",
                            "--guidance", "5.5", "--width", "768", "--scheduler", "PNDMScheduler"])
    assert ns.use_20k is True and ns.guidance == 5.5 and ns.width == 768 and ns.scheduler == "PNDMScheduler"
    flags = {o for act in sub.choices["text-to-audio-batch"]._actions for o in act.option_strings}
    assert {"--input-json", "--output-dir", "--num-seeds", "--device"} <= flags
    ns = parser.parse_args(["text-to-audio-batch", "--input-json", "x.json", "--output-dir", "o"])
    assert ns.num_seeds == 1 and ns.device == "cuda"
    # the six reference commands stay as they are
    sub = next(a for a in cli.build_parser()._actions if a.dest == "command")
    assert len(sub.choices) == 6 and "text-to-audio" not in sub.choices


class _FakePipe:
    calls = []

    def txt2img(self, prompt, **kw):
        _FakePipe.calls.append(dict(prompt=prompt, **kw))
        n = len(kw["seed"])
        return {"images": [Image.new("RGB", (kw["width"], kw["height"]), (s % 256, 0, 0)) for s in kw["seed"]][:n]}


class _FakeConverter:
    def __init__(self, params, device):
        self.p = params

    def audio_from_spectrogram_image(self, image, apply_filters=True, max_value=30e6):
        from riffusion.util.audio_util import AudioSegment

        return AudioSegment(np.zeros((4410, 2 if self.p.stereo else 1), np.int16), self.p.sample_rate)


def _patch_front_end(monkeypatch):
    from riffusion import text_to_audio

    _FakePipe.calls.clear()
    loaded = []
    monkeypatch.setattr(text_to_audio, "_load_pipeline", lambda ck, dev: loaded.append(ck) or _FakePipe())
    monkeypatch.setattr(text_to_audio, "SpectrogramImageConverter", _FakeConverter)
    return text_to_audio, loaded


def test_text_to_audio_command_files(tmp_path, monkeypatch):
    from riffusion.spectrogram_params import SpectrogramParams

    t2a, loaded = _patch_front_end(monkeypatch)
    t2a.main(["text-to-audio", "--prompt", "church bells", "--checkpoint", "ck", "--output-dir", str(tmp_path),
              "--seed", "7", "--num-clips", "3", "--width", "768", "--use-20k"])
    assert loaded == ["ck"] and len(_FakePipe.calls) == 1
    c = _FakePipe.calls[0]
    assert c["prompt"] == "church bells" and c["seed"] == [7, 8, 9] and c["negative_prompt"] is None
    assert (c["num_inference_steps"], c["guidance_scale"], c["width"], c["height"]) == (30, 7.0, 768, 512)
    for s in (7, 8, 9):
        img = Image.open(tmp_path / f"church_bells_{s}.png")
        assert img.format == "PNG" and img.size == (768, 512)
        assert SpectrogramParams.from_exif(img.getexif()) == SpectrogramParams(min_frequency=10, max_frequency=20000,
                                                                               stereo=True)
        assert (tmp_path / f"church_bells_{s}.wav").exists()


def test_text_to_audio_batch_index_and_names(tmp_path, monkeypatch):
    t2a, loaded = _patch_front_end(monkeypatch)
    spec = {"params": [{"checkpoint": "ck1", "num_inference_steps": 20, "guidance": 6.0, "width": 640},
                       {"checkpoint": "ck1", "scheduler": "PNDMScheduler", "name": "pndm"}],
            "entries": [{"prompt": "Church bells", "seed": 42},
                        {"prompt": "electronic beats", "negative_prompt": "drums", "seed": 100}]}
    (tmp_path / "in.json").write_text(json.dumps(spec))
    out = tmp_path / "out"
    t2a.main(["text-to-audio-batch", "--input-json", str(tmp_path / "in.json"), "--output-dir", str(out),
              "--num-seeds", "2"])
    assert loaded == ["ck1"] and len(_FakePipe.calls) == 2            # one batched loop per parameter set
    c0, c1 = _FakePipe.calls
    assert c0["prompt"] == ["Church bells"] * 2 + ["electronic beats"] * 2
    assert c0["negative_prompt"] == [None, None, "drums", "drums"] and c0["seed"] == [42, 43, 100, 101]
    assert (c0["num_inference_steps"], c0["guidance_scale"], c0["width"], c0["scheduler"]) == (20, 6.0, 640,
                                                                                                "DPMSolverMultistepScheduler")
    assert (c1["num_inference_steps"], c1["guidance_scale"], c1["width"], c1["scheduler"]) == (50, 7.0, 512, "PNDMScheduler")
    index = json.loads((out / "index.json").read_text())
    assert [p["name"] for p in index["params"]] == ["params[0]", "pndm"]
    e1 = index["entries"][1]
    assert [(o["params"], o["seed"]) for o in e1["outputs"]] == [("params[0]", 100), ("params[0]", 101), ("pndm", 100),
                                                                 ("pndm", 101)]
    assert e1["image_path"] == str(out / "image_1_electronic_beats_neg_drums_seed_101.png")
    assert e1["audio_path"] == str(out / "audio_1_electronic_beats_neg_drums_seed_101.wav")
    names = sorted(p.name for p in out.iterdir())
    assert len(names) == 2 * 2 * 2 * 2 + 1                            # params x entries x seeds x (png, wav) + index
    assert "image_0_Church_bells_neg__seed_43.png" in names
    for o in e1["outputs"]:
        assert Image.open(o["image_path"]).size == ((640 if o["params"] == "params[0]" else 512), 512)


def test_dpmpp_step_rejects_bad_arguments(native_lib):
    """argument checks of the C-ABI return RF_ERR_INVALID before anything touches the device"""
    import ctypes

    p = ctypes.c_void_p(16)
    args = dict(eps_pair=p, n=8, guidance=7.0, sample=p, x0_prev=None, sigma_s=0.9, alpha_s=0.1, c_x=1.0, c_0=-0.1,
                inv_r0=0.0, c_d1=0.0, x0_out=ctypes.c_void_p(32), prev_sample=ctypes.c_void_p(48), stream=None)
    for bad in (dict(eps_pair=None), dict(sample=None), dict(x0_out=None), dict(prev_sample=None), dict(n=0), dict(n=-3),
                dict(alpha_s=0.0), dict(alpha_s=float("nan")), dict(x0_out=ctypes.c_void_p(48))):
        assert native_lib.rf_cfg_dpmpp_step_f16(*{**args, **bad}.values()) == 1, bad
    assert native_lib.rf_vae_image_to_u8_f32scale(None, 1, 8, 8, p, None) == 1
    assert native_lib.rf_vae_image_to_u8_f32scale(p, 1, 0, 8, p, None) == 1
