"""Audio to audio on the host: the Pillow BICUBIC restatement (tests/resample_oracle.py) against Pillow and against the
tables librf_b200 builds, the img2img timestep arithmetic (SURVEY Appendix D), the img2img control flow and generator
draw order against an oracle loop with the device ops replaced by torch stand-ins, clip slicing, the
`riffusion.audio_to_audio` front end with the pipeline faked, and argument errors.  No GPU, no kernels."""
import ctypes
import types

import numpy as np
import pytest
import torch
from PIL import Image

import resample_oracle as ro
from riffusion.riffusion_pipeline import RiffusionPipeline
from riffusion.scheduler_b200 import DPMSolverMultistepSchedulerB200, PNDMSchedulerB200
from riffusion.spectrogram_params import SpectrogramParams
from test_txt2img_cpu import _FakeUNet, _fake_ops, _model

# clip widths of 3 .. 20 s spectrograms and their 32-stride widths
WIDTHS = [(301, 320), (401, 416), (501, 512), (601, 608), (701, 704), (1001, 1024), (300, 1024)]


# ------------------------------------------------------------------------------------------------ Pillow BICUBIC
@pytest.mark.parametrize("w_in,w_out", WIDTHS)
def test_resample_oracle_equals_pillow(w_in, w_out):
    rng = np.random.default_rng(w_in)
    a = rng.integers(0, 256, (24, w_in, 3), dtype=np.uint8)
    up = np.asarray(Image.fromarray(a).resize((w_out, 24), Image.BICUBIC))
    assert np.array_equal(ro.resize(a, w_out, 24), up)
    down = np.asarray(Image.fromarray(up).resize((w_in, 24), Image.BICUBIC))
    assert np.array_equal(ro.resize(up, w_in, 24), down)


def test_resample_oracle_vertical_and_same_size():
    rng = np.random.default_rng(1)
    a = rng.integers(0, 256, (500, 37, 3), dtype=np.uint8)
    for w, h in ((37, 512), (64, 512), (37, 250), (37, 500)):
        want = np.asarray(Image.fromarray(a).resize((w, h), Image.BICUBIC))
        assert np.array_equal(ro.resize(a, w, h), want), (w, h)
    assert np.array_equal(ro.resize(a, 37, 500), a)
    # a spectrogram-like image (smooth, mostly dark) through the clip round trip
    x = np.linspace(0, 1, 501)[None, :, None] * np.linspace(0, 1, 512)[:, None, None]
    img = np.repeat((255 * x ** 3).astype(np.uint8), 3, axis=2)
    up = np.asarray(Image.fromarray(img).resize((512, 512), Image.BICUBIC))
    assert np.array_equal(ro.resize(img, 512, 512), up)
    assert np.array_equal(ro.resize(up, 501, 512), np.asarray(Image.fromarray(up).resize((501, 512), Image.BICUBIC)))


@pytest.mark.parametrize("w_in,w_out", WIDTHS + [(500, 512), (512, 250)])
def test_resample_tables_equal_native_tables(native_lib, w_in, w_out):
    from riffusion import tc_ops

    for n_in, n_out in ((w_in, w_out), (w_out, w_in)):
        b_ref, k_ref = ro.coeffs(n_in, n_out)
        b, k = tc_ops.resample_coeffs(n_in, n_out)
        assert np.array_equal(b, b_ref) and np.array_equal(k, k_ref), (n_in, n_out)


# ------------------------------------------------------------------------------------------------ img2img timesteps
DPM_TS_25 = [999, 959, 919, 879, 839, 799, 759, 719, 679, 639, 599, 559, 519, 480, 440, 400, 360, 320, 280, 240, 200, 160,
             120, 80, 40]


@pytest.mark.parametrize("offset", [1, 0])
def test_img2img_timesteps_dpm_25_steps(offset):
    s = DPMSolverMultistepSchedulerB200(steps_offset=offset)
    assert s.config["steps_offset"] == offset
    # strength: (t_start, evaluations) -- equal for both offsets except at 1.0, where the clamp bites
    want = {0.4: (15, 10), 0.55: (12, 13), 0.75: (7, 18), 1.0: (1, 24) if offset else (0, 25)}
    for strength, (t_start, n) in want.items():
        got_start, ts, t_noise = s.img2img_timesteps(25, strength)
        assert (got_start, len(ts)) == (t_start, n), strength
        assert ts.tolist() == DPM_TS_25[t_start:] and t_noise == DPM_TS_25[t_start]
    assert s.img2img_timesteps(25, 0.55)[2] == 519
    for bad in (0.02, 0.0):
        with pytest.raises(ValueError, match="no denoising step"):
            s.img2img_timesteps(25, bad)
    for bad in (-0.1, 1.5):
        with pytest.raises(ValueError, match="strength"):
            s.img2img_timesteps(25, bad)


@pytest.mark.parametrize("offset", [1, 0])
def test_img2img_timesteps_pndm_50_steps(offset):
    s = PNDMSchedulerB200(steps_offset=offset)
    s.set_timesteps(50)
    full = s.timesteps.tolist()
    assert len(full) == 51 and full[:3] == [980 + offset, 960 + offset, 960 + offset]
    want = {0.4: (30, 21), 0.55: (23, 28), 0.75: (13, 38), 1.0: (1, 50) if offset else (0, 51)}
    for strength, (t_start, n) in want.items():
        got_start, ts, t_noise = s.img2img_timesteps(50, strength)
        assert (got_start, len(ts)) == (t_start, n), strength
        assert ts.tolist() == full[t_start:] and t_noise == full[t_start]
    # PLMS keeps its duplicated timestep: even strength 0 leaves one evaluation
    assert len(s.img2img_timesteps(50, 0.0)[1]) == 1


def test_add_noise_scalars_are_fp16_tensor_ops():
    for sched in (DPMSolverMultistepSchedulerB200(), PNDMSchedulerB200()):
        ac = sched.alphas_cumprod.to(torch.float16)
        for t in (999, 981, 559, 519, 400, 40, 1, 0):
            s, s1 = sched.add_noise_scalars(t)
            assert s == float(ac[t] ** 0.5) and s1 == float((1 - ac[t]) ** 0.5), t
            assert float(np.float16(s)) == s and float(np.float16(s1)) == s1


# ------------------------------------------------------------------------------------------------ img2img control flow
def _r16(v):
    return v.to(torch.float16).to(torch.float32)


def _add_noise_stand_in(x, n, s, s1):
    return _r16(_r16(s * x.float()) + _r16(s1 * n.float())).half()


class _FakeVae:
    config = types.SimpleNamespace(block_out_channels=[1, 1, 1, 1])

    def encode_moments(self, image):
        m = torch.nn.functional.avg_pool2d(image.float(), 8)
        return torch.cat([m, -m[:, :1]], dim=1).half(), torch.full_like(torch.cat([m, m[:, :1]], dim=1), -3.0).half()


def _img2img_pipe(monkeypatch):
    from riffusion import tc_ops

    _fake_ops(monkeypatch)
    monkeypatch.setattr(tc_ops, "add_noise_f16_seq", _add_noise_stand_in)
    pipe = RiffusionPipeline(vae=_FakeVae(), unet=_FakeUNet(), device="cpu")
    pipe.use_cuda_graph = False
    return pipe


def _images(n, w=128, h=64):
    rng = np.random.default_rng(n)
    return [Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)) for _ in range(n)]


def _oracle_start(images, seeds, sched, steps, strength):
    """prepare_latents of img2img 0.9: one generator per clip, posterior sample first, then the fp16 noise"""
    from riffusion.riffusion_pipeline import preprocess_image

    lats = []
    for im, sd in zip(images, seeds):
        x = preprocess_image(im).half()
        mean, logvar = _FakeVae().encode_moments(x)
        g = torch.Generator().manual_seed(sd)
        std = torch.exp(0.5 * torch.clamp(logvar, -30.0, 20.0))
        post = (mean.float() + std.float() * torch.randn(mean.shape, generator=g)).half()
        lat = 0.18215 * post
        noise = torch.randn(lat.shape, generator=g, dtype=torch.float16)
        _, ts, t_noise = sched.img2img_timesteps(steps, strength)
        s, s1 = sched.add_noise_scalars(t_noise)
        lats.append(_add_noise_stand_in(lat, noise, s, s1))
    return torch.cat(lats), ts


def test_img2img_control_flow_matches_oracle_loop(monkeypatch):
    """encode -> one generator per clip (posterior, then noise) -> fp16 add_noise at timesteps[t_start] -> CFG loop over
    timesteps[t_start:] with a first-order start, against the fp64 DPM oracle / the PNDM oracle"""
    from oracle import unet_oracle as uo
    from txt2img_oracle import DPMSolverMultistepSchedulerOracle

    images, seeds = _images(2), [5, 9]
    torch.manual_seed(3)
    text, uncond = torch.randn(2, 77, 16).half(), torch.randn(1, 77, 16).half()
    for scheduler, steps, strength, n_want in (("DPMSolverMultistepScheduler", 25, 0.55, 13),
                                               ("PNDMScheduler", 50, 0.75, 38),
                                               ("DPMSolverMultistepScheduler", 25, 1.0, 24)):
        pipe = _img2img_pipe(monkeypatch)
        before = pipe.scheduler
        out = pipe.img2img(init_image=images, seed=seeds, strength=strength, num_inference_steps=steps,
                           guidance_scale=7.0, scheduler=scheduler, text_embeddings=text, uncond_embeddings=uncond,
                           output_type="latent")
        assert pipe.scheduler is before and out["images"] is None
        sched = DPMSolverMultistepSchedulerB200() if scheduler.startswith("DPM") else PNDMSchedulerB200()
        x0, ts = _oracle_start(images, seeds, sched, steps, strength)
        assert out["n_unet_evals"] == n_want == len(ts) == len(pipe.unet.calls)
        assert [t for _, t in pipe.unet.calls] == ts.tolist()
        oracle = DPMSolverMultistepSchedulerOracle() if scheduler.startswith("DPM") else uo.PNDMSchedulerOracle()
        oracle.set_timesteps(steps)
        ctx = torch.cat([uncond.float().expand(2, -1, -1), text.float()])
        x = x0.float()
        for t in ts.tolist():
            eu, et = _model(torch.cat([x, x]), t, ctx).chunk(2)
            x = oracle.step(eu + 7.0 * (et - eu), t, x)
        err = float((out["latents_unscaled"].float() - x).norm() / x.norm())
        print(f"img2img {scheduler} {steps} steps strength {strength}: fp16 stand-ins vs oracle loop rel L2 {err:.2e}")
        assert err < 2e-2, (scheduler, strength, err)
        assert torch.equal(out["latents"], (1.0 / 0.18215) * out["latents_unscaled"])


def test_img2img_draw_order_and_batching(monkeypatch):
    """the first UNet input is exactly add_noise(0.18215 * posterior, noise) with both draws from one generator per clip;
    a clip list equals single calls; one image broadcasts over a seed list; injected noise replaces the second draw"""
    images, seeds = _images(3), [1, 2, 3]
    torch.manual_seed(4)
    text, uncond = torch.randn(3, 77, 16).half(), torch.randn(1, 77, 16).half()
    firsts = []

    def record(x, t, encoder_hidden_states=None, **kw):
        firsts.append(x[: x.shape[0] // 2].clone())
        return types.SimpleNamespace(sample=_model(x, int(t), encoder_hidden_states).to(torch.float16))

    pipe = _img2img_pipe(monkeypatch)
    pipe.unet = record
    kw = dict(strength=0.55, num_inference_steps=25, guidance_scale=7.0, uncond_embeddings=uncond, output_type="latent")
    batch = pipe.img2img(init_image=images, seed=seeds, text_embeddings=text, **kw)
    x0, _ = _oracle_start(images, seeds, DPMSolverMultistepSchedulerB200(), 25, 0.55)
    assert torch.equal(firsts[0], x0)
    for i in range(3):
        single = pipe.img2img(init_image=images[i], seed=seeds[i], text_embeddings=text[i:i + 1], **kw)
        assert torch.equal(single["latents_unscaled"], batch["latents_unscaled"][i:i + 1])
    firsts.clear()
    pipe.img2img(init_image=images[0], seed=[1, 7], text_embeddings=text[:2], **kw)
    x0, _ = _oracle_start([images[0]] * 2, [1, 7], DPMSolverMultistepSchedulerB200(), 25, 0.55)
    assert torch.equal(firsts[0], x0)
    noise = torch.randn(3, 4, 8, 16).half()
    firsts.clear()
    pipe.img2img(init_image=images, seed=seeds, text_embeddings=text, noise=noise, **kw)
    assert not torch.equal(firsts[0], x0[:1].expand(3, -1, -1, -1))
    with pytest.raises(ValueError, match="batch size"):
        pipe.img2img(init_image=images[:2], seed=seeds, text_embeddings=text, **kw)


def test_img2img_argument_errors(monkeypatch):
    pipe = _img2img_pipe(monkeypatch)
    u8 = torch.zeros(1, 512, 416, 3, dtype=torch.uint8)                    # a 4 s clip at the 32-stride width
    with pytest.raises(NotImplementedError, match="multiples of 64"):
        pipe.img2img("a", init_images_u8=u8)
    with pytest.raises(ValueError, match="multiples of 32"):
        pipe.img2img("a", init_images_u8=torch.zeros(1, 512, 501, 3, dtype=torch.uint8))
    with pytest.raises(ValueError, match="exactly one"):
        pipe.img2img("a")
    with pytest.raises(ValueError, match="no denoising step"):
        pipe.img2img("a", init_image=_images(1)[0], strength=0.02, num_inference_steps=25)
    with pytest.raises(NotImplementedError, match="EulerDiscreteScheduler"):
        pipe.img2img("a", init_image=_images(1)[0], scheduler="EulerDiscreteScheduler")


def test_audio_to_audio_clips_argument_errors():
    pipe = RiffusionPipeline(vae=None, unet=None, device="cpu")
    mono = types.SimpleNamespace(p=SpectrogramParams(min_frequency=0, max_frequency=10000))
    for seconds in (4, 6, 9):
        with pytest.raises(NotImplementedError, match="multiples of 64"):
            pipe.audio_to_audio_clips(torch.zeros(1, 44100 * seconds), converter=mono, prompt="a")
    stereo_20k = types.SimpleNamespace(p=SpectrogramParams(min_frequency=10, max_frequency=20000, stereo=True))
    with pytest.raises(NotImplementedError, match="20 kHz"):
        pipe.audio_to_audio_clips(torch.zeros(1, 220500), converter=stereo_20k, prompt="a")
    # 3, 5, 7, 8 and 10 s clips pass the size check (and then need a CUDA tensor)
    from riffusion._native import NativeError

    for seconds in (3, 5, 7, 8, 10):
        with pytest.raises(NativeError, match="CUDA"):
            pipe.audio_to_audio_clips(torch.zeros(1, 44100 * seconds), converter=mono, prompt="a")


# ------------------------------------------------------------------------------------------------ track slicing
def test_clip_start_times_reference_formula():
    from riffusion.audio_to_audio import clip_start_times

    assert np.allclose(clip_start_times(0.0, 20.0), [0.0, 4.8, 9.6, 14.4])
    assert len(clip_start_times(0.0, 180.0)) == 37
    assert np.allclose(clip_start_times(2.0, 10.2), [2.0, 6.8])
    assert np.allclose(clip_start_times(0.0, 12.0, 3.0, 0.5), 0.0 + np.arange(0, 9.0, 2.5))
    assert len(clip_start_times(0.0, 5.0)) == 0


def test_slice_audio_into_clips_pads_the_last_clip():
    from riffusion.audio_to_audio import slice_audio_into_clips
    from riffusion.util.audio_util import AudioSegment

    rng = np.random.default_rng(0)
    track = rng.integers(-3000, 3000, (12 * 44100, 1)).astype(np.int16)
    seg = AudioSegment(track, 44100)
    clips = slice_audio_into_clips(seg, [0.0, 4.8, 9.6], 5.0)
    assert [c.frame_count() for c in clips] == [220500.0] * 3
    for c, t in zip(clips, (0.0, 4.8, 9.6)):
        a = int(int(t * 1000) * 44.1)
        n = min(220500, track.shape[0] - a)
        assert np.array_equal(c._s[:n], track[a:a + n])
    assert not clips[2]._s[12 * 44100 - 423360:].any()          # 2.6 s of silence after the end of the track


# ------------------------------------------------------------------------------------------------ front end
def test_audio_to_audio_parser():
    from riffusion import audio_to_audio, cli

    parser = cli.build_parser(audio_to_audio.COMMANDS, prog="riffusion.audio_to_audio")
    sub = next(a for a in parser._actions if a.dest == "command")
    assert set(sub.choices) == {"audio-to-audio"}
    flags = {o for act in sub.choices["audio-to-audio"]._actions for o in act.option_strings}
    assert {"--audio", "--prompt", "--output", "--checkpoint", "--negative-prompt", "--seed", "--denoising",
            "--num-inference-steps", "--guidance", "--scheduler", "--start-time-s", "--duration-s", "--clip-duration-s",
            "--overlap-duration-s", "--prompt-b", "--seed-b", "--denoising-b", "--image-dir", "--device"} <= flags
    ns = parser.parse_args(["audio-to-audio", "--audio", "a.wav", "--prompt", "p", "--output", "o.wav"])
    assert (ns.seed, ns.denoising, ns.num_inference_steps, ns.guidance, ns.scheduler, ns.start_time_s, ns.duration_s,
            ns.clip_duration_s, ns.overlap_duration_s, ns.prompt_b, ns.seed_b, ns.image_dir) == (
        42, 0.55, 25, 7.0, "DPMSolverMultistepScheduler", 0.0, 20.0, 5.0, 0.2, "", None, "")
    ns = parser.parse_args(["audio-to-audio", "--audio", "a.wav", "--prompt", "p", "--output", "o.wav", "--prompt-b",
                            "q", "--seed-b", "7", "--denoising-b", "0.6", "--start-time-s", "1.5"])
    assert (ns.prompt_b, ns.seed_b, ns.denoising_b, ns.start_time_s) == ("q", 7, 0.6, 1.5)


class _FakeA2APipe:
    def __init__(self):
        self.calls = []

    def audio_to_audio_clips(self, waveforms, **kw):
        self.calls.append(dict(n=waveforms.shape[0], samples=waveforms.shape[1], **kw))
        B = waveforms.shape[0]
        g = torch.Generator().manual_seed(B)
        return dict(source_images=torch.zeros(B, 512, 501, 3, dtype=torch.uint8),
                    images=torch.full((B, 512, 501, 3), 7, dtype=torch.uint8),
                    waveform=torch.randn(B, 441 * 500, generator=g))

    def riffuse_batch(self, inputs, init_images):
        self.calls.append(dict(inputs=inputs, sizes=[im.size for im in init_images]))
        return [Image.new("RGB", (512, 512), (9, 9, 9)) for _ in inputs]


class _FakeImageConverter:
    def __init__(self, params, device):
        self.p = params

    def spectrogram_image_from_audio(self, segment):
        return Image.new("RGB", (1 + int(segment.frame_count()) // 441, 512))

    def audio_from_spectrogram_image(self, image, apply_filters=True, max_value=30e6):
        from riffusion.util.audio_util import AudioSegment

        return AudioSegment(np.full((441 * (image.width - 1), 1), 100, np.int16), 44100)


def _write_wav(path, seconds, rate=44100, channels=2):
    from scipy.io import wavfile

    rng = np.random.default_rng(0)
    wavfile.write(path, rate, rng.integers(-8000, 8000, (int(seconds * rate), channels)).astype(np.int16))


def _patch(monkeypatch, pipe):
    from riffusion import audio_to_audio

    monkeypatch.setattr(audio_to_audio, "_load_pipeline", lambda ck, dev: pipe)
    monkeypatch.setattr(audio_to_audio, "SpectrogramConverter", lambda params, device: types.SimpleNamespace(p=params))
    monkeypatch.setattr(audio_to_audio, "SpectrogramImageConverter", _FakeImageConverter)
    return audio_to_audio


def test_audio_to_audio_command_length_and_images(tmp_path, monkeypatch):
    from scipy.io import wavfile

    pipe = _FakeA2APipe()
    a2a = _patch(monkeypatch, pipe)
    _write_wav(tmp_path / "in.wav", 10.2)
    out = tmp_path / "out.wav"
    a2a.main(["audio-to-audio", "--audio", str(tmp_path / "in.wav"), "--prompt", "jazz", "--output", str(out),
              "--seed", "3", "--denoising", "0.4", "--scheduler", "PNDMScheduler", "--image-dir", str(tmp_path / "img"),
              "--device", "cpu"])
    (c,) = pipe.calls
    assert (c["n"], c["samples"], c["prompt"], c["seed"], c["strength"], c["scheduler"], c["guidance_scale"],
            c["num_inference_steps"], c["negative_prompt"]) == (2, 220500, "jazz", 3, 0.4, "PNDMScheduler", 7.0, 25, None)
    rate, data = wavfile.read(out)
    assert rate == 44100 and data.ndim == 1 and data.shape[0] == 2 * 220500 - 8820     # n clip - (n - 1) overlap
    for i in range(2):
        for kind in ("source", "riffed"):
            img = Image.open(tmp_path / "img" / f"clip_{i}_{kind}.png")
            assert img.size == (501, 512)
            assert SpectrogramParams.from_exif(img.getexif()) == SpectrogramParams(max_frequency=10000)


def test_audio_to_audio_batches_of_32_clips(monkeypatch):
    from riffusion.util.audio_util import AudioSegment

    pipe = _FakeA2APipe()
    a2a = _patch(monkeypatch, pipe)
    seg = AudioSegment(np.zeros((180 * 44100, 1), np.int16), 44100)
    result, starts, sources, riffed = a2a.audio_to_audio(seg, pipe=pipe, prompt="p", duration_s=180.0, device="cpu")
    assert len(starts) == 37 and [c["n"] for c in pipe.calls] == [32, 5] and len(riffed) == len(sources) == 37
    assert result.frame_count() == 37 * 220500 - 36 * 8820


def test_audio_to_audio_interpolation(tmp_path, monkeypatch):
    from scipy.io import wavfile

    pipe = _FakeA2APipe()
    a2a = _patch(monkeypatch, pipe)
    _write_wav(tmp_path / "in.wav", 15.0, channels=1)
    out = tmp_path / "out.wav"
    a2a.main(["audio-to-audio", "--audio", str(tmp_path / "in.wav"), "--prompt", "jazz", "--output", str(out),
              "--prompt-b", "rock", "--seed-b", "9", "--device", "cpu"])
    (c,) = pipe.calls
    inputs = c["inputs"]
    assert [i.alpha for i in inputs] == [0.0, 0.5, 1.0] and c["sizes"] == [(512, 512)] * 3
    assert (inputs[0].start.prompt, inputs[0].start.seed, inputs[0].start.denoising) == ("jazz", 42, 0.55)
    assert (inputs[0].end.prompt, inputs[0].end.seed, inputs[0].end.denoising) == ("rock", 9, 0.55)
    assert inputs[0].num_inference_steps == 25 and inputs[0].start.guidance == 7.0
    rate, data = wavfile.read(out)
    assert data.shape[0] == 3 * 220500 - 2 * 8820


def test_audio_to_audio_rejects_other_sample_rates(tmp_path, monkeypatch):
    from riffusion.util.audio_util import AudioSegment

    pipe = _FakeA2APipe()
    a2a = _patch(monkeypatch, pipe)
    _write_wav(tmp_path / "in.wav", 6.0, rate=22050)
    with pytest.raises(ValueError, match="44100 Hz"):
        a2a.main(["audio-to-audio", "--audio", str(tmp_path / "in.wav"), "--prompt", "p", "--output",
                  str(tmp_path / "o.wav"), "--device", "cpu"])
    with pytest.raises(ValueError, match="44100 Hz"):
        a2a.audio_to_audio(AudioSegment(np.zeros((48000 * 6, 1), np.int16), 48000), pipe=pipe, prompt="p")
    with pytest.raises(ValueError, match="no clip"):
        a2a.audio_to_audio(AudioSegment(np.zeros((44100 * 4, 1), np.int16), 44100), pipe=pipe, prompt="p")
    assert pipe.calls == []


# ------------------------------------------------------------------------------------------------ C-ABI arguments
def test_image_entries_reject_bad_arguments(native_lib):
    """argument checks of the C-ABI return RF_ERR_INVALID before anything touches the device"""
    p, q = ctypes.c_void_p(16), ctypes.c_void_p(32)
    args = dict(x=p, B=1, H_in=8, W_in=8, H_out=8, W_out=16, y=q, stream=None)
    for bad in (dict(x=None), dict(y=None), dict(y=p), dict(B=0), dict(H_in=0), dict(W_in=-1), dict(H_out=0),
                dict(W_out=0)):
        assert native_lib.rf_resample_u8(*{**args, **bad}.values()) == 1, bad
    k = ctypes.c_int()
    assert native_lib.rf_resample_coeffs(0, 5, ctypes.byref(k), None, None) == 1
    assert native_lib.rf_resample_coeffs(5, 0, ctypes.byref(k), None, None) == 1
    assert native_lib.rf_resample_coeffs(5, 7, None, None, None) == 1
    assert native_lib.rf_resample_coeffs(501, 512, ctypes.byref(k), None, None) == 0 and k.value == 5
    assert native_lib.rf_resample_coeffs(512, 250, ctypes.byref(k), None, None) == 0 and k.value == 11
    for bad in ((None, 1, 8, 8, q), (p, 0, 8, 8, q), (p, 1, 8, 0, q), (p, 1, 8, 8, None)):
        assert native_lib.rf_image_u8_to_f16(*bad, None) == 1, bad
    s, s1 = 0.5, 0.75                                                 # fp16 values
    for bad in ((None, p, s, s1, 8, q), (p, None, s, s1, 8, q), (p, p, s, s1, 8, None), (p, p, s, s1, 0, q),
                (p, p, 0.1, s1, 8, q), (p, p, s, float("nan"), 8, q), (p, p, s, 70000.0, 8, q)):
        assert native_lib.rf_add_noise_f16_seq(*bad, None) == 1, bad
