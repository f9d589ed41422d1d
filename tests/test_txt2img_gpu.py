"""Text to image / text to audio on the B200: rf_cfg_dpmpp_step_f16 against the reference's own torch-CUDA fp16 op
sequence, the txt2img uint8 rounding, the denoising loop against the fp32 oracle loop and its fp16-storage emulation
(tests/txt2img_oracle.py), CUDA-graph replay, seed-list batching, `text_to_audio_clips` end to end and both
`riffusion.text_to_audio` commands on a small random-init pipeline."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DPM = "DPMSolverMultistepScheduler"


def rel_l2(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm())


def _check_vs_floor(got, ref32, emul, what, floor_factor=1.25):
    """tests/test_parity_bench_gpu.py's bars: kernels vs fp32 oracle within floor_factor x the fp16-storage floor
    (emulation vs fp32), kernels vs emulation within 1.25 x the spread of two independent fp16 evaluations"""
    e_k, e_f, e_o = rel_l2(got, emul), rel_l2(emul, ref32), rel_l2(got, ref32)
    print(f"{what}: kernels vs fp32 oracle {e_o:.3e} | fp16-storage floor (emulation vs fp32) {e_f:.3e} | "
          f"kernels vs emulation {e_k:.3e}")
    assert torch.isfinite(got.float()).all()
    assert e_o <= floor_factor * e_f + 1e-4, f"{what}: kernels vs fp32 {e_o:.3e}, floor {e_f:.3e}"
    spread = 2 ** 0.5 * floor_factor * e_f
    assert e_k <= 1.25 * spread + 1e-4, f"{what}: kernels vs emulation {e_k:.3e}, spread {spread:.3e}"


@pytest.fixture(scope="module", autouse=True)
def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


def _round_params(m):
    with torch.no_grad():
        for p in m.parameters():
            p.copy_(p.half().float())
    return m


@pytest.fixture(scope="module")
def sd15(native_lib):
    from oracle import unet_oracle as uo
    from riffusion.unet_b200 import UNetB200

    oracle = _round_params(uo.init_weights_(uo.UNet2DConditionOracle(), seed=0)).cuda().eval()
    return oracle, UNetB200(oracle.state_dict(), device="cuda")


@pytest.fixture(scope="module")
def small_unet(native_lib):
    from oracle import unet_oracle as uo
    from riffusion.unet_b200 import UNetB200

    cfg = dict(block_out_channels=(64, 128, 128, 128), heads=4, cross_attention_dim=64)
    oracle = _round_params(uo.init_weights_(uo.UNet2DConditionOracle(**cfg), seed=21)).cuda().eval()
    return oracle, UNetB200(oracle.state_dict(), device="cuda", block_out_channels=cfg["block_out_channels"], heads=4)


@pytest.fixture(scope="module")
def vae_pair(native_lib):
    from oracle.unet_oracle import init_weights_
    from oracle.vae_oracle import AutoencoderKLOracle
    from riffusion.vae_b200 import VaeB200

    oracle = _round_params(init_weights_(AutoencoderKLOracle(), seed=5, std=0.03)).cuda().eval()
    return oracle, VaeB200(oracle.state_dict(), device="cuda")


class _StubTextEncoder:
    def __init__(self, dim=64):
        g = torch.Generator().manual_seed(123)
        self.table = torch.randn(49408, dim, generator=g).cuda()
        self.pos = torch.randn(77, dim, generator=g).cuda() * 0.3

    def __call__(self, ids):
        return ((self.table[ids.cuda()] + self.pos[None]).half(),)


def _small_pipe(small_unet, vae_pair):
    import sys
    from pathlib import Path

    from riffusion.riffusion_pipeline import RiffusionPipeline

    sys.path.insert(0, str(Path(__file__).parent / "golden"))
    from prompt_stub import StubTokenizer

    return RiffusionPipeline(vae=vae_pair[1], unet=small_unet[1], text_encoder=_StubTextEncoder(), tokenizer=StubTokenizer(),
                             device="cuda")


# ----------------------------------------------------------------------------------------------- the fused step
def _reference_step(s, eps_pair, g, x, m1, i):
    """DPMSolverMultistepScheduler.step as the reference runs it: fp16 CUDA tensors, 0-dim fp32 CPU scalars"""
    ts = s.timesteps.tolist()
    t, s0 = (ts[i + 1] if i + 1 < len(ts) else 0), ts[i]
    n = x.shape[0]
    eu, et = eps_pair[:n], eps_pair[n:]
    e = eu + g * (et - eu)
    m0 = (x - s.sigma_t[s0] * e) / s.alpha_t[s0]
    lam, al, sg = s.lambda_t, s.alpha_t, s.sigma_t
    h = lam[t] - lam[s0]
    if m1 is None:
        return m0, (sg[t] / sg[s0]) * x - (al[t] * (torch.exp(-h) - 1.0)) * m0
    r0 = (lam[s0] - lam[ts[i - 1]]) / h
    d1 = (1.0 / r0) * (m0 - m1)
    return m0, (sg[t] / sg[s0]) * x - (al[t] * (torch.exp(-h) - 1.0)) * m0 - 0.5 * (al[t] * (torch.exp(-h) - 1.0)) * d1


@torch.no_grad()
def test_dpmpp_step_kernel_bit_exact_vs_reference_ops(native_lib):
    from riffusion import tc_ops as ops
    from riffusion.scheduler_b200 import DPMSolverMultistepSchedulerB200

    s = DPMSolverMultistepSchedulerB200()
    s.set_timesteps(30)
    torch.manual_seed(3)
    # odd n: 16-byte groups with element-wise loads of the (misaligned) text half, then a 5-element tail; n % 8 == 0: all
    # six streams in 16-byte accesses
    for n in (3 * 16384 + 5, 2 * 4 * 64 * 64):
        for g in (1.0, 7.0):
            for i, second in ((0, False), (1, True), (17, True), (29, True)):
                eps_pair = torch.randn(2 * n, device="cuda").half()
                x = (torch.randn(n, device="cuda") * 3).half()
                m1 = torch.randn(n, device="cuda").half() if second else None
                m0_ref, xt_ref = _reference_step(s, eps_pair, g, x, m1, i)
                s.lower_order_nums = 2 if second else 0
                c = s.coefficients(s.timesteps[i])
                assert c["second"] == second
                xt = x.clone()
                m0, out = ops.cfg_dpmpp_step(eps_pair, g, xt, m1, c["sigma_s"], c["alpha_s"], c["c_x"], c["c_0"], c["inv_r0"],
                                             c["c_d1"], out=xt)                         # in place
                assert out.data_ptr() == xt.data_ptr()
                bad_m0 = int((m0.view(torch.int16) != m0_ref.view(torch.int16)).sum())
                bad_xt = int((xt.view(torch.int16) != xt_ref.view(torch.int16)).sum())
                print(f"rf_cfg_dpmpp_step_f16 n={n} g={g} step {i} ({'2nd' if second else '1st'} order): "
                      f"x0 differs in {bad_m0}, x_t in {bad_xt} of {n} elements")
                assert bad_m0 == 0 and bad_xt == 0


@torch.no_grad()
def test_dpmpp_exact_denoiser_through_the_kernel(native_lib):
    """true eps of x = a_s x0* + s_s eps* at every step: the trajectory stays on a_t x0* + s_t eps* (fp16 storage)"""
    from riffusion.scheduler_b200 import DPMSolverMultistepSchedulerB200

    for steps in (10, 30):
        s = DPMSolverMultistepSchedulerB200()
        s.set_timesteps(steps)
        a, sg = s.alpha_t.double(), s.sigma_t.double()
        g = torch.Generator(device="cuda").manual_seed(steps)
        x0s = torch.randn(2, 4, 64, 64, generator=g, device="cuda", dtype=torch.float64)
        epss = torch.randn(2, 4, 64, 64, generator=g, device="cuda", dtype=torch.float64)
        ts = s.timesteps.tolist()
        x = (float(a[ts[0]]) * x0s + float(sg[ts[0]]) * epss).half()
        worst = 0.0
        for i, t in enumerate(ts):
            eps = ((x.double() - float(a[t]) * x0s) / float(sg[t])).half()
            x = s.step_cfg(torch.cat([eps, eps]), 7.0, t, x)
            t_next = ts[i + 1] if i + 1 < len(ts) else 0
            worst = max(worst, rel_l2(x, float(a[t_next]) * x0s + float(sg[t_next]) * epss))
        print(f"exact denoiser, {steps} DPM steps through rf_cfg_dpmpp_step_f16: worst rel L2 off the trajectory {worst:.2e}")
        assert worst < 3e-3


def test_vae_to_u8_f32scale_bit_exact(native_lib):
    from riffusion import tc_ops as ops

    torch.manual_seed(9)
    for img in ((torch.rand(2, 3, 64, 512, device="cuda") * 2.6 - 1.3).half(),
                torch.linspace(-1.2, 1.2, 3 * 256 * 256, device="cuda").reshape(1, 3, 256, 256).half()):
        want = ((img / 2 + 0.5).clamp(0, 1).float() * 255).round().to(torch.uint8).permute(0, 2, 3, 1)
        got = ops.vae_image_to_u8(img, fp32_scale=True)
        fp16_path = ops.vae_image_to_u8(img)
        print(f"uint8 rounding: fp32 vs fp16 scale differ on {100 * (got != fp16_path).float().mean():.2f} % of values")
        assert torch.equal(got, want)


# ----------------------------------------------------------------------------------------------- loop parity
def _loop_case(oracle, unet, scheduler, steps, width, B, ctx_dim, seed):
    from oracle import unet_oracle as uo
    from riffusion.riffusion_pipeline import RiffusionPipeline
    from txt2img_oracle import DPMSolverMultistepSchedulerOracle, txt2img_loop, txt2img_loop_emul

    pipe = RiffusionPipeline(vae=None, unet=unet, device="cuda")
    torch.manual_seed(seed)
    text = torch.randn(B, 77, ctx_dim, device="cuda").half()
    uncond = torch.randn(1, 77, ctx_dim, device="cuda").half()
    seeds = [seed + 10 * i for i in range(B)]
    out = pipe.txt2img(text_embeddings=text, uncond_embeddings=uncond, seed=seeds, num_inference_steps=steps,
                       guidance_scale=7.0, width=width, height=512, scheduler=scheduler, output_type="latent")
    lat = torch.cat([torch.randn((1, 4, 64, width // 8), generator=torch.Generator(device="cuda").manual_seed(sd),
                                 device="cuda", dtype=torch.float16) for sd in seeds])
    n_want = steps + 1 if scheduler == "PNDMScheduler" else steps
    assert out["n_unet_evals"] == n_want and out["latents_unscaled"].shape == (B, 4, 64, width // 8)
    refs, emuls = [], []
    for i in range(B):
        sch = DPMSolverMultistepSchedulerOracle() if scheduler == DPM else uo.PNDMSchedulerOracle()
        r, n = txt2img_loop(oracle, sch, text[i:i + 1].float(), uncond.float(), lat[i:i + 1].float(), steps, 7.0)
        e, n2 = txt2img_loop_emul(oracle, scheduler, text[i:i + 1], uncond, lat[i:i + 1], steps, 7.0)
        assert n == n2 == n_want
        refs.append(r)
        emuls.append(e)
    return pipe, out, torch.cat(refs), torch.cat(emuls), text, uncond, lat


@torch.no_grad()
def test_txt2img_full_size_768_wide_10_dpm_steps(sd15):
    oracle, unet = sd15
    _, out, ref, emul, *_ = _loop_case(oracle, unet, DPM, 10, 768, 2, 768, 70)
    _check_vs_floor(out["latents_unscaled"], ref, emul, "txt2img SD-1.5 64x96 latents, 2 clips, 10 DPM steps")


@torch.no_grad()
def test_txt2img_small_unet_30_dpm_steps_and_graph_replay(small_unet):
    oracle, unet = small_unet
    pipe, out, ref, emul, text, uncond, lat = _loop_case(oracle, unet, DPM, 30, 512, 1, 64, 30)
    _check_vs_floor(out["latents_unscaled"], ref, emul, "txt2img small UNet 64x64 latents, 30 DPM steps")
    pipe.use_cuda_graph = False
    eager = pipe.txt2img(text_embeddings=text, uncond_embeddings=uncond, latents=lat, num_inference_steps=30,
                         guidance_scale=7.0, width=512, output_type="latent")
    assert torch.equal(eager["latents_unscaled"], out["latents_unscaled"]), "CUDA-graph replay differs from eager"


@torch.no_grad()
def test_txt2img_small_unet_50_pndm_steps_640_wide(small_unet):
    oracle, unet = small_unet
    _, out, ref, emul, *_ = _loop_case(oracle, unet, "PNDMScheduler", 50, 640, 1, 64, 50)
    _check_vs_floor(out["latents_unscaled"], ref, emul, "txt2img small UNet 64x80 latents, 50 PNDM steps (51 evals)")


@torch.no_grad()
def test_txt2img_seed_list_equals_single_calls(small_unet, vae_pair):
    pipe = _small_pipe(small_unet, vae_pair)
    prompts = ["church bells", "jazz with piano", "church bells", "lo-fi beat"]
    seeds = [42, 43, 7, 1000]
    batch = pipe.txt2img(prompts, negative_prompt=[None, "drums", None, ""], seed=seeds, num_inference_steps=20,
                         guidance_scale=7.0)
    assert len(batch["images"]) == 4 and all(im.size == (512, 512) for im in batch["images"])
    for i in range(4):
        single = pipe.txt2img(prompts[i], negative_prompt=[None, "drums", None, ""][i], seed=seeds[i], num_inference_steps=20,
                              guidance_scale=7.0)
        d = np.abs(np.array(batch["images"][i]).astype(np.int16) - np.array(single["images"][0]).astype(np.int16))
        print(f"txt2img seed list clip {i}: vs single call mean |diff| {d.mean():.4f} LSB, max {d.max()}, "
              f"within 1 LSB {100 * (d <= 1).mean():.2f} %")
        assert d.mean() < 0.25 and (d <= 1).mean() >= 0.98
    lat = torch.cat([torch.randn((1, 4, 64, 64), generator=torch.Generator(device="cuda").manual_seed(sd), device="cuda",
                                 dtype=torch.float16) for sd in seeds])
    inj = pipe.txt2img(prompts, negative_prompt=[None, "drums", None, ""], latents=lat, num_inference_steps=20,
                       guidance_scale=7.0)
    assert torch.equal(inj["latents_unscaled"], batch["latents_unscaled"])
    assert all(np.array_equal(np.array(a), np.array(b)) for a, b in zip(inj["images"], batch["images"]))


# ----------------------------------------------------------------------------------------------- text -> audio
@torch.no_grad()
def test_text_to_audio_clips_chain(small_unet, vae_pair):
    """device path: txt2img latents -> VAE decode -> fp32-scaled uint8 -> mel -> inverse mel + Griffin-Lim, each stage
    re-synchronised on ours: uint8 vs the torch rounding of our decode, waveform vs torchaudio on our uint8 image"""
    from oracle import audio_oracle as ao
    from oracle.torchaudio_ref import TorchaudioConverter
    from riffusion.spectrogram_converter import SpectrogramConverter, mel_filterbank
    from riffusion.spectrogram_params import SpectrogramParams

    pipe = _small_pipe(small_unet, vae_pair)
    conv = SpectrogramConverter(SpectrogramParams(), device="cuda")
    for W in (512, 768):
        angles = torch.rand(2, 8821, W, dtype=torch.complex64, device="cuda")
        out = pipe.text_to_audio_clips(["church bells", "jazz"], converter=conv, seed=[1, 2], num_inference_steps=10,
                                       guidance_scale=7.0, width=W, init_angles=angles)
        u8, wave = out["images"], out["waveform"]
        assert u8.shape == (2, 512, W, 3) and wave.shape == (2, 441 * (W - 1)) and out["n_unet_evals"] == 10
        img = pipe.vae.decode(out["latents"]).sample
        want = ((img / 2 + 0.5).clamp(0, 1).float() * 255).round().to(torch.uint8).permute(0, 2, 3, 1)
        assert torch.equal(u8, want)
        u8n = u8.cpu().numpy()
        mel_ref = np.concatenate([ao.spectrogram_from_image_array(u8n[i], power=0.25, stereo=False, max_value=30e6)
                                  for i in range(2)])
        wave_ref = TorchaudioConverter().waveform_from_mel_amplitudes(torch.from_numpy(mel_ref), angles.cpu())
        w = wave.cpu()

        def nrms(a, b):
            return float((((a - b) / b.abs().amax(dim=-1, keepdim=True)) ** 2).mean().sqrt())

        rms = nrms(w, wave_ref)
        print(f"text_to_audio_clips W={W}: waveform vs torchaudio on our uint8 image: normalised RMS {rms:.3e}")
        if rms >= 1e-4:            # ill-conditioned Griffin-Lim input: the fp64 recurrence referees (test_parity_bench_gpu)
            fb = mel_filterbank(8821, 0.0, 10000.0, 512, 44100).numpy()
            o64 = torch.from_numpy(ao.waveform_from_mel_amplitudes(mel_ref[:1], fb, 17640, 441, ao.hann_window(4410).double().numpy(),
                                                                   32, angles[:1].cpu().numpy())).float()
            e_ta, e_us = nrms(wave_ref[:1], o64), nrms(w[:1], o64)
            print(f"text_to_audio_clips W={W}: vs the fp64 recurrence: torchaudio {e_ta:.3e}, kernels {e_us:.3e}")
            assert e_us <= max(2 * e_ta, 2e-5)


def test_text_to_audio_commands_end_to_end(small_unet, vae_pair, tmp_path, monkeypatch):
    import json

    from PIL import Image
    from scipy.io import wavfile

    from riffusion import text_to_audio
    from riffusion.riffusion_pipeline import RiffusionPipeline
    from riffusion.spectrogram_params import SpectrogramParams

    pipe = _small_pipe(small_unet, vae_pair)
    monkeypatch.setattr(RiffusionPipeline, "load_checkpoint", classmethod(lambda cls, *a, **k: pipe))
    for use_20k, channels in ((False, 1), (True, 2)):
        out = tmp_path / f"t2a_{use_20k}"
        args = ["text-to-audio", "--prompt", "church bells", "--checkpoint", "ck", "--output-dir", str(out), "--seed", "5",
                "--num-clips", "2", "--num-inference-steps", "4", "--width", "768"] + (["--use-20k"] if use_20k else [])
        text_to_audio.main(args)
        for s in (5, 6):
            img = Image.open(out / f"church_bells_{s}.png")
            assert img.size == (768, 512)
            p = SpectrogramParams.from_exif(img.getexif())
            assert (p.stereo, p.min_frequency, p.max_frequency) == (use_20k, 10 if use_20k else 0, 20000 if use_20k else 10000)
            rate, data = wavfile.read(out / f"church_bells_{s}.wav")
            dur = data.shape[0] / rate
            print(f"text-to-audio use_20k={use_20k} seed {s}: {dur:.3f} s, {data.shape[1] if data.ndim == 2 else 1} channel(s)")
            assert rate == 44100 and (data.shape[1] if data.ndim == 2 else 1) == channels
            assert abs(dur - 441 * 767 / 44100) < 0.05
    spec = {"params": {"num_inference_steps": 3, "width": 640},
            "entries": [{"prompt": "Church bells", "seed": 42}, {"prompt": "beats", "negative_prompt": "drums", "seed": 9}]}
    (tmp_path / "in.json").write_text(json.dumps(spec))
    text_to_audio.main(["text-to-audio-batch", "--input-json", str(tmp_path / "in.json"), "--output-dir",
                        str(tmp_path / "batch")])
    index = json.loads((tmp_path / "batch" / "index.json").read_text())
    for e in index["entries"]:
        img = Image.open(e["image_path"])
        assert img.size == (640, 512) and SpectrogramParams.from_exif(img.getexif()) == SpectrogramParams(max_frequency=10000)
        rate, data = wavfile.read(e["audio_path"])
        assert (data.shape[1] if data.ndim == 2 else 1) == 1 and abs(data.shape[0] / rate - 441 * 639 / 44100) < 0.05
