/*
 * rf_b200.h — C-ABI of the B200-native Riffusion hot paths (librf_b200.so).
 *
 * The reference (riffusion/riffusion-hobby, pure Python) has no FFI; its seams are
 * duck-typed Python callables.  Each entry point below replaces the arithmetic behind
 * one of those seams and is what a ctypes binding in the reference would call
 * (INTEGRATION.md shows the stub).  Citations are into /root/reference unless
 * prefixed TA/ (= site-packages/torchaudio, the third-party package that holds the
 * arithmetic of path (a)).
 *
 * Conventions
 *   - every pointer named d_* is a DEVICE pointer (e.g. torch.Tensor.data_ptr()); the
 *     caller allocates inputs, outputs and the workspace (size from *_workspace_bytes);
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - all functions return 0 on success, non-zero on error; rf_last_error() returns a
 *     thread-local message.  There is NO CPU fallback: device entry points fail with
 *     RF_ERR_CUDA when no sm_100 device is usable;
 *   - no global mutable state: a plan is immutable after its first upload, so
 *     concurrent calls on different streams with different workspaces are safe
 *     (the reference shares one converter across a ThreadPool, riffusion/cli.py:172-204).
 */
#ifndef RF_B200_H
#define RF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RF_OK 0
#define RF_ERR_INVALID 1     /* bad argument / unsupported geometry */
#define RF_ERR_CUDA 2        /* CUDA runtime error or no usable device */
#define RF_ERR_UNSUPPORTED 3 /* valid reference parameters this build has no kernel for */

typedef struct rf_plan rf_plan;

/* Mirrors riffusion/spectrogram_params.py:8-81 (SpectrogramParams + derived n_fft /
 * win_length / hop_length) and the MelScale arguments of
 * riffusion/spectrogram_converter.py:75-99.
 * Geometry: win 4410 / n_fft 17640 / hop dividing 4410 (44.1 kHz defaults) runs on the prime-factor
 * engine; any other even n_fft <= 28000 with n_fft/2 = 2^a 3^b 5^c 7^d (48 kHz: 19200, 22.05 kHz: 8820,
 * custom window / padding / step durations) runs on the generic mixed-radix engine; everything else is
 * RF_ERR_UNSUPPORTED from rf_plan_create. */
typedef struct rf_plan_desc {
    int32_t sample_rate;  /* 44100 */
    int32_t n_fft;        /* 17640  (padded_duration_ms) */
    int32_t win_length;   /* 4410   (window_duration_ms) */
    int32_t hop_length;   /* 441    (step_size_ms) */
    int32_t n_mels;       /* 512    (num_frequencies) */
    float f_min;          /* 0      (min_frequency) */
    float f_max;          /* 10000  (max_frequency) */
    int32_t mel_norm_slaney; /* 0: norm=None, 1: "slaney" (mel_scale_norm) */
    int32_t mel_scale_slaney; /* 0: "htk", 1: "slaney" (mel_scale_type) */
    int32_t full_band;    /* 0: prune STFT bins to the mel filterbank's support
                             (rows of fb that are not identically zero);
                             1: keep all n_fft/2+1 bins (generic GriffinLim input) */
} rf_plan_desc;

typedef struct rf_plan_info {
    int32_t n_freq;      /* n_fft/2 + 1 */
    int32_t n_live;      /* STFT bins carried through Griffin-Lim */
    int32_t k_lo, k_hi;  /* smallest / largest live bin */
    int32_t n_even;      /* live bins with even k (first in the private bin order) */
    int32_t fb_nnz;      /* non-zeros of the mel filterbank */
    int32_t chunk_frames; /* frames per overlap-add chunk used by the iSTFT kernel */
} rf_plan_info;

const char* rf_last_error(void);
const char* rf_version(void);

/* Build the host side of a plan (all tables in fp64, rounded once to fp32).
 *   window : optional host float[win_length] (e.g. torch.hann_window, periodic) — NULL =
 *            computed here as 0.5-0.5cos(2 pi n/win) (TA/transforms/_transforms.py:94).
 *   fb     : optional host float[n_freq][n_mels], row-major, the torchaudio
 *            melscale_fbanks matrix (TA/functional/functional.py:518-587) — NULL =
 *            computed here following the same formula.
 * Device tables are uploaded lazily by the first device call. */
int rf_plan_create(const rf_plan_desc* desc, const float* window, const float* fb, rf_plan** out);
void rf_plan_destroy(rf_plan* plan);
int rf_plan_get_info(const rf_plan* plan, rf_plan_info* info);
/* Griffin-Lim runs its inner loop on every second waveform sample when the live band allows it (2*k_hi + 800 <=
 * n_fft/2: aliasing below fp32 rounding; the final reconstruction is always full rate).  enable = 0 forces the
 * full-rate loop.  Returns 1 if the decimated loop will be used, 0 otherwise (not an error code). */
int rf_plan_set_decimation(rf_plan* plan, int enable);
/* Copy a named host table (for tests): "bins" int32[n_live], "pp" uint32[n_live],
 * "wt_fwd"/"wt_inv" float[4][win][2], "window" float[win], "fb" float[n_freq][n_mels],
 * "pinv" float[n_freq][n_mels] (= min-norm inverse-mel operator, dense),
 * "tri" double[3][n_mels] (Gram tridiagonal: sub, diag, super), and for the decimated loop "pp2" uint32[n_live],
 * "wt2_fwd"/"wt2_inv" float[2][4][win/2][2], "ph_odd" float[n_live][2]; the kernel-side forms derived from them:
 * "bt" uint32[n_live] (V offset | partner offset << 14 | self-paired << 31), "ab_inv"/"ab_fwd" float[n_live][4]
 * (per-bin phase constants of the inverse / forward pair packing), "bt2"/"ab2_inv"/"ab2_fwd" for the decimated loop,
 * "items"/"items2" uint32[49 * 10 | 49 * 5] (radix-9 pass: V position a*441 + c | first sample index << 12 of slot tau),
 * "wg2_inv" float[9][245][4] (per sample of the decimated grid: window of frame t0, of frame t0+1, cos, sin) and the
 * other-parity tables of the hybrid loop's edge chunks "wg2o_inv" (the two windows swapped), "ab2o_inv" float[n_live][4].
 * Returns RF_ERR_INVALID if
 * `bytes` does not match the table size. */
int rf_plan_table(const rf_plan* plan, const char* name, void* dst, size_t bytes);

/* ---- path (a), inverse: mel amplitudes -> waveform ---------------------------------
 * replaces SpectrogramConverter.waveform_from_mel_amplitudes
 * (riffusion/spectrogram_converter.py:187-204). */

/* InverseMelScale.forward (TA/transforms/_transforms.py:491-512): relu(min-norm lstsq).
 * d_mel f32[B][n_mels][T] -> d_lin f32[B][n_freq][T] (torchaudio layout). */
int rf_inverse_mel(rf_plan* plan, const float* d_mel, int B, int T, float* d_lin, void* stream);

/* GriffinLim.forward -> F.griffinlim (TA/functional/functional.py:255-353), power=1.
 *   d_lin         f32[B][n_freq][T]  magnitudes (bins outside the plan's live set must be 0;
 *                                    use a full_band plan for arbitrary input)
 *   d_init_angles c64[B][n_freq][T]  initial "angles" (torch.rand(cfloat), :310) or NULL for
 *                                    rand_init=False (all ones, :312)
 *   d_wave        f32[B][hop*(T-1)]
 * Requires hop*(T-1) > n_fft/2 (torch.stft reflect padding limit, same error as torch). */
size_t rf_griffinlim_workspace_bytes(const rf_plan* plan, int B, int T);
int rf_griffinlim(rf_plan* plan, const float* d_lin, const void* d_init_angles, int B, int T,
                  int n_iter, float momentum, float* d_wave, void* d_workspace,
                  size_t workspace_bytes, void* stream);

/* Fused inverse-mel + Griffin-Lim (no [B][n_freq][T] intermediate). Requires a pruned
 * (full_band=0) plan. Same workspace size as rf_griffinlim. */
int rf_mel_to_wave(rf_plan* plan, const float* d_mel, const void* d_init_angles, int B, int T,
                   int n_iter, float momentum, float* d_wave, void* d_workspace,
                   size_t workspace_bytes, void* stream);

/* rf_mel_to_wave with every Griffin-Lim kernel launch bracketed by CUDA events on `stream`
 * (measurement aid for bench.py's roofline; synchronises the stream before returning).
 *   ms_out[3]       host: summed device ms of {iSTFT chunk kernel, overlap-add assembly, STFT pair kernel}
 *   launches_out[3] host: launches per class */
int rf_mel_to_wave_profiled(rf_plan* plan, const float* d_mel, const void* d_init_angles, int B,
                            int T, int n_iter, float momentum, float* d_wave, void* d_workspace,
                            size_t workspace_bytes, void* stream, float* ms_out, int* launches_out);

/* ---- path (a), forward: waveform -> mel amplitudes ---------------------------------
 * replaces SpectrogramConverter.mel_amplitudes_from_waveform
 * (riffusion/spectrogram_converter.py:165-185): Spectrogram(power=None) -> abs -> MelScale.
 * d_wave f32[B][L] -> d_mel f32[B][n_mels][T], T = 1 + L/hop. Requires L > n_fft/2. */
int rf_stft_mel(rf_plan* plan, const float* d_wave, int B, int L, float* d_mel, void* stream);
/* Complex STFT only (Spectrogram(power=None), TA/functional/functional.py:54-145):
 * d_spec c64[B][n_freq][T]; bins outside the live set are written as 0 unless full_band. */
int rf_stft(rf_plan* plan, const float* d_wave, int B, int L, void* d_spec, void* stream);
/* MelScale.forward (TA/transforms/_transforms.py:407-419) on its own:
 * d_spec f32[B][n_freq][T] -> d_mel f32[B][n_mels][T]. */
int rf_mel_scale(rf_plan* plan, const float* d_spec, int B, int T, float* d_mel, void* stream);

/* ---- image <-> spectrogram quantisation, int16 waveform --------------------------- */
/* image_util.spectrogram_from_image (riffusion/util/image_util.py:59-110) after the
 * P/L->RGB conversion: d_img u8[Hh][Ww][3] -> d_mel f32[C][Hh][Ww] (C = stereo?2:1),
 * flip-Y, mono = R plane, stereo = G,B planes, ((255-u8)/255)^(1/power) * max_value. */
int rf_image_to_mel(const uint8_t* d_img, int height, int width, int stereo, float power,
                    float max_value, float* d_mel, void* stream);
/* image_util.image_from_spectrogram (riffusion/util/image_util.py:13-56):
 * d_mel f32[C][Hh][Ww] -> d_img u8[Hh][Ww][3]; d_max receives max over all channels
 * (written to EXIF MAX_VALUE by spectrogram_image_converter.py:59). d_scratch: >= 4 bytes. */
int rf_mel_to_image(const float* d_mel, int channels, int height, int width, float power,
                    uint8_t* d_img, float* d_max, void* stream);
/* audio_util.audio_from_waveform(normalize=True) (riffusion/util/audio_util.py:13-28):
 * d_wave f32[C][L] -> d_pcm i16[L][C]; x *= 32767/max|x| over all channels, truncate. */
int rf_wave_to_int16(const float* d_wave, int channels, int L, int normalize, int16_t* d_pcm,
                     float* d_scratch, void* stream);


/* ==== path (b): tensor-core building blocks (tcgen05 / TMEM / TMA) ========================
 * The reference reaches these through diffusers' UNet2DConditionModel / AutoencoderKL forward
 * (riffusion/riffusion_pipeline.py:255,406-408,428): torch.nn.Linear / Conv2d / attention bmm.
 * All tensors fp16, device pointers; activations are NHWC ("channels last"). */

/* D[b2][b1][m][n] = act(alpha * sum_k A[..][m][k] * B[..][n][k] + bias) + residual  (both operands K-major).
 * Strides are in elements; ld* = row pitch, s*1 / s*2 = strides of the two batch dimensions
 * (ignored when the batch extent is 1).  Pointers 16-byte aligned, pitches multiples of 8. */
typedef struct rf_gemm_desc {
    int32_t M, N, K;
    int32_t batch1, batch2;
    const void* A; int64_t lda, sa1, sa2;
    const void* B; int64_t ldb, sb1, sb2;
    void* D;       int64_t ldd, sd1, sd2;
    const void* bias;          /* fp16 [N] (bias_mode 1) or [M] (bias_mode 2), or NULL */
    int32_t bias_mode;
    const void* residual;      /* fp16, indexed like D with ldr/sr1/sr2, or NULL */
    int64_t ldr, sr1, sr2;
    float alpha;               /* 0 is treated as 1 */
    int32_t act;               /* 0 none, 1 SiLU, 3 quick_gelu x*sigmoid(1.702x), 2 GEGLU: B rows come in runs of [16 value | 16 gate] rows of the
                                  same 16 outputs, D has N/2 columns, D[m][16 r + j] = v_j * gelu(g_j) (exact erf) */
    int32_t out_f32;           /* 1: D is fp32 */
    void* workspace;           /* optional device scratch for split-K (problems with fewer tiles than SMs); NULL: never split */
    int64_t workspace_bytes;   /* its size; rf_gemm_workspace_bytes(desc) returns what this problem would use (0: none) */
} rf_gemm_desc;
int rf_gemm_f16(const rf_gemm_desc* desc, void* stream);
size_t rf_gemm_workspace_bytes(const rf_gemm_desc* desc);

/* torch.nn.Conv2d (3x3 pad 1 or 1x1 pad 0, stride 1 or 2) as an implicit GEMM over NHWC input;
 * the input may be the channel concatenation of two tensors (UNet skip connections,
 * torch.cat([hidden, skip], dim=1)).  Weights are [Cout][ky][kx][C1+C2] fp16 (see
 * riffusion.unet weight packing).  out = act(conv + bias + bias_per_image[b]) + residual. */
typedef struct rf_conv_desc {
    int32_t B, H, W;           /* input images, height, width */
    int32_t C1, C2;            /* channels of x1 and x2 (C2 = 0 without x2); multiples of 64 */
    int32_t Cout, ksize, stride;
    const void* x1; const void* x2;
    const void* w;
    const void* bias;          /* fp16 [Cout] or NULL */
    const void* bias_per_image;/* fp16 [B][Cout] or NULL (time-embedding projection) */
    const void* residual;      /* fp16 NHWC like out, or NULL */
    void* out;                 /* fp16 [B][Ho][Wo][Cout] */
    float alpha;               /* 0 is treated as 1 */
    int32_t act;
    int32_t bias_per_image_pitch; /* row pitch (elements) of bias_per_image; 0 = Cout */
    int32_t pad_mode;          /* 0: symmetric padding ksize/2 (torch padding=1 for 3x3);
                                  1: no left/top padding, implicit zero padding on the right/bottom edge
                                     (diffusers VAE Downsample2D: F.pad(x, (0,1,0,1)) then conv padding=0)
                                  2: nearest-2x upsample fused in (diffusers Upsample2D: F.interpolate(scale 2, nearest) then
                                     conv 3x3 pad 1): ksize = 2, w = the four sub-pixel phase kernels [4][Cout][2][2][C1]
                                     (3x3 taps that land on the same input pixel pre-summed), out is [B][2H][2W][Cout] */
    void* workspace;           /* optional split-K scratch, as in rf_gemm_desc */
    int64_t workspace_bytes;
} rf_conv_desc;
int rf_conv2d_f16(const rf_conv_desc* desc, void* stream);
size_t rf_conv2d_workspace_bytes(const rf_conv_desc* desc);

/* Fused attention softmax(Q K^T * scale) V per (image, head) — diffusers CrossAttention's baddbmm/softmax/bmm
 * [restated from memory] without materialising the scores.  q [B][Nq][heads*d], k [B][Nk][heads*d],
 * vt [B][heads*d][vt_pitch] (V transposed, as produced by rf_gemm_f16 with swapped operands), out [B][Nq][heads*d];
 * fp16, d a multiple of 8 and <= 192, vt_pitch a multiple of 8 >= Nk. */
int rf_attention_f16(const void* q, const void* k, const void* vt, void* out, int B, int heads, int Nq, int Nk,
                     int d, int vt_pitch, float scale, void* stream);

/* Same with an optional causal mask (key j visible to query i iff j <= i): transformers CLIPTextModel's self-attention
 * (causal_attention_mask), the text encoder behind RiffusionPipeline.embed_text (riffusion/riffusion_pipeline.py:177-191).
 * causal != 0 requires Nk <= 128 and d <= 112. */
int rf_attention_masked_f16(const void* q, const void* k, const void* vt, void* out, int B, int heads, int Nq, int Nk,
                            int d, int vt_pitch, float scale, int causal, void* stream);

/* Measurement aid (bench.py roofline): between begin and end every rf_gemm_f16 / rf_conv2d_f16 launch is bracketed by
 * CUDA events on its stream; end synchronises the device and returns the summed kernel time (ms), the algorithmic
 * FLOPs (2*M*N*K, true extents) and the launch count.  Not for use inside CUDA-graph capture. */
int rf_tc_profile_begin(void);
int rf_tc_profile_end(double* ms_out, double* flops_out, long* launches_out);

/* Memory-bound UNet/VAE operators (fp16 activations, fp32 statistics).  NHWC images, row-major tokens.
 * Each restates the torch op diffusers calls [diffusers 0.9, absent here: restated from memory]. */
/* torch.nn.GroupNorm(groups, C, eps) (+ optional SiLU): x,y fp16 [B][HW][C]; d_scratch: fp32 device scratch of
 * rf_group_norm_scratch_floats(B, HW, groups) floats.  Deterministic (fixed-order reductions, no atomics). */
size_t rf_group_norm_scratch_floats(int B, int HW, int groups);
int rf_group_norm_f16(const void* x, int B, int HW, int C, int groups, const void* gamma, const void* beta,
                      float eps, int act, void* y, float* d_scratch, void* stream);
/* Same on the channel concatenation [x | x2] read in place: x [B][HW][C1], x2 [B][HW][C - C1], y [B][HW][C] — the
 * `torch.cat([hidden_states, res_hidden_states], dim=1)` of the UNet up blocks (diffusers unet_2d_blocks.py UpBlock2D /
 * CrossAttnUpBlock2D [restated from memory]) followed by the resnet's norm1, without materialising the concatenation.
 * x2 == NULL: identical to rf_group_norm_f16. */
int rf_group_norm_cat_f16(const void* x, const void* x2, int C1, int B, int HW, int C, int groups, const void* gamma,
                          const void* beta, float eps, int act, void* y, float* d_scratch, void* stream);
/* torch.nn.LayerNorm(C, eps) over rows */
int rf_layer_norm_f16(const void* x, int rows, int C, const void* gamma, const void* beta, float eps, void* y,
                      void* stream);
/* GEGLU: x [rows][2*inner] = (hidden | gate) -> y [rows][inner] = hidden * gelu_erf(gate) */
int rf_geglu_f16(const void* x, long rows, int inner, void* y, void* stream);
/* softmax over the first n entries of each row (row pitch `pitch` elements); padding is zeroed */
int rf_softmax_rows_f16(const void* x, long rows, int n, int pitch, void* y, void* stream);
/* F.interpolate(scale_factor=2, mode="nearest"): [B][H][W][C] -> [B][2H][2W][C] */
int rf_upsample2x_f16(const void* x, int B, int H, int W, int C, void* y, void* stream);
/* torch.cat([a, b], dim=1) for NHWC tensors: [pixels][Ca] + [pixels][Cb] -> [pixels][Ca+Cb] */
int rf_concat_channels_f16(const void* a, const void* b, long pixels, int Ca, int Cb, void* y, void* stream);
/* Conv2d(Cin<=8 -> Cout<=8, 1x1) on NCHW fp16 with an input pre-scale: the VAE's quant_conv / post_quant_conv
 * (and the latents / 0.18215 of riffusion_pipeline.py:427 folded into in_scale) */
int rf_conv1x1_small_f16(const void* x_nchw, const void* w, const void* bias, int B, int Cin, int Cout, long HW,
                         float in_scale, void* y_nchw, void* stream);
/* decoded image -> uint8 RGB: (x/2 + 0.5).clamp(0,1) then (x*255).round() (riffusion_pipeline.py:430-434 + diffusers
 * numpy_to_pil); x fp16 NCHW (B,3,H,W) -> y uint8 NHWC (B,H,W,3).  Device-side glue between VAE decode and
 * rf_image_to_mel (SURVEY 8(f)-1). */
int rf_vae_image_to_u8(const void* x_nchw, int B, int H, int W, uint8_t* y_nhwc, void* stream);
/* the same with `* 255` and the round in fp32 (txt2img decode_latents: `.float()` after the fp16 clamp) */
int rf_vae_image_to_u8_f32scale(const void* x_nchw, int B, int H, int W, uint8_t* y_nhwc, void* stream);
/* conv_in: Conv2d(Cin<=8 -> Cout, 3x3, pad 1) reading NCHW fp16, writing NHWC; w = torch layout [Cout][Cin][3][3] */
int rf_conv_in_f16(const void* x_nchw, const void* w, const void* bias, int B, int Cin, int H, int W, int Cout,
                   void* y_nhwc, void* stream);
/* conv_out: Conv2d(Cin -> Cout<=8, 3x3, pad 1) reading NHWC, writing NCHW fp16; w packed [Cout][3][3][Cin] */
int rf_conv_out_f16(const void* x_nhwc, const void* w_packed, const void* bias, int B, int H, int W, int Cin,
                    int Cout, void* y_nchw, void* stream);
/* diffusers Timesteps(dim, flip_sin_to_cos=True, downscale_freq_shift=0): t fp32 [B] -> fp16 [B][dim] */
int rf_timestep_embedding_f16(const float* d_t, int B, int dim, void* out, void* stream);
int rf_silu_f16(const void* x, long n, void* y, void* stream);
/* torch_util.slerp (riffusion/util/torch_util.py:21-48) per sample on the device: v0, v1, out fp16 [B][n]; d_alphas fp32
 * device [B]; d_scratch fp32 device [3*B].  fp32 reductions (the reference reduces in the tensors' dtype on the host). */
int rf_slerp_f16(const void* v0, const void* v1, int B, long n, const float* d_alphas, float dot_threshold, void* out,
                 float* d_scratch, void* stream);
/* classifier-free guidance + PNDM/PLMS multistep update on n = elements of ONE batch half:
 *   eps = eps_u + g (eps_t - eps_u) (riffusion_pipeline.py:411-415); e = c0 eps + c1 h1 + c2 h2 + c3 h3;
 *   prev = ca * sample - cb * e (PNDMScheduler._get_prev_sample).  eps_pair = [uncond | text] (2n). coef4: HOST float[4].
 *   eps_out (optional) receives the guided eps for the scheduler history. */
int rf_cfg_pndm_step_f16(const void* eps_pair, long n, float guidance, const void* h1, const void* h2,
                         const void* h3, const float* coef4, const void* sample, float ca, float cb,
                         void* eps_out, void* prev_sample, void* stream);
/* Guidance combine + DPMSolverMultistepScheduler(dpmsolver++, midpoint, order 2).step in one pass, reproducing the
 * reference's fp16 tensor-op sequence (one fp16 rounding per op, scalars at full fp32, division by alpha_s as a multiply
 * by its fp32 reciprocal):
 *   e = eu + g (et - eu);  m0 = (x - sigma_s e) / alpha_s;
 *   x0_prev == NULL (first order):  prev = c_x x - c_0 m0
 *   otherwise (second order):       prev = c_x x - c_0 m0 - c_d1 (inv_r0 (m0 - x0_prev))
 * eps_pair = [uncond | text] (2n), sample / x0_prev / x0_out / prev_sample n fp16 each.  x0_out receives m0, the next
 * step's history entry.  prev_sample may alias sample.  Every coefficient is an argument: the library keeps no state. */
int rf_cfg_dpmpp_step_f16(const void* eps_pair, long n, float guidance, const void* sample, const void* x0_prev,
                          float sigma_s, float alpha_s, float c_x, float c_0, float inv_r0, float c_d1, void* x0_out,
                          void* prev_sample, void* stream);
/* y = a*x + b*noise (scheduler.add_noise), optionally y = y*mask + z*(1-mask) (riffusion_pipeline.py:421-425) */
int rf_axpby_f16(const void* x, const void* noise, float a, float b, const void* mask, const void* z, long n,
                 void* y, void* stream);

/* diffusers 0.9 add_noise with its fp16 op sequence: y = s * x + s1 * noise, rounded to fp16 after each op.  s and s1 are
 * the fp16 values alphas_cumprod[t] ** 0.5 and (1 - alphas_cumprod[t]) ** 0.5 with alphas_cumprod cast to fp16 first
 * (img2img's prepare_latents); values not representable in fp16 are rejected.  x, noise, y: n fp16; y may alias x. */
int rf_add_noise_f16_seq(const void* x, const void* noise, float s, float s1, long n, void* y, void* stream);

/* ---- spectrogram-image glue of audio to audio (rf_image_ops.cu) ---- */
/* Pillow-exact Image.resize(..., BICUBIC) of B uint8 RGB images: x (B, H_in, W_in, 3) -> y (B, H_out, W_out, 3), NHWC.
 * Horizontal pass, then vertical, each skipped when its size is unchanged; taps in int32 fixed point with 22 fractional
 * bits, built on the host as Pillow builds them and cached on the device per (device, n_in, n_out).  y must not alias x. */
int rf_resample_u8(const uint8_t* x_nhwc, int B, int H_in, int W_in, int H_out, int W_out, uint8_t* y_nhwc, void* stream);
/* Host only: the fixed-point taps rf_resample_u8 uses along one axis of n_in -> n_out pixels.  *ksize receives the taps
 * per output pixel; bounds (optional, [n_out][2] = first input pixel, tap count) and kk (optional, [n_out][ksize]) are
 * filled when given. */
int rf_resample_coeffs(int n_in, int n_out, int* ksize, int32_t* bounds, int32_t* kk);
/* img2img preprocess: uint8 NHWC (B, H, W, 3) -> fp16 NCHW (B, 3, H, W), 2 * (u / 255) - 1 in fp32 rounded once to fp16 */
int rf_image_u8_to_f16(const uint8_t* x_nhwc, int B, int H, int W, void* y_nchw, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RF_B200_H */
