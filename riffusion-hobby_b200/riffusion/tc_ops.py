"""Thin tensor wrappers over the tensor-core C-ABI entry points (rf_gemm_f16, rf_conv2d_f16, ...).

Activations are fp16, NHWC for images and (rows, channels) for token matrices.  These helpers only
marshal pointers/strides; every FLOP runs in the tcgen05 kernels of librf_b200.so.
"""
from __future__ import annotations

import ctypes as C
import typing as T

import torch

from riffusion import _native

ACT_NONE, ACT_SILU, ACT_GEGLU, ACT_QUICK_GELU = 0, 1, 2, 3


def _f16(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda or t.dtype != torch.float16:
        raise _native.NativeError(f"{name} must be a CUDA fp16 tensor (got {t.dtype} on {t.device})")
    return t


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _workspace(nbytes: int, desc, device) -> T.Optional[torch.Tensor]:
    """split-K scratch of one call, from torch's caching allocator (stream-ordered, CUDA-graph safe): the library itself
    keeps no device state, so calls on different streams never share it"""
    if not nbytes:
        return None
    ws = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
    desc.workspace, desc.workspace_bytes = ws.data_ptr(), int(nbytes)
    return ws


def gemm(
    a: torch.Tensor, b: torch.Tensor, *, bias: T.Optional[torch.Tensor] = None, bias_per_row: bool = False,
    residual: T.Optional[torch.Tensor] = None, alpha: float = 1.0, act: int = ACT_NONE,
    out: T.Optional[torch.Tensor] = None, out_dtype: torch.dtype = torch.float16,
) -> torch.Tensor:
    """D[..., m, n] = act(alpha * A[..., m, :] . B[..., n, :] + bias) + residual.

    a: (..., M, K), b: (..., N, K) with up to two leading batch dims (strided views are fine as long
    as the last dim is contiguous and pitches are multiples of 8 elements).
    """
    _f16(a, "a"), _f16(b, "b")
    while a.dim() < 4:
        a = a.unsqueeze(0)
    while b.dim() < 4:
        b = b.unsqueeze(0)
    M, K, N = a.shape[2], a.shape[3], b.shape[2]
    B2, B1 = max(a.shape[0], b.shape[0]), max(a.shape[1], b.shape[1])
    a = a.expand(B2, B1, M, K)          # broadcast batch dims get stride 0 (handled in the C-ABI)
    b = b.expand(B2, B1, N, K)
    assert b.shape[3] == K and a.stride(3) == 1 and b.stride(3) == 1
    n_out = N // 2 if act == ACT_GEGLU else N       # GEGLU epilogue: b packed with interleave_geglu()
    if out is None:
        out = torch.empty((B2, B1, M, n_out), dtype=out_dtype, device=a.device)
    o4 = out
    while o4.dim() < 4:
        o4 = o4.unsqueeze(0)
    assert o4.shape == (B2, B1, M, n_out) and o4.stride(3) == 1
    d = _native.GemmDesc()
    d.M, d.N, d.K, d.batch1, d.batch2 = M, N, K, B1, B2
    d.A, d.lda, d.sa1, d.sa2 = a.data_ptr(), a.stride(2), a.stride(1), a.stride(0)
    d.B, d.ldb, d.sb1, d.sb2 = b.data_ptr(), b.stride(2), b.stride(1), b.stride(0)
    d.D, d.ldd, d.sd1, d.sd2 = o4.data_ptr(), o4.stride(2), o4.stride(1), o4.stride(0)
    d.bias = None if bias is None else _f16(bias, "bias").data_ptr()
    d.bias_mode = 0 if bias is None else (2 if bias_per_row else 1)
    if residual is not None:
        r4 = _f16(residual, "residual")
        while r4.dim() < 4:
            r4 = r4.unsqueeze(0)
        assert r4.shape == (B2, B1, M, N) and r4.stride(3) == 1
        d.residual, d.ldr, d.sr1, d.sr2 = r4.data_ptr(), r4.stride(2), r4.stride(1), r4.stride(0)
    d.alpha, d.act, d.out_f32 = float(alpha), int(act), int(o4.dtype == torch.float32)
    with torch.cuda.device(a.device):
        ws = _workspace(_native.lib().rf_gemm_workspace_bytes(C.byref(d)), d, a.device)     # keeps the scratch alive
        _native.check(_native.lib().rf_gemm_f16(C.byref(d), _stream(a)))
    del ws
    return out


def interleave_geglu(t: torch.Tensor) -> torch.Tensor:
    """Row order the GEGLU epilogue of rf_gemm_f16 expects.  t: (2*inner, ...) = diffusers GEGLU.proj weight or bias,
    rows [0, inner) the value half and [inner, 2*inner) the gate half (models/activations.py GEGLU.forward: chunk(2));
    result: runs of [16 value rows | 16 gate rows] of the same 16 outputs."""
    inner = t.shape[0] // 2
    assert t.shape[0] == 2 * inner and inner % 16 == 0
    v = t[:inner].reshape(inner // 16, 16, *t.shape[1:])
    g = t[inner:].reshape(inner // 16, 16, *t.shape[1:])
    return torch.stack((v, g), dim=1).reshape(t.shape).contiguous()


def pack_conv_weight(w: torch.Tensor) -> torch.Tensor:
    """torch Conv2d weight (Cout, Cin, kh, kw) -> (Cout, kh, kw, Cin) fp16 contiguous, the K-major
    layout the implicit-GEMM kernel streams with TMA."""
    return w.permute(0, 2, 3, 1).contiguous().to(torch.float16)


def conv2d(
    x: torch.Tensor, w_packed: torch.Tensor, *, x2: T.Optional[torch.Tensor] = None,
    bias: T.Optional[torch.Tensor] = None, bias_per_image: T.Optional[torch.Tensor] = None,
    residual: T.Optional[torch.Tensor] = None, stride: int = 1, act: int = ACT_NONE, pad_far_edge_only: bool = False,
) -> torch.Tensor:
    """x (and optional x2, concatenated along channels): (B, H, W, C) fp16 NHWC contiguous.
    w_packed: (Cout, k, k, C1+C2).  Returns (B, Ho, Wo, Cout).  `pad_far_edge_only`: F.pad(x,(0,1,0,1)) + padding=0."""
    _f16(x, "x"), _f16(w_packed, "w")
    B, H, W, C1 = x.shape
    C2 = 0 if x2 is None else x2.shape[3]
    Cout, k, _, Cin = w_packed.shape
    assert Cin == C1 + C2 and x.is_contiguous() and w_packed.is_contiguous()
    pad = 1 if (k == 3 and not pad_far_edge_only) else 0
    extra = 1 if (k == 3 and pad_far_edge_only) else 0
    Ho, Wo = (H + 2 * pad + extra - k) // stride + 1, (W + 2 * pad + extra - k) // stride + 1
    out = torch.empty((B, Ho, Wo, Cout), dtype=torch.float16, device=x.device)
    d = _native.ConvDesc()
    d.B, d.H, d.W, d.C1, d.C2, d.Cout, d.ksize, d.stride = B, H, W, C1, C2, Cout, k, stride
    d.x1 = x.data_ptr()
    d.x2 = None if x2 is None else _f16(x2, "x2").contiguous().data_ptr()
    d.w = w_packed.data_ptr()
    d.bias = None if bias is None else _f16(bias, "bias").data_ptr()
    if bias_per_image is not None:      # (B, Cout) view; rows may be slices of a wider matrix
        assert bias_per_image.shape == (B, Cout) and bias_per_image.stride(1) == 1
        d.bias_per_image = _f16(bias_per_image, "bias_per_image").data_ptr()
        d.bias_per_image_pitch = bias_per_image.stride(0)
    if residual is not None:
        assert residual.shape == out.shape and residual.is_contiguous()
        d.residual = _f16(residual, "residual").data_ptr()
    d.out, d.alpha, d.act, d.pad_mode = out.data_ptr(), 1.0, int(act), int(pad_far_edge_only)
    with torch.cuda.device(x.device):
        ws = _workspace(_native.lib().rf_conv2d_workspace_bytes(C.byref(d)), d, x.device)
        _native.check(_native.lib().rf_conv2d_f16(C.byref(d), _stream(x)))
    del ws
    return out


def pack_upsample_weight(w: torch.Tensor) -> torch.Tensor:
    """torch Conv2d weight (Cout, Cin, 3, 3) of an `Upsample2D` (nearest 2x, then conv 3x3 pad 1) -> the four 2x2 sub-pixel
    phase kernels (4, Cout, 2, 2, Cin) fp16 for `conv2d_upsample2x`: output pixel (2y + py, 2x + px) only sees the input
    pixels (y + py - 1 + a, x + px - 1 + b), a, b in {0, 1}; the 3x3 taps that land on the same input pixel are summed
    (in fp32, then rounded once).  phase = 2 py + px."""
    assert w.dim() == 4 and w.shape[2:] == (3, 3)
    wf = w.detach().float()
    rows = {0: ((0,), (1, 2)), 1: ((0, 1), (2,))}
    out = torch.empty((4, w.shape[0], 2, 2, w.shape[1]), dtype=torch.float32, device=w.device)
    for py in (0, 1):
        for px in (0, 1):
            for a in (0, 1):
                for b in (0, 1):
                    acc = 0
                    for dy in rows[py][a]:
                        for dx in rows[px][b]:
                            acc = acc + wf[:, :, dy, dx]
                    out[2 * py + px, :, a, b, :] = acc
    return out.to(torch.float16).contiguous()


def conv2d_upsample2x(x: torch.Tensor, w_phases: torch.Tensor, *, bias: T.Optional[torch.Tensor] = None) -> torch.Tensor:
    """conv3x3(pad 1)(nearest_upsample_2x(x)) without materialising the upsampled tensor and with 4/9 of the FLOPs.
    x: (B, H, W, C) NHWC fp16; w_phases from `pack_upsample_weight`; returns (B, 2H, 2W, Cout)."""
    _f16(x, "x"), _f16(w_phases, "w_phases")
    B, H, W, Cin = x.shape
    assert w_phases.dim() == 5 and w_phases.shape[0] == 4 and w_phases.shape[2:] == (2, 2, Cin) and x.is_contiguous()
    Cout = w_phases.shape[1]
    out = torch.empty((B, 2 * H, 2 * W, Cout), dtype=torch.float16, device=x.device)
    d = _native.ConvDesc()
    d.B, d.H, d.W, d.C1, d.C2, d.Cout, d.ksize, d.stride = B, H, W, Cin, 0, Cout, 2, 1
    d.x1, d.x2, d.w = x.data_ptr(), None, w_phases.data_ptr()
    d.bias = None if bias is None else _f16(bias, "bias").data_ptr()
    d.out, d.alpha, d.act, d.pad_mode = out.data_ptr(), 1.0, ACT_NONE, 2
    with torch.cuda.device(x.device):
        _native.check(_native.lib().rf_conv2d_f16(C.byref(d), _stream(x)))
    return out


# ------------------------------------------------------------------------------ memory-bound operators
def group_norm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, groups: int, eps: float, silu: bool,
               x2: T.Optional[torch.Tensor] = None) -> torch.Tensor:
    """x: (B, H, W, C) or (B, HW, C) fp16 NHWC -> same shape; GroupNorm (+ SiLU).  With `x2` the input is the channel
    concatenation [x | x2] (torch.cat(dim=1) of the up blocks), read in place; the result has C1 + C2 channels."""
    _f16(x, "x")
    assert x.is_contiguous()
    B, C1 = x.shape[0], x.shape[-1]
    C = C1
    if x2 is not None:
        _f16(x2, "x2")
        assert x2.is_contiguous() and x2.shape[:-1] == x.shape[:-1]
        C = C1 + x2.shape[-1]
    HW = x.numel() // (B * C1)
    y = torch.empty(x.shape[:-1] + (C,), dtype=torch.float16, device=x.device)
    stats = torch.empty((_native.lib().rf_group_norm_scratch_floats(B, HW, groups),), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(_native.lib().rf_group_norm_cat_f16(
            x.data_ptr(), None if x2 is None else x2.data_ptr(), C1, B, HW, C, groups, gamma.data_ptr(), beta.data_ptr(),
            float(eps), int(silu), y.data_ptr(), stats.data_ptr(), _stream(x)))
    return y


def layer_norm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    _f16(x, "x")
    assert x.is_contiguous()
    C = x.shape[-1]
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _native.check(_native.lib().rf_layer_norm_f16(x.data_ptr(), x.numel() // C, C, gamma.data_ptr(), beta.data_ptr(),
                                                      float(eps), y.data_ptr(), _stream(x)))
    return y


def geglu(x: torch.Tensor) -> torch.Tensor:
    _f16(x, "x")
    assert x.is_contiguous()
    inner = x.shape[-1] // 2
    y = torch.empty(x.shape[:-1] + (inner,), dtype=torch.float16, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(_native.lib().rf_geglu_f16(x.data_ptr(), x.numel() // (2 * inner), inner, y.data_ptr(), _stream(x)))
    return y


def softmax_rows_(x: torch.Tensor, n: int) -> torch.Tensor:
    """In-place softmax over the first n entries of every row of a contiguous (..., pitch) fp16 tensor."""
    _f16(x, "x")
    assert x.is_contiguous()
    pitch = x.shape[-1]
    with torch.cuda.device(x.device):
        _native.check(_native.lib().rf_softmax_rows_f16(x.data_ptr(), x.numel() // pitch, n, pitch, x.data_ptr(), _stream(x)))
    return x


def upsample2x(x: torch.Tensor) -> torch.Tensor:
    _f16(x, "x")
    B, H, W, C = x.shape
    y = torch.empty((B, 2 * H, 2 * W, C), dtype=torch.float16, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(_native.lib().rf_upsample2x_f16(x.data_ptr(), B, H, W, C, y.data_ptr(), _stream(x)))
    return y


def concat_channels(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    _f16(a, "a"), _f16(b, "b")
    assert a.shape[:-1] == b.shape[:-1] and a.is_contiguous() and b.is_contiguous()
    Ca, Cb = a.shape[-1], b.shape[-1]
    y = torch.empty(a.shape[:-1] + (Ca + Cb,), dtype=torch.float16, device=a.device)
    with torch.cuda.device(a.device):
        _native.check(_native.lib().rf_concat_channels_f16(a.data_ptr(), b.data_ptr(), a.numel() // Ca, Ca, Cb,
                                                           y.data_ptr(), _stream(a)))
    return y


def conv_in(x_nchw: torch.Tensor, w: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """(B, Cin<=8, H, W) NCHW fp16 -> (B, H, W, Cout) NHWC; w: torch layout (Cout, Cin, 3, 3) fp16."""
    _f16(x_nchw, "x")
    B, Cin, H, W = x_nchw.shape
    Cout = w.shape[0]
    y = torch.empty((B, H, W, Cout), dtype=torch.float16, device=x_nchw.device)
    with torch.cuda.device(x_nchw.device):
        _native.check(_native.lib().rf_conv_in_f16(x_nchw.contiguous().data_ptr(), w.data_ptr(), bias.data_ptr(), B, Cin,
                                                   H, W, Cout, y.data_ptr(), _stream(x_nchw)))
    return y


def conv_out(x_nhwc: torch.Tensor, w_packed: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """(B, H, W, Cin) NHWC -> (B, Cout<=8, H, W) NCHW; w_packed: (Cout, 3, 3, Cin)."""
    _f16(x_nhwc, "x")
    B, H, W, Cin = x_nhwc.shape
    Cout = w_packed.shape[0]
    y = torch.empty((B, Cout, H, W), dtype=torch.float16, device=x_nhwc.device)
    with torch.cuda.device(x_nhwc.device):
        _native.check(_native.lib().rf_conv_out_f16(x_nhwc.data_ptr(), w_packed.data_ptr(), bias.data_ptr(), B, H, W, Cin,
                                                    Cout, y.data_ptr(), _stream(x_nhwc)))
    return y


def timestep_embedding(t: torch.Tensor, dim: int) -> torch.Tensor:
    """t: fp32 (B,) device tensor -> (B, dim) fp16 [cos | sin]."""
    assert t.is_cuda and t.dtype == torch.float32
    out = torch.empty((t.shape[0], dim), dtype=torch.float16, device=t.device)
    with torch.cuda.device(t.device):
        _native.check(_native.lib().rf_timestep_embedding_f16(t.data_ptr(), t.shape[0], dim, out.data_ptr(), _stream(t)))
    return out


def silu(x: torch.Tensor) -> torch.Tensor:
    _f16(x, "x")
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _native.check(_native.lib().rf_silu_f16(x.data_ptr(), x.numel(), y.data_ptr(), _stream(x)))
    return y


def cfg_pndm_step(eps_pair, guidance, hist, coef, sample, ca, cb, want_eps=True):
    """eps_pair: (2B, ...) fp16 [uncond | text]; hist: up to 3 earlier guided eps tensors (most recent first);
    coef: 4 floats; returns (guided eps or None, prev_sample)."""
    _f16(eps_pair, "eps_pair"), _f16(sample, "sample")
    n = sample.numel()
    assert eps_pair.numel() == 2 * n and eps_pair.is_contiguous() and sample.is_contiguous()
    eps_out = torch.empty_like(sample) if want_eps else None
    prev = torch.empty_like(sample)
    h = [None if i >= len(hist) else hist[i].data_ptr() for i in range(3)]
    c4 = (C.c_float * 4)(*[float(v) for v in coef])
    with torch.cuda.device(sample.device):
        _native.check(_native.lib().rf_cfg_pndm_step_f16(
            eps_pair.data_ptr(), n, float(guidance), h[0], h[1], h[2], c4, sample.data_ptr(), float(ca), float(cb),
            None if eps_out is None else eps_out.data_ptr(), prev.data_ptr(), _stream(sample)))
    return eps_out, prev


def cfg_dpmpp_step(eps_pair, guidance, sample, x0_prev, sigma_s, alpha_s, c_x, c_0, inv_r0=0.0, c_d1=0.0, x0_out=None,
                   out=None):
    """Guidance combine + one DPM-Solver++ update (rf_cfg_dpmpp_step_f16).  eps_pair: (2B, ...) fp16 [uncond | text];
    x0_prev: the previous step's x0 prediction (second order) or None (first order).  Returns (x0 prediction, prev_sample);
    `x0_out` / `out` receive them when given (`out` may be `sample`)."""
    _f16(eps_pair, "eps_pair"), _f16(sample, "sample")
    n = sample.numel()
    assert eps_pair.numel() == 2 * n and eps_pair.is_contiguous() and sample.is_contiguous()
    for t in (x0_prev, x0_out, out):
        if t is not None:
            _f16(t, "history / output")
            assert t.numel() == n and t.is_contiguous()
    x0_out = torch.empty_like(sample) if x0_out is None else x0_out
    out = torch.empty_like(sample) if out is None else out
    with torch.cuda.device(sample.device):
        _native.check(_native.lib().rf_cfg_dpmpp_step_f16(
            eps_pair.data_ptr(), n, float(guidance), sample.data_ptr(), None if x0_prev is None else x0_prev.data_ptr(),
            float(sigma_s), float(alpha_s), float(c_x), float(c_0), float(inv_r0), float(c_d1), x0_out.data_ptr(),
            out.data_ptr(), _stream(sample)))
    return x0_out, out


def axpby(x, noise, a, b, mask=None, z=None):
    _f16(x, "x")
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _native.check(_native.lib().rf_axpby_f16(x.data_ptr(), noise.data_ptr(), float(a), float(b),
                                                 None if mask is None else mask.data_ptr(),
                                                 None if z is None else z.data_ptr(), x.numel(), y.data_ptr(), _stream(x)))
    return y


def add_noise_f16_seq(x, noise, s, s1):
    """diffusers 0.9 add_noise as its fp16 ops run it (rf_add_noise_f16_seq): fp16(fp16(s x) + fp16(s1 noise)), with s and
    s1 the fp16 values of sqrt(a[t]) and sqrt(1 - a[t])."""
    _f16(x, "x"), _f16(noise, "noise")
    assert noise.shape == x.shape
    x, noise = x.contiguous(), noise.contiguous()
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _native.check(_native.lib().rf_add_noise_f16_seq(x.data_ptr(), noise.data_ptr(), float(s), float(s1), x.numel(),
                                                         y.data_ptr(), _stream(x)))
    return y


def resample_u8(x_nhwc: torch.Tensor, height: int, width: int) -> torch.Tensor:
    """Pillow-exact `Image.resize((width, height), Image.BICUBIC)` of a batch: (B, H, W, 3) uint8 -> (B, height, width, 3)
    uint8 (rf_resample_u8)."""
    x = _native.require_cuda(x_nhwc, "image", torch.uint8)
    B, H, W, Cc = x.shape
    assert Cc == 3
    y = torch.empty((B, height, width, 3), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(_native.lib().rf_resample_u8(x.data_ptr(), B, H, W, height, width, y.data_ptr(), _stream(x)))
    return y


def resample_coeffs(n_in: int, n_out: int):
    """Host tables of rf_resample_u8 along one axis: (bounds (n_out, 2) int32, taps (n_out, ksize) int32)."""
    import numpy as np

    ksize = C.c_int()
    _native.check(_native.lib().rf_resample_coeffs(n_in, n_out, C.byref(ksize), None, None))
    bounds = np.zeros((n_out, 2), np.int32)
    kk = np.zeros((n_out, ksize.value), np.int32)
    _native.check(_native.lib().rf_resample_coeffs(n_in, n_out, C.byref(ksize), bounds.ctypes.data, kk.ctypes.data))
    return bounds, kk


def image_u8_to_f16(x_nhwc: torch.Tensor) -> torch.Tensor:
    """(B, H, W, 3) uint8 -> (B, 3, H, W) fp16 in [-1, 1]: img2img's preprocess (`/ 255`, `2x - 1` in fp32) + `.half()`."""
    x = _native.require_cuda(x_nhwc, "image", torch.uint8)
    B, H, W, Cc = x.shape
    assert Cc == 3
    y = torch.empty((B, 3, H, W), dtype=torch.float16, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(_native.lib().rf_image_u8_to_f16(x.data_ptr(), B, H, W, y.data_ptr(), _stream(x)))
    return y


def conv1x1_small(x_nchw: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, in_scale: float = 1.0) -> torch.Tensor:
    """(B, Cin<=8, H, W) NCHW -> (B, Cout<=8, H, W); w: (Cout, Cin) fp16."""
    _f16(x_nchw, "x")
    B, Cin, H, W = x_nchw.shape
    Cout = w.shape[0]
    y = torch.empty((B, Cout, H, W), dtype=torch.float16, device=x_nchw.device)
    with torch.cuda.device(x_nchw.device):
        _native.check(_native.lib().rf_conv1x1_small_f16(x_nchw.contiguous().data_ptr(), w.data_ptr(), bias.data_ptr(), B, Cin,
                                                         Cout, H * W, float(in_scale), y.data_ptr(), _stream(x_nchw)))
    return y


def attention(q: torch.Tensor, k: torch.Tensor, vt: torch.Tensor, heads: int, nk: int, causal: bool = False) -> torch.Tensor:
    """q: (B, Nq, C), k: (B, >=nk, C), vt: (B, C, pitch>=nk) fp16 contiguous -> (B, Nq, C); fused tcgen05 kernel.
    causal: key j is visible to query i iff j <= i (text encoder; nk <= 128)."""
    _f16(q, "q"), _f16(k, "k"), _f16(vt, "vt")
    B, Nq, C = q.shape
    d = C // heads
    assert q.is_contiguous() and k.is_contiguous() and vt.is_contiguous() and k.shape[1] == nk
    out = torch.empty_like(q)
    with torch.cuda.device(q.device):
        _native.check(_native.lib().rf_attention_masked_f16(q.data_ptr(), k.data_ptr(), vt.data_ptr(), out.data_ptr(), B, heads,
                                                            Nq, nk, d, vt.shape[-1], float(d) ** -0.5, int(causal), _stream(q)))
    return out


def vae_image_to_u8(x_nchw: torch.Tensor, fp32_scale: bool = False) -> torch.Tensor:
    """(B, 3, H, W) fp16 in [-1, 1] -> (B, H, W, 3) uint8, the array PIL images are built from.  `fp32_scale`: `* 255`
    and the round in fp32, as the txt2img pipeline does; otherwise in fp16, as the img2img pipeline does."""
    _f16(x_nchw, "x")
    B, Cc, H, W = x_nchw.shape
    assert Cc == 3
    y = torch.empty((B, H, W, 3), dtype=torch.uint8, device=x_nchw.device)
    fn = _native.lib().rf_vae_image_to_u8_f32scale if fp32_scale else _native.lib().rf_vae_image_to_u8
    with torch.cuda.device(x_nchw.device):
        _native.check(fn(x_nchw.contiguous().data_ptr(), B, H, W, y.data_ptr(), _stream(x_nchw)))
    return y


def slerp(alphas, v0: torch.Tensor, v1: torch.Tensor, dot_threshold: float = 0.9995) -> torch.Tensor:
    """Per-sample spherical interpolation on the device.  v0, v1: (B, ...) fp16; alphas: float or sequence of B floats."""
    _f16(v0, "v0"), _f16(v1, "v1")
    B = v0.shape[0]
    n = v0.numel() // B
    if not torch.is_tensor(alphas):
        alphas = torch.tensor([float(alphas)] * B if not hasattr(alphas, "__len__") else [float(a) for a in alphas],
                              dtype=torch.float32)
    al = alphas.to(device=v0.device, dtype=torch.float32).contiguous()
    out = torch.empty_like(v0)
    scratch = torch.empty(3 * B, dtype=torch.float32, device=v0.device)
    with torch.cuda.device(v0.device):
        _native.check(_native.lib().rf_slerp_f16(v0.contiguous().data_ptr(), v1.contiguous().data_ptr(), B, n, al.data_ptr(),
                                                 float(dot_threshold), out.data_ptr(), scratch.data_ptr(), _stream(v0)))
    return out
