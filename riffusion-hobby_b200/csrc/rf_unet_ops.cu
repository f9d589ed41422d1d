// Path (b) memory-bound operators around the tensor-core GEMM/conv kernel: GroupNorm(+SiLU),
// LayerNorm, GEGLU, row softmax, nearest-2x upsample, the 4-/3-channel edge convolutions, the
// sinusoidal timestep embedding, and the scheduler / guidance element-wise steps.
// Activations fp16 (NHWC), statistics and arithmetic fp32.
//
// Reference arithmetic (reached from riffusion/riffusion_pipeline.py:379,403-425 through diffusers
// 0.9 [restated from memory, package absent]): torch.nn.GroupNorm / LayerNorm / F.gelu / softmax /
// F.interpolate(nearest) / Conv2d, PNDMScheduler.step, classifier-free guidance combine.
#include <cuda_fp16.h>
#include <cmath>
#include <cstdlib>
#include <cuda_runtime.h>

#include <algorithm>
#include <string>

#include "rf_common.h"

namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float silu(float v) { return v / (1.f + __expf(-v)); }

// ---------------------------------------------------------------- GroupNorm (NHWC), deterministic
// pass 1: per (image, slab of pixels, group) partial sum and sum of squares.  Threads read 16-byte channel octets,
//         park their partials in shared memory, and one thread per group adds them in a fixed order (no atomics:
//         repeated runs are bit-identical).
// pass 2 (inside the apply kernel): the slab partials are added in a fixed order -> (mean, rstd) per group.
// pass 3: y = (x - mean) * rstd * gamma + beta, optional SiLU.
// Vectorised pass 1 (C % 8 == 0, C <= 2560): blockDim = PPI * C/8 threads; a thread owns 8 fixed channels (one 16-byte
// load per pixel) and walks every PPI-th pixel of the slab, four loads in flight.  Same deterministic two-level sum.
// Two-source form (x2 != nullptr): the input is the channel concatenation [x | x2] (C1 + (C - C1) channels,
// torch.cat([x, skip], dim=1) of the up blocks) read in place — a thread's 8 channels come from one of the two tensors.
__global__ void k_gn_partial_v(const __half* __restrict__ x, const __half* __restrict__ x2, int C1, int HW, int C, int G,
                               int slab, int nslabs, float* __restrict__ part /*[B][nslabs][G][2]*/) {
    extern __shared__ float2 shp[];  // [PPI][C/2]
    rf_pdl_trigger();      // PDL (rf_common.h)
    rf_pdl_wait();
    const int b = blockIdx.y;
    const int C2 = C >> 1;
    const int c8 = threadIdx.x % (C >> 3), pp = threadIdx.x / (C >> 3), PPI = blockDim.x / (C >> 3);
    const int p0 = blockIdx.x * slab, p1 = min(HW, p0 + slab);
    const bool second = x2 != nullptr && c8 * 8 >= C1;
    const int C8 = (second ? C - C1 : C1) >> 3;              // row pitch of the source tensor in 16-byte units
    const uint4* xb = reinterpret_cast<const uint4*>((second ? x2 : x) + static_cast<size_t>(b) * HW * (C8 * 8)) +
                      (second ? c8 - (C1 >> 3) : c8);
    float s[4] = {0.f, 0.f, 0.f, 0.f}, ss[4] = {0.f, 0.f, 0.f, 0.f};
    auto acc = [&](const uint4& v) {
        const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float2 f = __half22float2(h[j]);
            s[j] += f.x + f.y;
            ss[j] = fmaf(f.x, f.x, fmaf(f.y, f.y, ss[j]));
        }
    };
    int p = p0 + pp;
    for (; p + 3 * PPI < p1; p += 4 * PPI) {
        const uint4 v0 = xb[static_cast<size_t>(p) * C8], v1 = xb[static_cast<size_t>(p + PPI) * C8];
        const uint4 v2 = xb[static_cast<size_t>(p + 2 * PPI) * C8], v3 = xb[static_cast<size_t>(p + 3 * PPI) * C8];
        acc(v0); acc(v1); acc(v2); acc(v3);
    }
    for (; p < p1; p += PPI) acc(xb[static_cast<size_t>(p) * C8]);
#pragma unroll
    for (int j = 0; j < 4; ++j) shp[pp * C2 + c8 * 4 + j] = make_float2(s[j], ss[j]);
    __syncthreads();
    const int cpg2 = (C / G) >> 1;
    for (int g = threadIdx.x; g < G; g += blockDim.x) {
        float a = 0.f, q = 0.f;
        for (int w = 0; w < PPI; ++w)
            for (int k = 0; k < cpg2; ++k) {
                const float2 v = shp[w * C2 + g * cpg2 + k];
                a += v.x;
                q += v.y;
            }
        float* o = part + ((static_cast<size_t>(b) * nslabs + blockIdx.x) * G + g) * 2;
        o[0] = a;
        o[1] = q;
    }
}

// silu(x) = x * sigmoid(x) = h + h * tanh(h), h = x/2: one MUFU op (tanh.approx, 2^-11 relative) instead of ex2 + rcp
__device__ __forceinline__ float silu_tanh(float v) {
    const float h = 0.5f * v;
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    return fmaf(h, t, h);
}

// accurate form: x / (1 + 2^(-x log2 e)) with ex2.approx + rcp.approx (two MUFU ops, ~2^-21 relative).  The GroupNorm apply
// pass moves 4 bytes per element, so even at full HBM speed it needs < 80 % of the MUFU rate with two ops per element.
// tanh.approx (2^-11 relative = one fp16 ulp of extra noise on every GroupNorm+SiLU output) showed up as the largest
// difference between the kernels and the fp16-storage emulation of the oracle.
__device__ __forceinline__ float silu_exp(float v) {
    return __fdividef(v, 1.f + __expf(-v));
}

// Vectorised pass 3, same thread -> channel mapping: the affine form y = x * sc + sh (sc = rstd * gamma,
// sh = beta - mean * sc) of the thread's 8 channels lives in registers for the whole slab.
__global__ void k_gn_apply_v(const __half* __restrict__ x, const __half* __restrict__ x2, int C1,
                             const float* __restrict__ part, int nslabs, float inv_n,
                             float eps, const __half* __restrict__ gamma, const __half* __restrict__ beta, int HW, int C,
                             int G, int act, int slab, __half* __restrict__ y) {
    // pass 2 folded in: every CTA reduces the slab partials of its image to (mean, rstd) per group — a few KB from L2, in a
    // fixed order (P strided sub-sums per group, then added in index order), instead of a separate launch
    __shared__ float st[64 * 2];              // [G][2] mean, rstd   (G <= 64)
    rf_pdl_trigger();      // PDL (rf_common.h)
    rf_pdl_wait();
    __shared__ float sub[64 * 8 * 2];
    const int b = blockIdx.y;
    {
        const int P = min(8, static_cast<int>(blockDim.x) / G);
        const int t = threadIdx.x;
        if (t < G * P) {
            const int g = t / P, pi = t - g * P;
            float s = 0.f, ss = 0.f;
            for (int i = pi; i < nslabs; i += P) {
                const float* o = part + ((static_cast<size_t>(b) * nslabs + i) * G + g) * 2;
                s += o[0];
                ss += o[1];
            }
            sub[(g * 8 + pi) * 2] = s;
            sub[(g * 8 + pi) * 2 + 1] = ss;
        }
        __syncthreads();
        if (t < G) {
            float s = 0.f, ss = 0.f;
            for (int pi = 0; pi < P; ++pi) {
                s += sub[(t * 8 + pi) * 2];
                ss += sub[(t * 8 + pi) * 2 + 1];
            }
            const float mean = s * inv_n;
            const float var = fmaxf(ss * inv_n - mean * mean, 0.f);
            st[2 * t] = mean;
            st[2 * t + 1] = rsqrtf(var + eps);
        }
        __syncthreads();
    }
    const int C8 = C >> 3;
    const int c8 = threadIdx.x % C8, pp = threadIdx.x / C8, PPI = blockDim.x / C8;
    const int p0 = blockIdx.x * slab, p1 = min(HW, p0 + slab);
    const int cpg = C / G;
    float sc[8], sh[8];
    {
        const uint4 gv = *reinterpret_cast<const uint4*>(gamma + c8 * 8);
        const uint4 bv = *reinterpret_cast<const uint4*>(beta + c8 * 8);
        const __half* gh = reinterpret_cast<const __half*>(&gv);
        const __half* bh = reinterpret_cast<const __half*>(&bv);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int g = (c8 * 8 + e) / cpg;
            const float mean = st[2 * g], rstd = st[2 * g + 1];
            sc[e] = rstd * __half2float(gh[e]);
            sh[e] = fmaf(-mean, sc[e], __half2float(bh[e]));
        }
    }
    const bool second = x2 != nullptr && c8 * 8 >= C1;
    const int S8 = (second ? C - C1 : C1) >> 3;             // row pitch of the source tensor in 16-byte units
    const uint4* xb = reinterpret_cast<const uint4*>((second ? x2 : x) + static_cast<size_t>(b) * HW * (S8 * 8)) +
                      (second ? c8 - (C1 >> 3) : c8);
    uint4* yb = reinterpret_cast<uint4*>(y + static_cast<size_t>(b) * HW * C) + c8;
    auto xf = [&](uint4 v) -> uint4 {
        __half2* h = reinterpret_cast<__half2*>(&v);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float2 f = __half22float2(h[j]);
            float o0 = fmaf(f.x, sc[2 * j], sh[2 * j]), o1 = fmaf(f.y, sc[2 * j + 1], sh[2 * j + 1]);
            if (act == 1) {
                o0 = silu_exp(o0);
                o1 = silu_exp(o1);
            } else if (act == 2) {
                o0 = silu_tanh(o0);
                o1 = silu_tanh(o1);
            }
            h[j] = __floats2half2_rn(o0, o1);
        }
        return v;
    };
    int p = p0 + pp;
    for (; p + 3 * PPI < p1; p += 4 * PPI) {
        const uint4 v0 = xb[static_cast<size_t>(p) * S8], v1 = xb[static_cast<size_t>(p + PPI) * S8];
        const uint4 v2 = xb[static_cast<size_t>(p + 2 * PPI) * S8], v3 = xb[static_cast<size_t>(p + 3 * PPI) * S8];
        yb[static_cast<size_t>(p) * C8] = xf(v0);
        yb[static_cast<size_t>(p + PPI) * C8] = xf(v1);
        yb[static_cast<size_t>(p + 2 * PPI) * C8] = xf(v2);
        yb[static_cast<size_t>(p + 3 * PPI) * C8] = xf(v3);
    }
    for (; p < p1; p += PPI) yb[static_cast<size_t>(p) * C8] = xf(xb[static_cast<size_t>(p) * S8]);
}

// ---------------------------------------------------------------- LayerNorm over the last dim
__global__ void k_layernorm(const __half* __restrict__ x, const __half* __restrict__ gamma,
                            const __half* __restrict__ beta, int rows, int C, float eps, __half* __restrict__ y) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const __half2* xr = reinterpret_cast<const __half2*>(x + static_cast<size_t>(row) * C);
    float s = 0.f, ss = 0.f;
    for (int i = lane; i < C / 2; i += 32) {
        const float2 v = __half22float2(xr[i]);
        s += v.x + v.y;
        ss += v.x * v.x + v.y * v.y;
    }
    s = warp_sum(s);
    ss = warp_sum(ss);
    const float mean = s / C;
    const float rstd = rsqrtf(fmaxf(ss / C - mean * mean, 0.f) + eps);
    __half2* yr = reinterpret_cast<__half2*>(y + static_cast<size_t>(row) * C);
    const __half2* g2 = reinterpret_cast<const __half2*>(gamma);
    const __half2* b2 = reinterpret_cast<const __half2*>(beta);
    for (int i = lane; i < C / 2; i += 32) {
        const float2 v = __half22float2(xr[i]);
        const float2 ga = __half22float2(g2[i]);
        const float2 be = __half22float2(b2[i]);
        yr[i] = __floats2half2_rn((v.x - mean) * rstd * ga.x + be.x, (v.y - mean) * rstd * ga.y + be.y);
    }
}

// Vectorised LayerNorm for C = 40 * LPR (320, 640, 1280): LPR lanes per row (8 / 16 / 32), 32 / LPR rows per warp; a lane
// holds five 16-byte vectors of its row in registers between the statistics and the normalisation, so the row is read
// once (the scalar kernel above issues 4-byte loads and reads the row twice: 93 us for the 64x64 level at batch 64, i.e.
// 3.6 TB/s).
template <int LPR>
__global__ void __launch_bounds__(256) k_layernorm_v(const __half* __restrict__ x, const __half* __restrict__ gamma,
                                                     const __half* __restrict__ beta, int rows, float eps,
                                                     __half* __restrict__ y) {
    constexpr int NV = 5, C = 8 * NV * LPR, RPW = 32 / LPR;
    rf_pdl_trigger();      // PDL (rf_common.h)
    rf_pdl_wait();
    const int lane = threadIdx.x & 31, sub = lane % LPR;
    const int row = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RPW + lane / LPR;
    const bool ok = row < rows;
    const uint4* xr = reinterpret_cast<const uint4*>(x + static_cast<size_t>(ok ? row : 0) * C);
    uint4 v[NV];
    float s = 0.f, ss = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        v[i] = ok ? xr[sub + LPR * i] : make_uint4(0, 0, 0, 0);
        const __half2* h = reinterpret_cast<const __half2*>(&v[i]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float2 f = __half22float2(h[j]);
            s += f.x + f.y;
            ss += f.x * f.x + f.y * f.y;
        }
    }
#pragma unroll
    for (int o = LPR / 2; o; o >>= 1) {       // the lanes of a row are consecutive: xor-shuffles stay inside the group
        s += __shfl_xor_sync(0xffffffffu, s, o);
        ss += __shfl_xor_sync(0xffffffffu, ss, o);
    }
    const float mean = s * (1.f / C);
    const float rstd = rsqrtf(fmaxf(ss * (1.f / C) - mean * mean, 0.f) + eps);
    if (!ok) return;
    uint4* yr = reinterpret_cast<uint4*>(y + static_cast<size_t>(row) * C);
    const uint4* g4 = reinterpret_cast<const uint4*>(gamma);
    const uint4* b4 = reinterpret_cast<const uint4*>(beta);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const uint4 gv = g4[sub + LPR * i], bv = b4[sub + LPR * i];
        const __half2* gh = reinterpret_cast<const __half2*>(&gv);
        const __half2* bh = reinterpret_cast<const __half2*>(&bv);
        __half2* h = reinterpret_cast<__half2*>(&v[i]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float2 f = __half22float2(h[j]);
            const float2 ga = __half22float2(gh[j]);
            const float2 be = __half22float2(bh[j]);
            h[j] = __floats2half2_rn((f.x - mean) * rstd * ga.x + be.x, (f.y - mean) * rstd * ga.y + be.y);
        }
        yr[sub + LPR * i] = v[i];
    }
}

// ---------------------------------------------------------------- GEGLU: y = h * gelu(gate), [rows][2*inner] -> [rows][inner]
__global__ void k_geglu(const __half* __restrict__ x, size_t rows, int inner, __half* __restrict__ y) {
    const size_t n2 = rows * (inner / 2);
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n2;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t r = i / (inner / 2);
        const int c2 = static_cast<int>(i % (inner / 2));
        const __half2* xr = reinterpret_cast<const __half2*>(x + r * 2 * inner);
        const float2 h = __half22float2(xr[c2]);
        const float2 g = __half22float2(xr[inner / 2 + c2]);
        const float g0 = 0.5f * g.x * (1.f + erff(g.x * 0.70710678118654752f));  // exact (erf) GELU
        const float g1 = 0.5f * g.y * (1.f + erff(g.y * 0.70710678118654752f));
        reinterpret_cast<__half2*>(y + r * inner)[c2] = __floats2half2_rn(h.x * g0, h.y * g1);
    }
}

// ---------------------------------------------------------------- row softmax (fp16 in/out, fp32 math), one warp per row
__global__ void k_softmax_rows(const __half* __restrict__ x, size_t rows, int n, int pitch, __half* __restrict__ y) {
    const size_t row = static_cast<size_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const __half* xr = x + row * pitch;
    __half* yr = y + row * pitch;
    float m = -INFINITY;
    for (int i = lane; i < n; i += 32) m = fmaxf(m, __half2float(xr[i]));
    m = warp_max(m);
    float s = 0.f;
    for (int i = lane; i < n; i += 32) s += __expf(__half2float(xr[i]) - m);
    s = warp_sum(s);
    const float inv = 1.f / s;
    for (int i = lane; i < n; i += 32) yr[i] = __float2half_rn(__expf(__half2float(xr[i]) - m) * inv);
    for (int i = n + lane; i < pitch; i += 32) yr[i] = __float2half_rn(0.f);  // zero the pitch padding
}

// ---------------------------------------------------------------- nearest 2x upsample (NHWC)
__global__ void k_upsample2x(const __half* __restrict__ x, int B, int H, int W, int C, __half* __restrict__ y) {
    const int C8 = C / 8;
    const size_t n = static_cast<size_t>(B) * 2 * H * 2 * W * C8;
    const uint4* xs = reinterpret_cast<const uint4*>(x);
    uint4* ys = reinterpret_cast<uint4*>(y);
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int c = static_cast<int>(i % C8);
        size_t p = i / C8;
        const int xo = static_cast<int>(p % (2 * W));
        p /= 2 * W;
        const int yo = static_cast<int>(p % (2 * H));
        const int b = static_cast<int>(p / (2 * H));
        ys[i] = xs[((static_cast<size_t>(b) * H + yo / 2) * W + xo / 2) * C8 + c];
    }
}

// ---------------------------------------------------------------- edge convolutions (tiny channel counts)
// conv_in: NCHW fp16 (B, Cin<=8, H, W) -> NHWC fp16 (B, H, W, Cout), 3x3 pad 1. weights [Cout][Cin][3][3] fp16.
// CTA = 64 consecutive pixels (8 per warp); the weights are staged once per CTA, transposed to [k][cout] so that
// lanes (consecutive couts) read conflict-free and write coalesced NHWC rows.
__global__ void k_conv_in_generic(const __half* __restrict__ x, const __half* __restrict__ w, const __half* __restrict__ bias,
                          int B, int Cin, int H, int W, int Cout, __half* __restrict__ y) {
    extern __shared__ float wsm[];  // [Cin*9][Cout]
    const int K = Cin * 9;
    for (int i = threadIdx.x; i < Cout * K; i += blockDim.x) {
        const int co = i / K, k = i - co * K;
        wsm[k * Cout + co] = __half2float(w[i]);
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const size_t npix = static_cast<size_t>(B) * H * W;
    for (int j = 0; j < 8; ++j) {
        const size_t pix = static_cast<size_t>(blockIdx.x) * 64 + warp * 8 + j;
        if (pix >= npix) break;
        const int xq = static_cast<int>(pix % W), yq = static_cast<int>((pix / W) % H);
        const int b = static_cast<int>(pix / (static_cast<size_t>(W) * H));
        float in[72];
#pragma unroll 1
        for (int k = 0; k < K; ++k) {
            const int c = k / 9, t = k - c * 9;
            const int yy = yq + t / 3 - 1, xx = xq + t % 3 - 1;
            in[k] = (yy >= 0 && yy < H && xx >= 0 && xx < W)
                        ? __half2float(x[((static_cast<size_t>(b) * Cin + c) * H + yy) * W + xx])
                        : 0.f;
        }
        for (int co = lane; co < Cout; co += 32) {
            float acc = bias ? __half2float(bias[co]) : 0.f;
            for (int k = 0; k < K; ++k) acc += wsm[k * Cout + co] * in[k];
            y[pix * Cout + co] = __float2half_rn(acc);
        }
    }
}

// conv_out: NHWC fp16 (B, H, W, Cin) -> NCHW fp16/fp32 (B, Cout<=8, H, W), 3x3 pad 1. weights packed [Cout][3][3][Cin].
// One warp per output pixel; lanes split the channels.
__global__ void k_conv_out_generic(const __half* __restrict__ x, const __half* __restrict__ w, const __half* __restrict__ bias,
                           int B, int H, int W, int Cin, int Cout, __half* __restrict__ y) {
    const size_t pix = static_cast<size_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (pix >= static_cast<size_t>(B) * H * W) return;
    const int xq = static_cast<int>(pix % W), yq = static_cast<int>((pix / W) % H), b = static_cast<int>(pix / (static_cast<size_t>(W) * H));
    float acc[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) acc[o] = 0.f;
    for (int t = 0; t < 9; ++t) {
        const int yy = yq + t / 3 - 1, xx = xq + t % 3 - 1;
        if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
        const __half* xp = x + ((static_cast<size_t>(b) * H + yy) * W + xx) * Cin;
        for (int c = lane; c < Cin; c += 32) {
            const float v = __half2float(xp[c]);
            for (int o = 0; o < Cout; ++o) acc[o] += v * __half2float(w[(static_cast<size_t>(o) * 9 + t) * Cin + c]);
        }
    }
    for (int o = 0; o < Cout; ++o) {
        const float s = warp_sum(acc[o]);
        if (lane == 0)
            y[((static_cast<size_t>(b) * Cout + o) * H + yq) * W + xq] = __float2half_rn(s + (bias ? __half2float(bias[o]) : 0.f));
    }
}

// conv_in, register-blocked: a warp computes 4 horizontally adjacent pixels x all Cout.  Lane owns the cout pairs
// {2 lane + 64 i}, i < NCO2 (half2 stores: one 128-byte row segment per warp store), weights fp32 [k][Cout] in shared
// memory (LDS.64, conflict-free), the 3 x 6 x Cin input patch of the group staged per warp and read by broadcast.
// Persistent grid: every CTA stages the weights once and its warps stride over the pixel groups.  Needs W % 4 == 0.
template <int NCO2>
__global__ void __launch_bounds__(256)
k_conv_in_blk(const __half* __restrict__ x, const __half* __restrict__ w, const __half* __restrict__ bias, int B, int Cin,
              int H, int W, __half* __restrict__ y) {
    constexpr int Cout = 64 * NCO2;
    extern __shared__ float wsm[];                 // [Cin*9][Cout], then 8 warps x 18*Cin patch floats
    const int K = Cin * 9;
    for (int i = threadIdx.x; i < Cout * K; i += blockDim.x) {
        const int co = i / K, k = i - co * K;      // torch layout [Cout][Cin][3][3] -> k = c*9 + dy*3 + dx
        wsm[k * Cout + co] = __half2float(w[i]);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* patch = wsm + K * Cout + warp * (18 * 8);   // [c][dy][col 6]
    __syncthreads();
    float2 bz[NCO2];
#pragma unroll
    for (int i = 0; i < NCO2; ++i)
        bz[i] = bias ? __half22float2(*reinterpret_cast<const __half2*>(bias + 2 * lane + 64 * i)) : make_float2(0.f, 0.f);
    const int gpr = W / 4;                          // groups per row
    const long ngroups = static_cast<long>(B) * H * gpr;
    for (long g = static_cast<long>(blockIdx.x) * 8 + warp; g < ngroups; g += static_cast<long>(gridDim.x) * 8) {
        const int x0 = static_cast<int>(g % gpr) * 4, yq = static_cast<int>((g / gpr) % H);
        const int b = static_cast<int>(g / (static_cast<long>(gpr) * H));
        __syncwarp();
        for (int e = lane; e < 18 * Cin; e += 32) {
            const int c = e / 18, r = e - c * 18, dy = r / 6, col = r - dy * 6;
            const int yy = yq + dy - 1, xx = x0 + col - 1;
            patch[e] = (yy >= 0 && yy < H && xx >= 0 && xx < W)
                           ? __half2float(x[((static_cast<size_t>(b) * Cin + c) * H + yy) * W + xx])
                           : 0.f;
        }
        __syncwarp();
        float2 acc[4][NCO2];
#pragma unroll
        for (int p_ = 0; p_ < 4; ++p_)
#pragma unroll
            for (int i = 0; i < NCO2; ++i) acc[p_][i] = bz[i];
        for (int c = 0; c < Cin; ++c)
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                const int dy = t / 3, dx = t % 3;
                const float* pr = patch + c * 18 + dy * 6 + dx;
                const float i0 = pr[0], i1 = pr[1], i2 = pr[2], i3 = pr[3];
                const float2* wr = reinterpret_cast<const float2*>(wsm + (c * 9 + t) * Cout) + lane;
#pragma unroll
                for (int i = 0; i < NCO2; ++i) {
                    const float2 wv = wr[32 * i];
                    acc[0][i].x += wv.x * i0; acc[0][i].y += wv.y * i0;
                    acc[1][i].x += wv.x * i1; acc[1][i].y += wv.y * i1;
                    acc[2][i].x += wv.x * i2; acc[2][i].y += wv.y * i2;
                    acc[3][i].x += wv.x * i3; acc[3][i].y += wv.y * i3;
                }
            }
        __half* yp = y + ((static_cast<size_t>(b) * H + yq) * W + x0) * Cout + 2 * lane;
#pragma unroll
        for (int p_ = 0; p_ < 4; ++p_)
#pragma unroll
            for (int i = 0; i < NCO2; ++i)
                *reinterpret_cast<__half2*>(yp + static_cast<size_t>(p_) * Cout + 64 * i) =
                    __floats2half2_rn(acc[p_][i].x, acc[p_][i].y);
    }
}

// conv_out, register-blocked: a warp computes 4 horizontally adjacent pixels x Cout (<= 4) outputs.  Lane owns the
// channel pairs {2 lane + 64 s}, s < NSTEP (coalesced 128-byte loads), weights fp32 in shared memory as
// [tap][s][2 halves of the cout quad][lane][4] (LDS.128, conflict-free).  The 6 input columns of a kernel row are
// loaded once and shared by the 3 horizontal taps of the 4 pixels.  Persistent grid.  Needs W % 4 == 0.
template <int NSTEP>
__global__ void __launch_bounds__(256)
k_conv_out_blk(const __half* __restrict__ x, const __half* __restrict__ w, const __half* __restrict__ bias, int B, int H,
               int W, int Cout, __half* __restrict__ y) {
    constexpr int Cin = 64 * NSTEP;
    extern __shared__ float wsm[];                 // [9][NSTEP][2][32][4]
    for (int i = threadIdx.x; i < 9 * NSTEP * 256; i += blockDim.x) {
        const int e = i & 3, ln = (i >> 2) & 31, hf = (i >> 7) & 1, s_ = (i >> 8) % NSTEP, t = i / (256 * NSTEP);
        const int o = 2 * hf + (e >> 1), c = 2 * ln + 64 * s_ + (e & 1);
        wsm[i] = o < Cout ? __half2float(w[(static_cast<size_t>(o) * 9 + t) * Cin + c]) : 0.f;   // packed [Cout][3][3][Cin]
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int gpr = W / 4;
    const long ngroups = static_cast<long>(B) * H * gpr;
    for (long g = static_cast<long>(blockIdx.x) * 8 + warp; g < ngroups; g += static_cast<long>(gridDim.x) * 8) {
        const int x0 = static_cast<int>(g % gpr) * 4, yq = static_cast<int>((g / gpr) % H);
        const int b = static_cast<int>(g / (static_cast<long>(gpr) * H));
        float acc[4][4];
#pragma unroll
        for (int p_ = 0; p_ < 4; ++p_)
#pragma unroll
            for (int o = 0; o < 4; ++o) acc[p_][o] = 0.f;
#pragma unroll 1
        for (int dy = 0; dy < 3; ++dy) {
            const int yy = yq + dy - 1;
            if (yy < 0 || yy >= H) continue;
            float2 in[6][NSTEP];
            const __half* row = x + ((static_cast<size_t>(b) * H + yy) * W) * Cin + 2 * lane;
#pragma unroll
            for (int col = 0; col < 6; ++col) {
                const int xx = x0 + col - 1;
                const bool ok = xx >= 0 && xx < W;
#pragma unroll
                for (int s_ = 0; s_ < NSTEP; ++s_)
                    in[col][s_] = ok ? __half22float2(*reinterpret_cast<const __half2*>(row + static_cast<size_t>(xx) * Cin + 64 * s_))
                                     : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int dx = 0; dx < 3; ++dx)
#pragma unroll
                for (int s_ = 0; s_ < NSTEP; ++s_) {
                    const float4* wq = reinterpret_cast<const float4*>(wsm) + (((dy * 3 + dx) * NSTEP + s_) * 2) * 32 + lane;
                    const float4 w01 = wq[0], w23 = wq[32];   // (o0c0, o0c1, o1c0, o1c1), (o2c0, o2c1, o3c0, o3c1)
#pragma unroll
                    for (int p_ = 0; p_ < 4; ++p_) {
                        const float2 v = in[p_ + dx][s_];
                        acc[p_][0] += v.x * w01.x + v.y * w01.y;
                        acc[p_][1] += v.x * w01.z + v.y * w01.w;
                        acc[p_][2] += v.x * w23.x + v.y * w23.y;
                        acc[p_][3] += v.x * w23.z + v.y * w23.w;
                    }
                }
        }
#pragma unroll
        for (int p_ = 0; p_ < 4; ++p_)
#pragma unroll
            for (int o = 0; o < 4; ++o) acc[p_][o] = warp_sum(acc[p_][o]);
#pragma unroll
        for (int o = 0; o < 4; ++o)
            if (lane == o && o < Cout) {
                const float bo = bias ? __half2float(bias[o]) : 0.f;
                const __half2 h01 = __floats2half2_rn(acc[0][o] + bo, acc[1][o] + bo);
                const __half2 h23 = __floats2half2_rn(acc[2][o] + bo, acc[3][o] + bo);
                uint2 pk;
                pk.x = *reinterpret_cast<const uint32_t*>(&h01);
                pk.y = *reinterpret_cast<const uint32_t*>(&h23);
                *reinterpret_cast<uint2*>(y + ((static_cast<size_t>(b) * Cout + o) * H + yq) * W + x0) = pk;
            }
    }
}

// ---------------------------------------------------------------- sinusoidal timestep embedding
// diffusers Timesteps(dim, flip_sin_to_cos=True, downscale_freq_shift=0): [cos(t f_i), sin(t f_i)], f_i = 10000^(-i/half)
__global__ void k_timestep_embedding(const float* __restrict__ t, int B, int dim, __half* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int half_dim = dim / 2;
    if (i >= B * half_dim) return;
    const int b = i / half_dim, k = i % half_dim;
    const float freq = expf(-logf(10000.f) * static_cast<float>(k) / static_cast<float>(half_dim));
    const float a = t[b] * freq;
    out[static_cast<size_t>(b) * dim + k] = __float2half_rn(cosf(a));
    out[static_cast<size_t>(b) * dim + half_dim + k] = __float2half_rn(sinf(a));
}

__global__ void k_silu(const __half* __restrict__ x, size_t n, __half* __restrict__ y) {
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<size_t>(gridDim.x) * blockDim.x)
        y[i] = __float2half_rn(silu(__half2float(x[i])));
}

// ---------------------------------------------------------------- guidance + scheduler element-wise step
// eps = eps_u + g (eps_t - eps_u)            (riffusion_pipeline.py:411-415, fp16 arithmetic like torch)
// e   = sum_j coef[j] * hist_j  (hist_0 = eps)  PNDM/PLMS linear multistep combination
// x'  = ca * x - cb * e                       PNDMScheduler._get_prev_sample
// All tensors fp16 NCHW (B,4,64,64); eps_pair holds [uncond batch | text batch].
__global__ void k_cfg_pndm_step(const __half* __restrict__ eps_pair, size_t n, float guidance,
                                const __half* __restrict__ h1, const __half* __restrict__ h2,
                                const __half* __restrict__ h3, float c0, float c1, float c2, float c3,
                                const __half* __restrict__ sample, float ca, float cb,
                                __half* __restrict__ eps_out, __half* __restrict__ prev_sample) {
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const __half eu = eps_pair[i], et = eps_pair[n + i];
        // torch evaluates this in fp16: (et - eu) rounded, * g rounded, + eu rounded
        const __half d = __hsub(et, eu);
        const __half gd = __float2half_rn(__half2float(d) * guidance);
        const __half e0 = __hadd(eu, gd);
        if (eps_out) eps_out[i] = e0;
        float e = c0 * __half2float(e0);
        if (h1) e += c1 * __half2float(h1[i]);
        if (h2) e += c2 * __half2float(h2[i]);
        if (h3) e += c3 * __half2float(h3[i]);
        prev_sample[i] = __float2half_rn(ca * __half2float(sample[i]) - cb * e);
    }
}

// ---------------------------------------------------------------- guidance + DPM-Solver++(2M) element-wise step
// The reference applies DPMSolverMultistepScheduler.step to fp16 CUDA tensors with 0-dim fp32 CPU scalars: every tensor
// op widens its fp16 operands, computes in fp32 with the scalar at full fp32 and rounds the result to fp16 once.
// torch divides by a CPU scalar as a multiply by its fp32 reciprocal.  This reproduces that op sequence, left to right:
//   e   = eu + g (et - eu)                                   (fp16, as k_cfg_pndm_step)
//   m0  = (x - sigma_s * e) * (1 / alpha_s)                  convert_model_output, x0 prediction
//   x_t = c_x * x - c_0 * m0                                 first order
//   x_t = c_x * x - c_0 * m0 - c_d1 * (inv_r0 * (m0 - m1))   second order (midpoint), m1 = the previous step's m0
struct DpmppCoef {
    float g, sigma_s, inv_alpha_s, c_x, c_0, inv_r0, c_d1;
};

__device__ __forceinline__ __half rn(float v) { return __float2half_rn(v); }
__device__ __forceinline__ float wf(__half v) { return __half2float(v); }

template <bool SECOND>
__device__ __forceinline__ void dpmpp_elem(__half eu, __half et, __half x, __half m1, const DpmppCoef& c, __half& m0_out,
                                           __half& xt_out) {
    const __half d = __hsub(et, eu);
    const __half e = __hadd(eu, rn(wf(d) * c.g));
    const __half m0 = rn(wf(rn(wf(x) - wf(rn(c.sigma_s * wf(e))))) * c.inv_alpha_s);
    __half xt = rn(wf(rn(c.c_x * wf(x))) - wf(rn(c.c_0 * wf(m0))));
    if constexpr (SECOND) {
        const __half d1 = rn(c.inv_r0 * wf(rn(wf(m0) - wf(m1))));
        xt = rn(wf(xt) - wf(rn(c.c_d1 * wf(d1))));
    }
    m0_out = m0;
    xt_out = xt;
}

// n8 elements (a multiple of 8, every stream 16-byte aligned except possibly the text half of eps_pair) in 16-byte
// groups, the remaining n - n8 < 8 one by one.  sample may alias prev_sample: each element is read before it is written
// by the same thread.
template <bool SECOND>
__global__ void k_cfg_dpmpp_step(const __half* __restrict__ eps_pair, size_t n, size_t n8, bool et_vec,
                                 const __half* sample, const __half* x0_prev, DpmppCoef c, __half* x0_out,
                                 __half* prev_sample) {
    const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
    const __half* et_base = eps_pair + n;
    for (size_t gi = tid; gi < n8 / 8; gi += stride) {
        const size_t i = gi * 8;
        union V8 { uint4 u; __half h[8]; };
        V8 eu, et, x, m1, m0, xt;
        eu.u = *reinterpret_cast<const uint4*>(eps_pair + i);
        if (et_vec) {
            et.u = *reinterpret_cast<const uint4*>(et_base + i);
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) et.h[k] = et_base[i + k];
        }
        x.u = *reinterpret_cast<const uint4*>(sample + i);
        if constexpr (SECOND) m1.u = *reinterpret_cast<const uint4*>(x0_prev + i);
        else m1.u = make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int k = 0; k < 8; ++k) dpmpp_elem<SECOND>(eu.h[k], et.h[k], x.h[k], m1.h[k], c, m0.h[k], xt.h[k]);
        *reinterpret_cast<uint4*>(x0_out + i) = m0.u;
        *reinterpret_cast<uint4*>(prev_sample + i) = xt.u;
    }
    for (size_t i = n8 + tid; i < n; i += stride) {
        __half m0, xt;
        dpmpp_elem<SECOND>(eps_pair[i], et_base[i], sample[i], SECOND ? x0_prev[i] : __half(), c, m0, xt);
        x0_out[i] = m0;
        prev_sample[i] = xt;
    }
}

// add_noise / mask blend: y = a*x + b*n (scheduler.add_noise), optionally blended y*m + z*(1-m)
__global__ void k_axpby(const __half* __restrict__ x, const __half* __restrict__ nz, float a, float b,
                        const __half* __restrict__ mask, const __half* __restrict__ z, size_t n,
                        __half* __restrict__ y) {
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        float v = a * __half2float(x[i]) + b * __half2float(nz[i]);
        if (mask) {
            const float m = __half2float(mask[i]);
            v = v * m + __half2float(z[i]) * (1.f - m);
        }
        y[i] = __float2half_rn(v);
    }
}

// diffusers 0.9 `add_noise` on fp16 tensors (DDPM / PNDM / DPM-Solver share it): alphas_cumprod is cast to the sample
// dtype, s = a[t] ** 0.5 and s1 = (1 - a[t]) ** 0.5 are fp16 values (computed on the host), and
//   y = s * x + s1 * n
// rounds to fp16 after every op (each op widens to fp32 and rounds its result once, as torch does).  n8 elements (a
// multiple of 8, every stream 16-byte aligned) in 16-byte groups, the remaining n - n8 < 8 one by one.
__device__ __forceinline__ __half add_noise_elem(__half x, __half nz, float s, float s1) {
    return rn(wf(rn(s * wf(x))) + wf(rn(s1 * wf(nz))));
}

__global__ void k_add_noise_seq(const __half* x, const __half* nz, float s, float s1, size_t n, size_t n8, __half* y) {
    const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
    for (size_t gi = tid; gi < n8 / 8; gi += stride) {
        const size_t i = gi * 8;
        union V8 { uint4 u; __half h[8]; };
        V8 a, b, o;
        a.u = *reinterpret_cast<const uint4*>(x + i);
        b.u = *reinterpret_cast<const uint4*>(nz + i);
#pragma unroll
        for (int k = 0; k < 8; ++k) o.h[k] = add_noise_elem(a.h[k], b.h[k], s, s1);
        *reinterpret_cast<uint4*>(y + i) = o.u;
    }
    for (size_t i = n8 + tid; i < n; i += stride) y[i] = add_noise_elem(x[i], nz[i], s, s1);
}

// channel concatenation of two NHWC tensors (torch.cat([a, b], dim=1) in NCHW terms)
__global__ void k_concat_channels(const __half* __restrict__ a, const __half* __restrict__ b, size_t pixels, int Ca,
                                  int Cb, __half* __restrict__ y) {
    const int C8 = (Ca + Cb) / 8, A8 = Ca / 8;
    const size_t n = pixels * C8;
    const uint4* as = reinterpret_cast<const uint4*>(a);
    const uint4* bs = reinterpret_cast<const uint4*>(b);
    uint4* ys = reinterpret_cast<uint4*>(y);
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t p = i / C8;
        const int c = static_cast<int>(i % C8);
        ys[i] = c < A8 ? as[p * A8 + c] : bs[p * (Cb / 8) + (c - A8)];
    }
}

// 1x1 convolution on tiny channel counts, NCHW: y[b][o][p] = bias[o] + sum_i w[o][i] * (in_scale * x[b][i][p])
__global__ void k_conv1x1_small(const __half* __restrict__ x, const __half* __restrict__ w, const __half* __restrict__ bias,
                                int B, int Cin, int Cout, size_t HW, float in_scale, __half* __restrict__ y) {
    const size_t n = static_cast<size_t>(B) * HW;
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t b = i / HW, p = i % HW;
        float in[8];
        for (int c = 0; c < Cin; ++c) in[c] = in_scale * __half2float(x[(b * Cin + c) * HW + p]);
        for (int o = 0; o < Cout; ++o) {
            float acc = bias ? __half2float(bias[o]) : 0.f;
            for (int c = 0; c < Cin; ++c) acc += __half2float(w[o * Cin + c]) * in[c];
            y[(b * Cout + o) * HW + p] = __float2half_rn(acc);
        }
    }
}

// VAE output -> PIL-equivalent uint8 image: (x/2 + 0.5).clamp(0,1) * 255, round half to even (numpy .round()),
// NCHW fp16 (B,3,H,W) -> NHWC uint8 (B,H,W,3)      (riffusion_pipeline.py:430-434 + numpy_to_pil)
// F32_SCALE: the txt2img pipeline's decode_latents, which calls `.float()` after the clamp, so `* 255` and the round
// happen in fp32 instead of fp16.
template <bool F32_SCALE>
__global__ void k_vae_to_u8(const __half* __restrict__ x, int B, size_t HW, uint8_t* __restrict__ y) {
    const size_t n = static_cast<size_t>(B) * HW;
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t b = i / HW, p = i % HW;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            // riffusion_pipeline.py:430-434 on the reference's fp16 CUDA path: `(image / 2 + 0.5).clamp(0, 1)` is fp16
            // tensor arithmetic (one rounding per op), `.numpy()` keeps float16, and numpy_to_pil's `(images * 255).round()`
            // is float16 arithmetic too (product rounded to fp16, then round-half-even) -> the same ops in __half here
            const __half h = __hadd(__hmul(x[(b * 3 + c) * HW + p], __float2half(0.5f)), __float2half(0.5f));
            const __half cl = __hmin(__hmax(h, __float2half(0.f)), __float2half(1.f));
            if constexpr (F32_SCALE)
                y[i * 3 + c] = static_cast<uint8_t>(__float2int_rn(__half2float(cl) * 255.f));
            else
                y[i * 3 + c] = static_cast<uint8_t>(__half2int_rn(hrint(__hmul(cl, __float2half(255.f)))));
        }
    }
}

// ---------------------------------------------------------------- slerp of noise tensors, per sample
// riffusion/util/torch_util.py:21-48 on the device: dot = <v0,v1>/(|v0||v1|); |dot| > thr -> lerp, else
// s0 = sin((1-t) th)/sin th, s1 = sin(t th)/sin th.  Reductions in fp32, fixed order (one CTA per sample).
__global__ void k_slerp_stats(const __half* __restrict__ v0, const __half* __restrict__ v1, size_t n,
                              float* __restrict__ stats /*[B][3]*/) {
    __shared__ float sh[3][32];
    const size_t b = blockIdx.x;
    const __half* a = v0 + b * n;
    const __half* c = v1 + b * n;
    float d = 0.f, aa = 0.f, cc = 0.f;
    for (size_t i = threadIdx.x; i < n; i += blockDim.x) {
        const float x = __half2float(a[i]), y = __half2float(c[i]);
        d += x * y;
        aa += x * x;
        cc += y * y;
    }
    d = warp_sum(d);
    aa = warp_sum(aa);
    cc = warp_sum(cc);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) {
        sh[0][w] = d;
        sh[1][w] = aa;
        sh[2][w] = cc;
    }
    __syncthreads();
    if (w == 0) {
        const int nw = blockDim.x >> 5;
        d = l < nw ? sh[0][l] : 0.f;
        aa = l < nw ? sh[1][l] : 0.f;
        cc = l < nw ? sh[2][l] : 0.f;
        d = warp_sum(d);
        aa = warp_sum(aa);
        cc = warp_sum(cc);
        if (l == 0) {
            stats[b * 3] = d;
            stats[b * 3 + 1] = aa;
            stats[b * 3 + 2] = cc;
        }
    }
}

__global__ void k_slerp_apply(const __half* __restrict__ v0, const __half* __restrict__ v1, size_t n,
                              const float* __restrict__ stats, const float* __restrict__ alphas, float thr,
                              __half* __restrict__ out) {
    const size_t b = blockIdx.y;
    const float t = alphas[b];
    const float dot = stats[b * 3] / (sqrtf(stats[b * 3 + 1]) * sqrtf(stats[b * 3 + 2]));
    float s0, s1;
    if (fabsf(dot) > thr) {
        s0 = 1.f - t;
        s1 = t;
    } else {
        const float th = acosf(dot), sn = sinf(th);
        s0 = sinf(th - th * t) / sn;
        s1 = sinf(th * t) / sn;
    }
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<size_t>(gridDim.x) * blockDim.x)
        out[b * n + i] = __float2half_rn(s0 * __half2float(v0[b * n + i]) + s1 * __half2float(v1[b * n + i]));
}

inline unsigned grid_for(size_t n, int block) {
    size_t g = (n + block - 1) / block;
    return static_cast<unsigned>(g > 148 * 16 ? 148 * 16 : (g ? g : 1));
}

}  // namespace

extern "C" size_t rf_group_norm_scratch_floats(int B, int HW, int groups) {
    const int nslabs = (HW + 31) / 32;
    return static_cast<size_t>(B) * groups * 2 * (static_cast<size_t>(nslabs) + 1);
}

extern "C" int rf_group_norm_f16(const void* x, int B, int HW, int C, int groups, const void* gamma, const void* beta,
                                 float eps, int act, void* y, float* d_scratch, void* stream) {
    return rf_group_norm_cat_f16(x, nullptr, C, B, HW, C, groups, gamma, beta, eps, act, y, d_scratch, stream);
}

extern "C" int rf_group_norm_cat_f16(const void* x, const void* x2, int C1, int B, int HW, int C, int groups,
                                     const void* gamma, const void* beta, float eps, int act, void* y, float* d_scratch,
                                     void* stream) {
    if (!x || !y || !gamma || !beta || !d_scratch || B <= 0 || HW <= 0 || C <= 0 || groups <= 0 || C % groups ||
        ((C / groups) & 1))
        return rf_fail(RF_ERR_INVALID, "rf_group_norm_f16: bad argument (channels per group must be even)");
    if (!x2) C1 = C;
    if (x2 && (C1 <= 0 || C1 >= C || (C1 % 8) || ((C - C1) % 8)))
        return rf_fail(RF_ERR_INVALID, "rf_group_norm_cat_f16: both channel counts must be positive multiples of 8");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (C > 2560 || (C % 8)) return rf_fail(RF_ERR_UNSUPPORTED, "rf_group_norm_f16: C must be a multiple of 8, <= 2560");
    // thread -> (pixel phase, 8-channel column): blockDim = PPI * C/8 (<= 320 threads)
    const int C8 = C / 8;
    const int PPI = C8 >= 256 ? 1 : 256 / C8;
    const int threads = PPI * C8;
    // slab: >= 32 pixels (the scratch is sized for HW/32 slabs); large images take longer slabs (still >= 4 waves)
    int slab = 32;
    while (slab < 256 && static_cast<long>(B) * (HW / (2 * slab)) >= 4 * 148) slab *= 2;
    const int nslabs = (HW + slab - 1) / slab;
    float* part = d_scratch + static_cast<size_t>(B) * groups * 2;     // [B][nslabs][G][2]
    const size_t smem = static_cast<size_t>(PPI) * (C / 2) * sizeof(float2);
    dim3 grid(nslabs, B);
    RF_LAUNCH_PDL("k_gn_partial_v", k_gn_partial_v, grid, dim3(threads), smem, st, grid.x * grid.y <= 600u, static_cast<const __half*>(x),
                  static_cast<const __half*>(x2), C1, HW, C, groups, slab, nslabs, part);
    if (groups > 64 || threads < groups) return rf_fail(RF_ERR_UNSUPPORTED, "rf_group_norm_f16: at most 64 groups (and not more groups than threads)");
    // tanh form by default: measured on the full-size UNet, both forms leave the kernels AT the fp16-storage floor
    // (1.420e-3 vs 1.418e-3 from the fp32 oracle) and the exp form costs +0.4 ms per evaluation at batch 64
    static const int silu_form = getenv("RF_SILU_EXACT") ? 1 : 2;
    RF_LAUNCH_PDL("k_gn_apply_v", k_gn_apply_v, grid, dim3(threads), size_t(0), st, grid.x * grid.y <= 600u, static_cast<const __half*>(x),
                  static_cast<const __half*>(x2), C1, static_cast<const float*>(part), nslabs,
                  1.f / (static_cast<float>(HW) * (C / groups)), eps, static_cast<const __half*>(gamma),
                  static_cast<const __half*>(beta), HW, C, groups, act ? silu_form : 0, slab, static_cast<__half*>(y));
    return RF_OK;
}

extern "C" int rf_layer_norm_f16(const void* x, int rows, int C, const void* gamma, const void* beta, float eps, void* y,
                                 void* stream) {
    if (!x || !y || !gamma || !beta || rows <= 0 || C <= 0 || (C & 1)) return rf_fail(RF_ERR_INVALID, "rf_layer_norm_f16: bad argument");
    const bool aligned = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(gamma) |
                           reinterpret_cast<uintptr_t>(beta)) & 15) == 0;
    if (aligned && (C == 320 || C == 640 || C == 1280)) {
        const int rpb = 8 * (C == 320 ? 4 : C == 640 ? 2 : 1);     // 8 warps x rows per warp
        const int blocks = (rows + rpb - 1) / rpb;
        cudaStream_t st = static_cast<cudaStream_t>(stream);
        const __half *xp = static_cast<const __half*>(x), *gp = static_cast<const __half*>(gamma),
                     *bp = static_cast<const __half*>(beta);
        __half* yp = static_cast<__half*>(y);
        if (C == 320) RF_LAUNCH_PDL("k_layernorm_v", k_layernorm_v<8>, dim3(blocks), dim3(256), size_t(0), st, blocks <= 600, xp, gp, bp, rows, eps, yp);
        else if (C == 640) RF_LAUNCH_PDL("k_layernorm_v", k_layernorm_v<16>, dim3(blocks), dim3(256), size_t(0), st, blocks <= 600, xp, gp, bp, rows, eps, yp);
        else RF_LAUNCH_PDL("k_layernorm_v", k_layernorm_v<32>, dim3(blocks), dim3(256), size_t(0), st, blocks <= 600, xp, gp, bp, rows, eps, yp);
        return RF_OK;
    }
    k_layernorm<<<(rows + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(x), static_cast<const __half*>(gamma), static_cast<const __half*>(beta), rows, C, eps,
        static_cast<__half*>(y));
    RF_CUDA_LAUNCH_CHECK("k_layernorm");
    return RF_OK;
}

extern "C" int rf_geglu_f16(const void* x, long rows, int inner, void* y, void* stream) {
    if (!x || !y || rows <= 0 || inner <= 0 || (inner & 1)) return rf_fail(RF_ERR_INVALID, "rf_geglu_f16: bad argument");
    const size_t n2 = static_cast<size_t>(rows) * (inner / 2);
    k_geglu<<<grid_for(n2, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __half*>(x),
                                                                             static_cast<size_t>(rows), inner,
                                                                             static_cast<__half*>(y));
    RF_CUDA_LAUNCH_CHECK("k_geglu");
    return RF_OK;
}

extern "C" int rf_softmax_rows_f16(const void* x, long rows, int n, int pitch, void* y, void* stream) {
    if (!x || !y || rows <= 0 || n <= 0 || pitch < n) return rf_fail(RF_ERR_INVALID, "rf_softmax_rows_f16: bad argument");
    const size_t blocks = (static_cast<size_t>(rows) + 7) / 8;
    k_softmax_rows<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(x), static_cast<size_t>(rows), n, pitch, static_cast<__half*>(y));
    RF_CUDA_LAUNCH_CHECK("k_softmax_rows");
    return RF_OK;
}

extern "C" int rf_upsample2x_f16(const void* x, int B, int H, int W, int C, void* y, void* stream) {
    if (!x || !y || B <= 0 || H <= 0 || W <= 0 || C <= 0 || (C % 8)) return rf_fail(RF_ERR_INVALID, "rf_upsample2x_f16: bad argument");
    const size_t n = static_cast<size_t>(B) * 4 * H * W * (C / 8);
    k_upsample2x<<<grid_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __half*>(x), B, H, W,
                                                                                 C, static_cast<__half*>(y));
    RF_CUDA_LAUNCH_CHECK("k_upsample2x");
    return RF_OK;
}

extern "C" int rf_concat_channels_f16(const void* a, const void* b, long pixels, int Ca, int Cb, void* y, void* stream) {
    if (!a || !b || !y || pixels <= 0 || Ca <= 0 || Cb <= 0 || (Ca % 8) || (Cb % 8))
        return rf_fail(RF_ERR_INVALID, "rf_concat_channels_f16: bad argument");
    const size_t n = static_cast<size_t>(pixels) * ((Ca + Cb) / 8);
    k_concat_channels<<<grid_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(a), static_cast<const __half*>(b), static_cast<size_t>(pixels), Ca, Cb,
        static_cast<__half*>(y));
    RF_CUDA_LAUNCH_CHECK("k_concat_channels");
    return RF_OK;
}

extern "C" int rf_slerp_f16(const void* v0, const void* v1, int B, long n, const float* d_alphas, float dot_threshold,
                            void* out, float* d_scratch, void* stream) {
    if (!v0 || !v1 || !out || !d_alphas || !d_scratch || B <= 0 || n <= 0) return rf_fail(RF_ERR_INVALID, "rf_slerp_f16: bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    k_slerp_stats<<<B, 256, 0, st>>>(static_cast<const __half*>(v0), static_cast<const __half*>(v1), static_cast<size_t>(n),
                                     d_scratch);
    RF_CUDA_LAUNCH_CHECK("k_slerp_stats");
    dim3 grid(grid_for(static_cast<size_t>(n), 256), B);
    k_slerp_apply<<<grid, 256, 0, st>>>(static_cast<const __half*>(v0), static_cast<const __half*>(v1), static_cast<size_t>(n),
                                        d_scratch, d_alphas, dot_threshold, static_cast<__half*>(out));
    RF_CUDA_LAUNCH_CHECK("k_slerp_apply");
    return RF_OK;
}

extern "C" int rf_conv1x1_small_f16(const void* x_nchw, const void* w, const void* bias, int B, int Cin, int Cout, long HW,
                                    float in_scale, void* y_nchw, void* stream) {
    if (!x_nchw || !w || !y_nchw || B <= 0 || Cin <= 0 || Cin > 8 || Cout <= 0 || Cout > 8 || HW <= 0)
        return rf_fail(RF_ERR_INVALID, "rf_conv1x1_small_f16: bad argument");
    k_conv1x1_small<<<grid_for(static_cast<size_t>(B) * HW, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(x_nchw), static_cast<const __half*>(w), static_cast<const __half*>(bias), B, Cin, Cout,
        static_cast<size_t>(HW), in_scale, static_cast<__half*>(y_nchw));
    RF_CUDA_LAUNCH_CHECK("k_conv1x1_small");
    return RF_OK;
}

extern "C" int rf_vae_image_to_u8(const void* x_nchw, int B, int H, int W, uint8_t* y_nhwc, void* stream) {
    if (!x_nchw || !y_nhwc || B <= 0 || H <= 0 || W <= 0) return rf_fail(RF_ERR_INVALID, "rf_vae_image_to_u8: bad argument");
    const size_t HW = static_cast<size_t>(H) * W;
    k_vae_to_u8<false><<<grid_for(static_cast<size_t>(B) * HW, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(x_nchw), B, HW, y_nhwc);
    RF_CUDA_LAUNCH_CHECK("k_vae_to_u8");
    return RF_OK;
}

extern "C" int rf_vae_image_to_u8_f32scale(const void* x_nchw, int B, int H, int W, uint8_t* y_nhwc, void* stream) {
    if (!x_nchw || !y_nhwc || B <= 0 || H <= 0 || W <= 0)
        return rf_fail(RF_ERR_INVALID, "rf_vae_image_to_u8_f32scale: bad argument");
    const size_t HW = static_cast<size_t>(H) * W;
    k_vae_to_u8<true><<<grid_for(static_cast<size_t>(B) * HW, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(x_nchw), B, HW, y_nhwc);
    RF_CUDA_LAUNCH_CHECK("k_vae_to_u8_f32scale");
    return RF_OK;
}

template <int NCO2>
static int launch_conv_in_blk(const void* x, const void* w, const void* bias, int B, int Cin, int H, int W, void* y,
                              cudaStream_t st) {
    const size_t smem = (static_cast<size_t>(64 * NCO2) * Cin * 9 + 8 * 18 * 8) * sizeof(float);
    RF_CUDA_TRY(cudaFuncSetAttribute(k_conv_in_blk<NCO2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    const long ngroups = static_cast<long>(B) * H * (W / 4);
    const unsigned grid = static_cast<unsigned>(std::min<long>((ngroups + 7) / 8, 2 * 148));
    k_conv_in_blk<NCO2><<<grid, 256, smem, st>>>(static_cast<const __half*>(x), static_cast<const __half*>(w),
                                                 static_cast<const __half*>(bias), B, Cin, H, W, static_cast<__half*>(y));
    RF_CUDA_LAUNCH_CHECK("k_conv_in_blk");
    return RF_OK;
}

extern "C" int rf_conv_in_f16(const void* x_nchw, const void* w, const void* bias, int B, int Cin, int H, int W,
                              int Cout, void* y_nhwc, void* stream) {
    if (!x_nchw || !w || !y_nhwc || B <= 0 || Cin <= 0 || Cin > 8 || Cout <= 0) return rf_fail(RF_ERR_INVALID, "rf_conv_in_f16: bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (W % 4 == 0 && (!bias || (reinterpret_cast<uintptr_t>(bias) & 3) == 0) &&
        (reinterpret_cast<uintptr_t>(y_nhwc) & 3) == 0) {
        if (Cout == 512) return launch_conv_in_blk<8>(x_nchw, w, bias, B, Cin, H, W, y_nhwc, st);   // VAE decoder
        if (Cout == 320) return launch_conv_in_blk<5>(x_nchw, w, bias, B, Cin, H, W, y_nhwc, st);
        if (Cout == 128) return launch_conv_in_blk<2>(x_nchw, w, bias, B, Cin, H, W, y_nhwc, st);
        if (Cout == 64) return launch_conv_in_blk<1>(x_nchw, w, bias, B, Cin, H, W, y_nhwc, st);
    }
    const size_t smem = static_cast<size_t>(Cout) * Cin * 9 * sizeof(float);
    if (smem > 96 * 1024) return rf_fail(RF_ERR_UNSUPPORTED, "rf_conv_in_f16: weights too large");
    static bool attr = false;
    if (!attr) {
        RF_CUDA_TRY(cudaFuncSetAttribute(k_conv_in_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        attr = true;
    }
    const size_t npix = static_cast<size_t>(B) * H * W;
    k_conv_in_generic<<<static_cast<unsigned>((npix + 63) / 64), 256, smem, st>>>(
        static_cast<const __half*>(x_nchw), static_cast<const __half*>(w), static_cast<const __half*>(bias), B, Cin, H, W,
        Cout, static_cast<__half*>(y_nhwc));
    RF_CUDA_LAUNCH_CHECK("k_conv_in");
    return RF_OK;
}

template <int NSTEP>
static int launch_conv_out_blk(const void* x, const void* w, const void* bias, int B, int H, int W, int Cout, void* y,
                               cudaStream_t st) {
    const size_t smem = static_cast<size_t>(9) * NSTEP * 256 * sizeof(float);
    RF_CUDA_TRY(cudaFuncSetAttribute(k_conv_out_blk<NSTEP>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    const long ngroups = static_cast<long>(B) * H * (W / 4);
    const unsigned grid = static_cast<unsigned>(std::min<long>((ngroups + 7) / 8, 2 * 148));
    k_conv_out_blk<NSTEP><<<grid, 256, smem, st>>>(static_cast<const __half*>(x), static_cast<const __half*>(w),
                                                   static_cast<const __half*>(bias), B, H, W, Cout, static_cast<__half*>(y));
    RF_CUDA_LAUNCH_CHECK("k_conv_out_blk");
    return RF_OK;
}

extern "C" int rf_conv_out_f16(const void* x_nhwc, const void* w_packed, const void* bias, int B, int H, int W, int Cin,
                               int Cout, void* y_nchw, void* stream) {
    if (!x_nhwc || !w_packed || !y_nchw || B <= 0 || Cout <= 0 || Cout > 8) return rf_fail(RF_ERR_INVALID, "rf_conv_out_f16: bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (W % 4 == 0 && Cout <= 4 && (reinterpret_cast<uintptr_t>(y_nchw) & 7) == 0) {
        if (Cin == 320) return launch_conv_out_blk<5>(x_nhwc, w_packed, bias, B, H, W, Cout, y_nchw, st);
        if (Cin == 128) return launch_conv_out_blk<2>(x_nhwc, w_packed, bias, B, H, W, Cout, y_nchw, st);
        if (Cin == 64) return launch_conv_out_blk<1>(x_nhwc, w_packed, bias, B, H, W, Cout, y_nchw, st);
    }
    const size_t pix = static_cast<size_t>(B) * H * W;
    k_conv_out_generic<<<static_cast<unsigned>((pix + 7) / 8), 256, 0, st>>>(
        static_cast<const __half*>(x_nhwc), static_cast<const __half*>(w_packed), static_cast<const __half*>(bias), B, H,
        W, Cin, Cout, static_cast<__half*>(y_nchw));
    RF_CUDA_LAUNCH_CHECK("k_conv_out");
    return RF_OK;
}

extern "C" int rf_timestep_embedding_f16(const float* d_t, int B, int dim, void* out, void* stream) {
    if (!d_t || !out || B <= 0 || dim <= 0 || (dim & 1)) return rf_fail(RF_ERR_INVALID, "rf_timestep_embedding_f16: bad argument");
    k_timestep_embedding<<<(B * dim / 2 + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
        d_t, B, dim, static_cast<__half*>(out));
    RF_CUDA_LAUNCH_CHECK("k_timestep_embedding");
    return RF_OK;
}

extern "C" int rf_silu_f16(const void* x, long n, void* y, void* stream) {
    if (!x || !y || n <= 0) return rf_fail(RF_ERR_INVALID, "rf_silu_f16: bad argument");
    k_silu<<<grid_for(static_cast<size_t>(n), 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(x), static_cast<size_t>(n), static_cast<__half*>(y));
    RF_CUDA_LAUNCH_CHECK("k_silu");
    return RF_OK;
}

extern "C" int rf_cfg_pndm_step_f16(const void* eps_pair, long n, float guidance, const void* h1, const void* h2,
                                    const void* h3, const float* coef4, const void* sample, float ca, float cb,
                                    void* eps_out, void* prev_sample, void* stream) {
    if (!eps_pair || !sample || !prev_sample || !coef4 || n <= 0) return rf_fail(RF_ERR_INVALID, "rf_cfg_pndm_step_f16: bad argument");
    k_cfg_pndm_step<<<grid_for(static_cast<size_t>(n), 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(eps_pair), static_cast<size_t>(n), guidance, static_cast<const __half*>(h1),
        static_cast<const __half*>(h2), static_cast<const __half*>(h3), coef4[0], coef4[1], coef4[2], coef4[3],
        static_cast<const __half*>(sample), ca, cb, static_cast<__half*>(eps_out), static_cast<__half*>(prev_sample));
    RF_CUDA_LAUNCH_CHECK("k_cfg_pndm_step");
    return RF_OK;
}

extern "C" int rf_cfg_dpmpp_step_f16(const void* eps_pair, long n, float guidance, const void* sample, const void* x0_prev,
                                     float sigma_s, float alpha_s, float c_x, float c_0, float inv_r0, float c_d1,
                                     void* x0_out, void* prev_sample, void* stream) {
    if (!eps_pair || !sample || !x0_out || !prev_sample || n <= 0 || !(alpha_s > 0.f) || x0_out == prev_sample)
        return rf_fail(RF_ERR_INVALID, "rf_cfg_dpmpp_step_f16: bad argument");
    const size_t N = static_cast<size_t>(n);
    const auto a16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    const bool vec = a16(eps_pair) && a16(sample) && (!x0_prev || a16(x0_prev)) && a16(x0_out) && a16(prev_sample);
    const size_t n8 = vec ? (N & ~static_cast<size_t>(7)) : 0;
    const bool et_vec = (N & 7) == 0;
    const DpmppCoef c{guidance, sigma_s, 1.f / alpha_s, c_x, c_0, inv_r0, c_d1};
    const unsigned grid = grid_for(n8 / 8 + (N - n8), 256);
    const auto* ep = static_cast<const __half*>(eps_pair);
    const auto* xs = static_cast<const __half*>(sample);
    const auto* m1 = static_cast<const __half*>(x0_prev);
    auto* m0 = static_cast<__half*>(x0_out);
    auto* xt = static_cast<__half*>(prev_sample);
    if (x0_prev)
        k_cfg_dpmpp_step<true><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(ep, N, n8, et_vec, xs, m1, c, m0, xt);
    else
        k_cfg_dpmpp_step<false><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(ep, N, n8, et_vec, xs, m1, c, m0, xt);
    RF_CUDA_LAUNCH_CHECK("k_cfg_dpmpp_step");
    return RF_OK;
}

extern "C" int rf_axpby_f16(const void* x, const void* noise, float a, float b, const void* mask, const void* z, long n,
                            void* y, void* stream) {
    if (!x || !noise || !y || n <= 0 || (mask && !z)) return rf_fail(RF_ERR_INVALID, "rf_axpby_f16: bad argument");
    k_axpby<<<grid_for(static_cast<size_t>(n), 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(x), static_cast<const __half*>(noise), a, b, static_cast<const __half*>(mask),
        static_cast<const __half*>(z), static_cast<size_t>(n), static_cast<__half*>(y));
    RF_CUDA_LAUNCH_CHECK("k_axpby");
    return RF_OK;
}

extern "C" int rf_add_noise_f16_seq(const void* x, const void* noise, float s, float s1, long n, void* y, void* stream) {
    // s and s1 are the fp16 values a[t] ** 0.5 and (1 - a[t]) ** 0.5: anything not representable in fp16 is a caller bug
    const auto is_f16 = [](float v) { return std::isfinite(v) && __half2float(__float2half_rn(v)) == v; };
    if (!x || !noise || !y || n <= 0 || !is_f16(s) || !is_f16(s1))
        return rf_fail(RF_ERR_INVALID, "rf_add_noise_f16_seq: bad argument");
    const size_t N = static_cast<size_t>(n);
    const auto a16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    const size_t n8 = (a16(x) && a16(noise) && a16(y)) ? (N & ~static_cast<size_t>(7)) : 0;
    k_add_noise_seq<<<grid_for(n8 / 8 + (N - n8), 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(x), static_cast<const __half*>(noise), s, s1, N, n8, static_cast<__half*>(y));
    RF_CUDA_LAUNCH_CHECK("k_add_noise_seq");
    return RF_OK;
}
