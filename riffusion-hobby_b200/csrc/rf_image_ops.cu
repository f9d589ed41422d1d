// Spectrogram-image glue of the audio-to-audio chain: Pillow's BICUBIC resize of a batch of uint8 RGB images and the
// uint8 -> fp16 [-1, 1] conversion that feeds the VAE encoder.
//
// Neither kernel is about FLOPs (a 512 x 501 clip image is 0.8 MB).  They exist so that a batch of clips stays on the
// device from the STFT to Griffin-Lim: without them the chain would leave the GPU twice per clip for two PIL resizes.
//
// Reference arithmetic: Pillow's libImaging/Resample.c (8 bits per channel) as the reference reaches it through
// `Image.resize(size, Image.BICUBIC)` (streamlit/tasks/audio_to_audio.py scale_image_to_32_stride and the resize back),
// and diffusers 0.9 img2img `preprocess` (`/ 255`, `2x - 1` in fp32, then `.half()`).
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <vector>

#include "rf_common.h"

namespace {

// ---------------------------------------------------------------- Pillow's separable resample, coefficient tables
// Pillow computes each output pixel's filter taps in double, normalises them to sum 1, converts them to int32 fixed
// point with PRECISION_BITS = 32 - 8 - 2 fractional bits (rounding away from zero) and accumulates
// `(1 << (PRECISION_BITS - 1)) + sum(pixel * tap)` in int32; the output is that sum >> PRECISION_BITS clipped to
// [0, 255].  The tables are built here on the host exactly as Pillow builds them, so the device only does integer
// multiply-adds and is bit-exact by construction.
constexpr int RS_PRECISION_BITS = 22;
constexpr double RS_BICUBIC_SUPPORT = 2.0;

double bicubic_filter(double x) {
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1.0;
    if (x < 2.0) return (((x - 5.0) * x + 8.0) * x - 4.0) * a;
    return 0.0;
}

struct RsTables {
    int ksize = 0;
    std::vector<int32_t> bounds;   // [n_out][2]: first input index, number of taps
    std::vector<int32_t> kk;       // [n_out][ksize]: fixed-point taps, zero past the tap count
};

RsTables rs_tables(int n_in, int n_out) {
    RsTables t;
    const double scale = static_cast<double>(n_in) / n_out;
    const double filterscale = scale < 1.0 ? 1.0 : scale;         // downscaling widens the filter
    const double support = RS_BICUBIC_SUPPORT * filterscale;
    t.ksize = static_cast<int>(std::ceil(support)) * 2 + 1;
    t.bounds.assign(static_cast<size_t>(n_out) * 2, 0);
    t.kk.assign(static_cast<size_t>(n_out) * t.ksize, 0);
    std::vector<double> k(t.ksize);
    const double ss = 1.0 / filterscale;
    for (int xx = 0; xx < n_out; ++xx) {
        const double center = (xx + 0.5) * scale;
        int xmin = static_cast<int>(center - support + 0.5);
        if (xmin < 0) xmin = 0;
        int xmax = static_cast<int>(center + support + 0.5);
        if (xmax > n_in) xmax = n_in;
        xmax -= xmin;
        double ww = 0.0;
        for (int x = 0; x < xmax; ++x) {
            const double w = bicubic_filter((x + xmin - center + 0.5) * ss);
            k[x] = w;
            ww += w;
        }
        for (int x = 0; x < xmax; ++x) {
            if (ww != 0.0) k[x] /= ww;
            const double v = k[x] * (1 << RS_PRECISION_BITS);
            t.kk[static_cast<size_t>(xx) * t.ksize + x] = static_cast<int32_t>(k[x] < 0 ? -0.5 + v : 0.5 + v);
        }
        t.bounds[2 * xx] = xmin;
        t.bounds[2 * xx + 1] = xmax;
    }
    return t;
}

// Device copies, one per (device, n_in, n_out), uploaded at first use and kept for the life of the process (a handful
// of sizes in practice: the clip width and its 32-stride width, in both directions).
struct RsAxis {
    const int32_t* bounds = nullptr;   // nullptr: the axis keeps its size and the pass is skipped
    const int32_t* kk = nullptr;
    int ksize = 0;
};

std::mutex g_rs_mu;
std::map<std::tuple<int, int, int>, RsAxis> g_rs_cache;

int rs_device_axis(int n_in, int n_out, RsAxis* out) {
    int dev = 0;
    RF_CUDA_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_rs_mu);
    const auto key = std::make_tuple(dev, n_in, n_out);
    const auto it = g_rs_cache.find(key);
    if (it != g_rs_cache.end()) {
        *out = it->second;
        return RF_OK;
    }
    const RsTables t = rs_tables(n_in, n_out);
    int32_t* d = nullptr;
    const size_t nb = t.bounds.size(), nk = t.kk.size();
    RF_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d), (nb + nk) * sizeof(int32_t)));
    cudaError_t e = cudaMemcpy(d, t.bounds.data(), nb * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d + nb, t.kk.data(), nk * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        cudaFree(d);
        return rf_fail(RF_ERR_CUDA, std::string("rf_resample_u8: table upload: ") + cudaGetErrorString(e));
    }
    RsAxis a;
    a.bounds = d;
    a.kk = d + nb;
    a.ksize = t.ksize;
    g_rs_cache.emplace(key, a);
    *out = a;
    return RF_OK;
}

__device__ __forceinline__ int clip8(int acc) { return min(max(acc >> RS_PRECISION_BITS, 0), 255); }

// One thread per output pixel (all three channels).  Pillow runs the horizontal pass into a uint8 image and the
// vertical pass over that; here each output pixel recomputes the horizontal results of the rows its vertical taps read
// (same integers, clipped to uint8 the same way), so no intermediate image is needed.
template <bool HORIZ, bool VERT>
__global__ void k_resample_u8(const uint8_t* __restrict__ x, int B, int Hi, int Wi, int Ho, int Wo, RsAxis hx,
                              RsAxis vy, uint8_t* __restrict__ y) {
    const size_t n = static_cast<size_t>(B) * Ho * Wo;
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int ox = static_cast<int>(i % Wo);
        const size_t r = i / Wo;
        const int oy = static_cast<int>(r % Ho);
        const size_t b = r / Ho;
        const uint8_t* img = x + b * Hi * Wi * 3;
        int ymin = oy, ylen = 1, xmin = ox, xlen = 1;
        const int32_t* kv = nullptr;
        const int32_t* kh = nullptr;
        if constexpr (VERT) {
            ymin = vy.bounds[2 * oy];
            ylen = vy.bounds[2 * oy + 1];
            kv = vy.kk + static_cast<size_t>(oy) * vy.ksize;
        }
        if constexpr (HORIZ) {
            xmin = hx.bounds[2 * ox];
            xlen = hx.bounds[2 * ox + 1];
            kh = hx.kk + static_cast<size_t>(ox) * hx.ksize;
        }
        int acc[3] = {1 << (RS_PRECISION_BITS - 1), 1 << (RS_PRECISION_BITS - 1), 1 << (RS_PRECISION_BITS - 1)};
        int h[3];
        for (int j = 0; j < ylen; ++j) {
            const uint8_t* row = img + (static_cast<size_t>(ymin + j) * Wi + xmin) * 3;
            if constexpr (HORIZ) {
                int a0 = 1 << (RS_PRECISION_BITS - 1), a1 = a0, a2 = a0;
                for (int k = 0; k < xlen; ++k) {
                    const int w = kh[k];
                    a0 += row[3 * k] * w;
                    a1 += row[3 * k + 1] * w;
                    a2 += row[3 * k + 2] * w;
                }
                h[0] = clip8(a0);
                h[1] = clip8(a1);
                h[2] = clip8(a2);
            } else {
                h[0] = row[0];
                h[1] = row[1];
                h[2] = row[2];
            }
            if constexpr (VERT) {
                const int w = kv[j];
#pragma unroll
                for (int c = 0; c < 3; ++c) acc[c] += h[c] * w;
            }
        }
        uint8_t* o = y + i * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) o[c] = static_cast<uint8_t>(VERT ? clip8(acc[c]) : h[c]);
    }
}

// diffusers img2img `preprocess`: np.float32(u8) / 255, then 2x - 1 in fp32, then `.half()` (one rounding to fp16).
// 2x is exact, so a contraction of 2x - 1 into an FMA gives the same fp32 value.
__global__ void k_u8_to_f16_nchw(const uint8_t* __restrict__ x, int B, size_t HW, __half* __restrict__ y) {
    const size_t n = static_cast<size_t>(B) * HW;
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t b = i / HW, p = i % HW;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float v = static_cast<float>(x[i * 3 + c]) / 255.f;
            y[(b * 3 + c) * HW + p] = __float2half_rn(2.f * v - 1.f);
        }
    }
}

unsigned grid_1d(size_t n, int block) {
    const size_t g = (n + block - 1) / block;
    return static_cast<unsigned>(g > 148 * 16 ? 148 * 16 : (g ? g : 1));
}

}  // namespace

extern "C" int rf_resample_coeffs(int n_in, int n_out, int* ksize, int32_t* bounds, int32_t* kk) {
    if (n_in <= 0 || n_out <= 0 || !ksize) return rf_fail(RF_ERR_INVALID, "rf_resample_coeffs: bad argument");
    const RsTables t = rs_tables(n_in, n_out);
    *ksize = t.ksize;
    if (bounds) std::copy(t.bounds.begin(), t.bounds.end(), bounds);
    if (kk) std::copy(t.kk.begin(), t.kk.end(), kk);
    return RF_OK;
}

extern "C" int rf_resample_u8(const uint8_t* x_nhwc, int B, int H_in, int W_in, int H_out, int W_out, uint8_t* y_nhwc,
                              void* stream) {
    if (!x_nhwc || !y_nhwc || x_nhwc == y_nhwc || B <= 0 || H_in <= 0 || W_in <= 0 || H_out <= 0 || W_out <= 0)
        return rf_fail(RF_ERR_INVALID, "rf_resample_u8: bad argument");
    const bool horiz = W_in != W_out, vert = H_in != H_out;
    RsAxis hx, vy;
    if (horiz) {
        const int rc = rs_device_axis(W_in, W_out, &hx);
        if (rc != RF_OK) return rc;
    }
    if (vert) {
        const int rc = rs_device_axis(H_in, H_out, &vy);
        if (rc != RF_OK) return rc;
    }
    const unsigned grid = grid_1d(static_cast<size_t>(B) * H_out * W_out, 256);
    const auto st = static_cast<cudaStream_t>(stream);
    if (horiz && vert)
        k_resample_u8<true, true><<<grid, 256, 0, st>>>(x_nhwc, B, H_in, W_in, H_out, W_out, hx, vy, y_nhwc);
    else if (horiz)
        k_resample_u8<true, false><<<grid, 256, 0, st>>>(x_nhwc, B, H_in, W_in, H_out, W_out, hx, vy, y_nhwc);
    else if (vert)
        k_resample_u8<false, true><<<grid, 256, 0, st>>>(x_nhwc, B, H_in, W_in, H_out, W_out, hx, vy, y_nhwc);
    else
        k_resample_u8<false, false><<<grid, 256, 0, st>>>(x_nhwc, B, H_in, W_in, H_out, W_out, hx, vy, y_nhwc);
    RF_CUDA_LAUNCH_CHECK("k_resample_u8");
    return RF_OK;
}

extern "C" int rf_image_u8_to_f16(const uint8_t* x_nhwc, int B, int H, int W, void* y_nchw, void* stream) {
    if (!x_nhwc || !y_nchw || B <= 0 || H <= 0 || W <= 0) return rf_fail(RF_ERR_INVALID, "rf_image_u8_to_f16: bad argument");
    const size_t HW = static_cast<size_t>(H) * W;
    k_u8_to_f16_nchw<<<grid_1d(static_cast<size_t>(B) * HW, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        x_nhwc, B, HW, static_cast<__half*>(y_nchw));
    RF_CUDA_LAUNCH_CHECK("k_u8_to_f16_nchw");
    return RF_OK;
}
