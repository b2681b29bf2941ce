// Data movement around the tensor-core GEMM for the HMR ResNet-50 feature extractor (reference lib/models/spin.py:59-141,
// caller demo.py:183-198): activations live in HBM as NHWC bf16, every convolution (BatchNorm folded into weights and bias at
// pack time, eval mode) is  im2col rows x [Cout, kh*kw*Cin] weights  on tp_gemm_bf16_tc with the ReLU / shortcut-add epilogue;
// 1x1 stride-1 convolutions read the activation tensor directly as the GEMM operand.
#include "common.cuh"

namespace tp {

// x [N,C,H,W] fp32 -> y [N,H,W,CP] bf16 (channels c >= C are zero); CP = 4 for the RGB stem.
// SPLIT: y [N,H,W,3 CP], [hi | lo | hi] per pixel, hi = RN_bf16(v), lo = RN_bf16(v - hi).
template <bool SPLIT>
__global__ void k_nchw_to_nhwc(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int N, int C, int H, int W, int CP) {
  const int64_t total = (int64_t)N * H * W;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = i / ((int64_t)H * W), hw = i - n * H * W;
    for (int c = 0; c < CP; ++c) {
      const float v = c < C ? x[(n * C + c) * (int64_t)H * W + hw] : 0.0f;
      const __nv_bfloat16 hi = __float2bfloat16_rn(v);
      if (SPLIT) {
        y[i * 3 * CP + c] = hi;
        y[i * 3 * CP + CP + c] = __float2bfloat16_rn(v - __bfloat162float(hi));
        y[i * 3 * CP + 2 * CP + c] = hi;
      } else {
        y[i * CP + c] = hi;
      }
    }
  }
}

// in [N,H,W,C] bf16 -> out [N*Ho*Wo, KP] bf16, column (ky*kw + kx)*C + c; taps outside the image and columns >= kh*kw*C are zero.
// VEC channels (16 or 8 bytes) per thread and copy.  IdxT = unsigned int whenever the vector count fits 31 bits: the index
// arithmetic (five divisions per copy) in 64 bits made the kernel compute-bound (1.8 TB/s of stores, 0.95 TB/s for the stem).
template <int VEC, typename IdxT>
__global__ void k_im2col(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int N, int H, int W, int C,
                         int kh, int kw, int stride, int pad, int Ho, int Wo, int KP) {
  const IdxT kv = (IdxT)(KP / VEC);                           // vectors per output row
  const IdxT total = (IdxT)N * (IdxT)Ho * (IdxT)Wo * kv;
  const unsigned K = (unsigned)(kh * kw * C), cv = (unsigned)(C / VEC);      // vectors per tap
  for (IdxT i = blockIdx.x * (IdxT)blockDim.x + threadIdx.x; i < total; i += (IdxT)gridDim.x * blockDim.x) {
    const IdxT row = i / kv;
    const unsigned v = (unsigned)(i - row * kv);
    const unsigned col = v * VEC;
    const IdxT t1 = row / (IdxT)Wo;
    const int wo = (int)(row - t1 * (IdxT)Wo);
    const IdxT n = t1 / (IdxT)Ho;
    const int ho = (int)(t1 - n * (IdxT)Ho);
    const unsigned tap = v / cv, c = (v - tap * cv) * VEC;
    const int ky = (int)(tap / (unsigned)kw), kx = (int)(tap - (unsigned)ky * (unsigned)kw);
    const int hi = ho * stride - pad + ky, wi = wo * stride - pad + kx;
    const bool ok = col < K && hi >= 0 && hi < H && wi >= 0 && wi < W;
    const size_t src = (((size_t)n * H + hi) * W + wi) * C + c;
    if (VEC == 8) {
      uint4 val = make_uint4(0u, 0u, 0u, 0u);
      if (ok) val = *reinterpret_cast<const uint4*>(in + src);
      *reinterpret_cast<uint4*>(out + (size_t)row * KP + col) = val;
    } else {
      uint2 val = make_uint2(0u, 0u);
      if (ok) val = *reinterpret_cast<const uint2*>(in + src);
      *reinterpret_cast<uint2*>(out + (size_t)row * KP + col) = val;
    }
  }
}

// MaxPool2d(kernel 3, stride 2, padding 1) on NHWC bf16 (lib/models/spin.py:70): 8 channels per thread
__global__ void k_maxpool3x3s2(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int N, int H, int W, int C, int Ho, int Wo) {
  const int cv = C / 8;
  const int64_t total = (int64_t)N * Ho * Wo * cv;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % cv) * 8;
    const int64_t pix = i / cv;
    const int wo = (int)(pix % Wo), ho = (int)((pix / Wo) % Ho), n = (int)(pix / ((int64_t)Wo * Ho));
    float m[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) m[u] = -INFINITY;
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) {
        const int hi = ho * 2 - 1 + ky, wi = wo * 2 - 1 + kx;
        if (hi < 0 || hi >= H || wi < 0 || wi >= W) continue;
        const uint4 v = *reinterpret_cast<const uint4*>(in + (((int64_t)n * H + hi) * W + wi) * C + c);
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
        for (int u = 0; u < 4; ++u) { const float2 f = __bfloat1622float2(h[u]); m[2 * u] = fmaxf(m[2 * u], f.x); m[2 * u + 1] = fmaxf(m[2 * u + 1], f.y); }
      }
    __nv_bfloat162 o[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) o[u] = __floats2bfloat162_rn(m[2 * u], m[2 * u + 1]);
    *reinterpret_cast<uint4*>(out + pix * C + c) = *reinterpret_cast<const uint4*>(o);
  }
}

// AvgPool2d over the whole HW x HW map (lib/models/spin.py:75,139-140): [N,HW,C] bf16 -> [N,C] fp32 (+ optional bf16 copy)
__global__ void k_avgpool(const __nv_bfloat16* __restrict__ in, float* __restrict__ out, int N, int HW, int C) {
  const int64_t total = (int64_t)N * C;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = i / C;
    const int c = (int)(i - n * C);
    float s = 0.0f;
    for (int p = 0; p < HW; ++p) s += __bfloat162float(in[(n * HW + p) * C + c]);
    out[i] = s / (float)HW;
  }
}

// MaxPool2d(3, 2, 1) on split rows [N,H,W,3C]: the represented value hi + lo is exact in fp64; strict '>' keeps the first
// maximum in (ky, kx) order.  8 channels per thread.
__global__ void k_maxpool3x3s2_split3(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int N, int H, int W, int C,
                                      int Ho, int Wo) {
  const int cv = C / 8;
  const int64_t total = (int64_t)N * Ho * Wo * cv;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % cv) * 8;
    const int64_t pix = i / cv;
    const int wo = (int)(pix % Wo), ho = (int)((pix / Wo) % Ho), n = (int)(pix / ((int64_t)Wo * Ho));
    double m[8];
    __align__(16) __nv_bfloat16 bh[8], bl[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) { m[u] = -INFINITY; bh[u] = __float2bfloat16_rn(-INFINITY); bl[u] = __float2bfloat16_rn(0.0f); }
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) {
        const int hi = ho * 2 - 1 + ky, wi = wo * 2 - 1 + kx;
        if (hi < 0 || hi >= H || wi < 0 || wi >= W) continue;
        const __nv_bfloat16* src = in + (((int64_t)n * H + hi) * W + wi) * 3 * C + c;
        __align__(16) __nv_bfloat16 h[8], l[8];
        *reinterpret_cast<uint4*>(h) = *reinterpret_cast<const uint4*>(src);
        *reinterpret_cast<uint4*>(l) = *reinterpret_cast<const uint4*>(src + C);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const double v = (double)__bfloat162float(h[u]) + (double)__bfloat162float(l[u]);
          if (v > m[u]) { m[u] = v; bh[u] = h[u]; bl[u] = l[u]; }
        }
      }
    __nv_bfloat16* dst = out + pix * 3 * C + c;
    *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(bh);
    *reinterpret_cast<uint4*>(dst + C) = *reinterpret_cast<const uint4*>(bl);
    *reinterpret_cast<uint4*>(dst + 2 * C) = *reinterpret_cast<const uint4*>(bh);
  }
}

// mean of hi + lo over HW positions of split rows [N,HW,3C] -> [N,C] fp32 (hi + lo is exact in fp32 for a split the GEMM
// epilogue wrote)
__global__ void k_avgpool_split3(const __nv_bfloat16* __restrict__ in, float* __restrict__ out, int N, int HW, int C) {
  const int64_t total = (int64_t)N * C;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = i / C;
    const int c = (int)(i - n * C);
    float s = 0.0f;
    for (int p = 0; p < HW; ++p) {
      const __nv_bfloat16* r = in + (n * HW + p) * 3 * C + c;
      s += __bfloat162float(r[0]) + __bfloat162float(r[C]);
    }
    out[i] = s / (float)HW;
  }
}

static unsigned grid_for(int64_t total) {
  int64_t g = (total + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 16;
  return (unsigned)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace tp

using namespace tp;

extern "C" int tp_nchw_to_nhwc_bf16(const float* x, void* y, int N, int C, int H, int W, int CP, void* stream) {
  TP_CHECK_ARG(x && y && N > 0 && C > 0 && H > 0 && W > 0 && CP >= C, "tp_nchw_to_nhwc_bf16: bad arguments");
  k_nchw_to_nhwc<false><<<grid_for((int64_t)N * H * W), 256, 0, (cudaStream_t)stream>>>(x, reinterpret_cast<__nv_bfloat16*>(y), N, C, H, W, CP);
  TP_LAUNCH_CHECK();
  return TP_OK;
}

extern "C" int tp_nchw_to_nhwc_split3(const float* x, void* y, int N, int C, int H, int W, int CP, void* stream) {
  TP_CHECK_ARG(x && y && N > 0 && C > 0 && H > 0 && W > 0 && CP >= C, "tp_nchw_to_nhwc_split3: bad arguments");
  k_nchw_to_nhwc<true><<<grid_for((int64_t)N * H * W), 256, 0, (cudaStream_t)stream>>>(x, reinterpret_cast<__nv_bfloat16*>(y), N, C, H, W, CP);
  TP_LAUNCH_CHECK();
  return TP_OK;
}

extern "C" int tp_maxpool3x3s2_nhwc_split3(const void* in, void* out, int N, int H, int W, int C, void* stream) {
  TP_CHECK_ARG(in && out && N > 0 && H > 0 && W > 0 && C > 0 && C % 8 == 0, "tp_maxpool3x3s2_nhwc_split3: bad arguments (C %% 8 == 0)");
  TP_CHECK_ARG(aligned16(in) && aligned16(out), "tp_maxpool3x3s2_nhwc_split3: pointers must be 16-byte aligned");
  const int Ho = (H + 2 - 3) / 2 + 1, Wo = (W + 2 - 3) / 2 + 1;
  k_maxpool3x3s2_split3<<<grid_for((int64_t)N * Ho * Wo * (C / 8)), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(in), reinterpret_cast<__nv_bfloat16*>(out), N, H, W, C, Ho, Wo);
  TP_LAUNCH_CHECK();
  return TP_OK;
}

extern "C" int tp_avgpool_nhwc_split3(const void* in, float* out, int N, int HW, int C, void* stream) {
  TP_CHECK_ARG(in && out && N > 0 && HW > 0 && C > 0, "tp_avgpool_nhwc_split3: bad arguments");
  k_avgpool_split3<<<grid_for((int64_t)N * C), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __nv_bfloat16*>(in), out, N, HW, C);
  TP_LAUNCH_CHECK();
  return TP_OK;
}

extern "C" int tp_im2col_nhwc_bf16(const void* in, void* out, int N, int H, int W, int C, int kh, int kw, int stride, int pad, int KP,
                                   void* stream) {
  TP_CHECK_ARG(in && out && N > 0 && H > 0 && W > 0 && C > 0 && kh > 0 && kw > 0 && stride > 0 && pad >= 0, "tp_im2col_nhwc_bf16: bad arguments");
  TP_CHECK_ARG(C % 4 == 0 && KP % 8 == 0 && KP >= kh * kw * C, "tp_im2col_nhwc_bf16: need C %% 4 == 0 and KP %% 8 == 0, KP >= kh*kw*C (C=%d KP=%d)", C, KP);
  TP_CHECK_ARG(aligned16(in) && aligned16(out), "tp_im2col_nhwc_bf16: pointers must be 16-byte aligned");
  const int Ho = (H + 2 * pad - kh) / stride + 1, Wo = (W + 2 * pad - kw) / stride + 1;
  TP_CHECK_ARG(Ho > 0 && Wo > 0, "tp_im2col_nhwc_bf16: empty output");
  const __nv_bfloat16* i = reinterpret_cast<const __nv_bfloat16*>(in);
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
  const int vec = C % 8 == 0 ? 8 : 4;
  const int64_t nvec = (int64_t)N * Ho * Wo * (KP / vec);
  const bool small = nvec < ((int64_t)1 << 31) - ((int64_t)1 << 24);       // 32-bit indices (with room for the grid stride)
  const unsigned grid = grid_for(nvec);
  cudaStream_t st = (cudaStream_t)stream;
  if (vec == 8 && small) k_im2col<8, unsigned int><<<grid, 256, 0, st>>>(i, o, N, H, W, C, kh, kw, stride, pad, Ho, Wo, KP);
  else if (vec == 8) k_im2col<8, unsigned long long><<<grid, 256, 0, st>>>(i, o, N, H, W, C, kh, kw, stride, pad, Ho, Wo, KP);
  else if (small) k_im2col<4, unsigned int><<<grid, 256, 0, st>>>(i, o, N, H, W, C, kh, kw, stride, pad, Ho, Wo, KP);
  else k_im2col<4, unsigned long long><<<grid, 256, 0, st>>>(i, o, N, H, W, C, kh, kw, stride, pad, Ho, Wo, KP);
  TP_LAUNCH_CHECK();
  return TP_OK;
}

extern "C" int tp_maxpool3x3s2_nhwc_bf16(const void* in, void* out, int N, int H, int W, int C, void* stream) {
  TP_CHECK_ARG(in && out && N > 0 && H > 0 && W > 0 && C > 0 && C % 8 == 0, "tp_maxpool3x3s2_nhwc_bf16: bad arguments (C %% 8 == 0)");
  TP_CHECK_ARG(aligned16(in) && aligned16(out), "tp_maxpool3x3s2_nhwc_bf16: pointers must be 16-byte aligned");
  const int Ho = (H + 2 - 3) / 2 + 1, Wo = (W + 2 - 3) / 2 + 1;
  k_maxpool3x3s2<<<grid_for((int64_t)N * Ho * Wo * (C / 8)), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(in), reinterpret_cast<__nv_bfloat16*>(out), N, H, W, C, Ho, Wo);
  TP_LAUNCH_CHECK();
  return TP_OK;
}

extern "C" int tp_avgpool_nhwc_bf16(const void* in, float* out, int N, int HW, int C, void* stream) {
  TP_CHECK_ARG(in && out && N > 0 && HW > 0 && C > 0, "tp_avgpool_nhwc_bf16: bad arguments");
  k_avgpool<<<grid_for((int64_t)N * C), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __nv_bfloat16*>(in), out, N, HW, C);
  TP_LAUNCH_CHECK();
  return TP_OK;
}
