// Person crop of the demo front end (reference lib/data_utils/_img_utils.py: get_single_image_crop_demo ->
// generate_patch_image_cv with rot = 0, no flip; convert_cvimg_to_tensor) on the device: uint8 RGB frames -> the stem's
// [N,224,224,4] bf16 NHWC input.  The arithmetic is cv2's, restated in oracle/crop_ref.py and pinned there against cv2:
//   - the source points of gen_trans_from_patch_cv, rounded to float32 as the reference stores them;
//   - cv2.getAffineTransform: the 6x6 system by Gaussian elimination with partial pivoting (cv::LU64f), back substitution by
//     division; then the inversion cv2.warpAffine applies.  Every double operation is separately rounded (__d*_rn: no FMA
//     contraction), in cv2's order;
//   - cv2.warpAffine's uint8 INTER_LINEAR: positions in 1/1024 pixel rounded to 1/32, 15-bit bilinear weights, taps outside
//     the frame read 0;
//   - ((v / 255) - mean[c]) / std[c] in fp32 (ToTensor + Normalize), then one round to bf16.
#include "common.cuh"

#include <algorithm>
#include <vector>

namespace tp {

constexpr int kCrop = 224;                          // patch size (the demo's crop_size; HMR's input)
constexpr int kPairsPerRow = kCrop / 2;             // a thread writes two adjacent output pixels: one 16-byte store
constexpr int kPairs = kCrop * kPairsPerRow;
constexpr int kThreads = 256;

__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }

// Inverse map (destination pixel -> source position, 2x3 row-major) of one crop, computed by warp 0: lane j < 6 owns row j of
// the 6x6 system of cv2.getAffineTransform.  Returns the map in every lane.
__device__ __forceinline__ void crop_inverse_map(const tp_crop& c, double iM[6]) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  // gen_trans_from_patch_cv: float32 half extents, double sums, float32 points
  const double cx = c.cx, cy = c.cy;
  const float hh = __double2float_rn(dmul(dmul((double)c.h, (double)c.scale), 0.5));
  const float hw = __double2float_rn(dmul(dmul((double)c.w, (double)c.scale), 0.5));
  const int pt = lane >> 1;                                            // the point this row comes from
  const double px = pt == 2 ? (double)__double2float_rn(dadd(cx, (double)hw)) : (double)(float)cx;
  const double py = pt == 1 ? (double)__double2float_rn(dadd(cy, (double)hh)) : (double)(float)cy;
  const double half = kCrop * 0.5;
  const double qx = pt == 2 ? half + half : half, qy = pt == 1 ? half + half : half;
  double a[6], b;
  const bool odd = lane & 1, row = lane < 6;
  a[0] = row && !odd ? px : 0.0; a[1] = row && !odd ? py : 0.0; a[2] = row && !odd ? 1.0 : 0.0;
  a[3] = row && odd ? px : 0.0;  a[4] = row && odd ? py : 0.0;  a[5] = row && odd ? 1.0 : 0.0;
  b = row ? (odd ? qy : qx) : 0.0;
  bool singular = false;
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    // pivot: the first row j >= i with the largest |a[j][i]|
    const double v = fabs(a[i]);
    double best = __shfl_sync(full, v, i);
    int k = i;
#pragma unroll
    for (int j = i + 1; j < 6; ++j) {
      const double vj = __shfl_sync(full, v, j);
      if (vj > best) { best = vj; k = j; }
    }
    singular |= best < 100.0 * 2.220446049250313e-16;                   // cv::LU64f's DBL_EPSILON * 100
    const int src = lane == i ? k : (lane == k ? i : lane);
#pragma unroll
    for (int col = 0; col < 6; ++col) a[col] = __shfl_sync(full, a[col], src);
    b = __shfl_sync(full, b, src);
    const double d = __ddiv_rn(-1.0, __shfl_sync(full, a[i], i));
    double p[6];
#pragma unroll
    for (int col = i + 1; col < 6; ++col) p[col] = __shfl_sync(full, a[col], i);
    const double pb = __shfl_sync(full, b, i);
    if (lane > i && lane < 6) {
      const double alpha = dmul(a[i], d);
#pragma unroll
      for (int col = i + 1; col < 6; ++col) a[col] = dadd(a[col], dmul(alpha, p[col]));
      b = dadd(b, dmul(alpha, pb));
    }
  }
  double m[6];
#pragma unroll
  for (int i = 5; i >= 0; --i) {
    double s = b;
#pragma unroll
    for (int col = i + 1; col < 6; ++col) s = dsub(s, dmul(a[col], m[col]));
    m[i] = __shfl_sync(full, __ddiv_rn(s, a[i]), i);
  }
  if (singular) {                                                        // cv::solve fails: getAffineTransform returns zeros
#pragma unroll
    for (int i = 0; i < 6; ++i) m[i] = 0.0;
  }
  // cv2.warpAffine without WARP_INVERSE_MAP inverts the matrix it is given
  double D = dsub(dmul(m[0], m[4]), dmul(m[1], m[3]));
  D = D != 0.0 ? __ddiv_rn(1.0, D) : 0.0;
  const double a11 = dmul(m[4], D), a22 = dmul(m[0], D), a12 = dmul(m[1], -D), a21 = dmul(m[3], -D);
  iM[0] = a11; iM[1] = a12; iM[2] = dsub(dmul(-a11, m[2]), dmul(a12, m[5]));
  iM[3] = a21; iM[4] = a22; iM[5] = dsub(dmul(-a21, m[2]), dmul(a22, m[5]));
}

// grid (blocks per crop, N); every block covers the pairs p = blockIdx.x * kThreads + threadIdx.x (+ gridDim.x * kThreads) of
// its crop.  out [N,224,224,4] bf16; channel 3 is zero.
__global__ void __launch_bounds__(kThreads) k_crop_normalize(const uint8_t* __restrict__ frames, int F, int H, int W,
                                                             const tp_crop* __restrict__ crops, __nv_bfloat16* __restrict__ out) {
  __shared__ double s_map[6];
  __shared__ __nv_bfloat16 s_lut[3][256];                // byte value -> normalized bf16, per channel
  __shared__ int s_frame;
  const int n = blockIdx.y;
  for (int i = threadIdx.x; i < 3 * 256; i += kThreads) {
    const int ch = i >> 8;
    const float mean = ch == 0 ? 0.485f : (ch == 1 ? 0.456f : 0.406f), stdv = ch == 0 ? 0.229f : (ch == 1 ? 0.224f : 0.225f);
    s_lut[ch][i & 255] = __float2bfloat16_rn(__fdiv_rn(__fsub_rn(__fdiv_rn((float)(i & 255), 255.0f), mean), stdv));
  }
  if (threadIdx.x < 32) {
    const tp_crop c = crops[n];
    double iM[6];
    crop_inverse_map(c, iM);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int i = 0; i < 6; ++i) s_map[i] = iM[i];
      // the entry point checks frame indices when it is not being captured; a replayed graph may see a bad one: zeros, no read
      s_frame = (c.frame >= 0 && c.frame < F) ? c.frame : -1;
    }
  }
  __syncthreads();
  const double m0 = s_map[0], m1 = s_map[1], m2 = s_map[2], m3 = s_map[3], m4 = s_map[4], m5 = s_map[5];
  const int f = s_frame;
  const uint8_t* img = frames + (size_t)(f < 0 ? 0 : f) * H * W * 3;
  uint4* dst = reinterpret_cast<uint4*>(out + (size_t)n * kCrop * kCrop * 4);
  for (int p = blockIdx.x * kThreads + threadIdx.x; p < kPairs; p += gridDim.x * kThreads) {
    const int y = p / kPairsPerRow, x0 = (p - y * kPairsPerRow) * 2;
    __align__(16) __nv_bfloat16 o[8];
    if (f < 0) {
#pragma unroll
      for (int u = 0; u < 8; ++u) o[u] = __float2bfloat16_rn(0.0f);
    } else {
      // cv2 WarpAffineInvoker: X0, Y0 per row (+ 16: half of a 1/32 step), adelta / bdelta per column, in 1/1024 pixel
      const int X0 = __double2int_rn(dmul(dadd(dmul(m1, (double)y), m2), 1024.0)) + 16;
      const int Y0 = __double2int_rn(dmul(dadd(dmul(m4, (double)y), m5), 1024.0)) + 16;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const double x = (double)(x0 + u);
        const int X = (X0 + __double2int_rn(dmul(dmul(m0, x), 1024.0))) >> 5;     // 1/32 pixel
        const int Y = (Y0 + __double2int_rn(dmul(dmul(m3, x), 1024.0))) >> 5;
        const int sx = min(max(X >> 5, -32768), 32767), sy = min(max(Y >> 5, -32768), 32767);   // saturate_cast<short>
        const int fx = X & 31, fy = Y & 31;
        int acc[3] = {0, 0, 0};
#pragma unroll
        for (int dy = 0; dy < 2; ++dy) {
          const int yy = sy + dy;
          const int wy = dy ? fy : 32 - fy;
#pragma unroll
          for (int dx = 0; dx < 2; ++dx) {
            const int xx = sx + dx;
            const int w = wy * (dx ? fx : 32 - fx) * 32;
            if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
              const uint8_t* px = img + ((size_t)yy * W + xx) * 3;
#pragma unroll
              for (int ch = 0; ch < 3; ++ch) acc[ch] += w * (int)__ldg(px + ch);
            }
          }
        }
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) o[4 * u + ch] = s_lut[ch][(acc[ch] + (1 << 14)) >> 15];
        o[4 * u + 3] = __float2bfloat16_rn(0.0f);
      }
    }
    dst[p] = *reinterpret_cast<const uint4*>(o);
  }
}

}  // namespace tp

using namespace tp;

extern "C" int tp_crop_normalize_bf16(const void* frames, int F, int H, int W, const tp_crop* crops, int N, void* out,
                                      void* stream) {
  TP_CHECK_ARG(frames && crops && out, "tp_crop_normalize_bf16: null pointer");
  TP_CHECK_ARG(F > 0 && H > 0 && W > 0 && N > 0 && N <= 65535,
               "tp_crop_normalize_bf16: need F, H, W > 0 and 0 < N <= 65535 (F=%d H=%d W=%d N=%d)", F, H, W, N);
  TP_CHECK_ARG((reinterpret_cast<uintptr_t>(crops) & 3u) == 0 && aligned16(out),
               "tp_crop_normalize_bf16: crops must be 4-byte and out 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  TP_CUDA(cudaStreamIsCapturing(st, &cap));
  if (cap == cudaStreamCaptureStatusNone) {                 // the table is device data: read it back to check the frame indices
    std::vector<tp_crop> host((size_t)N);
    TP_CUDA(cudaMemcpyAsync(host.data(), crops, (size_t)N * sizeof(tp_crop), cudaMemcpyDefault, st));
    TP_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < N; ++i)
      TP_CHECK_ARG(host[i].frame >= 0 && host[i].frame < F, "tp_crop_normalize_bf16: crop %d names frame %d of %d", i,
                   host[i].frame, F);
  }
  const int per_crop = (int)ceil_div(kPairs, kThreads);
  const int bx = (int)std::min<int64_t>(per_crop, std::max<int64_t>(1, ceil_div((int64_t)sm_count() * 8, N)));
  k_crop_normalize<<<dim3(bx, N), kThreads, 0, st>>>(reinterpret_cast<const uint8_t*>(frames), F, H, W, crops,
                                                      reinterpret_cast<__nv_bfloat16*>(out));
  TP_LAUNCH_CHECK();
  return TP_OK;
}
