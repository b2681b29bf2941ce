// Pose smoothing of the demo's output path (lib/utils/smooth_pose.py with lib/utils/one_euro_filter.py): the One-Euro filter
// as a ragged, batched scan whose state survives between calls, so one kernel serves a whole clip (tepose_b200.smooth) and the
// per-frame step of tepose_b200.tracks.  A thread owns one channel of one sequence and walks its rows in order; the row loads
// do not depend on the recurrence, so kSmoothU of them are in flight before the rows are filtered.  Rows of a column view such
// as theta[:, 3:75] are only 4-byte aligned, so every access is a scalar fp32 one.
//
// Arithmetic: the reference runs in float32 with every operation rounded on its own (Python scalars are weak under numpy's
// rules, so 2*pi is rounded to float32 before it meets an array, and t_e is always 1).  The explicit __f*_rn intrinsics keep
// nvcc from contracting a*b + c into an FMA, which would change the bits.
#include <cmath>

#include "common.cuh"

namespace tp {

constexpr int kSmoothThreads = 128;
constexpr int kSmoothU = 8;                         // rows a thread has in flight
constexpr float kTwoPi = 6.28318530717958647692f;   // fl32(2*pi)

struct OneEuro {
  float mc, beta, a_d, one_m_a_d;                   // fl32(min_cutoff), fl32(beta), K/(K+1), 1 - a_d

  // x_hat of x given x_prev and dx_prev (which become x_hat and dx_hat)
  __device__ __forceinline__ float step(float x, float& xp, float& dxp) const {
    const float dx = __fsub_rn(x, xp);
    const float dxh = __fadd_rn(__fmul_rn(a_d, dx), __fmul_rn(one_m_a_d, dxp));
    const float cutoff = __fadd_rn(mc, __fmul_rn(beta, fabsf(dxh)));
    const float r = __fmul_rn(kTwoPi, cutoff);
    // r/(r+1) correctly rounded: the float64 quotient of two floats rounded to float is the float32 quotient (53 >= 2*24+2, so
    // the double rounding is innocuous), and it keeps fp32 FFMA out of the recurrence (__fdiv_rn refines a reciprocal with FFMA)
    const float a = __double2float_rn(__ddiv_rn((double)r, (double)__fadd_rn(r, 1.0f)));
    const float xh = __fadd_rn(__fmul_rn(a, x), __fmul_rn(__fsub_rn(1.0f, a), xp));
    xp = xh;
    dxp = dxh;
    return xh;
  }
};

// one thread per (sequence, channel), flattened over S*C; see tp_one_euro_filter for the contract
__global__ void __launch_bounds__(kSmoothThreads) k_one_euro_filter(const float* __restrict__ x, int64_t ldsx, int64_t ldrx,
                                                                   float* __restrict__ out, int64_t ldso, int64_t ldro,
                                                                   float* __restrict__ state, const int32_t* __restrict__ count,
                                                                   const int32_t* __restrict__ reset, int S, int K, int C,
                                                                   OneEuro f) {
  pdl_wait();                                       // x and the tables come from earlier work in the stream
  pdl_launch_dependents();
  const int64_t idx = (int64_t)blockIdx.x * kSmoothThreads + threadIdx.x;
  if (idx >= (int64_t)S * C) return;
  const int s = (int)(idx / C), c = (int)(idx % C);
  const int n = count[s];
  if (n <= 0 || n > K) return;
  const float* xs = x + (int64_t)s * ldsx + c;
  float* os = out + (int64_t)s * ldso + c;
  float* st = state + (int64_t)s * 2 * C + c;
  float xp, dxp;
  int t = 0;
  if (reset[s]) {                                   // row 0 passes through and starts the state
    xp = xs[0];
    dxp = 0.0f;
    os[0] = xp;
    t = 1;
  } else {
    xp = st[0];
    dxp = st[C];
  }
  for (; t + kSmoothU <= n; t += kSmoothU) {
    float v[kSmoothU];
#pragma unroll
    for (int u = 0; u < kSmoothU; ++u) v[u] = xs[(int64_t)(t + u) * ldrx];
#pragma unroll
    for (int u = 0; u < kSmoothU; ++u) os[(int64_t)(t + u) * ldro] = f.step(v[u], xp, dxp);
  }
  for (; t < n; ++t) os[(int64_t)t * ldro] = f.step(xs[(int64_t)t * ldrx], xp, dxp);
  st[0] = xp;
  st[C] = dxp;
}

}  // namespace tp

using namespace tp;

extern "C" int tp_one_euro_filter(const float* x, int64_t ld_seq_x, int64_t ld_row_x, float* out, int64_t ld_seq_out,
                                  int64_t ld_row_out, float* state, const int32_t* count, const int32_t* reset, int S, int K,
                                  int C, float min_cutoff, float beta, void* stream) {
  TP_CHECK_ARG(x && out && state && count && reset, "tp_one_euro_filter: null pointer");
  TP_CHECK_ARG(S >= 1 && K >= 1 && C >= 1, "tp_one_euro_filter: need S, K, C >= 1 (S=%d K=%d C=%d)", S, K, C);
  TP_CHECK_ARG(ld_seq_x >= C && ld_row_x >= C && ld_seq_out >= C && ld_row_out >= C,
               "tp_one_euro_filter: strides must be >= C=%d (x %lld/%lld, out %lld/%lld)", C, (long long)ld_seq_x,
               (long long)ld_row_x, (long long)ld_seq_out, (long long)ld_row_out);
  TP_CHECK_ARG(std::isfinite(min_cutoff) && min_cutoff >= 0.0f && std::isfinite(beta) && beta >= 0.0f,
               "tp_one_euro_filter: min_cutoff and beta must be finite and >= 0 (got %g, %g)", (double)min_cutoff, (double)beta);
  const int64_t blocks = ceil_div((int64_t)S * C, kSmoothThreads);
  TP_CHECK_ARG(blocks <= 0x7fffffff, "tp_one_euro_filter: S*C too large (S=%d C=%d)", S, C);
  OneEuro f;
  f.mc = min_cutoff;
  f.beta = beta;
  f.a_d = kTwoPi / (kTwoPi + 1.0f);                 // host fp32, each operation rounded (no contraction on these two)
  f.one_m_a_d = 1.0f - f.a_d;
  PdlConfig lc(dim3((unsigned)blocks), dim3(kSmoothThreads), 0, (cudaStream_t)stream);
  TP_CUDA(cudaLaunchKernelEx(&lc.cfg, k_one_euro_filter, x, ld_seq_x, ld_row_x, out, ld_seq_out, ld_row_out, state, count, reset,
                             S, K, C, f));
  TP_LAUNCH_CHECK();
  return TP_OK;
}
