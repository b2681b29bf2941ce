// Slot-managed windows of the windowed loop (tepose_b200.tracks): the per-row feature roll and theta roll of
// tepose_b200.stream.WindowedTePose, driven by a device table so that one captured graph follows tracks as they start, pause
// and end.  x is the loop's window [S,T,ld] fp32 (features in columns 0..2047, the theta ring in 2048..2132).  Rows of 2133
// floats are only 4-byte aligned, so every access is a scalar fp32 one; a thread owns one column of one slot and walks its T
// frames, which makes the in-place shift race-free without a barrier.
#include "common.cuh"

namespace tp {

constexpr int kSlotFeat = 2048;                     // static features per frame
constexpr int kSlotCols = kSlotFeat + 85;           // features + theta: the columns a window row uses
constexpr int kSlotThreads = 256;
constexpr int kSlotColThreads = 96;                 // the commit kernel: one thread per theta column
constexpr int kSlotU = 8;                           // frames a thread has in flight while shifting

// p[0..n-1] <- p[1..n] along a column of stride ld; kSlotU loads are issued before their stores
__device__ __forceinline__ void shift_column(float* p, int64_t ld, int n) {
  int t = 0;
  for (; t + kSlotU <= n; t += kSlotU) {
    float v[kSlotU];
#pragma unroll
    for (int u = 0; u < kSlotU; ++u) v[u] = p[(int64_t)(t + 1 + u) * ld];
#pragma unroll
    for (int u = 0; u < kSlotU; ++u) p[(int64_t)(t + u) * ld] = v[u];
  }
  for (; t < n; ++t) p[(int64_t)t * ld] = p[(int64_t)(t + 1) * ld];
}

// grid (S, ceil(kSlotCols / kSlotThreads)).  op 2 zeroes columns 0..2132 of every frame, then writes feats[src] as the newest
// frame; op 1 shifts the features by one frame and writes feats[src] as the newest; op 0, an unknown op or src outside [0, S)
// leave the slot untouched and read nothing.
__global__ void __launch_bounds__(kSlotThreads) k_window_slots_push(float* __restrict__ x, int S, int T, int64_t ld,
                                                                   const float* __restrict__ feats,
                                                                   const int32_t* __restrict__ src,
                                                                   const int32_t* __restrict__ op) {
  pdl_wait();                                       // the features come from the previous kernel
  pdl_launch_dependents();
  const int s = blockIdx.x;
  const int o = op[s], r = src[s];
  if ((o != 1 && o != 2) || r < 0 || r >= S) return;
  const int c = blockIdx.y * kSlotThreads + threadIdx.x;
  if (c >= kSlotCols || (o == 1 && c >= kSlotFeat)) return;
  float* col = x + (int64_t)s * T * ld + c;
  const float f = c < kSlotFeat ? feats[(int64_t)r * kSlotFeat + c] : 0.0f;
  if (o == 2) {
    for (int t = 0; t < T - 1; ++t) col[(int64_t)t * ld] = 0.0f;
  } else {
    shift_column(col, ld, T - 1);
  }
  col[(int64_t)(T - 1) * ld] = f;
}

// grid S, kSlotColThreads threads.  Slots with op 1 or 2: theta[0..T-3] <- theta[1..T-2], theta[T-2] <- theta_new[s]
// (WindowedTePose._body's roll); theta slot T-1 is never written.
__global__ void __launch_bounds__(kSlotColThreads) k_window_slots_commit(float* __restrict__ x, int T, int64_t ld,
                                                                        const float* __restrict__ theta,
                                                                        const int32_t* __restrict__ op) {
  pdl_wait();                                       // theta comes from the window step
  pdl_launch_dependents();
  const int s = blockIdx.x;
  const int o = op[s];
  const int c = threadIdx.x;
  if ((o != 1 && o != 2) || c >= 85) return;
  float* col = x + (int64_t)s * T * ld + kSlotFeat + c;
  const float v = theta[(int64_t)s * 85 + c];
  shift_column(col, ld, T - 2);
  col[(int64_t)(T - 2) * ld] = v;
}

static bool aligned4(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; }

}  // namespace tp

using namespace tp;

extern "C" int tp_window_slots_push(float* x, int S, int T, int64_t ld, const float* feats, const int32_t* src,
                                    const int32_t* op, void* stream) {
  TP_CHECK_ARG(x && feats && src && op, "tp_window_slots_push: null pointer");
  TP_CHECK_ARG(S >= 1 && T >= 2 && ld >= kSlotCols, "tp_window_slots_push: need S >= 1, T >= 2, ld >= %d (S=%d T=%d ld=%lld)",
               kSlotCols, S, T, (long long)ld);
  TP_CHECK_ARG(aligned4(x) && aligned4(feats) && aligned4(src) && aligned4(op), "tp_window_slots_push: pointers must be 4-byte aligned");
  PdlConfig lc(dim3((unsigned)S, (unsigned)ceil_div(kSlotCols, kSlotThreads)), dim3(kSlotThreads), 0, (cudaStream_t)stream);
  TP_CUDA(cudaLaunchKernelEx(&lc.cfg, k_window_slots_push, x, S, T, ld, feats, src, op));
  TP_LAUNCH_CHECK();
  return TP_OK;
}

extern "C" int tp_window_slots_commit(float* x, int S, int T, int64_t ld, const float* theta, const int32_t* op, void* stream) {
  TP_CHECK_ARG(x && theta && op, "tp_window_slots_commit: null pointer");
  TP_CHECK_ARG(S >= 1 && T >= 2 && ld >= kSlotCols, "tp_window_slots_commit: need S >= 1, T >= 2, ld >= %d (S=%d T=%d ld=%lld)",
               kSlotCols, S, T, (long long)ld);
  TP_CHECK_ARG(aligned4(x) && aligned4(theta) && aligned4(op), "tp_window_slots_commit: pointers must be 4-byte aligned");
  PdlConfig lc(dim3((unsigned)S), dim3(kSlotColThreads), 0, (cudaStream_t)stream);
  TP_CUDA(cudaLaunchKernelEx(&lc.cfg, k_window_slots_commit, x, T, ld, theta, op));
  TP_LAUNCH_CHECK();
  return TP_OK;
}
