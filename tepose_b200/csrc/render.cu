// Mesh overlay of the demo (lib/utils/renderer.py: Renderer.render, once per person present, each over the previous result) on
// the device.  The contract is stated in include/tepose_b200.h and restated in oracle/render_ref.py; every rounding step here
// has its twin there, so frames are bit-identical.  Three launches:
//   k_render_project  vertices -> snapped pixel coordinates + depth, vertex normals from the vertex -> face CSR; resets the keys
//   k_render_raster   one thread per triangle over its frame-clipped box; a box above kAloneMax pixels goes to a shared list
//                     that the whole CTA (and gridDim.y CTAs side by side) sweeps; atomicMin of a 64-bit key per pixel
//   k_render_resolve  one thread per pixel: decode the key, recompute the barycentrics, shade in float64, write out
#include "common.cuh"

#include <algorithm>

namespace tp {
namespace {

constexpr int kProjThreads = 256;
constexpr int kRasterThreads = 128;
constexpr int kAloneMax = 64;                  // clipped box pixels a thread rasterises on its own
constexpr float kGuard = 32768.0f;             // guard band, pixels
constexpr unsigned long long kEmpty = ~0ull;
constexpr int kMaxPeople = 65535;              // key bits 48..63: n - 1 - person (never all ones)
constexpr int kMaxFaces = 65536;               // key bits 0..15: face index

__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }

// n / |n| when |n| is finite and > 0, else 0 (degenerate and non-finite faces contribute nothing)
__device__ __forceinline__ void normalize3(double n[3]) {
  const double len = __dsqrt_rn(dadd(dadd(dmul(n[0], n[0]), dmul(n[1], n[1])), dmul(n[2], n[2])));
  const bool ok = len > 0.0 && len <= 1.7976931348623157e308;
#pragma unroll
  for (int k = 0; k < 3; ++k) n[k] = ok ? __ddiv_rn(n[k], len) : 0.0;
}

// order-preserving bits of an fp32 value: a < b  <=>  key(a) < key(b)
__device__ __forceinline__ unsigned int depth_bits(float z) {
  const unsigned int u = __float_as_uint(z);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// one screen triangle: snapped coordinates oriented to positive area, its vertex ids in that order, depths, clipped box
struct Tri {
  int x[3], y[3], id[3];
  float z[3];
  long long area;
  int bx0, by0, bx1, by1;
  int p, f;
};

// Loads face f of person p from the projected vertices; false when the face draws nothing.
__device__ __forceinline__ bool setup_tri(const int4* __restrict__ proj, const int* __restrict__ faces, int p, int f, int V, int H,
                                          int W, Tri& t) {
  const int4* pv = proj + (size_t)p * V;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int id = __ldg(faces + 3 * f + k);
    if (id < 0 || id >= V) return false;
    const int4 q = __ldg(pv + id);
    if (!q.w) return false;
    t.x[k] = q.x; t.y[k] = q.y; t.z[k] = __int_as_float(q.z); t.id[k] = id;
  }
  long long a = (long long)(t.x[1] - t.x[0]) * (t.y[2] - t.y[0]) - (long long)(t.y[1] - t.y[0]) * (t.x[2] - t.x[0]);
  if (a == 0) return false;
  if (a < 0) {                                   // both windings: swap vertices 1 and 2
    int s;
    s = t.x[1]; t.x[1] = t.x[2]; t.x[2] = s;
    s = t.y[1]; t.y[1] = t.y[2]; t.y[2] = s;
    s = t.id[1]; t.id[1] = t.id[2]; t.id[2] = s;
    const float zz = t.z[1]; t.z[1] = t.z[2]; t.z[2] = zz;
    a = -a;
  }
  t.area = a;
  t.p = p; t.f = f;
  // pixel x is inside [lo, hi] when lo <= 256x + 128 <= hi
  const int lox = min(t.x[0], min(t.x[1], t.x[2])) - 128, hix = max(t.x[0], max(t.x[1], t.x[2])) - 128;
  const int loy = min(t.y[0], min(t.y[1], t.y[2])) - 128, hiy = max(t.y[0], max(t.y[1], t.y[2])) - 128;
  t.bx0 = max(-((-lox) >> 8), 0); t.bx1 = min(hix >> 8, W - 1);
  t.by0 = max(-((-loy) >> 8), 0); t.by1 = min(hiy >> 8, H - 1);
  return t.bx0 <= t.bx1 && t.by0 <= t.by1;
}

__device__ __forceinline__ long long edge(int ax, int ay, int bx, int by, int px, int py) {
  return (long long)(bx - ax) * (py - ay) - (long long)(by - ay) * (px - ax);
}

// 1 when a sample exactly on edge a -> b is NOT the triangle's: the top-left rule is "nudge the sample right, then down"
__device__ __forceinline__ long long edge_bias(int ax, int ay, int bx, int by) {
  const int dx = bx - ax, dy = by - ay;
  return (dy < 0 || (dy == 0 && dx > 0)) ? 0 : 1;
}

// barycentric weights (w[k] of vertex k, sum = area) of pixel (px, py); true when the pixel is covered
__device__ __forceinline__ bool cover(const Tri& t, int px, int py, long long w[3]) {
  w[0] = edge(t.x[1], t.y[1], t.x[2], t.y[2], px, py);
  w[1] = edge(t.x[2], t.y[2], t.x[0], t.y[0], px, py);
  w[2] = edge(t.x[0], t.y[0], t.x[1], t.y[1], px, py);
  return ((w[0] - edge_bias(t.x[1], t.y[1], t.x[2], t.y[2])) | (w[1] - edge_bias(t.x[2], t.y[2], t.x[0], t.y[0])) |
          (w[2] - edge_bias(t.x[0], t.y[0], t.x[1], t.y[1]))) >= 0;
}

__device__ __forceinline__ void raster_pixel(const Tri& t, double inv, unsigned long long base, int x, int y, int W,
                                             unsigned long long* __restrict__ keys) {
  long long w[3];
  if (!cover(t, 256 * x + 128, 256 * y + 128, w)) return;
  const double s = dadd(dadd(dmul((double)w[0], (double)t.z[0]), dmul((double)w[1], (double)t.z[1])),
                        dmul((double)w[2], (double)t.z[2]));
  const unsigned long long key = base | ((unsigned long long)depth_bits(__double2float_rn(dmul(s, inv))) << 16);
  unsigned long long* k = keys + (size_t)y * W + x;
  if (key < __ldcg(k)) atomicMin(k, key);      // keys only decrease: a stale read can only cost an extra atomic
}

__global__ void __launch_bounds__(kProjThreads) k_render_project(const float* __restrict__ verts, const float* __restrict__ cam,
                                                                 const int* __restrict__ faces, const int* __restrict__ vf_off,
                                                                 const int* __restrict__ vf_faces, int n, int V, int F, int H,
                                                                 int W, int4* __restrict__ proj, double* __restrict__ vnorm,
                                                                 unsigned long long* __restrict__ keys) {
  const size_t stride = (size_t)gridDim.x * blockDim.x, t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (size_t i = t0; i < (size_t)H * W; i += stride) keys[i] = kEmpty;
  const float hw = 0.5f * (float)W, hh = 0.5f * (float)H;
  for (size_t i = t0; i < (size_t)n * V; i += stride) {
    const int p = (int)(i / V), v = (int)(i - (size_t)p * V);
    const float X = verts[3 * i], Y = verts[3 * i + 1], Z = verts[3 * i + 2];
    const float sx = cam[4 * p], sy = cam[4 * p + 1], tx = cam[4 * p + 2], ty = cam[4 * p + 3];
    const float u = __fmul_rn(__fadd_rn(__fmul_rn(sx, __fadd_rn(X, tx)), 1.0f), hw);
    const float w = __fmul_rn(__fadd_rn(__fmul_rn(sy, __fadd_rn(Y, ty)), 1.0f), hh);
    const bool ok = isfinite(X) && isfinite(Y) && isfinite(Z) && fabsf(u) <= kGuard && fabsf(w) <= kGuard;
    proj[i] = make_int4(ok ? __float2int_rn(__fmul_rn(u, 256.0f)) : 0, ok ? __float2int_rn(__fmul_rn(w, 256.0f)) : 0,
                        __float_as_int(Z), ok ? 1 : 0);
    // vertex normal: the adjacent unit face normals summed in CSR order, then normalised
    const float* pv = verts + (size_t)p * V * 3;
    double s[3] = {0.0, 0.0, 0.0};
    for (int e = vf_off[v]; e < vf_off[v + 1]; ++e) {
      const int f = vf_faces[e];
      if (f < 0 || f >= F) continue;
      const int a = faces[3 * f], b = faces[3 * f + 1], c = faces[3 * f + 2];
      if (a < 0 || a >= V || b < 0 || b >= V || c < 0 || c >= V) continue;
      double e1[3], e2[3], fn[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const double o = (double)pv[3 * a + k];
        e1[k] = dsub((double)pv[3 * b + k], o);
        e2[k] = dsub((double)pv[3 * c + k], o);
      }
      fn[0] = dsub(dmul(e1[1], e2[2]), dmul(e1[2], e2[1]));
      fn[1] = dsub(dmul(e1[2], e2[0]), dmul(e1[0], e2[2]));
      fn[2] = dsub(dmul(e1[0], e2[1]), dmul(e1[1], e2[0]));
      normalize3(fn);
#pragma unroll
      for (int k = 0; k < 3; ++k) s[k] = dadd(s[k], fn[k]);
    }
    normalize3(s);
#pragma unroll
    for (int k = 0; k < 3; ++k) vnorm[3 * i + k] = s[k];
  }
}

// grid (ceil(n*F / kRasterThreads), split): thread x of CTA column bx owns triangle bx*kRasterThreads + x; the split CTAs of a
// column share the pixels of its large triangles (pixel i of a box goes to CTA i / kRasterThreads % split)
__global__ void __launch_bounds__(kRasterThreads) k_render_raster(const int4* __restrict__ proj, const int* __restrict__ faces,
                                                                  int n, int V, int F, int H, int W,
                                                                  unsigned long long* __restrict__ keys) {
  __shared__ Tri s_big[kRasterThreads];
  __shared__ int s_count;
  if (threadIdx.x == 0) s_count = 0;
  __syncthreads();
  const long long tri = (long long)blockIdx.x * kRasterThreads + threadIdx.x;
  Tri t;
  if (tri < (long long)n * F) {
    const int p = (int)(tri / F), f = (int)(tri - (long long)p * F);
    if (setup_tri(proj, faces, p, f, V, H, W, t)) {
      const int bw = t.bx1 - t.bx0 + 1, bh = t.by1 - t.by0 + 1;
      if ((long long)bw * bh > kAloneMax) {
        s_big[atomicAdd(&s_count, 1)] = t;
      } else if (blockIdx.y == 0) {
        const double inv = __drcp_rn((double)t.area);
        const unsigned long long base = ((unsigned long long)(n - 1 - p) << 48) | (unsigned long long)f;
        for (int y = t.by0; y <= t.by1; ++y)
          for (int x = t.bx0; x <= t.bx1; ++x) raster_pixel(t, inv, base, x, y, W, keys);
      }
    }
  }
  __syncthreads();
  const int nbig = s_count;
  for (int b = 0; b < nbig; ++b) {
    const Tri& u = s_big[b];
    const int bw = u.bx1 - u.bx0 + 1, total = bw * (u.by1 - u.by0 + 1);
    const double inv = __drcp_rn((double)u.area);
    const unsigned long long base = ((unsigned long long)(n - 1 - u.p) << 48) | (unsigned long long)u.f;
    for (int i = blockIdx.y * kRasterThreads + threadIdx.x; i < total; i += gridDim.y * kRasterThreads) {
      const int y = i / bw;
      raster_pixel(u, inv, base, u.bx0 + i - y * bw, u.by0 + y, W, keys);
    }
  }
}

__global__ void __launch_bounds__(kProjThreads) k_render_resolve(const uint8_t* __restrict__ frame, const int4* __restrict__ proj,
                                                                 const double* __restrict__ vnorm, const int* __restrict__ faces,
                                                                 const float* __restrict__ colors, int n, int V, int H, int W,
                                                                 const unsigned long long* __restrict__ keys,
                                                                 uint8_t* __restrict__ out) {
  const size_t HW = (size_t)H * W;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += (size_t)gridDim.x * blockDim.x) {
    const unsigned long long key = keys[i];
    uint8_t rgb[3] = {frame[3 * i], frame[3 * i + 1], frame[3 * i + 2]};
    Tri t;
    const int p = n - 1 - (int)(key >> 48), f = (int)(key & 0xffffu);
    const int y = (int)(i / W), x = (int)(i - (size_t)y * W);
    if (key != kEmpty && setup_tri(proj, faces, p, f, V, H, W, t)) {
      long long w[3];
      cover(t, 256 * x + 128, 256 * y + 128, w);
      double nn[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const double* a = vnorm + ((size_t)p * V + t.id[0]) * 3;
        const double* b = vnorm + ((size_t)p * V + t.id[1]) * 3;
        const double* c = vnorm + ((size_t)p * V + t.id[2]) * 3;
        nn[k] = dadd(dadd(dmul((double)w[0], a[k]), dmul((double)w[1], b[k])), dmul((double)w[2], c[k]));
      }
      normalize3(nn);
      const double shade = dadd(0.3, dmul(0.7, fabs(nn[2])));
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const double v = dmul(dmul((double)colors[3 * p + k], shade), 255.0);
        rgb[k] = (uint8_t)__double2int_rn(fmin(fmax(v, 0.0), 255.0));      // fmax(NaN, 0) = 0
      }
    }
    out[3 * i] = rgb[0]; out[3 * i + 1] = rgb[1]; out[3 * i + 2] = rgb[2];
  }
}

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

struct Layout {
  size_t keys, proj, vnorm, total;
};

Layout layout(int n, int V, int H, int W) {
  Layout l;
  l.keys = 0;
  l.proj = align256((size_t)H * W * sizeof(unsigned long long));
  l.vnorm = l.proj + align256((size_t)n * V * sizeof(int4));
  l.total = l.vnorm + align256((size_t)n * V * 3 * sizeof(double));
  return l;
}

bool dims_ok(int n, int V, int H, int W) {
  return n >= 0 && n <= kMaxPeople && V >= 1 && H >= 1 && W >= 1 && H <= 32768 && W <= 32768;
}

}  // namespace
}  // namespace tp

using namespace tp;

extern "C" size_t tp_render_workspace_bytes(int n, int V, int H, int W) {
  return dims_ok(n, V, H, W) ? layout(n, V, H, W).total : 0;
}

extern "C" int tp_render_meshes(const void* frame, const float* verts, const float* orig_cam, const float* colors,
                                const int32_t* faces, const int32_t* vf_offsets, const int32_t* vf_faces, int n, int V, int F,
                                int H, int W, void* out, void* workspace, size_t workspace_bytes, void* stream) {
  TP_CHECK_ARG(frame && out && faces && vf_offsets && vf_faces && workspace, "tp_render_meshes: null pointer");
  TP_CHECK_ARG(n == 0 || (verts && orig_cam && colors), "tp_render_meshes: null verts, orig_cam or colors with n = %d", n);
  TP_CHECK_ARG(dims_ok(n, V, H, W) && F >= 1 && F <= kMaxFaces,
               "tp_render_meshes: need 0 <= n <= %d, V >= 1, 1 <= F <= %d, 1 <= H, W <= 32768 (n=%d V=%d F=%d H=%d W=%d)",
               kMaxPeople, kMaxFaces, n, V, F, H, W);
  TP_CHECK_ARG(aligned16(workspace), "tp_render_meshes: workspace must be 16-byte aligned");
  const Layout l = layout(n, V, H, W);
  TP_CHECK_ARG(workspace_bytes >= l.total, "tp_render_meshes: workspace of %zu bytes, need %zu", workspace_bytes, l.total);
  char* ws = reinterpret_cast<char*>(workspace);
  auto* keys = reinterpret_cast<unsigned long long*>(ws + l.keys);
  auto* proj = reinterpret_cast<int4*>(ws + l.proj);
  auto* vnorm = reinterpret_cast<double*>(ws + l.vnorm);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t grid_cap = (int64_t)sm_count() * 8;
  const int64_t proj_work = std::max<int64_t>((int64_t)H * W, (int64_t)n * V);
  const int proj_blocks = (int)std::min<int64_t>(ceil_div(proj_work, kProjThreads), grid_cap);
  k_render_project<<<proj_blocks, kProjThreads, 0, st>>>(verts, orig_cam, faces, vf_offsets, vf_faces, n, V, F, H, W, proj,
                                                         vnorm, keys);
  TP_LAUNCH_CHECK();
  if (n > 0) {
    const int64_t cols = ceil_div((int64_t)n * F, kRasterThreads);
    // enough CTAs to fill the device when there are few triangles: the split CTAs share the pixels of the large ones
    const int split = (int)std::min<int64_t>(16, std::max<int64_t>(1, ceil_div(grid_cap, cols)));
    k_render_raster<<<dim3((unsigned)cols, split), kRasterThreads, 0, st>>>(proj, faces, n, V, F, H, W, keys);
    TP_LAUNCH_CHECK();
  }
  const int res_blocks = (int)std::min<int64_t>(ceil_div((int64_t)H * W, kProjThreads), grid_cap);
  k_render_resolve<<<res_blocks, kProjThreads, 0, st>>>(reinterpret_cast<const uint8_t*>(frame), proj, vnorm, faces, colors, n,
                                                        V, H, W, keys, reinterpret_cast<uint8_t*>(out));
  TP_LAUNCH_CHECK();
  return TP_OK;
}
