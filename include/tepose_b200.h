/*
 * tepose_b200 -- C ABI of the B200 (sm_100a) implementation of TePose's per-sequence
 * inference hot path.
 *
 * The reference (ostadabbas/TePose) is pure Python/PyTorch and has no FFI of its own;
 * the boundary it exposes is the Python module API of lib.models (SURVEY.md 8b).  The
 * entry points below are what a reference-side ctypes binding for that path calls:
 * each comment names the reference code the entry point replaces (paths relative to
 * the reference repository).  See INTEGRATION.md for the binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless it says "host"; the library never
 *     allocates or frees caller memory (scratch comes in through `workspace`);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*), no host
 *     synchronisation, safe to capture in a CUDA graph;
 *   - return value: 0 = ok, <0 = error (see TP_ERR_*); tp_last_error() gives the text
 *     for the calling thread;
 *   - matrices are row-major float32 unless stated; `ld*` are row strides in ELEMENTS.
 */
#ifndef TEPOSE_B200_H
#define TEPOSE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define TP_API __attribute__((visibility("default")))
#else
#define TP_API
#endif

#define TP_OK 0
#define TP_ERR_INVALID (-1)     /* bad argument (null pointer, misaligned, bad size)   */
#define TP_ERR_UNSUPPORTED (-2) /* shape / device not supported by this build           */
#define TP_ERR_CUDA (-3)        /* a CUDA runtime / driver call failed                  */

#define TP_PRECISION_FP32 0 /* fp32 operands, FFMA, fp32 accumulate (strict parity mode)   */
#define TP_PRECISION_BF16 1 /* bf16 operands on tensor cores, fp32 accumulate + fp32 state */
#define TP_PRECISION_BF16X3 2 /* tp_gru_recurrence only: fp32-grade recurrent matmul on tensor cores.  Both operands are split
                                 x = hi + lo with hi = bf16(x), lo = bf16(x - hi); h.W^T = hi.W_hi + lo.W_hi + hi.W_lo (the lo.lo
                                 term, 2^-18 relative, is dropped) runs as ONE bf16 contraction over the K-concatenated operands
                                 [h_hi | h_lo | h_hi] x [W_hi | W_hi | W_lo]: w_hh is tp_pack_mma_a_bf16 of that [3H, 3H] matrix.
                                 State, gates and accumulation stay fp32 (exact expf / tanhf).                                 */

#define TP_POSE_ROTMAT 0     /* [n,24,3,3]  (smplx pose2rot=False, lib/models/spin.py:265-270) */
#define TP_POSE_AXIS_ANGLE 1 /* [n,72]      (smplx pose2rot=True,  lib/utils/eval_utils.py:168) */
#define TP_POSE_ROT6D 2      /* [n,144]     (rot6d_to_rotmat fused, lib/models/spin.py:263)     */

#define TP_RODRIGUES_SMPLX 0 /* smplx.lbs.batch_rodrigues                         */
#define TP_RODRIGUES_QUAT 1  /* lib/utils/geometry.py:22-65 (quaternion form)     */

/* joint source codes for tp_smpl_forward (composition of lib/models/smpl.py:75-77 and
 * lib/models/spin.py:275-278): */
#define TP_JSRC_POSED(j) (j)            /* 0..23  : posed kinematic-chain joint          */
#define TP_JSRC_REGRESSED(r) (100 + (r)) /* row r of the caller-supplied joint regressor  */
#define TP_JSRC_VERTEX(v) (1000 + (v))   /* mesh vertex v (smplx vertex_joint_selector)   */

TP_API int tp_version(void);
TP_API const char* tp_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
TP_API unsigned long long tp_launch_count(void);
/* Programmatic dependent launch between the kernels of a forward (each kernel's set-up overlaps the tail of its
 * predecessor).  On by default; profiling passes that bracket single kernels with events switch it off.  Returns the
 * previous setting. */
TP_API int tp_set_pdl(int enable);
/* The iterations of the fused IEF loop (lib/models/spin.py:250-261) as ONE 16-CTA thread-block cluster with the weights
 * on chip (csrc/ief_cluster.inl), instead of one grid barrier per layer.  On by default where the device can host the
 * cluster; 0 keeps the iterations inside the grid-barrier kernel (A/B tests).  Returns the previous setting. */
TP_API int tp_set_ief_cluster(int enable);
/* host out-params; any may be NULL */
TP_API int tp_device_info(int device, int* sm_count, int* cc_major, int* cc_minor, size_t* smem_per_block_optin);

/* ------------------------------------------------------------------ rotation utilities
 * lib/utils/geometry.py:330-343  rot6d_to_rotmat          x [n,6]   -> R [n,3,3]          */
TP_API int tp_rot6d_to_rotmat(const float* x, float* R, int64_t n, void* stream);
/* lib/utils/geometry.py:68-233   rotation_matrix_to_angle_axis   R [n,3,3] -> aa [n,3]   */
TP_API int tp_rotmat_to_angle_axis(const float* R, float* aa, int64_t n, void* stream);
/* smplx.lbs.batch_rodrigues / lib/utils/geometry.py:22-65   aa [n,3] -> R [n,3,3]        */
TP_API int tp_batch_rodrigues(const float* aa, float* R, int64_t n, int form, void* stream);
/* lib/models/spin.py:307-351  projection   joints [n,nj,3], cam [n,3] -> kp2d [n,nj,2]   */
TP_API int tp_projection(const float* joints, const float* cam, float* kp2d, int n, int nj, void* stream);

/* ------------------------------------------------------------------ operand packing
 * Gathers a [rows_b, rows_t, k] fp32 tensor (element (b,t,c) at src[b*stride_b + t*stride_t + c])
 * into a dense, zero-padded [rows_t*rows_b, kp] matrix whose row index is t*rows_b + b
 * (time-major, what the recurrence consumes), as fp32 (dst_precision 0) or bf16 (1).
 * Replaces x.permute(1,0,2) (lib/models/tepose.py:73,76).  kp >= k, kp % 8 == 0.        */
TP_API int tp_pack_rows(const float* src, int64_t stride_b, int64_t stride_t, int rows_b, int rows_t, int k,
                 void* dst, int kp, int dst_precision, int relu, void* stream);
/* Same; additionally clears `zero_bytes` bytes at `zero` (the grid-barrier slots of the persistent kernels that follow in
 * the step: tp_gru_recurrence_ex, tp_heads_ief_forward), so the step needs no separate fill.  zero may be NULL.           */
TP_API int tp_pack_rows_ex(const float* src, int64_t stride_b, int64_t stride_t, int rows_b, int rows_t, int k,
                    void* dst, int kp, int dst_precision, int relu, void* zero, size_t zero_bytes, void* stream);
/* tp_pack_rows_ex for a float16 source (strides in elements): the reference's datasets keep features and thetas as float16 on
 * the host (lib/dataset/dataset_3d.py:244-248), so a caller may ship them as they are -- half the host -> device bytes.   */
TP_API int tp_pack_rows_f16(const void* src_f16, int64_t stride_b, int64_t stride_t, int rows_b, int rows_t, int k,
                     void* dst, int kp, int dst_precision, int relu, void* zero, size_t zero_bytes, void* stream);
/* dst [rows, 3 k] bf16 = [hi | lo | hi] of src [rows, k] fp32 (row stride ld_src): the A operand of a bf16 x 3 contraction whose
 * weight side is [W_hi | W_hi | W_lo] (see TP_PRECISION_BF16X3).  k % 8 == 0.                                             */
TP_API int tp_split3_bf16(const float* src, int64_t ld_src, int rows, int k, void* dst, void* stream);
/* The way back, with the residual of lib/models/vibe.py:60-63 folded in (y + x, then TNF -> NTF):
 * out[b*rows_t + t, c] = y[(t*rows_b + b)*ld_y + c] + x[b*stride_b + t*stride_t + c]   (x may be NULL: no residual).
 * out is dense [rows_b*rows_t, k] fp32; out_bf16 (optional) receives the same rows in bf16.  k even.              */
TP_API int tp_unpack_rows_residual(const float* y, int64_t ld_y, const float* x, int64_t stride_b, int64_t stride_t,
                            int rows_b, int rows_t, int k, float* out, void* out_bf16, void* stream);

/* ------------------------------------------------------------------ GEMMs (torch.nn.Linear / GRU input projection)
 * C[M,N] = alpha * ( act(A)[M,K] . W[N,K]^T + bias[N] ) + beta * Cin[M,N]
 * fp32 FFMA path.  bias / Cin may be NULL; Cin may alias C.  K % 4 == 0, lda/ldw % 4 == 0,
 * A and W 16-byte aligned.  relu_a applies max(.,0) to A on load (F.relu before Linear,
 * lib/models/tepose.py:79-80).                                                           */
TP_API int tp_gemm_f32(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                const float* Cin, int64_t ldcin, float* C, int64_t ldc,
                int M, int N, int K, float alpha, float beta, int relu_a, void* stream);

/* Same GEMM with the K loop split over `splits` CTAs per output tile (skinny M: lets every SM
 * stream a slice of W).  Partials are reduced in split order by the last CTA to arrive, so the
 * result is deterministic.  workspace: tp_gemm_f32_splitk_workspace_bytes(M,N,splits) bytes,
 * 16-byte aligned, whose first 4096 bytes must be ZERO before the first use (the kernel leaves
 * them zero again).                                                                       */
TP_API size_t tp_gemm_f32_splitk_workspace_bytes(int M, int N, int splits);
TP_API int tp_gemm_f32_splitk(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                       const float* Cin, int64_t ldcin, float* C, int64_t ldc,
                       int M, int N, int K, float alpha, float beta, int relu_a, int splits,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ---- skinny (M <= 64) tensor-core GEMM with fragment-packed bf16 weights (nn.Linear at batch 32/64)
 * tp_pack_mma_a_bf16: W [rows, cols] fp32 (row stride ld) -> tp_pack_mma_a_bytes(rows, cols) bytes at
 * dst in mma.sync A-fragment order (done once per weight update).
 * tp_skinny_bf16: C[M,N] = alpha*(act(A)[M,K] . W^T + bias) + beta*Cin, A fp32 (rounded to bf16 on
 * the fly), fp32 accumulate.  splits > 1 splits K over CTAs; workspace as for tp_gemm_f32_splitk
 * (tp_skinny_bf16_workspace_bytes, first 4096 bytes zero).  K % 4 == 0, lda % 4 == 0.            */
TP_API size_t tp_pack_mma_a_bytes(int rows, int cols);
TP_API int tp_pack_mma_a_bf16(const float* w, int64_t ld, int rows, int cols, void* dst, void* stream);
TP_API size_t tp_skinny_bf16_workspace_bytes(int M, int N, int splits);
TP_API int tp_skinny_bf16(const float* A, int64_t lda, int M, int K, const void* Wp, int N, const float* bias,
                   const float* Cin, int64_t ldcin, float* C, int64_t ldc, float alpha, float beta,
                   int relu_a, int splits, void* workspace, size_t workspace_bytes, void* stream);

/* Extended form: A may also be given as a bf16 copy (A_bf16 [M, lda_bf16], read instead of A when
 * non-NULL; K % 8 == 0), and the output can additionally be written as bf16 (C_bf16) for the next
 * layer.  mode 0 = auto, 1 = split-K kernel (128 rows per CTA), 2 = single-phase kernel (one 16-row
 * tile per CTA, K split over the warps; no workspace needed).                                    */
TP_API int tp_skinny_bf16_ex(const float* A, int64_t lda, const void* A_bf16, int64_t lda_bf16, int M, int K,
                      const void* Wp, int N, const float* bias, const float* Cin, int64_t ldcin, float* C,
                      int64_t ldc, void* C_bf16, int64_t ldc_bf16, float alpha, float beta, int relu_a,
                      int splits, int mode, void* workspace, size_t workspace_bytes, void* stream);

/* One segment of a tensor-core GEMM launch: rows [m_start, m_start+m_rows) of A against rows
 * [n_start, n_start+n_cols) of W;  out[(m-m_start)*ldc + (n-n_start)] = dot + bias[n-n_start].
 * Epilogue options (flags; 0 = the plain fp32 output above): TP_GEMM_RELU clamps at zero, TP_GEMM_OUT_BF16 makes `out` a bf16
 * matrix (ldc in elements, ldc % 8 == 0), and a non-NULL `residual` (bf16 [m_rows, ldr], ldr % 8 == 0) is added before the clamp
 * -- the conv + folded BatchNorm (+ shortcut) + ReLU of a ResNet bottleneck (lib/models/spin.py:35-54) as one GEMM.
 * Split layout (fp32-grade activations on bf16 operands): a row of C values v is stored as bf16 [hi(C) | lo(C) | hi(C)] with
 * hi = RN_bf16(v), lo = RN_bf16(v - hi).  TP_GEMM_OUT_SPLIT3 writes the fp32 result v (after bias, residual and ReLU) that way:
 * `out` is bf16, hi at column c, lo at n_cols + c, hi at 2 n_cols + c (ldc % 8 == 0, ldc >= 3 n_cols; TP_GEMM_OUT_BF16 is then
 * ignored).  TP_GEMM_RES_SPLIT3: the residual rows are in split layout (ldr >= 3 n_cols) and hi + lo is added.              */
#define TP_GEMM_RELU 1
#define TP_GEMM_OUT_BF16 2
#define TP_GEMM_OUT_SPLIT3 4
#define TP_GEMM_RES_SPLIT3 8
typedef struct tp_gemm_seg {
  int32_t m_start, m_rows;
  int32_t n_start, n_cols; /* n_cols % 16 == 0 */
  float* out;
  int64_t ldc;
  const float* bias; /* [n_cols] or NULL */
  int32_t flags;
  int32_t ldr;
  const void* residual;
} tp_gemm_seg;

/* tcgen05 / TMEM GEMM fed by TMA (GRU input projection over all timesteps, K1):
 * A [a_rows, kp] bf16 and W [w_rows, kp] bf16, both K-major, kp % 64 == 0, 16-byte aligned.
 * `segs` is a HOST array (nseg <= 8).  Requires an sm_100 device.                        */
TP_API int tp_gemm_bf16_tc(const void* A, int a_rows, const void* W, int w_rows, int kp,
                    const tp_gemm_seg* segs, int nseg, void* stream);

/* ------------------------------------------------------------------ HMR ResNet-50 feature extractor (SURVEY 8 f-5)
 * Data movement around tp_gemm_bf16_tc for lib/models/spin.py:59-141 (feature_extractor; caller demo.py:183-198).
 * Activations are NHWC bf16; a convolution is  im2col rows x [Cout, kh*kw*Cin (padded to KP)]  with BatchNorm folded into
 * the weights / bias (eval mode) and ReLU / shortcut in the GEMM epilogue (TP_GEMM_RELU, TP_GEMM_OUT_BF16, residual).     */
/* x [N,C,H,W] fp32 -> y [N,H,W,CP] bf16, channels C..CP-1 zero */
TP_API int tp_nchw_to_nhwc_bf16(const float* x, void* y, int N, int C, int H, int W, int CP, void* stream);
/* in [N,H,W,C] bf16 -> out [N*Ho*Wo, KP] bf16, column (ky*kw + kx)*C + c, zero outside the image and beyond kh*kw*C;
 * Ho = (H + 2 pad - kh) / stride + 1 (nn.Conv2d); C % 4 == 0, KP % 8 == 0 */
TP_API int tp_im2col_nhwc_bf16(const void* in, void* out, int N, int H, int W, int C, int kh, int kw, int stride, int pad,
                        int KP, void* stream);
/* nn.MaxPool2d(kernel_size=3, stride=2, padding=1) on NHWC bf16 (lib/models/spin.py:70); C % 8 == 0 */
TP_API int tp_maxpool3x3s2_nhwc_bf16(const void* in, void* out, int N, int H, int W, int C, void* stream);
/* mean over the HW positions of [N, HW, C] bf16 -> [N, C] fp32 (nn.AvgPool2d(7) on the 7x7 map + view, spin.py:75,139-140) */
TP_API int tp_avgpool_nhwc_bf16(const void* in, float* out, int N, int HW, int C, void* stream);
/* Split-layout counterparts (precision "fp32_tc": every activation of C channels is bf16 [N,H,W,3C], [hi | lo | hi] per pixel as
 * TP_GEMM_OUT_SPLIT3 writes it; tp_im2col_nhwc_bf16 gathers it unchanged with C' = 3C).
 * x [N,C,H,W] fp32 -> y [N,H,W,3 CP] bf16, channels C..CP-1 of each block zero (CP = 4 for the RGB stem: 12 channels) */
TP_API int tp_nchw_to_nhwc_split3(const float* x, void* y, int N, int C, int H, int W, int CP, void* stream);
/* nn.MaxPool2d(3, 2, 1) on [N,H,W,3C] split rows: compares the represented values hi + lo exactly and writes the winning
 * (hi, lo) pair (the first in (ky, kx) order on a tie); C % 8 == 0 */
TP_API int tp_maxpool3x3s2_nhwc_split3(const void* in, void* out, int N, int H, int W, int C, void* stream);
/* mean over the HW positions of hi + lo of [N, HW, 3C] split rows -> [N, C] fp32 (sequential fp32 sum, one division) */
TP_API int tp_avgpool_nhwc_split3(const void* in, float* out, int N, int HW, int C, void* stream);

/* ------------------------------------------------------------------ demo front end: person crops on the device
 * One row of the crop table: the box of a tracked person (lib/data_utils/_img_utils.py: get_single_image_crop_demo, bbox =
 * centre x, centre y, width, height in pixels) in frame `frame`, enlarged by `scale` (the demo passes 1.2).  24 bytes. */
typedef struct tp_crop {
  int32_t frame;
  float cx, cy, w, h;
  float scale;
} tp_crop;
/* frames uint8 [F,H,W,3] RGB -> out [N,224,224,4] bf16 NHWC, channel 3 zero (the layout tp_im2col_nhwc_bf16 takes for the HMR
 * stem).  Crop n is generate_patch_image_cv(frames[crops[n].frame], cx, cy, w, h, 224, 224, do_flip=False, scale, rot=0)
 * (gen_trans_from_patch_cv -> cv2.getAffineTransform -> cv2.warpAffine INTER_LINEAR / BORDER_CONSTANT 0, all with cv2's
 * double and fixed-point rounding) followed by ToTensor + Normalize(ImageNet mean / std) in fp32 and one round to bf16:
 * bit-identical to that host pipeline (oracle/crop_ref.py).  `crops` is a DEVICE table (N <= 65535) read when the kernel
 * runs, so a captured graph follows boxes rewritten between replays.  Outside graph capture the call reads the frame indices
 * back (one stream synchronisation) and rejects an index outside [0, F); a captured launch that meets one writes zeros for
 * that crop and reads no frame.  Source positions must stay within 2^20 pixels of the origin (cv2's positions are int32 in
 * 1/1024 pixel).  crops 4-byte, out 16-byte aligned. */
TP_API int tp_crop_normalize_bf16(const void* frames, int F, int H, int W, const tp_crop* crops, int N, void* out,
                                  void* stream);
/* The same crop and the same fp32 normalisation, written in split layout instead of rounded: out [N,224,224,12] bf16,
 * [hi(4) | lo(4) | hi(4)] per pixel with channel 3 of each block zero (the stem input of precision "fp32_tc").  Same argument
 * checks and the same behaviour for a bad frame index under capture. */
TP_API int tp_crop_normalize_split3(const void* frames, int F, int H, int W, const tp_crop* crops, int N, void* out,
                                    void* stream);

/* ------------------------------------------------------------------ demo output: mesh overlay
 * The demo's overlay (lib/utils/renderer.py: Renderer.render, called once per person present, each over the previous result)
 * with a contract of this library's own (tepose_b200/render.py, oracle/render_ref.py restate it):
 *   - person i's vertex (X,Y,Z) of verts [n,V,3] fp32 lands at pixel u = (sx*(X+tx)+1)*W/2, v = (sy*(Y+ty)+1)*H/2 with
 *     orig_cam[i] = (sx, sy, tx, ty) fp32 (the reference's weak-perspective camera with the mesh turned 180 degrees about x),
 *     every fp32 operation separately rounded, snapped to 1/256 pixel; depth is Z, smaller nearer;
 *   - a triangle with a non-finite vertex, a vertex more than 2^15 pixels from the origin, or zero snapped area draws nothing;
 *   - pixel (x,y) is sampled at its centre; int64 edge functions with a top-left rule (both windings), so a pixel on an edge
 *     shared by two triangles belongs to exactly one;
 *   - visibility: later person first, then nearer, then lower face index (64-bit key: person 16 | depth 32 | face 16 bits);
 *   - shading in float64: vertex normals are the normalised sums of the adjacent unit face normals in CSR order,
 *     interpolated with the integer barycentrics and normalised; colour = colors[i] * (0.3 + 0.7*|n_z|), *255, clamped to
 *     [0,255], rounded to nearest even.  Uncovered pixels copy the frame.
 * frame, out uint8 [H,W,3] (frame is only read); colors [n,3] fp32; faces int32 [F,3]; vf_offsets int32 [V+1] and vf_faces
 * int32 [vf_offsets[V]]: the faces of vertex v are vf_faces[vf_offsets[v] .. vf_offsets[v+1]) in ascending order.
 * 0 <= n <= 65535, 1 <= F <= 65536, 1 <= H, W <= 32768.  workspace: tp_render_workspace_bytes(n, V, H, W) bytes, 16-byte
 * aligned, any content (the first kernel resets what it reads).  Three kernels (project, raster, resolve), no host sync. */
TP_API size_t tp_render_workspace_bytes(int n, int V, int H, int W);
TP_API int tp_render_meshes(const void* frame, const float* verts, const float* orig_cam, const float* colors,
                            const int32_t* faces, const int32_t* vf_offsets, const int32_t* vf_faces, int n, int V, int F,
                            int H, int W, void* out, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ tracked people: slot-managed windows
 * The windowed loop's state x [S,T,ld] fp32 (ld >= 2133; frame t of slot s is the row x + (s*T + t)*ld: features in columns
 * 0..2047, the theta ring in 2048..2132) for S slots, each holding one tracked person.  Two DEVICE tables of S int32 drive a
 * push, read when the kernels run, so a captured graph follows tracks that start, pause and end between replays:
 *   op[s]  0 = no frame for slot s this push, 1 = the next frame of the slot's track, 2 = the first frame of a new track;
 *   src[s] the row of feats [>= S, 2048] fp32 holding slot s's frame.
 * Rows are only 4-byte aligned (no 16-byte access is assumed).  The push leaves a slot whose op is outside {0,1,2} or whose
 * src is outside [0,S) untouched and reads nothing for it; the commit (which reads no src) leaves a slot whose op is outside
 * {0,1,2} untouched.  The callers validate the tables they write; a replayed graph cannot check them.  Every pointer 4-byte
 * aligned. */
/* Before the window step.  op 2: columns 0..2132 of every frame of the slot become 0, then feats[src[s]] is frame T-1;
 * op 1: the slot's features shift one frame towards 0 and feats[src[s]] becomes frame T-1 (theta columns untouched);
 * op 0: nothing. */
TP_API int tp_window_slots_push(float* x, int S, int T, int64_t ld, const float* feats, const int32_t* src, const int32_t* op,
                                void* stream);
/* After the window step, with theta [S,85] fp32 its newest predictions: for op 1 or 2, theta ring [0..T-3] <- [1..T-2] and
 * ring[T-2] <- theta[s] (evaluate.py:268-269 per slot); op 0 keeps the slot's ring.  Ring slot T-1 is never written. */
TP_API int tp_window_slots_commit(float* x, int S, int T, int64_t ld, const float* theta, const int32_t* op, void* stream);

/* ------------------------------------------------------------------ demo output: pose smoothing
 * The One-Euro filter of lib/utils/one_euro_filter.py as lib/utils/smooth_pose.py runs it (t_e = 1 on every row), as a
 * ragged batched scan that carries its state between calls.  Sequence s of S filters its rows 0..count[s]-1 in order: row r of
 * x is x + s*ld_seq_x + r*ld_row_x (C fp32 channels), and its result goes to the same place in out.  state [S,2,C] fp32 is
 * x_prev | dx_prev per sequence.  With reset[s] != 0, row 0 is copied through unchanged and starts the state (x_prev = row 0,
 * dx_prev = 0); otherwise filtering continues from state[s].  After the call state[s] holds the last row's x_hat | dx_hat.
 * Per channel, with K = fl32(2*pi), every operation rounded on its own in fp32 (no FMA contraction):
 *   a_d = K/(K+1);  dx = x - x_prev;  dx_hat = a_d*dx + (1-a_d)*dx_prev;  cutoff = min_cutoff + beta*|dx_hat|;
 *   r = K*cutoff;  a = r/(r+1);  x_hat = a*x + (1-a)*x_prev
 * which is bit-identical to the reference's float32 numpy arithmetic.  count and reset are DEVICE int32 [S], read when the
 * kernel runs (a captured graph follows new tables); count[s] == 0, or outside [0,K], reads and writes nothing for sequence s.
 * Strides >= C; rows need only 4-byte alignment (x may be the view theta[:, 3:75] of [N,85] rows).  min_cutoff and beta finite
 * and >= 0.  One kernel, no host sync. */
TP_API int tp_one_euro_filter(const float* x, int64_t ld_seq_x, int64_t ld_row_x, float* out, int64_t ld_seq_out,
                              int64_t ld_row_out, float* state, const int32_t* count, const int32_t* reset, int S, int K, int C,
                              float min_cutoff, float beta, void* stream);

/* ------------------------------------------------------------------ GRU recurrence (K2)
 * One direction of one torch.nn.GRU layer (lib/models/tepose.py:53-64,73,76) given the
 * input projections gi = x.W_ih^T + b_ih.  Step s (0-based) reads gi row block
 * (t_in0 + s*t_in_step) and writes outputs at time index (t_out0 + s*t_out_step).          */
typedef struct tp_gru_job {
  const float* gi;   /* [T, B, ldg] fp32, columns ordered r|z|n (3H wide)                  */
  int64_t ldg;
  const void* w_hh;  /* fp32: [3H,H] row-major.  bf16: fragment-packed by tp_pack_whh_bf16      */
  const float* b_hh; /* [3H]                                                                */
  const float* h0;   /* [B,H] (ld = H) initial state, or NULL for zeros                     */
  float* y;          /* optional [T,B,ldy] fp32 sequence output, or NULL                    */
  int64_t ldy;
  void* y_lp;        /* optional bf16 copy of the sequence output [T,B,ldy_lp], or NULL     */
  int64_t ldy_lp;
  float* h_final;    /* optional [B,ld_hf] state after the last step, or NULL               */
  int64_t ld_hf;
  int32_t steps;
  int32_t t_in0, t_in_step;
  int32_t t_out0, t_out_step;
  float* gates;          /* optional [T,B,4H] fp32 (indexed like y): r | z | n | (W_hn h + b_hn) of every step, saved for the
                            backward pass (tp_gru_cell_backward); NULL = not stored                                      */
  const void* w_hh_umma; /* optional (bf16 mode): tp_pack_whh_umma image of the same weight_hh -> the tcgen05 kernel
                            with W_hh resident in TMEM + shared memory takes jobs that provide it; NULL = not provided */
} tp_gru_job;

/* Packs weight_hh [3H,H] fp32 into the bf16 tensor-core fragment order the bf16 recurrence
 * streams (3*H*H bf16 = 6*H*H bytes at dst, 16-byte aligned).  Done once per weight update.  */
TP_API int tp_pack_whh_bf16(const float* w_hh, void* dst, int H, void* stream);
/* Packs weight_hh [3H,H] fp32 (H % 128 == 0) into the per-CTA images k_gru_umma keeps resident: for each of the H/32
 * CTAs of a direction, tile 1 (128 rows: r,z,n of 32 units + r of the next 32) for K < 896 in TMEM row order, its K tail
 * and tile 2 (z,n of the second 32 units) as UMMA 128-byte-swizzle K-major shared-memory images; CTA 2p+k holds the K
 * half k of pair p's 64 units.  tp_whh_umma_bytes(H) = 6 H^2 bytes at dst (16-byte aligned); 0 if H is unsupported. */
TP_API size_t tp_whh_umma_bytes(int H);
TP_API int tp_pack_whh_umma(const float* w_hh, void* dst, int H, void* stream);
/* debug hook: when non-NULL, the bf16 recurrence kernel writes SM-clock stamps
 * [grid][max_steps][8] (int64) into this device buffer; NULL (default) disables it. */
TP_API void tp_gru_set_trace(void* device_buffer);
/* bytes of scratch tp_gru_recurrence needs for (njobs, B, H) */
TP_API size_t tp_gru_workspace_bytes(int njobs, int B, int H);
/* Runs up to 4 independent jobs (directions) concurrently in ONE persistent cooperative
 * kernel that grid-synchronises once per timestep.  `jobs` is a HOST array.  B <= 64.
 * H % 32 == 0.  workspace must be 256-byte aligned.                                        */
TP_API int tp_gru_recurrence(const tp_gru_job* jobs, int njobs, int B, int H, int precision,
                      void* workspace, size_t workspace_bytes, void* stream);
/* Same, with the grid-barrier slot supplied by the caller: `barrier` (128-byte aligned, 1024 bytes = 8 sharded counters
 * on their own cache lines) must be ZERO when the kernel starts -- zeroed by an operation ordered BEFORE the previous kernel in the stream, so that no memset node
 * separates this launch from its programmatic-dependent-launch predecessor (the input-projection GEMM).  NULL = the
 * plain entry point's behaviour (barrier inside the workspace, zeroed by a memset right before the launch).          */
TP_API int tp_gru_recurrence_ex(const tp_gru_job* jobs, int njobs, int B, int H, int precision,
                         void* workspace, size_t workspace_bytes, void* barrier, void* stream);

/* ------------------------------------------------------------------ Regressor (K3)
 * Linear heads of the encoder (lib/models/tepose.py:79-85):
 *   is_train = 0: feat [B,2048]   = (linear_fwd(relu(h_fwd)) + linear_rec(relu(h_rec))) / 2
 *   is_train = 1: feat [B,2,2048] = stack(linear_fwd(..), linear_rec(..))
 * h_fwd [B, ld_hf] is y[-1] of gru_fwd (H wide), h_rec [B, ld_hr] is y_rec[0] (2H wide).
 * precision fp32: w_fwd [2048,H], w_rec [2048,2H] row-major fp32 (nn.Linear layout);
 * precision bf16: the tp_pack_mma_a_bf16 copies of the same matrices.                     */
TP_API size_t tp_encoder_heads_workspace_bytes(int B);
TP_API int tp_encoder_heads(int precision, const void* w_fwd, const float* b_fwd, const void* w_rec, const float* b_rec,
                     const float* h_fwd, int64_t ld_hf, const float* h_rec, int64_t ld_hr,
                     int B, int H, int is_train, float* feat, void* feat_bf16 /* optional bf16 copy, same shape */,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Eval-mode heads as one GEMM over the concatenated state h_cat [B,3H] = [y[-1] | y_rec[0]] with
 * w_cat = [0.5 W_fwd | 0.5 W_rec] ([2048,3H]; fp32 row-major or tp_pack_mma_a_bf16) and
 * b_cat = 0.5 (b_fwd + b_rec): identical to (linear_fwd(relu) + linear_rec(relu)) / 2.            */
TP_API int tp_encoder_heads_cat(int precision, const void* w_cat, const float* b_cat, const float* h_cat, int64_t ld_h,
                         int B, int H, float* feat, void* feat_bf16, void* workspace, size_t workspace_bytes,
                         void* stream);

/* 3-iteration IEF loop (lib/models/spin.py:250-261).  fc1 is split into its feature columns
 * (w1x, iteration-invariant) and its [pose|shape|cam] columns (w1p, zero-padded 157 -> 160);
 * decpose/decshape/deccam are stacked into one [160,1024] matrix.                         */
typedef struct tp_ief_weights { /* matrices: fp32 row-major, or tp_pack_mma_a_bf16 copies (bf16) */
  const void* w1x;   /* [1024, 2048] fc1.weight[:, :2048] */
  const float* b1;   /* [1024] */
  const void* w1p;   /* [1024, 160]  fc1.weight[:, 2048:2205] zero-padded */
  const void* w2;    /* [1024, 1024] */
  const float* b2;   /* [1024] */
  const void* wdec;  /* [160, 1024]  rows: decpose(144) | decshape(10) | deccam(3) | 0(3) */
  const float* bdec; /* [160] */
} tp_ief_weights;

TP_API size_t tp_ief_workspace_bytes(int n_rows);
/* feat [n_rows,2048]; init [init_rows,160] = pose6d(144)|shape(10)|cam(3)|0(3) with
 * init_rows == 1 (broadcast, the init_* buffers) or n_rows; psc [n_rows,160] receives the
 * refined pose6d | shape | cam | pad.                                                      */
TP_API int tp_ief_forward(int precision, const tp_ief_weights* w, const float* feat,
                   const void* feat_bf16 /* optional bf16 copy of feat (bf16 precision) */, int n_rows, const float* init,
                   int init_rows, int n_iter, float* psc, void* workspace, size_t workspace_bytes, void* stream);

/* Eval-mode heads + IEF as ONE persistent kernel (bf16 operands, n_rows <= 32): tp_encoder_heads_cat's GEMM becomes the
 * leading layers of the fused IEF kernel (lib/models/tepose.py:79-85 + lib/models/spin.py:250-261).  w_cat / b_cat as for
 * tp_encoder_heads_cat (packed bf16), h_cat [n_rows, 3H] fp32 (row stride ld_h); workspace: tp_ief_workspace_bytes.   */
TP_API int tp_heads_ief_forward(const void* w_cat, const float* b_cat, const float* h_cat, int64_t ld_h, int H,
                         const tp_ief_weights* w, int n_rows, const float* init, int init_rows, int n_iter, float* psc,
                         void* workspace, size_t workspace_bytes, void* barrier /* as for tp_gru_recurrence_ex, or NULL */,
                         void* stream);


/* ------------------------------------------------------------------ SMPL forward (K4 + K5)
 * Packed, device-resident body-model constants (built once by the host, see
 * tepose_b200/smpl.py:pack_smpl_model).                                                    */
typedef struct tp_smpl_model {
  const float* blend;    /* [218][3][vp]: rows 0..206 posedirs, 207..216 shapedirs, 217 v_template;
                            plane c of row k holds coordinate c of every vertex (padded to vp)  */
  const float* j_template; /* [24,3]     J_regressor . v_template                               */
  const float* j_shapedirs;/* [24,3,10]  J_regressor . shapedirs                                 */
  const int32_t* parents;  /* [24], parents[0] = -1, parents[i] < i                              */
  const int32_t* skin_idx; /* [vp, ks] joint index of each retained skinning weight             */
  const float* skin_w;     /* [vp, ks]                                                           */
  int32_t ks;              /* retained weights per vertex (4 for SMPL; up to 24)                */
  int32_t n_verts;         /* 6890 */
  int32_t vp;              /* n_verts rounded up to a multiple of 128 */
  /* optional tables of the tensor-core blend path (blend_mode 1); NULL disables it:
   * blend_tc    : tp_pack_mma_a_bf16 of the [3*vp, 256] matrix whose row ((v/16)*3 + c)*16 + v%16 holds, for
   *               vertex v / coordinate c: 207 pose-blend columns | S_hi (10) | S_hi (10) | S_lo (10) | 0,
   *               with S_hi = bf16(shapedirs), S_lo = shapedirs - S_hi
   * template_pad: [vp,3] fp32 v_template (zero rows beyond n_verts)                                      */
  const void* blend_tc;
  const float* template_pad;
  /* blend_km (optional): the same [3*vp, 256] bf16 matrix in plain row-major order, row v*3 + c -- the B operand of the
   * tcgen05 GEMM that the large-batch path (>= 1024 bodies) runs per chunk of bodies before skinning.     */
  const void* blend_km;
  /* blend_um (optional): the same bf16 matrix as the A-operand image of the fused tcgen05 blend + skinning kernel of the
   * large-batch path: [vertex tile of 128][plane c 3][K block of 64: 4][row 128][128 B], the eight 16-byte chunks of a row
   * stored at position chunk ^ (row & 7).  NULL: the large-batch path runs the GEMM + skinning pair instead.             */
  const void* blend_um;
  /* skin_um (optional, with blend_um): the skinning weights as the A operand of the skinning MMA of the large-batch path:
   * [vertex tile of 128][row 128][128 B] bf16 with k = joint: W_hi = bf16(w) at k 0..23, W_lo = bf16(w - W_hi) at k 32..55, zeros
   * elsewhere; same chunk swizzle as blend_um.  NULL: the skinning of the large-batch path gathers transforms from shared memory. */
  const void* skin_um;
} tp_smpl_model;

/* A joint regressor folded through the skinning weights and the blend matrix (optional, large-batch path): with
 * G[(r,j),v] = jreg[r,v] w[v,j], sum_v jreg[r,v] verts[v] = sum_j ( R_j q[r,j] + t_j g0[r,j] ), q = coef . M^T + q_bias:
 *   m_km   [nq_pad, 512] bf16 row-major: columns [0, 256) = bf16(M), [256, 512) = bf16(M - bf16(M)) (contracted with the coefficient
 *          row twice); row (r*24 + j)*3 + c, column k in the coefficient order of blend_tc (M = G . blend_km as stored, i.e. from
 *          the bf16 blend matrix)
 *   q_bias [nq_pad] = G . v_template;   g0 [nreg*24] = sum_v G;   nq_pad = nreg*72 rounded up to a multiple of 16.            */
typedef struct tp_smpl_regfold {
  const void* m_km;
  const float* q_bias;
  const float* g0;
  int32_t nreg, nq_pad;
} tp_smpl_regfold;

TP_API size_t tp_smpl_workspace_bytes(const tp_smpl_model* m, int n, int nreg, int blend_mode);
/* smplx.SMPL.forward + lbs (restated third-party code, SURVEY.md App. A.6), the wrapper
 * lib/models/smpl.py:72-84, the optional H36M regression lib/models/spin.py:275-278, the
 * projection spin.py:280 and the theta assembly spin.py:282-285 in three launches:
 * verts never round-trip HBM between stages.
 *   pose      : per pose_kind, row stride ld_pose   betas : [n,10] (row stride ld_betas)
 *   cam       : [n,3] or NULL (then kp2d/theta are not produced)
 *   jreg      : [nreg, vp] dense joint regressor rows (zero padded to vp), nreg <= 32
 *   joint_src : [nj] device array of TP_JSRC_* codes
 * outputs (any may be NULL; verts is required when nj > 0): verts [n,n_verts,3], joints [n,nj,3], kp2d [n,nj,2],
 *   rotmat [n,24,3,3], theta [n,85] = cam | axis-angle(72) | betas(10).                    */
TP_API int tp_smpl_forward(const tp_smpl_model* m, int n, const float* pose, int64_t ld_pose, int pose_kind,
                    const float* betas, int64_t ld_betas, const float* cam, int64_t ld_cam,
                    const float* jreg, int nreg, const int32_t* joint_src, int nj,
                    float* verts, float* joints, float* kp2d, float* rotmat, float* theta,
                    int blend_mode /* 0: fp32 FFMA blend (strict); 1: bf16 tensor-core blend (needs blend_tc) */,
                    void* workspace, size_t workspace_bytes, void* stream);
/* Same with an optional folded form of jreg (NULL = tp_smpl_forward): the large-batch path (>= 1024 bodies, blend_mode 1) then takes
 * the regressed joints from one small GEMM over all bodies instead of a pass over every body's skinned vertices.             */
TP_API int tp_smpl_forward_ex(const tp_smpl_model* m, int n, const float* pose, int64_t ld_pose, int pose_kind,
                       const float* betas, int64_t ld_betas, const float* cam, int64_t ld_cam,
                       const float* jreg, int nreg, const tp_smpl_regfold* fold, const int32_t* joint_src, int nj,
                       float* verts, float* joints, float* kp2d, float* rotmat, float* theta, int blend_mode,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ evaluation metrics (lib/utils/eval_utils.py)
 * All take fp32 device arrays; pelvis0 / pelvis1 select the root alignment applied to BOTH point sets first
 * (evaluate.py:420-428): both >= 0: subtract the mean of the two joints (hips 2, 3 of the 14-joint set);
 * pelvis1 < 0: subtract joint pelvis0 (mpii3d: joint J-3); pelvis0 < 0: none.
 *
 * tp_pose_metrics -- pred / target [n, n_joints, 3].  Any output may be NULL:
 *   aligned  [n, n_joints, 3] = batch_compute_similarity_transform_torch(pred, target)  (eval_utils.py:287-337:
 *            orthogonal Procrustes, R = V diag(1,1,sign det(U V^T)) U^T from the SVD of X1 X2^T, scale, translation)
 *   mpjpe    [n] = mean_j ||pred_j - target_j||                     (evaluate.py:433; lib/core/tester.py:286)
 *   pa_mpjpe [n] = mean_j ||aligned_j - target_j||                  (evaluate.py:435-437; lib/core/tester.py:287-288) */
TP_API int tp_pose_metrics(const float* pred, const float* target, int n, int n_joints, int pelvis0, int pelvis1,
                    float* aligned, float* mpjpe, float* pa_mpjpe, void* stream);
/* tp_accel_error -- pred / target [n_seq, len, n_joints, 3] -> out [n_seq, len-2]:
 *   out[s,i] = mean_j || (p_i - 2 p_{i+1} + p_{i+2}) - (g_i - 2 g_{i+1} + g_{i+2}) ||   (compute_error_accel_eval /
 *   compute_error_accel, eval_utils.py:79-138); target NULL: the norm of pred's own acceleration (compute_accel, :53-76). */
TP_API int tp_accel_error(const float* pred, const float* target, int n_seq, int len, int n_joints, int pelvis0, int pelvis1,
                   float* out, void* stream);
/* tp_vertex_error -- verts_a / verts_b [n, n_verts, 3] -> out [n] = mean_v ||a_v - b_v||   (compute_error_verts,
 * eval_utils.py:141-175; the target mesh comes from tp_smpl_forward with TP_POSE_AXIS_ANGLE).                        */
TP_API int tp_vertex_error(const float* verts_a, const float* verts_b, int n, int n_verts, float* out, void* stream);

/* ------------------------------------------------------------------ training step: backward kernels
 * The reference trains through torch.autograd (lib/core/trainer.py:203,235-237); these are the adjoints of the path's
 * stages.  GEMM-shaped adjoints (dX = dY.W, dW = dY^T.X) run on tp_gemm_f32 / tp_gemm_bf16_tc over operands transposed by
 * tp_transpose_f32.  All arrays fp32 device memory unless noted.                                                         */
/* dst[c][r] = src[r][c] (max(.,0) first when relu) for r < rows, c < cols; dst has dst_rows rows (>= cols, extra rows zero)
 * of ld_dst elements (columns rows..ld_dst-1 zero); dst_precision selects fp32 or bf16 output.                            */
TP_API int tp_transpose_f32(const float* src, int64_t ld_src, int rows, int cols, void* dst, int64_t ld_dst, int dst_rows,
                     int dst_precision, int relu, void* stream);
/* out[c] = beta*out[c] + sum_r A[r][c]  (bias gradients; fixed summation order) */
TP_API int tp_colsum_f32(const float* A, int64_t lda, int rows, int cols, float* out, float beta, void* stream);
/* a *= mask * scale  (nn.Dropout with the mask as an input: forward and backward are the same op; spin.py:216-218,256-258) */
TP_API int tp_mask_scale(float* a, int64_t ld, const float* mask, int64_t ldm, int rows, int cols, float scale, void* stream);
/* g = h > 0 ? g : 0  (F.relu backward, lib/models/tepose.py:79-80) */
TP_API int tp_relu_backward(float* g, int64_t ld, const float* h, int64_t ldh, int rows, int cols, void* stream);
/* dst = alpha*src + beta*dst */
TP_API int tp_axpby_f32(const float* src, int64_t lds, float* dst, int64_t ldd, int rows, int cols, float alpha, float beta, void* stream);
/* One step of back-propagation through time of a torch.nn.GRU direction: g_h [B,H] holds dL/dh_t on entry and
 * dL/dh_t * z_t on exit (add d_gh . W_hh for the full dL/dh_{t-1}); gates = the [B,4H] block tp_gru_recurrence saved for
 * the step; h_prev = h_{t-1} [B,H] or NULL for zeros; d_gi / d_gh [B,3H] = gradients w.r.t. the input-side and
 * hidden-side gate pre-activations (r|z|n).                                                                              */
TP_API int tp_gru_cell_backward(float* g_h, int64_t ldg, const float* gates, int64_t ld_gates, const float* h_prev, int64_t ldh,
                         float* d_gi, int64_t ld_dgi, float* d_gh, int64_t ld_dgh, int B, int H, void* stream);
/* adjoint of rot6d_to_rotmat (lib/utils/geometry.py:330-343): x6 [n,6], g_R [n,9] -> g_x6 [n,6] */
TP_API int tp_rot6d_backward(const float* x6, const float* g_R, float* g_x6, int64_t n, void* stream);
/* adjoint of rotation_matrix_to_angle_axis (lib/utils/geometry.py:68-233): R [n,9]; rotation i takes its gradient from
 * g_aa + (i / per_row) * ld_gaa + 3 * (i % per_row)  (theta rows: per_row = 24, ld_gaa = 85); g_R [n,9] is overwritten or
 * accumulated into.                                                                                                       */
TP_API int tp_rotmat_to_angle_axis_backward(const float* R, const float* g_aa, int64_t ld_gaa, int per_row, float* g_R, int64_t n,
                                     int accumulate, void* stream);
/* Adjoint of tp_smpl_forward with pose_kind = rotation matrices (SMPL lbs + joint selection + projection):
 *   inputs  R [n,24,9], betas, cam (as in the forward), jreg / joint_src (as in the forward), joints [n,nj,3] = the forward's
 *           joint output; gradients g_verts [n,n_verts,3], g_joints [n,nj,3], g_kp2d [n,nj,2], g_R_extra [n,24,9] (any NULL)
 *   outputs g_R [n,24,9] (= LBS + pose-blend + chain terms + g_R_extra), g_betas [n,10], g_cam [n,3] (NULL without cam).
 * Four launches: chain recompute + projection adjoint, skinning adjoint (v_posed recomputed, per-joint sums reduced in a
 * fixed order), one GEMM against the blend table for the pose-feature / shape gradients, kinematic-chain adjoint.       */
TP_API size_t tp_smpl_backward_workspace_bytes(const tp_smpl_model* m, int n);
TP_API int tp_smpl_backward(const tp_smpl_model* m, int n, const float* R, const float* betas, int64_t ld_betas, const float* cam,
                     int64_t ld_cam, const float* jreg, int nreg, const int32_t* joint_src, int nj, const float* joints,
                     const float* g_verts, const float* g_joints, const float* g_kp2d, const float* g_R_extra,
                     float* g_R, float* g_betas, float* g_cam, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ generator loss, data terms (lib/core/loss.py:59-171)
 * Value and gradient of TePoseLoss's data terms in one pass (the reference: ~40 torch ops + autograd):
 *   losses4 = { e_loss_weight * keypoint_loss (loss.py:179-192), e_3d_loss_weight * keypoint_3d_loss (:194-217),
 *               e_pose_loss_weight * MSE of quaternion-Rodrigues rotation matrices, e_shape_loss_weight * MSE of betas (:219-231) }
 *   kp2d [n2,49,2] vs real2d [n2,49,3] (x, y, confidence);  kp3d / real3d [n3,49,3] (rows with 3-D labels; joints 25..38 count);
 *   theta / real_theta [ns,85] (rows with SMPL labels).  weights6 (HOST array) = { e_loss_weight, e_3d_loss_weight,
 *   e_pose_loss_weight, e_shape_loss_weight, openpose_weight, gt_weight }.
 *   g_kp2d / g_kp3d / g_theta: d(sum of the four terms) / d(prediction), same shapes as the predictions.                    */
TP_API size_t tp_tepose_loss_workspace_bytes(int n2, int n3, int ns);
TP_API int tp_tepose_loss(const float* kp2d, const float* real2d, int n2, const float* kp3d, const float* real3d, int n3,
                   const float* theta, const float* real_theta, int ns, const float* weights6,
                   float* losses4, float* g_kp2d, float* g_kp3d, float* g_theta, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TEPOSE_B200_H */
