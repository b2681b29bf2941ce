"""NumPy restatement of the reference's person crop -- TEST INFRASTRUCTURE (tests/ and scripts/ import it; the product never does).

The reference's demo crops each tracked box on the host (lib/data_utils/_img_utils.py: get_single_image_crop_demo ->
generate_patch_image_cv -> gen_trans_from_patch_cv with rot = 0 and no flip, then cv2.warpAffine(INTER_LINEAR, BORDER_CONSTANT),
then torchvision ToTensor + Normalize(ImageNet mean / std)).  This module states that arithmetic exactly, so that the device
kernel (tp_crop_normalize_bf16) can be pinned against it bit for bit on a machine without OpenCV:

- patch_points: the three source / destination points of gen_trans_from_patch_cv, including their float32 rounding;
- solve_affine: cv2.getAffineTransform, i.e. the 6x6 system solved by cv::solve(DECOMP_LU) (Gaussian elimination with
  partial pivoting, back substitution by division, every operation a separately rounded double);
- invert_affine: the inversion cv2.warpAffine applies when WARP_INVERSE_MAP is not set;
- warp_linear: cv2.warpAffine's uint8 INTER_LINEAR on the inverse map: source positions in 1/32 pixel from 1/1024-pixel fixed
  point, bilinear weights (32 - f) * (32 - g) * 32 out of 2^15, rounding (sum + 2^14) >> 15; taps outside the frame read 0;
- normalize: ((v / 255) - mean[c]) / std[c] in float32, the order ToTensor + Normalize use.

tests/test_crop_ref.py checks each piece against cv2 and torchvision.  Valid for boxes whose sampled source positions stay within
2^20 pixels of the origin (cv2's 1/1024-pixel positions are int32).
"""
import numpy as np

SIZE = 224
MEAN = np.array([0.485, 0.456, 0.406], np.float32)       # lib/data_utils/_img_utils.py: convert_cvimg_to_tensor
STD = np.array([0.229, 0.224, 0.225], np.float32)
LU_EPS = np.finfo(np.float64).eps * 100                   # cv::LU64f: a pivot below this means a singular system


def patch_points(cx, cy, w, h, scale, size=SIZE):
    """gen_trans_from_patch_cv(cx, cy, w, h, size, size, scale, rot=0): (src, dst) float32 [3, 2] (centre, centre + down
    half-extent, centre + right half-extent).  The half extents are rounded to float32 first, the sums in double after."""
    cx, cy, w, h, scale = (float(v) for v in (cx, cy, w, h, scale))
    hh = np.float32(h * scale * 0.5)
    hw = np.float32(w * scale * 0.5)
    src = np.array([[cx, cy], [cx, cy + float(hh)], [cx + float(hw), cy]], np.float32)
    d = size * 0.5
    dst = np.array([[d, d], [d, d + d], [d + d, d]], np.float32)
    return src, dst


def solve_affine(src, dst):
    """cv2.getAffineTransform(src, dst) -> [2, 3] float64."""
    a = [[0.0] * 6 for _ in range(6)]
    b = [0.0] * 6
    for i in range(3):
        x, y = float(src[i][0]), float(src[i][1])
        a[2 * i][0:3] = [x, y, 1.0]
        a[2 * i + 1][3:6] = [x, y, 1.0]
        b[2 * i], b[2 * i + 1] = float(dst[i][0]), float(dst[i][1])
    m = 6
    for i in range(m):
        k = i
        for j in range(i + 1, m):
            if abs(a[j][i]) > abs(a[k][i]):
                k = j
        if abs(a[k][i]) < LU_EPS:
            return np.zeros((2, 3))                       # cv::solve reports failure and leaves a zero matrix
        if k != i:
            a[i], a[k] = a[k], a[i]
            b[i], b[k] = b[k], b[i]
        d = -1.0 / a[i][i]
        for j in range(i + 1, m):
            alpha = a[j][i] * d
            for c in range(i + 1, m):
                a[j][c] += alpha * a[i][c]
            b[j] += alpha * b[i]
    for i in range(m - 1, -1, -1):
        s = b[i]
        for c in range(i + 1, m):
            s -= a[i][c] * b[c]
        b[i] = s / a[i][i]
    return np.array(b).reshape(2, 3)


def invert_affine(M):
    """The inverse map cv2.warpAffine samples with when WARP_INVERSE_MAP is not set (imgwarp.cpp)."""
    m = [float(v) for v in np.asarray(M, np.float64).reshape(-1)]
    D = m[0] * m[4] - m[1] * m[3]
    D = 1.0 / D if D != 0 else 0.0
    a11, a22 = m[4] * D, m[0] * D
    a12, a21 = m[1] * -D, m[3] * -D
    b1 = -a11 * m[2] - a12 * m[5]
    b2 = -a21 * m[2] - a22 * m[5]
    return np.array([[a11, a12, b1], [a21, a22, b2]])


def crop_transform(cx, cy, w, h, scale, size=SIZE):
    """The inverse map (destination pixel -> source position) of one crop."""
    return invert_affine(solve_affine(*patch_points(cx, cy, w, h, scale, size)))


def warp_linear(img, iM, size=SIZE):
    """cv2.warpAffine(img, iM, (size, size), INTER_LINEAR | WARP_INVERSE_MAP, BORDER_CONSTANT 0): img uint8 [H, W, C]."""
    H, W = img.shape[:2]
    m = [float(v) for v in np.asarray(iM, np.float64).reshape(-1)]
    t = np.arange(size, dtype=np.float64)
    adelta = np.rint(m[0] * t * 1024).astype(np.int64)
    bdelta = np.rint(m[3] * t * 1024).astype(np.int64)
    X0 = np.rint((m[1] * t + m[2]) * 1024).astype(np.int64) + 16       # + half a 1/32 step: round to the nearest 1/32
    Y0 = np.rint((m[4] * t + m[5]) * 1024).astype(np.int64) + 16
    X = (X0[:, None] + adelta[None, :]) >> 5
    Y = (Y0[:, None] + bdelta[None, :]) >> 5
    sx, sy = np.clip(X >> 5, -32768, 32767), np.clip(Y >> 5, -32768, 32767)
    fx, fy = X & 31, Y & 31
    acc = np.zeros((size, size, img.shape[2]), np.int64)
    for dy, wy in ((0, 32 - fy), (1, fy)):
        for dx, wx in ((0, 32 - fx), (1, fx)):
            yy, xx = sy + dy, sx + dx
            inside = (yy >= 0) & (yy < H) & (xx >= 0) & (xx < W)
            v = img[np.clip(yy, 0, H - 1), np.clip(xx, 0, W - 1)].astype(np.int64) * inside[..., None]
            acc += v * (wy * wx * 32)[..., None]
    return np.clip((acc + (1 << 14)) >> 15, 0, 255).astype(np.uint8)


def crop(frame, cx, cy, w, h, scale, size=SIZE):
    """generate_patch_image_cv(frame, cx, cy, w, h, size, size, do_flip=False, scale, rot=0)[0]: uint8 [size, size, 3]."""
    return warp_linear(frame, crop_transform(cx, cy, w, h, scale, size), size)


def normalize(patch):
    """uint8 [..., 3] -> float32 [..., 3]: ToTensor (/255) then Normalize(MEAN, STD), channels last."""
    v = patch.astype(np.float32) / np.float32(255)
    return (v - MEAN) / STD


def sample_frames(seed, F, H, W):
    """uint8 [F, H, W, 3] RGB frames: smooth gradients plus noise, so that every bilinear tap matters."""
    rs = np.random.RandomState(seed)
    yy, xx = np.meshgrid(np.linspace(0, 1, H), np.linspace(0, 1, W), indexing="ij")
    out = []
    for _ in range(F):
        a, b, c = rs.uniform(0.5, 4, 3)
        base = np.stack([np.sin(a * 6 * xx) * 90, np.cos(b * 5 * yy) * 90, (xx - yy) * c * 40], -1) + 128
        out.append(np.clip(base + rs.normal(0, 25, (H, W, 3)), 0, 255))
    return np.stack(out).astype(np.uint8)


def sample_boxes(seed, F, H, W):
    """Crop-table rows (frame, cx, cy, w, h, scale), float32 values: boxes fully inside, partly outside and fully outside the
    frame, smaller than the patch (upsampling) and several times larger (downsampling), integer and non-integer centres,
    scale 1 and 1.2 (the demo's) and others, square and elongated."""
    rs = np.random.RandomState(seed)
    s = min(H, W)
    rows = [
        (0, W / 2, H / 2, s / 2, s / 2, 1.0),                          # inside, integer-ish centre
        (0, W / 2 + 0.37, H / 3 + 0.81, s * 0.3, s * 0.45, 1.2),       # inside, non-integer centre, demo scale
        (0, 3.25, 5.5, s * 0.6, s * 0.8, 1.1),                         # partly outside (top-left)
        (0, W - 2.0, H - 7.75, s * 0.7, s * 0.5, 1.3),                 # partly outside (bottom-right)
        (0, -3.0 * W, 2.5 * H, s * 0.4, s * 0.4, 1.0),                 # fully outside
        (0, W * 0.4 + 0.5, H * 0.6 + 0.25, 37.0, 53.0, 1.2),           # much smaller than 224: upsampling
        (0, W * 0.5, H * 0.5, 3.1 * s, 2.3 * s, 0.9),                  # much larger than the frame: downsampling
        (0, W * 0.7 + 0.123, H * 0.4 + 0.456, 11.0, 11.0, 2.5),        # tiny box, large scale
        (0, W * 0.3, H * 0.3, 0.0, s * 0.5, 1.0),                      # zero width: singular system, zero matrix in cv2
    ]
    while len(rows) < 32:
        rows.append((rs.randint(F), rs.uniform(-0.2, 1.2) * W, rs.uniform(-0.2, 1.2) * H, rs.uniform(0.05, 1.5) * s,
                     rs.uniform(0.05, 1.5) * s, rs.choice([1.0, 1.2, rs.uniform(0.7, 1.6)])))
    rows = [(f % F,) + tuple(float(np.float32(v)) for v in r) for f, *r in rows]
    return rows


def crops_nhwc4_bf16(frames, table, size=SIZE):
    """What tp_crop_normalize_bf16 writes: frames uint8 [F, H, W, 3], table rows (frame, cx, cy, w, h, scale) ->
    torch.bfloat16 [N, size, size, 4] with channel 3 zero."""
    import torch
    out = torch.zeros(len(table), size, size, 4, dtype=torch.bfloat16)
    for i, (f, cx, cy, w, h, s) in enumerate(table):
        out[i, ..., :3] = torch.from_numpy(normalize(crop(frames[int(f)], cx, cy, w, h, s, size))).to(torch.bfloat16)
    return out
