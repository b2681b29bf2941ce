"""CPU: oracle/crop_ref.py restates the reference demo's crop (gen_trans_from_patch_cv + cv2.warpAffine + ToTensor + Normalize)
bit for bit.  The device kernel tp_crop_normalize_bf16 is pinned against this restatement (tests/test_video.py), so the GPU
machine needs no OpenCV."""
import numpy as np
import pytest
import torch

from oracle import crop_ref

cv2 = pytest.importorskip("cv2")

SIZES = [(97, 131), (1080, 1920), (224, 224)]


def _frames(H, W, F=2):
    return crop_ref.sample_frames(H * 7 + W, F, H, W)


def _reference_crop(frame, cx, cy, w, h, scale, size=224):
    """generate_patch_image_cv of the reference (lib/data_utils/_img_utils.py) with cv2 doing the arithmetic."""
    src, dst = crop_ref.patch_points(cx, cy, w, h, scale, size)
    trans = cv2.getAffineTransform(np.float32(src), np.float32(dst))
    return cv2.warpAffine(frame, trans, (size, size), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT), trans


def test_patch_points_follow_gen_trans_from_patch_cv():
    """The reference builds the points from python floats / float64 arrays and stores them as float32."""
    cx, cy, w, h, s = 100.37, 50.81, 80.0, 120.0, 1.2
    src_w, src_h = w * s, h * s
    centre = np.zeros(2); centre[0], centre[1] = cx, cy
    down = np.array([0, src_h * 0.5], dtype=np.float32)
    right = np.array([src_w * 0.5, 0], dtype=np.float32)
    want = np.zeros((3, 2), np.float32)
    want[0, :], want[1, :], want[2, :] = centre, centre + down, centre + right
    src, dst = crop_ref.patch_points(cx, cy, w, h, s)
    assert np.array_equal(src, want)
    assert np.array_equal(dst, np.float32([[112, 112], [112, 224], [224, 112]]))


@pytest.mark.parametrize("H,W", SIZES)
def test_solve_affine_equals_getAffineTransform(H, W):
    for _, cx, cy, w, h, s in crop_ref.sample_boxes(3, 1, H, W):
        src, dst = crop_ref.patch_points(cx, cy, w, h, s)
        assert np.array_equal(crop_ref.solve_affine(src, dst), cv2.getAffineTransform(src, dst)), (cx, cy, w, h, s)


def test_solve_affine_random_systems():
    """Arbitrary (non-axis-aligned) triangles exercise every pivot order of the 6x6 elimination."""
    rs = np.random.RandomState(11)
    for _ in range(500):
        src = rs.uniform(-500, 2500, (3, 2)).astype(np.float32)
        dst = rs.uniform(-10, 300, (3, 2)).astype(np.float32)
        assert np.array_equal(crop_ref.solve_affine(src, dst), cv2.getAffineTransform(src, dst)), (src, dst)


@pytest.mark.parametrize("H,W", SIZES)
def test_warp_on_the_inverse_map_equals_cv2(H, W):
    frames = _frames(H, W)
    for f, cx, cy, w, h, s in crop_ref.sample_boxes(5, 2, H, W):
        iM = crop_ref.crop_transform(cx, cy, w, h, s)
        want = cv2.warpAffine(frames[f], iM, (224, 224), flags=cv2.INTER_LINEAR | cv2.WARP_INVERSE_MAP,
                              borderMode=cv2.BORDER_CONSTANT)
        got = crop_ref.warp_linear(frames[f], iM)
        assert np.array_equal(got, want), ((cx, cy, w, h, s), int((got != want).sum()))


@pytest.mark.parametrize("H,W", SIZES)
def test_crop_equals_the_reference_getAffineTransform_path(H, W):
    frames = _frames(H, W)
    boxes = crop_ref.sample_boxes(7, 2, H, W)
    outside = 0
    for f, cx, cy, w, h, s in boxes:
        want, trans = _reference_crop(frames[f], cx, cy, w, h, s)
        assert np.array_equal(crop_ref.solve_affine(*crop_ref.patch_points(cx, cy, w, h, s)), trans)
        got = crop_ref.crop(frames[f], cx, cy, w, h, s)
        assert np.array_equal(got, want), ((cx, cy, w, h, s), int((got != want).sum()))
        outside += int(not want.any())
    assert outside >= 1                       # the fully-outside box is all zeros, not skipped


def test_random_affine_warps_equal_cv2():
    """General inverse maps (shear, rotation, mirror) on an odd-sized frame, including subpixel ties."""
    rs = np.random.RandomState(5)
    img = _frames(97, 131, 1)[0]
    for t in range(60):
        iM = np.array([[rs.uniform(-2, 2), rs.uniform(-0.5, 0.5), rs.uniform(-60, 160)],
                       [rs.uniform(-0.5, 0.5), rs.uniform(-2, 2), rs.uniform(-60, 120)]])
        if t % 4 == 0:
            iM = np.round(iM * 64) / 64               # exact multiples of 1/64: positions on rounding ties
        want = cv2.warpAffine(img, iM, (224, 224), flags=cv2.INTER_LINEAR | cv2.WARP_INVERSE_MAP, borderMode=cv2.BORDER_CONSTANT)
        assert np.array_equal(crop_ref.warp_linear(img, iM), want), t


def test_normalize_bf16_equals_torchvision():
    tvt = pytest.importorskip("torchvision.transforms")
    rs = np.random.RandomState(1)
    patch = rs.randint(0, 256, (224, 224, 3)).astype(np.uint8)
    patch.reshape(-1, 3)[:256] = np.arange(256)[:, None]          # every byte value in every channel
    ref = tvt.Compose([tvt.ToTensor(), tvt.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])(patch)
    got = torch.from_numpy(crop_ref.normalize(patch)).permute(2, 0, 1)
    assert torch.equal(got.view(torch.int32), ref.view(torch.int32))
    assert torch.equal(got.bfloat16().view(torch.int16), ref.bfloat16().view(torch.int16))


def test_crops_nhwc4_layout():
    frames = _frames(97, 131)
    table = crop_ref.sample_boxes(9, 2, 97, 131)[:3]
    out = crop_ref.crops_nhwc4_bf16(frames, table)
    assert out.shape == (3, 224, 224, 4) and out.dtype == torch.bfloat16
    assert torch.equal(out[..., 3].view(torch.int16), torch.zeros(3, 224, 224, dtype=torch.int16))
    f, cx, cy, w, h, s = table[1]
    want = torch.from_numpy(crop_ref.normalize(crop_ref.crop(frames[f], cx, cy, w, h, s))).bfloat16()
    assert torch.equal(out[1, ..., :3].view(torch.int16), want.view(torch.int16))
