"""HMR ResNet-50 feature extractor + regressor -- drop-in for lib/models/spin.py:16-204 (`Bottleneck`, `HMR`, `hmr`), SURVEY 8 f-5.

The reference extracts the 2048-d per-frame features TePose consumes with `hmr.feature_extractor(batch.reshape(-1,3,224,224))`
(demo.py:183-198; lib/data_utils/_feature_extractor.py).  Same constructor, attribute names and `state_dict` keys, so the SPIN
checkpoint (`checkpoint['model']`, strict=False as in demo.py:120) loads; the nn.Conv2d / nn.BatchNorm2d members are parameter
containers whose forward is never called.

Compute path (eval mode -- the reference calls `.eval()` before use, demo.py:121): activations NHWC bf16 in HBM; BatchNorm is
folded into the conv weights / bias at pack time (float64); every convolution is a tcgen05 GEMM (`tp_gemm_bf16_tc`) over im2col
rows (1x1 stride-1 convolutions read the activation tensor directly) with ReLU and the shortcut add in the epilogue.  The IEF
loop, SMPL and projection of `HMR.forward` are the Regressor kernels (`tepose_b200.spin.Regressor`).  No CPU / torch fallback.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _native as nv
from .spin import Regressor
from .smpl import SMPL_MEAN_PARAMS


class Bottleneck(nn.Module):
    """Parameter container with the reference's member names (lib/models/spin.py:16-56)."""
    expansion = 4

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, kernel_size=1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, kernel_size=3, stride=stride, padding=1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.conv3 = nn.Conv2d(planes, planes * 4, kernel_size=1, bias=False)
        self.bn3 = nn.BatchNorm2d(planes * 4)
        self.relu = nn.ReLU(inplace=True)
        self.downsample = downsample
        self.stride = stride

    def forward(self, x):
        raise RuntimeError("tepose_b200.hmr.Bottleneck is a parameter container; call HMR.feature_extractor / HMR.forward")


CROP = 224                     # the demo's crop_size (get_single_image_crop_demo), HMR's input size
CROP_FIELDS = 6                # crop-table row: frame, cx, cy, w, h, scale (tp_crop, include/tepose_b200.h)


def make_crop_table(crops, device):
    """[N,6] rows (frame, cx, cy, w, h, scale) -> the table tp_crop_normalize_bf16 reads, on `device`: [N,6] int32 storage, the
    frame index as int32 and the other five fields as float32 bit patterns (the 24-byte tp_crop of include/tepose_b200.h)."""
    t = torch.as_tensor(crops, dtype=torch.float64)
    if t.dim() != 2 or t.shape[1] != CROP_FIELDS or t.shape[0] < 1:
        raise ValueError(f"crops must be [N,{CROP_FIELDS}] rows (frame, cx, cy, w, h, scale), got {tuple(t.shape)}")
    frame = t[:, 0]
    if not t.is_cuda and not torch.equal(frame, frame.round()):          # (a check of device rows would synchronise)
        raise ValueError("crop frame indices must be integers")
    table = torch.empty(t.shape[0], CROP_FIELDS, dtype=torch.int32, device=t.device)
    table[:, 0] = frame.to(torch.int32)
    table[:, 1:] = t[:, 1:].to(torch.float32).view(torch.int32)
    return table.to(device)


def _fold(conv: nn.Conv2d, bn: nn.BatchNorm2d, cin_pad=None):
    """conv (no bias) followed by eval-mode BatchNorm -> ([Cout, KP] bf16 weight matrix in (ky, kx, c) column order, fp32 bias)."""
    w = conv.weight.detach().double()                     # [Cout, Cin, kh, kw]
    scale = bn.weight.detach().double() / torch.sqrt(bn.running_var.detach().double() + bn.eps)
    bias = bn.bias.detach().double() - bn.running_mean.detach().double() * scale
    w = w * scale[:, None, None, None]
    cout, cin, kh, kw = w.shape
    if cin_pad is not None and cin_pad > cin:
        w = torch.cat([w, torch.zeros(cout, cin_pad - cin, kh, kw, dtype=w.dtype, device=w.device)], 1)
        cin = cin_pad
    m = w.permute(0, 2, 3, 1).reshape(cout, kh * kw * cin)
    kp = (m.shape[1] + 63) // 64 * 64
    out = torch.zeros(cout, kp, dtype=torch.float64, device=w.device)
    out[:, :m.shape[1]] = m
    return out.to(torch.bfloat16).contiguous(), bias.float().contiguous()


class HMR(Regressor):
    """SMPL Iterative Regressor with ResNet50 backbone (lib/models/spin.py:59-204)."""

    def __init__(self, block=Bottleneck, layers=(3, 4, 6, 3), smpl_mean_params=SMPL_MEAN_PARAMS, precision="bf16"):
        if precision != "bf16":
            raise ValueError("tepose_b200.HMR runs its convolutions on the bf16 tensor-core GEMM only (precision='bf16')")
        super().__init__(smpl_mean_params, precision=precision)       # fc1, fc2, dec*, smpl, init_* (spin.py:75-105)
        self.inplanes = 64
        self.conv1 = nn.Conv2d(3, 64, kernel_size=7, stride=2, padding=3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        self.relu = nn.ReLU(inplace=True)
        self.maxpool = nn.MaxPool2d(kernel_size=3, stride=2, padding=1)
        self.layer1 = self._make_layer(block, 64, layers[0])
        self.layer2 = self._make_layer(block, 128, layers[1], stride=2)
        self.layer3 = self._make_layer(block, 256, layers[2], stride=2)
        self.layer4 = self._make_layer(block, 512, layers[3], stride=2)
        self.avgpool = nn.AvgPool2d(7, stride=1)
        import math
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                n = m.kernel_size[0] * m.kernel_size[1] * m.out_channels
                m.weight.data.normal_(0, math.sqrt(2. / n))
            elif isinstance(m, nn.BatchNorm2d):
                m.weight.data.fill_(1)
                m.bias.data.zero_()
        self._cpack = None
        self._cpack_key = None

    def _make_layer(self, block, planes, blocks, stride=1):
        downsample = None
        if stride != 1 or self.inplanes != planes * block.expansion:
            downsample = nn.Sequential(
                nn.Conv2d(self.inplanes, planes * block.expansion, kernel_size=1, stride=stride, bias=False),
                nn.BatchNorm2d(planes * block.expansion))
        layers = [block(self.inplanes, planes, stride, downsample)]
        self.inplanes = planes * block.expansion
        for _ in range(1, blocks):
            layers.append(block(self.inplanes, planes))
        return nn.Sequential(*layers)

    # ------------------------------------------------------------------ packing
    def _conv_key(self):
        ts = []
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                ts.append(m.weight)
            elif isinstance(m, nn.BatchNorm2d):
                ts += [m.weight, m.bias, m.running_mean, m.running_var]
        return tuple((t.device, t.data_ptr(), t._version) for t in ts)

    def conv_packed(self):
        key = self._conv_key()
        if self._cpack is None or self._cpack_key != key:
            nv.require_cuda(self.conv1.weight, "HMR parameters (call .cuda() first)")
            pk = {"stem": _fold(self.conv1, self.bn1, cin_pad=4), "blocks": []}
            for layer in (self.layer1, self.layer2, self.layer3, self.layer4):
                for b in layer:
                    e = {"c1": _fold(b.conv1, b.bn1), "c2": _fold(b.conv2, b.bn2), "c3": _fold(b.conv3, b.bn3), "stride": b.stride,
                         "planes": b.conv1.out_channels, "down": None}
                    if b.downsample is not None:
                        e["down"] = _fold(b.downsample[0], b.downsample[1])
                    pk["blocks"].append(e)
            self._cpack, self._cpack_key = pk, key
        return self._cpack

    # ------------------------------------------------------------------ forward
    @staticmethod
    def _gemm(a, rows, wb, out, relu, residual=None):
        """out[rows, Cout] (bf16) = act(a[rows, KP] . W^T + bias (+ residual))"""
        w, bias = wb
        cout, kp = w.shape
        assert a.shape[1] == kp and a.is_contiguous(), (a.shape, kp)
        seg = (nv.GemmSeg * 1)()
        seg[0] = nv.GemmSeg(0, rows, 0, cout, nv.ptr(out), cout, nv.ptr(bias),
                            (nv.GEMM_RELU if relu else 0) | nv.GEMM_OUT_BF16, cout if residual is not None else 0,
                            nv.ptr(residual) if residual is not None else None)
        nv.check(nv.lib().tp_gemm_bf16_tc(nv.ptr(a), rows, nv.ptr(w), cout, kp, seg, 1, nv.stream()), "tp_gemm_bf16_tc")

    @nv.device_guard
    def feature_extractor(self, x):
        """x [N,3,224,224] fp32 (any H, W whose final map the 7x7 average pool covers) -> [N,2048] fp32 (spin.py:127-141)."""
        if self.training:
            raise NotImplementedError("tepose_b200.HMR implements the eval-mode feature extractor (BatchNorm folded); call .eval()")
        nv.require_cuda(x, "x")
        x = x.detach().contiguous().float()
        N, C, H, W = x.shape
        if C != 3:
            raise ValueError(f"HMR.feature_extractor expects [N,3,H,W] input, got {tuple(x.shape)}")
        x4 = torch.empty(N, H, W, 4, device=x.device, dtype=torch.bfloat16)
        nv.check(nv.lib().tp_nchw_to_nhwc_bf16(nv.ptr(x), nv.ptr(x4), N, 3, H, W, 4, nv.stream()), "tp_nchw_to_nhwc_bf16")
        return self.features_nhwc4(x4)

    @nv.device_guard
    def features_nhwc4(self, x4):
        """x4 [N,H,W,4] bf16 NHWC, channel 3 zero (RGB normalised as feature_extractor's input) -> [N,2048] fp32: everything of
        feature_extractor from the stem's im2col to the average pool."""
        if self.training:
            raise NotImplementedError("tepose_b200.HMR implements the eval-mode feature extractor (BatchNorm folded); call .eval()")
        nv.require_cuda(x4, "x4")
        if x4.dim() != 4 or x4.shape[3] != 4 or x4.dtype != torch.bfloat16:
            raise ValueError(f"HMR.features_nhwc4 expects [N,H,W,4] bf16 input, got {tuple(x4.shape)} {x4.dtype}")
        pk = self.conv_packed()
        L = nv.lib()
        dev = x4.device
        N, H, W, _ = x4.shape
        bf = lambda *s: torch.empty(*s, device=dev, dtype=torch.bfloat16)
        st = nv.stream()
        # stem: 7x7 stride-2 conv (+BN+ReLU) as im2col over RGB0 pixels, then 3x3 stride-2 max pool
        Ho, Wo = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
        kp = pk["stem"][0].shape[1]
        cols = bf(N * Ho * Wo, kp)
        nv.check(L.tp_im2col_nhwc_bf16(nv.ptr(x4), nv.ptr(cols), N, H, W, 4, 7, 7, 2, 3, kp, st), "tp_im2col_nhwc_bf16")
        y = bf(N * Ho * Wo, 64)
        self._gemm(cols, N * Ho * Wo, pk["stem"], y, relu=True)
        H, W = Ho, Wo
        Ho, Wo = (H + 2 - 3) // 2 + 1, (W + 2 - 3) // 2 + 1
        cur = bf(N * Ho * Wo, 64)
        nv.check(L.tp_maxpool3x3s2_nhwc_bf16(nv.ptr(y), nv.ptr(cur), N, H, W, 64, st), "tp_maxpool3x3s2_nhwc_bf16")
        H, W, Cin = Ho, Wo, 64
        nv.mark("hmr_stem")
        for e in pk["blocks"]:
            planes, s = e["planes"], e["stride"]
            rows = N * H * W
            t1 = bf(rows, planes)
            self._gemm(cur, rows, e["c1"], t1, relu=True)                         # 1x1
            Ho, Wo = (H + 2 - 3) // s + 1, (W + 2 - 3) // s + 1
            rows_o = N * Ho * Wo
            cols = bf(rows_o, 9 * planes)
            nv.check(L.tp_im2col_nhwc_bf16(nv.ptr(t1), nv.ptr(cols), N, H, W, planes, 3, 3, s, 1, 9 * planes, st), "tp_im2col_nhwc_bf16")
            t2 = bf(rows_o, planes)
            self._gemm(cols, rows_o, e["c2"], t2, relu=True)                      # 3x3 (stride s)
            if e["down"] is not None:
                if s == 1:
                    src = cur
                else:                                                              # 1x1 stride-s shortcut: gather the strided pixels
                    src = bf(rows_o, Cin)
                    nv.check(L.tp_im2col_nhwc_bf16(nv.ptr(cur), nv.ptr(src), N, H, W, Cin, 1, 1, s, 0, Cin, st), "tp_im2col_nhwc_bf16")
                res = bf(rows_o, planes * 4)
                self._gemm(src, rows_o, e["down"], res, relu=False)
            else:
                res = cur
            out = bf(rows_o, planes * 4)
            self._gemm(t2, rows_o, e["c3"], out, relu=True, residual=res)         # 1x1 + shortcut + ReLU
            cur, H, W, Cin = out, Ho, Wo, planes * 4
        nv.mark("hmr_blocks")
        if H != 7 or W != 7:
            raise ValueError(f"HMR.feature_extractor: the final feature map is {H}x{W}; nn.AvgPool2d(7) + view(N, -1) of the reference "
                             "yields 2048 features for 224x224 inputs only")
        xf = torch.empty(N, Cin, device=dev, dtype=torch.float32)
        nv.check(L.tp_avgpool_nhwc_bf16(nv.ptr(cur), nv.ptr(xf), N, H * W, Cin, st), "tp_avgpool_nhwc_bf16")
        nv.mark("hmr_pool")
        return xf

    @nv.device_guard
    def features_from_frames(self, frames, crops):
        """frames uint8 [F,H,W,3] RGB (CUDA), crops: the crop table (make_crop_table) -> [N,2048] fp32.  The device version of the
        demo's crop + feature extraction (demo.py:183-198, lib/data_utils/_img_utils.py: get_single_image_crop_demo): each box is
        cropped to 224x224 and normalised by tp_crop_normalize_bf16, bit-identical to the reference's cv2 / torchvision crop
        rounded to bf16, then runs features_nhwc4."""
        nv.require_cuda(frames, "frames")
        if frames.dim() != 4 or frames.shape[3] != 3 or frames.dtype != torch.uint8:
            raise ValueError(f"HMR.features_from_frames expects uint8 [F,H,W,3] frames, got {tuple(frames.shape)} {frames.dtype}")
        crops = make_crop_table(crops, frames.device)
        frames = frames.contiguous()
        F, H, W, _ = frames.shape
        N = crops.shape[0]
        x4 = torch.empty(N, CROP, CROP, 4, device=frames.device, dtype=torch.bfloat16)
        nv.check(nv.lib().tp_crop_normalize_bf16(nv.ptr(frames), F, H, W, nv.ptr(crops), N, nv.ptr(x4), nv.stream()),
                 "tp_crop_normalize_bf16")
        return self.features_nhwc4(x4)

    @nv.device_guard
    def forward(self, x, init_pose=None, init_shape=None, init_cam=None, n_iter=3, return_features=False):
        xf = self.feature_extractor(x)
        out = Regressor.forward(self, xf, init_pose=init_pose, init_shape=init_shape, init_cam=init_cam, n_iter=n_iter)
        output = [{k: out[0][k] for k in ("theta", "verts", "kp_2d", "kp_3d")}]      # (the reference's HMR returns no 'rotmat')
        if return_features:
            return xf, output
        return output


def hmr(smpl_mean_params=SMPL_MEAN_PARAMS, pretrained=True, **kwargs):
    """lib/models/spin.py:294-305.  `pretrained=True` loads torchvision's ImageNet ResNet-50 weights in the reference (a download);
    here the caller loads the SPIN checkpoint afterwards as demo.py:118-120 does, so the flag is accepted and ignored."""
    return HMR(Bottleneck, [3, 4, 6, 3], smpl_mean_params, **kwargs)
