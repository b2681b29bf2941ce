"""TePose with the reference's module API (lib/models/tepose.py:44-147) on sm_100a kernels.

  TemporalEncoder(n_layers=1, seq_len=16, hidden_size=2048)
  TePose(seqlen, batch_size=64, n_layers=1, hidden_size=2048, pretrained=..., precision='fp32')
  TePose.forward(input [B,T,2133], is_train=False, J_regressor=None) -> [ {theta, verts, kp_2d, kp_3d, rotmat} ]

The nn.GRU / nn.Linear members are PARAMETER CONTAINERS only (same state_dict keys and
default init as the reference, SURVEY.md App. A.1); their forward is never called.  The
arithmetic is: K1 input-projection GEMM (tcgen05 in bf16 mode, FFMA in fp32 mode), K2
persistent GRU recurrence, K3 linear heads + IEF, K4/K5 fused SMPL.

Encoder schedule (SURVEY.md F2/F3): with x_rec = flip(x), gru_rec's backward direction runs
over x in ORIGINAL order and only its final state is consumed; its forward direction is
consumed only at x_rec index 0 -- one step from h0 = 0 for the last layer.
"""
from __future__ import annotations

import os
import os.path as osp

import torch
import torch.nn as nn

from . import _native as nv
from .smpl import BASE_DATA_DIR
from .spin import Regressor

INPUT_SIZE = 2133


def _round_up(v, m):
    return (v + m - 1) // m * m


class GruKernels:
    """K1 / K2 launch helpers shared by the encoders (needs self.precision and self.hidden_size)."""

    @staticmethod
    def _pack_whh(w: torch.Tensor, lp: bool) -> torch.Tensor:
        """fp32 mode: [3H,H] fp32 as is.  bf16 mode: tensor-core fragment order (tp_pack_whh_bf16)."""
        w = w.contiguous()
        if not lp:
            return w
        out = torch.empty(w.shape[0], w.shape[1], device=w.device, dtype=torch.bfloat16)
        nv.check(nv.lib().tp_pack_whh_bf16(nv.ptr(w), nv.ptr(out), w.shape[1], nv.stream()), "tp_pack_whh_bf16")
        return out

    def uses_umma(self, batch: int) -> bool:
        """Whether tp_gru_recurrence takes the tcgen05 resident-weight kernel (k_gru_umma) for this model's two full directions at
        this batch: the host-side mirror of the dispatch conditions in csrc/gru.cu (for reporting; the library decides)."""
        import os
        H = self.hidden_size
        return (self.precision == "bf16" and H % 128 == 0 and batch <= 32 and 2 * (H // 32) <= 148
                and "TP_GRU_NO_UMMA" not in os.environ and self.n_layers == 1)

    @staticmethod
    def _pack_whh_umma(w: torch.Tensor, lp: bool):
        """bf16 mode, H % 128 == 0: the per-CTA images the tcgen05 recurrence keeps resident in TMEM + shared memory
        (tp_pack_whh_umma); None otherwise (the streaming kernels take the job)."""
        H = w.shape[1]
        nbytes = nv.lib().tp_whh_umma_bytes(H) if lp else 0
        if nbytes == 0:
            return None
        w = w.contiguous()
        out = torch.empty(nbytes, device=w.device, dtype=torch.uint8)
        nv.check(nv.lib().tp_pack_whh_umma(nv.ptr(w), nv.ptr(out), H, nv.stream()), "tp_pack_whh_umma")
        return out

    def _input_proj(self, A, a_rows, W, kp, bias, segs, outs):
        """K1: outs[i] = A[m-range] . W[n-range]^T + bias[n-range]."""
        L = nv.lib()
        if self.precision == "bf16" or A.dtype == torch.bfloat16:      # bf16 mode, or the [hi | lo | hi] operands of fp32_tc
            arr = (nv.GemmSeg * len(segs))()
            for i, ((m0, mr, n0, nc), out) in enumerate(zip(segs, outs)):
                arr[i] = nv.GemmSeg(m0, mr, n0, nc, nv.ptr(out), out.shape[1], nv.vp(bias.data_ptr() + 4 * n0))
            nv.check(L.tp_gemm_bf16_tc(nv.ptr(A), a_rows, nv.ptr(W), W.shape[0], kp, arr, len(segs), nv.stream()),
                     "tp_gemm_bf16_tc")
        else:
            for (m0, mr, n0, nc), out in zip(segs, outs):
                nv.check(L.tp_gemm_f32(nv.vp(A.data_ptr() + 4 * m0 * kp), kp, nv.vp(W.data_ptr() + 4 * n0 * kp), kp,
                                       nv.vp(bias.data_ptr() + 4 * n0), nv.vp(0), 0, nv.ptr(out), out.shape[1],
                                       mr, nc, kp, 1.0, 0.0, 0, nv.stream()), "tp_gemm_f32")

    def _recurrence(self, jobs, B, barrier=None, precision=None):
        """barrier: a zeroed 1 KB slot (cleared by the pack kernel at the top of the step) -> no memset node between this
        launch and the GEMM before it, so the two stay linked by programmatic dependent launch."""
        L = nv.lib()
        H = self.hidden_size
        arr = (nv.GruJob * len(jobs))(*jobs)
        ws = nv.workspace(L.tp_gru_workspace_bytes(len(jobs), B, H), jobs[0]._dev)
        nv.check(L.tp_gru_recurrence_ex(arr, len(jobs), B, H, nv.PRECISIONS[self.precision] if precision is None else precision, nv.ptr(ws), ws.numel(),
                                        nv.vp(0 if barrier is None else barrier.data_ptr()), nv.stream()), "tp_gru_recurrence")


    @staticmethod
    def _job(dev, gi, col0, w_hh, b_hh, steps, t_in0, t_in_step, h0=None, y=None, ycol=0, y_lp=None,
             t_out0=0, t_out_step=1, h_final=None, hcol=0, w_umma=None, gates=None):
        j = nv.GruJob()
        j.w_hh_umma = 0 if w_umma is None else w_umma.data_ptr()
        j.gates = 0 if gates is None else gates.data_ptr()
        j.gi = gi.data_ptr() + 4 * col0
        j.ldg = gi.shape[-1]
        j.w_hh = w_hh.data_ptr()
        j.b_hh = b_hh.data_ptr()
        j.h0 = 0 if h0 is None else h0.data_ptr()
        j.y = 0 if y is None else y.data_ptr() + 4 * ycol
        j.ldy = 0 if y is None else y.shape[-1]
        j.y_lp = 0 if y_lp is None else y_lp.data_ptr() + 2 * ycol
        j.ldy_lp = 0 if y_lp is None else y_lp.shape[-1]
        j.h_final = 0 if h_final is None else h_final.data_ptr() + 4 * hcol
        j.ld_hf = 0 if h_final is None else h_final.stride(0)
        j.steps, j.t_in0, j.t_in_step, j.t_out0, j.t_out_step = steps, t_in0, t_in_step, t_out0, t_out_step
        j._dev = dev
        return j


class TemporalEncoder(nn.Module, GruKernels):
    def __init__(self, n_layers=1, seq_len=16, hidden_size=2048, precision="fp32"):
        super().__init__()
        self.gru_fwd = nn.GRU(input_size=INPUT_SIZE, hidden_size=hidden_size, bidirectional=False, num_layers=n_layers)
        self.gru_rec = nn.GRU(input_size=INPUT_SIZE, hidden_size=hidden_size, bidirectional=True, num_layers=n_layers)
        self.mid_frame = int(seq_len / 2)
        self.hidden_size = hidden_size
        self.n_layers = n_layers
        self.linear_fwd = nn.Linear(hidden_size, 2048)
        self.linear_rec = nn.Linear(hidden_size * 2, 2048)
        self.precision = precision
        self._pack = None
        self._pack_key = None
        if hidden_size % 32 != 0:
            raise ValueError("tepose_b200 needs hidden_size to be a multiple of 32")

    # ------------------------------------------------------------------ packing
    def _key(self):
        ts = list(self.gru_fwd.parameters()) + list(self.gru_rec.parameters()) + \
            list(self.linear_fwd.parameters()) + list(self.linear_rec.parameters())
        return (self.precision,) + tuple((t.device, t.data_ptr(), t._version) for t in ts)

    def packed(self):
        key = self._key()
        if self._pack is not None and self._pack_key == key:
            return self._pack
        w0 = self.gru_fwd.weight_ih_l0
        nv.require_cuda(w0, "encoder parameters (call .cuda() first)")
        dev, H, Ln = w0.device, self.hidden_size, self.n_layers
        lp = self.precision == "bf16"
        wdt = torch.bfloat16 if lp else torch.float32
        f = lambda t: t.detach().to(dev, torch.float32)
        g = lambda mod, name: f(getattr(mod, name))

        def pad_k(w, kp):
            out = torch.zeros(w.shape[0], kp, device=dev, dtype=wdt)
            out[:, :w.shape[1]] = w.to(wdt)
            return out

        layers = []
        for l in range(Ln):
            in_f = INPUT_SIZE if l == 0 else H
            in_r = INPUT_SIZE if l == 0 else 2 * H
            kpf, kpr = _round_up(in_f, 64), _round_up(in_r, 64)
            wf = g(self.gru_fwd, f"weight_ih_l{l}")
            wr = g(self.gru_rec, f"weight_ih_l{l}")
            wb = g(self.gru_rec, f"weight_ih_l{l}_reverse")
            d = {"kpf": kpf, "kpr": kpr}
            if l == 0:
                # all three directions read the same packed x: stack [fwd | rec-backward | rec-forward]
                d["w_ih"] = torch.cat([pad_k(wf, kpf), pad_k(wb, kpf), pad_k(wr, kpf)], dim=0).contiguous()
                d["b_ih"] = torch.cat([g(self.gru_fwd, "bias_ih_l0"), g(self.gru_rec, "bias_ih_l0_reverse"),
                                       g(self.gru_rec, "bias_ih_l0")]).contiguous()
            else:
                d["w_ih_f"] = pad_k(wf, kpf).contiguous()
                d["b_ih_f"] = g(self.gru_fwd, f"bias_ih_l{l}").contiguous()
                d["w_ih_r"] = torch.cat([pad_k(wb, kpr), pad_k(wr, kpr)], dim=0).contiguous()   # [backward | forward]
                d["b_ih_r"] = torch.cat([g(self.gru_rec, f"bias_ih_l{l}_reverse"), g(self.gru_rec, f"bias_ih_l{l}")]).contiguous()
            d["w_hh"] = [self._pack_whh(g(self.gru_fwd, f"weight_hh_l{l}"), lp),
                         self._pack_whh(g(self.gru_rec, f"weight_hh_l{l}_reverse"), lp),
                         self._pack_whh(g(self.gru_rec, f"weight_hh_l{l}"), lp)]
            if self.precision == "fp32_tc" and l == 0 and Ln == 1 and H % 128 == 0:
                # fp32-grade tensor-core operands (TP_PRECISION_BF16X3): [W_hi | W_hi | W_lo] against [x_hi | x_lo | x_hi]
                def split3(w):
                    hi = w.to(torch.bfloat16)
                    lo = (w - hi.float()).to(torch.bfloat16)
                    return torch.cat([hi, hi, lo], dim=1).contiguous()
                d["w_ih3"] = split3(d["w_ih"])
                d["w_hh3"] = []
                for w in (g(self.gru_fwd, "weight_hh_l0"), g(self.gru_rec, "weight_hh_l0_reverse")):
                    w3 = split3(w).float()
                    out = torch.empty(nv.lib().tp_pack_mma_a_bytes(3 * H, 3 * H), dtype=torch.uint8, device=dev)
                    nv.check(nv.lib().tp_pack_mma_a_bf16(nv.ptr(w3), 3 * H, 3 * H, 3 * H, nv.ptr(out), nv.stream()), "tp_pack_mma_a_bf16")
                    d["w_hh3"].append(out)
                    del w3
            d["w_um"] = [self._pack_whh_umma(g(self.gru_fwd, f"weight_hh_l{l}"), lp),
                         self._pack_whh_umma(g(self.gru_rec, f"weight_hh_l{l}_reverse"), lp),
                         self._pack_whh_umma(g(self.gru_rec, f"weight_hh_l{l}"), lp) if Ln > 1 and l < Ln - 1 else None]
            d["b_hh"] = [g(self.gru_fwd, f"bias_hh_l{l}").contiguous(),
                         g(self.gru_rec, f"bias_hh_l{l}_reverse").contiguous(),
                         g(self.gru_rec, f"bias_hh_l{l}").contiguous()]
            layers.append(d)
        pk = {"layers": layers,
              "w_fwd": nv.pack_linear(g(self.linear_fwd, "weight"), self.precision), "b_fwd": g(self.linear_fwd, "bias").contiguous(),
              "w_rec": nv.pack_linear(g(self.linear_rec, "weight"), self.precision), "b_rec": g(self.linear_rec, "bias").contiguous(),
              "w_cat": nv.pack_linear(torch.cat([0.5 * g(self.linear_fwd, "weight"), 0.5 * g(self.linear_rec, "weight")], dim=1),
                                      self.precision),
              "b_cat": (0.5 * (g(self.linear_fwd, "bias") + g(self.linear_rec, "bias"))).contiguous()}
        self._pack, self._pack_key = pk, key
        return pk

    # ------------------------------------------------------------------ kernels
    def encode_states(self, x: torch.Tensor, h0=None, return_states=False, train_ctx=None):
        """Runs K1 + K2.  Returns (h_fwd [B,H], h_rec [B,2H]) = (y[-1], y_rec[0]) of
        lib/models/tepose.py:73-80.  h0 = (hF0, hB0) carries state (live-stream mode, L=1);
        with return_states the per-step states (yF [T,B,H], yB [T,B,H]) of the two causal
        directions are returned as well.  train_ctx (a dict, training path): per layer, the per-step states of every full
        direction in its run order, the gate activations of every step (tp_gru_job.gates, indexed like the direction's
        output) and the fp32 input of the layer are stored into train_ctx["layers"] for the backward pass."""
        nv.require_cuda(x, "input")
        if x.dim() != 3 or x.shape[2] != INPUT_SIZE:
            raise ValueError(f"expected input [B,T,{INPUT_SIZE}], got {tuple(x.shape)}")
        pk = self.packed()
        L = nv.lib()
        dev, H, Ln = x.device, self.hidden_size, self.n_layers
        B, T = x.shape[0], x.shape[1]
        lp = self.precision == "bf16"
        adt = torch.bfloat16 if lp else torch.float32
        prec = nv.PRECISIONS[self.precision]
        x = x.detach()
        if x.dtype != torch.float16 or train_ctx is not None:      # float16 rows (how the reference's datasets store them) are packed as they are
            x = x.float()
        if x.stride(2) != 1:
            x = x.contiguous()
        if (h0 is not None or return_states) and Ln != 1:
            raise ValueError("carried state is only defined for n_layers == 1 (SURVEY.md H5)")
        # grid-barrier slots: one per layer's recurrence + one for the heads/IEF kernel; cleared by the pack kernel
        sync = torch.empty(Ln + 1, 256, device=dev, dtype=torch.int32)
        self._sync_tail = sync[Ln]
        keep = return_states or train_ctx is not None
        seq_f = torch.empty(T, B, H, device=dev, dtype=torch.float32) if keep else None
        seq_b = torch.empty(T, B, H, device=dev, dtype=torch.float32) if keep else None
        gates_f = gates_b = gates_s = None
        saved = []          # train_ctx["layers"]: one dict per layer
        if train_ctx is not None:
            gates_f = torch.empty(T, B, 4 * H, device=dev, dtype=torch.float32)
            gates_b = torch.empty(T, B, 4 * H, device=dev, dtype=torch.float32)
            gates_s = torch.empty(1, B, 4 * H, device=dev, dtype=torch.float32)
        h_cat = torch.empty(B, 3 * H, device=dev, dtype=torch.float32)     # [y[-1] | y_rec[0]]
        h_fwd, h_rec = h_cat[:, :H], h_cat[:, H:]
        y_f = y_r = y_f_lp = y_r_lp = None
        for l in range(Ln):
            d = pk["layers"][l]
            last = l == Ln - 1
            if l == 0:
                kp = d["kpf"]
                xp = torch.empty(T * B, kp, device=dev, dtype=adt)
                pack_fn = L.tp_pack_rows_f16 if x.dtype == torch.float16 else L.tp_pack_rows_ex
                nv.check(pack_fn(nv.vp(x.data_ptr()), x.stride(0), x.stride(1), B, T, INPUT_SIZE, nv.ptr(xp), kp,
                                 prec, 0, nv.ptr(sync), sync.numel() * 4, nv.stream()), "tp_pack_rows")
                nv.mark("pack")
                if train_ctx is not None:
                    if lp:      # the weight-gradient GEMM reads the packed input in fp32
                        xp32 = torch.empty(T * B, kp, device=dev, dtype=torch.float32)
                        nv.check(L.tp_pack_rows(nv.vp(x.data_ptr()), x.stride(0), x.stride(1), B, T, INPUT_SIZE, nv.ptr(xp32), kp,
                                                nv.PRECISION_FP32, 0, nv.stream()), "tp_pack_rows")
                        x_in = xp32
                    else:
                        x_in = xp
                    saved.append({"x": {"f": x_in, "r": x_in}})
                if last:
                    gi = torch.empty(T * B, 6 * H, device=dev, dtype=torch.float32)      # [fwd | rec-backward]
                    gs = torch.empty(B, 3 * H, device=dev, dtype=torch.float32)          # rec-forward, newest frame only
                    if "w_ih3" in d:             # fp32_tc: x -> [hi | lo | hi] bf16, one tcgen05 GEMM over K = 3 kp
                        xp3 = torch.empty(T * B, 3 * kp, device=dev, dtype=torch.bfloat16)
                        nv.check(L.tp_split3_bf16(nv.ptr(xp), kp, T * B, kp, nv.ptr(xp3), nv.stream()), "tp_split3_bf16")
                        self._input_proj(xp3, T * B, d["w_ih3"], 3 * kp, d["b_ih"],
                                         [(0, T * B, 0, 6 * H), ((T - 1) * B, B, 6 * H, 3 * H)], [gi, gs])
                    else:
                        self._input_proj(xp, T * B, d["w_ih"], kp, d["b_ih"],
                                         [(0, T * B, 0, 6 * H), ((T - 1) * B, B, 6 * H, 3 * H)], [gi, gs])
                    gi_f, c_f, gi_b, c_b, gi_s, c_s = gi, 0, gi, 3 * H, gs, 0
                    s_t0 = 0     # gs holds a single time block
                else:
                    gi = torch.empty(T * B, 9 * H, device=dev, dtype=torch.float32)
                    self._input_proj(xp, T * B, d["w_ih"], kp, d["b_ih"], [(0, T * B, 0, 9 * H)], [gi])
                    gi_f, c_f, gi_b, c_b, gi_s, c_s = gi, 0, gi, 3 * H, gi, 6 * H
                    s_t0 = T - 1
                # layer-0 rows are in ORIGINAL time order; x_rec index tau = T-1-t
                f_in, b_in, s_in = (0, 1), (0, 1), (s_t0, -1)
            else:
                gi_f = torch.empty(T * B, 3 * H, device=dev, dtype=torch.float32)
                self._input_proj(y_f_lp if lp else y_f, T * B, d["w_ih_f"], d["kpf"], d["b_ih_f"],
                                 [(0, T * B, 0, 3 * H)], [gi_f])
                src = y_r_lp if lp else y_r
                if last:
                    gi_b = torch.empty(T * B, 3 * H, device=dev, dtype=torch.float32)
                    gi_s = torch.empty(B, 3 * H, device=dev, dtype=torch.float32)
                    self._input_proj(src, T * B, d["w_ih_r"], d["kpr"], d["b_ih_r"],
                                     [(0, T * B, 0, 3 * H), (0, B, 3 * H, 3 * H)], [gi_b, gi_s])
                    c_b, c_s = 0, 0
                else:
                    gi_r = torch.empty(T * B, 6 * H, device=dev, dtype=torch.float32)
                    self._input_proj(src, T * B, d["w_ih_r"], d["kpr"], d["b_ih_r"], [(0, T * B, 0, 6 * H)], [gi_r])
                    gi_b, c_b, gi_s, c_s = gi_r, 0, gi_r, 3 * H
                c_f = 0
                # deeper layers of gru_rec are indexed by x_rec time tau: backward dir walks tau = T-1..0
                f_in, b_in, s_in = (0, 1), (T - 1, -1), (0, 1)
                if train_ctx is not None:         # the fp32 outputs of the layer below (zero-padded to kpf / kpr)
                    saved.append({"x": {"f": y_f, "r": y_r}})
            gl = [None, None, None]
            if train_ctx is not None and not last:
                gl = [torch.empty(T, B, 4 * H, device=dev, dtype=torch.float32) for _ in range(3)]
            if not last:
                kpn_f, kpn_r = pk["layers"][l + 1]["kpf"], pk["layers"][l + 1]["kpr"]
                ny_f = torch.zeros(T * B, kpn_f, device=dev, dtype=torch.float32)
                ny_r = torch.zeros(T * B, kpn_r, device=dev, dtype=torch.float32)
                ny_f_lp = torch.zeros(T * B, kpn_f, device=dev, dtype=torch.bfloat16) if lp else None
                ny_r_lp = torch.zeros(T * B, kpn_r, device=dev, dtype=torch.bfloat16) if lp else None
            nv.mark(f"k1_input_proj_l{l}")
            hF0, hB0 = (None, None) if h0 is None else h0
            w, b, wu = d["w_hh"], d["b_hh"], d["w_um"]
            k2_prec = None
            # T == 1: every job is a single step from zero (gate math, no recurrent matmul), which BF16X3 does not take
            if last and "w_hh3" in d and h0 is None and T > 1 and B <= 32 and H // 16 <= 148 and "TP_FP32TC_NO_K2" not in os.environ:
                w = [d["w_hh3"][0], d["w_hh3"][1], w[2]]           # the single-step direction has no recurrent matmul
                k2_prec = nv.PRECISION_BF16X3
            if last:
                jobs = [
                    self._job(dev, gi_f, c_f, w[0], b[0], T, f_in[0], f_in[1], h0=hF0, h_final=h_fwd, hcol=0, y=seq_f, w_umma=wu[0],
                              gates=gates_f),
                    self._job(dev, gi_b, c_b, w[1], b[1], T, b_in[0], b_in[1], h0=hB0, h_final=h_rec, hcol=H, y=seq_b, w_umma=wu[1],
                              gates=gates_b),
                    self._job(dev, gi_s, c_s, w[2], b[2], 1, s_in[0] if gi_s.shape[0] != B else 0, s_in[1],
                              h_final=h_rec, hcol=0, gates=gates_s),
                ]
            else:
                # outputs of gru_rec are stored by x_rec index tau: forward dir writes tau = s,
                # backward dir writes tau = T-1-s
                jobs = [
                    self._job(dev, gi_f, c_f, w[0], b[0], T, f_in[0], f_in[1], y=ny_f, y_lp=ny_f_lp, w_umma=wu[0], gates=gl[0]),
                    self._job(dev, gi_b, c_b, w[1], b[1], T, b_in[0], b_in[1], y=ny_r, ycol=H, y_lp=ny_r_lp,
                              t_out0=T - 1, t_out_step=-1, w_umma=wu[1], gates=gl[1]),
                    self._job(dev, gi_s, c_s, w[2], b[2], T, s_in[0], s_in[1], y=ny_r, ycol=0, y_lp=ny_r_lp, w_umma=wu[2],
                              gates=gl[2]),
                ]
            self._recurrence(jobs, B, barrier=sync[l], precision=k2_prec)
            nv.mark(f"k2_recurrence_l{l}")
            if train_ctx is not None:
                if last:
                    saved[l].update(seq={"f": seq_f, "b": seq_b}, gates={"f": gates_f, "b": gates_b, "s": gates_s})
                else:
                    # states in each direction's run order (the backward direction wrote tau = T-1-s); gates stay indexed
                    # like the outputs
                    st = lambda c0: ny_r[:, c0:c0 + H].reshape(T, B, H)
                    saved[l].update(seq={"f": ny_f[:, :H].reshape(T, B, H).contiguous(), "b": st(H).flip(0).contiguous(),
                                         "s": st(0).contiguous()},
                                    gates={"f": gl[0], "b": gl[1], "s": gl[2]})
            if not last:
                y_f, y_r, y_f_lp, y_r_lp = ny_f, ny_r, ny_f_lp, ny_r_lp
        if train_ctx is not None:
            train_ctx["layers"] = saved
        if return_states:
            return h_fwd, h_rec, seq_f, seq_b
        return h_fwd, h_rec

    def heads(self, h_fwd, h_rec, is_train=False):
        """K3 (first half): lib/models/tepose.py:79-85."""
        pk = self.packed()
        B, H = h_fwd.shape[0], self.hidden_size
        feat = torch.empty((B, 2, 2048) if is_train else (B, 2048), device=h_fwd.device, dtype=torch.float32)
        L = nv.lib()
        feat_lp = torch.empty_like(feat, dtype=torch.bfloat16) if self.precision == "bf16" else None
        ws = nv.workspace(L.tp_encoder_heads_workspace_bytes(B), h_fwd.device)
        P = lambda t: nv.vp(0) if t is None else nv.vp(t.data_ptr())
        adjacent = (h_fwd.stride(0) == 3 * H and h_rec.stride(0) == 3 * H
                    and h_rec.data_ptr() == h_fwd.data_ptr() + 4 * H)
        if not is_train and adjacent:      # one GEMM over the concatenated state
            nv.check(L.tp_encoder_heads_cat(nv.PRECISIONS[self.precision], P(pk["w_cat"]), P(pk["b_cat"]), P(h_fwd), 3 * H,
                                            B, H, P(feat), P(feat_lp), P(ws), ws.numel(), nv.stream()), "tp_encoder_heads_cat")
        else:
            nv.check(L.tp_encoder_heads(nv.PRECISIONS[self.precision], P(pk["w_fwd"]), P(pk["b_fwd"]), P(pk["w_rec"]), P(pk["b_rec"]),
                                        P(h_fwd), h_fwd.stride(0), P(h_rec), h_rec.stride(0), B, H,
                                        1 if is_train else 0, P(feat), P(feat_lp), P(ws), ws.numel(), nv.stream()),
                     "tp_encoder_heads")
        feat._tp_bf16 = feat_lp          # bf16 copy rides along for the IEF (same storage order)
        nv.mark("k3_heads")
        return feat

    @nv.device_guard
    def forward(self, x, is_train=False):
        h_fwd, h_rec = self.encode_states(x)
        return self.heads(h_fwd, h_rec, is_train=is_train)


class TePose(nn.Module):
    def __init__(self, seqlen, batch_size=64, n_layers=1, hidden_size=2048,
                 pretrained=osp.join(BASE_DATA_DIR, 'spin_model_checkpoint.pth.tar'), precision="fp32", fold_linear=False):
        super().__init__()
        if precision not in nv.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(nv.PRECISIONS)}")
        self.fold_linear = bool(fold_linear)
        self.fuse_heads = os.environ.get("TP_NO_FUSED_HEADS") is None     # bf16, B <= 32: heads run as the first layers of the IEF kernel
        self.seqlen = seqlen
        self.batch_size = batch_size
        self.encoder = TemporalEncoder(seq_len=seqlen, n_layers=n_layers, hidden_size=hidden_size, precision=precision)
        self.regressor = Regressor(precision=precision)
        if pretrained and os.path.isfile(pretrained):       # lib/models/tepose.py:115-119
            pretrained_dict = torch.load(pretrained)['model']
            self.regressor.load_state_dict(pretrained_dict, strict=False)
            print(f'=> loaded pretrained model from \'{pretrained}\'')

    @property
    def precision(self):
        return self.encoder.precision

    @precision.setter
    def precision(self, value):
        if value not in nv.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(nv.PRECISIONS)}")
        self.encoder.precision = value
        self.regressor.precision = value

    # ------------------------------------------------------------------ heads + IEF as one affine map (opt-in)
    def folded(self, n_iter=3):
        """fold_linear: the eval-mode heads (lib/models/tepose.py:79-85) and the IEF loop (lib/models/spin.py:250-261)
        are both linear AFTER the relu on the encoder states, so

            psc = relu([y[-1] | y_rec[0]]) . (G [0.5 W_fwd | 0.5 W_rec])^T + G (b_fwd + b_rec)/2 + g + A^n p_0

        with G, g, A^n from Regressor.folded().  Composed in float64 at pack time, applied as ONE fp32 GEMM
        [B,3H] x [3H,160] (2-4 MB of weights instead of 25 MB + 7 MB streamed through 11 dependent layers)."""
        enc, reg = self.encoder, self.regressor
        key = (enc._key(), reg._key(), int(n_iter))
        if getattr(self, "_fold_key", None) != key:
            fd, pk = reg.folded(n_iter), reg.packed()
            with torch.no_grad():
                d = lambda t: t.detach().double()
                Wcat = torch.cat([0.5 * d(enc.linear_fwd.weight), 0.5 * d(enc.linear_rec.weight)], dim=1)      # [2048,3H]
                bcat = 0.5 * (d(enc.linear_fwd.bias) + d(enc.linear_rec.bias))
                Gh = fd["G64"] @ Wcat
                gh = fd["G64"] @ bcat + fd["g64"] + fd["An64"] @ pk["init"][0].double()
            self._fold = {"Gh": Gh.float().contiguous(), "gh": gh.float().contiguous()}
            self._fold_key = key
        return self._fold

    def _psc_from_states(self, h_fwd, h_rec):
        """Eval heads + IEF from the encoder states -> IEF state [B,160], through the folded map or the fused persistent
        kernel; None when neither applies (fp32 mode, more than 32 rows, states not adjacent in memory)."""
        H = self.encoder.hidden_size
        B = h_fwd.shape[0]
        adjacent = (h_fwd.stride(0) == 3 * H and h_rec.stride(0) == 3 * H and h_rec.data_ptr() == h_fwd.data_ptr() + 4 * H)
        if not adjacent:
            return None
        if self.fold_linear:
            from .spin import folded_gemm
            fd = self.folded()
            h_cat = torch.as_strided(h_fwd, (B, 3 * H), (3 * H, 1))
            psc = folded_gemm(h_cat, fd["Gh"], fd["gh"], relu_a=True)
            nv.mark("k3_folded")
            return psc
        if self.precision == "bf16" and B <= 32 and self.fuse_heads:
            # heads + IEF in one persistent kernel (the [B,2048] feature stays inside it)
            from .spin import PSC
            L = nv.lib()
            pe, pr = self.encoder.packed(), self.regressor.packed()
            psc = torch.empty(B, PSC, device=h_fwd.device, dtype=torch.float32)
            ws = nv.workspace(L.tp_ief_workspace_bytes(B), h_fwd.device)
            bar = getattr(self.encoder, "_sync_tail", None)      # zeroed at the top of encode_states (same stream, same step)
            self.encoder._sync_tail = None                       # one use per fill
            nv.check(L.tp_heads_ief_forward(nv.ptr(pe["w_cat"]), nv.ptr(pe["b_cat"]), nv.vp(h_fwd.data_ptr()), 3 * H, H, pr["c"], B,
                                            nv.ptr(pr["init"]), 1, 3, nv.ptr(psc), nv.ptr(ws), ws.numel(),
                                            nv.vp(0 if bar is None else bar.data_ptr()), nv.stream()),
                     "tp_heads_ief_forward")
            nv.mark("k3_heads_ief")
            return psc
        return None

    def regress_states(self, h_fwd, h_rec, is_train=False, J_regressor=None):
        """K3..K5 from the encoder states (y[-1], y_rec[0]): heads + Regressor, or their fused / folded form."""
        if not is_train:
            psc = self._psc_from_states(h_fwd, h_rec)
            if psc is not None:
                return self.regressor.decode(psc, is_train=False, J_regressor=J_regressor)
        feature = self.encoder.heads(h_fwd, h_rec, is_train=is_train)
        lp = getattr(feature, "_tp_bf16", None)
        feature = feature.reshape(-1, feature.size(-1))
        if lp is not None:
            feature._tp_bf16 = lp.reshape(-1, lp.size(-1))
        return self.regressor(feature, is_train=is_train, J_regressor=J_regressor)

    # sequences per pass of the encoder + regressor kernels: their fast paths (interleaved recurrence, fused heads + IEF)
    # hold one 32-row batch tile; larger batches run as balanced groups and share ONE SMPL pass
    GROUP = 32

    @nv.device_guard
    def forward(self, input, is_train=False, J_regressor=None, dropout_masks=None):
        if self.training:
            # lib/core/trainer.py:137,203: generator.train(); generator(inp, is_train=True) -- dropout active, outputs [B,2,...],
            # gradients to every encoder / regressor parameter through the hand-written backward (tepose_b200/train.py)
            if not is_train:
                raise NotImplementedError("tepose_b200.TePose in .train() mode implements the reference's training call "
                                          "(is_train=True); call .eval() for inference")
            from .train import train_forward
            return train_forward(self, input, dropout_masks)
        batch_size = input.shape[0]
        nv.mark("start")
        smpl_output = None
        if batch_size > self.GROUP and not is_train and (self.precision == "bf16" or self.fold_linear):
            # measured (B = 64, bf16): 0.81 ms on the generic batch-tiled kernels vs 0.52 ms as two groups of 32
            ngroups = (batch_size + self.GROUP - 1) // self.GROUP
            per = (batch_size + ngroups - 1) // ngroups
            pscs = []
            for b0 in range(0, batch_size, per):
                h_fwd, h_rec = self.encoder.encode_states(input[b0:b0 + per])
                psc = self._psc_from_states(h_fwd, h_rec)
                if psc is None:
                    pscs = None
                    break
                pscs.append(psc)
            if pscs is not None:
                smpl_output = self.regressor.decode(torch.cat(pscs, dim=0), is_train=False, J_regressor=J_regressor)
        if smpl_output is None:
            h_fwd, h_rec = self.encoder.encode_states(input)
            smpl_output = self.regress_states(h_fwd, h_rec, is_train=is_train, J_regressor=J_regressor)
        lead = (batch_size, 2) if is_train else (batch_size,)
        for s in smpl_output:                                  # lib/models/tepose.py:130-145
            s['theta'] = s['theta'].reshape(*lead, -1)
            s['verts'] = s['verts'].reshape(*lead, -1, 3)
            s['kp_2d'] = s['kp_2d'].reshape(*lead, -1, 2)
            s['kp_3d'] = s['kp_3d'].reshape(*lead, -1, 3)
            s['rotmat'] = s['rotmat'].reshape(*lead, -1, 3, 3)
        return smpl_output
