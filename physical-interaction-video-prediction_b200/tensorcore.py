"""bf16 tensor-core plan for the seven ConvLSTM layers: bf16 operand shadows, prepared weights, tcgen05 launches.

Created by ``Engine`` when ``compute="bf16"``.  fp32 stays the master format of every activation that the
bandwidth-bound kernels consume (cell state, LayerNorm input, gradients); this class only adds the bf16 GEMM operands:
  xh_bf16[l][t]  (M, Kpad)   concatenated layer input [x | h_{t-1}], channels padded to a multiple of 64 (fwd GEMM A operand)
  dg_bf16[l][t]  (M, 4C)     gate pre-activation gradients (input-gradient GEMM A operand)
  (the weight-gradient GEMM reads xh_bf16 / dg_bf16 of ALL time steps MN-major, straight from these NHWC tensors)
  Wf[l], Wd[l]               K-major bf16 weights (forward / tap-flipped input-gradient), refreshed after every Adam step
"""
import ctypes

import numpy as np
import torch

from .engine import LSTM_IN, LSTM_SIZES, LSTM_LEVEL, View, _ptr
from ._lib import PivpError


class TensorCorePlan(object):
    store_gates = True                                   # ConvLSTM forward keeps its activated gates (bf16, dg_bf16) for the backward pass

    def __init__(self, eng, ws):
        self.eng = eng
        self.ws = ws
        dev = eng.dev
        B, T = ws["B"], ws["T"]
        S = T - 1
        self.S = S
        self.Kpad = [(cin + c + 63) // 64 * 64 for cin, c in zip(LSTM_IN, LSTM_SIZES)]
        self.xh_all, self.dg_all, self.xh_bf16, self.dg_bf16 = [], [], [], []
        self.Wf, self.Wd = [], []
        wsb = 16
        for li, (cin, c, lv) in enumerate(zip(LSTM_IN, LSTM_SIZES, LSTM_LEVEL)):
            M = ws["Mr"][lv]
            h, w = eng.H // lv, eng.W // lv
            if M % 128 or (h * w) % 64:
                raise PivpError("bf16 tensor-core path: ConvLSTM layer %d has B*H*W = %d (needs a multiple of 128) and H*W = %d "
                                "(needs a multiple of 64); use an even batch / 64x64 or larger images, or compute='f32'"
                                % (li + 1, M, h * w))
            xa = torch.zeros(T, M, self.Kpad[li], dtype=torch.bfloat16, device=dev)      # zeros: h_{-1}, pad channels
            da = torch.empty(S, M, 4 * c, dtype=torch.bfloat16, device=dev)      # forward: activated gates; backward: overwritten by dG
            self.xh_all.append(xa)
            self.dg_all.append(da)
            self.xh_bf16.append([xa[t] for t in range(T)])
            self.dg_bf16.append([da[t] for t in range(S)])
            self.Wf.append(torch.empty(4 * c, 25, self.Kpad[li], dtype=torch.bfloat16, device=dev))
            self.Wd.append(torch.empty(cin + c, 25, 4 * c, dtype=torch.bfloat16, device=dev))
            wsb = max(wsb, eng.L.query("pivp_tc_wgrad_workspace_bytes", S * B, h, w, cin + c, 4 * c))
        self.wgrad_ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        self.accurate = 0
        import os
        # LayerNorm of the ConvLSTM output applied inside the gate epilogue (pivp_tc_conv5x5_ln): per-layer arrival counters, zeroed once.
        # OFF by default: measured on the b32 step (profiles/r02_halo_epilogue.md) the per-sample rendezvous (publish, atomic arrival, poll,
        # fetch of the sample's pairs: three dependent L2 round trips behind the slowest tile of the sample) adds 4.2 us to each forward
        # launch, while the LayerNorm kernel it removes costs 3.1 us inside the graph: 8.81 ms per step fused against 8.75 ms unfused.
        self.ln_counter = [torch.zeros(B, dtype=torch.int32, device=dev) for _ in LSTM_SIZES]
        self.fuse_ln = os.environ.get("PIVP_TC_FUSE_LN", "0") != "0"
        self.split_n = int(os.environ.get("PIVP_TC_SPLIT_N", "0"))       # tuning switch for the input-gradient N split
        self.pair_bn = int(os.environ.get("PIVP_TC_PAIR_BN", "96"))      # N tile of the 8x8-map input gradient (0: per-tap kernel's choice)
        # layers whose maps the halo-patch kernel tiles (H % 16 == 0, W % 8 == 0): its epilogue also produces the LayerNorm statistics
        self.ln_fused = [(eng.H // lv) % 16 == 0 and (eng.W // lv) % 8 == 0 and ((eng.H // lv) * (eng.W // lv) * c) % 4096 == 0
                         for c, lv in zip(LSTM_SIZES, LSTM_LEVEL)]
        # bf16 weight operands of the tap GEMMs live in ONE flat buffer filled by ONE gather launch per parameter update
        self._wflat = torch.zeros(2 << 20, dtype=torch.bfloat16, device=dev)
        self._wofs, self._widx = 0, []
        # ---- stride-2 Deconvolution2D layers enc4/enc5/enc6 (train_model.py:505-507) as 4 output phases each
        M8, M4, M2 = ws["Mr"][8], ws["Mr"][4], ws["Mr"][2]
        self.hid5_b = [torch.zeros(M8, 128, dtype=torch.bfloat16, device=dev) for _ in range(S)]
        self.cat5_b = [torch.zeros(M4, 128, dtype=torch.bfloat16, device=dev) for _ in range(S)]     # 96 used, 32 zero pad
        self.cat6_b = [torch.zeros(M2, 64, dtype=torch.bfloat16, device=dev) for _ in range(S)]
        self.dec = {}
        for name, cin, cout, lv in (("enc4", 128, 128, 8), ("enc5", 96, 96, 4), ("enc6", 64, 64, 2)):
            self.dec[name] = self._plan_deconv(name, cin, cout, lv)
        # input gradients of the stride-2 convolutions enc1 / enc2 are transposed convolutions too: same phase decomposition
        # (conv weight [N][ky][kx][C] has the deconv form with in := N, out := C)
        self.dec["enc1"] = self._plan_deconv("enc1", 32, 32, 4)
        self.dec["enc2"] = self._plan_deconv("enc2", 64, 64, 8)
        # forward of the stride-2 convolutions enc1 / enc2: 9-tap stride-1 GEMM on the space-to-depth bf16 input (half grid, 4 phases x cb ch)
        self.s2f = {"enc1": self._plan_conv_s2_fwd("enc1", 32, 32, 2), "enc2": self._plan_conv_s2_fwd("enc2", 64, 64, 4)}
        # bf16 d(pre-activation) of enc1 (32 of 64 used) / enc2, all time steps kept: operand of the input gradient AND of the deferred weight gradient
        self.de_b = {"enc1": torch.zeros(S, M4, 64, dtype=torch.bfloat16, device=dev), "enc2": torch.zeros(S, M8, 64, dtype=torch.bfloat16, device=dev)}
        # ---- deconvolution backward: dY in space-to-depth bf16 (all time steps kept for the deferred weight gradient)
        self.dbw = {}
        wsb2 = 16
        for name, cin, cout, lv, xs in (("enc4", 128, 128, 8, self.hid5_b), ("enc5", 96, 96, 4, self.cat5_b), ("enc6", 64, 64, 2, self.cat6_b)):
            self.dbw[name] = self._plan_deconv_bwd(name, cin, cout, lv)
            wsb2 = max(wsb2, eng.L.query("pivp_tc_wgrad_taps_workspace_bytes", S * B, eng.H // lv, eng.W // lv, cout, cin, 9))
        for name, d in self.s2f.items():
            wsb2 = max(wsb2, eng.L.query("pivp_tc_wgrad_taps_workspace_bytes", S * B, eng.H // d["lv"], eng.W // d["lv"], d["cin"], d["cout"], 9))
        if wsb2 > self.wgrad_ws.numel():
            self.wgrad_ws = torch.empty(wsb2, dtype=torch.uint8, device=dev)
        # the deferred weight gradient needs the deconv inputs of all time steps stacked: re-home them in one tensor each
        for nm in ("hid5_b", "cat5_b", "cat6_b"):
            old = getattr(self, nm)
            allt = torch.zeros(S, old[0].shape[0], old[0].shape[1], dtype=torch.bfloat16, device=dev)
            setattr(self, nm + "_all", allt)
            setattr(self, nm, [allt[t] for t in range(S)])
        self._widx_all = torch.from_numpy(np.concatenate(self._widx)).to(dev)
        # parallel branches for the deferred weight gradients (wgrad_all): PIVP_WGRAD_STREAMS = total branches (1 = one chain)
        nbr = max(1, min(3, int(os.environ.get("PIVP_WGRAD_STREAMS", "3"))))       # measured on the b32 step: 8.61 / 8.37 / 8.31 ms with 1 / 2 / 3
        self.wg_streams = [torch.cuda.Stream(device=dev) for _ in range(nbr - 1)]
        self.wg_ws = [torch.empty_like(self.wgrad_ws) for _ in range(nbr - 1)]
        self.early_on = os.environ.get("PIVP_WGRAD_EARLY", "1") != "0"
        self.wg_ws_early = [torch.empty_like(self.wgrad_ws) for _ in range(2)] if (nbr == 3 and self.early_on) else []
        self._early = set()
        self.refresh_weights()

    def _walloc(self, idx, shape):
        """Carve a bf16 operand of `shape` out of the flat weight buffer; idx (int32, flat parameter offsets, -1 = zero) says how to fill it."""
        idx = np.ascontiguousarray(idx, np.int32).reshape(-1)
        n = idx.size
        npad = (n + 63) // 64 * 64                       # 128-byte aligned operands (TMA global addresses)
        if self._wofs + npad > self._wflat.numel():
            raise PivpError("tensor-core weight buffer too small")
        view = self._wflat[self._wofs:self._wofs + n].view(*shape)
        self._widx.append(np.concatenate([idx, np.full(npad - n, -1, np.int32)]))
        self._wofs += npad
        return view

    def _plan_conv_s2_fwd(self, name, cin, cout, lv_in):
        """out[oy,ox][n] = sum_{ky,kx,c} W[n][ky][kx][c] in[2oy+ky-1, 2ox+kx-1][c]: on the space-to-depth input (pixel (y', x') of the half
        grid holds the 2x2 phases (py,px) in channel blocks of cb) tap k reads half-grid offset {0:-1, 1:0, 2:0}[k] and phase {0:1, 1:0, 2:1}[k]."""
        e = self.eng
        dev = e.dev
        cb = (cin + 63) // 64 * 64
        lv = 2 * lv_in
        M = self.ws["Mr"][lv]
        tapdef = {0: (-1, 1), 1: (0, 0), 2: (0, 1)}
        taps = []
        for ky in range(3):
            for kx in range(3):
                (dy, py), (dx, px) = tapdef[ky], tapdef[kx]
                taps.append((dy, dx, (py * 2 + px) * cb))
        base = e.spec[name + "/W"].offset                      # internal conv layout [N][ky][kx][C]
        idx = np.full((cout, 9, cb), -1, np.int32)
        c = np.arange(cin)
        for n in range(cout):
            for tp in range(9):
                idx[n, tp, :cin] = base + (n * 9 + tp) * cin + c
        arr = lambda v: (ctypes.c_int * 9)(*v)
        return dict(cin=cin, cout=cout, cb=cb, lv=lv, dy=arr([q[0] for q in taps]), dx=arr([q[1] for q in taps]), co=arr([q[2] for q in taps]),
                    wt=self._walloc(idx, (cout, 9 * cb)),
                    xs=torch.zeros(self.S, M, 4 * cb, dtype=torch.bfloat16, device=dev))      # kept per time step for the weight gradient

    def s2d_operand(self, name, t, width):
        """(bf16 View, (map width, channel block)) of the space-to-depth GEMM operand of stride-2 convolution `name` at step t: what the
        LayerNorm in front of it writes directly (Engine._ln_fwd(..., y_bf16, s2d))."""
        d = self.s2f[name]
        return View(d["xs"][t], 4 * d["cb"], 0, d["cin"]), (width, d["cb"])

    def conv_s2_fwd(self, name, t, x_f32, x_cs, out, out_cs, out_bf16, ob_cs):
        """Stride-2 Convolution2D + bias + ReLU (train_model.py:501-502): one tcgen05 launch on the space-to-depth bf16 input, which the
        producing LayerNorm wrote (x_f32 None) or which is cast from the fp32 input here."""
        e, d = self.eng, self.s2f[name]
        h, w = e.H // d["lv"], e.W // d["lv"]
        B = self.ws["B"]
        xs = d["xs"][t]
        if x_f32 is not None:
            e.L.call("pivp_cast_bf16", _ptr(x_f32), x_cs, 0, _ptr(xs), 4 * d["cb"], 0, B * 4 * h * w, d["cin"], 2 * h, 2 * w, 1, d["cb"], e._s())
        e.L.call("pivp_tc_conv_taps", _ptr(xs), 4 * d["cb"], B, h, w, d["cb"], 9, d["dy"], d["dx"], d["co"], _ptr(d["wt"]),
                 d["cout"], d["cout"], _ptr(e.p[name + "/b"]), 1, 0, _ptr(out), out_cs, 0, _ptr(out_bf16), ob_cs, 0, h, w, 1, 0, 0, e._s())

    def _plan_deconv_bwd(self, name, cin, cout, lv):
        """Backward of a stride-2 deconvolution on the tensor cores.  dY (big grid) is cast to space-to-depth bf16
        [B][h][w][4*cb]; then d_in[i,j][ci] = sum_{ky,kx,co} dY[2i+ky-1, 2j+kx-1][co] W[ci][ky][kx][co] is a 9-tap stride-1
        implicit GEMM on the small grid (tap -> pixel offset {-1,0} and phase channel block), and dW[ci][ky][kx][co] is the
        MN-major weight-gradient GEMM with the same taps (its output layout IS the internal [ci][ky][kx][co] layout)."""
        e = self.eng
        dev = e.dev
        cb = (cout + 63) // 64 * 64
        S, M = self.S, self.ws["Mr"][lv]
        tapdef = {0: (-1, 1), 1: (0, 0), 2: (0, 1)}                     # k -> (pixel offset, phase)
        taps = []
        for ky in range(3):
            for kx in range(3):
                (dy, py), (dx, px) = tapdef[ky], tapdef[kx]
                taps.append((dy, dx, (py * 2 + px) * cb))
        base = e.spec[name + "/W"].offset
        idx = np.full((cin, 9, cb), -1, np.int32)
        co = np.arange(cout)
        for ci in range(cin):
            for t in range(9):
                idx[ci, t, :cout] = base + (ci * 9 + t) * cout + co
        arr = lambda v: (ctypes.c_int * 9)(*v)
        bn = cin if cin <= 128 else 128
        if (M // 128) * (cin // bn) < 64 and cin % 64 == 0:
            bn = 64
        return dict(cin=cin, cout=cout, cb=cb, lv=lv, bn=bn, dy=arr([t[0] for t in taps]), dx=arr([t[1] for t in taps]),
                    co=arr([t[2] for t in taps]), wt=self._walloc(idx, (cin, 9 * cb)),
                    dys=torch.zeros(S, M, 4 * cb, dtype=torch.bfloat16, device=dev))

    def _plan_deconv(self, name, cin, cout, lv):
        """Sub-pixel decomposition: output pixel (2i+a, 2j+b) only sees taps ky = a+1 (mod 2), kx = b+1 (mod 2):
        1 / 2 / 2 / 4 taps for the four phases, each a stride-1 implicit GEMM on the INPUT grid (oy = 2*iy + ky - 1)."""
        e = self.eng
        dev = e.dev
        kc = (cin + 63) // 64 * 64
        base = e.spec[name + "/W"].offset                 # internal layout [cin][ky][kx][cout]
        sel = {0: [(0, 1)], 1: [(1, 0), (0, 2)]}          # phase -> [(pixel offset, kernel index)]
        phases = []
        for a in (0, 1):
            for b in (0, 1):
                taps = [(dy, dx, ky, kx) for (dy, ky) in sel[a] for (dx, kx) in sel[b]]
                idx = np.full((cout, len(taps), kc), -1, np.int32)
                ci = np.arange(cin)
                for t, (dy, dx, ky, kx) in enumerate(taps):
                    for co in range(cout):
                        idx[co, t, :cin] = base + ((ci * 3 + ky) * 3 + kx) * cout + co
                arr = lambda v: (ctypes.c_int * len(taps))(*v)
                phases.append(dict(a=a, b=b, n=len(taps), dy=arr([t[0] for t in taps]), dx=arr([t[1] for t in taps]),
                                   co=arr([0] * len(taps)), wt=self._walloc(idx, (cout, len(taps) * kc))))
        bn = cout if cout <= 128 else 128
        if 4 * (self.ws["Mr"][lv] // 128) * (cout // bn) < 120 and cout % 64 == 0:      # the four phases share one launch
            bn = 64
        # flattened per-phase lists for pivp_tc_conv_taps_multi (4 slots per phase)
        flat = lambda key: (ctypes.c_int * 16)(*[(list(ph[key]) + [0] * 4)[:4][i] for ph in phases for i in range(4)])
        multi = dict(ntaps=(ctypes.c_int * 4)(*[ph["n"] for ph in phases]), dy=flat("dy"), dx=flat("dx"), co=flat("co"),
                     wt=(ctypes.c_void_p * 4)(*[ph["wt"].data_ptr() for ph in phases]),
                     oa=(ctypes.c_int * 4)(*[ph["a"] for ph in phases]), ob=(ctypes.c_int * 4)(*[ph["b"] for ph in phases]))
        return dict(cin=cin, cout=cout, kc=kc, lv=lv, phases=phases, bn=bn, multi=multi)

    def refresh_weights(self):
        e = self.eng
        for li, (cin, c) in enumerate(zip(LSTM_IN, LSTM_SIZES)):
            e.L.call("pivp_tc_prep_weights", _ptr(e.p["lstm%d/conv/W" % (li + 1)]), 4 * c, cin + c, self.Kpad[li],
                     _ptr(self.Wf[li]), _ptr(self.Wd[li]), e._s())
        if getattr(self, "_widx_all", None) is not None:
            e.L.call("pivp_gather_bf16", _ptr(e.flat_p), _ptr(self._widx_all), self._wofs, _ptr(self._wflat), e._s())

    def deconv_bwd_data(self, name, t, dy_f32, out, accumulate):
        """dY (fp32, big grid, dense rows of cout) -> space-to-depth bf16 (kept for wgrad) -> d_in (fp32, dense rows of cin)."""
        e, d = self.eng, self.dbw[name]
        h, w = e.H // d["lv"], e.W // d["lv"]
        B = self.ws["B"]
        e.L.call("pivp_cast_bf16", _ptr(dy_f32), d["cout"], 0, _ptr(d["dys"][t]), 4 * d["cb"], 0, B * 4 * h * w, d["cout"], 2 * h, 2 * w, 1,
                 d["cb"], e._s())
        e.L.call("pivp_tc_conv_taps", _ptr(d["dys"][t]), 4 * d["cb"], B, h, w, d["cb"], 9, d["dy"], d["dx"], d["co"], _ptr(d["wt"]),
                 d["cin"], d["bn"], 0, 0, accumulate, _ptr(out), d["cin"], 0, 0, 0, 0, h, w, 1, 0, 0, e._s())

    def deconv_handover(self, name, t, width, db):
        """What Engine._ln_bwd(handover=...) needs to write the bf16 space-to-depth operand of deconvolution `name`'s backward itself:
        (operand tensor of step t, its row stride, width of the big map, channel block, bias-gradient tensor)."""
        d = self.dbw[name]
        return d["dys"][t], 4 * d["cb"], width, d["cb"], db

    def deconv_bwd_fused(self, name, t, out, ga, gb, db, d_in, accumulate, handover=True):
        """Backward of a stride-2 deconvolution fed by a ReLU (``out`` = its output view, or None for a plain gradient):
        ONE hand-over launch masks the gradient, accumulates the bias gradient and writes the space-to-depth bf16 operand
        (kept for the deferred weight gradient), then the 9-tap tcgen05 GEMM produces d_in."""
        e, d = self.eng, self.dbw[name]
        h, w = e.H // d["lv"], e.W // d["lv"]
        B = self.ws["B"]
        z = lambda v: (0, 0, 0) if v is None else (v.ptr, v.cs, v.co)
        if handover:                         # else: the producer (LayerNorm backward) already wrote d["dys"][t] and the bias gradient
            e.L.call("pivp_grad_handover", *z(out), *z(ga), *z(gb), 0, 0, 0, _ptr(d["dys"][t]), 4 * d["cb"], 0, 2 * h, 2 * w, 1, d["cb"],
                     _ptr(db), B * 4 * h * w, d["cout"], e._s())
        e.L.call("pivp_tc_conv_taps", _ptr(d["dys"][t]), 4 * d["cb"], B, h, w, d["cb"], 9, d["dy"], d["dx"], d["co"], _ptr(d["wt"]),
                 d["cin"], d["bn"], 0, 0, accumulate, _ptr(d_in), d["cin"], 0, 0, 0, 0, h, w, 1, 0, 0, e._s())

    def conv_s2_dgrad_fused(self, name, t, out, ga, gb, db, M, C, d_in, d_in_cs):
        """ReLU backward of a stride-2 convolution's output + its input gradient: the hand-over masks the gradient, accumulates the bias
        gradient and writes the bf16 GEMM operand (kept for the deferred weight gradient) in one launch; then the four output phases
        of the transposed convolution in one tcgen05 launch."""
        e = self.eng
        z = lambda v: (0, 0, 0) if v is None else (v.ptr, v.cs, v.co)
        dy_b = self.de_b[name][t]
        e.L.call("pivp_grad_handover", *z(out), *z(ga), *z(gb), 0, 0, 0, _ptr(dy_b), dy_b.shape[1], 0, 0, 0, 0, 0,
                 _ptr(db), M, C, e._s())
        self.deconv_fwd(name, dy_b, d_in, d_in_cs, None, 0, 0, bias=False)

    def conv_s2_wgrad_all(self, wsb=None):
        """Deferred weight gradients of the stride-2 convolutions enc1 / enc2 over all time steps: dW[n][ky][kx][c] contracts the bf16
        d(pre-activation) with the tap-shifted space-to-depth input the forward already wrote (train_model.py:501-502 backward)."""
        e, S, B = self.eng, self.S, self.ws["B"]
        for name in ("enc1", "enc2"):
            d = self.s2f[name]
            h, w = e.H // d["lv"], e.W // d["lv"]
            a = self.de_b[name]
            wsb_ = self.wgrad_ws if wsb is None else wsb
            e.L.call("pivp_tc_wgrad_taps", _ptr(a), a.shape[2], _ptr(d["xs"]), 4 * d["cb"], S * B, h, w, d["cin"], d["cout"], 9,
                     d["dy"], d["dx"], d["co"], _ptr(e.g[name + "/W"]), _ptr(wsb_), wsb_.numel(), e._s())

    def deconv_wgrad_all(self, wsb=None):
        """Deferred weight gradients of enc4/5/6 over all time steps (one MN-major GEMM each)."""
        e, S, B = self.eng, self.S, self.ws["B"]
        for name, xall in (("enc4", self.hid5_b_all), ("enc5", self.cat5_b_all), ("enc6", self.cat6_b_all)):
            d = self.dbw[name]
            h, w = e.H // d["lv"], e.W // d["lv"]
            wsb_ = self.wgrad_ws if wsb is None else wsb
            e.L.call("pivp_tc_wgrad_taps", _ptr(xall), xall.shape[2], _ptr(d["dys"]), 4 * d["cb"], S * B, h, w, d["cout"], d["cin"], 9,
                     d["dy"], d["dx"], d["co"], _ptr(e.g[name + "/W"]), _ptr(wsb_), wsb_.numel(), e._s())

    def deconv_fwd(self, name, x_bf16, out, out_cs, out_bf16, ob_cs, relu, bias=True, ln_partial=None):
        """Deconvolution2D forward (+bias, optional ReLU) -> fp32 view `out` (row stride out_cs, channel offset 0) and an
        optional bf16 copy (the next ConvLSTM's x slot): the four output phases in one tcgen05 launch.  ``ln_partial``: the epilogue
        also writes the (mean, M2) partials of the LayerNorm that follows (norm_enc6), so that LayerNorm skips its statistics launch."""
        e, d = self.eng, self.dec[name]
        h, w = e.H // d["lv"], e.W // d["lv"]
        m = d["multi"]                       # the four output phases in one launch (grid z = phase, or walked inside each CTA)
        e.L.call("pivp_tc_conv_taps_multi_ln", _ptr(x_bf16), d["kc"], self.ws["B"], h, w, d["kc"], 4, m["ntaps"], m["dy"], m["dx"], m["co"],
                 m["wt"], d["cout"], d["bn"], _ptr(e.p[name + "/b"]) if bias else 0, relu, 0,
                 _ptr(out), out_cs, 0, _ptr(out_bf16), ob_cs, 0, 2 * h, 2 * w, 2, m["oa"], m["ob"], _ptr(ln_partial), e._s())

    def xview(self, li, t):
        """bf16 x-slot of layer li at time t (what the producer of the layer input also writes)."""
        return View(self.xh_bf16[li][t], self.Kpad[li], 0, LSTM_IN[li])

    def ln_fusable(self, li):
        """The LayerNorm behind ConvLSTM layer li can run inside the layer's gate epilogue: halo geometry with fused statistics and a launch
        of at most 148 CTAs (one per SM: the per-sample rendezvous needs all of them resident)."""
        e = self.eng
        C, lv = LSTM_SIZES[li], LSTM_LEVEL[li]
        h, w = e.H // lv, e.W // lv
        tiles = self.ws["B"] * (h // 16) * (w // 8) if self.ln_fused[li] else 0
        ctas_one, ctas_two = tiles * (C // 32), (tiles // 2) * (C // 32)
        ctas = ctas_two if (tiles % 2 == 0 and ctas_two >= 96) else ctas_one          # launch_conv5x5_halo's choice of tiles per CTA
        return self.fuse_ln and self.ln_fused[li] and 0 < ctas <= 148

    def lstm_fwd(self, li, t, ln=None):
        """conv + bias + gates + cell + h of BasicConvLSTMCell (train_model.py:262-272) in ONE tcgen05 kernel.
        ``ln`` = (name, y View, y_bf16 View or None, stats): also apply the LayerNorm of the layer's output there (train_model.py:596-601)."""
        e, ws = self.eng, self.ws
        cin, C, lv = LSTM_IN[li], LSTM_SIZES[li], LSTM_LEVEL[li]
        h, w = e.H // lv, e.W // lv
        if ln is not None:
            name, y, yb, stats = ln
            e.L.call("pivp_tc_conv5x5_ln", _ptr(self.xh_bf16[li][t]), self.Kpad[li], ws["B"], h, w, self.Kpad[li], _ptr(self.Wf[li]), C,
                     _ptr(e.p["lstm%d/conv/b" % (li + 1)]), _ptr(self.dg_bf16[li][t]), _ptr(ws["c"][li][t - 1]) if t > 0 else 0, _ptr(ws["c"][li][t]),
                     _ptr(ws["xh"][li][t + 1]), cin + C, cin, _ptr(self.xh_bf16[li][t + 1]), self.Kpad[li], cin, 1.0, self.accurate, _ptr(ws["ln_ws"]),
                     _ptr(e.p[name + "/norm/gamma"]), _ptr(e.p[name + "/norm/beta"]), 1e-6, y.ptr, y.cs, y.co,
                     0 if yb is None else yb.ptr, 0 if yb is None else yb.cs, 0 if yb is None else yb.co, _ptr(stats), _ptr(self.ln_counter[li]), e._s())
            return
        e.L.call("pivp_tc_conv5x5", _ptr(self.xh_bf16[li][t]), self.Kpad[li], ws["B"], h, w, self.Kpad[li],
                 _ptr(self.Wf[li]), 4 * C, 128, 1, _ptr(e.p["lstm%d/conv/b" % (li + 1)]),
                 0, 0, 0,
                 _ptr(self.dg_bf16[li][t]), _ptr(ws["c"][li][t - 1]) if t > 0 else 0, _ptr(ws["c"][li][t]),
                 _ptr(ws["xh"][li][t + 1]), cin + C, cin, _ptr(self.xh_bf16[li][t + 1]), self.Kpad[li], cin,
                 0, 0, 0,
                 C, 1.0, self.accurate | (2 if self.store_gates else 4), _ptr(ws["ln_ws"]) if self.ln_fused[li] else 0, e._s())
        # flags bit 1: the activated gates are stored bf16, in dg_bf16[li][t] (bit 2 instead: not stored); ln_ws: LayerNorm statistics of h
        # from the epilogue

    def lstm_dgrad(self, li, t):
        """dxh = conv(dG_t, tap-flipped W): gradient w.r.t. the concatenated input [x | h_{t-1}] (D.5)."""
        e, ws = self.eng, self.ws
        cin, C, lv = LSTM_IN[li], LSTM_SIZES[li], LSTM_LEVEL[li]
        h, w = e.H // lv, e.W // lv
        cx = cin + C
        bn = cx                                # one N tile if that already fills the GPU, else the largest split reaching ~1 wave
        mt = ws["Mr"][lv] // 128
        halo = h % 16 == 0 and w % 8 == 0      # halo-patch kernel: one CTA per SM, so 64 pixel tiles leave half the GPU idle:
        if halo and mt < 100 and (cx // 2) % 16 == 0 and self.split_n:      # two N tiles of cx/2 (narrower tiles starve the weight ring)
            bn = cx // 2
        if h == 8 and w == 8 and ws["B"] % 2 == 0 and self.pair_bn:        # 8x8 maps: halo kernel in its two-image geometry, 16 pixel tiles only
            halo = True
            bn = self.pair_bn if cx % self.pair_bn == 0 else cx
        for cand in (cx, cx // 2, cx // 3, cx // 6):      # multiples of 32 only: N=48 tiles measured 2.4x slower than N=96
            if halo:
                break
            if cand >= 32 and cand % 32 == 0 and cx % cand == 0:
                bn = cand
                if mt * (cx // cand) >= 120:
                    break
        e.L.call("pivp_tc_conv5x5", _ptr(self.dg_bf16[li][t]), 4 * C, ws["B"], h, w, 4 * C,
                 _ptr(self.Wd[li]), cx, bn, 0, 0,
                 _ptr(ws["dxh"][li]), cx, 0,
                 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                 C, 0.0, 0, 0, e._s())

    def _lstm_wgrad(self, li, wsb):
        e, ws = self.eng, self.ws
        S, B = self.S, ws["B"]
        cin, C, lv = LSTM_IN[li], LSTM_SIZES[li], LSTM_LEVEL[li]
        M = ws["Mr"][lv]
        h, w = e.H // lv, e.W // lv
        cx = cin + C
        name = "lstm%d/conv" % (li + 1)
        e.L.call("pivp_tc_colsum_bf16", _ptr(self.dg_all[li]), 4 * C, S * M, 4 * C, _ptr(e.g[name + "/b"]), e._s())
        e.L.call("pivp_tc_wgrad5x5", _ptr(self.dg_all[li]), _ptr(self.xh_all[li]), self.Kpad[li], S * B, h, w, cx, 4 * C,
                 _ptr(e.g[name + "/W"]), _ptr(wsb), wsb.numel(), e._s())

    def wgrad_jobs(self, jobs, wsb):
        """Deferred weight-gradient jobs on the CURRENT stream: ConvLSTM layer index, "deconv" (enc4/5/6) or "s2" (enc1/2)."""
        for j in jobs:
            if j == "deconv":
                self.deconv_wgrad_all(wsb)
            elif j == "s2":
                self.conv_s2_wgrad_all(wsb)
            else:
                self._lstm_wgrad(j, wsb)

    def wgrad_early(self, stream_a, stream_b):
        """Called by the backward pipeline when its decoder half is done (all gate gradients of lstm5-7 and the dY of enc4-6 exist) while the
        encoder half of the last time step still runs: the decoder-side weight gradients start on the two idle pipeline streams, with
        workspaces of their own, and are joined with the rest in wgrad_all()."""
        if len(self.wg_streams) != 2 or not self.early_on:
            return
        with torch.cuda.stream(stream_a):
            self.wgrad_jobs([6, 4], self.wg_ws_early[0])
        with torch.cuda.stream(stream_b):
            self.wgrad_jobs([5, "deconv"], self.wg_ws_early[1])
        self._early = {6, 4, 5, "deconv"}

    def wgrad_all(self, grad_sync=None):
        """After BPTT: weight and bias gradients of all seven ConvLSTM convolutions, each as ONE GEMM over all time steps.
        Data parallel (``grad_sync``): the small encoder / decoder gradients go first and are all-reduced as one block, then the ConvLSTM
        layers from the largest parameter tensor to the smallest, each layer's all-reduce running under the next layer's GEMM, so only the
        smallest tensor's reduction (0.8 MB) is exposed behind the last GEMM."""
        e = self.eng
        lstm_wgrad = self._lstm_wgrad
        early = self._early
        self._early = set()
        if grad_sync is not None:
            self.deconv_wgrad_all()
            self.conv_s2_wgrad_all()
            grad_sync.ready("enc")
            for li in sorted(range(7), key=lambda li: -(LSTM_IN[li] + LSTM_SIZES[li]) * LSTM_SIZES[li]):
                lstm_wgrad(li, self.wgrad_ws)
                grad_sync.ready("lstm%d" % (li + 1))
            return
        if self.wg_streams:
            # The twelve deferred weight-gradient GEMMs are independent of one another: issued on parallel branches (forked side streams,
            # one split-K workspace each; parallel branches of the captured graph) a GEMM's tail -- its last partial wave and its split-K
            # reduce -- overlaps the head of a GEMM on another branch instead of leaving SMs idle.  Jobs balanced by measured duration.
            # Jobs in `early` were already issued by the backward pipeline beside its last stage (wgrad_early).
            cur = torch.cuda.current_stream(e.dev)
            if early:
                branches = [[0, 2], [1, "s2"], [3]] if len(self.wg_streams) == 2 else [[0, 2, 3], [1, "s2"]]
            else:
                branches = [[6, 0, 2], [5, 1, 4], [3, "deconv", "s2"]] if len(self.wg_streams) == 2 else [[6, 0, 2, 3], [5, 1, 4, "deconv", "s2"]]
            for sd in self.wg_streams:
                sd.wait_stream(cur)
            for k, jobs in enumerate(branches):
                wsb = self.wgrad_ws if k == 0 else self.wg_ws[k - 1]
                if k == 0:
                    self.wgrad_jobs(jobs, wsb)
                else:
                    with torch.cuda.stream(self.wg_streams[k - 1]):
                        self.wgrad_jobs(jobs, wsb)
            for sd in self.wg_streams:
                cur.wait_stream(sd)
            return
        for li in range(7):
            if li not in early:
                lstm_wgrad(li, self.wgrad_ws)
        if "deconv" not in early:
            self.deconv_wgrad_all()
        self.conv_s2_wgrad_all()
