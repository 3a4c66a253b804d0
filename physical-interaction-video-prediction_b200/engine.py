"""Forward / backward orchestration of the training step over libpivp.so.

This is the host side of ``Model.__call__`` (train_model.py:620-764) and of ``loss.backward()``
(train_model.py:950): an explicit time loop forward that keeps every activation the reverse sweep needs,
and an explicit reverse-time loop (BPTT) that launches the backward kernels.  torch is used ONLY to own
device memory and to provide the CUDA stream; every arithmetic operation is a libpivp.so kernel.
There is no CPU / PyTorch fallback: if the library is missing, construction fails.

Buffers (NHWC views, see include/pivp.h).  ``xhL[t]`` holds the concatenated ConvLSTM input of layer L at
time t: channels [0,Cin) = layer input x_t, channels [Cin,Cin+C) = h_{t-1}; the gate kernel of step t writes
h_t straight into ``xhL[t+1]``, so the reference's F.concat (train_model.py:262) never materialises.
"""
import math
import os

import numpy as np
import torch

from . import layout
from ._lib import lib, PivpError

LSTM_SIZES = layout.LSTM_SIZES
LSTM_IN = layout.LSTM_IN
# spatial level of each ConvLSTM layer (divisor of H, W)
LSTM_LEVEL = (2, 2, 4, 4, 8, 4, 2)
LN_OF_LSTM = ("hidden1", "hidden2", "hidden3", "hidden4", "hidden5", "hidden6", "hidden7")


class View(object):
    """(tensor, row stride, channel offset, channels) -- an NHWC slice."""
    __slots__ = ("t", "cs", "co", "C")

    def __init__(self, t, cs, co, C):
        self.t, self.cs, self.co, self.C = t, cs, co, C

    @property
    def ptr(self):
        return self.t.data_ptr()


def _ptr(t):
    return 0 if t is None else t.data_ptr()


class Engine(object):
    def __init__(self, model_type="CDNA", num_masks=10, use_state=True, height=64, width=64, context_frames=2,
                 device="cuda", compute="f32", stp_oob="zeros", params=None):
        """``params``: the flat parameter buffer of another engine of the same configuration, shared by reference (a forward-only engine:
        the parameters are not re-initialised and no gradient buffer is allocated).  None: own parameters, LeCun-normal initialised."""
        if model_type not in ("CDNA", "DNA", "STP"):
            raise ValueError("No network specified")
        if model_type == "DNA" and num_masks != 1:
            raise ValueError("Only one mask is supported for DNA model.")          # train_model.py:389-390
        if height % 8 or width % 8:
            raise ValueError("height and width must be multiples of 8")
        if compute not in ("f32", "bf16"):
            raise ValueError("compute must be 'f32' or 'bf16'")
        self.L = lib()                                   # raises if libpivp.so is absent: no fallback
        if not torch.cuda.is_available():
            raise PivpError("a CUDA device is required: this path has no CPU fallback")
        self.model_type, self.M, self.use_state = model_type, int(num_masks), bool(use_state)
        self.H, self.W, self.ctx = int(height), int(width), int(context_frames)
        self.dev = torch.device(device)
        self.compute = compute
        self.oob = 1 if stp_oob == "border" else 0
        self.Ne = {"CDNA": 3, "DNA": 25, "STP": 3}[model_type]
        self.M1 = self.M + 1
        self.Nh = self.Ne + self.M1
        self.sa = 10 if self.use_state else 0
        self.cs3 = (64 + self.sa + 3) // 4 * 4          # row stride of the enc3 input [enc2 out | smear]: 74 channels in 76-float rows (16-B aligned)
        self.specs, self.nparam = layout.param_specs(model_type, self.M, self.use_state, self.H, self.W)
        self.spec = {s.name: s for s in self.specs}
        self.ws = None
        self.tc = None                                   # tensor-core (bf16) plan, created lazily
        self.grad_sync = None                            # parallel.GradSync when the all-reduce is overlapped with the deferred weight gradients
        if params is not None:
            if params.numel() != self.nparam or params.dtype != torch.float32 or not params.is_cuda:
                raise ValueError("params: a CUDA float32 buffer of %d parameters is required" % self.nparam)
            self.flat_p, self.flat_g = params, None
            self.p = {s.name: self.flat_p[s.offset:s.offset + s.size] for s in self.specs}
            self.g = {}
            return
        self.flat_p = torch.zeros(self.nparam, dtype=torch.float32, device=self.dev)
        self.flat_g = torch.zeros(self.nparam, dtype=torch.float32, device=self.dev)
        self.p = {s.name: self.flat_p[s.offset:s.offset + s.size] for s in self.specs}
        self.g = {s.name: self.flat_g[s.offset:s.offset + s.size] for s in self.specs}
        self.load_chainer_params(layout.lecun_normal_init(self.specs))

    # ------------------------------------------------------------------ parameters
    def load_chainer_params(self, params):
        """params: dict Chainer path -> ndarray in Chainer layout (A.9)."""
        host = np.zeros(self.nparam, np.float32)
        for s in self.specs:
            if s.name not in params:
                raise KeyError("missing parameter %s" % s.name)
            host[s.offset:s.offset + s.size] = s.to_internal(params[s.name]).reshape(-1)
        self.flat_p.copy_(torch.from_numpy(host))
        self.params_changed()

    def export_chainer(self, flat):
        host = flat.detach().cpu().numpy()
        return {s.name: s.to_chainer(host[s.offset:s.offset + s.size]) for s in self.specs}

    def chainer_params(self):
        return self.export_chainer(self.flat_p)

    def chainer_grads(self):
        return self.export_chainer(self.flat_g)

    def params_changed(self):
        if self.tc is not None:
            self.tc.refresh_weights()

    # ------------------------------------------------------------------ workspace
    def _alloc(self, *shape, zero=False, dtype=torch.float32):
        f = torch.zeros if zero else torch.empty
        return f(*shape, dtype=dtype, device=self.dev)

    def _workspace(self, B, T):
        if self.ws is not None and self.ws["B"] == B and self.ws["T"] == T:
            return self.ws
        H, W = self.H, self.W
        ws = {"B": B, "T": T}
        HW = {1: H * W, 2: (H // 2) * (W // 2), 4: (H // 4) * (W // 4), 8: (H // 8) * (W // 8)}
        Mr = {k: B * v for k, v in HW.items()}
        ws["HW"], ws["Mr"] = HW, Mr
        A = self._alloc
        S = T - 1
        # inputs of the four encoder convolutions, stacked over time: their weight gradients are ONE launch each over all T-1 steps
        stack = lambda rows, ch: (lambda t_: [t_[i] for i in range(S)])(A(S, rows, ch))
        ws["img_nhwc"] = stack(Mr[1], 3)
        ws["enc0_pre"] = [A(Mr[2], 32) for _ in range(S)]
        ws["xh"], ws["G"], ws["c"] = [], [], []
        for cin, c, lv in zip(LSTM_IN, LSTM_SIZES, LSTM_LEVEL):
            ws["xh"].append([A(Mr[lv], cin + c, zero=(t == 0)) for t in range(T)])     # xh[.][0] h-slot = zeros
            # activated gates saved for BPTT: fp32 here; in bf16 mode they live (as bf16) in TensorCorePlan.dg_bf16 instead
            ws["G"].append([A(Mr[lv], 4 * c) if self.compute == "f32" else None for _ in range(S)])
            ws["c"].append([A(Mr[lv], c) for _ in range(S)])
        ws["hid2"] = stack(Mr[2], 32)
        ws["hid4"] = stack(Mr[4], 64)
        ws["in3"] = stack(Mr[8], self.cs3)
        ws["hid5"] = stack(Mr[8], 128)                 # stacked over time: operand of the deferred kernel-Linear weight gradient
        ws["cat5"] = [A(Mr[4], 96) for _ in range(S)]
        ws["cat6"] = [A(Mr[2], 64) for _ in range(S)]
        ws["e6pre"] = [A(Mr[1], 64) for _ in range(S)]
        ws["e6"] = [A(Mr[1], 64) for _ in range(S)]
        ws["head"] = [A(Mr[1], self.Nh) for _ in range(S)]
        ws["enc7_pre"] = [A(B, self.Ne, H, W) for _ in range(S)]
        ws["mask_pre"] = [A(B, self.M1, H, W) for _ in range(S)]
        ws["gen"] = [A(B, 3, H, W) for _ in range(S)]
        ws["prev_buf"] = [A(B, 3, H, W) for _ in range(S)]
        ws["sa"] = [A(B, 10) for _ in range(S)]
        ws["cur"] = [A(B, 5) for _ in range(T)]
        ws["ln_stats"] = {name: [A(B, 2) for _ in range(S)] for name in
                          ("norm_enc0", "norm_enc6") + LN_OF_LSTM}
        if self.model_type == "CDNA":
            ws["kern_raw"] = [A(B, 25 * self.M) for _ in range(S)]
        elif self.model_type == "STP":
            ws["stp_s"] = [A(B, 100) for _ in range(S)]
            ws["theta_raw"] = [A(B, 6) for _ in range(S)]
        ws["take"] = torch.zeros(S, B, dtype=torch.int32, device=self.dev)
        # Per-step host <-> device hand-over goes through RINGS of pinned slots, one slot per step in flight, each guarded by an event:
        # the scheduled-sampling select travels host -> device (a stream-ordered copy in front of the step, NOT a node of the captured
        # graph, so the host may write step k+1's select while step k still runs) and the loss sums travel device -> host behind the
        # step (so every loss handle is bound to the numbers of ITS step, train_model.py:951-956).
        ws["take_host"] = torch.zeros(self.RING, S, B, dtype=torch.int32).pin_memory()
        ws["take_event"] = [None] * self.RING
        ws["loss_slots"] = A(2 * S, zero=True)
        ws["loss_host"] = torch.zeros(self.RING, 2 * S, dtype=torch.float32).pin_memory()
        ws["loss_event"] = [None] * self.RING
        ws["loss_owner"] = [None] * self.RING          # weak reference to the report that reads slot i (materialised before the slot is reused)
        ws["step_no"] = 0
        # ---- backward temporaries
        ws["dxh"] = [A(Mr[lv], cin + c) for cin, c, lv in zip(LSTM_IN, LSTM_SIZES, LSTM_LEVEL)]
        ws["dln"] = [A(Mr[lv], c) for c, lv in zip(LSTM_SIZES, LSTM_LEVEL)]
        ws["dc"] = [A(Mr[lv], c) for c, lv in zip(LSTM_SIZES, LSTM_LEVEL)]
        ws["d_gen"] = [A(B, 3, H, W, zero=True) for _ in range(S)]
        ws["d_gs"] = [A(B, 5, zero=True) for _ in range(S)]
        ws["d_cur"] = [A(B, 5), A(B, 5)]
        ws["d_e6"] = A(Mr[1], 64)
        ws["d_e6pre"] = A(Mr[1], 64)
        ws["d_head"] = A(Mr[1], self.Nh)
        ws["d_enc7_pre"] = A(B, self.Ne, H, W)
        ws["d_mask_pre"] = A(B, self.M1, H, W)
        ws["d_prev"] = A(B, 3, H, W)
        ws["d_img_nhwc"] = A(Mr[1], 3)
        # what crosses the stages of the backward pipeline (Engine.backward) is multi-buffered by time step
        ws["d_hid5"] = [A(Mr[8], 128), A(Mr[8], 128)]
        ws["d_cat6"] = [A(Mr[2], 64), A(Mr[2], 64), A(Mr[2], 64)]
        ws["d_cat5"] = [A(Mr[4], 96), A(Mr[4], 96)]
        ws["d_e5pre"] = A(Mr[2], 96)
        ws["d_e4pre"] = A(Mr[4], 128)
        ws["d_e3pre"] = stack(Mr[8], 64)               # d(pre-activation) of enc0..enc3 kept per time step for the deferred weight gradients
        ws["d_in3"] = [A(Mr[8], self.cs3), A(Mr[8], self.cs3)]
        ws["d_e2pre"] = stack(Mr[8], 64)
        ws["d_hid4"] = A(Mr[4], 64)
        ws["d_e1pre"] = stack(Mr[4], 32)
        ws["d_hid2"] = A(Mr[2], 32)
        ws["d_enc0pre"] = stack(Mr[2], 32)
        if self.model_type == "CDNA":
            ws["d_kern_raw"] = stack(B, 25 * self.M)   # kept per time step for the deferred kernel-Linear weight gradient
            nb = self.L.query("pivp_cdna_fused_bwd_workspace_bytes", B, H, W, self.M)
        elif self.model_type == "DNA":
            nb = self.L.query("pivp_dna_fused_bwd_workspace_bytes", B, H, W)
        else:
            ws["d_theta"] = A(B, 6)
            ws["d_stp_s"] = A(B, 100)
            nb = self.L.query("pivp_stp_fused_bwd_workspace_bytes", B, H, W, self.M)
        ws["fused_ws"] = torch.empty(nb, dtype=torch.uint8, device=self.dev)
        ws["lin_ws"] = torch.empty(max(16, self.L.query("pivp_linear_fwd_workspace_bytes", B, 128 * HW[8], max(25 * self.M, 100))),
                                   dtype=torch.uint8, device=self.dev)
        nb = self.L.query("pivp_layernorm_workspace_bytes", B, 64 * H * W)
        ws["ln_ws"] = torch.empty(max(nb, 16), dtype=torch.uint8, device=self.dev)
        ws["ln_ws_head"] = torch.empty(max(nb, 16), dtype=torch.uint8, device=self.dev)     # LayerNorm workspaces of the other two backward stages
        ws["ln_ws_upper"] = torch.empty(max(nb, 16), dtype=torch.uint8, device=self.dev)
        self.ws = ws
        if self.compute == "bf16":
            from .tensorcore import TensorCorePlan
            self.tc = TensorCorePlan(self, ws)
        return ws

    # ------------------------------------------------------------------ parallel branches
    # The step is one dependent chain of ~780 small kernels, but a few pieces hang off it sideways: the kernel Linear (needs hidden5, is
    # needed only by the transform at the end of the time step), its input gradient (needed only when BPTT reaches enc4), the loss
    # reductions, the deferred weight gradients.  They are issued on forked side streams (``with self._fork(k): ...``) and joined where
    # their result is consumed; under CUDA-graph capture fork / join become parallel branches of the graph, so these kernels fill SMs the
    # chain leaves idle instead of lengthening it.
    def _side(self, k):
        if not hasattr(self, "_side_streams"):
            import os
            self._side_streams = {}
            # branch ids: 0 kernel Linear (forward / backward), 1 loss terms, 2 small deferred weight gradients.  Measured on the b32 step
            # (one id at a time, against 8.353 ms with none): 0 -> 8.248, 1 -> 8.274, 2 -> 8.280 ms.  (Also measured: the eight bf16
            # weight-refresh launches behind Adam on three branches -> 8.57 ms, WORSE -- the forks delay the first kernels of the next
            # step -- so they stay on the main chain.)  PIVP_BRANCHES="" keeps everything on one stream.
            # 3: the backward pipeline (Engine.backward); 5: bf16 / fp32 copies of the two skip connections (forward).
            self._branches = set(int(v) for v in os.environ.get("PIVP_BRANCHES", "0,1,2,3,5").split(",") if v.strip() != "")
        if k not in self._side_streams:
            self._side_streams[k] = torch.cuda.Stream(device=self.dev)
        return self._side_streams[k]

    def _fork(self, k):
        """Context manager: work inside runs on side stream k, ordered after everything issued on the current stream so far."""
        import contextlib
        side = self._side(k)
        if k not in self._branches:
            return contextlib.nullcontext()
        side.wait_stream(torch.cuda.current_stream(self.dev))
        return torch.cuda.stream(side)

    def _join(self, k):
        """The current stream waits for side stream k."""
        side = self._side(k)
        if k in self._branches:
            torch.cuda.current_stream(self.dev).wait_stream(side)

    # ------------------------------------------------------------------ thin kernel wrappers
    def _s(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def _conv_fwd(self, x, B, H, W, w, b, N, k, stride, pad, y, relu=0, acc=0):
        Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
        self.L.call("pivp_conv2d_fwd", x.ptr, x.cs, x.co, B, H, W, x.C, _ptr(w), _ptr(b), N, k, k, stride, pad,
                    y.ptr, y.cs, y.co, Ho, Wo, relu, acc, self._s())

    def _conv_dgrad(self, dy, B, Ho, Wo, w, b, k, stride, pad, dx, H, W, relu=0, acc=0):
        self.L.call("pivp_conv2d_dgrad", dy.ptr, dy.cs, dy.co, B, Ho, Wo, dy.C, _ptr(w), _ptr(b), k, k, stride, pad,
                    dx.ptr, dx.cs, dx.co, H, W, dx.C, relu, acc, self._s())

    def _conv_wgrad(self, x, B, H, W, dy, Ho, Wo, k, stride, pad, dw, db):
        self.L.call("pivp_conv2d_wgrad", x.ptr, x.cs, x.co, B, H, W, x.C, dy.ptr, dy.cs, dy.co, Ho, Wo, dy.C,
                    k, k, stride, pad, _ptr(dw), _ptr(db), self._s())

    def _ln_fwd(self, name, x, B, HW, y, y2, relu, stats, y_bf16=None, have_stats=False, s2d=None):
        """``s2d`` = (map width, channel block): the bf16 copy is written in the space-to-depth layout of the stride-2 convolution that reads it."""
        ws = self.ws
        relu = relu | (2 if have_stats else 0)          # bit 1: the producing tcgen05 epilogue already wrote the (mean, M2) partials
        s2d_w, s2d_cb = (0, 0) if s2d is None else s2d
        self.L.call("pivp_layernorm_fwd_s2d", x.ptr, x.cs, x.co, _ptr(self.p[name + "/norm/gamma"]), _ptr(self.p[name + "/norm/beta"]),
                    B, HW, x.C, 1e-6, y.ptr, y.cs, y.co, 0 if y2 is None else y2.ptr, 0 if y2 is None else y2.cs,
                    0 if y2 is None else y2.co, 0 if y_bf16 is None else y_bf16.ptr, 0 if y_bf16 is None else y_bf16.cs,
                    0 if y_bf16 is None else y_bf16.co, relu, _ptr(stats), _ptr(ws["ln_ws"]), ws["ln_ws"].numel(), s2d_w, s2d_cb, self._s())

    def _ln_bwd(self, name, x, g1, g2, B, HW, relu, stats, dx, ln_ws=None, handover=None):
        """``handover`` = (bf16 tensor, row stride, map width, channel block, bias-gradient tensor): dx leaves as the space-to-depth bf16 operand of
        the transposed convolution below this LayerNorm plus that convolution's bias gradient (dx may then be None)."""
        ws = self.ws
        ln_ws = ws["ln_ws"] if ln_ws is None else ln_ws
        ho = (0, 0, 0, 0, 0, 0) if handover is None else (_ptr(handover[0]), handover[1], 0, handover[2], handover[3], _ptr(handover[4]))
        self.L.call("pivp_layernorm_bwd_handover", x.ptr, x.cs, x.co, g1.ptr, g1.cs, g1.co, 0 if g2 is None else g2.ptr,
                    0 if g2 is None else g2.cs, 0 if g2 is None else g2.co, _ptr(self.p[name + "/norm/gamma"]),
                    _ptr(self.p[name + "/norm/beta"]), _ptr(stats), B, HW, x.C, relu, 0 if dx is None else dx.ptr, 0 if dx is None else dx.cs,
                    0 if dx is None else dx.co, _ptr(self.g[name + "/norm/gamma"]), _ptr(self.g[name + "/norm/beta"]), _ptr(ln_ws),
                    ln_ws.numel(), *ho, self._s())

    def _ln_lstm_bwd(self, name, li, t, x, g1, g2, B, HW, last, ln_ws=None):
        """LayerNorm backward of ConvLSTM layer li's output at step t, then the layer's gate / input-gradient backward.
        Tensor-core mode: ONE kernel does the LayerNorm dx and the gate backward (d h_t never reaches memory), then the tcgen05 dgrad."""
        ws = self.ws
        ln_ws = ws["ln_ws"] if ln_ws is None else ln_ws
        cin, C, lv = LSTM_IN[li], LSTM_SIZES[li], LSTM_LEVEL[li]
        if self.tc is None:
            self._ln_bwd(name, x, g1, g2, B, HW, 0, ws["ln_stats"][name][t], View(ws["dln"][li], C, 0, C), ln_ws=ln_ws)
            self._lstm_bwd(li, t, B, last)
            return
        dgb = self.tc.dg_bf16[li][t]
        self.L.call("pivp_layernorm_bwd_lstm", x.ptr, x.cs, x.co, g1.ptr, g1.cs, g1.co, 0 if g2 is None else g2.ptr,
                    0 if g2 is None else g2.cs, 0 if g2 is None else g2.co, _ptr(self.p[name + "/norm/gamma"]),
                    _ptr(self.p[name + "/norm/beta"]), _ptr(ws["ln_stats"][name][t]), B, HW, C,
                    _ptr(self.g[name + "/norm/gamma"]), _ptr(self.g[name + "/norm/beta"]), _ptr(dgb),
                    _ptr(ws["c"][li][t - 1]) if t > 0 else 0, _ptr(ws["c"][li][t]), 0 if last else _ptr(ws["dxh"][li]), cin + C, cin,
                    _ptr(ws["dc"][li]), 0 if last else 1, _ptr(ln_ws), ln_ws.numel(), self._s())
        self.tc.lstm_dgrad(li, t)

    def _relu_bwd(self, out, ga, gb, dst, M):
        self.L.call("pivp_relu_bwd", out.ptr, out.cs, out.co, ga.ptr, ga.cs, ga.co, 0 if gb is None else gb.ptr,
                    0 if gb is None else gb.cs, 0 if gb is None else gb.co, dst.ptr, dst.cs, dst.co, M, dst.C, self._s())

    # ------------------------------------------------------------------ ConvLSTM layer (fwd / bwd)
    def _lstm_ln_fwd(self, li, t, B, name, y, y_bf16=None, s2d=None):
        """ConvLSTM layer li at step t followed by the LayerNorm `name` of its output h_t (train_model.py:596-601): one kernel on the tensor-core
        path when the launch fits (TensorCorePlan.ln_fusable), else the cell and then the LayerNorm kernel(s)."""
        ws = self.ws
        cin, C, lv = LSTM_IN[li], LSTM_SIZES[li], LSTM_LEVEL[li]
        stats = ws["ln_stats"][name][t]
        if self.tc is not None and self.tc.ln_fusable(li) and s2d is None:
            self.tc.lstm_fwd(li, t, ln=(name, y, y_bf16, stats))
            return
        self._lstm_fwd(li, t, B)
        self._ln_fwd(name, View(ws["xh"][li][t + 1], cin + C, cin, C), B, ws["HW"][lv], y, None, 0, stats, y_bf16,
                     have_stats=self.tc is not None and self.tc.ln_fused[li], s2d=s2d)

    def _lstm_fwd(self, li, t, B):
        ws = self.ws
        cin, C, lv = LSTM_IN[li], LSTM_SIZES[li], LSTM_LEVEL[li]
        h, w = self.H // lv, self.W // lv
        name = "lstm%d/conv" % (li + 1)
        xh, Gt = ws["xh"][li][t], ws["G"][li][t]
        if self.tc is not None:
            self.tc.lstm_fwd(li, t)            # conv + bias + gates + cell + h in ONE tcgen05 kernel
            return
        self._conv_fwd(View(xh, cin + C, 0, cin + C), B, h, w, self.p[name + "/W"], self.p[name + "/b"], 4 * C, 5, 1, 2,
                       View(Gt, 4 * C, 0, 4 * C))
        self.L.call("pivp_lstm_gates_fwd", _ptr(Gt), _ptr(ws["c"][li][t - 1]) if t > 0 else 0, _ptr(ws["c"][li][t]),
                    _ptr(ws["xh"][li][t + 1]), cin + C, cin, 0, 0, 0, ws["Mr"][lv], C, 1.0, self._s())

    def _lstm_bwd(self, li, t, B, last):
        """dln[li] holds the LN-path gradient of h_t; dxh[li] (from step t+1) holds d h_t via the recurrent input."""
        ws = self.ws
        cin, C, lv = LSTM_IN[li], LSTM_SIZES[li], LSTM_LEVEL[li]
        h, w = self.H // lv, self.W // lv
        name = "lstm%d/conv" % (li + 1)
        Gt, dxh = ws["G"][li][t], ws["dxh"][li]
        if self.tc is not None:       # bf16 mode: gates were stored bf16 in dg_bf16[li][t]; dG overwrites them in place
            dgb = self.tc.dg_bf16[li][t]
            self.L.call("pivp_lstm_gates_bwd_bf16", _ptr(dgb), _ptr(ws["c"][li][t - 1]) if t > 0 else 0, _ptr(ws["c"][li][t]),
                        _ptr(ws["dln"][li]), 0 if last else _ptr(dxh), cin + C, cin, _ptr(ws["dc"][li]), 0 if last else 1,
                        _ptr(dgb), ws["Mr"][lv], C, self._s())
        else:
            self.L.call("pivp_lstm_gates_bwd", _ptr(Gt), _ptr(ws["c"][li][t - 1]) if t > 0 else 0, _ptr(ws["c"][li][t]),
                        _ptr(ws["dln"][li]), 0 if last else _ptr(dxh), cin + C, cin, _ptr(ws["dc"][li]), 0 if last else 1,
                        0, ws["Mr"][lv], C, self._s())
        dG = View(Gt, 4 * C, 0, 4 * C)
        xh = View(ws["xh"][li][t], cin + C, 0, cin + C)
        if self.tc is not None:
            self.tc.lstm_dgrad(li, t)          # dxh = conv(dG_bf16, tap-flipped W) on tcgen05; wgrad is deferred (wgrad_all)
        else:
            self._conv_wgrad(xh, B, h, w, dG, h, w, 5, 1, 2, self.g[name + "/W"], self.g[name + "/b"])
            self._conv_dgrad(dG, B, h, w, self.p[name + "/W"], None, 5, 1, 2, View(dxh, cin + C, 0, cin + C), h, w)

    # ------------------------------------------------------------------ forward
    RING = 4                                            # steps that may be in flight between the host and the device

    def stage_schedule(self, take_gt):
        """Host part of a step: put the scheduled-sampling select (int32 (T-1,B)) into the next pinned ring slot and queue its copy
        into the device buffer the step reads, on the current stream.  The slot is reused RING steps later, after the event recorded
        behind its copy has fired, so a caller that does not synchronise every step can never overwrite a select that is still to be read."""
        ws = self.ws
        slot = ws["step_no"] % self.RING
        ev = ws["take_event"][slot]
        if ev is not None:
            ev.synchronize()
        else:
            ev = ws["take_event"][slot] = torch.cuda.Event()
        ws["take_host"][slot].copy_(torch.from_numpy(np.ascontiguousarray(take_gt, dtype=np.int32)))
        ws["take"].copy_(ws["take_host"][slot], non_blocking=True)
        ev.record(torch.cuda.current_stream(self.dev))

    def snapshot_loss(self, owner=None):
        """Device -> host copy of this step's loss sums into a pinned ring slot (stream-ordered behind the step, no synchronisation here).
        Returns a reader ``() -> (loss, psnr_all, recon_costs)`` bound to THIS step's numbers: it waits for the slot's event only."""
        import weakref
        ws = self.ws
        slot = ws["step_no"] % self.RING
        ws["step_no"] += 1
        old = ws["loss_owner"][slot]
        old = old() if old is not None else None
        if old is not None:
            old()                                       # a report RING steps old that nobody read yet: materialise it before its slot is reused
        ev = ws["loss_event"][slot]
        if ev is None:
            ev = ws["loss_event"][slot] = torch.cuda.Event()
        ws["loss_host"][slot].copy_(ws["loss_slots"], non_blocking=True)
        ev.record(torch.cuda.current_stream(self.dev))
        T, B = self.T, self.B
        cache = {}

        def read():
            if not cache:
                ev.synchronize()
                cache["v"] = self.loss_values(ws["loss_host"][slot].numpy().copy(), T, B)
            return cache["v"]
        ws["loss_owner"][slot] = weakref.ref(read)
        return read

    def forward(self, images, actions, states, take_gt=None, feedself=True):
        """images (T,B,3,H,W), actions/states (T,B,5) fp32 CUDA tensors.  ``take_gt``: int32 (T-1,B) host array with the
        scheduled-sampling select for steps t >= ctx (rows before are ignored) or None when ``feedself``."""
        self._workspace(int(images.shape[1]), int(images.shape[0]))
        if not feedself:
            self.stage_schedule(take_gt)
        return self.forward_device(images, actions, states, feedself)

    def forward_device(self, images, actions, states, feedself=True, steps=None, loss=True):
        """Device part of the forward pass: stream-ordered work only (CUDA-graph capturable).
        ``steps``: sequence length T when ``images`` holds the context frames only (feedself reads images[t] for t < context_frames);
        ``loss=False``: no loss terms (states[0] is then the only state read)."""
        T, B = int(images.shape[0]) if steps is None else int(steps), int(images.shape[1])
        H, W = self.H, self.W
        assert images.shape[2:] == (3, H, W) and images.dtype == torch.float32 and images.is_contiguous()
        ws = self._workspace(B, T)
        L, s = self.L, self._s()
        HW, Mr = ws["HW"], ws["Mr"]
        self.feedself = bool(feedself)
        self.images, self.states = images, states
        ws["cur"][0].copy_(states[0])
        if loss:
            ws["loss_slots"].zero_()
        self.prev = []
        p = self.p
        n_img, n_sta = B * 3 * H * W, B * 5
        div = float(T - self.ctx)
        for t in range(T - 1):
            # ---- previous frame (train_model.py:663-673)
            if t < self.ctx:
                prev = images[t]
            elif feedself:
                prev = ws["gen"][t - 1]
            else:
                prev = ws["prev_buf"][t]             # the select also writes the NHWC rows enc0 reads (no nchw_to_nhwc launch on this path)
                L.call("pivp_sched_select_nhwc", _ptr(images[t]), _ptr(ws["gen"][t - 1]), _ptr(ws["take"][t]), _ptr(prev),
                       _ptr(ws["img_nhwc"][t]), B, 3, HW[1], s)
            self.prev.append(prev)
            # state predictor + smear (train_model.py:563-565, 676, 730): needs the action and the previous state only -> side branch 5;
            # it fills the smear columns of enc3's input, enc2 fills the others; joined in front of enc3
            with self._fork(5):
                L.call("pivp_state_fwd", _ptr(actions[t]), _ptr(ws["cur"][t]), _ptr(p["current_state/W"]), _ptr(p["current_state/b"]),
                       _ptr(ws["sa"][t]), _ptr(ws["cur"][t + 1]), _ptr(ws["in3"][t]) if self.use_state else 0, self.cs3, 64,
                       HW[8], B, self._s())
            if t < self.ctx or feedself:
                L.call("pivp_nchw_to_nhwc", _ptr(prev), _ptr(ws["img_nhwc"][t]), 3, 0, B, 3, HW[1], s)
            # ---- group 0: enc0 -> LN -> relu  (goes to lstm1's x slot and to the enc6 skip slot)
            self._conv_fwd(View(ws["img_nhwc"][t], 3, 0, 3), B, H, W, p["enc0/W"], p["enc0/b"], 32, 5, 2, 2,
                           View(ws["enc0_pre"][t], 32, 0, 32))
            self._ln_fwd("norm_enc0", View(ws["enc0_pre"][t], 32, 0, 32), B, HW[2], View(ws["xh"][0][t], 64, 0, 32),
                         View(ws["cat6"][t], 64, 32, 32), 1, ws["ln_stats"]["norm_enc0"][t],
                         None if self.tc is None else self.tc.xview(0, t))
            if self.tc is not None:
                with self._fork(5):            # bf16 copy of the enc0 skip: needed by the enc6 deconvolution at the end of the step only
                    L.call("pivp_copy_view", _ptr(ws["cat6"][t]), 64, 32, 0, 0, 0, _ptr(self.tc.cat6_b[t]), 64, 32, Mr[2], 32, self._s())
            # ---- group 1
            self._lstm_ln_fwd(0, t, B, "hidden1", View(ws["xh"][1][t], 64, 0, 32), None if self.tc is None else self.tc.xview(1, t))
            if self.tc is not None:       # the LayerNorm writes enc1's GEMM operand itself: bf16, space-to-depth (no separate cast launch)
                self._lstm_ln_fwd(1, t, B, "hidden2", View(ws["hid2"][t], 32, 0, 32), *self.tc.s2d_operand("enc1", t, W // 2))
            else:
                self._lstm_ln_fwd(1, t, B, "hidden2", View(ws["hid2"][t], 32, 0, 32))
            if self.tc is not None:       # stride-2 conv as a 9-tap tcgen05 GEMM on the space-to-depth bf16 input; bf16 x slot from the epilogue
                self.tc.conv_s2_fwd("enc1", t, None, 32, ws["xh"][2][t], 96, self.tc.xview(2, t).t, self.tc.Kpad[2])
                with self._fork(5):            # enc1 skip (fp32 + bf16): needed by the enc5 deconvolution only
                    L.call("pivp_copy_view", _ptr(ws["xh"][2][t]), 96, 0, _ptr(ws["cat5"][t]), 96, 64, _ptr(self.tc.cat5_b[t]), 128, 64, Mr[4], 32, self._s())
            else:
                self._conv_fwd(View(ws["hid2"][t], 32, 0, 32), B, H // 2, W // 2, p["enc1/W"], p["enc1/b"], 32, 3, 2, 1,
                               View(ws["xh"][2][t], 96, 0, 32), relu=1)
                with self._fork(5):
                    L.call("pivp_copy_view", _ptr(ws["xh"][2][t]), 96, 0, _ptr(ws["cat5"][t]), 96, 64, 0, 0, 0, Mr[4], 32, self._s())
            # ---- group 2
            self._lstm_ln_fwd(2, t, B, "hidden3", View(ws["xh"][3][t], 128, 0, 64), None if self.tc is None else self.tc.xview(3, t))
            if self.tc is not None:
                self._lstm_ln_fwd(3, t, B, "hidden4", View(ws["hid4"][t], 64, 0, 64), *self.tc.s2d_operand("enc2", t, W // 4))
                self.tc.conv_s2_fwd("enc2", t, None, 64, ws["in3"][t], self.cs3, None, 0)
            else:
                self._lstm_ln_fwd(3, t, B, "hidden4", View(ws["hid4"][t], 64, 0, 64))
                self._conv_fwd(View(ws["hid4"][t], 64, 0, 64), B, H // 4, W // 4, p["enc2/W"], p["enc2/b"], 64, 3, 2, 1,
                               View(ws["in3"][t], self.cs3, 0, 64), relu=1)
            # ---- group 3: enc3 on [enc2 out | smear]; the smear and the state predictor (train_model.py:676,730) ran on side branch 5
            self._join(5)
            self._conv_fwd(View(ws["in3"][t], self.cs3, 0, 64 + self.sa), B, H // 8, W // 8, p["enc3/W"], p["enc3/b"], 64, 1, 1, 0,
                           View(ws["xh"][4][t], 192, 0, 64), relu=1)
            if self.tc is not None:
                L.call("pivp_copy_view", _ptr(ws["xh"][4][t]), 192, 0, 0, 0, 0, self.tc.xview(4, t).ptr, self.tc.Kpad[4], 0, Mr[8], 64, s)
            # ---- group 4
            self._lstm_ln_fwd(4, t, B, "hidden5", View(ws["hid5"][t], 128, 0, 128), None if self.tc is None else View(self.tc.hid5_b[t], 128, 0, 128))
            # (the enc0 skip copy on branch 5 is joined with the enc1 skip above: same side stream, issued earlier)
            # the kernel / theta Linear needs hidden5 only and is consumed by the transform at the end of the step: side branch 0
            K5 = 128 * HW[8]
            with self._fork(0):
                s0 = self._s()
                if self.model_type == "CDNA":
                    L.call("pivp_linear_fwd_splitk", _ptr(ws["hid5"][t]), K5, _ptr(p["model/cdna_kerns/W"]), _ptr(p["model/cdna_kerns/b"]),
                           _ptr(ws["kern_raw"][t]), B, K5, 25 * self.M, 0, _ptr(ws["lin_ws"]), ws["lin_ws"].numel(), s0)
                elif self.model_type == "STP":
                    L.call("pivp_linear_fwd_splitk", _ptr(ws["hid5"][t]), K5, _ptr(p["model/stp_input/W"]), _ptr(p["model/stp_input/b"]),
                           _ptr(ws["stp_s"][t]), B, K5, 100, 1, _ptr(ws["lin_ws"]), ws["lin_ws"].numel(), s0)
                    L.call("pivp_linear_fwd", _ptr(ws["stp_s"][t]), 100, _ptr(p["model/identity_params/W"]),
                           _ptr(p["model/identity_params/b"]), _ptr(ws["theta_raw"][t]), B, 100, 6, 0, s0)
            if self.tc is not None:
                self.tc.deconv_fwd("enc4", self.tc.hid5_b[t], ws["xh"][5][t], 192, self.tc.xh_bf16[5][t], self.tc.Kpad[5], 1)
            else:
                self._conv_dgrad(View(ws["hid5"][t], 128, 0, 128), B, H // 8, W // 8, p["enc4/W"], p["enc4/b"], 3, 2, 1,
                                 View(ws["xh"][5][t], 192, 0, 128), H // 4, W // 4, relu=1)
            # ---- group 5
            self._lstm_ln_fwd(5, t, B, "hidden6", View(ws["cat5"][t], 96, 0, 64), None if self.tc is None else View(self.tc.cat5_b[t], 128, 0, 64))
            self._join(5)                              # the enc1 skip copies
            if self.tc is not None:
                self.tc.deconv_fwd("enc5", self.tc.cat5_b[t], ws["xh"][6][t], 128, self.tc.xh_bf16[6][t], self.tc.Kpad[6], 1)
            else:
                self._conv_dgrad(View(ws["cat5"][t], 96, 0, 96), B, H // 4, W // 4, p["enc5/W"], p["enc5/b"], 3, 2, 1,
                                 View(ws["xh"][6][t], 128, 0, 96), H // 2, W // 2, relu=1)
            # ---- group 6
            self._lstm_ln_fwd(6, t, B, "hidden7", View(ws["cat6"][t], 64, 0, 32), None if self.tc is None else View(self.tc.cat6_b[t], 64, 0, 32))
            if self.tc is not None:
                e6_stats = ((H // 2) * (W // 2)) % 128 == 0          # the deconvolution's epilogue also writes norm_enc6's (mean, M2) partials
                self.tc.deconv_fwd("enc6", self.tc.cat6_b[t], ws["e6pre"][t], 64, None, 0, 0, ln_partial=ws["ln_ws"] if e6_stats else None)
            else:
                e6_stats = False
                self._conv_dgrad(View(ws["cat6"][t], 64, 0, 64), B, H // 2, W // 2, p["enc6/W"], p["enc6/b"], 3, 2, 1,
                                 View(ws["e6pre"][t], 64, 0, 64), H, W, relu=0)
            heads_ln = e6_stats and self.Nh in (14, 27) and os.environ.get("PIVP_HEADS_LN", "1") != "0"
            if not heads_ln:
                self._ln_fwd("norm_enc6", View(ws["e6pre"][t], 64, 0, 64), B, HW[1], View(ws["e6"][t], 64, 0, 64), None, 1,
                             ws["ln_stats"]["norm_enc6"][t], have_stats=e6_stats)
            # ---- heads (enc7 + masks 1x1), NCHW planes out
            if heads_ln:                  # norm_enc6 + ReLU applied while the heads kernel stages its tile (statistics from the enc6 epilogue)
                L.call("pivp_heads_fwd_ln", _ptr(ws["e6pre"][t]), 64, 0, _ptr(p["norm_enc6/norm/gamma"]), _ptr(p["norm_enc6/norm/beta"]),
                       _ptr(ws["ln_ws"]), 1e-6, _ptr(ws["ln_stats"]["norm_enc6"][t]), _ptr(ws["e6"][t]), 64, 0,
                       _ptr(p["model/enc7/W"]), _ptr(p["model/enc7/b"]), _ptr(ws["enc7_pre"][t]), self.Ne, _ptr(ws["mask_pre"][t]), self.Nh,
                       B, HW[1], s)
            elif self.Nh in (14, 27):     # fused heads: e6 read once, planes written directly (heads.cu)
                L.call("pivp_heads_fwd", _ptr(ws["e6"][t]), 64, 0, _ptr(p["model/enc7/W"]), _ptr(p["model/enc7/b"]),
                       _ptr(ws["enc7_pre"][t]), self.Ne, _ptr(ws["mask_pre"][t]), self.Nh, B, HW[1], s)
            else:
                self._conv_fwd(View(ws["e6"][t], 64, 0, 64), B, H, W, p["model/enc7/W"], p["model/enc7/b"], self.Nh, 1, 1, 0,
                               View(ws["head"][t], self.Nh, 0, self.Nh))
                L.call("pivp_nhwc_to_nchw", _ptr(ws["head"][t]), self.Nh, 0, _ptr(ws["enc7_pre"][t]), B, self.Ne, HW[1], 0, s)
                L.call("pivp_nhwc_to_nchw", _ptr(ws["head"][t]), self.Nh, self.Ne, _ptr(ws["mask_pre"][t]), B, self.M1, HW[1], 0, s)
            # ---- transform + masks + composite
            self._join(0)                                  # kernel / theta Linear of this step
            if self.model_type == "CDNA":
                L.call("pivp_cdna_fused_fwd", _ptr(prev), _ptr(ws["enc7_pre"][t]), _ptr(ws["mask_pre"][t]), _ptr(ws["kern_raw"][t]),
                       _ptr(ws["gen"][t]), B, H, W, self.M, s)
            elif self.model_type == "DNA":
                L.call("pivp_dna_fused_fwd", _ptr(prev), _ptr(ws["enc7_pre"][t]), _ptr(ws["mask_pre"][t]), _ptr(ws["gen"][t]), B, H, W, s)
            else:
                L.call("pivp_stp_fused_fwd", _ptr(prev), _ptr(ws["enc7_pre"][t]), _ptr(ws["mask_pre"][t]), _ptr(ws["theta_raw"][t]),
                       _ptr(ws["gen"][t]), B, H, W, self.M, self.oob, s)
            # ---- loss terms of this step (train_model.py:737-758) on side branch 1: sums to loss_slots, loss gradients to d_gen / d_gs
            if not loss:
                continue
            with self._fork(1):
                s1 = self._s()
                if t >= self.ctx - 1:
                    L.call("pivp_mse", _ptr(ws["gen"][t]), _ptr(images[t + 1]), n_img, 2.0 / (n_img * div), _ptr(ws["d_gen"][t]),
                           ws["loss_slots"][t:].data_ptr(), s1)
                    L.call("pivp_mse", _ptr(ws["cur"][t + 1]), _ptr(states[t + 1]), n_sta, 1e-4 * 2.0 / (n_sta * div), _ptr(ws["d_gs"][t]),
                           ws["loss_slots"][T - 1 + t:].data_ptr(), s1)
                else:
                    ws["d_gen"][t].zero_()
                    ws["d_gs"][t].zero_()
        if loss:
            self._join(1)
        self.T, self.B = T, B
        return ws["gen"]

    def loss_values(self, slots=None, T=None, B=None):
        """Host-side finish of train_model.py:739-758.  ``slots``: the step's loss sums on the host (snapshot_loss); None reads the
        device buffer directly (a D2H sync, like ref:955-956).  Returns (loss, psnr_all, recon_costs, state_costs)."""
        ws = self.ws
        T, B = (self.T if T is None else T), (self.B if B is None else B)
        if slots is None:
            slots = ws["loss_slots"].cpu().numpy()
        n_img, n_sta = np.float32(B * 3 * self.H * self.W), np.float32(B * 5)
        loss, psnr, recon, state = np.float32(0), 0.0, [], []
        for t in range(self.ctx - 1, T - 1):
            c = np.float32(slots[t]) / n_img
            recon.append(float(c))
            # ref:124-134: 10 log10(1 / MSE); an exact match (MSE == 0) is +inf there too (NumPy division), not an exception
            psnr += 10.0 * math.log(1.0 / float(c)) / math.log(10.0) if c > 0 else float("inf")
            loss = np.float32(loss + c)
        for t in range(self.ctx - 1, T - 1):
            sc = np.float32(slots[T - 1 + t]) / n_sta * np.float32(1e-4)
            state.append(float(sc))
            loss = np.float32(loss + sc)
        loss = np.float32(loss / np.float32(T - self.ctx))
        return float(loss), psnr, recon, state

    # ------------------------------------------------------------------ backward (BPTT)
    def _stop_after_step(self, t):
        """Hook for the stage-by-stage gradient diagnostics (scripts/dbg_bwd_stage.py subclasses Engine and overrides this to leave one
        step's backward temporaries in place).  The production engine never stops early."""
        return False

    def cleargrads(self):
        self.flat_g.zero_()

    def _bwd_head(self, t, inline):
        """The part of backward step t that hangs off the loss only (when the previous frame is detached, i.e. under scheduled sampling):
        fused transform backward, kernel / theta Linear input gradient, the two 1x1 heads, LayerNorm norm_enc6 and the enc6 deconvolution
        input gradient.  Its outputs for the recurrent chain are d_cat6[t % 3] (gradient of [hidden7 | enc0 skip]) and d_hid5[t & 1] (gradient
        of hidden5 through the Linear); everything else it touches is private to heads, which never overlap one another.
        ``inline``: the Linear runs on the head's own stream (the head itself is a side branch); else on side branch 0, joined at enc4."""
        import contextlib
        ws, L = self.ws, self.L
        s = self._s()
        T, B, H, W = self.T, self.B, self.H, self.W
        HW, Mr = ws["HW"], ws["Mr"]
        p, g = self.p, self.g
        K5 = 128 * HW[8]
        s2, s3 = t & 1, t % 3
        prev = self.prev[t]
        need_dprev = self.feedself and t >= self.ctx          # prev_t = gen_{t-1} keeps the graph (ref:664-666)
        d_prev = ws["d_prev"] if need_dprev else None
        # ---- fused transform backward
        if self.model_type == "CDNA":
            L.call("pivp_cdna_fused_bwd", _ptr(ws["d_gen"][t]), _ptr(prev), _ptr(ws["enc7_pre"][t]), _ptr(ws["mask_pre"][t]),
                   _ptr(ws["kern_raw"][t]), _ptr(ws["d_enc7_pre"]), _ptr(ws["d_mask_pre"]), _ptr(ws["d_kern_raw"][t]),
                   _ptr(d_prev), 0, B, H, W, self.M, _ptr(ws["fused_ws"]), ws["fused_ws"].numel(), s)
            with (contextlib.nullcontext() if inline else self._fork(0)):       # d hidden5 through the kernel Linear: needed only when BPTT reaches enc4
                L.call("pivp_linear_bwd", _ptr(ws["d_kern_raw"][t]), _ptr(ws["hid5"][t]), K5, _ptr(p["model/cdna_kerns/W"]),
                       _ptr(ws["d_hid5"][s2]), K5, 0, 0, 0, B, K5, 25 * self.M, self._s())       # dx only; dW / db after the time loop
            hid5_has_grad = True
        elif self.model_type == "DNA":
            L.call("pivp_dna_fused_bwd", _ptr(ws["d_gen"][t]), _ptr(prev), _ptr(ws["enc7_pre"][t]), _ptr(ws["mask_pre"][t]),
                   _ptr(ws["d_enc7_pre"]), _ptr(ws["d_mask_pre"]), _ptr(d_prev), 0, B, H, W, _ptr(ws["fused_ws"]),
                   ws["fused_ws"].numel(), s)
            hid5_has_grad = False
        else:
            if need_dprev:
                d_prev.zero_()
            L.call("pivp_stp_fused_bwd", _ptr(ws["d_gen"][t]), _ptr(prev), _ptr(ws["enc7_pre"][t]), _ptr(ws["mask_pre"][t]),
                   _ptr(ws["theta_raw"][t]), _ptr(ws["d_enc7_pre"]), _ptr(ws["d_mask_pre"]), _ptr(ws["d_theta"]), _ptr(d_prev),
                   B, H, W, self.M, self.oob, _ptr(ws["fused_ws"]), ws["fused_ws"].numel(), s)
            with (contextlib.nullcontext() if inline else self._fork(0)):
                s0 = self._s()
                L.call("pivp_linear_bwd", _ptr(ws["d_theta"]), _ptr(ws["stp_s"][t]), 100, _ptr(p["model/identity_params/W"]),
                       _ptr(ws["d_stp_s"]), 100, 0, _ptr(g["model/identity_params/W"]), _ptr(g["model/identity_params/b"]), B, 100, 6, s0)
                L.call("pivp_relu_mask", _ptr(ws["stp_s"][t]), _ptr(ws["d_stp_s"]), B * 100, s0)
                L.call("pivp_linear_bwd", _ptr(ws["d_stp_s"]), _ptr(ws["hid5"][t]), K5, _ptr(p["model/stp_input/W"]),
                       _ptr(ws["d_hid5"][s2]), K5, 0, _ptr(g["model/stp_input/W"]), _ptr(g["model/stp_input/b"]), B, K5, 100, s0)
            hid5_has_grad = True
        # ---- heads backward: planes -> NHWC, then 1x1 conv dgrad / wgrad
        if self.Nh in (14, 27):
            L.call("pivp_heads_bwd", _ptr(ws["e6"][t]), 64, 0, _ptr(p["model/enc7/W"]), _ptr(ws["d_enc7_pre"]), self.Ne,
                   _ptr(ws["d_mask_pre"]), self.Nh, _ptr(ws["d_e6"]), 64, 0, _ptr(g["model/enc7/W"]), _ptr(g["model/enc7/b"]),
                   B, HW[1], s)
        else:
            L.call("pivp_nchw_to_nhwc", _ptr(ws["d_enc7_pre"]), _ptr(ws["d_head"]), self.Nh, 0, B, self.Ne, HW[1], s)
            L.call("pivp_nchw_to_nhwc", _ptr(ws["d_mask_pre"]), _ptr(ws["d_head"]), self.Nh, self.Ne, B, self.M1, HW[1], s)
            dhead = View(ws["d_head"], self.Nh, 0, self.Nh)
            self._conv_wgrad(View(ws["e6"][t], 64, 0, 64), B, H, W, dhead, H, W, 1, 1, 0, g["model/enc7/W"], g["model/enc7/b"])
            self._conv_dgrad(dhead, B, H, W, p["model/enc7/W"], None, 1, 1, 0, View(ws["d_e6"], 64, 0, 64), H, W)
        # ---- norm_enc6 (+relu) and enc6 deconv
        de6 = View(ws["d_e6pre"], 64, 0, 64)
        ho = self.tc.deconv_handover("enc6", t, W, g["enc6/b"]) if (self.tc is not None and os.environ.get("PIVP_LN_HANDOVER", "1") != "0") else None
        self._ln_bwd("norm_enc6", View(ws["e6pre"][t], 64, 0, 64), View(ws["d_e6"], 64, 0, 64), None, B, HW[1], 1,
                     ws["ln_stats"]["norm_enc6"][t], None if ho is not None else de6, ln_ws=ws["ln_ws_head"], handover=ho)
        if self.tc is not None:           # bias gradient + bf16 space-to-depth operand: from the LayerNorm backward itself (or one hand-over launch)
            self.tc.deconv_bwd_fused("enc6", t, None, de6, None, g["enc6/b"], ws["d_cat6"][s3], 0, handover=ho is None)
        else:
            L.call("pivp_colsum", de6.ptr, 64, 0, Mr[1], 64, _ptr(g["enc6/b"]), s)
            self._conv_wgrad(de6, B, H, W, View(ws["cat6"][t], 64, 0, 64), H // 2, W // 2, 3, 2, 1, g["enc6/W"], None)
            self._conv_fwd(de6, B, H, W, p["enc6/W"], None, 64, 3, 2, 1, View(ws["d_cat6"][s3], 64, 0, 64))
        return hid5_has_grad

    def _bwd_upper(self, t, hid5_has_grad, inline_head, ln_ws):
        """Backward step t, decoder half: lstm7, enc5, lstm6, enc4, lstm5, enc3 and the state predictor.  Reads d_cat6 / d_hid5 of HEAD(t);
        hands d_in3 (gradient of [enc2 out | smear]) and d_cat5[:, 64:96] (the enc1 skip) to the encoder half."""
        ws, L = self.ws, self.L
        s = self._s()
        T, B, H, W = self.T, self.B, self.H, self.W
        HW, Mr = ws["HW"], ws["Mr"]
        p, g = self.p, self.g
        last = (t == T - 2)
        s2, s3 = t & 1, t % 3
        # ---- lstm7
        self._ln_lstm_bwd("hidden7", 6, t, View(ws["xh"][6][t + 1], 128, 96, 32), View(ws["d_cat6"][s3], 64, 0, 32), None, B, HW[2], last, ln_ws)
        # ---- enc5 deconv (input concat(hidden6, encs[1]))
        de5 = View(ws["d_e5pre"], 96, 0, 96)
        if self.tc is not None:
            self.tc.deconv_bwd_fused("enc5", t, View(ws["xh"][6][t], 128, 0, 96), View(ws["dxh"][6], 128, 0, 96), None, g["enc5/b"],
                                     ws["d_cat5"][s2], 0)
        else:
            self._relu_bwd(View(ws["xh"][6][t], 128, 0, 96), View(ws["dxh"][6], 128, 0, 96), None, de5, Mr[2])
            L.call("pivp_colsum", de5.ptr, 96, 0, Mr[2], 96, _ptr(g["enc5/b"]), s)
            self._conv_wgrad(de5, B, H // 2, W // 2, View(ws["cat5"][t], 96, 0, 96), H // 4, W // 4, 3, 2, 1, g["enc5/W"], None)
            self._conv_fwd(de5, B, H // 2, W // 2, p["enc5/W"], None, 96, 3, 2, 1, View(ws["d_cat5"][s2], 96, 0, 96))
        # ---- lstm6
        self._ln_lstm_bwd("hidden6", 5, t, View(ws["xh"][5][t + 1], 192, 128, 64), View(ws["d_cat5"][s2], 96, 0, 64), None, B, HW[4], last, ln_ws)
        # ---- enc4 deconv (input hidden5); d_hid5 may already hold the kernel-Linear contribution (side branch 0)
        if hid5_has_grad and not inline_head:                   # an in-line head put the Linear on side branch 0
            self._join(0)
        de4 = View(ws["d_e4pre"], 128, 0, 128)
        if self.tc is not None:
            self.tc.deconv_bwd_fused("enc4", t, View(ws["xh"][5][t], 192, 0, 128), View(ws["dxh"][5], 192, 0, 128), None, g["enc4/b"],
                                     ws["d_hid5"][s2], 1 if hid5_has_grad else 0)
        else:
            self._relu_bwd(View(ws["xh"][5][t], 192, 0, 128), View(ws["dxh"][5], 192, 0, 128), None, de4, Mr[4])
            L.call("pivp_colsum", de4.ptr, 128, 0, Mr[4], 128, _ptr(g["enc4/b"]), s)
            self._conv_wgrad(de4, B, H // 4, W // 4, View(ws["hid5"][t], 128, 0, 128), H // 8, W // 8, 3, 2, 1, g["enc4/W"], None)
            self._conv_fwd(de4, B, H // 4, W // 4, p["enc4/W"], None, 128, 3, 2, 1, View(ws["d_hid5"][s2], 128, 0, 128),
                           acc=1 if hid5_has_grad else 0)
        # ---- lstm5
        self._ln_lstm_bwd("hidden5", 4, t, View(ws["xh"][4][t + 1], 192, 64, 128), View(ws["d_hid5"][s2], 128, 0, 128), None, B, HW[8], last, ln_ws)
        # ---- enc3 (1x1 on concat(enc2 out, smear))
        self._relu_bwd(View(ws["xh"][4][t], 192, 0, 64), View(ws["dxh"][4], 192, 0, 64), None, View(ws["d_e3pre"][t], 64, 0, 64), Mr[8])
        de3 = View(ws["d_e3pre"][t], 64, 0, 64)
        cin3, cs3 = 64 + self.sa, self.cs3
        self._conv_dgrad(de3, B, H // 8, W // 8, p["enc3/W"], None, 1, 1, 0, View(ws["d_in3"][s2], cs3, 0, cin3), H // 8, W // 8)
        # ---- state predictor + smear backward; produces d cur[t] for step t-1
        d_cur_out = ws["d_cur"][t & 1]
        d_cur_in = None if last else ws["d_cur"][(t + 1) & 1]       # gradient w.r.t. cur[t+1] from step t+1's state_action
        L.call("pivp_state_bwd", _ptr(ws["d_gs"][t]), _ptr(d_cur_in), _ptr(ws["sa"][t]), _ptr(p["current_state/W"]),
               _ptr(ws["d_in3"][s2]) if self.use_state else 0, cs3, 64, HW[8], B, _ptr(d_cur_out),
               _ptr(g["current_state/W"]), _ptr(g["current_state/b"]), s)

    def _bwd_lower(self, t, ln_ws):
        """Backward step t, encoder half: enc2, lstm4, lstm3, enc1, lstm2, lstm1, norm_enc0 (and, in feedself mode, enc0 back to the frame)."""
        ws, L = self.ws, self.L
        s = self._s()
        T, B, H, W = self.T, self.B, self.H, self.W
        HW, Mr = ws["HW"], ws["Mr"]
        p, g = self.p, self.g
        last = (t == T - 2)
        s2, s3 = t & 1, t % 3
        need_dprev = self.feedself and t >= self.ctx          # prev_t = gen_{t-1} keeps the graph (ref:664-666)
        d_prev = ws["d_prev"] if need_dprev else None
        cs3 = self.cs3
        # ---- enc2
        de2 = View(ws["d_e2pre"][t], 64, 0, 64)
        if self.tc is not None:
            self.tc.conv_s2_dgrad_fused("enc2", t, View(ws["in3"][t], cs3, 0, 64), View(ws["d_in3"][s2], cs3, 0, 64), None, g["enc2/b"],
                                        Mr[8], 64, ws["d_hid4"], 64)
        else:
            self._relu_bwd(View(ws["in3"][t], cs3, 0, 64), View(ws["d_in3"][s2], cs3, 0, 64), None, de2, Mr[8])
            self._conv_dgrad(de2, B, H // 8, W // 8, p["enc2/W"], None, 3, 2, 1, View(ws["d_hid4"], 64, 0, 64), H // 4, W // 4)
        # ---- lstm4, lstm3
        self._ln_lstm_bwd("hidden4", 3, t, View(ws["xh"][3][t + 1], 128, 64, 64), View(ws["d_hid4"], 64, 0, 64), None, B, HW[4], last, ln_ws)
        self._ln_lstm_bwd("hidden3", 2, t, View(ws["xh"][2][t + 1], 96, 32, 64), View(ws["dxh"][3], 128, 0, 64), None, B, HW[4], last, ln_ws)
        # ---- enc1: encs[1] feeds lstm3 (x slot) and the enc5 skip slot
        de1 = View(ws["d_e1pre"][t], 32, 0, 32)
        if self.tc is not None:
            self.tc.conv_s2_dgrad_fused("enc1", t, View(ws["xh"][2][t], 96, 0, 32), View(ws["dxh"][2], 96, 0, 32), View(ws["d_cat5"][s2], 96, 64, 32),
                                        g["enc1/b"], Mr[4], 32, ws["d_hid2"], 32)
        else:
            self._relu_bwd(View(ws["xh"][2][t], 96, 0, 32), View(ws["dxh"][2], 96, 0, 32), View(ws["d_cat5"][s2], 96, 64, 32), de1, Mr[4])
            self._conv_dgrad(de1, B, H // 4, W // 4, p["enc1/W"], None, 3, 2, 1, View(ws["d_hid2"], 32, 0, 32), H // 2, W // 2)
        # ---- lstm2, lstm1
        self._ln_lstm_bwd("hidden2", 1, t, View(ws["xh"][1][t + 1], 64, 32, 32), View(ws["d_hid2"], 32, 0, 32), None, B, HW[2], last, ln_ws)
        self._ln_lstm_bwd("hidden1", 0, t, View(ws["xh"][0][t + 1], 64, 32, 32), View(ws["dxh"][1], 64, 0, 32), None, B, HW[2], last, ln_ws)
        # ---- norm_enc0 (+relu): encs[0] feeds lstm1 (x slot) and the enc6 skip slot; enc0
        self._ln_bwd("norm_enc0", View(ws["enc0_pre"][t], 32, 0, 32), View(ws["dxh"][0], 64, 0, 32), View(ws["d_cat6"][s3], 64, 32, 32),
                     B, HW[2], 1, ws["ln_stats"]["norm_enc0"][t], View(ws["d_enc0pre"][t], 32, 0, 32), ln_ws=ln_ws)
        de0 = View(ws["d_enc0pre"][t], 32, 0, 32)
        if need_dprev:
            self._conv_dgrad(de0, B, H // 2, W // 2, p["enc0/W"], None, 5, 2, 2, View(ws["d_img_nhwc"], 3, 0, 3), H, W)
            L.call("pivp_nhwc_to_nchw", _ptr(ws["d_img_nhwc"]), 3, 0, _ptr(d_prev), B, 3, HW[1], 1, s)
            L.call("pivp_axpy", _ptr(d_prev), _ptr(ws["d_gen"][t - 1]), B * 3 * H * W, s)

    def backward(self):
        """BPTT.  Backward step t = HEAD(t) (loss side: transform, heads, norm_enc6, enc6 -- see _bwd_head), UPPER(t) (lstm7 .. lstm5, enc3, state
        predictor) and LOWER(t) (enc2 .. lstm1, norm_enc0).  UPPER(t) needs HEAD(t) and UPPER(t+1); LOWER(t) needs UPPER(t) and LOWER(t+1);
        under scheduled sampling HEAD(t) needs nothing from the other two (the previous frame is detached).  So the three run as a software
        pipeline over three streams -- tick k issues HEAD(T-2-k), UPPER(T-1-k), LOWER(T-k), with a cross-stream barrier between ticks -- and
        a time step costs max(HEAD, UPPER, LOWER) (about 155 us each at b32) instead of their sum.  What crosses stages is multi-buffered by
        time step: d_cat6 x3, d_hid5 / d_in3 / d_cat5 x2, one LayerNorm workspace per stage; everything else is private to a layer, hence to
        a stage.  Under CUDA-graph capture the streams become parallel branches of the graph.  In feedself mode the previous frame keeps the
        graph (ref:664-666): d_gen[t-1] receives d_prev at the end of LOWER(t), so the stages run in line on one stream."""
        ws, T = self.ws, self.T
        self._side(3)
        pipelined = (not self.feedself) and 3 in self._branches
        if not pipelined:
            for t in range(T - 2, -1, -1):
                flag = self._bwd_head(t, False)
                self._bwd_upper(t, flag, False, ws["ln_ws"])
                self._bwd_lower(t, ws["ln_ws"])
                if self._stop_after_step(t):
                    return
        else:
            cur = torch.cuda.current_stream(self.dev)
            st_h, st_u = self._side(3), self._side(4)
            flags = {}
            streams = (cur, st_u, st_h)
            st_u.wait_stream(cur)                      # fork: the two side streams join the (possibly capturing) current stream first --
            st_h.wait_stream(cur)                      # a capturing stream must not wait on a stream that is not part of the capture yet
            for k in range(T - 1 + 2):
                for a in streams:                      # barrier between ticks: every stage waits for what the other two were given so far
                    for b in streams:
                        if a is not b and k > 0:
                            a.wait_stream(b)
                h, u, l = T - 2 - k, T - 1 - k, T - k
                if 0 <= h <= T - 2:
                    with torch.cuda.stream(st_h):
                        flags[h] = self._bwd_head(h, True)
                if 0 <= u <= T - 2:
                    with torch.cuda.stream(st_u):
                        self._bwd_upper(u, flags[u], True, ws["ln_ws_upper"])
                if u < 0 <= l and self.tc is not None and self.grad_sync is None:
                    self.tc.wgrad_early(st_u, st_h)    # decoder half finished: its weight gradients start beside LOWER(0)
                if 0 <= l <= T - 2:
                    self._bwd_lower(l, ws["ln_ws"])
            cur.wait_stream(st_u)
            cur.wait_stream(st_h)
        L, s = self.L, self._s()
        B, H, W = self.B, self.H, self.W
        HW, Mr = ws["HW"], ws["Mr"]
        p, g = self.p, self.g
        # ---- deferred weight gradients of enc0..enc3: the per-step tensors are stacked over time, so each is ONE launch with
        # S*B "images" (9x longer reduction per launch instead of 9 launches that cannot fill the GPU)
        gs = self.grad_sync
        if gs is not None:
            gs.ready("tail")                   # LayerNorm / heads / state-predictor gradients are final: their all-reduce runs under the GEMMs below
        with self._fork(2):                    # small deferred weight gradients: a branch beside tc.wgrad_all()
            S = T - 1
            first = lambda lst: lst[0]
            cin3 = 64 + self.sa
            if self.model_type == "CDNA":              # kernel Linear 8192 -> 250: one pass over all steps instead of T-1 read-modify-writes of dW
                NK = 25 * self.M
                L.call("pivp_linear_wgrad_steps", _ptr(first(ws["d_kern_raw"])), B * NK, _ptr(first(ws["hid5"])), Mr[8] * 128, 128 * HW[8],
                       _ptr(g["model/cdna_kerns/W"]), _ptr(g["model/cdna_kerns/b"]), S, B, 128 * HW[8], NK, self._s())
            self._conv_wgrad(View(first(ws["img_nhwc"]), 3, 0, 3), S * B, H, W, View(first(ws["d_enc0pre"]), 32, 0, 32), H // 2, W // 2, 5, 2, 2,
                             g["enc0/W"], g["enc0/b"])
            if self.tc is None:                # bf16 mode: tcgen05 weight-gradient GEMMs in tc.wgrad_all(), bias gradients from the hand-over
                self._conv_wgrad(View(first(ws["hid2"]), 32, 0, 32), S * B, H // 2, W // 2, View(first(ws["d_e1pre"]), 32, 0, 32), H // 4, W // 4,
                                 3, 2, 1, g["enc1/W"], g["enc1/b"])
                self._conv_wgrad(View(first(ws["hid4"]), 64, 0, 64), S * B, H // 4, W // 4, View(first(ws["d_e2pre"]), 64, 0, 64), H // 8, W // 8,
                                 3, 2, 1, g["enc2/W"], g["enc2/b"])
            self._conv_wgrad(View(first(ws["in3"]), self.cs3, 0, cin3), S * B, H // 8, W // 8, View(first(ws["d_e3pre"]), 64, 0, 64), H // 8, W // 8,
                             1, 1, 0, g["enc3/W"], g["enc3/b"])
        if gs is not None:
            self._join(2)
            gs.ready("xform")
        if self.tc is not None:
            self.tc.wgrad_all(gs)              # ConvLSTM weight/bias gradients: one tcgen05 GEMM per layer over all time steps
        self._join(2)
        if gs is not None:
            gs.finish()
