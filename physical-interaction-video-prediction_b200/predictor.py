"""Forward-only batched prediction with a fixed memory footprint (planning: score many candidate action sequences).

``Predictor`` runs the test-mode forward pass (feedself: the first ``context_frames`` steps see the given frames, every later step its own
prediction, train_model.py:649-650, 663-666) of a ``Model`` on a workspace of its own:

* ``ForwardEngine`` shares the model's flat parameter buffer by reference -- never copied, never re-initialised -- and owns every buffer
  it writes, so the training engine's workspace, tensor-core plan and loss rings are never touched and a graph captured by ``Rollout`` or
  ``TrainStep`` on the same model stays valid.
* No backward state: no saved gates, no gradient temporaries, no weight-gradient workspaces or stacked operands, no loss kernels and no
  scheduled-sampling select.  The gate epilogue runs without its gate store (``pivp_tc_conv5x5`` flags bit 2) and the heads kernel without
  the normalised ``enc6`` rows (``pivp_heads_fwd_ln`` with ``y == NULL``).
* Per-time-step buffers are rings.  Depth 2 for the ConvLSTM inputs ``xh`` (step t reads slot t and writes h_t into slot t+1: one kernel
  must not read and write the same buffer) and, as a margin, for everything else produced and consumed inside a step; every side branch of
  the step (``_fork(5)``: state predictor, smear and skip copies; ``_fork(0)``: kernel / theta Linear) joins before the step ends, so a
  slot is never reused while a branch may still read it.  The cell state ``c`` has depth 1: the gate kernels update it in place
  (include/pivp.h).  Only the outputs -- predicted frames and states -- keep one slot per step.
* The bf16 weight refresh is the first node of the captured graph: every replay sees the current parameters (after ``Adam.apply``,
  ``load_params``) with no host bookkeeping.
"""
import numpy as np
import torch

from .engine import Engine, LSTM_IN, LSTM_SIZES, LSTM_LEVEL
from .tensorcore import TensorCorePlan
from ._lib import PivpError

RING = 2


def _ring(make, n, depth=RING):
    """n per-step entries over `depth` buffers: entry t is buffer t % depth (list aliasing keeps Engine.forward_device's indexing)."""
    bufs = [make() for _ in range(min(depth, n))]
    return [bufs[t % len(bufs)] for t in range(n)]


class ForwardPlan(TensorCorePlan):
    """The forward half of TensorCorePlan: bf16 operand rings, forward weights only, no gate storage, no backward operands."""
    store_gates = False

    def __init__(self, eng, ws):
        self.eng, self.ws = eng, ws
        dev = eng.dev
        B, T = ws["B"], ws["T"]
        S = T - 1
        self.S = RING                                   # time extent of the per-step operands _plan_conv_s2_fwd allocates
        self.Kpad = [(cin + c + 63) // 64 * 64 for cin, c in zip(LSTM_IN, LSTM_SIZES)]
        self.xh_bf16, self.dg_bf16, self.Wf, self.Wd = [], [], [], []
        for li, (cin, c, lv) in enumerate(zip(LSTM_IN, LSTM_SIZES, LSTM_LEVEL)):
            M = ws["Mr"][lv]
            h, w = eng.H // lv, eng.W // lv
            if M % 128 or (h * w) % 64:
                raise PivpError("bf16 tensor-core path: ConvLSTM layer %d has B*H*W = %d (needs a multiple of 128) and H*W = %d "
                                "(needs a multiple of 64); use an even batch / 64x64 or larger images, or compute='f32'"
                                % (li + 1, M, h * w))
            self.xh_bf16.append(_ring(lambda: torch.zeros(M, self.Kpad[li], dtype=torch.bfloat16, device=dev), T))   # pad channels stay 0
            self.dg_bf16.append([None] * S)             # no gate storage (flags bit 2)
            self.Wf.append(torch.empty(4 * c, 25, self.Kpad[li], dtype=torch.bfloat16, device=dev))
            self.Wd.append(None)                        # no input-gradient weights
        self.accurate = 0
        self.fuse_ln = False                            # the LayerNorm-fused cell stores its gates (pivp_tc_conv5x5_ln)
        self.split_n, self.pair_bn = 0, 0
        self.ln_fused = [(eng.H // lv) % 16 == 0 and (eng.W // lv) % 8 == 0 and ((eng.H // lv) * (eng.W // lv) * c) % 4096 == 0
                         for c, lv in zip(LSTM_SIZES, LSTM_LEVEL)]
        self._wflat = torch.zeros(2 << 20, dtype=torch.bfloat16, device=dev)
        self._wofs, self._widx = 0, []
        M8, M4, M2 = ws["Mr"][8], ws["Mr"][4], ws["Mr"][2]
        self.hid5_b = _ring(lambda: torch.zeros(M8, 128, dtype=torch.bfloat16, device=dev), S)
        self.cat5_b = _ring(lambda: torch.zeros(M4, 128, dtype=torch.bfloat16, device=dev), S)      # 96 used, 32 zero pad
        self.cat6_b = _ring(lambda: torch.zeros(M2, 64, dtype=torch.bfloat16, device=dev), S)
        self.dec = {}
        for name, cin, cout, lv in (("enc4", 128, 128, 8), ("enc5", 96, 96, 4), ("enc6", 64, 64, 2)):
            self.dec[name] = self._plan_deconv(name, cin, cout, lv)
        self.s2f = {"enc1": self._plan_conv_s2_fwd("enc1", 32, 32, 2), "enc2": self._plan_conv_s2_fwd("enc2", 64, 64, 4)}
        for d in self.s2f.values():
            d["xs"] = [d["xs"][t % RING] for t in range(S)]
        self._widx_all = torch.from_numpy(np.concatenate(self._widx)).to(dev)
        self.refresh_weights()


class ForwardEngine(Engine):
    """Forward-only engine over the parameters of `train_engine` (shared by reference): ring workspace, no backward state."""

    def __init__(self, train_engine):
        e = train_engine
        Engine.__init__(self, e.model_type, e.M, e.use_state, e.H, e.W, e.ctx, e.dev, e.compute, "border" if e.oob else "zeros",
                        params=e.flat_p)

    def _heads_ln(self):
        """Engine.forward_device's choice of the heads kernel that applies norm_enc6 itself (then e6 is never read in the forward pass)."""
        import os
        e6_stats = self.compute == "bf16" and ((self.H // 2) * (self.W // 2)) % 128 == 0
        return e6_stats and self.Nh in (14, 27) and os.environ.get("PIVP_HEADS_LN", "1") != "0"

    def _workspace(self, B, T):
        if self.ws is not None and self.ws["B"] == B and self.ws["T"] == T:
            return self.ws
        self.ws, self.tc = None, None
        H, W = self.H, self.W
        ws = {"B": B, "T": T}
        HW = {1: H * W, 2: (H // 2) * (W // 2), 4: (H // 4) * (W // 4), 8: (H // 8) * (W // 8)}
        Mr = {k: B * v for k, v in HW.items()}
        ws["HW"], ws["Mr"] = HW, Mr
        A = self._alloc
        S = T - 1
        ws["img_nhwc"] = _ring(lambda: A(Mr[1], 3), S)
        ws["enc0_pre"] = _ring(lambda: A(Mr[2], 32), S)
        ws["xh"], ws["G"], ws["c"] = [], [], []
        for cin, c, lv in zip(LSTM_IN, LSTM_SIZES, LSTM_LEVEL):
            ws["xh"].append(_ring(lambda: A(Mr[lv], cin + c, zero=True), T))
            # fp32 path: the gate pre-activations are scratch of the step (conv output, activated in place); bf16 path: not stored at all
            ws["G"].append(_ring(lambda: A(Mr[lv], 4 * c), S, 1) if self.compute == "f32" else [None] * S)
            ws["c"].append(_ring(lambda: A(Mr[lv], c), S, 1))       # updated in place
        ws["hid2"] = _ring(lambda: A(Mr[2], 32), S)
        ws["hid4"] = _ring(lambda: A(Mr[4], 64), S)
        ws["in3"] = _ring(lambda: A(Mr[8], self.cs3), S)
        ws["hid5"] = _ring(lambda: A(Mr[8], 128), S)
        ws["cat5"] = _ring(lambda: A(Mr[4], 96), S)
        ws["cat6"] = _ring(lambda: A(Mr[2], 64), S)
        ws["e6pre"] = _ring(lambda: A(Mr[1], 64), S)
        ws["e6"] = [None] * S if self._heads_ln() else _ring(lambda: A(Mr[1], 64), S)     # None: pivp_heads_fwd_ln gets y == NULL
        ws["head"] = [None] * S if self.Nh in (14, 27) else _ring(lambda: A(Mr[1], self.Nh), S)
        ws["enc7_pre"] = _ring(lambda: A(B, self.Ne, H, W), S)
        ws["mask_pre"] = _ring(lambda: A(B, self.M1, H, W), S)
        ws["gen_all"] = A(S, B, 3, H, W)               # the outputs: one slot per step
        ws["gen"] = [ws["gen_all"][t] for t in range(S)]
        ws["prev_buf"] = [None] * S                    # (scheduled sampling only)
        ws["sa"] = _ring(lambda: A(B, 10), S)
        ws["cur_all"] = A(T, B, 5)
        ws["cur"] = [ws["cur_all"][t] for t in range(T)]
        ws["ln_stats"] = {name: _ring(lambda: A(B, 2), S) for name in ("norm_enc0", "norm_enc6") + tuple("hidden%d" % i for i in range(1, 8))}
        if self.model_type == "CDNA":
            ws["kern_raw"] = _ring(lambda: A(B, 25 * self.M), S)
        elif self.model_type == "STP":
            ws["stp_s"] = _ring(lambda: A(B, 100), S)
            ws["theta_raw"] = _ring(lambda: A(B, 6), S)
        ws["lin_ws"] = torch.empty(max(16, self.L.query("pivp_linear_fwd_workspace_bytes", B, 128 * HW[8], max(25 * self.M, 100))),
                                   dtype=torch.uint8, device=self.dev)
        nb = self.L.query("pivp_layernorm_workspace_bytes", B, 64 * H * W)
        ws["ln_ws"] = torch.empty(max(nb, 16), dtype=torch.uint8, device=self.dev)
        self.ws = ws
        if self.compute == "bf16":
            self.tc = ForwardPlan(self, ws)
        return ws

    def predict_device(self, context, actions, state0, T, refresh=True):
        """context (>= min(T-1, context_frames), B, 3, H, W), actions (T-1, B, 5), state0 (1, B, 5): stream-ordered work only (capturable).
        ``refresh=False`` skips the bf16 weight refresh (a caller that runs several passes on unchanged parameters refreshes once)."""
        ws = self._workspace(int(context.shape[1]), int(T))
        if self.tc is not None and refresh:
            self.tc.refresh_weights()                  # bf16 weight operands from the current flat_p: first node of a captured graph
        for li, (cin, c) in enumerate(zip(LSTM_IN, LSTM_SIZES)):
            ws["xh"][li][0][:, cin:].zero_()           # h_{-1} = 0: slot 0 of the ring held h of an odd step of the previous pass
            if self.tc is not None:
                self.tc.xh_bf16[li][0][:, cin:cin + c].zero_()
        return self.forward_device(context, actions, state0, True, steps=T, loss=False)


class Predictor(object):
    """``predictor(context_images, actions, first_state)`` -> predicted frames (T-1, N, 3, H, W), CUDA float32; ``.gen_states`` (T-1, N, 5).

    context_images (C, N or 1, 3, H, W) with C >= model.num_frame_before_prediction (only the first context_frames are read), actions
    (T-1, N, 5), first_state (N or 1, 5); float32, on any device.  A batch of 1 in the context or the first state is broadcast to all N
    rows.  N may exceed ``batch_size``: the captured graph then runs over chunks of batch_size rows; a short last chunk (and an odd chunk
    on the bf16 path, which tiles the 8x8 maps in pairs of images) is padded by repeating its last row.  The returned tensors are the
    predictor's output buffers: the next call overwrites them (clone to keep)."""

    def __init__(self, model, batch_size, seq_len, graph=True):
        e = model.engine
        B, T = int(batch_size), int(seq_len)
        if B < 1 or T < 2:
            raise ValueError("batch_size must be >= 1 and seq_len >= 2 (got %d, %d)" % (B, T))
        self.model, self.B, self.T = model, B, T
        self.Bp = B + (B & 1) if e.compute == "bf16" else B
        self.ctx = e.ctx
        self.e = ForwardEngine(e)
        dev, H, W = e.dev, e.H, e.W
        self.context = torch.zeros(self.ctx, self.Bp, 3, H, W, dtype=torch.float32, device=dev)
        self.actions = torch.zeros(T - 1, self.Bp, 5, dtype=torch.float32, device=dev)
        self.state0 = torch.zeros(1, self.Bp, 5, dtype=torch.float32, device=dev)
        self.e._workspace(self.Bp, T)
        self.use_graph, self.graph = bool(graph), None
        self._out = None                                 # (N, frames, states) for calls with more rows than one chunk
        self.gen_states = None

    # ---- inputs
    def _check(self, context_images, actions, first_state):
        e = self.e

        def arr(x, what):
            if not isinstance(x, torch.Tensor):
                x = np.asarray(x)
                if x.dtype != np.float32:
                    raise ValueError("%s: float32 required, got %s" % (what, x.dtype))
                x = torch.from_numpy(x)
            elif x.dtype != torch.float32:
                raise ValueError("%s: float32 required, got %s" % (what, x.dtype))
            return x
        c, a, s = arr(context_images, "context_images"), arr(actions, "actions"), arr(first_state, "first_state")
        if a.dim() != 3 or a.shape[0] != self.T - 1 or a.shape[2] != 5 or a.shape[1] < 1:
            raise ValueError("actions: (T-1, N, 5) = (%d, N, 5) expected, got %s" % (self.T - 1, tuple(a.shape)))
        N = int(a.shape[1])
        if c.dim() != 5 or c.shape[0] < self.ctx or c.shape[1] not in (1, N) or tuple(c.shape[2:]) != (3, e.H, e.W):
            raise ValueError("context_images: (C >= %d, %d or 1, 3, %d, %d) expected, got %s" % (self.ctx, N, e.H, e.W, tuple(c.shape)))
        if s.dim() != 2 or s.shape[0] not in (1, N) or s.shape[1] != 5:
            raise ValueError("first_state: (%d or 1, 5) expected, got %s" % (N, tuple(s.shape)))
        return c[:self.ctx], a, s[None], N

    def _put(self, dst, src, n0, n):
        """Rows [n0, n0 + n) of src (batch dimension 1; a batch of 1 is broadcast) into dst, padded by repeating the last row."""
        dev = dst.device
        if src.shape[1] == 1:
            dst.copy_(src.to(dev, non_blocking=True).expand_as(dst))
            return
        dst[:, :n].copy_(src[:, n0:n0 + n].to(dev, non_blocking=True))
        if dst.shape[1] > n:
            dst[:, n:].copy_(dst[:, n - 1:n].expand(-1, dst.shape[1] - n, *dst.shape[2:]))

    # ---- the forward pass
    def _forward(self):
        self.e.predict_device(self.context, self.actions, self.state0, self.T)

    def _run(self):
        if not self.use_graph:
            self._forward()
            return
        if self.graph is None:
            dev = self.e.dev
            s = torch.cuda.Stream(device=dev)
            s.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(s):
                self._forward()                                           # lazy initialisation outside the capture
            torch.cuda.current_stream(dev).wait_stream(s)
            torch.cuda.synchronize(dev)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._forward()
        self.graph.replay()

    def __call__(self, context_images, actions, first_state):
        c, a, s, N = self._check(context_images, actions, first_state)
        ws = self.e.ws
        gen, cur = ws["gen_all"], ws["cur_all"]
        if N > self.B:
            if self._out is None or self._out[0] != N:
                e = self.e
                self._out = (N, torch.empty(self.T - 1, N, 3, e.H, e.W, dtype=torch.float32, device=e.dev),
                             torch.empty(self.T - 1, N, 5, dtype=torch.float32, device=e.dev))
        for n0 in range(0, N, self.B):
            n = min(self.B, N - n0)
            self._put(self.context, c, n0, n)
            self._put(self.actions, a, n0, n)
            self._put(self.state0, s, n0, n)
            self._run()
            if N > self.B:
                self._out[1][:, n0:n0 + n].copy_(gen[:, :n])
                self._out[2][:, n0:n0 + n].copy_(cur[1:, :n])
        if N > self.B:
            frames, self.gen_states = self._out[1], self._out[2]
        else:
            frames, self.gen_states = gen[:, :N], cur[1:, :N]
        return frames
