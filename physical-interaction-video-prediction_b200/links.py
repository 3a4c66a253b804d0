"""The reference's link surface (src/models/train_model.py) over the CUDA path.

Same class names, constructor arguments, call signatures and attributes as the reference:
``LayerNormalizationConv2D`` (:186-208), ``BasicConvLSTMCell`` (:216-276), ``StatelessCDNA/DNA/STP``
(:278-475), ``Model`` (:478-764) and the helpers ``concat_examples`` (:51-71), ``scheduled_sample`` (:73-122),
``peak_signal_to_noise_ratio`` (:124-134).  Tensors are torch CUDA fp32 in the reference's NCHW layout.
``Model`` runs the whole step through ``engine.Engine``; the small links run the same kernels stand-alone so
that they can be dropped into a Chainer graph one at a time (INTEGRATION.md).
"""
import math

import numpy as np
import torch

from . import functions as Fn
from .engine import Engine
from ._lib import lib, PivpError

RELU_SHIFT = 1e-12      # train_model.py:42
DNA_KERN_SIZE = 5       # train_model.py:45


# ----------------------------------------------------------------------------- helpers
def concat_examples(batch):
    """train_model.py:51-71 (host side, NumPy): list of [img (T,H,W,3), act (T,5), sta (T,5)] -> time-major, channel-first."""
    img = np.array([b[0] for b in batch])
    act = np.array([b[1] for b in batch])
    sta = np.array([b[2] for b in batch])
    return (np.ascontiguousarray(img.transpose(1, 0, 4, 2, 3)), np.ascontiguousarray(act.transpose(1, 0, 2)),
            np.ascontiguousarray(sta.transpose(1, 0, 2)))


from .parallel import num_ground_truth, scheduled_sample_mask, schedule_plan, allreduce_sum_   # noqa: E402,F401


def scheduled_sample(ground_truth_x, generated_x, batch_size, num_ground_truth):
    """train_model.py:73-122: batch with ``num_ground_truth`` samples from the ground truth and the rest generated.
    Same RNG consumption as the reference; the gather/stitch runs as one select kernel on the device (no D2H round trip)."""
    take = torch.from_numpy(scheduled_sample_mask(batch_size, num_ground_truth)).to(generated_x.device)
    out = torch.empty_like(generated_x)
    per = int(generated_x.numel() // int(batch_size))
    lib().call("pivp_sched_select", ground_truth_x.data_ptr(), generated_x.data_ptr(), take.data_ptr(), out.data_ptr(),
               int(batch_size), per, torch.cuda.current_stream(out.device).cuda_stream)
    return out


def peak_signal_to_noise_ratio(true, pred):
    """train_model.py:124-134: 10 log10(1 / MSE) with the batch-level MSE (computed by the mse kernel)."""
    slot = torch.zeros(1, dtype=torch.float32, device=pred.device)
    lib().call("pivp_mse", pred.data_ptr(), true.data_ptr(), pred.numel(), 0.0, 0, slot.data_ptr(),
               torch.cuda.current_stream(pred.device).cuda_stream)
    mse = float(slot.item()) / pred.numel()
    return 10.0 * math.log(1.0 / mse) / math.log(10.0)


class _Scalar(object):
    """Stands in for the 0-d ``chainer.Variable`` the reference returns as loss: ``.data`` / ``float()`` force the D2H read."""

    def __init__(self, getter):
        self._get, self._v = getter, None

    @property
    def data(self):
        if self._v is None:
            self._v = np.float32(self._get())
        return self._v

    def __float__(self):
        return float(self.data)

    def __repr__(self):
        return "loss(%r)" % float(self)


# ----------------------------------------------------------------------------- small links (stand-alone use)
class LayerNormalizationConv2D(object):
    """train_model.py:186-208.  gamma/beta are created lazily from the first input (size C*H*W), like L.LayerNormalization()."""

    def __init__(self):
        self.gamma = self.beta = None
        self._f = Fn.LayerNormalizationFunction()

    def __call__(self, inputs):
        n = inputs[0].numel()
        if self.gamma is None:
            self.gamma = torch.ones(n, dtype=torch.float32, device=inputs.device)
            self.beta = torch.zeros(n, dtype=torch.float32, device=inputs.device)
        self._x = inputs
        return self._f.forward((inputs, self.gamma, self.beta))[0]

    def backward(self, gy):
        gx, self.ggamma, self.gbeta = self._f.backward((self._x, self.gamma, self.beta), (gy,))
        return gx


class BasicConvLSTMCell(object):
    """train_model.py:216-276.  ``W`` (4*out, in+out, k, k) / ``b`` in Chainer layout, created on first call (LeCunNormal)."""

    def __init__(self, out_size=None, filter_size=5):
        self.out_size, self.filter_size = out_size, filter_size
        self.W = self.b = None
        self.reset_state()

    def reset_state(self):
        self.c = None
        self.h = None

    def __call__(self, inputs, forget_bias=1.0):
        B, Cin, H, W = inputs.shape
        C, k = self.out_size, self.filter_size
        dev = inputs.device
        if self.W is None:
            fan_in = (Cin + C) * k * k
            self.W = (torch.randn(4 * C, Cin + C, k, k, device=dev) * math.sqrt(1.0 / fan_in)).float()
            self.b = torch.zeros(4 * C, device=dev)
        if self.c is None:
            self.c = torch.zeros(B, C, H, W, device=dev)
        if self.h is None:
            self.h = torch.zeros(B, C, H, W, device=dev)
        from .layout import gate_perm
        L = lib()
        s = torch.cuda.current_stream(dev).cuda_stream
        M = B * H * W
        xh = torch.empty(M, Cin + C, device=dev)
        L.call("pivp_nchw_to_nhwc", inputs.data_ptr(), xh.data_ptr(), Cin + C, 0, B, Cin, H * W, s)
        L.call("pivp_nchw_to_nhwc", self.h.data_ptr(), xh.data_ptr(), Cin + C, Cin, B, C, H * W, s)
        perm = torch.from_numpy(gate_perm(C)).to(dev)
        wi = torch.empty_like(self.W)
        wi[perm] = self.W
        wi = wi.permute(0, 2, 3, 1).contiguous()
        bi = torch.empty_like(self.b)
        bi[perm] = self.b
        G = torch.empty(M, 4 * C, device=dev)
        L.call("pivp_conv2d_fwd", xh.data_ptr(), Cin + C, 0, B, H, W, Cin + C, wi.data_ptr(), bi.data_ptr(), 4 * C, k, k, 1, k // 2,
               G.data_ptr(), 4 * C, 0, H, W, 0, 0, s)
        cp = Fn.nchw_to_nhwc(self.c)
        cn, hn = torch.empty(M, C, device=dev), torch.empty(M, C, device=dev)
        L.call("pivp_lstm_gates_fwd", G.data_ptr(), cp.data_ptr(), cn.data_ptr(), hn.data_ptr(), C, 0, 0, 0, 0, M, C, float(forget_bias), s)
        self.c = Fn.nhwc_to_nchw(cn, B, C, H, W)
        self.h = Fn.nhwc_to_nchw(hn, B, C, H, W)
        return self.h


class _Stateless(object):
    """Common part of StatelessCDNA / DNA / STP (train_model.py:278-475).

    Two call forms:
      * the REFERENCE form ``link(encs, hiddens, batch_size, prev_image, num_masks, color_channels) -> (transformed_list, enc7)``
        (ref:293, 368, 434).  The link owns the reference's parameters (``enc7`` 1x1 Deconvolution2D, ``cdna_kerns`` / ``stp_input`` /
        ``identity_params`` Linear) in Chainer layout as attributes ``<name>_W`` / ``<name>_b``, created lazily with Chainer's default
        initialisers like ``L.Linear(in_size=None)``, or set by the caller (``load(params, prefix="model/")`` takes a checkpoint dict).
        ``transformed_list`` is the un-fused list Model.__call__ composites at ref:725-728.
        ``link.backward(g_transformed, g_enc7=None)`` is its backward, for a link dropped into the reference Model.
      * the FUSED form ``link.fused(prev_image, enc7_pre, mask_pre, ...) -> gen_image``: transform + mask softmax + composite in one
        kernel, which is what ``Model`` runs (the list never reaches memory).  A call with the fused arity is routed there.
    """
    NE = 3

    def __init__(self, num_masks):
        self.num_masks = num_masks
        self.enc7_W = self.enc7_b = None

    def load(self, params, prefix="model/"):
        """Take this link's parameters (Chainer layout) from a checkpoint-style dict: ``model/enc7/W`` -> ``self.enc7_W`` ..."""
        for k, v in params.items():
            if k.startswith(prefix):
                setattr(self, k[len(prefix):].replace("/", "_"), torch.as_tensor(np.asarray(v), dtype=torch.float32))
        return self

    def _param(self, name, shape, dev, fan_in=None):
        v = getattr(self, name, None)
        if v is None:
            v = torch.randn(*shape) * math.sqrt(1.0 / fan_in) if fan_in else torch.zeros(*shape)      # LeCunNormal / zeros (A.1)
        v = v.to(dev).float().contiguous()
        setattr(self, name, v)
        return v

    def _enc7(self, enc6):
        """ref:314 / 387 / 454: 1x1 Deconvolution2D(64 -> NE) on enc6 (B,64,H,W) -> pre-activation (B,NE,H,W)."""
        B, C, H, W = enc6.shape
        Wt = self._param("enc7_W", (C, self.NE, 1, 1), enc6.device, fan_in=self.NE)
        b = self._param("enc7_b", (self.NE,), enc6.device)
        self._enc6 = enc6.contiguous()                                                  # kept for backward()
        return Fn.Deconvolution2DFunction(1, 0, (H, W)).forward((self._enc6, Wt, b))[0]

    def _linear(self, name, x, out_size, relu=0):
        B, K = x.shape
        Wt = self._param(name + "_W", (out_size, K), x.device, fan_in=K)
        b = self._param(name + "_b", (out_size,), x.device)
        y = torch.empty(B, out_size, dtype=torch.float32, device=x.device)
        lib().call("pivp_linear_fwd", x.data_ptr(), K, Wt.data_ptr(), b.data_ptr(), y.data_ptr(), B, K, out_size, relu,
                   torch.cuda.current_stream(x.device).cuda_stream)
        return y

    def _linear_bwd(self, name, x, dy):
        """Backward of ``_linear`` (without its ReLU): returns dx, puts dW / db into ``self.grads``."""
        Wt = getattr(self, name + "_W")
        B, K = x.shape
        N = Wt.shape[0]
        dx = torch.empty_like(x)
        dW, db = torch.zeros_like(Wt), torch.zeros(N, dtype=torch.float32, device=x.device)      # accumulated into
        lib().call("pivp_linear_bwd", dy.data_ptr(), x.data_ptr(), K, Wt.data_ptr(), dx.data_ptr(), K, 0, dW.data_ptr(), db.data_ptr(),
                   B, K, N, torch.cuda.current_stream(x.device).cuda_stream)
        self.grads["model/%s/W" % name], self.grads["model/%s/b" % name] = dW, db
        return dx

    def backward(self, g_transformed, g_enc7=None):
        """Backward of the reference call form.  ``g_transformed``: the gradients of the returned list, one per entry, ``None`` for an
        entry without one (the reference Model composites with ``zip(transformed, mask_list[1:])``, ref:725-728, so the last CDNA entry
        never gets one); ``g_enc7``: that of the returned enc7, or ``None``.  Returns ``(g_enc6, g_hidden5, g_prev)`` shaped like
        ``encs[6]``, ``hiddens[4]`` and ``prev_image`` (``None`` where the link has no path: DNA's hidden5, and its prev_image, whose taps
        the reference detaches, ref:404).  The parameter gradients go to ``self.grads`` in Chainer layout, keyed as ``load()`` reads them
        (``model/enc7/W`` ...)."""
        g_list = tuple(None if g is None else g.contiguous() for g in g_transformed)
        if len(g_list) != self._nlist:
            raise ValueError("expected %d list gradients, got %d" % (self._nlist, len(g_list)))
        g_enc7 = None if g_enc7 is None else g_enc7.contiguous()
        self.grads = {}
        g_e7pre, g_hidden5, g_prev = self._transform_bwd(g_list, g_enc7)
        H, W = self._enc6.shape[2:]
        g_enc6, dW, db = Fn.Deconvolution2DFunction(1, 0, (H, W)).backward((self._enc6, self.enc7_W, self.enc7_b), (g_e7pre,))
        self.grads["model/enc7/W"], self.grads["model/enc7/b"] = dW, db
        return g_enc6, g_hidden5, g_prev


class StatelessCDNA(_Stateless):
    """train_model.py:278-351."""

    def __init__(self, num_masks):
        super(StatelessCDNA, self).__init__(num_masks)
        self.cdna_kerns_W = self.cdna_kerns_b = None

    def fused(self, prev_image, enc7_pre, mask_pre, kern_raw):
        return Fn.CDNACompositeFunction(self.num_masks).forward((prev_image, enc7_pre, mask_pre, kern_raw))[0]

    def __call__(self, *args):
        if len(args) == 4:
            return self.fused(*args)
        encs, hiddens, batch_size, prev_image, num_masks, color_channels = args
        B, _, H, W = prev_image.shape
        enc7_pre = self._enc7(encs[6])
        kern_raw = self._linear("cdna_kerns", hiddens[4].reshape(int(batch_size), -1).contiguous(), DNA_KERN_SIZE * DNA_KERN_SIZE * self.num_masks)
        out = torch.empty(self.num_masks + 1, B, 3, H, W, dtype=torch.float32, device=prev_image.device)
        lib().call("pivp_cdna_transform", prev_image.contiguous().data_ptr(), enc7_pre.data_ptr(), kern_raw.data_ptr(), out.data_ptr(), B, H, W,
                   self.num_masks, torch.cuda.current_stream(out.device).cuda_stream)
        self.enc7_pre, self.kern_raw = enc7_pre, kern_raw
        self._prev, self._h5, self._h5_shape = prev_image.contiguous(), hiddens[4].reshape(int(batch_size), -1).contiguous(), hiddens[4].shape
        self._nlist = self.num_masks + 1
        return [out[i] for i in range(self.num_masks + 1)], enc7_pre.clamp(min=0)          # ref:315 enc7 = relu(enc7)

    def _transform_bwd(self, g_list, g_enc7):
        g_prev, g_e, g_k = Fn.CDNATransformFunction(self.num_masks).backward((self._prev, self.enc7_pre, self.kern_raw), g_list + (g_enc7,))
        g_h5 = self._linear_bwd("cdna_kerns", self._h5, g_k)
        return g_e, g_h5.reshape(self._h5_shape), g_prev


class StatelessDNA(_Stateless):
    """train_model.py:354-417."""
    NE = DNA_KERN_SIZE * DNA_KERN_SIZE

    def fused(self, prev_image, enc7_pre, mask_pre):
        if self.num_masks != 1:
            raise ValueError("Only one mask is supported for DNA model.")
        return Fn.DNACompositeFunction().forward((prev_image, enc7_pre, mask_pre))[0]

    def __call__(self, *args):
        if len(args) == 3:
            return self.fused(*args)
        encs, hiddens, batch_size, prev_image, num_masks, color_channels = args
        if self.num_masks != 1:
            raise ValueError("Only one mask is supported for DNA model.")                # ref:389-390
        B, _, H, W = prev_image.shape
        enc7_pre = self._enc7(encs[6])
        out = torch.empty(1, B, 3, H, W, dtype=torch.float32, device=prev_image.device)
        lib().call("pivp_dna_transform", prev_image.contiguous().data_ptr(), enc7_pre.data_ptr(), out.data_ptr(), B, H, W,
                   torch.cuda.current_stream(out.device).cuda_stream)
        self.enc7_pre = enc7_pre
        self._prev, self._nlist = prev_image.contiguous(), 1
        return [out[0]], enc7_pre.clamp(min=0)

    def _transform_bwd(self, g_list, g_enc7):
        _, g_e = Fn.DNATransformFunction().backward((self._prev, self.enc7_pre), g_list + (g_enc7,))
        return g_e, None, None


class StatelessSTP(_Stateless):
    """train_model.py:419-475."""

    def __init__(self, num_masks):
        super(StatelessSTP, self).__init__(num_masks)
        self.stp_input_W = self.stp_input_b = self.identity_params_W = self.identity_params_b = None

    def fused(self, prev_image, enc7_pre, mask_pre, theta_raw, oob="zeros"):
        return Fn.STPCompositeFunction(self.num_masks, oob).forward((prev_image, enc7_pre, mask_pre, theta_raw))[0]

    def __call__(self, *args, **kw):
        if len(args) in (4, 5) and not isinstance(args[0], (list, tuple)):
            return self.fused(*args, **kw)
        encs, hiddens, batch_size, prev_image, num_masks, color_channels = args
        B, _, H, W = prev_image.shape
        enc7 = self._enc7(encs[6])                                                       # ref:454 no ReLU
        s_ = self._linear("stp_input", hiddens[4].reshape(int(batch_size), -1).contiguous(), 100, relu=1)
        theta_raw = self._linear("identity_params", s_, 6)                               # ONE Linear shared by all transformers (B.4)
        n = max(int(num_masks), 1)                                                       # ref:463 loops over the ARGUMENT num_masks - 1
        out = torch.empty(n, B, 3, H, W, dtype=torch.float32, device=prev_image.device)
        lib().call("pivp_stp_transform", prev_image.contiguous().data_ptr(), enc7.data_ptr(), theta_raw.data_ptr(), out.data_ptr(), B, H, W,
                   n, 1 if kw.get("oob", "zeros") == "border" else 0, torch.cuda.current_stream(out.device).cuda_stream)
        self.enc7_pre, self.theta_raw = enc7, theta_raw
        self._prev, self._h5, self._h5_shape = prev_image.contiguous(), hiddens[4].reshape(int(batch_size), -1).contiguous(), hiddens[4].shape
        self._s, self._nlist, self._oob = s_, n, kw.get("oob", "zeros")
        return [out[i] for i in range(n)], enc7

    def _transform_bwd(self, g_list, g_enc7):
        f = Fn.STPTransformFunction(self._nlist, self._oob)
        g_prev, g_e, g_th = f.backward((self._prev, self.enc7_pre, self.theta_raw), g_list + (g_enc7,))
        g_s = self._linear_bwd("identity_params", self._s, g_th)
        lib().call("pivp_relu_mask", self._s.data_ptr(), g_s.data_ptr(), g_s.numel(),       # the ReLU between the two Linears (ref:457)
                   torch.cuda.current_stream(g_s.device).cuda_stream)
        g_h5 = self._linear_bwd("stp_input", self._h5, g_s)
        return g_e, g_h5.reshape(self._h5_shape), g_prev


# ----------------------------------------------------------------------------- Model
class Model(object):
    """train_model.py:478-764.  Same constructor arguments; extra keyword-only geometry / device options.

    ``__call__(x, iter_num)`` runs the forward pass and returns the loss; ``backward()`` runs BPTT into ``.grads``;
    ``.loss .psnr_all .summaries .gen_images .conv_res .reset_state()`` exist as in the reference.
    """

    def __init__(self, num_masks, is_cdna=True, is_dna=False, is_stp=False, use_state=True, scheduled_sampling_k=-1,
                 num_frame_before_prediction=2, prefix=None, height=64, width=64, device="cuda", compute="f32",
                 stp_oob="zeros", rank=0, world_size=1):
        model_type = "CDNA" if is_cdna else ("STP" if is_stp else ("DNA" if is_dna else None))   # precedence as ref:532-537
        if model_type is None:
            raise ValueError("No network specified")
        self.engine = Engine(model_type, num_masks, use_state, height, width, num_frame_before_prediction, device, compute, stp_oob)
        self.num_masks, self.use_state = num_masks, use_state
        self.scheduled_sampling_k = scheduled_sampling_k
        self.num_frame_before_prediction = num_frame_before_prediction
        self.prefix = prefix
        self.train = True                      # stands in for chainer.config.train (ref:649)
        self.rank, self.world_size = rank, world_size
        self.reset_state()

    def reset_state(self):
        """ref:604-618.  The recurrent state lives in per-step buffers that every forward overwrites, so this only resets the report."""
        self.loss = 0.0
        self.psnr_all = 0.0
        self.summaries = []
        self._conv_res = []

    @property
    def conv_res(self):
        """ref:734 ``self.conv_res = encs``: the eight encoder outputs [enc0 .. enc6, enc7] of the LAST time step, (B,C,h,w) NCHW like the
        reference (visualize.py:443 reads them).  The engine keeps them as NHWC channel slices of the ConvLSTM input buffers, so the
        NCHW copies are made when the attribute is first looked at after a forward pass."""
        if callable(self._conv_res):
            self._conv_res = self._conv_res()
        return self._conv_res

    @conv_res.setter
    def conv_res(self, v):
        self._conv_res = v

    def _make_conv_res(self):
        e = self.engine
        ws, t, B, H, W = e.ws, e.T - 2, e.B, e.H, e.W
        src = [(ws["xh"][0][t], 64, 0, 32, 2), (ws["xh"][2][t], 96, 0, 32, 4), (ws["in3"][t], e.cs3, 0, 64, 8), (ws["xh"][4][t], 192, 0, 64, 8),
               (ws["xh"][5][t], 192, 0, 128, 4), (ws["xh"][6][t], 128, 0, 96, 2), (ws["e6"][t], 64, 0, 64, 1)]
        s = torch.cuda.current_stream(e.dev).cuda_stream
        out = []
        for buf, cs, co, C, lv in src:
            y = torch.empty(B, C, H // lv, W // lv, dtype=torch.float32, device=e.dev)
            lib().call("pivp_nhwc_to_nchw", buf.data_ptr(), cs, co, y.data_ptr(), B, C, (H // lv) * (W // lv), 0, s)
            out.append(y)
        enc7 = ws["enc7_pre"][t].clone()
        if e.model_type != "STP":                      # ref:315,388 relu(enc7) for CDNA / DNA; ref:454 STP keeps the raw deconvolution
            enc7.clamp_(min=0)
        out.append(enc7)
        return out

    # parameters in Chainer layout (npz-compatible, A.9)
    def params(self):
        return self.engine.chainer_params()

    def load_params(self, params):
        self.engine.load_chainer_params(params)

    @property
    def grads(self):
        return self.engine.chainer_grads()

    def cleargrads(self):
        self.engine.cleargrads()

    def save(self, filename):
        """``serializers.save_npz(filename, model)`` (ref:1035)."""
        from .serializers import save_npz
        save_npz(filename, self)

    def load(self, filename):
        """``serializers.load_npz(filename, model)`` (ref:865)."""
        from .serializers import load_npz
        load_npz(filename, self)

    def schedule(self, batch_size_global, T, iter_num):
        """Scheduled-sampling plan for one step (ref:649-657, 663-673): returns (feedself, take[T-1, B_local], n_gt).
        Every rank draws the SAME global permutations and keeps its slice (SURVEY 8e)."""
        return schedule_plan(batch_size_global, T, iter_num, self.scheduled_sampling_k, self.num_frame_before_prediction,
                             self.train, self.rank, self.world_size)

    def __call__(self, x, iter_num=-1.0):
        images, actions, states = x
        dev = self.engine.dev
        images, actions, states = [torch.as_tensor(a, dtype=torch.float32).to(dev).contiguous() for a in (images, actions, states)]
        T, B = images.shape[0], images.shape[1]
        feedself, take, self.num_ground_truth = self.schedule(B * self.world_size, T, iter_num)
        self.take_gt = take
        gen = self.engine.forward(images, actions, states, take, feedself)
        self.gen_images = gen
        self._bind_loss()
        return self.loss

    def _bind_loss(self):
        """Handles for .loss / .psnr_all bound to THIS step: the loss sums leave the device behind the step (a stream-ordered copy into
        a pinned ring slot, Engine.snapshot_loss), and the host read (ref:955-956) happens when a handle is first looked at -- it waits
        for that copy only, so step k's loss can be read after step k+1 was launched and still reports step k."""
        e = self.engine
        self.gen_states = e.ws["cur"][1:]
        self._conv_res = self._make_conv_res
        values = e.snapshot_loss()
        self.loss = _Scalar(lambda: values()[0])
        self.psnr_all = _Scalar(lambda: values()[1])
        self._values = values

    def make_summaries(self):
        """ref:744-759 strings, same order: recon_cost / psnr per predicted frame, state_cost per predicted state, psnr_all, loss."""
        loss, psnr, recon, state = self._values()
        p = self.prefix or ""
        out = []
        for i, c in enumerate(recon):
            out.append("%s_recon_cost%d: %s" % (p, i, c))
            out.append("%s_psnr%d: %s" % (p, i, 10.0 * math.log(1.0 / c) / math.log(10.0) if c > 0 else float("inf")))
        for i, c in enumerate(state):
            out.append("%s_state_cost%d: %s" % (p, i, c))
        out.append("%s_psnr_all: %s" % (p, psnr))
        out.append("%s_loss: %s" % (p, loss))
        self.summaries = out
        return out

    def backward(self):
        self.engine.backward()


class Adam(object):
    """chainer.optimizers.Adam as used at train_model.py:860-861,950 (Chainer 2.0.1 AdamRule, SURVEY A.8)."""

    def __init__(self, alpha=0.001, beta1=0.9, beta2=0.999, eps=1e-8):
        self.alpha, self.beta1, self.beta2, self.eps = alpha, beta1, beta2, eps
        self.target = None
        self.epoch = 0                         # chainer.Optimizer.epoch (serialised in the state file, ref:1037)

    def new_epoch(self):
        self.epoch += 1

    def setup(self, model):
        self.target = model
        e = model.engine
        self.m = torch.zeros_like(e.flat_p)
        self.v = torch.zeros_like(e.flat_p)
        self.step = torch.zeros(1, dtype=torch.int32, device=e.dev)
        return self

    @property
    def t(self):
        return int(self.step.item())

    def apply(self):
        """All-reduce (data parallel) + fused 1/N scale + Adam on the flat buffers."""
        e = self.target.engine
        ws = self.target.world_size
        if ws > 1:
            allreduce_sum_(e.flat_g)                          # NCCL sum over NVLink (SURVEY 8e)
        lib().call("pivp_adam_step", e.flat_p.data_ptr(), e.flat_g.data_ptr(), self.m.data_ptr(), self.v.data_ptr(), e.nparam,
                   self.step.data_ptr(), self.alpha, self.beta1, self.beta2, self.eps, 1.0 / ws,
                   torch.cuda.current_stream(e.dev).cuda_stream)
        e.params_changed()

    def update(self, lossfun, *args):
        """ref:950 ``optimizer.update(training_model, [imgs, acts, stas], itr)``: forward, cleargrads, backward, update."""
        loss = lossfun(*args)
        self.target.cleargrads()
        self.target.backward()
        self.apply()
        return loss
