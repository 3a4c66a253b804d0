"""Function-style (forward / backward pairs) wrappers over libpivp.so, on torch CUDA tensors.

Chainer 2.0.1 only has ``chainer.Function`` (``forward_gpu`` / ``backward_gpu``); each class here has the same
shape -- ``forward(inputs) -> outputs`` and ``backward(inputs, grad_outputs) -> grad_inputs`` -- so that
INTEGRATION.md's Chainer adapter is a three-line subclass.  Inputs are fp32, contiguous, NCHW like the
reference's Variables.  No arithmetic happens in torch: it only owns the memory and the stream.
"""
import ctypes

import numpy as np
import torch

from ._lib import lib, PivpError


def _s(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _chk(*ts):
    for t in ts:
        if t is None:
            continue
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise PivpError("expected contiguous fp32 CUDA tensors (no CPU fallback exists for this path)")


def _p(t):
    return 0 if t is None else t.data_ptr()


class CDNACompositeFunction(object):
    """train_model.py:315-317,326-349 (StatelessCDNA) fused with the mask softmax + compositing :719-728.

    inputs: prev (B,3,H,W), enc7_pre (B,3,H,W), mask_pre (B,M+1,H,W), kern_raw (B,25*M); output gen (B,3,H,W).
    """

    def __init__(self, num_masks):
        self.M = int(num_masks)

    def forward(self, inputs):
        prev, e, a, k = inputs
        _chk(prev, e, a, k)
        B, _, H, W = prev.shape
        out = torch.empty_like(prev)
        lib().call("pivp_cdna_fused_fwd", _p(prev), _p(e), _p(a), _p(k), _p(out), B, H, W, self.M, _s(prev))
        return (out,)

    def backward(self, inputs, grad_outputs, need_dprev=True):
        prev, e, a, k = inputs
        (g,) = grad_outputs
        _chk(prev, e, a, k, g)
        B, _, H, W = prev.shape
        L = lib()
        nb = L.query("pivp_cdna_fused_bwd_workspace_bytes", B, H, W, self.M)
        ws = torch.empty(nb, dtype=torch.uint8, device=prev.device)
        de, da, dk = torch.empty_like(e), torch.empty_like(a), torch.empty_like(k)
        dp = torch.empty_like(prev) if need_dprev else None
        L.call("pivp_cdna_fused_bwd", _p(g), _p(prev), _p(e), _p(a), _p(k), _p(de), _p(da), _p(dk), _p(dp), 0,
               B, H, W, self.M, _p(ws), nb, _s(prev))
        return dp, de, da, dk


class DNACompositeFunction(object):
    """train_model.py:388-415 (StatelessDNA) + :719-728.  inputs: prev, enc7_pre (B,25,H,W), mask_pre (B,2,H,W)."""

    def forward(self, inputs):
        prev, e, a = inputs
        _chk(prev, e, a)
        B, _, H, W = prev.shape
        out = torch.empty_like(prev)
        lib().call("pivp_dna_fused_fwd", _p(prev), _p(e), _p(a), _p(out), B, H, W, _s(prev))
        return (out,)

    def backward(self, inputs, grad_outputs, need_dprev=True):
        prev, e, a = inputs
        (g,) = grad_outputs
        _chk(prev, e, a, g)
        B, _, H, W = prev.shape
        L = lib()
        nb = L.query("pivp_dna_fused_bwd_workspace_bytes", B, H, W)
        ws = torch.empty(nb, dtype=torch.uint8, device=prev.device)
        de, da = torch.empty_like(e), torch.empty_like(a)
        dp = torch.empty_like(prev) if need_dprev else None
        L.call("pivp_dna_fused_bwd", _p(g), _p(prev), _p(e), _p(a), _p(de), _p(da), _p(dp), 0, B, H, W, _p(ws), nb, _s(prev))
        return dp, de, da


class STPCompositeFunction(object):
    """train_model.py:454-471 (StatelessSTP) + :719-728.  theta_raw (B,6) is the shared Linear output BEFORE the
    identity [1,0,0,0,1,0] is added (the kernel adds it)."""

    def __init__(self, num_masks, oob="zeros"):
        self.M, self.oob = int(num_masks), 1 if oob == "border" else 0

    def forward(self, inputs):
        prev, e, a, th = inputs
        _chk(prev, e, a, th)
        B, _, H, W = prev.shape
        out = torch.empty_like(prev)
        lib().call("pivp_stp_fused_fwd", _p(prev), _p(e), _p(a), _p(th), _p(out), B, H, W, self.M, self.oob, _s(prev))
        return (out,)

    def backward(self, inputs, grad_outputs, need_dprev=True):
        prev, e, a, th = inputs
        (g,) = grad_outputs
        _chk(prev, e, a, th, g)
        B, _, H, W = prev.shape
        L = lib()
        nb = L.query("pivp_stp_fused_bwd_workspace_bytes", B, H, W, self.M)
        ws = torch.empty(nb, dtype=torch.uint8, device=prev.device)
        de, da, dth = torch.empty_like(e), torch.empty_like(a), torch.empty_like(th)
        dp = torch.zeros_like(prev) if need_dprev else None
        L.call("pivp_stp_fused_bwd", _p(g), _p(prev), _p(e), _p(a), _p(th), _p(de), _p(da), _p(dth), _p(dp),
               B, H, W, self.M, self.oob, _p(ws), nb, _s(prev))
        return dp, de, da, dth


def _glist(grads):
    """Chainer-style grad_outputs of a list (None = no gradient) -> host array of device pointers (None -> NULL)."""
    _chk(*grads)
    return (ctypes.c_void_p * len(grads))(*[_p(g) for g in grads])


def _relu_out(e):
    """relu(e) through the library's mask kernel: the reference's returned enc7 (ref:315, 388)."""
    out = e.clone()
    lib().call("pivp_relu_mask", _p(e), _p(out), out.numel(), _s(e))
    return out


class CDNATransformFunction(object):
    """The reference call form of StatelessCDNA (train_model.py:315-347): transform list + enc7, un-fused.

    inputs: prev (B,3,H,W), enc7_pre (B,3,H,W), kern_raw (B,25*M).  outputs: the M+1 list entries (B,3,H,W) -- sigmoid(relu(enc7_pre)),
    then prev cross-correlated with each normalised kernel -- followed by enc7 = relu(enc7_pre).  backward takes the M+2 output gradients
    (None allowed) and returns the gradients of (prev, enc7_pre, kern_raw)."""

    def __init__(self, num_masks):
        self.M = int(num_masks)

    def forward(self, inputs):
        prev, e, k = inputs
        _chk(prev, e, k)
        B, _, H, W = prev.shape
        out = torch.empty(self.M + 1, B, 3, H, W, dtype=torch.float32, device=prev.device)
        lib().call("pivp_cdna_transform", _p(prev), _p(e), _p(k), _p(out), B, H, W, self.M, _s(prev))
        return tuple(out[i] for i in range(self.M + 1)) + (_relu_out(e),)

    def backward(self, inputs, grad_outputs, need_dprev=True):
        prev, e, k = inputs
        _chk(prev, e, k)
        B, _, H, W = prev.shape
        gl = _glist(grad_outputs[:self.M + 1])
        ge = grad_outputs[self.M + 1]
        _chk(ge)
        L = lib()
        nb = L.query("pivp_cdna_transform_bwd_workspace_bytes", B, H, W, self.M)
        ws = torch.empty(nb, dtype=torch.uint8, device=prev.device)
        de, dk = torch.empty_like(e), torch.empty_like(k)
        dp = torch.empty_like(prev) if need_dprev else None
        L.call("pivp_cdna_transform_bwd", gl, _p(ge), _p(prev), _p(e), _p(k), _p(de), _p(dk), _p(dp), 0, B, H, W, self.M, _p(ws), nb, _s(prev))
        return dp, de, dk


class DNATransformFunction(object):
    """The reference call form of StatelessDNA (train_model.py:388-414).  inputs: prev, enc7_pre (B,25,H,W); outputs: the one
    transformed image and enc7 = relu(enc7_pre).  The taps are detached in the reference (:404), so the gradient of prev is None."""

    def forward(self, inputs):
        prev, e = inputs
        _chk(prev, e)
        B, _, H, W = prev.shape
        out = torch.empty_like(prev)
        lib().call("pivp_dna_transform", _p(prev), _p(e), _p(out), B, H, W, _s(prev))
        return out, _relu_out(e)

    def backward(self, inputs, grad_outputs):
        prev, e = inputs
        _chk(prev, e)
        B, _, H, W = prev.shape
        gl = _glist(grad_outputs[:1])
        ge = grad_outputs[1]
        _chk(ge)
        de = torch.empty_like(e)
        lib().call("pivp_dna_transform_bwd", gl, _p(ge), _p(prev), _p(e), _p(de), B, H, W, _s(prev))
        return None, de


class STPTransformFunction(object):
    """The reference call form of StatelessSTP (train_model.py:454-470).  inputs: prev, enc7_pre (B,3,H,W), theta_raw (B,6) (the shared
    Linear output before the identity is added); outputs: the num_masks list entries -- sigmoid(enc7_pre), then num_masks - 1 samplings
    with the one theta -- followed by enc7 = enc7_pre.  backward returns the gradients of (prev, enc7_pre, theta_raw)."""

    def __init__(self, num_masks, oob="zeros"):
        self.M, self.oob = int(num_masks), 1 if oob == "border" else 0

    def forward(self, inputs):
        prev, e, th = inputs
        _chk(prev, e, th)
        B, _, H, W = prev.shape
        out = torch.empty(self.M, B, 3, H, W, dtype=torch.float32, device=prev.device)
        lib().call("pivp_stp_transform", _p(prev), _p(e), _p(th), _p(out), B, H, W, self.M, self.oob, _s(prev))
        return tuple(out[i] for i in range(self.M)) + (e,)

    def backward(self, inputs, grad_outputs, need_dprev=True):
        prev, e, th = inputs
        _chk(prev, e, th)
        B, _, H, W = prev.shape
        gl = _glist(grad_outputs[:self.M])
        ge = grad_outputs[self.M]
        _chk(ge)
        L = lib()
        nb = L.query("pivp_stp_transform_bwd_workspace_bytes", B, H, W, self.M)
        ws = torch.empty(nb, dtype=torch.uint8, device=prev.device)
        de, dth = torch.empty_like(e), torch.empty_like(th)
        dp = torch.empty_like(prev) if need_dprev else None
        L.call("pivp_stp_transform_bwd", gl, _p(ge), _p(prev), _p(e), _p(th), _p(de), _p(dth), _p(dp), 0, B, H, W, self.M, self.oob,
               _p(ws), nb, _s(prev))
        return dp, de, dth


def nchw_to_nhwc(x):
    """(B,C,H,W) -> (B*H*W, C) via the library's packing kernel."""
    _chk(x)
    B, C, H, W = x.shape
    y = torch.empty(B * H * W, C, dtype=torch.float32, device=x.device)
    lib().call("pivp_nchw_to_nhwc", _p(x), _p(y), C, 0, B, C, H * W, _s(x))
    return y


def nhwc_to_nchw(y, B, C, H, W):
    x = torch.empty(B, C, H, W, dtype=torch.float32, device=y.device)
    lib().call("pivp_nhwc_to_nchw", _p(y), C, 0, _p(x), B, C, H * W, 0, _s(y))
    return x


class Convolution2DFunction(object):
    """L.Convolution2D (A.2) on NCHW tensors with a Chainer-layout weight (O,I,kh,kw); cross-correlation."""

    def __init__(self, stride=1, pad=0):
        self.s, self.p = stride, pad

    def forward(self, inputs):
        x, W, b = inputs
        B, C, H, Wd = x.shape
        O, _, kh, kw = W.shape
        Ho, Wo = (H + 2 * self.p - kh) // self.s + 1, (Wd + 2 * self.p - kw) // self.s + 1
        xn = nchw_to_nhwc(x)
        wi = W.permute(0, 2, 3, 1).contiguous()
        yn = torch.empty(B * Ho * Wo, O, dtype=torch.float32, device=x.device)
        lib().call("pivp_conv2d_fwd", _p(xn), C, 0, B, H, Wd, C, _p(wi), _p(b), O, kh, kw, self.s, self.p, _p(yn), O, 0, Ho, Wo, 0, 0, _s(x))
        return (nhwc_to_nchw(yn, B, O, Ho, Wo),)

    def backward(self, inputs, grad_outputs):
        x, W, b = inputs
        (gy,) = grad_outputs
        B, C, H, Wd = x.shape
        O, _, kh, kw = W.shape
        Ho, Wo = gy.shape[2:]
        xn, gn = nchw_to_nhwc(x), nchw_to_nhwc(gy)
        wi = W.permute(0, 2, 3, 1).contiguous()
        dxn = torch.empty(B * H * Wd, C, dtype=torch.float32, device=x.device)
        dwi = torch.zeros_like(wi)
        db = torch.zeros(O, dtype=torch.float32, device=x.device)
        L = lib()
        L.call("pivp_conv2d_dgrad", _p(gn), O, 0, B, Ho, Wo, O, _p(wi), 0, kh, kw, self.s, self.p, _p(dxn), C, 0, H, Wd, C, 0, 0, _s(x))
        L.call("pivp_conv2d_wgrad", _p(xn), C, 0, B, H, Wd, C, _p(gn), O, 0, Ho, Wo, O, kh, kw, self.s, self.p, _p(dwi), _p(db), _s(x))
        return nhwc_to_nchw(dxn, B, C, H, Wd), dwi.permute(0, 3, 1, 2).contiguous(), db


class Deconvolution2DFunction(object):
    """L.Deconvolution2D with explicit outsize (A.3); W in Chainer layout (in,out,kh,kw)."""

    def __init__(self, stride, pad, outsize):
        self.s, self.p, self.outsize = stride, pad, outsize

    def forward(self, inputs):
        x, W, b = inputs
        B, Ci, ih, iw = x.shape
        _, Co, kh, kw = W.shape
        oh, ow = self.outsize
        xn = nchw_to_nhwc(x)
        wi = W.permute(0, 2, 3, 1).contiguous()
        yn = torch.empty(B * oh * ow, Co, dtype=torch.float32, device=x.device)
        lib().call("pivp_conv2d_dgrad", _p(xn), Ci, 0, B, ih, iw, Ci, _p(wi), _p(b), kh, kw, self.s, self.p, _p(yn), Co, 0, oh, ow, Co, 0, 0, _s(x))
        return (nhwc_to_nchw(yn, B, Co, oh, ow),)

    def backward(self, inputs, grad_outputs):
        x, W, b = inputs
        (gy,) = grad_outputs
        B, Ci, ih, iw = x.shape
        _, Co, kh, kw = W.shape
        oh, ow = self.outsize
        xn, gn = nchw_to_nhwc(x), nchw_to_nhwc(gy)
        wi = W.permute(0, 2, 3, 1).contiguous()
        dxn = torch.empty(B * ih * iw, Ci, dtype=torch.float32, device=x.device)
        dwi = torch.zeros_like(wi)
        db = torch.zeros(Co, dtype=torch.float32, device=x.device)
        L = lib()
        L.call("pivp_conv2d_fwd", _p(gn), Co, 0, B, oh, ow, Co, _p(wi), 0, Ci, kh, kw, self.s, self.p, _p(dxn), Ci, 0, ih, iw, 0, 0, _s(x))
        L.call("pivp_conv2d_wgrad", _p(gn), Co, 0, B, oh, ow, Co, _p(xn), Ci, 0, ih, iw, Ci, kh, kw, self.s, self.p, _p(dwi), 0, _s(x))
        L.call("pivp_colsum", _p(gn), Co, 0, B * oh * ow, Co, _p(db), _s(x))
        return nhwc_to_nchw(dxn, B, Ci, ih, iw), dwi.permute(0, 3, 1, 2).contiguous(), db


class LayerNormalizationFunction(object):
    """LayerNormalizationConv2D (train_model.py:186-208): per-sample LN over C*H*W, per-element gamma/beta in CHW order."""

    def __init__(self, relu=False):
        self.relu = 1 if relu else 0

    def forward(self, inputs):
        x, gamma, beta = inputs
        B, C, H, W = x.shape
        L = lib()
        xn = nchw_to_nhwc(x)
        gi = gamma.reshape(C, H, W).permute(1, 2, 0).contiguous().reshape(-1)
        bi = beta.reshape(C, H, W).permute(1, 2, 0).contiguous().reshape(-1)
        yn = torch.empty_like(xn)
        self.stats = torch.empty(B, 2, dtype=torch.float32, device=x.device)
        nb = max(16, L.query("pivp_layernorm_workspace_bytes", B, C * H * W))
        ws = torch.empty(nb, dtype=torch.uint8, device=x.device)
        L.call("pivp_layernorm_fwd", _p(xn), C, 0, _p(gi), _p(bi), B, H * W, C, 1e-6, _p(yn), C, 0, 0, 0, 0, 0, 0, 0, self.relu,
               _p(self.stats), _p(ws), nb, _s(x))
        return (nhwc_to_nchw(yn, B, C, H, W),)

    def backward(self, inputs, grad_outputs):
        x, gamma, beta = inputs
        (gy,) = grad_outputs
        B, C, H, W = x.shape
        L = lib()
        xn, gn = nchw_to_nhwc(x), nchw_to_nhwc(gy)
        gi = gamma.reshape(C, H, W).permute(1, 2, 0).contiguous().reshape(-1)
        bi = beta.reshape(C, H, W).permute(1, 2, 0).contiguous().reshape(-1)
        dxn = torch.empty_like(xn)
        dg, db = torch.zeros_like(gi), torch.zeros_like(bi)
        nb = max(16, L.query("pivp_layernorm_workspace_bytes", B, C * H * W))
        ws = torch.empty(nb, dtype=torch.uint8, device=x.device)
        L.call("pivp_layernorm_bwd", _p(xn), C, 0, _p(gn), C, 0, 0, 0, 0, _p(gi), _p(bi), _p(self.stats), B, H * W, C, self.relu,
               _p(dxn), C, 0, _p(dg), _p(db), _p(ws), nb, _s(x))
        to_chw = lambda v: v.reshape(H, W, C).permute(2, 0, 1).contiguous().reshape(-1)
        return nhwc_to_nchw(dxn, B, C, H, W), to_chw(dg), to_chw(db)
