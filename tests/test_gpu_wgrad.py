"""Deferred tensor-core weight gradients against float64, at the benchmark shapes and at the kernel edges.

Every reference is float64, computed with torch from the SAME bf16-rounded operands the kernels read.  A product of two bf16 values
is exact in fp32, so the only difference left is the order of the fp32 accumulation (in TMEM, across the K splits, in the reduce).
Errors are max-abs over max|reference| per tensor, bounded by TOL.

  * test_deferred_wgrad_b32: TensorCorePlan.wgrad_all() of a CDNA 64x64 bf16 engine at B = 32, T = 10 (SB = 288 images per GEMM, the
    benchmark's split plans), in the three orders the training step issues it, against operation-level references (conv2d weight
    gradient, stride-2 convolution, stride-2 transposed convolution by autograd, column sums) in Chainer layout.  That checks the
    plan's tap / phase / channel-offset tables as well as the GEMMs; every other gradient element must keep its prefill bit for bit.
  * test_wgrad_kernel_edges: the two C entry points directly, at the shapes production does not reach: the split-K workspace and both
    branches of its reduce, an operand ring too small for the TMA epilogue, N4 < 128 accumulator rows clipped by the TMA reduce-add,
    workspace and dW bounds.
  * test_linear_wgrad_steps: the kernel Linear's weight gradient over all time steps (fast kernel and per-step path).
  * unaligned dW / workspace: rejected with PivpError before any CUDA call (the CPU test runs without a GPU).

Each tensor of the b32 test also shows that TOL can fail: dropping the last 64-pixel K block of the last image (the tail of the
last K split) from the reference moves it by more than 10 x TOL of max-abs.

Measured on a B200 (1000 W power limit, two runs), max-abs error over max|reference|: b32 weight gradients 5.3e-7 ... 1.86e-5
(worst lstm7/conv/W; the ConvLSTM layers contract K = 294,912 down to 18,432 pixels), bias gradients <= 2.0e-6, kernel edge cases
<= 6.1e-7, linear_wgrad_steps <= 7.9e-7, alike in all three orders.  TOL = 2e-4 keeps 10x headroom above the worst; the smallest
effect of one K block is 1.35e-2 (lstm7/conv/b), 6.7x above 10 x TOL.  The float64 references of the b32 test take about 2 s, the
GPU tests of this file about 8 s.
"""
import ctypes
import os
import sys
import time

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch.nn.grad import conv2d_weight

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TOL = 2e-4


@pytest.fixture(scope="module")
def pk():
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.build()
    import pivp_b200
    return pivp_b200


def stream():
    return torch.cuda.current_stream().cuda_stream


def iarr(v):
    return (ctypes.c_int * len(v))(*v)


def tap_lists(taps):
    return iarr([t[0] for t in taps]), iarr([t[1] for t in taps]), iarr([t[2] for t in taps])


TAPS5 = [(t // 5 - 2, t % 5 - 2, 0) for t in range(25)]


def s2d_taps(cb):
    """3x3 stride-2 taps on a space-to-depth operand: tap k reads half-grid offset {0:-1, 1:0, 2:0}[k], phase {0:1, 1:0, 2:1}[k]."""
    tapdef = {0: (-1, 1), 1: (0, 0), 2: (0, 1)}
    return [(tapdef[ky][0], tapdef[kx][0], (tapdef[ky][1] * 2 + tapdef[kx][1]) * cb) for ky in range(3) for kx in range(3)]


# ---- split plans, as launch_wgrad5x5_halo and launch_wgrad plan them with the default tuning switches (for the tables; the per-tap
# kernel's count is also checked against its workspace query)
def halo_plan(SB, H, W, Cx, N4):
    tiles = (N4 + 127) // 128 * ((Cx + 63) // 64) * 4
    kb = SB * (H // 8) * (W // 8)
    s = max(1, min(148 // tiles, max(1, kb // 8)))
    kbps = -(-kb // s)
    return -(-kb // kbps), kbps


def taps_plan(SB, H, W, Cx, N4, ntaps):
    tmax = min(512 // Cx, ntaps)
    groups = -(-ntaps // tmax)
    tpg = -(-ntaps // groups)
    groups = -(-ntaps // tpg)
    tiles = (N4 + 127) // 128 * groups
    kb = SB * H * W // 64
    s = max(1, min(-(-296 // tiles), max(1, kb // 8)))
    kbps = -(-kb // s)
    return -(-kb // kbps), kbps


# ---- float64 references (NHWC tensors in, weight gradients out)
def ref_taps(A, X, H, W, Cx, N4, taps):
    """dW[n][t][c] = sum_p A[p][n] X[p + (dy_t, dx_t)][coff_t + c] over images of H x W pixels; out-of-image pixels read zero."""
    A = A[:, :N4].double()
    X = X.double().reshape(-1, H, W, X.shape[-1])
    pad = max(max(abs(t[0]), abs(t[1])) for t in taps)
    Xp = F.pad(X, (0, 0, pad, pad, pad, pad))
    out = [A.t() @ Xp[:, pad + dy:pad + dy + H, pad + dx:pad + dx + W, co:co + Cx].reshape(-1, Cx) for dy, dx, co in taps]
    return torch.stack(out, 1)


def nchw(t):
    return t.double().permute(0, 3, 1, 2).contiguous()


def ref_conv5x5(xh, dg):
    """ConvLSTM convolution (5x5, padding 2): (n, h, w, cx) input, (n, h, w, 4C) output gradient -> (4C, cx, 5, 5)."""
    return conv2d_weight(nchw(xh), (dg.shape[3], xh.shape[3], 5, 5), nchw(dg), padding=2)


def ref_conv_s2(x, dy):
    """Convolution2D(3x3, stride 2, pad 1): (n, 2h, 2w, cin) input, (n, h, w, cout) output gradient -> (cout, cin, 3, 3)."""
    return conv2d_weight(nchw(x), (dy.shape[3], x.shape[3], 3, 3), nchw(dy), stride=2, padding=1)


def ref_deconv_s2(x, dy):
    """Deconvolution2D(3x3, stride 2, pad 1, outsize 2h x 2w): (n, h, w, cin) input, (n, 2h, 2w, cout) output gradient -> (cin, cout, 3, 3)."""
    w = torch.zeros(x.shape[3], dy.shape[3], 3, 3, dtype=torch.float64, device=x.device, requires_grad=True)
    F.conv_transpose2d(nchw(x), w, stride=2, padding=1, output_padding=1).backward(nchw(dy))
    return w.grad


def last_block(t, square):
    """Copy of the last image of NHWC t with everything but its last 64-pixel K block zeroed: an 8 x 8 block in the bottom-right corner
    (halo kernel) or the last 64 pixels in raster order (per-tap kernel)."""
    x = t[-1:].double()
    keep = torch.zeros_like(x)
    h, w = x.shape[1], x.shape[2]
    if square:
        keep[:, h - 8:, w - 8:] = 1
    else:
        keep.view(1, h * w, -1)[:, h * w - 64:] = 1
    return x * keep


def maxrel(got, ref):
    return float(np.abs(np.asarray(got, np.float64) - ref).max() / (np.abs(ref).max() + 1e-300))


# =====================================================================================================================================
# unaligned dW / workspace: no CUDA call is made, so this runs without a GPU
def test_wgrad_rejects_unaligned_dw_and_workspace_without_gpu(pk):
    L = pk.lib()
    dy, dx, co = tap_lists(s2d_taps(64))
    for dW, ws in ((20, 32), (36, 64), (32, 20), (64, 40)):
        with pytest.raises(pk.PivpError) as ei:
            L.call("pivp_tc_wgrad5x5", 16, 16, 64, 4, 16, 16, 64, 128, dW, ws, 1 << 24, 0)
        assert "16-byte aligned" in str(ei.value)
        with pytest.raises(pk.PivpError) as ei:
            L.call("pivp_tc_wgrad_taps", 16, 64, 16, 256, 4, 16, 16, 64, 64, 9, dy, dx, co, dW, ws, 1 << 24, 0)
        assert "16-byte aligned" in str(ei.value)


# =====================================================================================================================================
# (a) the production deferred-gradient phase at the benchmark configuration
B32, T32 = 32, 10


class _Recorder(object):
    """Stands in for the engine's library handle: forwards every call and records (name, args, kernels launched)."""

    def __init__(self, L):
        self.L, self.calls = L, []

    def call(self, name, *args):
        n0 = self.L.query("pivp_launch_count")
        self.L.call(name, *args)
        self.calls.append((name, args, self.L.query("pivp_launch_count") - n0))

    def __getattr__(self, k):
        return getattr(self.L, k)


class _NoSync(object):
    def ready(self, name):
        pass


@pytest.fixture(scope="module")
def b32(pk):
    from pivp_b200 import engine as E, layout
    eng = E.Engine("CDNA", 10, True, 64, 64, compute="bf16")
    eng._workspace(B32, T32)
    tc = eng.tc
    S = T32 - 1
    SB = S * B32
    assert tc.S == S
    gen = torch.Generator(device="cuda")
    gen.manual_seed(20261020)
    rnd = lambda *shape, scale=1.0: torch.randn(*shape, generator=gen, device="cuda") * scale
    L, s = eng.L, stream()
    refs, deltas, shapes = {}, {}, {}
    t0 = time.time()
    # ConvLSTM layers: every element of xh_all (pad channels of lstm3, time step T-1 beyond the SB images) and dg_all is nonzero
    for li, (cin, C, lv) in enumerate(zip(E.LSTM_IN, E.LSTM_SIZES, E.LSTM_LEVEL)):
        h, w, cx = 64 // lv, 64 // lv, cin + C
        xa, da = tc.xh_all[li], tc.dg_all[li]
        xa.copy_(rnd(*xa.shape))
        da.copy_(rnd(*da.shape, scale=0.1))
        xh = xa[:S].reshape(SB, h, w, -1)[..., :cx]
        dg = da.reshape(SB, h, w, 4 * C)
        perm = torch.from_numpy(layout.gate_perm(C)).cuda()           # Chainer row r = internal row perm[r]
        name = "lstm%d/conv" % (li + 1)
        refs[name + "/W"] = ref_conv5x5(xh, dg)[perm]
        refs[name + "/b"] = dg.double().sum((0, 1, 2))[perm]
        deltas[name + "/W"] = ref_conv5x5(xh[-1:], last_block(dg, True))[perm]
        deltas[name + "/b"] = last_block(dg, True).sum((0, 1, 2))[perm]
        shapes[name + "/W"] = ("wgrad5x5", SB, h, w, cx, 4 * C, 25)
    # enc1 / enc2: the forward's space-to-depth input (pad channels of each phase block nonzero) and all 64 channels of d(pre-activation)
    for name, d in tc.s2f.items():
        h, w, cin, cout, cb = 64 // d["lv"], 64 // d["lv"], d["cin"], d["cout"], d["cb"]
        x = rnd(SB, 2 * h, 2 * w, cin).bfloat16().float()
        d["xs"].copy_(rnd(*d["xs"].shape))
        L.call("pivp_cast_bf16", x.data_ptr(), cin, 0, d["xs"].data_ptr(), 4 * cb, 0, SB * 4 * h * w, cin, 2 * h, 2 * w, 1, cb, s)
        a = tc.de_b[name]
        a.copy_(rnd(*a.shape, scale=0.1))
        dy = a.reshape(SB, h, w, -1)[..., :cout]
        refs[name + "/W"] = ref_conv_s2(x, dy)
        deltas[name + "/W"] = ref_conv_s2(x[-1:], last_block(dy, False))
        shapes[name + "/W"] = ("taps", SB, h, w, cin, cout, 9)
    # enc4 / enc5 / enc6: deconvolution inputs of all steps (the 32 pad channels of cat5_b nonzero), space-to-depth output gradients
    for name, xall in (("enc4", tc.hid5_b_all), ("enc5", tc.cat5_b_all), ("enc6", tc.cat6_b_all)):
        d = tc.dbw[name]
        h, w, cin, cout, cb = 64 // d["lv"], 64 // d["lv"], d["cin"], d["cout"], d["cb"]
        xall.copy_(rnd(*xall.shape))
        gy = (rnd(SB, 2 * h, 2 * w, cout) * 0.1).bfloat16().float()
        d["dys"].copy_(rnd(*d["dys"].shape))
        L.call("pivp_cast_bf16", gy.data_ptr(), cout, 0, d["dys"].data_ptr(), 4 * cb, 0, SB * 4 * h * w, cout, 2 * h, 2 * w, 1, cb, s)
        x = xall.reshape(SB, h, w, -1)[..., :cin]
        refs[name + "/W"] = ref_deconv_s2(x, gy)
        deltas[name + "/W"] = ref_deconv_s2(last_block(x, False), gy[-1:])
        shapes[name + "/W"] = ("taps", SB, h, w, cout, cin, 9)
    torch.cuda.synchronize()
    t_ref = time.time() - t0
    prefill = rnd(eng.nparam)
    torch.cuda.synchronize()
    return dict(eng=eng, tc=tc, prefill=prefill, t_ref=t_ref, shapes=shapes,
                refs={k: v.cpu().numpy() for k, v in refs.items()}, deltas={k: v.cpu().numpy() for k, v in deltas.items()})


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["branches", "early_then_all", "grad_sync"])
def test_deferred_wgrad_b32(pk, b32, mode, capsys):
    """TensorCorePlan.wgrad_all() at B = 32, T = 10: all twelve weight and seven bias gradients against float64 references, in the
    default parallel branches, after wgrad_early() (the order of the backward pipeline) and in the data-parallel sequential order."""
    eng, tc = b32["eng"], b32["tc"]
    if mode == "early_then_all" and not tc.wg_ws_early:
        pytest.skip("early weight-gradient branches are switched off (PIVP_WGRAD_STREAMS / PIVP_WGRAD_EARLY)")
    eng.flat_g.copy_(b32["prefill"])
    rec = _Recorder(eng.L)
    eng.L = rec
    try:
        cur = torch.cuda.current_stream()
        t0 = time.time()
        if mode == "early_then_all":
            sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
            sa.wait_stream(cur)
            sb.wait_stream(cur)
            tc.wgrad_early(sa, sb)
            tc.wgrad_all()
            cur.wait_stream(sa)
            cur.wait_stream(sb)
        else:
            tc.wgrad_all(_NoSync() if mode == "grad_sync" else None)
        torch.cuda.synchronize()
        t_gpu = time.time() - t0
    finally:
        eng.L = rec.L
    # every weight-gradient tensor is the target of exactly one GEMM call, every ConvLSTM bias of one column-sum call
    owner = {eng.g[k].data_ptr(): k for k in b32["refs"]}
    calls = {}
    for name, args, launched in rec.calls:
        dst = {"pivp_tc_wgrad5x5": 8, "pivp_tc_wgrad_taps": 13, "pivp_tc_colsum_bf16": 4}[name]
        key = owner[args[dst]]
        assert key not in calls, key
        calls[key] = (name, args, launched)
    assert sorted(calls) == sorted(b32["refs"])
    for key, (name, args, _) in calls.items():
        if name == "pivp_tc_wgrad5x5":
            assert ("wgrad5x5",) + tuple(args[3:8]) + (25,) == b32["shapes"][key], key
        elif name == "pivp_tc_wgrad_taps":
            assert ("taps",) + tuple(args[4:10]) == b32["shapes"][key], key
    got, pre = eng.export_chainer(eng.flat_g), eng.export_chainer(b32["prefill"])
    rows, bad = [], {}
    for key in sorted(b32["refs"]):
        ref, delta = b32["refs"][key], b32["deltas"][key]
        g = got[key].astype(np.float64) - pre[key].astype(np.float64)
        err = maxrel(g, ref)
        sens = float(np.abs(delta).max() / np.abs(ref).max())
        name, args, launched = calls[key]
        if key.endswith("/b"):
            plan = ""
        else:
            kind, SB, h, w, cx, n4, nt = b32["shapes"][key]
            sp, kbps = halo_plan(SB, h, w, cx, n4) if kind == "wgrad5x5" else taps_plan(SB, h, w, cx, n4, nt)
            plan = "%-8s %3d x %3d  %s" % (kind, sp, kbps, "TMA reduce-add" if launched == 1 else "workspace + reduce")
        rows.append((key, err, sens, plan))
        if err > TOL:
            bad[key] = ("error", err)
        if sens <= 10 * TOL:
            bad[key] = ("one K block is not visible at 10 x TOL", sens)
    # nothing outside the nineteen tensors was touched
    mask = torch.ones(eng.nparam, dtype=torch.bool, device="cuda")
    for key in b32["refs"]:
        sp = eng.spec[key]
        mask[sp.offset:sp.offset + sp.size] = False
    untouched = bool(torch.equal(eng.flat_g.view(torch.int32)[mask], b32["prefill"].view(torch.int32)[mask]))
    with capsys.disabled():
        print("\n[deferred wgrad, B=32 T=10, %s] float64 references %.1f s, wgrad + sync %.3f s, TOL %.1e" % (mode, b32["t_ref"], t_gpu, TOL))
        print("  %-16s %-10s %-12s %s" % ("tensor", "max err", "1 K block", "kernel  splits x 64-px blocks  epilogue"))
        for key, err, sens, plan in rows:
            print("  %-16s %.3e  %.3e    %s" % (key, err, sens, plan))
    assert untouched, "a weight-gradient GEMM wrote outside its tensor"
    assert not bad, bad


# =====================================================================================================================================
# (b) kernel-level edges through the C-ABI
EDGE_CASES = [
    # id, entry point, SB, H, W, Cx, N4, a_cs, x_cs, taps, epilogue, splits.  The workspace epilogues: Cx % 32 != 0 (both kernels), an
    # operand ring too small for two staging buffers (Cx > 192, per-tap kernel).  splitk_reduce_kernel adds more than 16 splits in chunks
    # with float4 atomics, up to 16 with a plain read-modify-write.
    ("halo_cx48_atomic_reduce", "5x5", 74, 16, 16, 48, 128, 128, 64, TAPS5, "workspace", 37),
    ("halo_cx48_plain_reduce", "5x5", 4, 16, 16, 48, 128, 128, 64, TAPS5, "workspace", 2),
    ("taps_cx48_atomic_reduce", "taps", 288, 16, 16, 48, 64, 64, 256, s2d_taps(64), "workspace", 144),
    ("taps_cx48_plain_reduce", "taps", 8, 16, 16, 48, 64, 64, 256, s2d_taps(64), "workspace", 4),
    ("taps_cx256_ring_too_small", "taps", 160, 8, 8, 256, 128, 128, 256, [(-1, -1, 0), (-1, 1, 0), (0, 0, 0), (1, -1, 0), (1, 1, 0)],
     "workspace", 20),
    ("taps_n4_32_tma_clip", "taps", 32, 8, 8, 64, 32, 64, 256, s2d_taps(64), "tma", 4),
    ("taps_n4_96_tma_clip", "taps", 16, 16, 16, 96, 96, 128, 512, s2d_taps(128), "tma", 8),
]

NEG0 = -2147483648          # bit pattern of -0.0f: any store or reduce-add (even of +0.0) changes it


def sentinel(n):
    return torch.full((n,), NEG0, dtype=torch.int32, device="cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("case", EDGE_CASES, ids=[c[0] for c in EDGE_CASES])
def test_wgrad_kernel_edges(pk, case, capsys):
    _, entry, SB, H, W, Cx, N4, a_cs, x_cs, taps, path, splits = case
    L = pk.lib()
    ntaps = len(taps)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(SB * 1000 + Cx + N4)
    P = SB * H * W
    A = (torch.randn(P, a_cs, generator=gen, device="cuda") * 0.1).bfloat16()        # channels N4..a_cs are nonzero and never read
    X = torch.randn(P, x_cs, generator=gen, device="cuda").bfloat16()                 # so are the channels no tap reaches
    if entry == "5x5":
        nb = L.query("pivp_tc_wgrad_workspace_bytes", SB, H, W, Cx, N4)
        sp, _ = halo_plan(SB, H, W, Cx, N4)
        assert nb >= sp * 128 * ((N4 + 127) // 128) * ntaps * Cx * 4
    else:
        nb = L.query("pivp_tc_wgrad_taps_workspace_bytes", SB, H, W, Cx, N4, ntaps)
        sp, _ = taps_plan(SB, H, W, Cx, N4, ntaps)
        assert nb == sp * 128 * ((N4 + 127) // 128) * ntaps * Cx * 4
    assert sp == splits
    # workspace of exactly the queried size, then a guard; dW a 16-byte aligned view between guards, room for 128 rows behind it
    guard = 1 << 14
    ws = sentinel(nb // 4 + guard)
    n = N4 * ntaps * Cx
    pre, post = 4, (128 - N4) * ntaps * Cx + guard
    buf = sentinel(pre + n + post)
    dW = buf[pre:pre + n].view(torch.float32)
    dW.copy_(torch.randn(n, generator=gen, device="cuda"))
    dW0 = dW.clone()
    n0 = L.query("pivp_launch_count")
    if entry == "5x5":
        L.call("pivp_tc_wgrad5x5", A.data_ptr(), X.data_ptr(), x_cs, SB, H, W, Cx, N4, dW.data_ptr(), ws.data_ptr(), nb, stream())
    else:
        dy, dx, co = tap_lists(taps)
        L.call("pivp_tc_wgrad_taps", A.data_ptr(), a_cs, X.data_ptr(), x_cs, SB, H, W, Cx, N4, ntaps, dy, dx, co, dW.data_ptr(),
               ws.data_ptr(), nb, stream())
    launched = L.query("pivp_launch_count") - n0
    ref = ref_taps(A, X, H, W, Cx, N4, taps).cpu().numpy()
    torch.cuda.synchronize()
    err = maxrel((dW.double() - dW0.double()).reshape(N4, ntaps, Cx).cpu().numpy(), ref)
    with capsys.disabled():
        print("\n[%s] SB %d %dx%d Cx %d N4 %d taps %d: %d splits, %s, max err %.3e" % (case[0], SB, H, W, Cx, N4, ntaps, sp,
              "TMA reduce-add" if launched == 1 else "workspace + reduce", err))
    assert launched == (1 if path == "tma" else 2)
    assert torch.equal(ws[nb // 4:], sentinel(guard)), "workspace written past the queried size"
    assert torch.equal(buf[:pre], sentinel(pre)) and torch.equal(buf[pre + n:], sentinel(post)), "dW written out of bounds"
    assert err <= TOL


@pytest.mark.gpu
def test_wgrad_rejects_unaligned_dw_and_workspace(pk):
    """Misaligned dW or workspace: PivpError, nothing launched, dW unchanged."""
    L = pk.lib()
    SB, H, W, Cx, N4 = 4, 16, 16, 64, 128
    A = torch.ones(SB * H * W, N4, device="cuda").bfloat16()
    X = torch.ones(SB * H * W, 256, device="cuda").bfloat16()
    n = N4 * 25 * Cx
    buf = torch.full((n + 64,), 0.5, device="cuda")
    ws = torch.zeros(max(L.query("pivp_tc_wgrad_workspace_bytes", SB, H, W, Cx, N4),
                         L.query("pivp_tc_wgrad_taps_workspace_bytes", SB, H, W, Cx, N4, 9)) + 64, dtype=torch.uint8, device="cuda")
    nb = ws.numel() - 64
    dy, dx, co = tap_lists(s2d_taps(64))
    n0 = L.query("pivp_launch_count")
    for dW, wsp in ((buf[1:].data_ptr(), ws.data_ptr()), (buf.data_ptr(), ws[4:].data_ptr())):
        with pytest.raises(pk.PivpError, match="16-byte aligned"):
            L.call("pivp_tc_wgrad5x5", A.data_ptr(), X.data_ptr(), 64, SB, H, W, Cx, N4, dW, wsp, nb, stream())
        with pytest.raises(pk.PivpError, match="16-byte aligned"):
            L.call("pivp_tc_wgrad_taps", A.data_ptr(), N4, X.data_ptr(), 256, SB, H, W, Cx, N4, 9, dy, dx, co, dW, wsp, nb, stream())
    torch.cuda.synchronize()
    assert L.query("pivp_launch_count") == n0
    assert bool((buf == 0.5).all())


# =====================================================================================================================================
# (c) kernel Linear weight gradient over all time steps
@pytest.mark.gpu
@pytest.mark.parametrize("B", [32, 40])          # 32: linear_dw_steps_kernel (the engine's b32 call); 40 > LW_B: the per-step path
def test_linear_wgrad_steps(pk, B, capsys):
    L = pk.lib()
    S, K, N = 9, 8192, 250
    gen = torch.Generator(device="cuda")
    gen.manual_seed(B)
    x = torch.randn(S, B, K, generator=gen, device="cuda")             # x rows at step stride B * K (the engine's hid5 stack)
    dy = torch.randn(S, B, N, generator=gen, device="cuda") * 0.1
    dW = torch.randn(N, K, generator=gen, device="cuda")
    db = torch.randn(N, generator=gen, device="cuda")
    dW0, db0 = dW.double(), db.double()
    L.call("pivp_linear_wgrad_steps", dy.data_ptr(), B * N, x.data_ptr(), B * K, K, dW.data_ptr(), db.data_ptr(), S, B, K, N, stream())
    ref_w = torch.einsum("sbn,sbk->nk", dy.double(), x.double())
    ref_b = dy.double().sum((0, 1))
    torch.cuda.synchronize()
    ew = float((dW.double() - dW0 - ref_w).abs().max() / ref_w.abs().max())
    eb = float((db.double() - db0 - ref_b).abs().max() / ref_b.abs().max())
    with capsys.disabled():
        print("\n[linear_wgrad_steps S=%d B=%d K=%d N=%d] max err dW %.3e, db %.3e" % (S, B, K, N, ew, eb))
    assert ew <= TOL and eb <= TOL
