"""Backward of the reference call form of StatelessCDNA / DNA / STP (train_model.py:293-351, 368-417, 434-475): the un-fused
transformation list + enc7, with the list's gradient given entry by entry (None = no gradient, as Chainer's grad_outputs).

Checked against the float64 oracle (oracle/model.py cdna_transform / dna_transform / stp_transform through npgrad), against the fused
backward of the same math (the list composited with the mask softmax, ref:725-728), at the link level in Chainer layout, under CUDA-graph
capture, and for the error contract of the C-ABI (CPU).  Tolerances as tests/test_gpu_ops.py: gradients 1e-3 relative to the tensor's
max-abs, the looser sampler bounds for STP.
"""
import ctypes
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import model as OM
from oracle import npgrad as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FWD_TOL = 1e-4
GRAD_TOL = 1e-3


def rel(a, b):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    return float(np.abs(a.astype(np.float64) - b).max() / (np.abs(b).max() + 1e-30))


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


@pytest.fixture(scope="module")
def pk():
    import pivp_b200
    pivp_b200.lib()
    return pivp_b200


# ---------------------------------------------------------------------------------------------- float64 oracle of the three lists
# The oracle's transforms start from enc6 / hidden5 and the link's own layers.  With identity layers (1x1 deconvolution W = I, b = 0;
# kernel Linear W = I, b = 0; for STP s = relu([x; -x]) and theta_raw = [I, -I] s = x) they are exactly the maps of the C-ABI entry
# points, and the gradients of enc6 / hidden5 are those of enc7_pre / kern_raw / theta_raw.
def oracle_list(mt, prev, e, aux, M, R, Re, oob="zeros"):
    """-> (list entries, enc7, grads dict prev / enc7_pre / aux) of loss = sum_i <R_i, list_i> + <Re, enc7> (R_i / Re may be None)."""
    B, _, H, W = prev.shape
    ne = e.shape[1]
    P = {"model/enc7/W": G.Var(np.eye(ne).reshape(ne, ne, 1, 1)), "model/enc7/b": G.Var(np.zeros(ne))}
    vp, ve = G.Var(prev.astype(np.float64)), G.Var(e.astype(np.float64))
    va = None if aux is None else G.Var(aux.astype(np.float64))
    cfg = types.SimpleNamespace(num_masks=M, stp_oob=oob)
    if mt == "CDNA":
        n = 25 * M
        P.update({"model/cdna_kerns/W": G.Var(np.eye(n)), "model/cdna_kerns/b": G.Var(np.zeros(n))})
        out, enc7 = OM.cdna_transform(P, cfg, ve, va, vp, {})
    elif mt == "DNA":
        out, enc7 = OM.dna_transform(P, cfg, ve, vp, {})
    else:
        P.update({"model/stp_input/W": G.Var(np.concatenate([np.eye(6), -np.eye(6)])), "model/stp_input/b": G.Var(np.zeros(12)),
                  "model/identity_params/W": G.Var(np.concatenate([np.eye(6), -np.eye(6)], 1)), "model/identity_params/b": G.Var(np.zeros(6))})
        out, enc7 = OM.stp_transform(P, cfg, ve, va, vp, {})
    terms = [G.sum_(o * G.Var(r.astype(np.float64)), (0, 1, 2, 3)) for o, r in zip(out, R) if r is not None]
    if Re is not None:
        terms.append(G.sum_(enc7 * G.Var(Re.astype(np.float64)), (0, 1, 2, 3)))
    loss = terms[0]
    for t in terms[1:]:
        loss = loss + t
    G.backward(loss)
    z = lambda v, like: np.zeros(like.shape) if v.grad is None else v.grad      # no path from the loss: zero gradient
    return [o.data for o in out], enc7.data, {"prev": vp.grad if mt == "DNA" else z(vp, prev), "enc7_pre": z(ve, e),
                                              "aux": None if aux is None else z(va, aux)}


def make_inputs(rs, mt, B, H, W, M):
    prev = rs.rand(B, 3, H, W).astype(np.float32)
    e = rs.standard_normal((B, 25 if mt == "DNA" else 3, H, W)).astype(np.float32)
    aux = {"CDNA": lambda: rs.standard_normal((B, 25 * M)).astype(np.float32),       # about half the taps clamped to RELU_SHIFT
           "STP": lambda: (0.4 * rs.standard_normal((B, 6))).astype(np.float32),      # a good share of the samples fall outside
           "DNA": lambda: None}[mt]()
    return prev, e, aux


def list_len(mt, M):
    return {"CDNA": M + 1, "DNA": 1, "STP": M}[mt]


def make_grads(rs, mt, B, H, W, M, nulls):
    """Random R_i for every list entry and R_e for enc7; with `nulls` some entries (always the last, for CDNA the one the reference
    composite's zip drops) and R_e are None."""
    L = list_len(mt, M)
    R = [rs.standard_normal((B, 3, H, W)).astype(np.float32) for _ in range(L)]
    Re = rs.standard_normal((B, 25 if mt == "DNA" else 3, H, W)).astype(np.float32)
    if nulls:
        R = [None if (i % 3 == 2 or i == L - 1) and L > 1 else r for i, r in enumerate(R)]
        Re = None
    return R, Re


def function(pk, mt, M, oob="zeros"):
    F = pk.functions
    return {"CDNA": lambda: F.CDNATransformFunction(M), "DNA": lambda: F.DNATransformFunction(),
            "STP": lambda: F.STPTransformFunction(M, oob)}[mt]()


def run_function(pk, mt, M, prev, e, aux, R, Re, oob="zeros"):
    f = function(pk, mt, M, oob)
    ins = (cu(prev), cu(e)) + (() if aux is None else (cu(aux),))
    outs = f.forward(ins)
    gouts = tuple(None if r is None else cu(r) for r in R) + (None if Re is None else cu(Re),)
    return outs, f.backward(ins, gouts)


# ---------------------------------------------------------------------------------------------- 1. op level against float64
SHAPES = [(2, 64, 64, 10), (3, 16, 24, 3), (1, 8, 8, 1), (2, 24, 40, 7)]


@pytest.mark.gpu
@pytest.mark.parametrize("nulls", [False, True])
@pytest.mark.parametrize("B,H,W,M", SHAPES)
def test_cdna_list_bwd_against_float64(pk, B, H, W, M, nulls):
    rs = np.random.RandomState(31)
    prev, e, k = make_inputs(rs, "CDNA", B, H, W, M)
    R, Re = make_grads(rs, "CDNA", B, H, W, M, nulls)
    out_ref, e7_ref, gr = oracle_list("CDNA", prev, e, k, M, R, Re)
    outs, (dp, de, dk) = run_function(pk, "CDNA", M, prev, e, k, R, Re)
    assert len(outs) == M + 2
    for o, w in zip(outs, out_ref + [e7_ref]):
        assert rel(o, w) < FWD_TOL
    assert rel(de, gr["enc7_pre"]) < GRAD_TOL and rel(dk, gr["aux"]) < GRAD_TOL and rel(dp, gr["prev"]) < GRAD_TOL
    if nulls:
        assert torch.all(dk.reshape(B, M, 25)[:, M - 1] == 0)        # the last entry had no gradient: its kernel gets exactly zero


@pytest.mark.gpu
@pytest.mark.parametrize("nulls", [False, True])
@pytest.mark.parametrize("B,H,W,M", SHAPES)
def test_dna_list_bwd_against_float64(pk, B, H, W, M, nulls):
    rs = np.random.RandomState(32)
    prev, e, _ = make_inputs(rs, "DNA", B, H, W, 1)
    R, Re = make_grads(rs, "DNA", B, H, W, 1, False)
    if nulls:                                                        # one of the two gradients missing, by shape
        R, Re = ([None], Re) if M % 2 else (R, None)
    out_ref, e7_ref, gr = oracle_list("DNA", prev, e, None, 1, R, Re)
    assert gr["prev"] is None                                        # the taps are detached (ref:404)
    outs, (dp, de) = run_function(pk, "DNA", 1, prev, e, None, R, Re)
    assert dp is None
    assert rel(outs[0], out_ref[0]) < FWD_TOL and rel(outs[1], e7_ref) < FWD_TOL
    assert rel(de, gr["enc7_pre"]) < GRAD_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("nulls", [False, True])
@pytest.mark.parametrize("B,H,W,M,oob", [(2, 64, 64, 10, "zeros"), (2, 64, 64, 10, "border"), (3, 16, 24, 3, "zeros"),
                                         (1, 8, 8, 1, "zeros"), (1, 8, 8, 1, "border"), (2, 24, 40, 7, "border")])
def test_stp_list_bwd_against_float64(pk, B, H, W, M, oob, nulls):
    rs = np.random.RandomState(33)
    prev, e, th = make_inputs(rs, "STP", B, H, W, M)
    R, Re = make_grads(rs, "STP", B, H, W, M, nulls)
    out_ref, e7_ref, gr = oracle_list("STP", prev, e, th, M, R, Re, oob)
    outs, (dp, de, dth) = run_function(pk, "STP", M, prev, e, th, R, Re, oob)
    assert len(outs) == M + 1
    for o, w in zip(outs, out_ref + [e7_ref]):
        assert rel(o, w) < 5e-4                                      # the sampler amplifies the rounding of the grid coordinates
    assert rel(de, gr["enc7_pre"]) < GRAD_TOL
    if all(r is None for r in R[1:]):                                # no sampled entry with a gradient: d_theta zero, d_prev zeroed
        assert torch.all(dth == 0) and torch.all(dp == 0)
        assert np.abs(gr["aux"]).max() == 0 and np.abs(gr["prev"]).max() == 0
    else:
        assert rel(dth, gr["aux"]) < 5e-3 and rel(dp, gr["prev"]) < 2e-3


# ---------------------------------------------------------------------------------------------- 2. benchmark geometry
@pytest.mark.gpu
def test_cdna_list_bwd_b32_per_sample_and_properties(pk):
    """B = 32, 64x64, 10 masks, every entry live, d_prev on: samples against the oracle one by one; batch reversal commutes bit for bit;
    linear in g; two calls bit-identical."""
    rs = np.random.RandomState(34)
    B, H, W, M = 32, 64, 64, 10
    prev, e, k = make_inputs(rs, "CDNA", B, H, W, M)
    R, Re = make_grads(rs, "CDNA", B, H, W, M, False)
    f = pk.functions.CDNATransformFunction(M)
    ins = (cu(prev), cu(e), cu(k))
    gouts = tuple(cu(r) for r in R) + (cu(Re),)
    dp, de, dk = f.backward(ins, gouts)
    for b in (0, 13, 31):
        sl = slice(b, b + 1)
        _, _, gr = oracle_list("CDNA", prev[sl], e[sl], k[sl], M, [r[sl] for r in R], Re[sl])
        assert rel(de[sl], gr["enc7_pre"]) < GRAD_TOL and rel(dk[sl], gr["aux"]) < GRAD_TOL and rel(dp[sl], gr["prev"]) < GRAD_TOL
    flip = lambda v: torch.flip(v, dims=[0]).contiguous()
    dp_r, de_r, dk_r = f.backward(tuple(flip(v) for v in ins), tuple(flip(g) for g in gouts))
    assert torch.equal(flip(dp_r), dp) and torch.equal(flip(de_r), de) and torch.equal(flip(dk_r), dk)
    dp2, de2, dk2 = f.backward(ins, tuple(2 * g for g in gouts))
    for a, b2 in ((dp, dp2), (de, de2), (dk, dk2)):
        assert rel(b2, 2 * a.double()) < 1e-6
    dp3, de3, dk3 = f.backward(ins, gouts)
    assert torch.equal(dk3, dk) and torch.equal(dp3, dp) and torch.equal(de3, de)


@pytest.mark.gpu
def test_stp_list_bwd_b32_per_sample_and_properties(pk):
    rs = np.random.RandomState(35)
    B, H, W, M = 32, 64, 64, 10
    prev, e, th = make_inputs(rs, "STP", B, H, W, M)
    R, Re = make_grads(rs, "STP", B, H, W, M, False)
    f = pk.functions.STPTransformFunction(M)
    ins = (cu(prev), cu(e), cu(th))
    gouts = tuple(cu(r) for r in R) + (cu(Re),)
    dp, de, dth = f.backward(ins, gouts)
    for b in (0, 13, 31):
        sl = slice(b, b + 1)
        _, _, gr = oracle_list("STP", prev[sl], e[sl], th[sl], M, [r[sl] for r in R], Re[sl])
        assert rel(de[sl], gr["enc7_pre"]) < GRAD_TOL and rel(dth[sl], gr["aux"]) < 5e-3 and rel(dp[sl], gr["prev"]) < 2e-3
    flip = lambda v: torch.flip(v, dims=[0]).contiguous()
    dp_r, de_r, dth_r = f.backward(tuple(flip(v) for v in ins), tuple(flip(g) for g in gouts))
    assert torch.equal(flip(de_r), de) and torch.equal(flip(dth_r), dth)
    assert rel(flip(dp_r), dp.double()) < 1e-6                        # d_prev is a scatter-add: summation order may differ
    dp2, de2, dth2 = f.backward(ins, tuple(2 * g for g in gouts))
    assert rel(de2, 2 * de.double()) < 1e-6 and rel(dth2, 2 * dth.double()) < 1e-6 and rel(dp2, 2 * dp.double()) < 1e-6
    _, _, dth3 = f.backward(ins, gouts)
    assert torch.equal(dth3, dth)


# ---------------------------------------------------------------------------------------------- 3. agreement with the fused backward
def mask_softmax(a, M):
    """ref:718-723: softmax over groups of (M+1) FLAT NCHW elements of relu(a) (B.1)."""
    z = np.maximum(a.astype(np.float64), 0).reshape(-1, M + 1)
    z = np.exp(z - z.max(1, keepdims=True))
    return (z / z.sum(1, keepdims=True)).reshape(a.shape)


@pytest.mark.gpu
@pytest.mark.parametrize("mt,B,H,W,M,oob", [("CDNA", 2, 64, 64, 10, "zeros"), ("CDNA", 3, 16, 24, 3, "zeros"), ("DNA", 2, 64, 64, 1, "zeros"),
                                            ("DNA", 3, 16, 24, 1, "zeros"), ("STP", 2, 64, 64, 10, "zeros"), ("STP", 3, 16, 24, 4, "border")])
def test_list_bwd_agrees_with_fused_bwd(pk, mt, B, H, W, M, oob):
    """The list fed g_list[i] = mu_{i+1} g (the reference composite, zip truncation included) gives the fused op's gradients."""
    rs = np.random.RandomState(36)
    prev, e, aux = make_inputs(rs, mt, B, H, W, M)
    a = (2 * rs.standard_normal((B, M + 1, H, W))).astype(np.float32)
    g = rs.standard_normal((B, 3, H, W)).astype(np.float32)
    mu = mask_softmax(a, M)
    L = list_len(mt, M)
    R = [(mu[:, i + 1:i + 2] * g).astype(np.float32) if i < M else None for i in range(L)]
    _, (dp, de, *rest) = run_function(pk, mt, M, prev, e, aux, R, None, oob)
    F = pk.functions
    fused = {"CDNA": lambda: F.CDNACompositeFunction(M), "DNA": lambda: F.DNACompositeFunction(), "STP": lambda: F.STPCompositeFunction(M, oob)}[mt]()
    fins = (cu(prev), cu(e), cu(a)) + (() if aux is None else (cu(aux),))
    fg = fused.backward(fins, (cu(g),))
    assert rel(de, fg[1]) < GRAD_TOL
    if mt == "DNA":
        return
    d_aux = rest[0]
    assert rel(d_aux, fg[3]) < GRAD_TOL
    assert rel(dp + cu(mu[:, 0:1] * g), fg[0]) < GRAD_TOL
    if mt == "CDNA":
        assert torch.all(d_aux.reshape(B, M, 25)[:, M - 1] == 0)    # B.3: the last kernel gets exactly zero gradient


# ---------------------------------------------------------------------------------------------- 4. link level
def oracle_step(mt, nm, H=32, B=2, T=3, oob="zeros"):
    cfg = OM.Config(mt, nm, schedsamp_k=900.0, height=H, width=H, stp_oob=oob, dtype=np.float64)
    params = OM.init_params(cfg)
    rs = np.random.RandomState(3)
    for k in sorted(params):                                   # biases off zero so that they matter
        if k.endswith("/b"):
            params[k] = params[k] + 0.1 * rs.standard_normal(params[k].shape)
    batch = OM.concat_examples(OM.synthetic_sequences(B, T, cfg))
    np.random.seed(99)
    return cfg, params, batch, OM.forward(params, batch, 6000, cfg)


LINK_PARAMS = {"CDNA": ("model/enc7/W", "model/enc7/b", "model/cdna_kerns/W", "model/cdna_kerns/b"),
               "DNA": ("model/enc7/W", "model/enc7/b"),
               "STP": ("model/enc7/W", "model/enc7/b", "model/stp_input/W", "model/stp_input/b", "model/identity_params/W",
                       "model/identity_params/b")}


@pytest.mark.gpu
@pytest.mark.parametrize("mt,nm,oob", [("CDNA", 10, "zeros"), ("CDNA", 4, "zeros"), ("DNA", 1, "zeros"), ("STP", 10, "zeros"),
                                       ("STP", 5, "border"), ("STP", 1, "zeros")])
def test_stateless_links_reference_call_form_backward(pk, mt, nm, oob):
    cfg, params, batch, ref = oracle_step(mt, nm, oob=oob)
    tr = ref["trace"][-1]
    t32 = lambda v: torch.from_numpy(np.ascontiguousarray(v, dtype=np.float32)).cuda()
    enc6, h5, prev = tr["encs"][6].data, tr["hiddens"][4].data, tr["prev_image"].data
    encs = [t32(x.data) for x in tr["encs"]]
    hiddens = [t32(x.data) for x in tr["hiddens"]]
    link = {"CDNA": pk.StatelessCDNA, "DNA": pk.StatelessDNA, "STP": pk.StatelessSTP}[mt](nm).load(params)
    B = prev.shape[0]
    kw = {"oob": oob} if mt == "STP" else {}
    transformed, enc7 = link(encs, hiddens, B, t32(prev), nm, 3, **kw)
    # oracle: the same link from enc6 / hidden5 / prev as leaves, loss = sum_i <R_i, list_i> + <Re, enc7>, the last CDNA entry without
    # gradient (the composite's zip)
    rs = np.random.RandomState(37)
    L = len(transformed)
    R = [rs.standard_normal(transformed[0].shape) if not (mt == "CDNA" and i == L - 1) else None for i in range(L)]
    Re = rs.standard_normal(enc7.shape)
    P = {k: G.Var(np.asarray(v, np.float64)) for k, v in params.items()}
    v6, vh, vp = G.Var(enc6.astype(np.float64)), G.Var(h5.astype(np.float64)), G.Var(prev.astype(np.float64))
    if mt == "CDNA":
        out, e7 = OM.cdna_transform(P, cfg, v6, vh, vp, {})
    elif mt == "DNA":
        out, e7 = OM.dna_transform(P, cfg, v6, vp, {})
    else:
        out, e7 = OM.stp_transform(P, cfg, v6, vh, vp, {})
    loss = G.sum_(e7 * G.Var(Re), (0, 1, 2, 3))
    for o, r in zip(out, R):
        if r is not None:
            loss = loss + G.sum_(o * G.Var(r), (0, 1, 2, 3))
    G.backward(loss)
    g6, gh, gp = link.backward([None if r is None else t32(r) for r in R], t32(Re))
    torch.cuda.synchronize()
    loose = 5e-3 if mt == "STP" else GRAD_TOL                            # the theta path goes through the sampler

    def check(got, v, like, tol, what):
        want = np.zeros(like.shape) if v.grad is None else v.grad      # no path from the loss (STP with one mask: theta unused)
        assert tuple(got.shape) == like.shape, what
        if np.abs(want).max() == 0:
            assert torch.all(got == 0), what
        else:
            assert rel(got, want) < tol, what
    check(g6, v6, enc6, GRAD_TOL, "enc6")
    if mt == "DNA":
        assert gh is None and gp is None and vp.grad is None
    else:
        check(gh, vh, h5, loose, "hidden5")
        check(gp, vp, prev, 2e-3 if mt == "STP" else GRAD_TOL, "prev")
    assert sorted(link.grads) == sorted(LINK_PARAMS[mt])
    for k in LINK_PARAMS[mt]:
        check(link.grads[k], P[k], params[k], GRAD_TOL if "enc7" in k else loose, k)


# ---------------------------------------------------------------------------------------------- 5. graph capture
@pytest.mark.gpu
@pytest.mark.parametrize("mt", ["CDNA", "DNA", "STP"])
def test_list_bwd_graph_capture_replays_the_eager_call(pk, mt):
    rs = np.random.RandomState(38)
    B, H, W, M = 4, 64, 64, 10 if mt != "DNA" else 1
    prev, e, aux = make_inputs(rs, mt, B, H, W, M)
    R, Re = make_grads(rs, mt, B, H, W, M, True)
    f = function(pk, mt, M)
    ins = (cu(prev), cu(e)) + (() if aux is None else (cu(aux),))
    gouts = tuple(None if r is None else cu(r) for r in R) + (None if Re is None else cu(Re),)
    eager = f.backward(ins, gouts)
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        captured = f.backward(ins, gouts)
    for t in captured:
        if t is not None:
            t.fill_(float("nan"))
    gr.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager, captured):
        assert (a is None) == (b is None)
        if a is None:
            continue
        if mt == "STP" and a.shape == ins[0].shape:                     # the STP d_prev is a scatter-add
            assert rel(b, a.double()) < 1e-6
        else:
            assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------- 6. error contract (CPU)
@pytest.fixture(scope="module")
def pk_cpu():
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.build()
    import pivp_b200
    return pivp_b200


def test_list_bwd_error_contract_without_gpu(pk_cpu):
    """Null pointers, a NULL g_list array, num_masks out of range and a short workspace are PIVP_EINVAL before any CUDA call (fake device
    pointers: nothing is dereferenced, nothing is launched)."""
    L = pk_cpu.lib()
    n0 = L.query("pivp_launch_count")
    B, H, W, M = 2, 64, 64, 10
    fake = 1 << 20
    gl = (ctypes.c_void_p * 65)(*([fake] * 65))
    ws = L.query("pivp_cdna_transform_bwd_workspace_bytes", B, H, W, M)
    assert ws == 4 * B * 8 * M * 25                                          # 8 bands of 8 rows at 64x64
    cdna = lambda g=gl, prev=fake, m=M, nb=ws: L.call("pivp_cdna_transform_bwd", g, fake, prev, fake, fake, fake, fake, fake, 0,
                                                       B, H, W, m, fake, nb, 0)
    wst = L.query("pivp_stp_transform_bwd_workspace_bytes", B, H, W, M)
    assert wst == 4 * B * 8 * 6
    stp = lambda g=gl, prev=fake, m=M, nb=wst: L.call("pivp_stp_transform_bwd", g, fake, prev, fake, fake, fake, fake, fake, 0,
                                                       B, H, W, m, 0, fake, nb, 0)
    dna = lambda g=gl, prev=fake, de=fake: L.call("pivp_dna_transform_bwd", g, fake, prev, fake, de, B, H, W, 0)
    bad = [lambda: cdna(prev=0), lambda: cdna(g=None), lambda: cdna(m=0), lambda: cdna(m=65), lambda: cdna(nb=ws - 1),
           lambda: stp(prev=0), lambda: stp(g=None), lambda: stp(m=0), lambda: stp(m=65), lambda: stp(nb=wst - 1),
           lambda: dna(prev=0), lambda: dna(g=None), lambda: dna(de=0)]
    for call in bad:
        with pytest.raises(pk_cpu.PivpError):
            call()
    assert L.query("pivp_launch_count") == n0
