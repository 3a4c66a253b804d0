"""Forward-only batched prediction (pivp_b200.Predictor): the frames of the training engine's rollout bit for bit, the float64 oracle in
test mode, a memory footprint that does not grow with the horizon, chunking and broadcasting, no interference with the training engine,
parameter updates seen by the next replay; and the kernel variants it runs on (no gate storage, in-place cell state, heads without y)."""
import gc
import os

import numpy as np
import pytest
import torch

from oracle import model as OM

pytestmark = pytest.mark.gpu

H = 64
NM = {"CDNA": 10, "DNA": 1, "STP": 10}


@pytest.fixture(scope="module")
def pk():
    import pivp_b200
    pivp_b200.lib()
    return pivp_b200


def make(pk, mt, compute, seed=4321):
    cfg = OM.Config(mt, NM[mt], height=H, width=H, dtype=np.float64, train=False)
    params = OM.init_params(cfg, seed=seed)
    m = pk.Model(NM[mt], is_cdna=mt == "CDNA", is_dna=mt == "DNA", is_stp=mt == "STP", height=H, width=H, compute=compute)
    m.load_params(params)
    m.train = False
    return m, cfg, params


def data(cfg, N, T, seed=1234):
    img, act, sta = OM.concat_examples(OM.synthetic_sequences(N, T, cfg, seed=seed))
    return img.astype(np.float32), act.astype(np.float32), sta.astype(np.float32)


def rollout(pk, m, img, act, sta):
    """Rollout on the training engine: frames (T-1, N, 3, H, W) and states (T-1, N, 5), cloned."""
    T, N = img.shape[0], img.shape[1]
    r = pk.Rollout(m, N, T, graph=True)
    r.load(img, act, sta)
    gen = torch.stack(list(r())).clone()
    states = torch.stack([s[:N] for s in m.gen_states]).clone()
    return gen, states


@pytest.mark.parametrize("N", [4, 3])
@pytest.mark.parametrize("compute", ["f32", "bf16"])
@pytest.mark.parametrize("mt", ["CDNA", "DNA", "STP"])
def test_predictor_equals_rollout_bit_for_bit(pk, mt, compute, N):
    T = 6
    m, cfg, _ = make(pk, mt, compute)
    img, act, sta = data(cfg, N, T)
    ctx = m.num_frame_before_prediction
    junk = img.copy()
    junk[ctx:] = np.random.RandomState(7).rand(T - ctx, N, 3, H, H).astype(np.float32)      # never read under feedself
    g1, s1 = rollout(pk, m, junk, act, sta)
    g2, s2 = rollout(pk, m, junk, act, sta)
    assert torch.equal(g1, g2) and torch.equal(s1, s2)                                      # the forward pass is deterministic
    p = pk.Predictor(m, N, T)
    for _ in range(2):                                                                      # second call replays the captured graph
        frames = p(img[:ctx], act[:T - 1], sta[0])
        torch.cuda.synchronize()
        assert frames.shape == (T - 1, N, 3, H, H) and frames.dtype == torch.float32 and frames.is_cuda
        assert tuple(p.gen_states.shape) == (T - 1, N, 5)
        assert torch.equal(frames, g1[:, :N]) and torch.equal(p.gen_states, s1)


@pytest.mark.parametrize("compute", ["f32", "bf16"])
@pytest.mark.parametrize("mt", ["CDNA", "DNA", "STP"])
def test_predictor_matches_oracle_test_mode(pk, mt, compute):
    N, T = 3, 8
    m, cfg, params = make(pk, mt, compute)
    img, act, sta = data(cfg, N, T)
    ref = OM.forward(params, (img.astype(np.float64), act.astype(np.float64), sta.astype(np.float64)), 0, cfg)
    assert ref["n_gt"] is None
    ctx = m.num_frame_before_prediction
    frames = pk.Predictor(m, N, T)(img[:ctx], act[:T - 1], sta[0]).double().cpu().numpy()
    errs = [np.linalg.norm(frames[t] - ref["gen_images"][t].data) / np.linalg.norm(ref["gen_images"][t].data) for t in range(T - 1)]
    print("\n%s %s relative L2 per predicted frame: %s" % (mt, compute, " ".join("%.3g" % e for e in errs)))
    for t, e in enumerate(errs):
        if compute == "f32":
            tol = 1e-4
        elif mt != "STP":
            tol = 2e-2
        else:
            # STP bf16: test_gpu_tc.py's 1e-1 over the three predicted frames it checks (T = 4).  Fed back through the bilinear sampler, the
            # bf16 error keeps growing with the horizon (measured on a B200: 0.024 0.019 0.062 0.114 0.216 0.315 0.325 for the seven
            # frames here), a property of the engine's STP bf16 path that
            # Predictor shares bit for bit (test_predictor_equals_rollout_bit_for_bit): later frames get a sanity bound only.
            tol = 1e-1 if t < 3 else 0.5
        assert e <= tol, (t, e)


def _peak(build_and_call):
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    keep = build_and_call()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    del keep
    gc.collect()
    torch.cuda.empty_cache()
    return peak


def test_predictor_memory_does_not_grow_with_the_horizon(pk):
    N = 64
    m, cfg, _ = make(pk, "CDNA", "bf16")
    img, act, sta = data(cfg, N, 20)
    ctx = m.num_frame_before_prediction
    c = torch.from_numpy(img[:ctx]).cuda()
    a = torch.from_numpy(act).cuda()
    s = torch.from_numpy(sta[0]).cuda()
    peak, peak_r = {}, {}
    for T in (6, 20):
        peak[T] = _peak(lambda: (lambda p: (p, p(c, a[:T - 1], s)))(pk.Predictor(m, N, T)))
    out_bytes = lambda T: (T - 1) * N * (3 * H * H + 5) * 4
    grow = peak[20] - peak[6]
    for T in (6, 20):
        mr, _, _ = make(pk, "CDNA", "bf16")
        peak_r[T] = _peak(lambda: (lambda r: (r, mr, r.load(img[:T], act[:T], sta[:T]), r()))(pk.Rollout(mr, N, T)))
        del mr
    print("\npeak allocated, bf16 CDNA 64x64, N=%d: Predictor T=6 %.1f MiB, T=20 %.1f MiB; Rollout T=6 %.1f MiB, T=20 %.1f MiB"
          % (N, peak[6] / 2**20, peak[20] / 2**20, peak_r[6] / 2**20, peak_r[20] / 2**20))
    assert grow <= out_bytes(20) - out_bytes(6) + 2**20, (grow, out_bytes(20) - out_bytes(6))
    assert peak[20] < peak_r[20]


def test_predictor_chunks_equal_one_launch(pk):
    T = 16
    m, cfg, _ = make(pk, "CDNA", "bf16")
    img, act, sta = data(cfg, 1024, T)
    ctx = m.num_frame_before_prediction
    c, a, s = torch.from_numpy(img[:ctx]).cuda(), torch.from_numpy(act[:T - 1]).cuda(), torch.from_numpy(sta[0]).cuda()
    big = pk.Predictor(m, 256, T)
    one = big(c[:, :256], a[:, :256], s[:256]).clone()
    one_s = big.gen_states.clone()
    small = pk.Predictor(m, 64, T)
    chunked = small(c[:, :256], a[:, :256], s[:256])
    assert chunked.shape == one.shape and torch.equal(chunked, one) and torch.equal(small.gen_states, one_s)
    del small, chunked
    all_rows = big(c, a, s)
    torch.cuda.synchronize()
    assert all_rows.shape == (T - 1, 1024, 3, H, H) and bool(torch.isfinite(all_rows).all())
    assert torch.equal(all_rows[:, :256], one) and torch.equal(big.gen_states[:, :256], one_s)


def test_predictor_broadcasts_a_context_batch_of_one(pk):
    N, T = 5, 6                                             # odd: the last chunk row is repeated on the bf16 path
    m, cfg, _ = make(pk, "CDNA", "bf16")
    img, act, sta = data(cfg, N, T)
    ctx = m.num_frame_before_prediction
    acts = np.random.RandomState(3).randn(T - 1, N, 5).astype(np.float32)                  # N candidate action sequences
    p = pk.Predictor(m, N, T)
    b = p(img[:ctx, :1], acts, sta[0, :1]).clone()
    bs = p.gen_states.clone()
    rep = p(np.repeat(img[:ctx, :1], N, axis=1), acts, np.repeat(sta[0, :1], N, axis=0))
    assert torch.equal(b, rep) and torch.equal(bs, p.gen_states)


def _ws_pointers(ws):
    out = []
    for k in sorted(ws, key=str):
        v = ws[k]
        for x in (v if isinstance(v, list) else list(v.values()) if isinstance(v, dict) else [v]):
            for y in (x if isinstance(x, list) else [x]):
                if isinstance(y, torch.Tensor):
                    out.append((k, y.data_ptr()))
    return out


def test_predictor_leaves_the_training_engine_untouched(pk):
    m, cfg, _ = make(pk, "CDNA", "bf16")
    img, act, sta = data(cfg, 4, 6)
    r = pk.Rollout(m, 4, 6, graph=True)
    r.load(img, act, sta)
    before = torch.stack(list(r())).clone()
    e = m.engine
    ws, tc, ptrs = e.ws, e.tc, _ws_pointers(e.ws)
    img2, act2, sta2 = data(cfg, 8, 10, seed=5)
    pk.Predictor(m, 8, 10)(img2[:2], act2[:9], sta2[0])                                     # another (N, T) on the same model
    after = torch.stack(list(r())).clone()                                                  # replay of the graph captured before
    torch.cuda.synchronize()
    assert torch.equal(before, after)
    assert e.ws is ws and e.tc is tc and _ws_pointers(e.ws) == ptrs


def test_predictor_follows_parameter_updates(pk):
    N, T = 4, 6
    m, cfg, params = make(pk, "CDNA", "bf16")
    img, act, sta = data(cfg, N, T)
    p = pk.Predictor(m, N, T)
    old = p(img[:2], act[:T - 1], sta[0]).clone()
    opt = pk.Adam().setup(m)
    torch.manual_seed(0)
    m.engine.flat_g.normal_()
    opt.apply()
    new = p(img[:2], act[:T - 1], sta[0]).clone()
    want, _ = rollout(pk, m, img, act, sta)
    assert not torch.equal(new, old) and torch.equal(new, want)
    m.load_params({k: (v * 0.9).astype(np.float32) for k, v in params.items()})
    new2 = p(img[:2], act[:T - 1], sta[0]).clone()
    want2, _ = rollout(pk, m, img, act, sta)
    assert not torch.equal(new2, new) and torch.equal(new2, want2)


def test_predictor_shape_errors_launch_nothing(pk):
    m, cfg, _ = make(pk, "CDNA", "f32")
    img, act, sta = data(cfg, 2, 6)
    p = pk.Predictor(m, 2, 6)
    L = pk.lib()
    n0, c0 = L.query("pivp_launch_count"), L.launches
    bad = [(img[:1], act[:5], sta[0]),                       # fewer context frames than context_frames
           (img[:2], act[:4], sta[0]),                       # T-1 = 4 action steps for T = 6
           (img[:2, :1], act[:5], sta[0, :1][:, :4]),        # state of 4 components
           (img[:2], act[:5], sta[0][None]),                 # state with an extra dimension
           (img[:2].astype(np.float64), act[:5], sta[0]),    # dtype
           (np.concatenate([img[:2]] * 2, axis=1)[:, :3], act[:5], sta[0])]     # context batch 3 for N = 2
    for c, a, s in bad:
        with pytest.raises(ValueError):
            p(c, a, s)
    assert L.query("pivp_launch_count") == n0 and L.launches == c0


# ----------------------------------------------------------------------------- kernel level
def _cell(pk, li, B, flags, in_place, lnp):
    """One launch of pivp_tc_conv5x5 mode 1 on ConvLSTM layer li's geometry with fixed random operands."""
    from pivp_b200.engine import LSTM_IN, LSTM_SIZES, LSTM_LEVEL
    cin, C, lv = LSTM_IN[li], LSTM_SIZES[li], LSTM_LEVEL[li]
    h = w = H // lv
    M, Kp = B * h * w, (cin + C + 63) // 64 * 64
    g = torch.Generator(device="cuda").manual_seed(li)
    rnd = lambda *s: torch.randn(*s, device="cuda", generator=g)
    xin = (rnd(M, Kp) * 0.5).to(torch.bfloat16)
    wt = (rnd(4 * C, 25, Kp) * 0.05).to(torch.bfloat16)
    bias, c_prev = rnd(4 * C), rnd(M, C)
    gates = torch.zeros(M, 4 * C, dtype=torch.bfloat16, device="cuda")
    c_out = c_prev.clone() if in_place else torch.zeros(M, C, device="cuda")
    xh = torch.zeros(M, cin + C, device="cuda")
    hb = torch.zeros(M, Kp, dtype=torch.bfloat16, device="cuda")
    part = torch.zeros(B * h * w * C // 4096 * 2 + 64, device="cuda") if lnp else None
    pk.lib().call("pivp_tc_conv5x5", xin.data_ptr(), Kp, B, h, w, Kp, wt.data_ptr(), 4 * C, 128, 1, bias.data_ptr(), 0, 0, 0,
                  gates.data_ptr() if flags & 2 else 0, c_out.data_ptr() if in_place else c_prev.data_ptr(), c_out.data_ptr(),
                  xh.data_ptr(), cin + C, cin, hb.data_ptr(), Kp, cin, 0, 0, 0, C, 1.0, flags, 0 if part is None else part.data_ptr(),
                  torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return dict(c=c_out, h=xh, hb=hb, part=part, gates=gates)


# the epilogue variants: TMA stores (default), staged per-thread stores (PIVP_TC_HALO_TMA=0), the per-tap kernel (PIVP_TC_HALO=0)
@pytest.mark.parametrize("variant", [{}, {"PIVP_TC_HALO_TMA": "0"}, {"PIVP_TC_HALO": "0"}])
@pytest.mark.parametrize("li,B", [(0, 2), (4, 4)])         # lstm1 on 32x32 maps; lstm5 on 8x8 maps (pair geometry of the halo kernel)
def test_cell_without_gate_store_and_in_place_state(pk, monkeypatch, li, B, variant):
    for k, v in variant.items():
        monkeypatch.setenv(k, v)
    lnp = li == 0 and "PIVP_TC_HALO" not in variant          # LayerNorm partials: halo kernel, tiled geometry only
    ref = _cell(pk, li, B, 2, False, lnp)
    assert bool(ref["gates"].abs().sum() > 0)
    for flags, in_place in ((4, False), (4, True), (2, True)):
        got = _cell(pk, li, B, flags, in_place, lnp)
        for k in ("c", "h", "hb") + (("part",) if lnp else ()):
            assert torch.equal(got[k], ref[k]), (flags, in_place, k)
        if flags & 4:
            assert not bool(got["gates"].abs().sum() > 0)    # no gate store


def test_heads_without_normalised_rows(pk):
    B, HW, Ne, Nh = 2, H * H, 3, 14
    g = torch.Generator(device="cuda").manual_seed(0)
    rnd = lambda *s: torch.randn(*s, device="cuda", generator=g)
    x, gamma, beta = rnd(B * HW, 64), rnd(HW * 64) * 0.2 + 1.0, rnd(HW * 64) * 0.2
    Wt, bias = rnd(Nh, 64) * 0.1, rnd(Nh)
    xs = x.view(B, -1, 4096).double()                          # (mean, M2) partials of 4096-value chunks
    mean = xs.mean(-1)
    part = torch.stack([mean, ((xs - mean[..., None]) ** 2).sum(-1)], -1).float().contiguous()
    na, nb, ny = B * Ne * HW, B * (Nh - Ne) * HW, B * HW * 64
    runs = []
    for with_y in (True, False):
        buf = torch.full((na + nb + ny,), 12345.0, device="cuda")          # planes, then a y-sized guard region right behind them
        y = torch.zeros(B * HW, 64, device="cuda")
        stats = torch.zeros(B, 2, device="cuda")
        pk.lib().call("pivp_heads_fwd_ln", x.data_ptr(), 64, 0, gamma.data_ptr(), beta.data_ptr(), part.data_ptr(), 1e-6, stats.data_ptr(),
                      y.data_ptr() if with_y else 0, 64, 0, Wt.data_ptr(), bias.data_ptr(), buf.data_ptr(), Ne, buf[na:].data_ptr(), Nh,
                      B, HW, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        runs.append((buf, stats, y))
    (b1, s1, y1), (b2, s2, y2) = runs
    assert torch.equal(b1[:na + nb], b2[:na + nb]) and torch.equal(s1, s2)
    assert bool((b2[na + nb:] == 12345.0).all()) and bool((y2 == 0).all()) and bool(y1.abs().sum() > 0)
