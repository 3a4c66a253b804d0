"""Cross-entropy-method planning (pivp_b200.CEMPlanner): the three kernels against float64 NumPy restatements (goal cost, sampling
statistics, elite refit with ties / NaN / inf), the CEM loop through the C-ABI on a known optimum, and the planner end to end -- costs and
best sequence reproduced by a fresh Predictor bit for bit, graph = eager, seeds, parameter updates, no interference with the training
engine, memory."""
import gc

import numpy as np
import pytest
import torch

from oracle import model as OM

pytestmark = pytest.mark.gpu

NM = {"CDNA": 10, "DNA": 1, "STP": 10}


@pytest.fixture(scope="module")
def pk():
    import pivp_b200
    pivp_b200.lib()
    return pivp_b200


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return 0 if t is None else t.data_ptr()


def make(pk, mt, compute, H=64, seed=4321):
    cfg = OM.Config(mt, NM[mt], height=H, width=H, dtype=np.float64, train=False)
    params = OM.init_params(cfg, seed=seed)
    m = pk.Model(NM[mt], is_cdna=mt == "CDNA", is_dna=mt == "DNA", is_stp=mt == "STP", height=H, width=H, compute=compute)
    m.load_params(params)
    m.train = False
    return m, cfg, params


def data(cfg, N, T, seed=1234):
    img, act, sta = OM.concat_examples(OM.synthetic_sequences(N, T, cfg, seed=seed))
    return img.astype(np.float32), act.astype(np.float32), sta.astype(np.float32)


# ----------------------------------------------------------------------------- goal cost
def goal_cost(pk, gen, Bp, N, goal, per_step, w, cost):
    T, H, W = gen.shape[0] + 1, gen.shape[-2], gen.shape[-1]
    pk.lib().call("pivp_goal_cost", _p(gen), T, Bp, N, H, W, _p(goal), int(per_step), _p(w), _p(cost), _st())


def ref_cost(gen, goal, w, N):
    g = gen[:, :N].astype(np.float64)
    q = goal.astype(np.float64)
    q = q[:, None] if q.ndim == 4 else q[None, None]
    per = ((g - q) ** 2).mean(axis=(2, 3, 4))                              # (T-1, N)
    return (w.astype(np.float64)[:, None] * np.where(w[:, None] == 0, 0.0, per)).sum(0)


@pytest.mark.parametrize("H,N,Bp,T,per_step,wkind", [
    (64, 7, 10, 6, True, "rand"),           # odd N, Bp > N
    (64, 7, 8, 6, False, "last"),           # one goal image, default-style weights
    (64, 5, 6, 2, False, "ones"),           # S = 1: one predicted frame
    (64, 9, 9, 7, True, "zeros"),           # zero-weight steps hold NaN: never read
    (128, 3, 4, 4, True, "rand"),
    (128, 4, 6, 5, False, "zeros")])
def test_goal_cost_matches_float64(pk, H, N, Bp, T, per_step, wkind):
    g = torch.Generator(device="cuda").manual_seed(N * 100 + T)
    gen = torch.rand(T - 1, Bp, 3, H, H, device="cuda", generator=g)
    goal = torch.rand(*((T - 1,) if per_step else ()), 3, H, H, device="cuda", generator=g)
    w = {"rand": torch.rand(T - 1, device="cuda", generator=g) + 0.1, "ones": torch.ones(T - 1, device="cuda"),
         "last": torch.zeros(T - 1, device="cuda").index_fill_(0, torch.tensor([T - 2], device="cuda"), 1.0),
         "zeros": torch.tensor([0.0 if t % 2 == 0 else 0.5 + t for t in range(T - 1)], device="cuda")}[wkind]
    gen[w == 0] = float("nan")
    guard = 8
    cost = torch.full((N + guard,), 4242.0, device="cuda")
    goal_cost(pk, gen, Bp, N, goal, per_step, w, cost)
    c1 = cost.clone()
    goal_cost(pk, gen, Bp, N, goal, per_step, w, cost)
    torch.cuda.synchronize()
    assert torch.equal(c1, cost)                                           # repeated calls: bit-identical
    assert bool((cost[N:] == 4242.0).all())                                # guard rows untouched
    ref = ref_cost(gen.cpu().numpy(), goal.cpu().numpy(), w.cpu().numpy(), N)
    got = cost[:N].double().cpu().numpy()
    assert np.isfinite(got).all()
    err = np.abs(got - ref) / np.abs(ref).max()
    assert err.max() <= 1e-5, err.max()
    # the same rows at another Bp: bit-identical costs
    Bp2 = Bp + 5
    gen2 = torch.zeros(T - 1, Bp2, 3, H, H, device="cuda")
    gen2[:, :Bp] = gen
    cost2 = torch.zeros(N, device="cuda")
    goal_cost(pk, gen2, Bp2, N, goal, per_step, w, cost2)
    torch.cuda.synchronize()
    assert torch.equal(cost2, cost[:N])


# ----------------------------------------------------------------------------- sample
def sample(pk, T, Bp, ctx, mean, std, seed, it, low=None, high=None, fill=777.0):
    a = torch.full((T - 1, Bp, 5), fill, device="cuda")
    sd = torch.tensor([seed], dtype=torch.int64, device="cuda")
    lo = None if low is None else np.ascontiguousarray(low, dtype=np.float32)
    hi = None if high is None else np.ascontiguousarray(high, dtype=np.float32)
    pk.lib().call("pivp_cem_sample", _p(a), T, Bp, ctx, _p(mean), _p(std), 0 if lo is None else lo.ctypes.data,
                  0 if hi is None else hi.ctypes.data, _p(sd), it, _st())
    torch.cuda.synchronize()
    return a


def test_sample_is_keyed_on_seed_and_iteration(pk):
    T, ctx, Bp = 8, 3, 33
    S = T - ctx
    g = torch.Generator(device="cuda").manual_seed(0)
    mean, std = torch.randn(S, 5, device="cuda", generator=g), torch.rand(S, 5, device="cuda", generator=g) + 0.5
    a = sample(pk, T, Bp, ctx, mean, std, 11, 2)
    assert torch.equal(a, sample(pk, T, Bp, ctx, mean, std, 11, 2))
    assert bool((a[:ctx - 1] == 777.0).all()) and not bool((a[ctx - 1:] == 777.0).any())   # context rows not written, every Bp row is
    for other in (sample(pk, T, Bp, ctx, mean, std, 11, 3), sample(pk, T, Bp, ctx, mean, std, 12, 2)):
        assert not bool((other[ctx - 1:] == a[ctx - 1:]).any())
    wide = sample(pk, T, Bp + 17, ctx, mean, std, 11, 2)                  # the value of (n, s, d) does not depend on Bp
    assert torch.equal(wide[:, :Bp], a)


def test_sample_statistics_at_8192(pk):
    T, ctx, N = 5, 2, 8192
    S = T - ctx
    g = torch.Generator(device="cuda").manual_seed(1)
    mean, std = torch.randn(S, 5, device="cuda", generator=g), torch.rand(S, 5, device="cuda", generator=g) * 2 + 0.1
    a = sample(pk, T, N, ctx, mean, std, 5, 0)[ctx - 1:].double()
    m, sd = mean.double(), std.double()
    z = (a.mean(1) - m) / (sd / N ** 0.5)
    rel = a.std(1, unbiased=False) / sd - 1
    print("\nsample mean |z| max %.2f, std rel err max %.4f" % (float(z.abs().max()), float(rel.abs().max())))
    assert float(z.abs().max()) < 5 and float(rel.abs().max()) < 0.05


def test_sample_clipping_and_zero_std(pk):
    T, ctx, Bp = 7, 2, 64
    S = T - ctx
    g = torch.Generator(device="cuda").manual_seed(2)
    mean, std = torch.randn(S, 5, device="cuda", generator=g), torch.rand(S, 5, device="cuda", generator=g) + 0.5
    lo, hi = np.array([-0.5, -1, -np.inf, 0.0, 0.2], np.float32), np.array([0.5, 0.3, 0.1, np.inf, 0.2], np.float32)
    free = sample(pk, T, Bp, ctx, mean, std, 3, 1)
    clipped = sample(pk, T, Bp, ctx, mean, std, 3, 1, lo, hi)
    want = torch.maximum(torch.minimum(free[ctx - 1:], torch.from_numpy(hi).cuda()), torch.from_numpy(lo).cuda())
    assert torch.equal(clipped[ctx - 1:], want)
    assert bool((clipped[ctx - 1:, :, 4] == 0.2).all())
    only_low = sample(pk, T, Bp, ctx, mean, std, 3, 1, lo, None)
    assert torch.equal(only_low[ctx - 1:], torch.maximum(free[ctx - 1:], torch.from_numpy(lo).cuda()))
    zero = sample(pk, T, Bp, ctx, mean, torch.zeros_like(std), 3, 1, lo, hi)
    want0 = torch.maximum(torch.minimum(mean, torch.from_numpy(hi).cuda()), torch.from_numpy(lo).cuda())
    assert torch.equal(zero[ctx - 1:], want0[:, None].expand(S, Bp, 5))
    assert torch.equal(sample(pk, T, Bp, ctx, mean, torch.zeros_like(std), 9, 4)[ctx - 1:], mean[:, None].expand(S, Bp, 5))


# ----------------------------------------------------------------------------- refit
def ref_refit(cost, a, ctx, N, K, alpha, min_std, mean, std, best_cost, best):
    c = cost[:N].astype(np.float64)
    nan = np.isnan(c)
    order = np.lexsort((np.arange(N), np.where(nan, 0.0, c), nan))        # (NaN last, cost, index): stable on ties
    el = order[:K]
    A = a[ctx - 1:, el, :].astype(np.float64)
    em, es = A.mean(1), A.std(1)
    nm = alpha * mean + (1 - alpha) * em
    ns = np.maximum(alpha * std + (1 - alpha) * es, min_std)
    c0 = c[order[0]]
    hist = (c0, c[el].mean())
    if c0 < best_cost:
        best_cost, best = c0, a[:, order[0], :].astype(np.float64)
    return nm, ns, best_cost, best, hist


def refit(pk, cost, a, ctx, N, K, alpha, min_std, mean, std, best_cost, best, history, it):
    T, Bp = a.shape[0] + 1, a.shape[1]
    pk.lib().call("pivp_cem_refit", _p(cost), _p(a), T, Bp, ctx, N, K, float(alpha), float(min_std), _p(mean), _p(std), _p(best_cost),
                  _p(best), _p(history), it, _st())
    torch.cuda.synchronize()


def _close(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    same_nan = np.isnan(got) == np.isnan(ref)
    ok = np.where(np.isnan(ref), True, np.where(np.isinf(ref), got == ref, np.abs(got - ref) <= 1e-5 * (1 + np.abs(np.nan_to_num(ref)))))
    return bool(same_nan.all() and ok.all())


@pytest.mark.parametrize("N,K,alpha,min_std,ties", [
    (100, 10, 0.0, 0.0, True),              # ties, NaN, +inf, -inf
    (37, 1, 0.5, 0.0, True),                # K = 1
    (64, 64, 0.0, 0.0, False),              # K = N
    (64, 64, 0.5, 0.0, True),               # K = N with NaN / inf among the elites
    (50, 5, 0.5, 0.3, False),               # min_std floor active
    (8192, 819, 0.5, 0.0, True)])           # N = pivp_cem_max_samples()
def test_refit_matches_float64(pk, N, K, alpha, min_std, ties):
    if N == 8192:
        N = pk.lib().query("pivp_cem_max_samples")
    T, ctx = 7, 2
    S, Bp = T - ctx, N + 3
    rs = np.random.RandomState(N + K)
    cost = (rs.randint(0, 6, N) / 4.0 if ties else rs.rand(N) * 10 + 1).astype(np.float32)
    if ties:
        cost[rs.choice(N, 3, replace=False)] = np.nan
        cost[rs.choice(N, 2, replace=False)] = np.inf
        cost[rs.choice(N, 1)] = -np.inf if N > 40 else 0.25
    a = (rs.rand(T - 1, Bp, 5) * (0.2 if min_std else 2.0) - (0.1 if min_std else 1.0)).astype(np.float32)
    a[:, N:] = 1e30                                                        # padding rows: never read
    mean0, std0 = rs.randn(S, 5).astype(np.float32), (rs.rand(S, 5) + 0.1).astype(np.float32)
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    c_d, a_d, m_d, s_d = dev(cost), dev(a), dev(mean0), dev(std0)
    bc = torch.full((), float("inf"), device="cuda")
    best = torch.zeros(T - 1, 5, device="cuda")
    hist = torch.full((3, 2), -7.0, device="cuda")
    refit(pk, c_d, a_d, ctx, N, K, alpha, min_std, m_d, s_d, bc, best, hist, 1)
    nm, ns, rbc, rbest, rh = ref_refit(cost, a, ctx, N, K, alpha, min_std, mean0.astype(np.float64), std0.astype(np.float64), np.inf, None)
    assert _close(m_d.cpu().numpy(), nm) and _close(s_d.cpu().numpy(), ns)
    if min_std:
        assert bool((s_d == float(np.float32(min_std))).any())                   # the floor is active somewhere
    h = hist.cpu().numpy()
    assert _close(h[1], rh) and (h[[0, 2]] == -7.0).all()
    assert float(bc) == rbc and np.array_equal(best.cpu().numpy(), rbest.astype(np.float32))   # replaced (from +inf)
    # kept: an equal (tie) or lower record stays, with its row
    for keep in (float(rbc), float(rbc) - 1.0):
        if not np.isfinite(keep):
            continue
        bc.fill_(keep)
        best.fill_(3.0)
        refit(pk, c_d, a_d, ctx, N, K, alpha, min_std, m_d.clone(), s_d.clone(), bc, best, hist, 2)
        assert float(bc) == keep and bool((best == 3.0).all())
        assert _close(hist[2].cpu().numpy(), rh)
    # repeated: bit-identical
    outs = []
    for _ in range(2):
        m2, s2, bc2, b2, h2 = dev(mean0), dev(std0), torch.full((), float("inf"), device="cuda"), torch.zeros(T - 1, 5, device="cuda"), \
            torch.zeros(1, 2, device="cuda")
        refit(pk, c_d, a_d, ctx, N, K, alpha, min_std, m2, s2, bc2, b2, h2, 0)
        outs.append(torch.cat([m2.flatten(), s2.flatten(), bc2.flatten(), b2.flatten(), h2.flatten()]))
    assert torch.equal(outs[0].nan_to_num(7.0), outs[1].nan_to_num(7.0))


# ----------------------------------------------------------------------------- the CEM loop on a known optimum
def test_cem_core_finds_a_known_optimum(pk):
    S, N, K, iters, ctx = 4, 512, 51, 15, 2
    T = S + ctx
    rs = np.random.RandomState(0)
    a_star = torch.from_numpy(rs.uniform(-0.5, 0.5, (S, 5)).astype(np.float32)).cuda()
    a = torch.zeros(T - 1, N, 5, device="cuda")
    mean, std = torch.zeros(S, 5, device="cuda"), torch.ones(S, 5, device="cuda")
    cost = torch.zeros(N, device="cuda")
    bc, best, hist = torch.full((), float("inf"), device="cuda"), torch.zeros(T - 1, 5, device="cuda"), torch.zeros(iters, 2, device="cuda")
    seed = torch.tensor([2024], dtype=torch.int64, device="cuda")
    lo, hi = np.full(5, -1.0, np.float32), np.full(5, 1.0, np.float32)
    L = pk.lib()
    for i in range(iters):
        L.call("pivp_cem_sample", _p(a), T, N, ctx, _p(mean), _p(std), lo.ctypes.data, hi.ctypes.data, _p(seed), i, _st())
        cost.copy_(((a[ctx - 1:] - a_star[:, None]) ** 2).sum((0, 2)))
        L.call("pivp_cem_refit", _p(cost), _p(a), T, N, ctx, N, K, 0.0, 0.0, _p(mean), _p(std), _p(bc), _p(best), _p(hist), i, _st())
    torch.cuda.synchronize()
    err = float((mean - a_star).abs().max())
    h = hist.cpu().numpy()
    print("\nCEM core: max |mean - a*| = %.2e after %d iterations; lowest cost per iteration %s" % (err, iters, np.array2string(h[:, 0], precision=4)))
    assert err < 2e-2
    assert float(bc) == h[:, 0].min()


# ----------------------------------------------------------------------------- the planner end to end
def _inputs(cfg, T, seed=1234):
    img, act, sta = data(cfg, 1, T, seed=seed)
    return img[:2], sta[0], img[T - 1, 0], act[:1, 0]                     # context (2, 1, 3, H, W), first_state (1, 5), goal, past


def _run(pl, *args, **kw):
    best = pl(*args, **kw).clone()
    torch.cuda.synchronize()
    return dict(best=best, best_cost=pl.best_cost.clone(), history=pl.history.clone(), mean=pl.mean.clone(), std=pl.std.clone(),
                actions=pl.last_actions.clone(), costs=pl.last_costs.clone())


def _equal(r1, r2):
    return all(torch.equal(r1[k], r2[k]) for k in r1)


def _frames_cost(pk, m, T, N, ctx_img, actions, state, goal):
    p = pk.Predictor(m, N, T)
    p(ctx_img, actions, state)
    gen = p.e.ws["gen_all"]
    w = torch.zeros(T - 1, device="cuda")
    w[-1] = 1.0
    cost = torch.zeros(N, device="cuda")
    goal_cost(pk, gen, p.Bp, N, torch.from_numpy(goal).cuda(), False, w, cost)
    torch.cuda.synchronize()
    return cost


@pytest.mark.parametrize("mt,compute,H", [("CDNA", "f32", 64), ("CDNA", "bf16", 64), ("DNA", "f32", 64), ("DNA", "bf16", 64),
                                          ("STP", "f32", 64), ("STP", "bf16", 64), ("STP", "bf16", 128)])
def test_planner_end_to_end(pk, mt, compute, H):
    T, N, K, I = 6, 64, 6, 3
    m, cfg, _ = make(pk, mt, compute, H)
    c, s, goal, past = _inputs(cfg, T)
    lo, hi = [-1.0] * 5, [1.0] * 5
    pl = pk.CEMPlanner(m, N, T, K, I, action_low=lo, action_high=hi, init_std=0.5)
    r = _run(pl, c, s, goal, past_actions=past, seed=3)
    assert r["best"].shape == (T - 1, 5) and r["actions"].shape == (T - 1, N, 5) and r["costs"].shape == (N,)
    assert torch.equal(r["best"][0], torch.from_numpy(past[0]).cuda()) and bool((r["actions"][0] == r["best"][0]).all())
    # the last iteration's costs: pivp_goal_cost on a fresh Predictor's frames of the same candidates, bit for bit
    assert torch.equal(r["costs"], _frames_cost(pk, m, T, N, c, r["actions"], s, goal))
    # the best sequence reproduces its cost; best_cost is the lowest of the per-iteration minima
    again = _frames_cost(pk, m, T, N, c, r["best"][:, None].expand(T - 1, N, 5).contiguous(), s, goal)
    h = r["history"].cpu().numpy()
    print("\n%s %s %dx%d: history %s" % (mt, compute, H, H, np.array2string(h, precision=5)))
    assert float(again[0]) == float(r["best_cost"]) == h[:, 0].min()
    assert bool(torch.isfinite(r["mean"]).all()) and bool((r["std"] >= 0).all())
    # graph = eager; same seed = same plan; another seed = another plan
    assert _equal(r, _run(pk.CEMPlanner(m, N, T, K, I, action_low=lo, action_high=hi, init_std=0.5, graph=False), c, s, goal,
                          past_actions=past, seed=3))
    assert _equal(r, _run(pl, c, s, goal, past_actions=past, seed=3))
    other = _run(pl, c, s, goal, past_actions=past, seed=4)
    assert not torch.equal(other["actions"], r["actions"]) and not torch.equal(other["best"], r["best"])


def test_planner_follows_parameter_updates(pk):
    T, N, K, I = 6, 64, 6, 2
    m, cfg, params = make(pk, "CDNA", "bf16")
    c, s, goal, past = _inputs(cfg, T)
    pl = pk.CEMPlanner(m, N, T, K, I)
    old = _run(pl, c, s, goal, seed=1)
    opt = pk.Adam().setup(m)
    torch.manual_seed(0)
    m.engine.flat_g.normal_()
    opt.apply()
    new = _run(pl, c, s, goal, seed=1)
    assert not torch.equal(new["costs"], old["costs"])
    assert _equal(new, _run(pk.CEMPlanner(m, N, T, K, I, graph=False), c, s, goal, seed=1))
    m.load_params({k: (v * 0.9).astype(np.float32) for k, v in params.items()})
    new2 = _run(pl, c, s, goal, seed=1)
    assert not torch.equal(new2["costs"], new["costs"])
    assert _equal(new2, _run(pk.CEMPlanner(m, N, T, K, I, graph=False), c, s, goal, seed=1))


def _ws_pointers(ws):
    out = []
    for k in sorted(ws, key=str):
        v = ws[k]
        for x in (v if isinstance(v, list) else list(v.values()) if isinstance(v, dict) else [v]):
            for y in (x if isinstance(x, list) else [x]):
                if isinstance(y, torch.Tensor):
                    out.append((k, y.data_ptr()))
    return out


def test_planner_leaves_the_training_engine_untouched(pk):
    m, cfg, _ = make(pk, "CDNA", "bf16")
    img, act, sta = data(cfg, 4, 6)
    r = pk.Rollout(m, 4, 6, graph=True)
    r.load(img, act, sta)
    before = torch.stack(list(r())).clone()
    e = m.engine
    ws, tc, ptrs = e.ws, e.tc, _ws_pointers(e.ws)
    c, s, goal, past = _inputs(cfg, 8, seed=5)
    pk.CEMPlanner(m, 16, 8, 4, 2)(c, s, goal)
    after = torch.stack(list(r())).clone()
    torch.cuda.synchronize()
    assert torch.equal(before, after)
    assert e.ws is ws and e.tc is tc and _ws_pointers(e.ws) == ptrs


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


def test_planner_memory_is_the_predictors_plus_its_buffers(pk):
    T, N, K, I = 6, 64, 6, 3
    m, cfg, _ = make(pk, "CDNA", "bf16")
    c, s, goal, past = _inputs(cfg, T)
    cd, sd = torch.from_numpy(c).cuda(), torch.from_numpy(s).cuda()
    a = torch.zeros(T - 1, N, 5, device="cuda")
    peak_p = _peak(lambda: (lambda p: (p, p(cd, a, sd)))(pk.Predictor(m, N, T)))
    holder = []
    peak_c = _peak(lambda: (lambda pl: (pl, pl(cd, sd, torch.from_numpy(goal).cuda()), holder.append(pl)))(pk.CEMPlanner(m, N, T, K, I)))
    pl = holder.pop()
    own = sum(t.numel() * t.element_size() for t in (pl.mean, pl.std, pl.goal, pl.weights, pl.cost, pl.best, pl.best_cost, pl.history,
                                                     pl.seed))
    del pl
    print("\npeak allocated, bf16 CDNA 64x64 N=%d T=%d: Predictor %.2f MiB, CEMPlanner %.2f MiB (own buffers %.3f MiB)"
          % (N, T, peak_p / 2**20, peak_c / 2**20, own / 2**20))
    assert peak_c <= peak_p + own + 2**20, (peak_c, peak_p, own)


def test_planned_cost_beats_the_zero_sequence(pk):
    """Goal = the last frame the model itself predicts under a known a*: the plan must get closer to it than the all-zero sequence."""
    T, N, K, I = 6, 128, 13, 5
    m, cfg, _ = make(pk, "CDNA", "bf16")
    c, s, _, past = _inputs(cfg, T)
    ctx = m.num_frame_before_prediction
    a_star = np.zeros((T - 1, 5), np.float32)
    a_star[:ctx - 1] = past
    a_star[ctx - 1:] = np.random.RandomState(8).uniform(-0.5, 0.5, (T - ctx, 5))
    p = pk.Predictor(m, 1, T)
    goal = p(c, a_star[:, None], s)[-1, 0].clone().cpu().numpy()
    pl = pk.CEMPlanner(m, N, T, K, I, action_low=[-1.0] * 5, action_high=[1.0] * 5, init_std=0.5)
    pl(c, s, goal, past_actions=past, seed=0)
    torch.cuda.synchronize()
    zero = np.zeros((T - 1, 1, 5), np.float32)
    zero[:ctx - 1, 0] = past
    z = _frames_cost(pk, m, T, 1, c, torch.from_numpy(zero).cuda(), s, goal)
    best = float(pl.best_cost)
    print("\nplanned best_cost %.4g, all-zero sequence %.4g: ratio %.3f" % (best, float(z[0]), best / float(z[0])))
    assert best < float(z[0])
