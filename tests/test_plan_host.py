"""CPU tests of the CEM planning contract: every bad argument of the three planning entry points is PIVP_EINVAL before any launch (fake
device pointers, as in test_predict_host.py), and CEMPlanner rejects bad configurations and inputs with ValueError before it touches the
device."""
import os
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EINVAL = -1
FAKE = 1 << 20                                   # 16-byte aligned, never dereferenced: every call below fails validation first


@pytest.fixture(scope="module")
def pk():
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.build()
    import pivp_b200
    return pivp_b200


def _f32(*v):
    return np.array(v, dtype=np.float32)


def test_max_samples_covers_8192(pk):
    assert pk.lib().query("pivp_cem_max_samples") >= 8192


def test_sample_einval(pk):
    L = pk.lib()
    n0 = L.query("pivp_launch_count")
    lo, hi = _f32(-1, -1, -1, -1, -1), _f32(1, 1, 1, 1, 1)
    inv = _f32(-1, -1, 2, -1, -1)                                   # low[2] > high[2]
    nan = _f32(-1, -1, np.nan, -1, -1)

    def call(actions=FAKE, T=6, Bp=4, ctx=2, mean=FAKE, std=FAKE, low=lo.ctypes.data, high=hi.ctypes.data, seed=FAKE, it=0):
        return L.query("pivp_cem_sample", actions, T, Bp, ctx, mean, std, low, high, seed, it, 0)
    bad = [dict(actions=0), dict(mean=0), dict(std=0), dict(seed=0),
           dict(Bp=0), dict(ctx=0), dict(T=2), dict(T=1), dict(it=-1),
           dict(low=hi.ctypes.data, high=lo.ctypes.data), dict(low=inv.ctypes.data), dict(high=nan.ctypes.data)]
    for kw in bad:
        assert call(**kw) == EINVAL, kw
    assert "low[2]" in (call(low=inv.ctypes.data), L.cdll.pivp_last_error().decode())[1]
    assert L.query("pivp_launch_count") == n0


def test_goal_cost_einval(pk):
    L = pk.lib()
    n0 = L.query("pivp_launch_count")

    def call(gen=FAKE, T=6, Bp=4, N=3, H=64, W=64, goal=FAKE, per_step=0, w=FAKE, cost=FAKE):
        return L.query("pivp_goal_cost", gen, T, Bp, N, H, W, goal, per_step, w, cost, 0)
    bad = [dict(gen=0), dict(goal=0), dict(w=0), dict(cost=0),
           dict(N=0), dict(N=5), dict(T=1), dict(H=0), dict(W=-64), dict(H=1, W=1),     # 3*H*W not a multiple of 4
           dict(gen=FAKE + 4), dict(goal=FAKE + 8)]                                      # float4 loads need 16-byte alignment
    for kw in bad:
        assert call(**kw) == EINVAL, kw
    assert L.query("pivp_launch_count") == n0


def test_refit_einval(pk):
    L = pk.lib()
    n0 = L.query("pivp_launch_count")
    nmax = L.query("pivp_cem_max_samples")

    def call(cost=FAKE, a=FAKE, T=6, Bp=4, ctx=2, N=3, K=2, alpha=0.0, min_std=0.0, mean=FAKE, std=FAKE, bc=FAKE, ba=FAKE, hist=FAKE, it=0):
        return L.query("pivp_cem_refit", cost, a, T, Bp, ctx, N, K, alpha, min_std, mean, std, bc, ba, hist, it, 0)
    bad = [dict(cost=0), dict(a=0), dict(mean=0), dict(std=0), dict(bc=0), dict(ba=0), dict(hist=0),
           dict(N=0), dict(N=5), dict(K=0), dict(K=4), dict(N=nmax + 1, Bp=nmax + 2, K=1),
           dict(ctx=0), dict(T=2), dict(it=-1),
           dict(alpha=1.0), dict(alpha=-0.1), dict(alpha=float("nan")), dict(min_std=-1e-3), dict(min_std=float("nan"))]
    for kw in bad:
        assert call(**kw) == EINVAL, kw
    assert L.query("pivp_launch_count") == n0


# ----------------------------------------------------------------------------- CEMPlanner validation
def _model(use_state=True, ctx=2, H=64, W=64):
    return types.SimpleNamespace(engine=types.SimpleNamespace(use_state=use_state, ctx=ctx, H=H, W=W))


def test_planner_rejects_bad_configurations(pk):
    P = pk.CEMPlanner
    nmax = pk.lib().query("pivp_cem_max_samples")
    bad = [dict(model=_model(use_state=False)),                        # actions never read
           dict(num_elites=65), dict(num_elites=0), dict(num_samples=0),
           dict(num_samples=nmax + 1, num_elites=1),
           dict(seq_len=2), dict(model=_model(ctx=6)),                 # T - ctx < 1
           dict(iterations=0), dict(alpha=1.0), dict(alpha=-0.5), dict(min_std=-1.0), dict(init_std=-1.0),
           dict(action_low=[0.0] * 4), dict(action_low=[1.0] * 5, action_high=[0.0] * 5), dict(action_high=[np.nan] * 5)]
    for kw in bad:
        args = dict(model=_model(), num_samples=64, seq_len=6, num_elites=6, iterations=3)
        args.update(kw)
        with pytest.raises(ValueError):
            P(**args)                                # raises before Predictor (and with it the device) is reached


def _stub(pk, T=6, ctx=2):
    """A CEMPlanner with the attributes its input check reads and no device state (this machine may have no GPU)."""
    P = pk.CEMPlanner
    p = P.__new__(P)
    p.T, p.ctx, p.S, p.e = T, ctx, T - ctx, types.SimpleNamespace(H=64, W=64)
    return p


def test_planner_rejects_malformed_inputs(pk):
    p = _stub(pk)
    rs = np.random.RandomState(0)
    img = rs.rand(3, 1, 3, 64, 64).astype(np.float32)
    sta = rs.rand(1, 5).astype(np.float32)
    goal = rs.rand(3, 64, 64).astype(np.float32)
    c, s, g, pa, w, m0, s0 = p._check(img, sta, goal, None, None, None, None)
    assert tuple(c.shape) == (2, 1, 3, 64, 64) and pa is None and w is None
    ok = dict(past_actions=rs.rand(1, 5).astype(np.float32), weights=np.ones(5, np.float32),
              init_mean=np.zeros((4, 5), np.float32), init_std=np.ones((4, 5), np.float32))
    p._check(img, sta, rs.rand(5, 3, 64, 64).astype(np.float32), *ok.values())            # per-step goal, every optional input
    base = (img, sta, goal, None, None, None, None)
    bad = [(img[:1],), (img[:, :1, :, :32],), (np.repeat(img, 2, axis=1),),               # context frames, size, batch
           (img.astype(np.float64),),
           (img, sta[0]), (img, np.repeat(sta, 2, axis=0)),                                # first_state (1, 5)
           (img, sta, goal[:2]), (img, sta, rs.rand(4, 3, 64, 64).astype(np.float32)),     # goal channels / steps
           (img, sta, goal, np.zeros((2, 5), np.float32)),                                 # past actions: ctx - 1 rows
           (img, sta, goal, None, np.ones(4, np.float32)),                                 # weights (T-1,)
           (img, sta, goal, None, _f32(1, 1, -1, 1, 1)),                                   # negative weight
           (img, sta, goal, None, _f32(1, 1, np.nan, 1, 1)),
           (img, sta, goal, None, None, np.zeros((5, 5), np.float32)),                     # init_mean (S, 5)
           (img, sta, goal, None, None, None, -np.ones((4, 5), np.float32)),               # negative init_std
           (img, sta, goal, None, None, None, np.ones((4, 5), np.float64))]
    for args in bad:
        with pytest.raises(ValueError):
            p._check(*(args + base[len(args):]))
