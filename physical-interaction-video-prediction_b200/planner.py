"""Cross-entropy-method (CEM) planning over ``Predictor`` with a goal-image cost, sampled, scored and refit on the device.

``CEMPlanner`` searches the S = T - context_frames future actions of one context for the sequence whose predicted frames come closest to a
goal image.  Each iteration draws N candidates from a per-(step, component) Gaussian, predicts their frames, scores them, and refits the
Gaussian to the K best:

* ``pivp_cem_sample`` writes the candidates straight into the predictor's action buffer (rows of the context steps hold the given past
  actions and are never sampled);
* the predictor's forward pass (``ForwardEngine.predict_device``, its ring workspace) predicts the T-1 frames of every candidate;
* ``pivp_goal_cost`` scores them: cost[n] = sum_t w[t] * mean (gen[t, n] - goal[t])^2;
* ``pivp_cem_refit`` ranks the costs in one CTA, refits mean / std to the elites and keeps the best sequence seen so far.

One call is the input copies plus one CUDA-graph replay: the bf16 weight refresh (so a plan follows ``Adam.apply`` / ``load_params``),
then ``iterations`` x (sample -> forward -> cost -> refit).  Nothing synchronises with the host until the caller reads a result.
"""
import numpy as np
import torch

from ._lib import lib
from .predictor import Predictor


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _arr(x, what):
    """float32 tensor (CPU or CUDA) from a tensor or array-like; ValueError for another dtype."""
    if not isinstance(x, torch.Tensor):
        x = np.asarray(x)
        if x.dtype != np.float32:
            raise ValueError("%s: float32 required, got %s" % (what, x.dtype))
        x = torch.from_numpy(x)
    elif x.dtype != torch.float32:
        raise ValueError("%s: float32 required, got %s" % (what, x.dtype))
    return x


def _host_values(x):
    """The values of a CPU tensor, None for a CUDA one (not inspected: that would synchronise with the device)."""
    return None if x.is_cuda else x.numpy()


class CEMPlanner(object):
    """``planner(context_images, first_state, goal, ...)`` -> the best action sequence found, (T-1, 5) CUDA float32, past actions included.

    model: a ``Model`` built with ``use_state=True`` (otherwise its actions are never read).  num_samples N (<= pivp_cem_max_samples()),
    num_elites K <= N, seq_len T with T - context_frames >= 1 planned steps, iterations >= 1.  action_low / action_high: 5 floats each or
    None (no bound).  init_std: the default initial standard deviation; min_std: its floor after every refit; alpha: the weight of the old
    mean / std in the refit, in [0, 1).  graph=False runs the same launches eagerly.

    After a call, the device tensors ``best_cost`` (0-d), ``mean`` / ``std`` (S, 5, the refit distribution), ``history`` (iterations, 2:
    lowest and mean elite cost of each iteration), ``last_actions`` (T-1, N, 5) and ``last_costs`` (N,) of the last iteration hold the
    plan's state; the next call overwrites them (clone to keep)."""

    def __init__(self, model, num_samples, seq_len, num_elites, iterations, action_low=None, action_high=None, init_std=1.0, min_std=0.0,
                 alpha=0.0, graph=True):
        e = model.engine
        N, T, K, I = int(num_samples), int(seq_len), int(num_elites), int(iterations)
        if not e.use_state:
            raise ValueError("CEMPlanner: the model was built with use_state=False, so its actions are never read")
        nmax = lib().query("pivp_cem_max_samples")
        if not 1 <= N <= nmax:
            raise ValueError("num_samples must be in [1, %d] (got %d)" % (nmax, N))
        if not 1 <= K <= N:
            raise ValueError("num_elites must be in [1, num_samples = %d] (got %d)" % (N, K))
        if T - e.ctx < 1:
            raise ValueError("seq_len - context_frames must be >= 1 planned step (got seq_len %d, context_frames %d)" % (T, e.ctx))
        if I < 1:
            raise ValueError("iterations must be >= 1 (got %d)" % I)
        if not 0.0 <= float(alpha) < 1.0:
            raise ValueError("alpha must be in [0, 1) (got %r)" % alpha)
        if not float(min_std) >= 0.0:
            raise ValueError("min_std must be >= 0 (got %r)" % min_std)
        if not float(init_std) >= 0.0:
            raise ValueError("init_std must be >= 0 (got %r)" % init_std)
        bounds = []
        for v, what in ((action_low, "action_low"), (action_high, "action_high")):
            if v is not None:
                v = np.asarray(v, dtype=np.float64)
                if v.shape != (5,) or np.isnan(v).any():
                    raise ValueError("%s: 5 numbers expected, got shape %s" % (what, v.shape))
                v = np.ascontiguousarray(v, dtype=np.float32)
            bounds.append(v)
        lo, hi = bounds
        if lo is not None and hi is not None and (lo > hi).any():
            raise ValueError("action_low > action_high in a component: %s > %s" % (lo, hi))
        self.N, self.T, self.K, self.I, self.ctx, self.S = N, T, K, I, e.ctx, T - e.ctx
        self.low, self.high = lo, hi                     # host arrays: pivp_cem_sample reads them at the call (baked into the graph)
        self.init_std, self.min_std, self.alpha = float(init_std), float(min_std), float(alpha)

        self.predictor = p = Predictor(model, N, T, graph=False)      # its engine and static buffers; the graph below is the planner's
        self.e, self.Bp = p.e, p.Bp
        dev, H, W = self.e.dev, self.e.H, self.e.W
        f32 = dict(dtype=torch.float32, device=dev)
        self.mean = torch.zeros(self.S, 5, **f32)
        self.std = torch.zeros(self.S, 5, **f32)
        self.goal = torch.zeros(T - 1, 3, H, W, **f32)
        self.weights = torch.zeros(T - 1, **f32)
        self.cost = torch.zeros(N, **f32)
        self.best = torch.zeros(T - 1, 5, **f32)
        self.best_cost = torch.full((), float("inf"), **f32)
        self.history = torch.zeros(I, 2, **f32)
        self.seed = torch.zeros(1, dtype=torch.int64, device=dev)
        self.use_graph, self.graph = bool(graph), None

    @property
    def last_actions(self):
        return self.predictor.actions[:, :self.N]

    @property
    def last_costs(self):
        return self.cost

    # ---- inputs
    def _check(self, context_images, first_state, goal, past_actions, weights, init_mean, init_std):
        e, T, ctx, S = self.e, self.T, self.ctx, self.S
        c, s, g = _arr(context_images, "context_images"), _arr(first_state, "first_state"), _arr(goal, "goal")
        if c.dim() != 5 or c.shape[0] < ctx or c.shape[1] != 1 or tuple(c.shape[2:]) != (3, e.H, e.W):
            raise ValueError("context_images: (C >= %d, 1, 3, %d, %d) expected, got %s" % (ctx, e.H, e.W, tuple(c.shape)))
        if tuple(s.shape) != (1, 5):
            raise ValueError("first_state: (1, 5) expected, got %s" % (tuple(s.shape),))
        if tuple(g.shape) not in ((3, e.H, e.W), (T - 1, 3, e.H, e.W)):
            raise ValueError("goal: (3, %d, %d) or (%d, 3, %d, %d) expected, got %s" % (e.H, e.W, T - 1, e.H, e.W, tuple(g.shape)))
        pa = None
        if past_actions is not None:
            pa = _arr(past_actions, "past_actions")
            if tuple(pa.shape) != (ctx - 1, 5):
                raise ValueError("past_actions: (context_frames - 1, 5) = (%d, 5) expected, got %s" % (ctx - 1, tuple(pa.shape)))
        w = None
        if weights is not None:
            w = _arr(weights, "weights")
            if tuple(w.shape) != (T - 1,):
                raise ValueError("weights: (T-1,) = (%d,) expected, got %s" % (T - 1, tuple(w.shape)))
            v = _host_values(w)
            if v is not None and not (v >= 0).all():
                raise ValueError("weights must be non-negative and not NaN")
        out = []
        for x, what in ((init_mean, "init_mean"), (init_std, "init_std")):
            if x is not None:
                x = _arr(x, what)
                if tuple(x.shape) != (S, 5):
                    raise ValueError("%s: (T - context_frames, 5) = (%d, 5) expected, got %s" % (what, S, tuple(x.shape)))
            out.append(x)
        m0, s0 = out
        if s0 is not None:
            v = _host_values(s0)
            if v is not None and not (v >= 0).all():
                raise ValueError("init_std must be non-negative and not NaN")
        return c[:ctx], s, g, pa, w, m0, s0

    # ---- the plan
    def _plan(self):
        e, p, L = self.e, self.predictor, self.e.L
        T, Bp, ctx, N = self.T, self.Bp, self.ctx, self.N
        st = e._s()
        lo = 0 if self.low is None else self.low.ctypes.data
        hi = 0 if self.high is None else self.high.ctypes.data
        if e.tc is not None:
            e.tc.refresh_weights()                       # once per plan: the parameters do not change between iterations
        for i in range(self.I):
            L.call("pivp_cem_sample", _ptr(p.actions), T, Bp, ctx, _ptr(self.mean), _ptr(self.std), lo, hi, _ptr(self.seed), i, st)
            e.predict_device(p.context, p.actions, p.state0, T, refresh=False)
            L.call("pivp_goal_cost", _ptr(e.ws["gen_all"]), T, Bp, N, e.H, e.W, _ptr(self.goal), 1, _ptr(self.weights), _ptr(self.cost), st)
            L.call("pivp_cem_refit", _ptr(self.cost), _ptr(p.actions), T, Bp, ctx, N, self.K, self.alpha, self.min_std, _ptr(self.mean),
                   _ptr(self.std), _ptr(self.best_cost), _ptr(self.best), _ptr(self.history), i, st)

    def _capture(self):
        dev = self.e.dev
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            self._plan()                                 # lazy initialisation outside the capture (on whatever the buffers hold)
        torch.cuda.current_stream(dev).wait_stream(s)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._plan()

    def __call__(self, context_images, first_state, goal, past_actions=None, weights=None, init_mean=None, init_std=None, seed=0):
        """context_images (C >= context_frames, 1, 3, H, W), first_state (1, 5), goal (3, H, W) or (T-1, 3, H, W); past_actions
        (context_frames - 1, 5), the executed actions of the context steps (default zeros); weights (T-1,) >= 0 per predicted frame
        (default: the last one only); init_mean / init_std (T - context_frames, 5) (default 0 / the constructor's init_std), e.g. a
        shifted previous plan; seed: a non-negative int.  float32 on any device.  Returns the planner's (T-1, 5) best-sequence buffer."""
        c, s, g, pa, w, m0, s0 = self._check(context_images, first_state, goal, past_actions, weights, init_mean, init_std)
        seed = int(seed)
        if not 0 <= seed < 2**63:
            raise ValueError("seed must be in [0, 2**63) (got %d)" % seed)
        if self.use_graph and self.graph is None:
            self._capture()                              # before the copies: the warm-up pass overwrites the plan's state
        p, dev, ctx = self.predictor, self.e.dev, self.ctx
        to = lambda x: x.to(dev, non_blocking=True)
        p.context.copy_(to(c).expand_as(p.context))
        p.state0.copy_(to(s)[None].expand_as(p.state0))
        self.best.zero_()
        if ctx > 1:
            if pa is None:
                p.actions[:ctx - 1].zero_()
            else:
                p.actions[:ctx - 1].copy_(to(pa)[:, None].expand(ctx - 1, self.Bp, 5))
                self.best[:ctx - 1].copy_(p.actions[:ctx - 1, 0])
        self.goal.copy_(to(g).expand_as(self.goal))
        if w is None:
            self.weights.zero_()
            self.weights[-1] = 1.0
        else:
            self.weights.copy_(to(w))
        if m0 is None:
            self.mean.zero_()
        else:
            self.mean.copy_(to(m0))
        if s0 is None:
            self.std.fill_(self.init_std)
        else:
            self.std.copy_(to(s0))
        self.seed.fill_(seed)
        self.best_cost.fill_(float("inf"))
        self.history.zero_()
        if self.use_graph:
            self.graph.replay()
        else:
            self._plan()
        return self.best
