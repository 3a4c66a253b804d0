"""Time of one cross-entropy-method plan (pivp_b200.CEMPlanner) against the forward pass it is built on, and the cost of its own kernels.

CDNA 64x64, bf16, T = 16 (two context frames, 14 planned steps), N candidates, K = N / 10 elites, I = 5 iterations, default weights (the
last predicted frame only).  For each N, one JSON line with:
  * plan ms per call (input copies + one graph replay, CUDA events around `steps` calls after warm-up) and per iteration;
  * the same N, T Predictor call (input copies + graph replay);
  * pivp_cem_sample, pivp_goal_cost and pivp_cem_refit on the planner's own buffers, each timed alone (CUDA events around single launches,
    L2 overwritten with a 256 MiB write before each so the cost kernel reads its frames from HBM), and their share of one plan iteration;
  * the cost kernel's bytes (gen rows of the weighted steps, the goal image once, weights, costs) over its time, against the
    7.7 TB/s HBM3e data-sheet figure of one B200.
The card and its power limit come from a read-only nvidia-smi query.

    python scripts/bench_plan.py [--n 256 1024] [--steps 10] [--warmup 2] [--reps 50]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_GBS = 7700.0


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except Exception as ex:                                  # the numbers stand without it, but say why it is missing
        return "unknown (%s)" % ex


def timed(fn, steps):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def kernel_us(launch, reps, flush):
    """Median of `reps` single launches, each after an L2-overwriting write, timed with CUDA events around the launch alone."""
    ts = []
    for _ in range(reps):
        flush.zero_()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        launch()
        t1.record()
        torch.cuda.synchronize()
        ts.append(t0.elapsed_time(t1) * 1e3)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, nargs="+", default=[256, 1024])
    ap.add_argument("--T", type=int, default=16)
    ap.add_argument("--iterations", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=50)
    a = ap.parse_args()
    import pivp_b200 as pk
    from oracle import model as OM
    T, H, I = a.T, 64, a.iterations
    print(json.dumps({"card": card(), "model": "CDNA", "compute": "bf16", "H": H, "W": H, "T": T, "context_frames": 2, "iterations": I}),
          flush=True)
    cfg = OM.Config("CDNA", 10, height=H, width=H)
    params = OM.init_params(cfg)
    rs = np.random.RandomState(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    L = pk.lib()
    for N in a.n:
        K = max(1, N // 10)
        ctx = torch.from_numpy(rs.rand(2, 1, 3, H, H).astype(np.float32)).cuda()
        st = torch.from_numpy(rs.randn(1, 5).astype(np.float32) * 0.1).cuda()
        goal = torch.from_numpy(rs.rand(3, H, H).astype(np.float32)).cuda()
        m = pk.Model(10, is_cdna=True, height=H, width=H, compute="bf16")
        m.load_params(params)
        m.train = False
        # the Predictor alone at the same N, T
        p = pk.Predictor(m, N, T)
        act = torch.from_numpy(rs.randn(T - 1, N, 5).astype(np.float32) * 0.1).cuda()
        for _ in range(a.warmup):
            p(ctx, act, st)
        ms_pred = timed(lambda: p(ctx, act, st), a.steps)
        del p
        pl = pk.CEMPlanner(m, N, T, K, I, action_low=[-1.0] * 5, action_high=[1.0] * 5, init_std=0.5)
        for _ in range(a.warmup):
            pl(ctx, st, goal)
        ms_plan = timed(lambda: pl(ctx, st, goal), a.steps)
        finite = bool(torch.isfinite(pl.best_cost).item())
        # the planner's own kernels, alone, on its buffers (as the last plan left them)
        e, pp = pl.e, pl.predictor
        s = lambda: torch.cuda.current_stream().cuda_stream
        lo, hi = pl.low.ctypes.data, pl.high.ctypes.data
        us_sample = kernel_us(lambda: L.call("pivp_cem_sample", pp.actions.data_ptr(), T, pl.Bp, pl.ctx, pl.mean.data_ptr(), pl.std.data_ptr(),
                                             lo, hi, pl.seed.data_ptr(), 0, s()), a.reps, flush)
        us_cost = kernel_us(lambda: L.call("pivp_goal_cost", e.ws["gen_all"].data_ptr(), T, pl.Bp, N, H, H, pl.goal.data_ptr(), 1,
                                           pl.weights.data_ptr(), pl.cost.data_ptr(), s()), a.reps, flush)
        mean, std, bc, best, hist = pl.mean.clone(), pl.std.clone(), pl.best_cost.clone(), pl.best.clone(), torch.zeros(1, 2, device="cuda")
        us_refit = kernel_us(lambda: L.call("pivp_cem_refit", pl.cost.data_ptr(), pp.actions.data_ptr(), T, pl.Bp, pl.ctx, N, K, 0.0, 0.0,
                                            mean.data_ptr(), std.data_ptr(), bc.data_ptr(), best.data_ptr(), hist.data_ptr(), 0, s()),
                             a.reps, flush)
        nw = int((pl.weights != 0).sum())
        cost_bytes = (N + 1) * nw * 3 * H * H * 4 + (T - 1) * 4 + N * 4    # gen rows + the goal once (re-reads hit L2) + weights + costs
        gbs = cost_bytes / (us_cost * 1e-6) / 1e9
        own_ms = (us_sample + us_cost + us_refit) * 1e-3
        rec = {"N": N, "K": K, "plan_ms_per_call": round(ms_plan, 3), "plan_ms_per_iteration": round(ms_plan / I, 3),
               "predictor_ms_per_call": round(ms_pred, 3), "iteration_minus_predictor_ms": round(ms_plan / I - ms_pred, 3),
               "sample_us": round(us_sample, 2), "goal_cost_us": round(us_cost, 2), "refit_us": round(us_refit, 2),
               "own_kernels_share_of_iteration": round(own_ms / (ms_plan / I), 5),
               "goal_cost_bytes": cost_bytes, "goal_cost_GBps": round(gbs, 1), "goal_cost_share_of_hbm_7700GBps": round(gbs / HBM_GBS, 3),
               "best_cost_finite": finite}
        print(json.dumps(rec), flush=True)
        del pl, m
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
