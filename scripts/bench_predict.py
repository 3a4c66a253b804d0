"""Throughput and memory of forward-only batched prediction (pivp_b200.Predictor) against the training engine's Rollout.

CDNA 64x64, bf16, T = 16 (two context frames, 15 predicted frames per candidate), N candidate action sequences in one call
(batch_size = N).  Reports predicted frames / s = N * (T - 1) / time of one call (CUDA events around the calls after warm-up: graph
replay plus the input copies) and the peak of torch.cuda.max_memory_allocated for building and calling each predictor.  The card and its
power limit are read with a read-only nvidia-smi query.  One JSON line per measurement.

    python scripts/bench_predict.py [--n 32 256 1024] [--steps 20] [--warmup 3]
"""
import argparse
import gc
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except Exception as ex:                                  # the numbers stand without it, but say why it is missing
        return "unknown (%s)" % ex


def fresh():
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    return torch.cuda.memory_allocated()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, nargs="+", default=[32, 256, 1024])
    ap.add_argument("--T", type=int, default=16)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    import pivp_b200 as pk
    from oracle import model as OM
    T, H = a.T, 64
    print(json.dumps({"card": card(), "model": "CDNA", "compute": "bf16", "H": H, "W": H, "T": T, "context_frames": 2}), flush=True)
    cfg = OM.Config("CDNA", 10, height=H, width=H)
    params = OM.init_params(cfg)
    rs = np.random.RandomState(0)
    for N in a.n:
        ctx = torch.from_numpy(rs.rand(2, N, 3, H, H).astype(np.float32)).cuda()
        act = torch.from_numpy(rs.randn(T - 1, N, 5).astype(np.float32) * 0.1).cuda()
        st = torch.from_numpy(rs.randn(N, 5).astype(np.float32) * 0.1).cuda()
        m = pk.Model(10, is_cdna=True, height=H, width=H, compute="bf16")
        m.load_params(params)
        m.train = False
        base = fresh()
        p = pk.Predictor(m, N, T)
        for _ in range(a.warmup):
            out = p(ctx, act, st)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(a.steps):
            out = p(ctx, act, st)
        t1.record()
        torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / a.steps
        finite = bool(torch.isfinite(out).all())
        del p, out
        rec = {"what": "Predictor", "N": N, "ms_per_call": round(ms, 3), "frames_per_s": round(N * (T - 1) / (ms * 1e-3), 1),
               "peak_allocated_MiB": round(peak / 2**20, 1), "finite": finite}
        print(json.dumps(rec), flush=True)
        # the training engine's rollout at the same shape: full training workspace (every activation of every step + backward buffers)
        base = fresh()
        try:
            r = pk.Rollout(m, N, T)
            imgs = torch.zeros(T, N, 3, H, H, device="cuda")
            imgs[:2].copy_(ctx)
            r.load(imgs, torch.cat([act, act[-1:]]), st[None].expand(T, N, 5))
            r()
            torch.cuda.synchronize()
            rec = {"what": "Rollout", "N": N, "peak_allocated_MiB": round((torch.cuda.max_memory_allocated() - base) / 2**20, 1)}
            del r, imgs
        except torch.cuda.OutOfMemoryError as ex:
            rec = {"what": "Rollout", "N": N, "fits": False, "error": str(ex).splitlines()[0][:160]}
        print(json.dumps(rec), flush=True)
        del m
        fresh()


if __name__ == "__main__":
    main()
