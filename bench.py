#!/usr/bin/env python
"""Benchmark of the hot path: CDNA 64x64 training step (forward + BPTT + gradient all-reduce + Adam).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path, one rank per GPU (torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (NumPy restatement), rank 0 only
    python bench.py ... --dump-outputs DIR                   # also write what the last timed step computed to DIR/<name>.npy

Prints ONE JSON line (rank 0).  Metric: train frames/sec = global_batch * T / step_time (BASELINE.json).
 value        : inputs resident in HBM, whole step replayed as a CUDA graph, CUDA-event time, max over ranks
 e2e          : same step through the public API (TrainStep.load_batch from pinned host memory + step + loss D2H read)
 roofline     : dominant kernel = the tcgen05 ConvLSTM implicit GEMM; algorithmic FLOPs / CUDA-event duration, measured
                live on the launching stream during one instrumented step
 cpu_baseline : the oracle (NumPy restatement of the reference's Chainer CPU path) timed on this box's host cores
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "train frames/sec (CDNA, 64x64, b32)"
T_SEQ, H, W, MASKS, K_SCHED, ITER0 = 10, 64, 64, 10, 900.0, 6000
DUMP_MAX_ELEMS = 1 << 22              # per dumped array: the three large ones stay under 64 MB together


def dump_outputs(out_dir, model):
    """Write what the last training step handed its caller to out_dir/<name>.npy (float32, float64 for the scalars): loss, psnr_all, the
    predicted frames and states, and the updated parameters and the gradients in Chainer layout, every tensor flattened and concatenated
    in sorted name order.  An array of more than DUMP_MAX_ELEMS elements is reduced to its elements at a fixed, seeded choice of flat
    indices, so that two builds run with the same arguments can be compared element for element.  The comparison needs a tolerance: the
    step adds fp32 partial sums with atomics, and Adam amplifies those last-bit differences over the steps."""
    import numpy as np
    import torch

    def flat(d):
        return np.concatenate([d[k].reshape(-1) for k in sorted(d)])
    arrays = {"loss": np.float64(float(model.loss)), "psnr_all": np.float64(float(model.psnr_all)),
              "gen_images": torch.stack(list(model.gen_images)).float().cpu().numpy(),
              "gen_states": torch.stack(list(model.gen_states)).float().cpu().numpy(),
              "params": flat(model.params()), "grads": flat(model.grads)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if a.size > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.RandomState(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines, self.t0 = gpu_index, None, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "25"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.monotonic(), line.strip()))

    def mark(self):
        """Start of the timed region: the process is started earlier (before the warm-up), because nvidia-smi needs a few hundred ms
        to print its first line and a short timed region would otherwise end without a sample."""
        self.t0 = time.monotonic()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t1 = time.monotonic()
        time.sleep(0.05)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0 = self.t0 if self.t0 is not None else 0.0
        window = [ln for ts, ln in self.lines if t0 <= ts <= t1 + 0.03]           # a line printed just after the region was sampled inside it
        for ln in window:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def lstm_flops(B):
    """Algorithmic FLOPs of one launch of the ConvLSTM GEMM per layer (2*M*N*K, K = 25*(Cin+C), un-padded)."""
    from importlib import import_module
    lay = import_module("physical-interaction-video-prediction_b200.layout")
    lv = (2, 2, 4, 4, 8, 4, 2)
    out = []
    for cin, c, l in zip(lay.LSTM_IN, lay.LSTM_SIZES, lv):
        M = B * (H // l) * (W // l)
        out.append(2.0 * M * 4 * c * 25 * (cin + c))
    return out


def run_reference(args, rank):
    """The reference's own CPU algorithm for this path.  Chainer 2.0.1 / Python 2 cannot run in this image, so this is the
    NumPy restatement (oracle/), all host threads the BLAS will use, on a bounded sample: ONE sequence of the b32 workload."""
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    # torchrun exports OMP_NUM_THREADS=1 to its workers, which would silently single-thread the BLAS under the CPU arm: the reference
    # arm is ONE process and gets every host core, whatever launched it (must be set before NumPy loads its BLAS)
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = str(cores)
    import numpy as np
    from oracle import model as OM
    blas_threads = None
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(cores)
        blas_threads = max([p_.get("num_threads", 0) for p_ in threadpool_info()] or [0]) or None
    except Exception:
        pass
    cfg = OM.Config("CDNA", MASKS, schedsamp_k=K_SCHED, height=H, width=W)
    params = OM.init_params(cfg)
    adam = OM.Adam()
    batch = OM.concat_examples(OM.synthetic_sequences(1, T_SEQ, cfg))
    np.random.seed(99)
    steps, warm = args.steps, max(1, min(args.warmup, 1))
    for i in range(warm):
        OM.train_step(params, adam, batch, ITER0 + i, cfg)
    t0 = time.perf_counter()
    for i in range(steps):
        OM.train_step(params, adam, batch, ITER0 + warm + i, cfg)
    dt = (time.perf_counter() - t0) / steps
    val = 1 * T_SEQ / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "CDNA 64x64 T=10 10 masks train step (fwd+bwd+Adam), CPU NumPy restatement of the Chainer path",
                       "sample": "1 sequence of the b32 batch per step"},
            "cpu_baseline": {"value": val, "unit": "frames/s", "cores": cores, "blas_threads": blas_threads, "kind": "port",
                             "sample": "CDNA b1 T=10 fwd+bwd+Adam, %d steps after %d warm-up" % (steps, warm)},
            "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def cpu_baseline():
    import numpy as np
    from oracle import model as OM
    cfg = OM.Config("CDNA", MASKS, schedsamp_k=K_SCHED, height=H, width=W)
    params = OM.init_params(cfg)
    batch = OM.concat_examples(OM.synthetic_sequences(1, T_SEQ, cfg))
    np.random.seed(99)
    OM.loss_and_grads(params, batch, ITER0, cfg)
    best = 1e9
    for i in range(3):
        t0 = time.perf_counter()
        OM.loss_and_grads(params, batch, ITER0, cfg)
        best = min(best, time.perf_counter() - t0)
    blas_threads = None
    try:
        from threadpoolctl import threadpool_info
        blas_threads = max([p_.get("num_threads", 0) for p_ in threadpool_info()] or [0]) or None
    except Exception:
        pass
    return {"value": T_SEQ / best, "unit": "frames/s", "cores": len(os.sched_getaffinity(0)), "blas_threads": blas_threads, "kind": "port",
            "sample": "oracle (NumPy restatement of the Chainer CPU path; Chainer 2.0.1 not installable): CDNA b1 T=10 fwd+bwd, best of 3 after 1 warm-up"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="per-GPU batch (weak scaling)")
    ap.add_argument("--compute", default="bf16", choices=["bf16", "f32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--global-batch", type=int, default=0, help="strong scaling: fixed GLOBAL batch split over the ranks (BASELINE config 3: 256)")
    ap.add_argument("--no-extras", action="store_true", help="skip the DNA-op (config 4) and STP 128x128 (config 5) measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import numpy as np
    import torch
    import __graft_entry__
    __graft_entry__.build()
    import pivp_b200 as pk
    from pivp_b200 import parallel
    rank, local, world = parallel.init_distributed()
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    W_ = max(3, args.warmup)
    B, T = args.batch, T_SEQ
    if args.global_batch:
        assert args.global_batch % world == 0, "--global-batch must be divisible by the number of ranks"
        B = args.global_batch // world

    model = pk.Model(MASKS, is_cdna=True, scheduled_sampling_k=K_SCHED, prefix="train", height=H, width=W, device=str(dev),
                     compute=args.compute, rank=rank, world_size=world)
    opt = pk.Adam(alpha=0.001).setup(model)
    seqs = pk.data.synthetic_sequences(B, T, H, W, seed=1234 + rank)
    host = [torch.from_numpy(a).pin_memory() for a in pk.concat_examples(seqs)]
    step = pk.TrainStep(model, opt, B, T, graph=not args.no_graph)
    step.load_batch(*host)
    np.random.seed(99)                      # every rank draws the same global permutations (SURVEY 8e)
    it = ITER0

    def barrier():
        if world > 1:
            torch.distributed.barrier()

    sampler = ClockSampler(local)
    sampler.start()                         # running before the warm-up; only lines inside the timed region are used (mark())
    for _ in range(W_):
        step(it); it += 1
    torch.cuda.synchronize()
    # ---------------- timed region: inputs resident, device time, max over ranks
    barrier(); torch.cuda.synchronize()
    sampler.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = pk.lib().query("pivp_launch_count")
    ev0.record()
    for _ in range(args.steps):
        step(it); it += 1
    ev1.record()
    torch.cuda.synchronize(); barrier()
    clocks = sampler.stop()
    ms = ev0.elapsed_time(ev1)
    launches = (step.launches_per_step or 0) * args.steps if step.use_graph else pk.lib().query("pivp_launch_count") - n0
    tmax = torch.tensor([ms], device=dev)
    if world > 1:
        torch.distributed.all_reduce(tmax, op=torch.distributed.ReduceOp.MAX)
    ms = float(tmax.item())
    ms_per_step = ms / args.steps
    value = B * world * T / (ms_per_step * 1e-3)
    loss_now = float(model.loss)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model)

    # ---------------- end to end: H2D of the batch from pinned memory + step + D2H loss read, every step
    barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    # the public data path: BatchPrefetcher copies batch k+1 from pinned host memory while step k computes (every batch is still
    # copied host -> device inside this timed region), TrainStep runs the step, float(loss) is the device -> host read
    e2e_path = "BatchPrefetcher"
    try:
        pf = pk.BatchPrefetcher(step, (host for _ in range(args.steps)))
        pending = None
        while pf.load_next():
            handle = step(it); it += 1
            if pending is not None:
                loss = float(pending)         # device -> host read of step k's loss, issued while step k+1 runs (every step's loss is read)
            pending = handle
        loss = float(pending)
    except RuntimeError as exc:               # keep the line valid if the side-stream path is unavailable: synchronous copy, and say so
        sys.stderr.write("bench: BatchPrefetcher failed (%s); timing the synchronous copy path\n" % exc)
        e2e_path = "load_batch (synchronous H2D)"
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step.load_batch(*host)
            loss = float(step(it)); it += 1
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    tmax = torch.tensor([e2e_s], device=dev)
    if world > 1:
        torch.distributed.all_reduce(tmax, op=torch.distributed.ReduceOp.MAX)
    e2e_val = B * world * T / (float(tmax.item()) / args.steps)
    h2d = sum(a.numel() * 4 for a in host) + (T - 1) * B * 4
    d2h = 2 * (T - 1) * 4

    # ---------------- roofline: the dominant kernel = the tcgen05 ConvLSTM implicit GEMM (forward with the fused gate epilogue and
    # input gradient; 126 launches per step).  One eager step records every launch with its real arguments; the recorded launches
    # are then replayed back to back as ONE CUDA graph on the same buffers and timed with CUDA events on the launching stream --
    # an eager event pair around a 20 us kernel mostly measures the host's launch cadence, not the kernel.
    roof, roof_wgrad, cdna_op = None, None, None

    def traffic_from_profile():
        """DRAM bytes (read + write) per launch of the dominant kernel from the committed `ncu --set full` capture of one step
        (profiles/r02_ncu_full_halo_traffic.json, else the round-1 file; written by scripts/ncu_traffic_summary.py); None when absent."""
        for nm in ("r02_ncu_full_halo_traffic.json", "r01_ncu_full_halo_traffic.json"):
            try:
                with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", nm)) as fh:
                    return json.load(fh)["dram_bytes_per_launch"]
            except (OSError, KeyError, ValueError):
                continue
        return None
    if True:                                  # every rank runs the instrumented step (it contains the all-reduce); rank 0 reports
        L = pk.lib()
        orig = L.call
        recs = []

        def recording_call(name, *a):
            if name in ("pivp_tc_conv5x5", "pivp_tc_conv5x5_ln", "pivp_tc_wgrad5x5"):
                recs.append((name, a))
            orig(name, *a)
        L.call = recording_call
        eager = pk.TrainStep(model, opt, B, T, graph=False)
        eager.images, eager.actions, eager.states = step.images, step.actions, step.states
        eager(it); it += 1
        torch.cuda.synchronize()
        L.call = orig
        pk_, src = peaks()
        fl = lstm_flops(B)
        tcp = model.engine.tc

        def replay_time(calls, reps=5):
            """Average device time per launch (s) of `calls` replayed back to back as one CUDA graph; best of `reps` replays."""
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                cur = torch.cuda.current_stream().cuda_stream
                for name, a in calls:
                    orig(name, *(a[:-1] + (cur,)))
            g.replay(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            best = 1e9
            for _ in range(reps):
                e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1) * 1e-3)
            return best / len(calls)

        if tcp is not None:
            by_ptr = {}
            for li, f in enumerate(fl):
                by_ptr[tcp.Wf[li].data_ptr()] = f          # forward launch of layer li
                by_ptr[tcp.Wd[li].data_ptr()] = f          # input-gradient launch: same 2*M*N*K
            conv_calls = [(n, a) for n, a in recs if n in ("pivp_tc_conv5x5", "pivp_tc_conv5x5_ln")]      # weights pointer = argument 6 of both
            if conv_calls:
                per = replay_time(conv_calls)
                flops = sum(by_ptr[a[6]] for _, a in conv_calls) / len(conv_calls)
                ach = flops / per / 1e12
                roof = {"bound": "tensor",
                        "kernel": "conv5x5_halo_tc_kernel (tcgen05 ConvLSTM implicit GEMM with halo-patch A operand; forward + fused gates, "
                                  "and input gradient; the 8x8 maps of layer 5 in the two-image pair geometry)",
                        "achieved": ach, "peak": pk_["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk_["bf16_tflops"],
                        "frac_of_sustained": ach / pk_["bf16_tflops_sustained"], "traffic": traffic_from_profile(), "traffic_unit": "bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum)",
                        "peak_source": src + " (burst figure: the step's %d launches are replayed back to back as one CUDA graph, "
                                             "about 3 ms, outside the long step)" % len(conv_calls),
                        "launches": len(conv_calls), "avg_launch_us": per * 1e6,
                        "flops_per_launch": flops, "how": "algorithmic 2*M*N*K (un-padded channels) / CUDA-event time of the graph replay"}
            wg_calls = [(n, a) for n, a in recs if n == "pivp_tc_wgrad5x5"]
            if wg_calls:
                per = replay_time(wg_calls)
                flops = sum(fl) * (T - 1) / len(wg_calls)
                ach = flops / per / 1e12
                roof_wgrad = {"bound": "tensor", "kernel": "wgrad5x5_halo_kernel + splitk_reduce (weight gradient over all T-1 steps, one launch "
                              "per layer)", "achieved": ach, "peak": pk_["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk_["bf16_tflops"],
                              "launches": len(wg_calls), "avg_launch_us": per * 1e6}
        # ---- fused CDNA transform + mask softmax + composite: graph of 20 launches walking input sets that exceed L2 ("cold")
        if model.engine.model_type == "CDNA":
            def cdna_time(Bc, nsets, iters=20):
                HWc = H * W
                sets = []
                for _ in range(nsets):
                    t = dict(prev=torch.rand(Bc, 3, H, W, device=dev), e=torch.randn(Bc, 3, H, W, device=dev),
                             a=2 * torch.randn(Bc, MASKS + 1, H, W, device=dev), k=torch.randn(Bc, 25 * MASKS, device=dev),
                             g=torch.randn(Bc, 3, H, W, device=dev))
                    t.update(out=torch.empty_like(t["prev"]), de=torch.empty_like(t["e"]), da=torch.empty_like(t["a"]), dk=torch.empty_like(t["k"]))
                    sets.append(t)
                nb = L.query("pivp_cdna_fused_bwd_workspace_bytes", Bc, H, W, MASKS)
                wsb = torch.empty(nb, dtype=torch.uint8, device=dev)

                def fwd(t, st):
                    orig("pivp_cdna_fused_fwd", t["prev"].data_ptr(), t["e"].data_ptr(), t["a"].data_ptr(), t["k"].data_ptr(), t["out"].data_ptr(),
                         Bc, H, W, MASKS, st)

                def bwd(t, st):
                    orig("pivp_cdna_fused_bwd", t["g"].data_ptr(), t["prev"].data_ptr(), t["e"].data_ptr(), t["a"].data_ptr(), t["k"].data_ptr(),
                         t["de"].data_ptr(), t["da"].data_ptr(), t["dk"].data_ptr(), 0, 0, Bc, H, W, MASKS, wsb.data_ptr(), nb, st)
                res = {}
                for nm, fn in (("fwd", fwd), ("bwd", bwd)):
                    for i in range(nsets):
                        fn(sets[i], torch.cuda.current_stream().cuda_stream)
                    torch.cuda.synchronize()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        for i in range(iters):
                            fn(sets[i % nsets], torch.cuda.current_stream().cuda_stream)
                    g.replay(); torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    best = 1e9
                    for _ in range(5):
                        e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
                        best = min(best, e0.elapsed_time(e1) * 1e-3 / iters)
                    res[nm] = best
                return res
            cdna_op = {"bound": "hbm", "unit": "GB/s", "peak": pk_["hbm_gbs"], "peak_source": src,
                       "bytes_per_sample": {"fwd": 328680, "bwd": 559056},
                       "note": "algorithmic bytes (SURVEY 8d): fwd reads prev, enc7_pre, mask_pre, kern_raw and writes gen; bwd reads g, prev, "
                               "enc7_pre, mask_pre, kern_raw and writes d_enc7_pre, d_mask_pre, d_kern_raw (no d_prev: the previous frame is "
                               "detached in scheduled-sampling training).  Cold = a CUDA graph of 20 launches walking input sets that "
                               "together exceed the 126 MB L2."}
            for Bc in sorted({B, 256}):
                per = Bc * 37 * H * W * 4
                tm = cdna_time(Bc, max(2, int(600e6 // per) + 1))
                cdna_op["b%d" % Bc] = {d: {"avg_launch_us": tm[d] * 1e6, "achieved": cdna_op["bytes_per_sample"][d] * Bc / tm[d] / 1e9,
                                           "frac": cdna_op["bytes_per_sample"][d] * Bc / tm[d] / 1e9 / pk_["hbm_gbs"]} for d in ("fwd", "bwd")}
            tw = cdna_time(B, 1)              # warm: one input set, resident in L2 after the first launch (what the op sees inside the step)
            cdna_op["b%d_warm_l2" % B] = {d: {"avg_launch_us": tw[d] * 1e6, "achieved": cdna_op["bytes_per_sample"][d] * B / tw[d] / 1e9}
                                          for d in ("fwd", "bwd")}

    # ---------------- BASELINE config 4: DNA fused transform + composite (num_masks = 1), b32, forward / backward GB/s on cold inputs
    dna_op, stp_step = None, None
    if rank == 0 and world == 1 and not args.no_extras:
        L = pk.lib()
        pk_, src = peaks()

        def op_time(fn, nsets, iters=20):
            for i in range(nsets):
                fn(i, torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for i in range(iters):
                    fn(i % nsets, torch.cuda.current_stream().cuda_stream)
            g.replay(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            best = 1e9
            for _ in range(5):
                e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1) * 1e-3 / iters)
            return best
        HWc = H * W
        dna_bytes = {"fwd": (25 + 3 + 2 + 3) * HWc * 4, "bwd": (3 + 3 + 25 + 2 + 25 + 2) * HWc * 4}
        dna_op = {"bound": "hbm", "unit": "GB/s", "peak": pk_["hbm_gbs"], "peak_source": src, "bytes_per_sample": dna_bytes,
                  "note": "BASELINE config 4. Algorithmic bytes (SURVEY 8d): fwd reads enc7_pre (25 planes), prev (3), mask_pre (2) and writes gen (3) = "
                          "540,672 B/sample; bwd reads g, prev, enc7_pre, mask_pre and writes d_enc7_pre, d_mask_pre (the taps are detached, "
                          "train_model.py:404, and prev is detached under scheduled sampling: no d_prev).  Cold = 20 launches walking input sets "
                          "that together exceed the 126 MB L2."}
        for Bc in sorted({args.batch, 256}):
            nsets = max(2, int(600e6 // (Bc * 60 * HWc * 4)) + 1)
            sets = [dict(prev=torch.rand(Bc, 3, H, W, device=dev), e=torch.randn(Bc, 25, H, W, device=dev), a=2 * torch.randn(Bc, 2, H, W, device=dev),
                         g=torch.randn(Bc, 3, H, W, device=dev)) for _ in range(nsets)]
            for t_ in sets:
                t_.update(out=torch.empty_like(t_["prev"]), de=torch.empty_like(t_["e"]), da=torch.empty_like(t_["a"]))
            nb = L.query("pivp_dna_fused_bwd_workspace_bytes", Bc, H, W)
            wsb = torch.empty(max(nb, 16), dtype=torch.uint8, device=dev)

            def fwd(i, st, sets=sets, Bc=Bc):
                t_ = sets[i]
                L.call("pivp_dna_fused_fwd", t_["prev"].data_ptr(), t_["e"].data_ptr(), t_["a"].data_ptr(), t_["out"].data_ptr(), Bc, H, W, st)

            def bwd(i, st, sets=sets, Bc=Bc, wsb=wsb, nb=nb):
                t_ = sets[i]
                L.call("pivp_dna_fused_bwd", t_["g"].data_ptr(), t_["prev"].data_ptr(), t_["e"].data_ptr(), t_["a"].data_ptr(), t_["de"].data_ptr(),
                       t_["da"].data_ptr(), 0, 0, Bc, H, W, wsb.data_ptr(), nb, st)
            tm = {"fwd": op_time(fwd, nsets), "bwd": op_time(bwd, nsets)}
            dna_op["b%d" % Bc] = {d: {"avg_launch_us": tm[d] * 1e6, "achieved": dna_bytes[d] * Bc / tm[d] / 1e9,
                                      "frac": dna_bytes[d] * Bc / tm[d] / 1e9 / pk_["hbm_gbs"]} for d in ("fwd", "bwd")}
            del sets
        # ------------ BASELINE config 5: STP, 10 transformers, 128x128, 20-frame sequences, scheduled sampling: whole training step
        try:
            Hs, Ts, Bs = 128, 20, 16
            m5 = pk.Model(MASKS, is_cdna=False, is_stp=True, scheduled_sampling_k=K_SCHED, prefix="stp", height=Hs, width=Hs, device=str(dev),
                          compute=args.compute)
            o5 = pk.Adam(alpha=0.001).setup(m5)
            s5 = pk.TrainStep(m5, o5, Bs, Ts, graph=not args.no_graph)
            s5.load_batch(*[torch.from_numpy(a) for a in pk.concat_examples(pk.data.synthetic_sequences(Bs, Ts, Hs, Hs, seed=77))])
            np.random.seed(7)
            for i in range(3):
                s5(ITER0 + i)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n5 = 5
            e0.record()
            for i in range(n5):
                s5(ITER0 + 3 + i)
            e1.record(); torch.cuda.synchronize()
            ms5 = e0.elapsed_time(e1) / n5
            stp_step = {"workload": "STP, 10 transformers, 128x128 RGB, T=20 (19 recurrent steps, 18 loss terms), batch %d, scheduled sampling k=900 at iter %d; "
                                    "forward + BPTT + Adam as one CUDA graph" % (Bs, ITER0), "value": Bs * Ts / (ms5 * 1e-3), "unit": "frames/s",
                        "ms_per_step": ms5, "steps": n5, "warmup": 3, "loss": float(m5.loss), "gpu_launches_per_step": s5.launches_per_step,
                        "stp_out_of_range_rule": "zeros (SURVEY A.7; the other rule is implemented and tested)"}
            del m5, o5, s5
        except Exception as exc:              # keep the headline line valid whatever happens in the extra configuration
            stp_step = {"error": "%s: %s" % (type(exc).__name__, exc)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": W_,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if args.global_batch else "weak", "vs_baseline": None,
                "dtype": "bf16" if args.compute == "bf16" else "f32", "data": "synthetic",
                "config": {"workload": "CDNA 64x64 RGB, batch %d per GPU, T=10, 10 masks, scheduled sampling k=900 at iter %d; "
                                       "one step = forward + BPTT + grad all-reduce + Adam" % (B, ITER0),
                           "global_batch": B * world, "seq_len": T, "parallelism": "dp%d" % world,
                           "l2": "per-step working set ~%.1f GB of activations >> 126 MB L2 (no flush needed)" % (2.2 * B / 32),
                           "cuda_graph": bool(step.use_graph), "lstm_gemm": "tcgen05 bf16: ConvLSTM fwd (+fused gates) / dgrad / wgrad with halo-patch operands, stride-2 convolutions / deconvolutions fwd+bwd+wgrad; enc0 (3 channels) and enc3 (1x1) SIMT fp32" if args.compute == "bf16" else "SIMT fp32"},
                "clocks": clocks, "gpu_launches": int(launches), "loss": loss_now,
                "e2e": {"value": e2e_val, "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "path": e2e_path}}
        if roof:
            line["roofline"] = roof
        if roof_wgrad:
            line["roofline_wgrad"] = roof_wgrad
        if cdna_op:
            line["cdna_op"] = cdna_op
        if dna_op:
            line["dna_op"] = dna_op
        if stp_step:
            line["stp_step"] = stp_step
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line))
    if world > 1:
        # CUDA graphs that hold NCCL kernels (PIVP_DP_OVERLAP=1) must be gone before the communicator is torn down
        step.graph = None
        del step
        import gc
        gc.collect()
        torch.cuda.synchronize()
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
