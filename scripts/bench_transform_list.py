"""Un-fused CDNA list (the links' reference call form) micro-benchmark: CUDA-event time per launch inside a CUDA graph, cold L2 (rotating
input sets > 126 MB) and warm L2, forward and backward, with the fused backward on the same inputs for comparison.

usage: python scripts/bench_transform_list.py [B ...]    -> the GPU line, then one JSON line per batch size (default 32 256)

Backward: every list entry live (M + 1 gradient planes), g_enc7 given, d_prev on.  Bytes are the algorithmic ones (each input read once,
each output written once); the HBM fraction is against MEASURED_PEAKS.json when present, else 6650 GB/s (the HBM rate bench_cdna.py
assumes).  FMA: backward 2 * 25 * M * 3 * HW per sample (dK and d_prev), forward 25 * M * 3 * HW.
"""
import json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import pivp_b200 as pk
from pivp_b200 import functions as Fn

H = W = 64
HW = H * W
M = 10
_pk = os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json")
peak = json.load(open(_pk))["hbm_gbs"] if os.path.exists(_pk) else 6650.0
L = pk.lib()


def cur():
    return torch.cuda.current_stream().cuda_stream


def gpu_line():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE,
                           stderr=subprocess.PIPE, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as ex:                    # the name still comes from the runtime
        q = "nvidia-smi unavailable (%s)" % ex
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q, "hbm_peak_gbs_used": peak}


def run(B, nsets, iters=20):
    fwd_bytes = B * ((3 + 3 + 3 * (M + 1)) * HW * 4 + 1000)
    bwd_bytes = B * ((3 * (M + 1) + 3 + 3 + 3 + 3 + 3) * HW * 4 + 2000)
    fused_bytes = B * ((3 + 3 + 3 + 11 + 3 + 11 + 3) * HW * 4 + 2000)     # fused backward with d_prev (DESIGN.md section 2)
    bwd_fma, fwd_fma = B * 2 * 25 * M * 3 * HW, B * 25 * M * 3 * HW
    sets = []
    for _ in range(nsets):
        prev = torch.rand(B, 3, H, W, device="cuda"); e = torch.randn(B, 3, H, W, device="cuda"); k = torch.randn(B, 25 * M, device="cuda")
        a = 2 * torch.randn(B, M + 1, H, W, device="cuda")
        g = torch.randn(M + 1, B, 3, H, W, device="cuda"); ge = torch.randn(B, 3, H, W, device="cuda")
        out = torch.empty(M + 1, B, 3, H, W, device="cuda")
        de, dk, dp, da = torch.empty_like(e), torch.empty_like(k), torch.empty_like(prev), torch.empty_like(a)
        gl = Fn._glist(tuple(g[i] for i in range(M + 1)))
        sets.append((prev, e, k, a, g, ge, out, de, dk, dp, da, gl))
    nb = L.query("pivp_cdna_transform_bwd_workspace_bytes", B, H, W, M)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    nbf = L.query("pivp_cdna_fused_bwd_workspace_bytes", B, H, W, M)
    wsf = torch.empty(nbf, dtype=torch.uint8, device="cuda")

    def fwd(s):
        prev, e, k, a, g, ge, out, de, dk, dp, da, gl = s
        L.call("pivp_cdna_transform", prev.data_ptr(), e.data_ptr(), k.data_ptr(), out.data_ptr(), B, H, W, M, cur())

    def bwd(s):
        prev, e, k, a, g, ge, out, de, dk, dp, da, gl = s
        L.call("pivp_cdna_transform_bwd", gl, ge.data_ptr(), prev.data_ptr(), e.data_ptr(), k.data_ptr(), de.data_ptr(), dk.data_ptr(),
               dp.data_ptr(), 0, B, H, W, M, ws.data_ptr(), nb, cur())

    def fused_bwd(s):
        prev, e, k, a, g, ge, out, de, dk, dp, da, gl = s
        L.call("pivp_cdna_fused_bwd", g[0].data_ptr(), prev.data_ptr(), e.data_ptr(), a.data_ptr(), k.data_ptr(), de.data_ptr(), da.data_ptr(),
               dk.data_ptr(), dp.data_ptr(), 0, B, H, W, M, wsf.data_ptr(), nbf, cur())

    res = {}
    for name, fn, nbytes, fma in (("list_fwd", fwd, fwd_bytes, fwd_fma), ("list_bwd", bwd, bwd_bytes, bwd_fma),
                                  ("fused_bwd_dprev", fused_bwd, fused_bytes, None)):
        for i in range(3 * nsets):
            fn(sets[i % nsets])
        torch.cuda.synchronize()
        # graph of `iters` launches walking the sets: launch gaps excluded, cold L2 when nsets * bytes >> 126 MB
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for i in range(iters):
                fn(sets[i % nsets])
        gr.replay(); torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = 1e9
        for _ in range(5):
            ev0.record(); gr.replay(); ev1.record(); torch.cuda.synchronize()
            best = min(best, ev0.elapsed_time(ev1) * 1e3 / iters)
        r = dict(us=round(best, 2), GBs=round(nbytes / best / 1e3, 1), hbm_frac=round(nbytes / best / 1e3 / peak, 3), MB=round(nbytes / 1e6, 2))
        if fma:
            r["TFMA_s"] = round(fma / best / 1e6, 2)
        res[name] = r
    return res


if __name__ == "__main__":
    print(json.dumps(gpu_line()))
    for B in [int(v) for v in sys.argv[1:]] or [32, 256]:
        per = B * (3 * (M + 1) + 15 + 11) * HW * 4
        cold = max(1, int(600e6 // per) + 1)
        print(json.dumps({"B": B, "H": H, "W": W, "M": M, "cold_sets": cold, "cold": run(B, cold), "warm": run(B, 1)}))
