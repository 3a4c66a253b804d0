"""GPU parity at the BASELINE.json metric configuration: CDNA 64x64, B=32, T=10, 10 masks, scheduled sampling at iteration 6000.

These are the shapes bench.py times, so this test runs the kernel instantiations of the benchmark (two-tile halo CTAs
``conv5x5_halo_tc_kernel<2,1>``, the b32 split-K counts of the weight-gradient GEMMs, the 4-split 8x8 input gradient) THROUGH the
benchmarked entry point: ``TrainStep(graph=True)`` -- one captured CUDA graph of forward + BPTT + Adam.

Reference: frozen float64 oracle vectors ``tests/golden/cdna_b32_t10.npz`` (``make_golden_b32.py``; the oracle needs ~16 GB and
~2.5 minutes for this case, so it is not re-run here).  Tolerances (stated per north_star):
  fp32 mode : loss / frames / states 1e-4 relative; gradients: relative L2 of the strided subsample <= 2e-3, norm 1e-3.
  bf16 mode : loss 2e-2; frames relative L2 <= 2e-2 at EVERY time step (incl. t = 8, after 9 recurrent steps) and 5e-2 of max-abs;
              mask logits relative L2 <= 2e-2; gradients per tensor: relative L2 of the subsample <= GRAD_L2_BF16, cosine >= GRAD_COS_BF16
              (the measured table is printed; see DESIGN.md section 4 for what bounds it).
Frames of SAMPLES and mask logits are compared at the stored quarter of the pixel positions (``MG.PIXELS``).
Index work (num_ground_truth, the seven scheduled-sampling selects) is bit-exact in both modes.
"""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import model as OM

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLD)

GRAD_L2_BF16, GRAD_COS_BF16 = 0.12, 0.99        # measured at B=32, T=10: worst tensor lstm1/conv/W 0.089 / 0.9962


@pytest.fixture(scope="module")
def pk():
    import pivp_b200
    pivp_b200.lib()
    return pivp_b200


def l2rel(a, b):
    a = a.detach().float().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    a, b = a.astype(np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))


def maxrel(a, b):
    a = a.detach().float().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    a, b = a.astype(np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


@pytest.mark.parametrize("compute", ["bf16", "f32"])
def test_b32_t10_train_step_matches_frozen_oracle(pk, compute, capsys):
    import make_golden_b32 as MG
    gold = np.load(os.path.join(GOLD, "cdna_b32_t10.npz"))
    B, T, H = MG.B, MG.T, MG.H
    cfg = OM.Config("CDNA", 10, schedsamp_k=MG.K, height=H, width=H)
    params = MG.params_for(cfg)
    batch = OM.concat_examples(OM.synthetic_sequences(B, T, cfg, seed=1234))
    model = pk.Model(10, is_cdna=True, scheduled_sampling_k=MG.K, prefix="b32", height=H, width=H, compute=compute)
    model.load_params(params)
    opt = pk.Adam().setup(model)
    step = pk.TrainStep(model, opt, B, T, graph=True)          # the benchmarked path: one CUDA graph per step
    step.load_batch(*[torch.from_numpy(a) for a in batch], non_blocking=False)
    np.random.seed(99)
    loss = step(MG.ITER)
    torch.cuda.synchronize()
    e = model.engine
    # ---- index work: bit-exact
    assert int(model.num_ground_truth) == int(gold["n_gt"]) == 17
    assert np.array_equal(model.take_gt[2:T - 1].astype(bool), gold["take_gt"])
    # ---- values
    ftol, ltol = (2e-2, 2e-2) if compute == "bf16" else (1e-4, 1e-4)
    assert abs(float(loss) - float(gold["loss"])) <= ltol * float(gold["loss"]), (float(loss), float(gold["loss"]))
    rows = []
    for t in range(T - 1):
        gen = model.gen_images[t]
        sub = MG.at_pixels(gen[list(MG.SAMPLES)].float().cpu().numpy())
        e_l2, e_max = l2rel(sub, gold["gen_sub"][t]), maxrel(sub, gold["gen_sub"][t])
        g64 = gen.double()
        mean_err = float((g64.mean(dim=(1, 2, 3)).cpu().numpy() - gold["gen_mean"][t]).__abs__().max())
        l2_err = float(np.abs(g64.pow(2).sum(dim=(1, 2, 3)).sqrt().cpu().numpy() / gold["gen_l2"][t] - 1).max())
        rows.append((t, e_l2, e_max, mean_err, l2_err))
        assert e_l2 < ftol, ("frames", t, e_l2)
        assert e_max < (5e-2 if compute == "bf16" else 1e-4), ("frames max", t, e_max)
        assert l2_err < ftol and mean_err < ftol, ("frame statistics of all 32 samples", t, mean_err, l2_err)
    for i, t in enumerate(MG.MASK_T):
        got = MG.at_pixels(e.ws["mask_pre"][t][list(MG.MASK_SAMPLES)].float().cpu().numpy())
        assert l2rel(got, gold["mask_pre_sub"][i].astype(np.float64)) < (2e-2 if compute == "bf16" else 2e-3), ("mask logits", t)   # fp16 storage of the reference: 1e-3
    gs = torch.stack(list(model.gen_states)).cpu().numpy()
    assert maxrel(gs, gold["gen_states"]) < (2e-2 if compute == "bf16" else 1e-4)
    # ---- gradients (flat_g is what Adam consumed; the step does not modify it)
    grads = e.chainer_grads()
    table, bad = [], {}
    for key in sorted(grads):
        g = grads[key].astype(np.float64).reshape(-1)
        ref = gold["gsub/" + key].astype(np.float64)
        sub = g[::MG.stride_of(g.size)]
        err = np.linalg.norm(sub - ref) / (np.linalg.norm(ref) + 1e-30)
        cos = float((sub * ref).sum() / (np.linalg.norm(sub) * np.linalg.norm(ref) + 1e-30))
        nrm = np.sqrt((g * g).sum()) / (float(gold["gl2/" + key]) + 1e-30)
        table.append((key, err, cos, nrm))
        if float(gold["gl2/" + key]) == 0.0:
            if np.abs(g).max() != 0.0:
                bad[key] = "expected an exactly zero gradient"
            continue
        if compute == "bf16":
            if err > GRAD_L2_BF16 or cos < GRAD_COS_BF16:
                bad[key] = (err, cos)
        elif err > 2e-3 or abs(nrm - 1) > 1e-3:
            bad[key] = (err, nrm)
    with capsys.disabled():
        print("\n[b32 T=10 %s] loss %.6f (oracle %.6f)" % (compute, float(loss), float(gold["loss"])))
        print("  t : frames relL2 / max-rel (3 samples) | all 32 samples: |mean err|, |L2 ratio - 1|")
        for r in rows:
            print("  %d : %.2e / %.2e | %.2e, %.2e" % r)
        print("  gradient, per tensor (strided subsample): relative L2, cosine, norm ratio")
        for key, err, cos, nrm in table:
            print("  %-28s %.3e  %.5f  %.4f" % (key, err, cos, nrm))
    assert not bad, bad


def test_steps_in_flight_keep_their_own_select_and_loss(pk):
    """Steps launched back to back WITHOUT a host synchronisation in between (what bench.py's timed loop does) must see the same
    scheduled-sampling selects and report the same per-step losses as the run that synchronises after every step: the select travels
    through a ring of pinned slots guarded by events, and every loss handle is bound to a snapshot of its own step."""
    H, B, T, N = 64, 2, 4, 7                      # N > Engine.RING: slots are reused
    cfg = OM.Config("CDNA", 10, schedsamp_k=900.0, height=H, width=H)
    params = OM.init_params(cfg)
    batch = [torch.from_numpy(a) for a in OM.concat_examples(OM.synthetic_sequences(B, T, cfg))]
    res = {}
    for mode in ("synced", "in_flight"):
        m = pk.Model(10, is_cdna=True, scheduled_sampling_k=900.0, prefix="q", height=H, width=H, compute="bf16")
        m.load_params(params)
        opt = pk.Adam().setup(m)
        step = pk.TrainStep(m, opt, B, T, graph=True)
        step.load_batch(*batch, non_blocking=False)
        np.random.seed(5)
        step(5990); torch.cuda.synchronize()       # capture outside the comparison
        handles, takes = [], []
        for i in range(N):
            handles.append(step(6000 + 150 * i))   # n_gt changes from step to step: a stale select would change the loss
            takes.append(m.take_gt.copy())
            if mode == "synced":
                float(handles[-1]); torch.cuda.synchronize()
        torch.cuda.synchronize()
        res[mode] = ([float(h) for h in handles], takes, m.engine.flat_p.clone())
    (l0, t0, p0), (l1, t1, p1) = res["synced"], res["in_flight"]
    assert all(np.array_equal(a, b) for a, b in zip(t0, t1))
    assert len(set(l0)) == N                       # the steps really differ
    # same kernels, same inputs, same order; the only run-to-run noise is the order of the fp32 atomics, which seven Adam updates of a
    # two-sample bf16 model amplify to ~2e-3 relative on the later losses (measured 1e-4 ... 2.0e-3 over repeated runs), whereas a select
    # or loss that belongs to another step moves the loss by several percent (neighbouring steps differ by 10-40 %)
    assert all(abs(a - b) <= 1e-2 * abs(a) for a, b in zip(l0, l1)), (l0, l1)
    assert float((p0 - p1).abs().max()) <= 2e-2
