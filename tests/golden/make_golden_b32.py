"""Frozen oracle vectors for the BASELINE.json metric configuration: CDNA 64x64, B=32, T=10, 10 masks, scheduled sampling at
iteration 6000 (17 of 32 samples take the ground truth) -- the exact shapes bench.py times, so the GPU parity test exercises the
kernel instantiations the benchmark runs (two-tile halo CTAs, b32-sized split-K weight gradients).

The float64 oracle needs ~16 GB and ~2 minutes for this case, too much for every test run; it is run ONCE here and a compact
summary is frozen: all scalars, the frames of SAMPLES and the mask logits of two samples at two time steps at the PIXELS (a fixed,
seeded quarter of the pixel positions, the same for every sample, time step and channel), per-(t, sample) frame statistics of every
sample, and for every parameter gradient its L2 norm, its sum and a strided subsample (every stride_of(n)-th element in Chainer
layout, C order; tensors of up to 8192 elements whole) from which the relative L2 error of the whole tensor is estimated without bias.
The pixel and gradient samples keep the file under 1 MB.

    python tests/golden/make_golden_b32.py        # from the repo root; writes tests/golden/cdna_b32_t10.npz
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import model as M  # noqa: E402

B, T, H, ITER, K = 32, 10, 64, 6000, 900.0
SAMPLES = (0, 13, 31)
MASK_T = (0, 8)
MASK_SAMPLES = (0, 31)
STRIDE = 61
PIXELS = np.sort(np.random.RandomState(0).choice(H * H, H * H // 4, replace=False))       # flat h * W + w


def stride_of(n):
    """Tensors up to 8192 elements are stored whole; larger ones every STRIDE-th element, or every k * STRIDE-th when that still
    leaves at least 4096 elements."""
    return 1 if n <= 8192 else STRIDE * max(1, n // (STRIDE * 4096))


def at_pixels(x):
    """(..., H, W) -> (..., len(PIXELS)): the values at the stored pixel positions."""
    return x.reshape(x.shape[:-2] + (-1,))[..., PIXELS]


def params_for(cfg):
    params = M.init_params(cfg, seed=4321)
    rs = np.random.RandomState(7)
    for key in sorted(params):            # move LN/bias params off their 1/0 init so their grads matter
        if not key.endswith("/W"):
            params[key] = (params[key] + 0.05 * rs.standard_normal(params[key].shape)).astype(np.float32)
    return params


def main():
    cfg = M.Config("CDNA", 10, schedsamp_k=K, height=H, width=H, dtype=np.float64)
    params = params_for(cfg)
    batch = M.concat_examples(M.synthetic_sequences(B, T, cfg, seed=1234))
    np.random.seed(99)
    take = []
    out = M.forward(params, batch, ITER, cfg, take_gt_log=take)
    M.G.backward(out["loss"])
    gen = np.stack([g.data for g in out["gen_images"]])                       # (T-1, B, 3, H, W)
    res = {
        "loss": np.float64(out["loss"].data),
        "psnr_all": np.float64(out["psnr_all"]),
        "recon_costs": np.array(out["recon_costs"], np.float64),
        "n_gt": np.int32(out["n_gt"]),
        "take_gt": np.array(take, dtype=np.bool_).reshape(len(take), B),
        "gen_sub": at_pixels(gen[:, list(SAMPLES)]).astype(np.float32),
        "gen_mean": gen.mean(axis=(2, 3, 4)),
        "gen_l2": np.sqrt((gen ** 2).sum(axis=(2, 3, 4))),
        "mask_pre_sub": np.stack([at_pixels(out["trace"][t]["mask_pre"].data[list(MASK_SAMPLES)]) for t in MASK_T]).astype(np.float16),
        "gen_states": np.stack([g.data for g in out["gen_states"]]).astype(np.float32),
    }
    for key, v in out["P"].items():
        g = (np.zeros_like(v.data) if v.grad is None else v.grad).astype(np.float64)
        res["gsum/" + key] = np.float64(g.sum())
        res["gl2/" + key] = np.float64(np.sqrt((g ** 2).sum()))
        res["gsub/" + key] = g.reshape(-1)[::stride_of(g.size)].astype(np.float32)
    np.savez_compressed(os.path.join(HERE, "cdna_b32_t10.npz"), **res)
    print("cdna_b32_t10", float(res["loss"]), int(res["n_gt"]))


if __name__ == "__main__":
    main()
