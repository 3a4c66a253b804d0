"""CPU tests of the forward-only prediction contract: the new flag values of the C-ABI are validated before any launch (fake pointers,
as in test_abi_host.py), and Predictor rejects malformed inputs with ValueError before it touches the device."""
import os
import sys

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


def conv5x5(L, mode, gates, flags, N=128, C=32):
    """pivp_tc_conv5x5 on a 2 x 32 x 32 map with 64 input channels; everything except `mode`, `gates` and `flags` is a valid launch."""
    return L.query("pivp_tc_conv5x5", FAKE, 64, 2, 32, 32, 64, FAKE, N, 128, mode, FAKE, FAKE if mode == 0 else 0, N, 0,
                   gates, 0, FAKE, FAKE, 64, 32, FAKE, 64, 32, 0, 0, 0, C, 1.0, flags, 0, 0)


def test_no_gate_flag_needs_mode_1(pk):
    L = pk.lib()
    n0 = L.query("pivp_launch_count")
    assert conv5x5(L, 0, 0, 4) == EINVAL                 # bit 2 ("no gate storage") with the plain epilogue
    assert conv5x5(L, 0, 0, 4 | 1) == EINVAL
    assert "bit 2" in L.cdll.pivp_last_error().decode()
    assert L.query("pivp_launch_count") == n0


def test_null_gates_need_the_no_gate_flag(pk):
    L = pk.lib()
    n0 = L.query("pivp_launch_count")
    assert conv5x5(L, 1, 0, 2) == EINVAL                 # NULL gates with bf16 gate storage requested
    assert conv5x5(L, 1, 0, 0) == EINVAL                 # NULL gates, fp32 gate storage
    assert L.query("pivp_launch_count") == n0


def test_fused_layernorm_cell_refuses_the_no_gate_flag(pk):
    L = pk.lib()
    n0 = L.query("pivp_launch_count")
    rc = L.query("pivp_tc_conv5x5_ln", FAKE, 64, 2, 32, 32, 64, FAKE, 32, FAKE, FAKE, 0, FAKE, FAKE, 64, 32, FAKE, 64, 32, 1.0, 4, FAKE,
                 FAKE, FAKE, 1e-6, FAKE, 32, 0, 0, 0, 0, FAKE, FAKE, 0)
    assert rc == EINVAL and L.query("pivp_launch_count") == n0


def test_heads_ln_still_checks_a_given_y(pk):
    """y == NULL is allowed (the normalised rows are not written); a y that is given must still be 16-byte aligned."""
    L = pk.lib()
    n0 = L.query("pivp_launch_count")
    args = lambda y: (FAKE, 64, 0, FAKE, FAKE, FAKE, 1e-6, FAKE, y, 64, 0, FAKE, FAKE, FAKE, 3, FAKE, 14, 2, 4096, 0)
    assert L.query("pivp_heads_fwd_ln", *args(FAKE + 4)) == EINVAL
    assert L.query("pivp_heads_fwd_ln", *(args(0)[:7] + (0,) + args(0)[8:])) == EINVAL       # stats stays required
    assert L.query("pivp_launch_count") == n0


class _Eng(object):
    H = W = 64


def _stub(pk, B=2, T=6, ctx=2):
    """A Predictor with the attributes its input check reads and no device state (this machine may have no GPU)."""
    P = pk.Predictor
    p = P.__new__(P)
    p.B, p.T, p.ctx, p.e = B, T, ctx, _Eng()
    return p


def test_predictor_rejects_malformed_inputs(pk):
    p = _stub(pk)
    rs = np.random.RandomState(0)
    img = rs.rand(2, 2, 3, 64, 64).astype(np.float32)
    act = rs.rand(5, 2, 5).astype(np.float32)
    sta = rs.rand(2, 5).astype(np.float32)
    c, a, s, N = p._check(img, act, sta)
    assert N == 2 and tuple(c.shape) == (2, 2, 3, 64, 64) and tuple(s.shape) == (1, 2, 5)
    assert p._check(np.concatenate([img, img]), act, sta[:1])[0].shape[0] == 2        # extra context frames are not read; state broadcast
    assert p._check(img[:, :1], rs.rand(5, 7, 5).astype(np.float32), sta[:1])[3] == 7   # N may exceed batch_size; context broadcast
    bad = [(img[:1], act, sta),                                    # fewer frames than context_frames
           (img, act[:4], sta),                                    # T-1 action steps expected
           (img, act[..., :4], sta),                               # 5 action components
           (img[..., :32], act, sta),                              # image size
           (img, act, sta[:, :4]),                                 # 5 state components
           (img, act, sta[None]),                                  # first_state rank
           (np.concatenate([img] * 2, axis=1)[:, :3], act, sta),   # context batch neither 1 nor N
           (img, act, np.concatenate([sta, sta])),                 # state batch neither 1 nor N
           (img.astype(np.float64), act, sta),                     # dtype
           (img, act.astype(np.float16), sta),
           (img, act[:, :0], sta[:0])]                             # no candidates
    for args in bad:
        with pytest.raises(ValueError):
            p._check(*args)
