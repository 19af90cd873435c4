"""CPU tests of SaveAt(ts): the Dopri5 dense output of the test reference (tests/dense_oracle.py) and the host side of
ecnf_solve_saveat (argument checks, workspace query), which need no device."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import ecnf_oracle as O
from ecnf_b200 import lib as L
from ecnf_b200.engine import CnfConfig, Engine
import dense_oracle as DO
from helpers import CASES, make_pair


def _random_step(S=5, seed=0):
    g = torch.Generator().manual_seed(seed)
    y0, y1 = torch.randn(S, generator=g, dtype=torch.float64), torch.randn(S, generator=g, dtype=torch.float64)
    k = [torch.randn(S, generator=g, dtype=torch.float64) for _ in range(7)]
    return y0, y1, k


def test_interpolant_hits_both_ends_and_the_midpoint():
    y0, y1, k = _random_step()
    assert torch.allclose(DO.dopri5_interp(y0, y1, k, 0.0), y0, rtol=0, atol=1e-14)
    assert torch.allclose(DO.dopri5_interp(y0, y1, k, 1.0), y1, rtol=0, atol=1e-12)
    y_mid = y0 + sum(c * kk for c, kk in zip(DO.DP_C_MID, k))
    assert torch.allclose(DO.dopri5_interp(y0, y1, k, 0.5), y_mid, rtol=0, atol=1e-12)


def _linear(Amat):
    A = torch.tensor(Amat, dtype=torch.float64)
    return lambda t, y: y @ A.T


@pytest.mark.parametrize("field", ["exp", "rotation"])
def test_dense_output_converges_at_fourth_order_or_better(field):
    """y' = lambda y and a rotation, fixed steps dt = 0.1, 0.05, 0.025: the dense-output error at interior times against
    the closed form falls by at least 2^4 per halving (the error of a 4th-order interpolant)."""
    ts = [0.137, 0.33, 0.5, 0.713, 0.9]
    if field == "exp":
        lam = -2.0
        func, y0 = _linear([[lam]]), torch.tensor([[1.0]], dtype=torch.float64)
        exact = np.array([[math.exp(lam * t)] for t in ts])
    else:
        w = 3.0
        func, y0 = _linear([[0.0, -w], [w, 0.0]]), torch.tensor([[1.0, 0.5]], dtype=torch.float64)
        exact = np.array([[math.cos(w * t) - 0.5 * math.sin(w * t), math.sin(w * t) + 0.5 * math.cos(w * t)] for t in ts])
    errs = []
    for dt in (0.1, 0.05, 0.025):
        _, st, path = DO.dopri5_saveat(func, y0, 0.0, 1.0, O.SolveControl(fixed=True, step_size=dt), ts)
        assert (st.status == 0).all()
        errs.append(np.abs(path[0].numpy() - exact).max())
    assert errs[2] > 1e-13, errs                              # far above fp64 rounding, so the ratios mean something
    assert errs[0] / errs[1] > 14 and errs[1] / errs[2] > 14, errs


@pytest.mark.parametrize("fixed", [True, False])
@pytest.mark.parametrize("mode", ["sample_logq", "logprob"])
def test_saving_leaves_the_oracle_solve_unchanged(fixed, mode):
    """fp64 solve of a small network with the exact trace: with ts the end state and the step counts are bit for bit
    those of oracle.dopri5, the start time returns the initial state (delta 0) and the end time the final state."""
    n, dim, blocks, units, H, nfeat = CASES["small_64_32"]
    ocfg, flat, _, _ = make_pair(n, dim, blocks, units, H, n_features=nfeat, head_variance=0.3, zero_time=True)
    p = O.to_torch(flat, torch.float64)
    rng = np.random.default_rng(3)
    B = 3
    x = O.base_sample_from_noise(ocfg, torch.tensor(rng.standard_normal((B, n * dim)))).double()
    feat = torch.tensor(rng.integers(0, nfeat, (B, n))).long()
    y0 = torch.cat([x, torch.zeros(B, 1, dtype=torch.float64)], dim=1)
    ctrl = O.SolveControl(fixed=fixed, step_size=0.1)
    t0, t1 = (0.0, 1.0) if mode == "sample_logq" else (1.0, 0.0)
    ts = [0.0, 0.05, 0.3, 0.61, 1.0] if t0 == 0.0 else [1.0, 0.95, 0.7, 0.39, 0.0]
    func = O._joint(p, ocfg, feat)
    y_ref, st_ref = O.dopri5(func, y0, t0, t1, ctrl)
    y, st, path = DO.dopri5_saveat(func, y0, t0, t1, ctrl, ts)
    assert torch.equal(y, y_ref)
    for name in ("n_steps", "n_accepted", "n_evals", "status"):
        assert np.array_equal(getattr(st, name), getattr(st_ref, name)), name
    assert torch.equal(path[:, 0], y0) and torch.equal(path[:, -1], y)
    assert torch.isfinite(path).all()
    y2, st2, none = DO.dopri5_saveat(func, y0, t0, t1, ctrl)
    assert none is None and torch.equal(y2, y_ref)


def test_early_stop_leaves_unreached_rows_nan():
    func = _linear([[-1.0]])
    y0 = torch.ones(1, 1, dtype=torch.float64)
    _, st, path = DO.dopri5_saveat(func, y0, 0.0, 1.0, O.SolveControl(fixed=True, step_size=0.1, max_steps=3),
                                   [0.0, 0.15, 0.3, 0.31, 0.9, 1.0])
    assert st.status[0] == 1
    assert torch.isfinite(path[0, :3]).all() and torch.isnan(path[0, 3:]).all()


# ---------------------------------------------------------------- C-ABI, host side
def _engine():
    return Engine(CnfConfig(13, 3, 0.01, 1.0, 3, (128,) * 3, 64, 8, 1))


def _saveat(lib, eng, mode, ts, B=2, traj=1, delta=1, ws=None, ws_bytes=0, logs=1):
    arr = (C.c_float * max(len(ts), 1))(*ts)
    return lib.ecnf_solve_saveat(eng.handle, mode, C.c_void_p(8), C.c_void_p(8), None, B, None, len(ts),
                                 arr if ts else None, C.c_void_p(8), C.c_void_p(logs), None, C.c_void_p(traj),
                                 C.c_void_p(delta), ws, ws_bytes, None)


def test_saveat_workspace_query():
    lib, eng = L.load(), _engine()
    for mode in (L.MODE_SAMPLE, L.MODE_SAMPLE_LOGQ, L.MODE_LOGPROB):
        for B in (1, 1000, 10_000):
            base = lib.ecnf_solve_workspace_bytes(eng.handle, mode, B)
            assert lib.ecnf_solve_saveat_workspace_bytes(eng.handle, mode, B, 0) == base
            for n in (1, 64, 65, 1024):
                got = lib.ecnf_solve_saveat_workspace_bytes(eng.handle, mode, B, n)
                assert got == (base + 255) // 256 * 256 + (4 * n + 255) // 256 * 256


def test_saveat_rejects_bad_arguments_with_messages():
    lib, eng = L.load(), _engine()
    S, LQ, LP = L.MODE_SAMPLE, L.MODE_SAMPLE_LOGQ, L.MODE_LOGPROB

    def err(rc, text):
        assert rc == -1, rc
        assert text in lib.ecnf_last_error().decode(), lib.ecnf_last_error()

    err(_saveat(lib, eng, LQ, [0.5] * (L.MAX_SAVE_TIMES + 1)), "n_save")
    arr = (C.c_float * 1)(0.5)
    err(lib.ecnf_solve_saveat(eng.handle, S, C.c_void_p(8), C.c_void_p(8), None, 2, None, -1, arr, C.c_void_p(8), None,
                              None, C.c_void_p(8), None, None, 0, None), "n_save")
    err(_saveat(lib, eng, LQ, [0.0, 1.5]), "outside [0, 1]")
    err(_saveat(lib, eng, LQ, [-0.1]), "outside [0, 1]")
    err(_saveat(lib, eng, LQ, [0.2, float("nan")]), "outside [0, 1]")
    err(_saveat(lib, eng, S, [0.2, 0.2]), "strictly increasing")
    err(_saveat(lib, eng, LQ, [0.7, 0.2]), "strictly increasing")
    err(_saveat(lib, eng, LP, [0.2, 0.7]), "strictly decreasing")
    err(_saveat(lib, eng, LP, [0.5], traj=0), "out_traj")
    err(lib.ecnf_solve_saveat(eng.handle, S, C.c_void_p(8), C.c_void_p(8), None, 2, None, 2, None, C.c_void_p(8), None,
                              None, C.c_void_p(8), None, None, 0, None), "ts_host")
    err(_saveat(lib, eng, LQ, [0.5], delta=0), "out_traj_delta")
    err(_saveat(lib, eng, LP, [0.5], logs=0), "out_logs")
    err(_saveat(lib, eng, 7, [0.5]), "bad mode")
    # valid arguments: a missing / short workspace is the workspace error, before any device work
    assert _saveat(lib, eng, LP, [1.0, 0.5, 0.0]) == -4
    need = lib.ecnf_solve_saveat_workspace_bytes(eng.handle, LP, 2, 3)
    assert _saveat(lib, eng, LP, [1.0, 0.5, 0.0], ws=C.c_void_p(256), ws_bytes=need - 1) == -4
    assert b"workspace" in lib.ecnf_last_error()
    assert _saveat(lib, eng, S, [0.0, 1.0], delta=0, logs=0) == -4       # out_traj_delta / out_logs unused in SAMPLE
    assert _saveat(lib, eng, S, [0.0, 1.0], B=0, delta=0, logs=0) == 0   # empty batch: nothing to do
