"""GPU tests of SaveAt(ts) (ecnf_solve_saveat, Engine.solve(ts=), the ts= keyword of the façade) on both solve engines:
the dense-output path against the test reference (tests/dense_oracle.py), bit-identity of everything else with and
without saving, an accuracy check independent of the interpolant weights, batch consistency and early stops."""
import numpy as np
import pytest
import torch

from oracle import ecnf_oracle as O
from ecnf_b200 import lib as L
from ecnf_b200.cnf import build_cnf, get_log_prob, sample_and_log_prob_cnf, sample_cnf
from ecnf_b200.engine import Engine
import dense_oracle as DO
from helpers import CASES, make_pair, rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-4
TS_FWD = [0.0, 0.013, 0.25, 0.5, 0.77, 0.999, 1.0]
TS_REV = [1.0, 0.987, 0.75, 0.5, 0.23, 0.001, 0.0]
MODES = {"sample": L.MODE_SAMPLE, "sample_logq": L.MODE_SAMPLE_LOGQ, "logprob": L.MODE_LOGPROB}

# (case, engine choice, engine the solve must run on: 0 tcgen05, 1 fp32 SIMT)
ROWS = [("small_64_32", 0, 0), ("lj13", 0, 0), ("qm9_like", 0, 1), ("lj13", 1, 1)]


def _setup(case, B, seed, engine, adaptive=False):
    n, dim, blocks, units, H, nfeat = CASES[case]
    kw = dict(head_variance=0.3, zero_time=True) if adaptive else {}
    ocfg, flat, tree, ecfg = make_pair(n, dim, blocks, units, H, n_features=nfeat, **kw)
    eng = Engine(ecfg)
    eng.set_engine(engine)
    rng = np.random.default_rng(seed)
    x = O.base_sample_from_noise(ocfg, torch.tensor(rng.standard_normal((B, n * dim)).astype(np.float32)))
    feat = rng.integers(0, nfeat, (B, n)).astype(np.int32)
    probe = rng.standard_normal((B, n * dim)).astype(np.float32)
    return ocfg, flat, tree, eng, x, feat, probe


def _oracle_path(flat, ocfg, mode, x, feat, ctrl, ts, eps=None):
    p32 = O.to_torch(flat, torch.float32)
    ft = torch.tensor(feat).long()
    if mode == L.MODE_SAMPLE:
        _, st, path = DO.sample_cnf(p32, ocfg, x, ft, ctrl, ts)
        return path, None, st
    if mode == L.MODE_SAMPLE_LOGQ:
        *_, st, path = DO.sample_and_log_prob_cnf(p32, ocfg, x, ft, ctrl, ts, eps)
    else:
        *_, st, path = DO.get_log_prob(p32, ocfg, x, ft, ctrl, ts, eps)
    return path[..., :-1], path[..., -1], st


def _check_parity(eng, tree, flat, ocfg, mode, x, feat, fixed, eps=None):
    ts = TS_REV if mode == L.MODE_LOGPROB else TS_FWD
    ctrl_o = O.SolveControl(fixed=fixed)
    traj_ref, dl_ref, st_ref = _oracle_path(flat, ocfg, mode, x, feat, ctrl_o, ts, None if eps is None else torch.tensor(eps))
    _, _, stats, traj, dl = eng.solve(tree, mode, x.numpy(), feat, L.make_ctrl(use_fixed_step_size=fixed), eps=eps, ts=ts)
    st = stats.cpu().numpy()
    assert (st[:, 3] == 0).all()
    assert np.abs(st[:, 1] - st_ref.n_accepted).max() <= (0 if fixed else 1), (st[:, 1], st_ref.n_accepted)
    assert traj.shape == (x.shape[0], len(ts), x.shape[1])
    assert rel_err(traj.cpu().numpy(), traj_ref.numpy()) < TOL
    if mode == L.MODE_SAMPLE:
        assert dl is None
    else:
        d, r = dl.cpu().numpy(), dl_ref.numpy()
        assert np.abs(d - r).max() < TOL * (np.abs(r).max() + 1), np.abs(d - r).max()


@pytest.mark.parametrize("stepping", ["fixed", "adaptive"])
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("row", ROWS, ids=[f"{c}-engine{e}" for c, e, _ in ROWS])
def test_path_matches_oracle_dense_output(row, mode, stepping, cuda_device):
    """Fixed step, and adaptive on the smooth (zero_time) field as in test_gpu_solve.py, exact trace."""
    case, engine, expect = row
    adaptive = stepping == "adaptive"
    B = 2 if case == "lj13" else 3
    ocfg, flat, tree, eng, x, feat, _ = _setup(case, B, 11, engine, adaptive)
    assert eng.lib.ecnf_solve_engine_for(eng.handle, MODES[mode]) == expect
    _check_parity(eng, tree, flat, ocfg, MODES[mode], x, feat, not adaptive)


@pytest.mark.parametrize("mode", ["sample_logq", "logprob"])
@pytest.mark.parametrize("row", ROWS, ids=[f"{c}-engine{e}" for c, e, _ in ROWS])
def test_path_matches_oracle_hutchinson(row, mode, cuda_device):
    case, engine, expect = row
    B = 2 if case == "lj13" else 3
    ocfg, flat, tree, eng, x, feat, probe = _setup(case, B, 12, engine)
    assert eng.lib.ecnf_solve_engine_for(eng.handle, MODES[mode]) == expect
    _check_parity(eng, tree, flat, ocfg, MODES[mode], x, feat, True, eps=probe)


@pytest.mark.parametrize("engine", [0, 1])
@pytest.mark.parametrize("mode", list(MODES))
def test_saving_does_not_perturb_the_solve(mode, engine, cuda_device):
    """out_x / out_logs / out_stats are bit-identical with and without ts; the start time saves x_init and 0, the end time
    saves out_x and the delta column bit for bit (adaptive LJ13 on the time-forced field, many steps, exact trace)."""
    m = MODES[mode]
    ocfg, flat, tree, eng, x, feat, _ = _setup("lj13", 40, 13, engine)
    assert eng.lib.ecnf_solve_engine_for(eng.handle, m) == engine
    ctrl = L.make_ctrl()
    ts = TS_REV if m == L.MODE_LOGPROB else TS_FWD
    x_a, logs_a, st_a = eng.solve(tree, m, x.numpy(), feat, ctrl)
    x_b, logs_b, st_b, traj, dl = eng.solve(tree, m, x.numpy(), feat, ctrl, ts=ts)
    assert torch.equal(x_a, x_b) and torch.equal(st_a, st_b)
    # not a vacuous check: the solves take several accepted steps on average and reject some
    assert st_a[:, 1].float().mean() > 3 and (st_a[:, 0] > st_a[:, 1]).any(), st_a[:, :2]
    assert torch.equal(traj[:, 0], x.to(traj.device)) and torch.equal(traj[:, -1], x_b)
    assert torch.isfinite(traj).all()
    if m == L.MODE_SAMPLE:
        assert logs_a is None and logs_b is None and dl is None
    else:
        assert torch.equal(logs_a, logs_b)
        assert (dl[:, 0] == 0).all() and torch.equal(dl[:, -1], logs_b[:, 2])
    x_c, _, st_c, traj_c, _ = eng.solve(tree, m, x.numpy(), feat, ctrl, ts=[])     # n_save = 0: the plain solve
    assert torch.equal(x_c, x_a) and torch.equal(st_c, st_a) and traj_c.shape == (40, 0, ocfg.D)


def test_adaptive_dense_output_agrees_with_a_fine_fixed_step_solve(cuda_device):
    """Independent of the interpolant weights: adaptive LJ13 (rtol = atol = 1e-5) at interior times against a fixed-step
    dt = 0.005 solve, whose own interpolation error is negligible at that step.  Bound: the interior error is at most 10x
    the adaptive solve's error at the end time (a 4th-order interpolant of 5th-order steps), floor 1e-4 relative."""
    ocfg, flat, tree, eng, x, feat, _ = _setup("lj13", 8, 14, 0, adaptive=True)
    ts = [0.0, 0.1, 0.237, 0.5, 0.618, 0.9, 1.0]
    _, logs_a, st_a, tr_a, dl_a = eng.solve(tree, L.MODE_SAMPLE_LOGQ, x.numpy(), feat, L.make_ctrl(), ts=ts)
    _, logs_f, st_f, tr_f, dl_f = eng.solve(tree, L.MODE_SAMPLE_LOGQ, x.numpy(), feat,
                                            L.make_ctrl(use_fixed_step_size=True, step_size=0.005), ts=ts)
    assert (st_f[:, 1] == 200).all() and (st_a[:, 1] < 100).all()
    a, f = tr_a.cpu().numpy(), tr_f.cpu().numpy()
    scale = np.abs(f).max()
    e_end = np.abs(a[:, -1] - f[:, -1]).max() / scale
    e_mid = np.abs(a[:, 1:-1] - f[:, 1:-1]).max() / scale
    d_end = np.abs((dl_a - dl_f).cpu().numpy()[:, -1]).max()
    d_mid = np.abs((dl_a - dl_f).cpu().numpy()[:, 1:-1]).max()
    dscale = np.abs(dl_f.cpu().numpy()).max() + 1
    print(f"adaptive vs dt=0.005: end {e_end:.2e} interior {e_mid:.2e}; delta end {d_end:.2e} interior {d_mid:.2e}; "
          f"accepted steps {st_a[:, 1].tolist()}")
    assert e_mid < max(10 * e_end, 1e-4), (e_mid, e_end)
    assert d_mid < max(10 * d_end, 1e-4 * dscale), (d_mid, d_end)


@pytest.mark.parametrize("engine", [0, 1])
def test_batch_copies_and_repeats_are_bit_identical(engine, cuda_device):
    """2 * #SMs + 5 copies of 4 trajectories (the work queue hands copies to different CTAs, several per CTA): every copy's
    path is bit-identical, and so is a second launch."""
    ocfg, flat, tree, eng, x4, feat4, _ = _setup("lj13", 4, 15, engine, adaptive=True)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 2 * sms + 5
    idx = np.arange(B) % 4
    x, feat = x4.numpy()[idx], feat4[idx]
    run = lambda: eng.solve(tree, L.MODE_SAMPLE_LOGQ, x, feat, L.make_ctrl(), ts=TS_FWD)
    a, b = run(), run()
    for k in (0, 1, 2, 3, 4):
        assert torch.equal(a[k], b[k]), k
    tr, dl = a[3], a[4]
    for j in range(4):
        assert torch.equal(tr[j::4], tr[j].expand_as(tr[j::4])) and torch.equal(dl[j::4], dl[j].expand_as(dl[j::4]))


@pytest.mark.parametrize("engine", [0, 1])
@pytest.mark.parametrize("mode", ["sample", "logprob"])
def test_early_stop_fills_unreached_rows_with_nan(mode, engine, cuda_device):
    """max_steps = 3 at dt = 0.05 stops at t = 0.15 (t = 0.85 backwards): status 1, NaN in exactly the later rows."""
    m = MODES[mode]
    ocfg, flat, tree, eng, x, feat, _ = _setup("lj13", 3, 16, engine)
    ts = [0.0, 0.1, 0.12, 0.2, 0.5, 1.0] if m == L.MODE_SAMPLE else [1.0, 0.9, 0.88, 0.8, 0.5, 0.0]
    ctrl = L.make_ctrl(use_fixed_step_size=True, max_steps=3)
    _, _, st, tr, dl = eng.solve(tree, m, x.numpy(), feat, ctrl, ts=ts)
    assert (st[:, 3] == 1).all() and (st[:, 0] == 3).all()
    assert torch.isfinite(tr[:, :3]).all() and torch.isnan(tr[:, 3:]).all()
    if dl is not None:
        assert torch.isfinite(dl[:, :3]).all() and torch.isnan(dl[:, 3:]).all()


def test_facade_shapes_squeeze_and_unchanged_default(cuda_device):
    n, dim, blocks, units, H, nfeat = CASES["dw4"]
    ocfg, flat, tree, _ = make_pair(n, dim, blocks, units, H, n_features=nfeat)
    cnf = build_cnf(n, dim, 0.01, 1.0, blocks, units, H, 8, nfeat)
    D, B, ts = n * dim, 5, np.linspace(0.0, 1.0, 11)
    rng = np.random.default_rng(17)
    x0 = O.base_sample_from_noise(ocfg, torch.tensor(rng.standard_normal((B, D)).astype(np.float32)))
    fx = dict(use_fixed_step_size=True, x0=x0)

    x1 = sample_cnf(cnf, tree, 0, **fx)
    x1s, xs = sample_cnf(cnf, tree, 0, **fx, ts=ts)
    assert torch.equal(x1, x1s) and xs.shape == (B, 11, D) and torch.equal(xs[:, -1], x1)
    x1_1, xs_1 = sample_cnf(cnf, tree, 0, use_fixed_step_size=True, x0=x0[0], ts=ts)
    assert x1_1.shape == (D,) and xs_1.shape == (11, D) and torch.equal(xs_1, xs[0])

    r0 = sample_and_log_prob_cnf(cnf, tree, 0, **fx)
    r1 = sample_and_log_prob_cnf(cnf, tree, 0, **fx, ts=ts)
    assert len(r0) == 2 and len(r1) == 4
    assert torch.equal(r0[0], r1[0]) and torch.equal(r0[1], r1[1])
    assert r1[2].shape == (B, 11, D) and r1[3].shape == (B, 11)
    # log q_t(x_t) = log p0(x0) - delta(t); at t = 1 this is the returned log q
    lq_path = cnf.engine.base_log_prob(x0)[:, None] - r1[3]
    assert torch.allclose(lq_path[:, -1], r1[1], rtol=0, atol=1e-5 * (float(r1[1].abs().max()) + 1))
    r1s = sample_and_log_prob_cnf(cnf, tree, 0, use_fixed_step_size=True, x0=x0[0], ts=ts, return_stats=True)
    assert len(r1s) == 5 and r1s[2].shape == (11, D) and r1s[3].shape == (11,)

    g0 = get_log_prob(cnf, tree, r0[0], use_fixed_step_size=True)
    g1 = get_log_prob(cnf, tree, r0[0], use_fixed_step_size=True, ts=ts[::-1].copy())
    assert len(g0) == 3 and len(g1) == 5
    for a, b in zip(g0, g1):
        assert torch.equal(a, b)
    assert g1[3].shape == (B, 11, D) and g1[4].shape == (B, 11) and torch.equal(g1[4][:, -1], g0[2])
    g1s = get_log_prob(cnf, tree, r0[0][0], use_fixed_step_size=True, ts=ts[::-1].copy())
    assert g1s[3].shape == (11, D) and g1s[4].shape == (11,)
    with pytest.raises(L.EcnfError, match="strictly decreasing"):
        get_log_prob(cnf, tree, r0[0], use_fixed_step_size=True, ts=ts)
