"""GPU parity over the space of networks ecnf_model_create accepts: both solve engines against the fp64 oracle at the shapes
where the tensor-core engine changes its internal structure (ecnf_solve_tc.cuh: tc_pick_mrows / tc_pack / tc_eligible) and
at the limits of the fp32 SIMT engine (Geo<U,H>::TR, 227 KB of shared memory).

Structure of the tcgen05 engine that the rows below aim at (MR = rows of the message accumulator, D = n * dim):
  * TT_MID (blocks after the first, exact trace): windows of whole receivers while 1 + D <= MR, else one receiver x a range
    of slot chunks, (MR - 1) / 7 chunks per window (MR = 8: one chunk per window);
  * TT_FIRST: windows of MR / (1 + dim) receivers;
  * tiles of 16 * SUB chunks (SUB = 128 / U: two sub-tiles stacked on the TMEM lanes for U = 64);
  * the dense kinds of sample-only solves (TT_NODE1 / TT_EDGE1) pack 8 primal rows per chunk.
Every row states the engine each call must run on (ecnf_solve_engine_for), or the error it must raise; the host test
tests/test_config_sweep_host.py checks, without a GPU, that the rows still reach the structures their reasons name.
"""
from collections import namedtuple

import numpy as np
import pytest
import torch

from oracle import ecnf_oracle as O
from ecnf_b200 import lib as L
from ecnf_b200.engine import Engine
from helpers import make_pair, rel_err

pytestmark = pytest.mark.gpu

TC, SIMT = 0, 1           # ecnf_solve_engine_for: tcgen05 tensor cores / fp32 SIMT
UNSUPPORTED = -3          # ... or ECNF_ERR_UNSUPPORTED: the call fails
SMEM = "exceeds 227 KB"   # expected EcnfError text of the shapes no engine runs

Row = namedtuple("Row", "name n dim U H blocks L T nfeat nc div sample simt_div why")
_D = dict(blocks=2, L=2, T=8, nfeat=1, nc=1.0)


def row(name, n, dim, U, div, sample, simt_div, why, **kw):
    a = {**_D, **kw}
    return Row(name, n, dim, U, {128: 64, 64: 32, 256: 32}[U], a["blocks"], a["L"], a["T"], a["nfeat"], a["nc"], div, sample,
               simt_div, why)


# div / sample: engine of the exact-trace (and Hutchinson) calls and of the sample-only / plain-VF calls on the automatic engine
# choice; simt_div: the exact-trace calls with ecnf_model_set_engine(1).  A string is the EcnfError those calls must raise.
SWEEP = [
    #    name                n  dim  U     div   sample simt_div  why
    # -- smallest graph: one edge per receiver, every tile nearly empty
    row("n2_d2_u128",        2, 2, 128,   TC,   TC,    SIMT,     "smallest graph"),
    row("n2_d3_u128",        2, 3, 128,   TC,   TC,    SIMT,     "smallest graph"),
    row("n2_d2_u64",         2, 2, 64,    TC,   TC,    SIMT,     "smallest graph, stacked sub-tiles"),
    row("n2_d3_u64",         2, 3, 64,    TC,   TC,    SIMT,     "smallest graph, stacked sub-tiles"),
    row("n2_d2_u256",        2, 2, 256,   SIMT, SIMT,  SIMT,     "smallest graph, SIMT-only pair"),
    row("n2_d3_u256",        2, 3, 256,   SIMT, SIMT,  SIMT,     "smallest graph, SIMT-only pair"),
    # -- window and tile structure, U = 128
    row("n15_d3_u128",      15, 3, 128,   TC,   TC,    SIMT,     "last whole-receiver TT_MID window (1 + D = 46 = MR)"),
    row("n16_d3_u128",      16, 3, 128,   TC,   TC,    SIMT,     "first TT_MID slot windows"),
    row("n17_d3_u128",      17, 3, 128,   TC,   TC,    SIMT,     "slot windows, 52 tangent rows"),
    row("n20_d3_u128",      20, 3, 128,   TC,   TC,    SIMT,     "slot windows, MR 29; last exact-trace shape the SIMT engine fits"),
    row("n21_d3_u128",      21, 3, 128,   TC,   TC,    SMEM,     "first shape whose SIMT exact trace is out of shared memory"),
    row("n23_d3_u128",      23, 3, 128,   TC,   TC,    SMEM,     "last sample-only shape on tcgen05 (dim 3)"),
    row("n24_d3_u128",      24, 3, 128,   TC,   SIMT,  SMEM,     "MR 15; first sample-only shape past tcgen05; SIMT div out of smem"),
    row("n26_d3_u128",      26, 3, 128,   TC,   SIMT,  SMEM,     "MR = 8 (one chunk per window), last exact-trace shape on tcgen05"),
    row("n27_d3_u128",      27, 3, 128,   SMEM, SIMT,  SMEM,     "first exact-trace shape past tcgen05: no engine has room"),
    row("n29_d2_u128",      29, 2, 128,   TC,   TC,    SIMT,     "last sample-only shape on tcgen05 (dim 2)"),
    row("n30_d2_u128",      30, 2, 128,   TC,   SIMT,  SIMT,     "first sample-only shape past tcgen05 (dim 2)"),
    row("n32_d2_u128",      32, 2, 128,   TC,   SIMT,  SMEM,     "992 edges, the largest edge table; last exact-trace shape (dim 2)"),
    # -- the same on U = 64 (two sub-tiles stacked on the lanes), dim 2 included
    row("n9_d2_u64",         9, 2, 64,    TC,   TC,    SIMT,     "72 edge groups: exactly 9 dense chunks"),
    row("n14_d3_u64",       14, 3, 64,    TC,   TC,    SIMT,     "last whole-receiver TT_MID window"),
    row("n15_d3_u64",       15, 3, 64,    TC,   TC,    SIMT,     "first TT_MID slot windows"),
    row("n22_d2_u64",       22, 2, 64,    TC,   TC,    SIMT,     "first slot windows (dim 2)"),
    row("n22_d3_u64",       22, 3, 64,    TC,   TC,    SIMT,     "last sample-only shape on tcgen05 (dim 3)"),
    row("n23_d3_u64",       23, 3, 64,    TC,   SIMT,  SIMT,     "MR 15; first sample-only shape past tcgen05 (dim 3)"),
    row("n24_d3_u64",       24, 3, 64,    TC,   SIMT,  SIMT,     "MR = 8, partial tiles only"),
    row("n25_d3_u64",       25, 3, 64,    TC,   SIMT,  SIMT,     "MR = 8, last exact-trace shape on tcgen05 (dim 3)"),
    row("n26_d3_u64",       26, 3, 64,    SIMT, SIMT,  SIMT,     "first exact-trace shape past tcgen05 (dim 3)"),
    row("n28_d2_u64",       28, 2, 64,    TC,   TC,    SIMT,     "last sample-only shape on tcgen05 (dim 2)"),
    row("n29_d2_u64",       29, 2, 64,    TC,   SIMT,  SIMT,     "first sample-only shape past tcgen05 (dim 2)"),
    row("n32_d2_u64",       32, 2, 64,    TC,   SIMT,  SIMT,     "992 edges, MR 15 (dim 2)"),
    # -- SIMT only (256, 32): TR = 64 tangent rows per tile
    row("n21_d3_u256",      21, 3, 256,   SIMT, SIMT,  SIMT,     "1 + D = 64 = TR exactly"),
    row("n22_d3_u256",      22, 3, 256,   "tangent slots exceed the 64-row tile", SIMT,
        "tangent slots exceed the 64-row tile",                  "1 + D = 67 > TR: exact trace fails, plain VF runs"),
    # -- depth and width axes on a small graph (n = 5, dim 3), both tensor-core pairs
    *[r for U in (128, 64) for r in (
        row(f"l1_u{U}",      5, 3, U,     TC,   TC,    SIMT,     "1 MLP layer: the first phi_e layer is the message layer", L=1),
        row(f"l6_u{U}",      5, 3, U,     TC,   TC,    SIMT,     "6 MLP layers", L=6),
        row(f"b1_u{U}",      5, 3, U,     TC,   TC,    SIMT,     "1 EGNN block: TT_FIRST is also the last block", blocks=1),
        row(f"b8l2_u{U}",    5, 3, U,     TC,   TC,    SIMT,     "8 blocks x 2 layers: 72 weight images (> 64)", blocks=8),
        row(f"b8l6_u{U}",    5, 3, U,     TC,   TC,    SIMT,     "8 blocks x 6 layers: 168 weight images", blocks=8, L=6),
        row(f"t4_u{U}",      5, 3, U,     TC,   TC,    SIMT,     "time_dim 4", T=4),
        row(f"t16_u{U}",     5, 3, U,     TC,   TC,    SIMT,     "time_dim 16", T=16),
        row(f"nc05_u{U}",    5, 3, U,     TC,   TC,    SIMT,     "normalization_constant 0.5", nc=0.5),
    )],
    row("nf5_u128",          5, 3, 128,   TC,   TC,    SIMT,     "5 node features on U = 128", nfeat=5),
    row("b6l3_u128",        13, 3, 128,   TC,   TC,    SIMT,     "LJ13 width with 6 blocks: 72 weight images", blocks=6, L=3),
]
ROWS = {r.name: r for r in SWEEP}

# one row per tensor-core branch for the ODE-loop checks (fixed-step solves, the work queue)
SOLVE_ROWS = ["n2_d3_u128", "n2_d2_u64", "n17_d3_u128", "n26_d3_u128", "n24_d3_u64", "l1_u128", "l1_u64", "b8l2_u128",
              "b8l2_u64", "n22_d2_u64"]
# depth / width rows (+ the smallest graph and dim 2 on U = 64) for the flow-matching gradient
TRAIN_ROWS = ["n2_d3_u128", "n2_d2_u64", "n22_d2_u64"] + [r.name for r in SWEEP if r.n == 5]

VF_TOL = 2e-5     # relative to max |f|
DIV_TOL = 5e-5    # relative to max |div| + 1
SOLVE_TOL = 1e-4
LOSS_TOL, GRAD_TOL = 1e-5, 1e-4
# 8 blocks x 6 layers: the attention-gate gradients of the middle blocks nearly cancel (|g| ~ 1e-9 on b8l6_u64), and fp32
# autograd on the CPU misses GRAD_TOL on them as well (4.5e-4 on EGNN_0/3/Dense_1/bias against fp64; the kernel: 4.0e-4).
# These rows are bounded by DEEP_MULT x the fp32 autograd error of the same tensor instead.
DEEP_ROWS, DEEP_MULT = ("b8l6_u128", "b8l6_u64"), 3.0

DIV_MODES = (L.MODE_VF_DIV, L.MODE_SAMPLE_LOGQ, L.MODE_LOGPROB)
PRIMAL_MODES = (L.MODE_VF, L.MODE_SAMPLE)


def build(r, **kw):
    ocfg, flat, tree, ecfg = make_pair(r.n, r.dim, r.blocks, (r.U,) * r.L, r.H, T=r.T, n_features=r.nfeat,
                                       normalization_constant=r.nc, **kw)
    return ocfg, flat, tree, Engine(ecfg)


def engine_for(eng, mode):
    return eng.lib.ecnf_solve_engine_for(eng.handle, mode)


def expected(r, engine):
    """(exact-trace, sample-only) expectation of a row under ecnf_model_set_engine(engine)."""
    return (r.div if engine == 0 else r.simt_div), (r.sample if engine == 0 else SIMT)


def check_engine_query(eng, r, engine):
    div, sample = expected(r, engine)
    for mode in DIV_MODES:
        assert engine_for(eng, mode) == (UNSUPPORTED if isinstance(div, str) else div), (r.name, engine, mode)
    for mode in PRIMAL_MODES:
        assert engine_for(eng, mode) == sample, (r.name, engine, mode)


def div_err(a, ref):
    a, ref = np.asarray(a, np.float64), np.asarray(ref, np.float64)
    return float(np.abs(a - ref).max() / (np.abs(ref).max() + 1.0))


@pytest.mark.parametrize("name", list(ROWS))
def test_vf_div_hutchinson_match_oracle(name, cuda_device):
    r = ROWS[name]
    ocfg, flat, tree, eng = build(r)
    B = 3
    rng = np.random.default_rng(101)
    x = rng.standard_normal((B, r.n * r.dim)).astype(np.float32) * 1.3 + 0.2
    t = rng.uniform(0, 1, B).astype(np.float32)
    eps = rng.standard_normal((B, r.n * r.dim)).astype(np.float32)
    feat = rng.integers(0, r.nfeat, (B, r.n)).astype(np.int32)
    p64 = O.to_torch(flat, torch.float64)
    x64, t64, ft = torch.tensor(x, dtype=torch.float64), torch.tensor(t, dtype=torch.float64), torch.tensor(feat).long()
    f_ref, div_ref = O.vf_and_exact_div(p64, ocfg, x64, t64, ft)
    _, h_ref = O.vf_and_hutchinson_div(p64, ocfg, x64, t64, ft, torch.tensor(eps, dtype=torch.float64))
    f_ref, div_ref, h_ref = f_ref.numpy(), div_ref.numpy(), h_ref.numpy()
    try:
        for engine in (0, 1):
            eng.set_engine(engine)
            check_engine_query(eng, r, engine)
            div, _ = expected(r, engine)
            e_f = rel_err(eng.apply(tree, x, t, feat).cpu().numpy(), f_ref)
            assert e_f < VF_TOL, (engine, e_f)
            if isinstance(div, str):
                with pytest.raises(L.EcnfError, match=div):
                    eng.apply_div(tree, x, t, feat)
                with pytest.raises(L.EcnfError, match=div):
                    eng.apply_hutchinson(tree, x, t, eps, feat)
                print(f"sweep {name} engine={engine}: vf {e_f:.2e}; div raises as expected")
                continue
            f2, d = eng.apply_div(tree, x, t, feat)
            f3, h = eng.apply_hutchinson(tree, x, t, eps, feat)
            e_f2, e_f3 = rel_err(f2.cpu().numpy(), f_ref), rel_err(f3.cpu().numpy(), f_ref)
            e_d, e_h = div_err(d.cpu().numpy(), div_ref), div_err(h.cpu().numpy(), h_ref)
            print(f"sweep {name} engine={engine}: vf {max(e_f, e_f2, e_f3):.2e} div {e_d:.2e} hutch {e_h:.2e}")
            assert e_f2 < VF_TOL and e_f3 < VF_TOL, (engine, e_f2, e_f3)
            assert e_d < DIV_TOL, (engine, e_d)
            assert e_h < DIV_TOL, (engine, e_h)
    finally:
        eng.set_engine(0)


def _solve_both(eng, tree, mode, x0, feat, ctrl):
    out = eng.solve(tree, mode, x0, feat, ctrl)
    return out[0].cpu().numpy(), (None if out[1] is None else out[1].cpu().numpy()), out[2].cpu().numpy()


@pytest.mark.parametrize("name", SOLVE_ROWS)
def test_fixed_step_solves_and_work_queue(name, cuda_device):
    """Fixed-step sample + log q and sample-only against the fp32 oracle; then one batch of 2 * #SMs + 5 trajectories (every
    CTA takes several trajectories from the work queue, reusing its scratch and tables) made of copies of the oracle's
    trajectories: bit-identical when repeated and between copies, equal to the oracle, and to the fp32 SIMT engine where
    that engine runs the shape."""
    r = ROWS[name]
    ocfg, flat, tree, eng = build(r, head_variance=0.3)
    B = 3
    rng = np.random.default_rng(7)
    x0 = O.base_sample_from_noise(ocfg, torch.tensor(rng.standard_normal((B, r.n * r.dim)), dtype=torch.float32))
    feat = rng.integers(0, r.nfeat, (B, r.n)).astype(np.int32)
    ft = torch.tensor(feat).long()
    p32 = O.to_torch(flat, torch.float32)
    octrl = O.SolveControl(fixed=True, step_size=0.25)
    ctrl = L.make_ctrl(use_fixed_step_size=True, step_size=0.25)
    x1_ref, lq_ref, _ = O.sample_and_log_prob_cnf(p32, ocfg, x0, ft, octrl)
    xs_ref, _ = O.sample_cnf(p32, ocfg, x0, ft, octrl)
    x1_ref, lq_ref, xs_ref = x1_ref.numpy(), lq_ref.numpy(), xs_ref.numpy()
    lq_scale = np.abs(lq_ref).max() + 1

    assert engine_for(eng, L.MODE_SAMPLE_LOGQ) == r.div and engine_for(eng, L.MODE_SAMPLE) == r.sample
    x1, logs, st = _solve_both(eng, tree, L.MODE_SAMPLE_LOGQ, x0.numpy(), feat, ctrl)
    assert (st[:, 2] == 25).all() and (st[:, 3] == 0).all()
    e_x, e_l = rel_err(x1, x1_ref), float(np.abs(logs[:, 0] - lq_ref).max() / lq_scale)
    xs, _, st = _solve_both(eng, tree, L.MODE_SAMPLE, x0.numpy(), feat, ctrl)
    e_s = rel_err(xs, xs_ref)
    print(f"solve {name}: sample_logq x {e_x:.2e} logq {e_l:.2e}; sample {e_s:.2e}")
    assert e_x < SOLVE_TOL and e_l < SOLVE_TOL and e_s < SOLVE_TOL

    nb = 2 * torch.cuda.get_device_properties(0).multi_processor_count + 5
    idx = np.arange(nb) % B
    xb, fb = x0.numpy()[idx], feat[idx]
    a = _solve_both(eng, tree, L.MODE_SAMPLE_LOGQ, xb, fb, ctrl)
    b = _solve_both(eng, tree, L.MODE_SAMPLE_LOGQ, xb, fb, ctrl)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    for k in range(B):            # a trajectory's result does not depend on the CTA or the queue position it ran at
        assert np.array_equal(a[0][idx == k], np.broadcast_to(a[0][k], a[0][idx == k].shape))
        assert np.array_equal(a[1][idx == k], np.broadcast_to(a[1][k], a[1][idx == k].shape))
    assert rel_err(a[0], x1_ref[idx]) < SOLVE_TOL
    assert np.abs(a[1][:, 0] - lq_ref[idx]).max() < SOLVE_TOL * lq_scale
    if r.simt_div == SIMT and r.div == TC:
        try:
            eng.set_engine(1)
            c = _solve_both(eng, tree, L.MODE_SAMPLE_LOGQ, xb, fb, ctrl)
        finally:
            eng.set_engine(0)
        assert rel_err(a[0], c[0]) < SOLVE_TOL
        assert np.abs(a[1][:, 0] - c[1][:, 0]).max() < SOLVE_TOL * (np.abs(c[1][:, 0]).max() + 1)


def _fm_batch(ocfg, B, nfeat, seed):
    rng = np.random.default_rng(seed)
    D = ocfg.D
    x_data = O.remove_mean(torch.tensor(rng.standard_normal((B, D)) * 1.5), ocfg.n_frames, ocfg.dim).float()
    x0 = O.base_sample_from_noise(ocfg, torch.tensor(rng.standard_normal((B, D)))).float()
    t = torch.tensor(rng.uniform(0, 1, B)).float()
    feat = torch.tensor(rng.integers(0, nfeat, (B, ocfg.n_frames)))
    return x_data, x0, t, feat


def _check_grad(eng, ocfg, grad, g_ref, blocks, what, g32=None):
    """Per-tensor error relative to the tensor's max |g| (fp64 reference).  g32: the same gradient from fp32 autograd; a tensor
    may then miss GRAD_TOL by as much as fp32 itself does, up to DEEP_MULT times fp32's own error."""
    g = eng.unpack(grad, to_numpy=True)["params"]
    worst = 0.0
    for path, _ in O.param_layout(ocfg):
        node = g
        for part in path.split("/"):
            node = node[part]
        ref = g_ref[path].numpy()
        parts = path.split("/")
        if parts[1].isdigit() and int(parts[1]) == blocks - 1 and parts[2] in ("phi_h", "Dense_1"):
            # the last block's phi_h and attention do not reach the output (egnn.py:180-190): exact zeros
            assert np.abs(node).max() == 0.0 and np.abs(ref).max() == 0.0, path
            continue
        err = float(np.abs(node - ref).max() / (np.abs(ref).max() + 1e-12))
        worst = max(worst, err)
        bound = GRAD_TOL
        if g32 is not None:
            err32 = float(np.abs(g32[path].numpy().astype(np.float64) - ref).max() / (np.abs(ref).max() + 1e-12))
            bound = max(GRAD_TOL, DEEP_MULT * err32)
        assert err < bound, (what, path, err, bound)
    return worst


@pytest.mark.parametrize("name", TRAIN_ROWS)
def test_fm_loss_grad_matches_autograd(name, cuda_device):
    r = ROWS[name]
    ocfg, flat, tree, eng = build(r)
    B = 7
    x_data, x0, t, feat = _fm_batch(ocfg, B, r.nfeat, 17)
    loss_ref, g_ref = O.fm_loss_and_grad(flat, ocfg, x_data, x0, t, feat, dtype=torch.float64)
    g32 = O.fm_loss_and_grad(flat, ocfg, x_data, x0, t, feat, dtype=torch.float32)[1] if name in DEEP_ROWS else None
    loss, grad = eng.fm_loss_grad(tree, x_data, x0, t, feat.int())
    e_loss = abs(float(loss[0]) - float(loss_ref)) / abs(float(loss_ref))
    worst = _check_grad(eng, ocfg, grad, g_ref, r.blocks, name, g32)
    print(f"train {name}: loss {e_loss:.2e} worst grad {worst:.2e}")
    assert e_loss < LOSS_TOL


def test_fm_tensor_core_gemms_smallest_graph(cuda_device):
    """n = 2, dim 3, U = 128 at B = 4200: M = 8400 edge rows, >= 8192 (the tcgen05 training GEMMs) and not a multiple of 128."""
    r = ROWS["n2_d3_u128"]
    ocfg, flat, tree, eng = build(r)
    B = 4200
    assert B * r.n * (r.n - 1) == 8400
    x_data, x0, t, feat = _fm_batch(ocfg, B, r.nfeat, 19)
    try:
        eng.set_engine(0)
        loss_tc, grad_tc = eng.fm_loss_grad(tree, x_data, x0, t, feat.int())
        loss_tc, grad_tc = float(loss_tc[0]), grad_tc.clone()
        eng.set_engine(1)
        loss_s, grad_s = eng.fm_loss_grad(tree, x_data, x0, t, feat.int())
        loss_s, grad_s = float(loss_s[0]), grad_s.clone()
    finally:
        eng.set_engine(0)
    assert not torch.equal(grad_tc, grad_s)          # the two paths really differ in arithmetic
    loss_ref, g_ref = O.fm_loss_and_grad(flat, ocfg, x_data, x0, t, feat, dtype=torch.float64)
    assert abs(loss_tc - float(loss_ref)) < LOSS_TOL * abs(float(loss_ref))
    assert abs(loss_s - float(loss_ref)) < LOSS_TOL * abs(float(loss_ref))
    w_tc = _check_grad(eng, ocfg, grad_tc, g_ref, r.blocks, "tcgen05")
    w_s = _check_grad(eng, ocfg, grad_s, g_ref, r.blocks, "simt")
    print(f"train n2_d3_u128 B=4200: worst grad tcgen05 {w_tc:.2e} simt {w_s:.2e}")
