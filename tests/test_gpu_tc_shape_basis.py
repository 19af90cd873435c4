"""Shape-space tangents of the tensor-core exact trace on the GPU (DESIGN 3.1): VF_DIV against the fp64 oracle and the
fp32 SIMT engine, including inputs whose rotations are degenerate (the canonical path), and fixed-step
sample_and_log_prob against the oracle."""
import numpy as np
import pytest
import torch

from oracle import ecnf_oracle as O
from ecnf_b200 import lib as L
from helpers import make_pair, rel_err

pytestmark = pytest.mark.gpu

VF_TOL = 2e-5     # relative to max |f|            (test_gpu_config_sweep.py)
DIV_TOL = 5e-5    # relative to max |div| + 1
SOLVE_TOL = 1e-4

CASES = {   # name: n, dim, blocks, units, H, n_features
    "lj13": (13, 3, 3, (128, 128, 128), 64, 1),
    "dw4": (4, 2, 3, (128, 128, 128), 64, 1),
    "aldp": (22, 3, 3, (64, 64), 32, 22),
    "small_64_32": (5, 3, 3, (64, 64), 32, 3),
    "b8_128": (5, 3, 8, (128, 128), 64, 1),
    "b6_lj13": (13, 3, 6, (128, 128, 128), 64, 1),   # four middle blocks on the shape-space path
    "b8_64": (6, 2, 8, (64, 64), 32, 1),
    "n2_d3": (2, 3, 3, (128, 128), 64, 1),       # s = 0: every evaluation on the canonical path
}


def div_err(a, ref):
    a, ref = np.asarray(a, np.float64), np.asarray(ref, np.float64)
    return float(np.abs(a - ref).max() / (np.abs(ref).max() + 1.0))


def inputs(name, B, kind, seed=5):
    n, dim = CASES[name][:2]
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, n * dim)) * 1.3 + 0.2
    if kind == "collinear":          # rows 0, 1: all particles on a line (row 1: nearly, below the rank threshold)
        d = np.array([0.3, -0.5, 0.8][:dim])
        for b in range(min(B, 2)):
            X = np.outer(rng.standard_normal(n), d) + rng.standard_normal(dim)
            if b == 1:
                X += 1e-3 * rng.standard_normal((n, dim))
            x[b] = X.reshape(-1)
    return x.astype(np.float32), rng.uniform(0, 1, B).astype(np.float32), rng.integers(0, CASES[name][5], (B, n)).astype(np.int32)


@pytest.mark.parametrize("name,kind", [(k, "generic") for k in CASES] + [("lj13", "collinear"), ("dw4", "collinear"),
                                                                         ("aldp", "collinear")])
def test_vf_div_matches_oracle_and_simt(name, kind, cuda_device):
    n, dim, blocks, units, H, nf = CASES[name]
    ocfg, flat, tree, ecfg = make_pair(n, dim, blocks, units, H, n_features=nf)
    from ecnf_b200.engine import Engine
    eng = Engine(ecfg)
    assert eng.lib.ecnf_solve_engine_for(eng.handle, L.MODE_VF_DIV) == 0
    x, t, feat = inputs(name, 4, kind)
    p64 = O.to_torch(flat, torch.float64)
    f_ref, div_ref = O.vf_and_exact_div(p64, ocfg, torch.tensor(x, dtype=torch.float64),
                                        torch.tensor(t, dtype=torch.float64), torch.tensor(feat).long())
    f_ref, div_ref = f_ref.numpy(), div_ref.numpy()
    f, d = eng.apply_div(tree, x, t, feat)
    f, d = f.cpu().numpy(), d.cpu().numpy()
    e_f, e_d = rel_err(f, f_ref), div_err(d, div_ref)
    msg = f"{name} {kind}: tcgen05 vf {e_f:.2e} div {e_d:.2e}"
    assert e_f < VF_TOL and e_d < DIV_TOL, msg
    try:
        eng.set_engine(1)
        if eng.lib.ecnf_solve_engine_for(eng.handle, L.MODE_VF_DIV) == 1:
            f1, d1 = eng.apply_div(tree, x, t, feat)
            e_s = div_err(d, d1.cpu().numpy())
            msg += f"; against SIMT div {e_s:.2e}"
            assert rel_err(f, f1.cpu().numpy()) < 2 * VF_TOL and e_s < 2 * DIV_TOL, msg
    finally:
        eng.set_engine(0)
    print(msg)


@pytest.mark.parametrize("name", ["lj13", "aldp"])
def test_fixed_step_sample_and_log_prob(name, cuda_device):
    n, dim, blocks, units, H, nf = CASES[name]
    ocfg, flat, tree, ecfg = make_pair(n, dim, blocks, units, H, n_features=nf, head_variance=0.3)
    from ecnf_b200.engine import Engine
    eng = Engine(ecfg)
    B = 2
    rng = np.random.default_rng(11)
    x0 = O.base_sample_from_noise(ocfg, torch.tensor(rng.standard_normal((B, n * dim)), dtype=torch.float32))
    feat = rng.integers(0, nf, (B, n)).astype(np.int32)
    octrl = O.SolveControl(fixed=True, step_size=0.25)
    x1_ref, lq_ref, _ = O.sample_and_log_prob_cnf(O.to_torch(flat, torch.float32), ocfg, x0, torch.tensor(feat).long(), octrl)
    x1, logs, st = eng.solve(tree, L.MODE_SAMPLE_LOGQ, x0.numpy(), feat, L.make_ctrl(use_fixed_step_size=True, step_size=0.25))
    x1, lq = x1.cpu().numpy(), logs.cpu().numpy()[:, 0]
    e_x = rel_err(x1, x1_ref.numpy())
    e_l = float(np.abs(lq - lq_ref.numpy()).max() / (np.abs(lq_ref.numpy()).max() + 1))
    print(f"{name}: sample_and_log_prob x {e_x:.2e} log q {e_l:.2e}")
    assert e_x < SOLVE_TOL and e_l < SOLVE_TOL
