"""Shape-space tangents of the tensor-core exact trace (DESIGN 3.1), no GPU needed.

The middle EGNN blocks carry only the s = D - dim - dim(dim-1)/2 centred directions Q_S orthogonal to the rotations
A_j x of the evaluation's input; the canonical directions P e_d are rebuilt before the last block from
    J P e_d = sum_k Q_S[d,k] J q_k + sum_j W[d,j] A_j f(x),   W = Q_R R_r^-T,  [A_j x] = Q_R R_r,
which holds because the vector field is rotation-equivariant (J A_j x = A_j f(x) for a centred x).  An input whose
rotations are (nearly) degenerate takes the canonical path.  Here: the identity on the fp64 oracle with the basis built
the way the kernel builds it, the rank test, and the invariants of the reduced tile tables (kind + 16 of
ecnf_solve_tc_tile_table)."""
import numpy as np
import pytest
import torch

from oracle import ecnf_oracle as O
from ecnf_b200.engine import CnfConfig, Engine
from test_tc_tiles_host import (FIRST, FLUSH, GRPEND, LAST, MID, N, NCH, NODE, NODE1, OWNER, P, RUNEND, SHAPES, VALID,
                                WIN_I, WIN_NR, WIN_NS, WIN_S, IFIRST, ILAST, MR, table, word_index)

MIN_SIGMA = 0.05     # EngineTC::TC_SHAPE_MIN_SIGMA: smallest singular value of [A_j x] relative to |x|
SHAPE = 16           # kind offset of the shape-space tables


def generators(dim):
    return [(p, q) for p in range(dim) for q in range(p + 1, dim)]


def rot(x, n, dim, p, q):
    """A_j x for the generator of the plane (p, q): (A x)_p = x_q, (A x)_q = -x_p per particle."""
    X = np.asarray(x, np.float64).reshape(n, dim)
    Y = np.zeros_like(X)
    Y[:, p], Y[:, q] = X[:, q], -X[:, p]
    return Y.reshape(-1)


def shape_basis(x, n, dim):
    """(Q_S, W, on the shape-space path) from the QR of [translations | A_j x], like EngineTC::shape_basis."""
    D, gens = n * dim, generators(dim)
    r, c = len(gens), dim + len(gens)
    T = np.zeros((D, dim))
    for a in range(dim):
        T[a::dim, a] = 1 / np.sqrt(n)
    R = np.stack([rot(x, n, dim, p, q) for p, q in gens], 1) if r else np.zeros((D, 0))
    Q, Rf = np.linalg.qr(np.concatenate([T, R], 1), mode="complete")
    QR_, QS = Q[:, dim:c], Q[:, c:]
    Rr = Rf[dim:c, dim:c]
    x2 = float(np.dot(x, x))
    lmin = np.linalg.eigvalsh(Rr.T @ Rr).min() if r else np.inf
    ok = D - c >= 1 and x2 > 0 and lmin > MIN_SIGMA ** 2 * x2
    W = QR_ @ np.linalg.inv(Rr).T if ok and r else np.zeros((D, r))
    return QS, W, ok


def sigma_ratio(x, n, dim):
    R = np.stack([rot(x, n, dim, p, q) for p, q in generators(dim)], 1)
    return np.linalg.svd(R, compute_uv=False).min() / np.linalg.norm(x)


MODELS = {   # name: n, dim, blocks, units, H, n_features
    "lj13": (13, 3, 3, (128, 128, 128), 64, 1),
    "dw4": (4, 2, 3, (128, 128, 128), 64, 1),
    "aldp": (22, 3, 3, (64, 64), 32, 22),
}


def model(name):
    n, dim, blocks, units, H, nf = MODELS[name]
    ocfg = O.CnfConfig(n_frames=n, dim=dim, n_blocks_egnn=blocks, mlp_units=units, n_invariant_feat_hidden=H,
                       n_features=nf)
    p = O.to_torch(O.init_params(ocfg, seed=0, head_variance=1.0), torch.float64)
    return ocfg, p


def centred(x, n, dim):
    X = np.asarray(x, np.float64).reshape(n, dim)
    return (X - X.mean(0)).reshape(-1)


def check_identity(name, x):
    """trace(J) from the s shape directions plus the rotation part, against the full fp64 Jacobian."""
    ocfg, p = model(name)
    n, dim = ocfg.n_frames, ocfg.dim
    D = n * dim
    QS, W, ok = shape_basis(x, n, dim)
    assert ok and QS.shape == (D, D - dim - dim * (dim - 1) // 2)
    t = torch.tensor([0.37], dtype=torch.float64)
    feat = (torch.arange(n) % ocfg.n_features)[None]
    f = lambda z: O.egnn_apply(p, ocfg, z[None], t, feat)[0]
    xt = torch.tensor(x)
    J = torch.autograd.functional.jacobian(f, xt).numpy()
    fx = f(xt).detach().numpy()
    fs = float(p["EGNN_0/final_scaling"])
    AF = np.stack([rot(fx, n, dim, pp, q) for pp, q in generators(dim)], 1)      # J A_j x = A_j f(x)
    JP = (J @ QS) @ QS.T + AF @ W.T                                             # columns J P e_d, rebuilt
    Pc = np.eye(D) - np.kron(np.ones((n, n)) / n, np.eye(dim))
    assert np.abs(JP - J @ Pc).max() <= 1e-12 * np.abs(J).max()
    tr, tr_red = np.trace(J), np.trace(JP) - fs * dim                           # J (I - P) = -fs (I - P)
    assert abs(tr_red - tr) <= 1e-12 * abs(tr), (name, tr, tr_red)
    return tr


@pytest.mark.parametrize("name", list(MODELS))
def test_trace_identity_on_oracle(name):
    n, dim = MODELS[name][:2]
    x = centred(np.random.default_rng(0).standard_normal(n * dim), n, dim)
    assert sigma_ratio(x, n, dim) > 0.3       # a generic state is far from the fallback
    check_identity(name, x)


def near_collinear(n, dim, ratio, seed=1):
    """A centred LJ13-like state on a line plus a perpendicular spread scaled so that sigma_min / |x| = ratio."""
    rng = np.random.default_rng(seed)
    line = np.outer(rng.standard_normal(n), np.eye(dim)[0])
    perp = rng.standard_normal((n, dim))
    perp[:, 0] = 0
    make = lambda a: centred(line + a * perp, n, dim)
    lo, hi = 0.0, 1.0
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if sigma_ratio(make(mid), n, dim) < ratio else (lo, mid)
    return make(hi)


def test_trace_identity_near_collinear():
    x = near_collinear(13, 3, 1.02 * MIN_SIGMA)
    assert MIN_SIGMA < sigma_ratio(x, 13, 3) < 1.05 * MIN_SIGMA
    check_identity("lj13", x)


def test_rank_test_takes_the_canonical_path():
    assert not shape_basis(near_collinear(13, 3, 0.98 * MIN_SIGMA), 13, 3)[2]
    line = centred(np.outer(np.arange(13.0), [0.3, -0.2, 0.9]), 13, 3)          # collinear
    assert not shape_basis(line, 13, 3)[2]
    assert not shape_basis(centred([0.1, 0.2, 0.3, -0.4, 0.5, 0.6], 2, 3), 2, 3)[2]   # n = 2 in 3-D: s = 0
    assert not shape_basis(np.zeros(12), 6, 2)[2]                               # coincident particles
    # 2-D: one generator with sigma = |x|, so any non-degenerate state is on the shape-space path
    assert shape_basis(centred(np.random.default_rng(3).standard_normal(8), 4, 2), 4, 2)[2]


def check_tiles(tab, SUB, r, ngroups, nb, kind):
    """The invariants test_tc_tiles_host.py checks for NODE / MID tables with r rows per group."""
    seen, owners = set(), set()
    for t in tab:
        h = t[32:48].astype(np.int64)
        npch = int(h[P])
        assert 1 <= npch <= 16 * SUB
        used = {word_index(p, SUB) for p in range(npch)}
        for wi in range(32):
            assert bool(t[wi] & VALID) == (wi in used)
        for sb in range(SUB):
            for hh in range(2):
                assert h[NCH + sb * 2 + hh] == sum(1 for p in range(npch) if p % SUB == sb and (p // SUB) % 2 == hh)
        n0 = max(h[NCH + sb * 2] for sb in range(SUB))
        n1 = max(h[NCH + sb * 2 + 1] for sb in range(SUB))
        assert h[N] % 16 == 0 and 16 <= h[N] <= 128 and h[N] >= (64 + 8 * n1 if n1 else 8 * n0)
        run_key, run_open = None, False
        for p in range(npch):
            w = int(t[word_index(p, SUB)])
            gid, qb, cnt = w & 1023, (w >> 10) & 255, (w >> 18) & 15
            assert qb >= 1 and (qb - 1) % 7 == 0 and cnt == 1 + min(7, r - qb)
            assert bool(w & OWNER) == (qb == 1)
            if w & OWNER:
                assert gid not in owners
                owners.add(gid)
                seen.add((gid, 0))
            for u in range(1, cnt):
                assert (gid, qb + u - 1) not in seen
                seen.add((gid, qb + u - 1))
            key = (gid // nb, qb) if kind == MID else (gid, qb)
            if run_open:
                assert key == run_key
            run_key, run_open = key, not (w & RUNEND)
        assert not run_open
        start = 0
        for p in range(npch):
            if int(t[word_index(p, SUB)]) & RUNEND:
                for q in range(start, p + 1):
                    assert bool(int(t[word_index(q, SUB)]) & GRPEND) == (q + 2 * SUB > p)
                start = p + 1
        if kind == MID:
            assert h[WIN_NR] * h[WIN_NS] <= h[MR] and 8 <= h[MR]
            assert h[WIN_I] <= h[IFIRST] <= h[ILAST] < h[WIN_I] + h[WIN_NR]
            for p in range(npch):
                w = int(t[word_index(p, SUB)])
                qb, cnt = (w >> 10) & 255, (w >> 18) & 15
                assert h[WIN_S] <= (0 if (w & OWNER) else qb) and qb + cnt - 2 < h[WIN_S] + h[WIN_NS]
    assert len(seen) == ngroups * r and len(owners) == ngroups
    if kind == MID:
        assert tab[-1][32 + FLUSH] == 1


@pytest.mark.parametrize("n,dim,U,H", SHAPES)
def test_shape_tables(n, dim, U, H):
    eng = Engine(CnfConfig(n, dim, 0.01, 1.0, 3, (U,) * 2, H, 8, 1))
    s = n * dim - dim - dim * (dim - 1) // 2
    for kind in (NODE, MID):
        tab = table(eng, kind + SHAPE)
        assert len(tab) > 0
        check_tiles(tab, 128 // U, 1 + s, n if kind == NODE else n * (n - 1), n - 1, kind)
        # the same window size as the canonical tables (one message accumulator for both)
        assert all(t[32 + MR] == table(eng, kind)[0][32 + MR] for t in tab)
    for kind in (NODE1, FIRST, LAST):
        assert eng.lib.ecnf_solve_tc_tile_table(eng.handle, kind + SHAPE, None, 0) == 0
    # two blocks: no middle block, no shape-space tables
    eng2 = Engine(CnfConfig(n, dim, 0.01, 1.0, 2, (U,) * 2, H, 8, 1))
    assert eng2.lib.ecnf_solve_tc_tile_table(eng2.handle, MID + SHAPE, None, 0) == 0


@pytest.mark.parametrize("name,mid_tiles,mid_s_tiles", [("lj13", 65, 52), ("aldp", 154, 132), ("dw4", 2, 1)])
def test_flagship_tiles_and_flop_count(name, mid_tiles, mid_s_tiles):
    """The middle blocks run fewer tiles, and the tensor-core FLOP count is that of the kinds the kernel runs: the
    shape-space kinds on the (128, 64) network where they save at least 8 middle-block tiles (LJ13), else the canonical
    ones (ALDP: the (64, 32) network; DW4: one tile saved)."""
    n, dim, blocks, units, H, nf = MODELS[name]
    L = len(units)
    eng = Engine(CnfConfig(n, dim, 0.01, 1.0, blocks, units, H, 8, nf))
    assert len(table(eng, MID)) == mid_tiles and len(table(eng, MID + SHAPE)) == mid_s_tiles
    sumN = lambda kind: int(sum(t[32 + N] for t in table(eng, kind)))
    layer = lambda cols, K: 3 * 2 * 128 * cols * K
    SUB = 128 // units[0]
    want = 0
    for b in range(blocks):
        last, mid = b == blocks - 1, 0 < b < blocks - 1 and units[0] == 128 and mid_tiles - mid_s_tiles >= 8
        node = NODE + SHAPE if mid else NODE
        want += (1 if last else 2) * layer(sumN(node if b > 0 else NODE1), SUB * H)
        want += 2 * L * layer(sumN(LAST if last else FIRST if b == 0 else MID + SHAPE if mid else MID), 128)
        if not last:
            want += (L + 1) * layer(sumN(node), 128)
    assert eng.lib.ecnf_solve_tensor_flops_per_eval(eng.handle) == want
