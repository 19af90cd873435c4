"""The configuration sweep of tests/test_gpu_config_sweep.py covers what it claims, checked on the host (no GPU): every row
runs on the engine it names (ecnf_solve_engine_for), and the rows together reach each structure of the tensor-core engine
(tile headers from ecnf_solve_tc_tile_table) and each eligibility limit.  If the eligibility rules or the tile packing
change, this test names the coverage property that no row has any more."""
import pytest

from ecnf_b200 import lib as L
from ecnf_b200.engine import CnfConfig, Engine
from test_gpu_config_sweep import SIMT, SWEEP, TC, UNSUPPORTED, build, engine_for
from test_tc_tiles_host import FIRST, LAST, MID, EDGE1, NODE1, MR, P, WIN_I, WIN_NR, WIN_NS, table


def engines(r):
    return build(r)[3]


@pytest.mark.parametrize("r", SWEEP, ids=[r.name for r in SWEEP])
def test_row_runs_on_the_engine_it_names(r):
    eng = engines(r)
    for engine in (0, 1):
        eng.set_engine(engine)
        div, sample = (r.div, r.sample) if engine == 0 else (r.simt_div, SIMT)
        for mode in (L.MODE_VF_DIV, L.MODE_SAMPLE_LOGQ, L.MODE_LOGPROB):
            got = engine_for(eng, mode)
            if isinstance(div, str):
                assert got == UNSUPPORTED and div in eng.lib.ecnf_last_error().decode(), (engine, mode)
            else:
                assert got == div, (engine, mode)
        for mode in (L.MODE_VF, L.MODE_SAMPLE):
            assert engine_for(eng, mode) == sample, (engine, mode)
    eng.set_engine(0)
    # the flop count (roofline reports) and the tile tables exist exactly when exact-trace calls run on the tensor cores
    assert (eng.lib.ecnf_solve_tensor_flops_per_eval(eng.handle) > 0) == (r.div == TC)
    assert (eng.lib.ecnf_solve_tc_tile_table(eng.handle, MID, None, 0) > 0) == (r.div == TC)


def test_engine_query_rejects_bad_arguments():
    eng = Engine(CnfConfig(4, 2, 0.01, 1.0, 1, (128,), 64, 8, 1))
    assert eng.lib.ecnf_solve_engine_for(None, L.MODE_VF) == -1
    assert eng.lib.ecnf_solve_engine_for(eng.handle, 5) == -1
    assert eng.lib.ecnf_solve_engine_for(eng.handle, -1) == -1


def _tc_rows():
    """(row, {kind: tiles}) of every row whose exact-trace calls run on the tensor cores."""
    out = []
    for r in SWEEP:
        if r.div != TC:
            continue
        eng = engines(r)
        out.append((r, {k: table(eng, k) for k in (NODE1, FIRST, MID, LAST, EDGE1)}))
    return out


def test_sweep_reaches_every_tensor_core_structure():
    rows = _tc_rows()
    have = set()
    for r, tabs in rows:
        D, sub = r.n * r.dim, 128 // r.U
        mid = tabs[MID][:, 32:]
        if ((mid[:, WIN_NR] == 1) & (mid[:, WIN_NS] < 1 + D)).any():
            have.add(("mid slot window", r.U))
        if (mid[:, MR] == 8).all():
            have.add(("MR = 8", r.U))
        if len(set(tabs[FIRST][:, 32 + WIN_I].tolist())) > 1:
            have.add(("first-block table with several windows", r.U))
        for k in (FIRST, MID, LAST, EDGE1):
            p = tabs[k][:, 32 + P]
            if (p == 16 * sub).any():
                have.add(("full edge tile", r.U))
            if (p < 16 * sub).any():
                have.add(("partial edge tile", r.U))
        for k, groups in ((NODE1, r.n), (EDGE1, r.n * (r.n - 1))):
            have.add(("dense groups multiple of 8" if groups % 8 == 0 else "dense groups not multiple of 8", r.U))
        if r.L in (1, 6):
            have.add((f"L = {r.L}", r.U))
        if r.blocks in (1, 8):
            have.add((f"{r.blocks} blocks", r.U))
        if r.blocks * (3 * r.L + 3) > 64:
            have.add(("more than 64 weight images", r.U))
    want = {(p, U) for U in (128, 64) for p in (
        "mid slot window", "MR = 8", "first-block table with several windows", "full edge tile", "partial edge tile",
        "dense groups multiple of 8", "dense groups not multiple of 8", "L = 1", "L = 6", "1 blocks", "8 blocks",
        "more than 64 weight images")}
    assert want <= have, sorted(want - have)


def _limit(U, H, dim, mode):
    """Last n (default depth) that runs on the tensor cores in `mode`."""
    last = None
    for n in range(2, 33):
        eng = Engine(CnfConfig(n, dim, 0.01, 1.0, 2, (U,) * 2, H, 8, 1))
        if engine_for(eng, mode) == TC:
            last = n
    return last


@pytest.mark.parametrize("U,H", [(128, 64), (64, 32)])
@pytest.mark.parametrize("dim", [2, 3])
def test_sweep_straddles_every_eligibility_limit(U, H, dim):
    """For each (U, dim), exact trace and sample-only: the last shape on the tensor cores and the first one past it are rows of
    the sweep (unless the last one is n = 32, the largest graph accepted)."""
    by_shape = {(r.U, r.dim, r.n): r for r in SWEEP if (r.blocks, r.L, r.T, r.nfeat, r.nc) == (2, 2, 8, 1, 1.0)}
    for mode, col in ((L.MODE_VF_DIV, "div"), (L.MODE_SAMPLE, "sample")):
        last = _limit(U, H, dim, mode)
        assert last is not None
        assert (U, dim, last) in by_shape, (col, last)
        assert getattr(by_shape[(U, dim, last)], col) == TC
        if last < 32:
            assert (U, dim, last + 1) in by_shape, (col, last + 1)
            assert getattr(by_shape[(U, dim, last + 1)], col) != TC
