"""INT8-slice condensation in column chunks under a bounded slice buffer (hb_ctx_set_oz_workspace_limit): same digits as the
unchunked kernel, the FP64 recombination regrouped at rounding level, bit-identical when the budget holds all columns, and the
AUTO / explicit-mode behaviour when not even one recombination chunk fits."""
import numpy as np
import pytest

from hiop_b200 import synth
from oracle import kkt_oracle as ko

pytestmark = pytest.mark.gpu

TOL_N = {6: 2e-10, 7: 2e-12, 8: 5e-14}      # tests/test_gpu_ozaki.py: int8 slices against the FP64 DMMA kernel
TOL_REGROUP = 1e-14                          # chunked against unchunked, relative to sqrt(N_ii N_jj)


def chunk_cols(S):
    """columns of one int32-safe recombination chunk (hb_ozaki.cu): chunk boundaries are multiples of this"""
    stages = (524288 // S) // 128
    while S * stages * 128 * 4096 >= 2 ** 31:
        stages -= 1
    return stages * 128


def slice_bytes(Ma, S, cols):
    return S * (-(-Ma // 128) * 128) * cols


@pytest.fixture(scope="module")
def ctx():
    from hiop_b200.engine import Context
    c = Context(0)
    yield c
    c.close()


@pytest.fixture
def budget(ctx):
    """sets the context's slice budget for one test and restores AUTO afterwards"""
    yield ctx.set_oz_workspace_limit
    ctx.set_oz_workspace_limit(0)


def _setup(ctx, P, mode):
    from hiop_b200.engine import KKTLinSysLowRank
    k = KKTLinSysLowRank(ctx, P.n, P.m_eq, P.m_ineq, max(P.l, 1))
    D = ctx.to_device
    T = {name: D(getattr(P, name)) for name in ("ixl", "ixu", "idl", "idu", "zl", "sxl", "zu", "sxu", "vl", "sdl", "vu", "sdu", "St", "Yt", "rx", "ryc", "ryd")}
    T["J"] = D(P.J)
    k.set_patterns(T["ixl"], T["ixu"], T["idl"], T["idu"])
    k.set_jacobian(T["J"][:P.m_eq], T["J"][P.m_eq:])
    k.set_secant(P.sigma, T["St"] if P.l else None, T["Yt"] if P.l else None, P.L, P.D)
    k.set_condense_mode(mode)
    k.update(T["zl"], T["sxl"], T["zu"], T["sxu"], T["vl"], T["sdl"], T["vu"], T["sdu"])
    return k, T


def _rel(A, B):
    d = np.abs(np.diag(B)).copy()
    d[d == 0] = 1.0
    return (np.abs(A - B) / np.sqrt(np.outer(d, d))).max()


def _condense(ctx, P, mode, limit, budget):
    budget(limit)
    k, T = _setup(ctx, P, mode)
    k.condense()
    return k, T, k.N(), k.condense_chunks()


@pytest.mark.parametrize("S", [6, 7, 8])
def test_chunked_matches_unchunked_fp64_and_is_deterministic(ctx, budget, S):
    # 3 full chunks + a ragged fourth of 3841 columns (odd n: the 8-byte row path; S = 8 is n = 200001 of the oracle test below)
    n, m, l = 3 * chunk_cols(S) + 3841 if S != 8 else 200001, 300, 6
    P = synth.make_qn_problem(n, m, l, seed=31 + S)
    lim = slice_bytes(m + 2 * l, S, chunk_cols(S))
    k0, _, N0, c0 = _condense(ctx, P, 0, 0, budget)
    k1, _, N1, c1 = _condense(ctx, P, S, 0, budget)
    k2, _, N2, c2 = _condense(ctx, P, S, lim, budget)
    assert (c0, c1, c2) == (0, 1, 4)
    assert _rel(N2, N1) <= TOL_REGROUP, _rel(N2, N1)
    assert _rel(N1, N0) <= TOL_N[S] and _rel(N2, N0) <= TOL_N[S], (_rel(N1, N0), _rel(N2, N0))
    assert np.array_equal(N2, N2.T)
    k2.condense()                                              # same budget again: bit for bit
    assert k2.condense_chunks() == 4
    assert np.array_equal(k2.N(), N2)
    for k in (k0, k1, k2):
        k.close()


def test_budget_that_holds_all_columns_is_bit_identical(ctx, budget):
    n, m, l = 70001, 130, 6
    P = synth.make_qn_problem(n, m, l, seed=3)
    k1, _, N1, c1 = _condense(ctx, P, 8, 0, budget)
    k2, _, N2, c2 = _condense(ctx, P, 8, slice_bytes(m + 2 * l, 8, -(-n // 128) * 128), budget)
    assert c1 == c2 == 1
    assert np.array_equal(N1, N2)
    k1.close()
    k2.close()


def test_chunked_against_oracle_at_scale_adversarial_scaling(ctx, budget):
    """the scaling of tests/test_gpu_ozaki.py::test_oz8_against_oracle_at_scale_adversarial_scaling (DhInv over 16 decades, rows over
    12 decades) with the columns sliced in 4 chunks"""
    n, m, l = 200001, 300, 4
    P = synth.make_qn_problem(n, m, l, seed=4242)
    r = np.random.default_rng(7)
    P.sxl[:] = 10.0 ** r.uniform(-8.0, 0.0, n)
    P.zl[:] = 10.0 ** r.uniform(0.0, 8.0, n)
    rowscale = 10.0 ** (12.0 * np.arange(m) / (m - 1) - 6.0)
    P.Jc *= rowscale[:P.m_eq, None]
    P.Jd *= rowscale[P.m_eq:, None]
    Dx, DhInv, Dd, Dd_inv = ko.kkt_update(P.zl, P.sxl, P.zu, P.sxu, P.ixl, P.ixu, P.vl, P.sdl, P.vu, P.sdu, P.idl, P.idu, P.sigma)
    No, _, _, _ = ko.condense(ko.QnState(P.Jc, P.Jd, DhInv, Dd_inv, P.St, P.Yt, P.L, P.D, P.sigma))
    k, _, Ng, chunks = _condense(ctx, P, 8, slice_bytes(m + 2 * l, 8, chunk_cols(8)), budget)
    assert chunks == 4
    assert _rel(Ng, No) <= 2e-12, _rel(Ng, No)
    k.close()


@pytest.mark.parametrize("n,m,l", [
    (65537, 64, 6),     # 2 chunks, the second 2 stages long: most split items of the last chunk are empty
    (130817, 64, 0),    # odd n, n not a multiple of the chunk width, l = 0
    (140000, 1, 6),     # m = 1
    (140000, 0, 6),     # m = 0: C_aug is the secant block only
    (9000, 40, 3),      # n smaller than one chunk: unchunked under the same budget
    (17, 5, 2),         # n = 17
])
def test_edge_shapes(ctx, budget, n, m, l):
    P = synth.make_qn_problem(n, m, l, seed=n % 1000 + m)
    lim = slice_bytes(max(m + 2 * l, 1), 8, chunk_cols(8))
    want_chunks = -(-(-(-n // 128) * 128) // chunk_cols(8))
    k1, T1, N1, c1 = _condense(ctx, P, 8, 0, budget)
    k2, T2, N2, c2 = _condense(ctx, P, 8, lim, budget)
    assert c1 == 1 and c2 == want_chunks, (c1, c2, want_chunks)
    if m:
        assert np.all(np.isfinite(N2))
        if c2 == 1:
            assert np.array_equal(N1, N2)
        else:
            assert _rel(N2, N1) <= TOL_REGROUP, _rel(N2, N1)
    res = []
    for k, T in ((k1, T1), (k2, T2)):
        dx, dyc, dyd = [ctx.zeros(s) for s in (P.n, P.m_eq, P.m_ineq)]
        assert k.solveCompressed(ctx.to_device(P.rx), T["ryc"], T["ryd"], dx, dyc, dyd)
        ctx.sync()
        res.append([v.cpu().numpy() for v in (dx, dyc, dyd)])
        k.close()
    for a, b in zip(*res):
        if b.size:
            assert np.abs(a - b).max() <= 1e-10 * max(1.0, np.abs(b).max())


def test_fused_rowmax_route_with_chunking(ctx, budget):
    """solveCompressed on a pending condensation takes J (H+Dx)^-1 rx from the row-maximum sweep over all columns; with the slices in
    chunks it must still give the direction of the two-pass route"""
    n, m, l = 200001, 120, 4
    P = synth.make_qn_problem(n, m, l, seed=17)
    budget(slice_bytes(m + 2 * l, 8, chunk_cols(8)))
    res = {}
    for fused in (True, False):
        k, T = _setup(ctx, P, 8)
        if not fused:
            k.condense()
        dx, dyc, dyd = [ctx.zeros(s) for s in (P.n, P.m_eq, P.m_ineq)]
        assert k.solveCompressed(ctx.to_device(P.rx), T["ryc"], T["ryd"], dx, dyc, dyd)
        k.check()
        ctx.sync()
        assert k.condense_mode_used() == 8 and k.condense_chunks() == 4
        res[fused] = [v.cpu().numpy().copy() for v in (dx, dyc, dyd)]
        k.close()
    for a, b in zip(res[True], res[False]):
        assert np.abs(a - b).max() <= 1e-10 * max(1.0, np.abs(b).max())


def test_budget_fallbacks(ctx, budget):
    n, m, l = 140000, 90, 4
    P = synth.make_qn_problem(n, m, l, seed=23)
    one = slice_bytes(m + 2 * l, 8, chunk_cols(8))
    # AUTO with a budget of one recombination chunk: still the int8 kernel, chunked, no fallback
    k, _, _, chunks = _condense(ctx, P, -1, one, budget)
    assert (k.condense_mode_used(), k.fallback_count(), chunks) == (8, 0, 3)
    k.close()
    # below one recombination chunk: AUTO redoes the condensation with the FP64 kernel and counts it
    k, _, N, chunks = _condense(ctx, P, -1, one - 1, budget)
    assert (k.condense_mode_used(), k.fallback_count(), chunks) == (0, 1, 0)
    k0, _, N0, _ = _condense(ctx, P, 0, 0, budget)
    assert _rel(N, N0) <= 1e-15
    k.close()
    k0.close()
    # an explicit int8 mode reports the allocation failure
    from hiop_b200._lib import EngineError
    budget(one - 1)
    k, _ = _setup(ctx, P, 8)
    with pytest.raises(EngineError, match=r"code -3"):
        k.condense()
    k.close()


def test_lsq_duals_with_chunking(ctx, budget):
    n, m = 200001, 100
    P = synth.make_qn_problem(n, m, 0, seed=41)
    D = ctx.to_device
    r = np.random.default_rng(5)
    g, zl, zu = D(r.standard_normal(n)), D(P.zl), D(P.zu)
    vl, vu = D(P.vl), D(P.vu)
    out = []
    for lim in (0, slice_bytes(m, 8, chunk_cols(8))):
        budget(lim)
        k, T = _setup(ctx, P, 8)
        yc, yd = ctx.zeros(P.m_eq), ctx.zeros(P.m_ineq)
        assert k.lsq_duals(g, zl, zu, vl, vu, yc, yd)
        ctx.sync()
        out.append(np.concatenate([yc.cpu().numpy(), yd.cpu().numpy()]))
        k.close()
    assert np.abs(out[1] - out[0]).max() <= 1e-12 * np.abs(out[0]).max()


def test_kkt_residual_with_independent_operators(ctx, budget):
    """through solveCompressed with 4 chunks: the compressed KKT residual evaluated with torch FP64 operators that never see N"""
    import torch
    import bench
    n, m, l = 200001, 300, 6
    from hiop_b200.engine import KKTLinSysLowRank
    budget(slice_bytes(m + 2 * l, 8, chunk_cols(8)))
    with ctx:                                                  # torch work on the engine stream (ordered with its kernels)
        T = bench.make_device_problem(ctx, torch, n, n, m, l, 0, 1, None)
        k = KKTLinSysLowRank(ctx, n, T["m_eq"], T["m_ineq"], l)
        k.set_patterns(T["ixl"], T["ixu"], T["idl"], T["idu"])
        k.set_jacobian(T["J"][:T["m_eq"]], T["J"][T["m_eq"]:])
        k.set_secant(1.0, T["St"], T["Yt"], T["L"], T["D"])
        k.update(T["zl"], T["sxl"], T["zu"], T["sxu"], T["vl"], T["sdl"], T["vu"], T["sdu"])
        dx, dyc, dyd = ctx.zeros(n), ctx.zeros(T["m_eq"]), ctx.zeros(T["m_ineq"])
        assert k.solveCompressed(T["rx"].clone(), T["ryc"], T["ryd"], dx, dyc, dyd)
        k.check()
        ctx.sync()
        assert k.condense_mode_used() == 8 and k.condense_chunks() == 4
        resid = bench.independent_kkt_residual(torch, None, 1, T, 1.0, dx, dyc, dyd)
    assert resid <= 1e-8, resid
    k.close()
