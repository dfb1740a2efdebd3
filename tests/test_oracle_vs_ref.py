"""Pins the numpy/C restatement (oracle/kkt_oracle.py) against the UNMODIFIED reference.
What the reference returned for every case below is stored in tests/golden/oracle_vs_ref.npz, so these tests need neither the
reference's sources nor its compiled library. `python tests/golden/make_golden.py` rewrites that file: it runs this module with
HB_RECORD_REFERENCE=1 against the reference compiled into oracle/_ref (oracle/Makefile), which calls the reference wherever the
tests otherwise read the stored outputs.

To keep the file small, an output the test compares bit for bit is stored as the SHA-256 of its values, and an output longer than
SAMPLE entries that the test compares within a tolerance is stored as SAMPLE entries at fixed, seeded positions together with the
largest magnitude of the whole output (the scale of the tolerance and, being NaN or inf otherwise, proof that all of it is finite)."""
import hashlib
import json
import os

import numpy as np
import pytest

from hiop_b200 import synth
from oracle import kkt_oracle as ko
from oracle import ref

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_vs_ref.npz")
RECORD = os.environ.get("HB_RECORD_REFERENCE") == "1"
SAMPLE = 512
_recorded = {}
_stored = {}


def _positions(size):
    return np.sort(np.random.default_rng(size).choice(size, SAMPLE, replace=False))


def _sha256(a):
    a = np.ascontiguousarray(a, dtype=np.float64) + 0.0          # -0.0 -> 0.0: equal, as for np.testing.assert_array_equal
    return np.frombuffer(hashlib.sha256(repr(a.shape).encode() + a.tobytes()).digest(), dtype=np.uint8)


def _shrink(out, exact):
    stored = {}
    for k, v in out.items():
        v = np.asarray(v)
        if k in exact:
            stored[k + "#sha256"] = _sha256(v)
        elif v.size > SAMPLE:
            stored[k] = v.reshape(-1)[_positions(v.size)]
            stored[k + "#absmax"] = np.abs(v).max()
        else:
            stored[k] = v
    return stored


def _save(entries):
    """One float64 array of all values (digests and counts are exact in float64) and a JSON index of offset, shape and dtype per
    entry; an entry equal to an earlier one (the sigma rules share their secant pairs) points at the earlier one's values."""
    chunks, index, offsets, size = [], {}, {}, 0
    for k, v in entries.items():
        flat = v.astype(np.float64).reshape(-1)
        if flat.tobytes() not in offsets:
            offsets[flat.tobytes()] = size
            chunks.append(flat)
            size += flat.size
        index[k] = [offsets[flat.tobytes()], list(v.shape), v.dtype.str]
    np.savez_compressed(GOLDEN, values=np.concatenate(chunks), index=np.array(json.dumps(index)))


def _load():
    with np.load(GOLDEN) as z:
        values, index = z["values"], json.loads(str(z["index"]))
    return {k: values[at:at + int(np.prod(shape))].reshape(shape).astype(dtype) for k, (at, shape, dtype) in index.items()}


class Reference:
    """The stored outputs of the reference for one call: r[k] is output k, or its sample when k is longer than SAMPLE."""

    def __init__(self, stored):
        self.stored = stored

    def __getitem__(self, k):
        return self.stored[k]

    def pick(self, k, a):
        """The entries of `a`, shaped like output k, at the positions stored for k."""
        a = np.asarray(a)
        return a.reshape(-1)[_positions(a.size)] if a.size > SAMPLE else a

    def absmax(self, k):
        """max |output k| over all its entries (0 when empty)."""
        return float(self.stored[k + "#absmax"] if k + "#absmax" in self.stored else np.abs(self.stored[k]).max(initial=0.0))

    def assert_same(self, k, a):
        np.testing.assert_array_equal(_sha256(a), self.stored[k + "#sha256"], err_msg=f"{k} differs from the reference's")


@pytest.fixture(scope="module", autouse=True)
def _golden_file():
    if not RECORD:
        _stored.update(_load())
    yield
    if RECORD:
        _save(_recorded)


@pytest.fixture
def reference(request):
    """reference(run, exact=()) -> Reference of what `run` computes through the compiled reference for this test case: the stored
    outputs, or (recording) run() itself. Outputs named in `exact` are compared bit for bit. Each call of one test case is a
    separate entry."""
    calls = []

    def get(run, exact=()):
        prefix = f"{request.node.name}/{len(calls)}/"
        calls.append(prefix)
        if RECORD:
            _recorded.update({prefix + k: v for k, v in _shrink(run(), exact).items()})
        out = {k[len(prefix):]: v for k, v in (_recorded if RECORD else _stored).items() if k.startswith(prefix)}
        assert out, f"{GOLDEN} holds no reference outputs for {prefix}: regenerate it with tests/golden/make_golden.py"
        return Reference(out)
    return get


def _ref_system(p):
    q = ref.RefQn(p.n, p.m_eq, p.m_ineq, max(p.l, 1), p.ixl, p.ixu, p.idl, p.idu)
    q.set_iterate(p.sxl, p.sxu, p.zl, p.zu, p.sdl, p.sdu, p.vl, p.vu)
    q.set_jac(p.Jc, p.Jd)
    q.set_secant(p.sigma, p.St, p.Yt, p.L, p.D)
    return q


def _oracle_state(p):
    Dx, DhInv, Dd, Dd_inv = ko.kkt_update(p.zl, p.sxl, p.zu, p.sxu, p.ixl, p.ixu, p.vl, p.sdl, p.vu, p.sdu, p.idl,
                                          p.idu, p.sigma)
    return Dx, ko.QnState(p.Jc, p.Jd, DhInv, Dd_inv, p.St, p.Yt, p.L, p.D, p.sigma)


@pytest.mark.parametrize("n,m,l,mz", [(500, 4, 6, False), (2000, 50, 6, True), (1000, 1, 3, False),
                                       (3000, 64, 0, False), (777, 33, 2, True)])
def test_qn_system_matches_reference(n, m, l, mz, reference):
    p = synth.make_qn_problem(n, m, l, masked_zero_divisors=mz)

    def run():
        q = _ref_system(p)
        out = dict(zip(("Dx", "DhInv", "Ddinv"), q.update()))
        out["N"] = q.condense()
        out["hs"] = q.hess_solve(p.rx)
        out.update(zip(("dx", "dyc", "dyd"), q.solve_compressed(p.rx, p.ryc, p.ryd)))
        q.close()
        return out
    r = reference(run, exact=("Dx", "DhInv", "Ddinv"))
    Dx, st = _oracle_state(p)
    r.assert_same("Dx", Dx)
    r.assert_same("DhInv", st.DhInv)
    r.assert_same("Ddinv", st.Dd_inv)
    N, W0, S1, Y1 = ko.condense(st)
    scale = r.absmax("N")
    assert np.abs(r.pick("N", N) - r["N"]).max() <= 1e-12 * scale
    hs = ko.hess_solve(st, p.rx)
    assert np.abs(r.pick("hs", hs) - r["hs"]).max() <= 1e-11 * r.absmax("hs")
    dx, dyc, dyd, _ = ko.solve_compressed(st, p.rx, p.ryc, p.ryd)
    for k, a in (("dx", dx), ("dyc", dyc), ("dyd", dyd)):
        if r[k].size:
            assert np.abs(r.pick(k, a) - r[k]).max() <= 1e-8 * max(1.0, r.absmax(k))


def test_compute_directions_matches_reference(reference):
    p = synth.make_qn_problem(1500, 20, 4, masked_zero_divisors=True)

    def run():
        q = _ref_system(p)
        q.update()
        d = q.compute_directions(p.res)
        q.close()
        return d
    d_r = reference(run)
    _, st = _oracle_state(p)
    it = dict(sxl=p.sxl, sxu=p.sxu, zl=p.zl, zu=p.zu, sdl=p.sdl, sdu=p.sdu, vl=p.vl, vu=p.vu)
    pat = dict(ixl=p.ixl, ixu=p.ixu, idl=p.idl, idu=p.idu)
    d = ko.compute_directions(st, it, pat, p.res)
    for k in ko.DIR_NAMES:
        assert np.isfinite(d_r.absmax(k)), k
        assert np.abs(d_r.pick(k, d[k]) - d_r[k]).max() <= 1e-8 * max(1.0, d_r.absmax(k)), k


def test_kkt_full_operator_matches_reference(reference):
    """hiopMatVecKKTFullOpr::times_vec on a random 12-block vector."""
    p = synth.make_qn_problem(700, 12, 4, masked_zero_divisors=True)
    rng = np.random.default_rng(17)
    x = {k: rng.standard_normal(np.asarray(p.res[rk]).size) for k, rk in zip(ko.DIR_NAMES, ko.RES_NAMES)}

    def run():
        q = _ref_system(p)
        Dx_r, _, _ = q.update()
        y_r = q.kkt_full_times_vec(x)
        q.close()
        return dict(Dx=Dx_r, **y_r)
    exact = [k for k in ko.RES_NAMES if k not in ("rx", "ryc", "ryd")]          # elementwise rows are bit-identical
    r = reference(run, exact=["Dx"] + exact)
    Dx_r, st = _oracle_state(p)
    r.assert_same("Dx", Dx_r)                                                 # the operator is applied with the reference's D_x
    it = dict(sxl=p.sxl, sxu=p.sxu, zl=p.zl, zu=p.zu, sdl=p.sdl, sdu=p.sdu, vl=p.vl, vu=p.vu)
    pat = dict(ixl=p.ixl, ixu=p.ixu, idl=p.idl, idu=p.idu)
    y = ko.kkt_full_times_vec(st, it, pat, x, Dx_r)
    for k in ko.RES_NAMES:
        if k in exact:
            r.assert_same(k, y[k])
        else:
            assert np.abs(r.pick(k, y[k]) - r[k]).max(initial=0.0) <= 1e-12 * max(1.0, r.absmax(k)), k


@pytest.mark.parametrize("mu,maxit", [(1e-1, 8), (1e-6, 8), (1e-3, 2), (1.0, 0)])
def test_compute_directions_w_ir_matches_reference(mu, maxit, reference):
    """hiopKKTLinSys::compute_directions_w_IR: BiCGStab on the full KKT system, preconditioned by computeDirections."""
    p = synth.make_qn_problem(1200, 16, 4, masked_zero_divisors=True)

    def run():
        q = _ref_system(p)
        Dx_r, _, _ = q.update()
        d_r, info_r = q.compute_directions_w_ir(p.res, mu, maxit)
        q.close()
        return dict(Dx=Dx_r, info=np.array(info_r), **d_r)
    r = reference(run, exact=("Dx",))
    Dx_r, st = _oracle_state(p)
    r.assert_same("Dx", Dx_r)                                                 # the oracle runs with the reference's D_x
    info_r = r["info"]
    it = dict(sxl=p.sxl, sxu=p.sxu, zl=p.zl, zu=p.zu, sdl=p.sdl, sdu=p.sdu, vl=p.vl, vu=p.vu)
    pat = dict(ixl=p.ixl, ixu=p.ixu, idl=p.idl, idu=p.idu)
    d, info = ko.compute_directions_w_ir(st, it, pat, p.res, mu, maxit, Dx=Dx_r)
    if maxit > 0:
        assert info[0] == info_r[0] and info[1] == info_r[1], (info, info_r)     # same exit flag, same (half-)iteration count
    for k in ko.DIR_NAMES:
        assert np.isfinite(r.absmax(k)), k
        assert np.abs(r.pick(k, d[k]) - r[k]).max(initial=0.0) <= 1e-8 * max(1.0, r.absmax(k)), k
    # the defining property: the returned direction solves the unreduced system to the BiCGStab tolerance
    if maxit > 0 and info_r[0] == 0:
        y = ko.kkt_full_times_vec(st, it, pat, d, Dx_r)
        rr = np.concatenate([y[k] - np.asarray(p.res[k]) for k in ko.RES_NAMES])
        bb = np.concatenate([np.asarray(p.res[k]) for k in ko.RES_NAMES])
        assert np.linalg.norm(rr) <= min(mu * 1e-2, 1e-6) * np.linalg.norm(bb) * 1.01


@pytest.mark.parametrize("case", ["good_prec", "rough_prec", "no_prec_budget", "singular", "zero_rhs"])
def test_bicgstab_recurrence_matches_reference(case, reference):
    """hiopBiCGStabSolver::solve on dense systems that need several iterations / hit the non-convergence exits."""
    rng = np.random.default_rng(21)
    n = 60
    A = rng.standard_normal((n, n)) + 8.0 * np.eye(n)
    b = rng.standard_normal(n)
    tol, maxit = 1e-10, 40
    if case == "good_prec":
        Minv = np.linalg.inv(A + 1e-3 * rng.standard_normal((n, n)))
    elif case == "rough_prec":
        Minv = np.linalg.inv(A + 0.15 * rng.standard_normal((n, n)))   # ~10 iterations; beyond that BiCGStab trajectories are rounding-chaotic
    elif case == "no_prec_budget":
        Minv, maxit = np.eye(n), 5                 # runs out of iterations -> minimal-residual fallback
    elif case == "singular":
        A = np.outer(rng.standard_normal(n), rng.standard_normal(n))   # rank 1: breakdown / stagnation exits
        Minv = np.eye(n)
    else:
        Minv, b = np.eye(n), np.zeros(n)

    def run():
        x_r, info_r = ref.bicgstab_dense(A, Minv, b, tol, maxit)
        return dict(x=x_r, info=np.array(info_r))
    r = reference(run)
    x_r, info_r = r["x"], r["info"]
    x, flag, it, a, rel = ko.bicgstab(lambda v: A @ v, lambda v: Minv @ v, b, tol, maxit)
    assert flag == info_r[0] and it == info_r[1], ((flag, it, a, rel), info_r)
    assert np.abs(x - x_r).max(initial=0.0) <= 1e-7 * max(1.0, np.abs(x_r).max(initial=0.0))
    assert abs(a - info_r[2]) <= 1e-3 * abs(info_r[2]) + 1e-13     # residual norms: same digits up to rounding amplification


@pytest.mark.parametrize("strategy", [1, 2, 3, 4, 5])
def test_secant_update_matches_reference(strategy, reference):
    """hiopHessianLowRank::update over a sequence: first call, appends, shifts (l_max = 3), both skip rules, all sigma rules."""
    n, me, mi, lmax = 300, 4, 3, 3
    seq = synth.make_secant_sequence(n, me, mi, steps=8)
    ones = np.ones(n)

    def run():
        q = ref.RefQn(n, me, mi, lmax, ones, np.zeros(n), np.ones(mi), np.zeros(mi))
        q.set_sigma_strategy(strategy, 1.0)
        out = {}
        for i, it in enumerate(seq):
            out.update({f"{i}/{k}": v for k, v in zip(("l", "St", "Yt", "L", "D", "sigma"),
                                                      q.hess_update(it["x"], it["grad_f"], it["yc"], it["yd"], it["Jc"], it["Jd"]))})
        q.close()
        return out
    r = reference(run, exact=[f"{i}/St" for i in range(len(seq))])
    mem = ko.SecantMemory(n, lmax, 1.0, strategy)
    statuses = []
    for i, it in enumerate(seq):
        l, L, D, sigma = (r[f"{i}/{k}"] for k in ("l", "L", "D", "sigma"))
        statuses.append(mem.update(it["x"], it["grad_f"], it["yc"], it["yd"], it["Jc"], it["Jd"]))
        assert mem.St.shape[0] == l
        r.assert_same(f"{i}/St", mem.St)                                # s = x - x_prev: one rounding, same bits
        Yt = f"{i}/Yt"
        assert np.abs(r.pick(Yt, mem.Yt) - r[Yt]).max(initial=0.0) <= 1e-13 * max(1.0, r.absmax(Yt))
        assert np.abs(np.tril(mem.L, -1) - np.tril(L, -1)).max(initial=0.0) <= 1e-12
        assert np.abs(mem.D - D).max(initial=0.0) <= 1e-12
        assert abs(mem.sigma - sigma) <= 1e-12 * sigma
    assert statuses == [0, 1, 1, 2, 1, 3, 1, 1], statuses


@pytest.mark.parametrize("form", [0, 1])
@pytest.mark.parametrize("nx,neq,nineq,dw,dc", [(40, 6, 9, 0.0, 0.0), (25, 10, 4, 1e-4, 1e-8), (12, 0, 5, 1e-3, 1e-6), (9, 3, 0, 0.0, 0.0)])
def test_dense_newton_kkt_matrix_matches_reference(form, nx, neq, nineq, dw, dc, reference):
    """hiopKKTLinSysDenseXYcYd / XDYcYd::build_kkt_matrix incl. non-zero regularisations (delta_cd lands on the first dual
    rows in the reference: reproduced)."""
    p = synth.make_mds_problem(0, nx, neq, nineq, seed=7 + nx, dwx=dw, dcc=dc)
    it = dict(zl=p.zl, sxl=p.sxl, zu=p.zu, sxu=p.sxu, vl=p.vl, sdl=p.sdl, vu=p.vu, sdu=p.sdu)
    pat = dict(ixl=p.ixl, ixu=p.ixu, idl=p.idl, idu=p.idu)
    deltas = (p.delta_wx, p.delta_wd, p.delta_cc, p.delta_cd)
    r = reference(lambda: dict(M=ref.densekkt_build(form, p.Hd, p.Jcd, p.Jdd, it, pat, deltas)), exact=("M",))
    M, _, _ = ko.dense_build_kkt_matrix(form, p.Hd, p.Jcd, p.Jdd, it, pat, deltas)
    r.assert_same("M", M)          # same additions in the same order: bit-identical, lower triangle zero


@pytest.mark.parametrize("n,m", [(800, 14), (300, 1), (500, 40)])
def test_lsq_duals_match_reference(n, m, reference):
    """hiopDualsLsqUpdateLinsysRedDenseSymPD::do_lsq_update (initial / recalculated multipliers)."""
    p = synth.make_qn_problem(n, m, 0)
    g = np.random.default_rng(8).standard_normal(n)

    def run():
        q = _ref_system(p)
        yc_r, yd_r = q.lsq_duals(g)
        q.close()
        return dict(yc=yc_r, yd=yd_r)
    r = reference(run)
    yc, yd = ko.lsq_duals(p.Jc, p.Jd, g, p.zl, p.zu, p.vl, p.vu)
    for a, b in ((yc, r["yc"]), (yd, r["yd"])):
        assert np.abs(a - b).max(initial=0.0) <= 1e-10 * max(1.0, np.abs(b).max(initial=0.0))


def test_iajaaa_writer_is_byte_identical_to_reference(tmp_path, reference):
    """write_kkt dumps: the C-ABI writer against hiopCSR_IO (matrix + rhs + solution), then the reader round-trips it."""
    from hiop_b200 import iajaaa
    K = np.triu(synth.make_kkt_like(23, 9, seed=4))
    K[2, 5] = 0.0                       # structural zeros are skipped (|a| <= 1e-25)
    K[7, 7] = 1e-30
    rhs = np.random.default_rng(2).standard_normal(32)
    sol = np.random.default_rng(3).standard_normal(32) * 1e3

    def run():
        with open(ref.write_iajaaa(tmp_path, 7, K, 23, 4, 5, rhs, sol), "rb") as f:
            return dict(file=np.frombuffer(f.read(), dtype=np.uint8))
    r = reference(run, exact=("file",))
    f_own = str(tmp_path / "own.iajaaa")
    iajaaa.write_system(f_own, K, 23, 4, 5, [(rhs, sol)])
    with open(f_own, "rb") as f:
        r.assert_same("file", np.frombuffer(f.read(), dtype=np.uint8))
    back = iajaaa.read_system(f_own)                  # byte for byte the reference's file
    assert (back["N"], back["nx"], back["meq"], back["mineq"]) == (32, 23, 4, 5)
    Kz = K.copy()
    Kz[np.abs(Kz) <= 1e-25] = 0.0
    assert np.abs(back["M"] - Kz).max() <= 1e-19 + 1e-15 * np.abs(Kz).max()          # "%.20f" text: absolute 1e-20 resolution
    assert np.abs(back["pairs"][0][0] - rhs).max() <= 1e-15 and np.abs(back["pairs"][0][1] - sol).max() <= 1e-12


@pytest.mark.parametrize("n,m,mz,mu,kd", [(900, 14, True, 0.1, 1e-5), (400, 1, False, 1e-4, 0.0), (300, 9, True, 1.0, 1e-5)])
def test_residual_update_matches_reference(n, m, mz, mu, kd, reference):
    """hiopResidual::update: the 12 residual blocks bit for bit (elementwise), J^T y to 1e-13, all 11 norms."""
    p = synth.make_qn_problem(n, m, 0, masked_zero_divisors=mz)
    itr, dat = synth.make_iterate(p)

    def run():
        q = _ref_system(p)
        r_r, n_r = q.residual_update(itr, dat["c"], dat["d"], dat["grad"], mu, kd, dat["xl"], dat["xu"], dat["dl"], dat["du"], dat["crhs"])
        q.close()
        return {**r_r, **n_r}
    out = reference(run, exact=[k for k in ko.RES_NAMES if k != "rx"])
    n_r = {k: out[k] for k in ko.NORM_NAMES}
    pat = dict(ixl=p.ixl, ixu=p.ixu, idl=p.idl, idu=p.idu)
    r, nm = ko.residual_update(itr, dat["c"], dat["d"], dat["grad"], p.Jc, p.Jd, mu, kd, pat, dat["xl"], dat["xu"], dat["dl"], dat["du"], dat["crhs"])
    for k in ko.RES_NAMES:
        if k == "rx":
            assert np.abs(out.pick(k, r[k]) - out[k]).max(initial=0.0) <= 1e-13 * max(1.0, out.absmax(k)), k
        else:
            out.assert_same(k, r[k])
    for k in ko.NORM_NAMES:
        assert abs(nm[k] - n_r[k]) <= 1e-12 * max(1.0, abs(n_r[k])), (k, nm[k], n_r[k])


@pytest.mark.parametrize("n,m,mz,mu,kd", [(900, 14, True, 0.1, 1e-5), (400, 1, False, 1e-4, 0.0)])
def test_logbar_and_fraction_to_bdry_match_reference(n, m, mz, mu, kd, reference):
    """hiopLogBarProblem::updateWithNlpInfo and hiopIterate::fractionToTheBdry."""
    p = synth.make_qn_problem(n, m, 0, masked_zero_divisors=mz)
    itr, dat = synth.make_iterate(p)
    pat = dict(ixl=p.ixl, ixu=p.ixu, idl=p.idl, idu=p.idu)
    # slacks must be positive where the pattern is set (log): masked-out entries may be anything
    for s, ptn in (("sxl", "ixl"), ("sxu", "ixu"), ("sdl", "idl"), ("sdu", "idu")):
        itr[s] = np.where(pat[ptn] == 1.0, np.abs(itr[s]) + 1e-3, itr[s])
    rng = np.random.default_rng(12)
    direction = {k: rng.standard_normal(np.asarray(v).size) * np.where(np.asarray(v) != 0, 1.0, 0.0) for k, v in itr.items()}
    # adjustDuals_primalLogHessian: duals scattered over several decades so that every branch of the clamp is taken
    itr2 = dict(itr)
    for zk in ("zl", "zu", "vl", "vu"):
        itr2[zk] = itr[zk] * 10.0 ** rng.integers(-6, 7, size=np.asarray(itr[zk]).size)

    def run():
        q = _ref_system(p)
        out = dict(zip(("fl", "gx", "gd"), q.logbar_update(itr, 3.25, mu, kd, dat["grad"])))
        out.update({f"adj{i}": a for i, a in enumerate(q.adjust_duals(itr2, mu, 1e10 if kd == 0.0 else 50.0))})
        out["ap"], out["ad"] = q.fraction_to_bdry(itr, direction, 0.995)
        q.close()
        return out
    r = reference(run, exact=("gx", "gd", "adj0", "adj1", "adj2", "adj3"))
    fl, gx, gd = ko.logbar_update(itr, 3.25, mu, kd, dat["grad"], pat)
    assert abs(fl - r["fl"]) <= 1e-13 * max(1.0, abs(r["fl"]))
    r.assert_same("gx", gx)
    r.assert_same("gd", gd)
    got = ko.iterate_adjust_duals(itr2, pat, mu, 1e10 if kd == 0.0 else 50.0)
    for i, a in enumerate(got):
        r.assert_same(f"adj{i}", a)
    ap, ad = ko.iterate_fraction_to_bdry(itr, direction, 0.995, pat)
    assert ap == r["ap"] and ad == r["ad"], ((ap, ad), (r["ap"], r["ad"]))


@pytest.mark.parametrize("mu", [1e-2, 10.0])
def test_adjust_small_slacks_matches_reference(mu, reference):
    """hiopIterate::adjust_small_slacks: slacks that collapsed to (or below) zero are pushed back; untouched when none is small."""
    p = synth.make_qn_problem(600, 12, 0, masked_zero_divisors=True)
    itr, dat = synth.make_iterate(p)
    pat = dict(ixl=p.ixl, ixu=p.ixu, idl=p.idl, idu=p.idu)
    rng = np.random.default_rng(4)
    for collapse in (True, False):
        trial = {k: np.array(v, dtype=np.float64) for k, v in itr.items()}
        for s_, ptn in (("sxl", "ixl"), ("sxu", "ixu"), ("sdl", "idl"), ("sdu", "idu")):
            trial[s_] = np.where(pat[ptn] == 1.0, np.abs(trial[s_]) + 1e-3, 0.0)
            if collapse:
                hit = (rng.random(trial[s_].size) < 0.2) & (pat[ptn] == 1.0)
                trial[s_] = np.where(hit, rng.choice([0.0, -1e-9, 1e-20, 3e-17], size=trial[s_].size), trial[s_])

        def run():
            q = _ref_system(p)
            num_r, got_r = q.adjust_small_slacks(trial, itr, mu, dat["xl"], dat["xu"], dat["dl"], dat["du"])
            q.close()
            return dict(num=num_r, **{f"s{i}": a for i, a in enumerate(got_r)})
        r = reference(run, exact=("s0", "s1", "s2", "s3"))
        num_r = r["num"]
        num = 0
        for i, (s_, ptn, bnd, dual) in enumerate((("sxl", "ixl", "xl", "zl"), ("sxu", "ixu", "xu", "zu"), ("sdl", "idl", "dl", "vl"),
                                                   ("sdu", "idu", "du", "vu"))):
            new, k = ko.adjust_small_slack(trial[s_], dat[bnd], itr[dual], pat[ptn], mu)
            num += k
            r.assert_same(f"s{i}", new)
        assert num == num_r and (num > 0) == collapse


def test_hess_times_vec_matches_reference(reference):
    p = synth.make_qn_problem(900, 3, 5)
    x = np.random.default_rng(3).standard_normal(p.n)
    y0 = np.random.default_rng(4).standard_normal(p.n)

    def run():
        q = _ref_system(p)
        Dx_r, _, _ = q.update()
        out = {f"y{int(add)}": q.hess_times_vec(0.5, y0, 2.0, x, add) for add in (False, True)}
        q.close()
        return dict(Dx=Dx_r, **out)
    r = reference(run, exact=("Dx",))
    Dx_r, _ = _oracle_state(p)
    r.assert_same("Dx", Dx_r)                                                 # the oracle runs with the reference's D_x
    for add in (False, True):
        k = f"y{int(add)}"
        y = ko.hess_times_vec(p.St, p.Yt, p.sigma, Dx_r, 0.5, y0, 2.0, x, add)
        assert np.abs(r.pick(k, y) - r[k]).max() <= 1e-10 * r.absmax(k)


@pytest.mark.parametrize("nx,m", [(30, 10), (120, 37), (5, 0), (1, 1)])
def test_symdense_matches_reference(nx, m, reference):
    K = synth.make_kkt_like(nx, m)
    rhs = np.random.default_rng(5).standard_normal(nx + m)
    r = reference(lambda: dict(zip(("ret", "sol"), ref.symdense_factor_solve(np.triu(K), rhs)[:2])))
    ret_r, sol_r = r["ret"], r["sol"]
    ret, f = ko.symdense_matrix_changed(np.triu(K))
    assert ret == ret_r == m
    sol = f.solve(rhs)
    assert np.abs(sol - sol_r).max() <= 1e-9 * np.abs(sol_r).max()
    assert np.abs(K @ sol - rhs).max() <= 1e-9 * np.abs(rhs).max()


def test_symdense_singular_matches_reference(reference):
    K = synth.make_kkt_like(20, 6)
    K[3, :] = 0.0
    K[:, 3] = 0.0
    ret_r = reference(lambda: dict(ret=ref.symdense_factor_solve(np.triu(K))[0]))["ret"]
    ret, _ = ko.symdense_matrix_changed(np.triu(K))
    assert ret == ret_r == -1


def test_vector_ops_match_reference(reference):
    r = np.random.default_rng(9)
    n = 1000
    y, x = r.standard_normal(n), r.standard_normal(n)
    z = r.uniform(0.5, 2.0, n)
    sel = (r.random(n) < 0.6).astype(np.float64)
    z0 = z * sel  # zero divisors on masked-out lanes
    ixu = (r.random(n) < 0.3).astype(np.float64)

    def run():
        out = {}
        for alpha in (1.0, -1.0, 0.37):
            out[f"axdzpy_w_pattern_{alpha}"] = ref.vec_op("axdzpy_w_pattern", y, x, z0, sel, alpha)[0]
            out[f"axzpy_{alpha}"] = ref.vec_op("axzpy", y, x, z, None, alpha)[0]
        out["component_div_w_sel"] = ref.vec_op("component_div_w_sel", y, z0, None, sel)[0]
        out["add_logbar_grad"] = ref.vec_op("add_logbar_grad", y, z0, None, sel, 0.1)[0]
        out["logbarrier"] = ref.vec_op("logbarrier", z, None, None, sel)[1]
        out["lin_damping_term"] = ref.vec_op("lin_damping_term", z, sel, ixu, None, 0.1, 1e-5)[1]
        out["add_lin_damping"] = ref.vec_op("add_lin_damping", y, sel, ixu, None, 0.9, 1e-6)[0]
        out["frac_to_bdry_w_sel"] = ref.vec_op("frac_to_bdry_w_sel", z, x, None, sel, 0.995)[1]
        out["frac_to_bdry"] = ref.vec_op("frac_to_bdry", z, x, None, None, 0.995)[1]
        return out
    vectors = [f"{op}_{alpha}" for alpha in (1.0, -1.0, 0.37) for op in ("axdzpy_w_pattern", "axzpy")]
    g = reference(run, exact=vectors + ["component_div_w_sel", "add_logbar_grad", "add_lin_damping"])
    for alpha in (1.0, -1.0, 0.37):
        g.assert_same(f"axdzpy_w_pattern_{alpha}", ko.axdzpy_w_pattern(y.copy(), alpha, x, z0, sel))
        g.assert_same(f"axzpy_{alpha}", ko.axzpy(y.copy(), alpha, x, z))
    g.assert_same("component_div_w_sel", ko.component_div_w_select(y.copy(), z0, sel))
    g.assert_same("add_logbar_grad", ko.add_log_barrier_grad(y.copy(), 0.1, z0, sel))
    assert g["logbarrier"] == ko.log_barrier(z, sel)
    assert g["lin_damping_term"] == ko.linear_damping_term(z, sel, ixu, 0.1, 1e-5)
    g.assert_same("add_lin_damping", ko.add_linear_damping_term(y.copy(), sel, ixu, 0.9, 1e-6))
    assert g["frac_to_bdry_w_sel"] == ko.fraction_to_the_bdry(z, x, 0.995, sel)
    assert g["frac_to_bdry"] == ko.fraction_to_the_bdry(z, x, 0.995)


def test_mds_assembly_ops_match_reference(reference):
    r = np.random.default_rng(21)
    Nw, m, n = 40, 7, 12
    A = r.standard_normal((m, n))
    W = r.standard_normal((Nw, Nw))
    H = r.standard_normal((n, n))
    # sparse Schur terms: sorted triplets, ~4 nnz per row
    ms, ns = 9, 30
    rows, cols = [], []
    for i in range(ms):
        cs = np.sort(r.choice(ns, 4, replace=False))
        rows += [i] * 4
        cols += list(cs)
    iR, jC = np.array(rows, dtype=np.int32), np.array(cols, dtype=np.int32)
    vals = r.standard_normal(iR.size)
    D = r.uniform(0.5, 2.0, ns)

    def run():
        W1, W2, W3 = W.copy(), W.copy(), W.copy()
        ref.lib().ref_mat_trans_add_to_sym_upper(m, n, A.ctypes.data_as(ref.dp), 3, 20, 0.7, Nw, W1.ctypes.data_as(ref.dp))
        ref.lib().ref_mat_add_upper_to_sym_upper(n, H.ctypes.data_as(ref.dp), 5, -1.3, Nw, W2.ctypes.data_as(ref.dp))
        ref.lib().ref_sp_add_MDinvMtrans(ms, ns, iR.size, iR.ctypes.data_as(ref.ip), jC.ctypes.data_as(ref.ip),
                                         vals.ctypes.data_as(ref.dp), 11, -1.0, D.ctypes.data_as(ref.dp), Nw,
                                         W3.ctypes.data_as(ref.dp))
        return dict(trans_add=W1, add_upper=W2, sp_MDinvMtrans=W3)
    g = reference(run, exact=("trans_add", "add_upper"))
    g.assert_same("trans_add", ko.trans_add_to_sym_upper(A, 3, 20, 0.7, W.copy()))
    g.assert_same("add_upper", ko.add_upper_to_sym_upper(H, 5, -1.3, W.copy()))
    Wo = ko.sp_add_MDinvMtrans(ms, ns, iR, jC, vals, 11, -1.0, D, W.copy())
    assert np.abs(g.pick("sp_MDinvMtrans", Wo) - g["sp_MDinvMtrans"]).max() <= 1e-13 * g.absmax("sp_MDinvMtrans")


def test_mds_build_kkt_matrix_matches_reference_methods(reference):
    """ko.mds_build_kkt_matrix against the reference's own matrix methods called in the order of
    hiopKKTLinSysCompressedMDSXYcYd::build_kkt_matrix (src/Optimization/hiopKKTLinSysMDS.cpp:196-290)."""
    p = synth.make_mds_problem(60, 25, 9, 14, dwx=1e-4, dcc=1e-6)
    M, Dx, Hxs, Dd_inv = ko.mds_build_kkt_matrix(p)

    def run():
        L, dp, ip = ref.lib(), ref.dp, ref.ip
        N = p.nxd + p.neq + p.nineq
        W = np.zeros((N, N))
        wp = W.ctypes.data_as(dp)

        def D(a):
            a = np.ascontiguousarray(a, dtype=np.float64)
            return a, a.ctypes.data_as(dp)

        def I(a):
            a = np.ascontiguousarray(a, dtype=np.int32)
            return a, a.ctypes.data_as(ip)
        Dx_r, _ = ref.vec_op("axdzpy_w_pattern", np.zeros(p.nxs + p.nxd), p.zl, p.sxl, p.ixl, 1.0)
        Dx_r, _ = ref.vec_op("axdzpy_w_pattern", Dx_r, p.zu, p.sxu, p.ixu, 1.0)
        a, pa = D(p.Hd); L.ref_mat_add_upper_to_sym_upper(p.nxd, pa, 0, 1.0, N, wp)
        a, pa = D(p.Jcd); L.ref_mat_trans_add_to_sym_upper(p.neq, p.nxd, pa, 0, p.nxd, 1.0, N, wp)
        a, pa = D(p.Jdd); L.ref_mat_trans_add_to_sym_upper(p.nineq, p.nxd, pa, 0, p.nxd + p.neq, 1.0, N, wp)
        a, pa = D(Dx[p.nxs:]); L.ref_mat_add_sub_diagonal(N, wp, 0, 1.0, p.nxd, pa)
        a, pa = D(p.delta_wx[p.nxs:]); L.ref_mat_add_sub_diagonal(N, wp, 0, 1.0, p.nxd, pa)
        hx, phx = D(Hxs)
        ic, pic = I(p.iRow_c); jc, pjc = I(p.jCol_c); vc, pvc = D(p.Jcs_vals)
        idd, pid = I(p.iRow_d); jd, pjd = I(p.jCol_d); vd, pvd = D(p.Jds_vals)
        L.ref_sp_add_MDinvMtrans(p.neq, p.nxs, ic.size, pic, pjc, pvc, p.nxd, -1.0, phx, N, wp)
        a, pa = D(p.delta_cc); L.ref_mat_add_sub_diagonal(N, wp, p.nxd, -1.0, p.neq, pa)
        L.ref_sp_add_MDinvMtrans(p.nineq, p.nxs, idd.size, pid, pjd, pvd, p.nxd + p.neq, -1.0, phx, N, wp)
        L.ref_sp_add_MDinvNtrans(p.neq, p.nxs, ic.size, pic, pjc, pvc, p.nineq, idd.size, pid, pjd, pvd, p.nxd, p.nxd + p.neq, -1.0, phx, N, wp)
        a, pa = D(Dd_inv); L.ref_mat_add_sub_diagonal(N, wp, p.nxd + p.neq, -1.0, p.nineq, pa)
        a, pa = D(p.delta_cd); L.ref_mat_add_sub_diagonal(N, wp, p.nxd + p.neq, -1.0, p.nineq, pa)
        ret_r, _, _, _ = ref.symdense_factor_solve(W)
        return dict(Dx=Dx_r, W=W, ret=ret_r)
    g = reference(run, exact=("Dx", "W"))
    g.assert_same("Dx", Dx)
    g.assert_same("W", M)
    # and the whole system is a valid KKT system: inertia (nxd, 0, neq+nineq) for the dense block
    ret, f = ko.mds_factorize_with_curv_check(M, Hxs)
    assert ret == g["ret"] == p.neq + p.nineq
    dx, dyc, dyd = ko.mds_solve_compressed(p, f, Hxs, p.rx, p.ryc, p.ryd)
    # residual of the full (unreduced) XYcYd system
    import scipy.sparse as sp
    Jc = np.hstack([sp.csr_matrix((p.Jcs_vals, (p.iRow_c, p.jCol_c)), shape=(p.neq, p.nxs)).toarray(), p.Jcd])
    Jd = np.hstack([sp.csr_matrix((p.Jds_vals, (p.iRow_d, p.jCol_d)), shape=(p.nineq, p.nxs)).toarray(), p.Jdd])
    H = np.zeros((p.nxs + p.nxd, p.nxs + p.nxd))
    H[:p.nxs, :p.nxs] = np.diag(p.Hs_diag)
    H[p.nxs:, p.nxs:] = p.Hd
    H += np.diag(Dx + p.delta_wx)
    r1 = H @ dx + Jc.T @ dyc + Jd.T @ dyd - p.rx
    r2 = Jc @ dx - p.delta_cc * dyc - p.ryc
    r3 = Jd @ dx - (Dd_inv + p.delta_cd) * dyd - p.ryd
    assert max(np.abs(r1).max(), np.abs(r2).max(), np.abs(r3).max()) <= 1e-9
