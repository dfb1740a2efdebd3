"""Generates tests/golden/*.npz by running the UNMODIFIED reference (oracle/_ref, built by `make -C oracle ref` from the
reference's sources, REF=<its checkout>) on seeded synthetic inputs:  python tests/golden/make_golden.py
The fixtures freeze (inputs, reference outputs) tuples so that the test suite -- which does not need the reference --
checks both the oracle restatement and the CUDA path against what the reference itself computed. The reference's outputs
for tests/test_oracle_vs_ref.py (tests/golden/oracle_vs_ref.npz) are recorded by that module itself."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from hiop_b200 import synth  # noqa: E402
from oracle import ref  # noqa: E402
from oracle.kkt_oracle import DIR_NAMES, RES_NAMES  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))

QN_CASES = [  # name, n, m, l, masked_zero_divisors
    ("qn_n400_m12_l4", 400, 12, 4, True),
    ("qn_n1500_m40_l6", 1500, 40, 6, False),
    ("qn_n300_m1_l2", 300, 1, 2, True),      # NlpDenseConsEx1 shape (m=1)
    ("qn_n640_m33_l0", 640, 33, 0, False),   # first IPM iteration: empty secant memory
]


def qn_case(name, n, m, l, mz):
    p = synth.make_qn_problem(n, m, l, masked_zero_divisors=mz)
    q = ref.RefQn(p.n, p.m_eq, p.m_ineq, max(p.l, 1), p.ixl, p.ixu, p.idl, p.idu)
    q.set_iterate(p.sxl, p.sxu, p.zl, p.zu, p.sdl, p.sdu, p.vl, p.vu)
    q.set_jac(p.Jc, p.Jd)
    q.set_secant(p.sigma, p.St, p.Yt, p.L, p.D)
    Dx, DhInv, Dd_inv = q.update()
    N = q.condense()
    hs = q.hess_solve(p.rx)
    dx, dyc, dyd = q.solve_compressed(p.rx, p.ryc, p.ryd)
    d = q.compute_directions(p.res)
    x = np.random.default_rng(77).standard_normal(n)
    Bx = q.hess_times_vec(0.0, np.zeros(n), 1.0, x, True)
    # outer refinement (a19): the full 12-block operator on a random compound vector, and compute_directions_w_IR
    rng = np.random.default_rng(78)
    kx_in = {k: rng.standard_normal(np.asarray(p.res[rk]).size) for k, rk in zip(DIR_NAMES, RES_NAMES)}
    kx_out = q.kkt_full_times_vec(kx_in)
    ir_mu, ir_maxit = 1e-3, 8
    d_ir, ir_info = q.compute_directions_w_ir(p.res, ir_mu, ir_maxit)
    out = dict(n=n, m_eq=p.m_eq, m_ineq=p.m_ineq, l=l, sigma=p.sigma, Jc=p.Jc, Jd=p.Jd, ixl=p.ixl, ixu=p.ixu, idl=p.idl,
               idu=p.idu, sxl=p.sxl, sxu=p.sxu, zl=p.zl, zu=p.zu, sdl=p.sdl, sdu=p.sdu, vl=p.vl, vu=p.vu, St=p.St, Yt=p.Yt,
               L=p.L, D=p.D, rx=p.rx, ryc=p.ryc, ryd=p.ryd, tv_x=x,
               ref_Dx=Dx, ref_DhInv=DhInv, ref_Dd_inv=Dd_inv, ref_N=N, ref_hess_solve=hs, ref_dx=dx, ref_dyc=dyc,
               ref_dyd=dyd, ref_Bx=Bx)
    for k in RES_NAMES:
        out["res_" + k] = p.res[k]
    for k in DIR_NAMES:
        out["ref_dir_" + k] = d[k]
        out["ref_ir_dir_" + k] = d_ir[k]
        out["kx_in_" + k] = kx_in[k]
    for k in RES_NAMES:
        out["ref_kx_out_" + k] = kx_out[k]
    out["ir_mu"], out["ir_maxit"], out["ref_ir_info"] = ir_mu, ir_maxit, np.array(ir_info)
    q.close()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "N cond ~", np.linalg.cond(N))


def densekkt_case():
    """hiopKKTLinSysDenseXYcYd / XDYcYd::build_kkt_matrix + LAPACK solve, nx=30, neq=7, nineq=11, non-zero regularisations."""
    p = synth.make_mds_problem(0, 30, 7, 11, seed=19, dwx=1e-4, dcc=1e-8)
    it = dict(zl=p.zl, sxl=p.sxl, zu=p.zu, sxu=p.sxu, vl=p.vl, sdl=p.sdl, vu=p.vu, sdu=p.sdu)
    pat = dict(ixl=p.ixl, ixu=p.ixu, idl=p.idl, idu=p.idu)
    deltas = (p.delta_wx, p.delta_wd, p.delta_cc, p.delta_cd)
    out = dict(nx=30, neq=7, nineq=11, H=p.Hd, Jc=p.Jcd, Jd=p.Jdd, dwx=p.delta_wx, dwd=p.delta_wd, dcc=p.delta_cc, dcd=p.delta_cd, **it, **pat)
    rng = np.random.default_rng(20)
    for form in (0, 1):
        M = ref.densekkt_build(form, p.Hd, p.Jcd, p.Jdd, it, pat, deltas)
        rhs = rng.standard_normal(M.shape[0])
        ret, sol, _, _ = ref.symdense_factor_solve(M, rhs)
        out[f"ref_M{form}"], out[f"rhs{form}"], out[f"ref_ret{form}"], out[f"ref_sol{form}"] = M, rhs, ret, sol
    np.savez_compressed(os.path.join(OUT, "densekkt_nx30.npz"), **out)
    print("densekkt rets", int(out["ref_ret0"]), int(out["ref_ret1"]))


def iajaaa_case():
    """write_kkt dump of a small KKT matrix + one rhs/solution pair, written by the reference's hiopCSR_IO."""
    import shutil
    import tempfile
    K = np.triu(synth.make_kkt_like(23, 9, seed=4))
    K[2, 5] = 0.0
    K[7, 7] = 1e-30
    rhs = np.random.default_rng(2).standard_normal(32)
    sol = np.random.default_rng(3).standard_normal(32) * 1e3
    with tempfile.TemporaryDirectory() as d:
        f = ref.write_iajaaa(d, 7, K, 23, 4, 5, rhs, sol)
        shutil.copy(f, os.path.join(OUT, "kkt_linsys_7.iajaaa"))
    np.savez_compressed(os.path.join(OUT, "iajaaa_case.npz"), K=K, rhs=rhs, sol=sol, nx=23, meq=4, mineq=5)
    print("iajaaa golden written")


def symdense_cases():
    out = {}
    for i, (nx, m) in enumerate([(24, 9), (70, 30), (3, 0), (1, 1), (130, 61)]):
        K = synth.make_kkt_like(nx, m, seed=100 + i)
        rhs = np.random.default_rng(200 + i).standard_normal(nx + m)
        ret, sol, _, _ = ref.symdense_factor_solve(np.triu(K), rhs)
        out[f"K{i}"] = np.triu(K)
        out[f"rhs{i}"] = rhs
        out[f"ret{i}"] = ret
        out[f"sol{i}"] = sol
    # general indefinite (needs 2x2 pivots) and singular
    M = synth.make_symmetric_indefinite(64, 20, seed=5)
    rhs = np.random.default_rng(6).standard_normal(64)
    ret, sol, _, _ = ref.symdense_factor_solve(np.triu(M), rhs)
    out["K5"], out["rhs5"], out["ret5"], out["sol5"] = np.triu(M), rhs, ret, sol
    Z = np.array([[0.0, 1.0, 2.0], [1.0, 0.0, 3.0], [2.0, 3.0, 0.0]])  # zero diagonal: forces 2x2 pivot
    rhs = np.array([1.0, 2.0, 3.0])
    ret, sol, _, _ = ref.symdense_factor_solve(np.triu(Z), rhs)
    out["K6"], out["rhs6"], out["ret6"], out["sol6"] = np.triu(Z), rhs, ret, sol
    S = synth.make_kkt_like(20, 6, seed=3)
    S[3, :] = 0.0
    S[:, 3] = 0.0
    ret, _, _, _ = ref.symdense_factor_solve(np.triu(S))
    out["K7"], out["rhs7"], out["ret7"], out["sol7"] = np.triu(S), np.zeros(26), ret, np.zeros(26)
    out["count"] = 8
    np.savez_compressed(os.path.join(OUT, "symdense.npz"), **out)
    print("symdense rets", [int(out[f"ret{i}"]) for i in range(8)])


def vec_cases():
    r = np.random.default_rng(9)
    n = 1000
    y, x = r.standard_normal(n), r.standard_normal(n)
    z = r.uniform(0.5, 2.0, n)
    sel = (r.random(n) < 0.6).astype(np.float64)
    ixu = (r.random(n) < 0.3).astype(np.float64)
    z0 = z * sel
    out = dict(y=y, x=x, z=z, sel=sel, ixu=ixu)
    for alpha in (1.0, -1.0, 0.37):
        out[f"axdzpy_w_pattern_{alpha}"] = ref.vec_op("axdzpy_w_pattern", y, x, z0, sel, alpha)[0]
        out[f"axzpy_{alpha}"] = ref.vec_op("axzpy", y, x, z, None, alpha)[0]
        out[f"axdzpy_{alpha}"] = ref.vec_op("axdzpy", y, x, z, None, alpha)[0]
    out["component_div_w_sel"] = ref.vec_op("component_div_w_sel", y, z0, None, sel)[0]
    out["component_mult"] = ref.vec_op("component_mult", y, x)[0]
    out["component_div"] = ref.vec_op("component_div", y, z)[0]
    out["invert"] = ref.vec_op("invert", z)[0]
    out["select_pattern"] = ref.vec_op("select_pattern", y, None, None, sel)[0]
    out["add_constant"] = ref.vec_op("add_constant", y, None, None, None, 0.25)[0]
    out["add_constant_w_sel"] = ref.vec_op("add_constant_w_sel", y, None, None, sel, 0.25)[0]
    out["add_logbar_grad"] = ref.vec_op("add_logbar_grad", y, z0, None, sel, 0.1)[0]
    out["add_lin_damping"] = ref.vec_op("add_lin_damping", y, sel, ixu, None, 0.9, 1e-6)[0]
    out["twonorm"] = ref.vec_op("twonorm", y)[1]
    out["dot"] = ref.vec_op("dot", y, x)[1]
    out["infnorm"] = ref.vec_op("infnorm", y)[1]
    out["onenorm"] = ref.vec_op("onenorm", y)[1]
    out["logbarrier"] = ref.vec_op("logbarrier", z, None, None, sel)[1]
    out["lin_damping_term"] = ref.vec_op("lin_damping_term", z, sel, ixu, None, 0.1, 1e-5)[1]
    out["min_w_pattern"] = ref.vec_op("min_w_pattern", y, None, None, sel)[1]
    out["frac_to_bdry"] = ref.vec_op("frac_to_bdry", z, x, None, None, 0.995)[1]
    out["frac_to_bdry_w_sel"] = ref.vec_op("frac_to_bdry_w_sel", z, x, None, sel, 0.995)[1]
    np.savez_compressed(os.path.join(OUT, "vector_ops.npz"), **out)


def mds_case():
    """MDS KKT assembly through the reference's own matrix methods (order of build_kkt_matrix) + LAPACK BK solve."""
    import ctypes
    from oracle import kkt_oracle as ko
    p = synth.make_mds_problem(50, 20, 8, 11, dwx=1e-4, dcc=1e-6, seed=77)
    M, Dx, Hxs, Dd_inv = ko.mds_build_kkt_matrix(p)     # bit-identical to the reference methods (tests/test_oracle_vs_ref.py)
    ret, sol, _, _ = ref.symdense_factor_solve(M, np.concatenate([p.rx[p.nxs:], p.ryc, p.ryd]))
    out = {k: getattr(p, k) for k in p.__dataclass_fields__}
    out.update(ref_M=M, ref_Dx=Dx, ref_Hxs=Hxs, ref_Dd_inv=Dd_inv, ref_ret=ret)
    np.savez_compressed(os.path.join(OUT, "mds_nxs50_nxd20.npz"), **out)
    print("mds ret", ret)


if __name__ == "__main__":
    assert ref.available(), "build oracle/_ref first: make -C oracle ref"
    for c in QN_CASES:
        qn_case(*c)
    symdense_cases()
    densekkt_case()
    iajaaa_case()
    vec_cases()
    mds_case()
    subprocess.check_call([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", os.path.join(ROOT, "tests", "test_oracle_vs_ref.py")],
                          cwd=ROOT, env=dict(os.environ, HB_RECORD_REFERENCE="1"))
