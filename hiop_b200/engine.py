"""Host-side (Python) mirror of the reference's plug-in interfaces for the KKT hot path, on top of the C-ABI.

Names, argument meaning and return conventions follow the reference classes so that the parity tests read like the
reference's own call sites:

  Context                      one device + one stream (+ optional NCCL communicator)
  Vector ops (vec_*)           hiopVector methods                        src/LinAlg/hiopVector.hpp
  LinSolverSymDense            hiopLinSolverSymDense{Lapack,MagmaBuKa,MagmaNopiv}::{matrixChanged, solve}
                                                                         src/LinAlg/hiopLinSolver.hpp:78-128
  KKTLinSysLowRank             hiopKKTLinSysLowRank::{update, solveCompressed, computeDirections} with the
                               hiopHessianLowRank state it owns          src/Optimization/hiopKKTLinSys.cpp:1031-1350

torch is used ONLY as the owner of device buffers (tensor.data_ptr()) and for stream/event plumbing; every
computation is a call into libhiopb200.so. Nothing here falls back to torch/numpy math.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import EngineError, check

RES_NAMES = ["rx", "rd", "ryc", "ryd", "rxl", "rxu", "rdl", "rdu", "rszl", "rszu", "rsvl", "rsvu"]
DIR_NAMES = ["x", "d", "yc", "yd", "sxl", "sxu", "sdl", "sdu", "zl", "zu", "vl", "vu"]


def _ptr(t):
    if t is None:
        return None
    if isinstance(t, torch.Tensor):
        assert t.dtype == torch.float64 and t.is_contiguous(), "engine buffers are contiguous float64"
        return ctypes.c_void_p(t.data_ptr())
    raise TypeError(type(t))


class Context:
    """One GPU, one stream. `with ctx:` makes the engine stream torch's current stream so that tensor allocations,
    copies and CUDA events are ordered with the engine's kernels."""

    def __init__(self, device: int = 0):
        if not torch.cuda.is_available():
            raise EngineError("hiop_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.L = _lib.lib()
        self.h = ctypes.c_void_p()
        check(self.L.hb_ctx_create(device, ctypes.byref(self.h)), "hb_ctx_create")
        self.device = torch.device("cuda", device)
        self.stream = torch.cuda.ExternalStream(self.L.hb_ctx_stream(self.h), device=self.device)
        self._guard = None

    def __enter__(self):
        self._guard = torch.cuda.stream(self.stream)
        self._guard.__enter__()
        return self

    def __exit__(self, *a):
        g, self._guard = self._guard, None
        return g.__exit__(*a)

    def sync(self):
        check(self.L.hb_ctx_sync(self.h), "hb_ctx_sync")

    PHASES = ("update", "row maxima (+fused row dots)", "slicing", "GEMM+fix-up (C_aug)", "all-reduce", "V/U/N assembly", "Cholesky", "H^-1 rx",
              "J dx (+all-reduce)", "SPD solve", "J^T dy", "H^-1 rx (2nd)")

    def phase_timeline(self, on: bool):
        """arm (on=True) / read (on=False -> dict phase -> ms) the per-phase event marks of one quasi-Newton step"""
        if on:
            check(self.L.hb_ctx_phase_timeline(self.h, 1, None), "hb_ctx_phase_timeline")
            return None
        ms = (ctypes.c_float * len(self.PHASES))()
        check(self.L.hb_ctx_phase_timeline(self.h, 0, ms), "hb_ctx_phase_timeline")
        return {name: float(ms[i]) for i, name in enumerate(self.PHASES)}

    def microbench_peak(self, which: int) -> float:
        """0: FP64 DMMA TFLOP/s, 1: int8 tcgen05 TOP/s -- measured on this device, now (hb_microbench_peak)"""
        v = ctypes.c_double()
        check(self.L.hb_microbench_peak(self.h, which, ctypes.byref(v)), "hb_microbench_peak")
        return v.value

    def close(self):
        if self.h:
            self.L.hb_ctx_destroy(self.h)
            self.h = None

    def enable_timing(self, on: bool = True):
        check(self.L.hb_ctx_enable_timing(self.h, int(on)), "hb_ctx_enable_timing")

    def last_syrk_ms(self) -> float:
        ms = ctypes.c_float()
        check(self.L.hb_ctx_last_syrk_ms(self.h, ctypes.byref(ms)), "hb_ctx_last_syrk_ms")
        return float(ms.value)

    def set_oz_workspace_limit(self, nbytes: int):
        """Bound on the int8 slice buffer of the condensation (0 = AUTO: free device memory minus 1 GiB). Above the bound the columns
        are sliced and multiplied in chunks; a buffer held above it is released now. See include/hiopb200.h."""
        check(self.L.hb_ctx_set_oz_workspace_limit(self.h, int(nbytes)), "hb_ctx_set_oz_workspace_limit")

    def launch_count(self) -> int:
        return int(self.L.hb_launch_count())

    # -- distributed -----------------------------------------------------------------------------------------
    def init_comm(self, nranks: int, rank: int, unique_id: bytes | None):
        buf = ctypes.create_string_buffer(unique_id, 128) if unique_id is not None else None
        check(self.L.hb_comm_init(self.h, nranks, rank, buf), "hb_comm_init")

    def unique_id(self) -> bytes:
        buf = ctypes.create_string_buffer(128)
        check(self.L.hb_comm_unique_id(buf), "hb_comm_unique_id")
        return buf.raw

    def to_device(self, a) -> torch.Tensor:
        t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))
        with torch.cuda.stream(self.stream):
            return t.to(self.device, non_blocking=False)

    def zeros(self, *shape) -> torch.Tensor:
        with torch.cuda.stream(self.stream):
            return torch.zeros(*shape, dtype=torch.float64, device=self.device)

    # -- hiopVector ops --------------------------------------------------------------------------------------
    def _v(self, name, n, *args):
        check(getattr(self.L, name)(self.h, n, *args), name)

    def vec_set(self, y, c): self._v("hb_vec_set", y.numel(), _ptr(y), c)
    def vec_copy(self, y, x): self._v("hb_vec_copy", y.numel(), _ptr(y), _ptr(x))
    def vec_scale(self, y, a): self._v("hb_vec_scale", y.numel(), _ptr(y), a)
    def vec_axpy(self, y, a, x): self._v("hb_vec_axpy", y.numel(), _ptr(y), a, _ptr(x))
    def vec_axzpy(self, y, a, x, z): self._v("hb_vec_axzpy", y.numel(), _ptr(y), a, _ptr(x), _ptr(z))
    def vec_axdzpy(self, y, a, x, z): self._v("hb_vec_axdzpy", y.numel(), _ptr(y), a, _ptr(x), _ptr(z))
    def vec_axdzpy_w_pattern(self, y, a, x, z, s): self._v("hb_vec_axdzpy_w_pattern", y.numel(), _ptr(y), a, _ptr(x), _ptr(z), _ptr(s))
    def vec_component_mult(self, y, x): self._v("hb_vec_component_mult", y.numel(), _ptr(y), _ptr(x))
    def vec_component_div(self, y, x): self._v("hb_vec_component_div", y.numel(), _ptr(y), _ptr(x))
    def vec_component_div_w_pattern(self, y, x, s): self._v("hb_vec_component_div_w_pattern", y.numel(), _ptr(y), _ptr(x), _ptr(s))
    def vec_invert(self, y): self._v("hb_vec_invert", y.numel(), _ptr(y))
    def vec_select_pattern(self, y, s): self._v("hb_vec_select_pattern", y.numel(), _ptr(y), _ptr(s))
    def vec_add_constant(self, y, c): self._v("hb_vec_add_constant", y.numel(), _ptr(y), c)
    def vec_add_constant_w_pattern(self, y, c, s): self._v("hb_vec_add_constant_w_pattern", y.numel(), _ptr(y), c, _ptr(s))
    def vec_add_log_barrier_grad(self, y, a, x, s): self._v("hb_vec_add_log_barrier_grad", y.numel(), _ptr(y), a, _ptr(x), _ptr(s))
    def vec_add_linear_damping_term(self, y, ixl, ixu, a, ct): self._v("hb_vec_add_linear_damping_term", y.numel(), _ptr(y), _ptr(ixl), _ptr(ixu), a, ct)

    def _r(self, name, n, *args) -> float:
        out = ctypes.c_double()
        check(getattr(self.L, name)(self.h, n, *args, ctypes.byref(out)), name)
        return out.value

    def vec_dot(self, x, y): return self._r("hb_vec_dot", x.numel(), _ptr(x), _ptr(y))
    def vec_twonorm(self, x): return self._r("hb_vec_twonorm", x.numel(), _ptr(x))
    def vec_infnorm(self, x): return self._r("hb_vec_infnorm", x.numel(), _ptr(x))
    def vec_onenorm(self, x): return self._r("hb_vec_onenorm", x.numel(), _ptr(x))
    def vec_min_w_pattern(self, x, s): return self._r("hb_vec_min_w_pattern", x.numel(), _ptr(x), _ptr(s))
    def vec_log_barrier(self, x, s): return self._r("hb_vec_log_barrier", x.numel(), _ptr(x), _ptr(s))
    def vec_linear_damping_term(self, x, ixl, ixu, mu, kd): return self._r("hb_vec_linear_damping_term", x.numel(), _ptr(x), _ptr(ixl), _ptr(ixu), mu, kd)
    def vec_fraction_to_bdry(self, x, dx, tau, s=None): return self._r("hb_vec_fraction_to_bdry", x.numel(), _ptr(x), _ptr(dx), tau, _ptr(s))

    def mat_times_vec(self, A, beta, y, alpha, x):
        m, n = A.shape
        check(self.L.hb_mat_times_vec(self.h, m, n, _ptr(A), n, beta, _ptr(y), alpha, _ptr(x)), "hb_mat_times_vec")

    def mat_trans_times_vec(self, A, beta, y, alpha, x):
        m, n = A.shape
        check(self.L.hb_mat_trans_times_vec(self.h, m, n, _ptr(A), n, beta, _ptr(y), alpha, _ptr(x)), "hb_mat_trans_times_vec")


class LinSolverSymDense:
    """hiopLinSolverSymDense: owns the N x N row-major system matrix (upper triangle valid), `matrixChanged()` returns
    the number of negative eigenvalues or -1, `solve(x)` overwrites the rhs (src/LinAlg/hiopLinSolver.hpp:78-128)."""

    BUNCH_KAUFMAN, NOPIV, CHOLESKY = _lib.HB_FACT_BUNCH_KAUFMAN, _lib.HB_FACT_NOPIV, _lib.HB_FACT_CHOLESKY

    def __init__(self, ctx: Context, n: int, mode: int = _lib.HB_FACT_BUNCH_KAUFMAN):
        self.ctx, self.n, self.mode = ctx, n, mode
        self.h = ctypes.c_void_p()
        check(ctx.L.hb_symdense_create(ctx.h, n, ctypes.byref(self.h)), "hb_symdense_create")
        self._mptr = ctx.L.hb_symdense_matrix(self.h)

    def close(self):
        if self.h:
            self.ctx.L.hb_symdense_destroy(self.h)
            self.h = None

    def set_matrix(self, M: torch.Tensor):
        """Fills sysMatrix() from a device tensor (what the KKT class's build_kkt_matrix does in place)."""
        assert M.shape == (self.n, self.n)
        check(self.ctx.L.hb_memcpy_d2d(self.ctx.h, ctypes.c_void_p(self._mptr), _ptr(M.contiguous()), 8 * self.n * self.n), "memcpy")

    def matrixChanged(self) -> int:
        rc = self.ctx.L.hb_symdense_matrix_changed(self.h, self.mode)
        if rc < -1:
            check(rc, "hb_symdense_matrix_changed")
        return rc

    def matrixChanged_host(self, M: np.ndarray) -> int:
        M = np.ascontiguousarray(M, dtype=np.float64)
        rc = self.ctx.L.hb_symdense_matrix_changed_host(self.h, M.ctypes.data_as(ctypes.c_void_p), self.mode)
        if rc < -1:
            check(rc, "hb_symdense_matrix_changed_host")
        return rc

    def inertia(self):
        a, b, c = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        check(self.ctx.L.hb_symdense_inertia(self.h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)), "hb_symdense_inertia")
        return a.value, b.value, c.value

    def solve(self, x: torch.Tensor) -> bool:
        nrhs = x.numel() // max(self.n, 1) if self.n else 0
        rc = self.ctx.L.hb_symdense_solve(self.h, _ptr(x), nrhs)
        if rc < 0:
            check(rc, "hb_symdense_solve")
        return rc == 1

    def solve_host(self, x: np.ndarray) -> bool:
        assert x.dtype == np.float64 and x.flags["C_CONTIGUOUS"]
        nrhs = x.size // max(self.n, 1) if self.n else 0
        rc = self.ctx.L.hb_symdense_solve_host(self.h, x.ctypes.data_as(ctypes.c_void_p), nrhs)
        if rc < 0:
            check(rc, "hb_symdense_solve_host")
        return rc == 1


class KKTLinSysLowRank:
    """hiopKKTLinSysLowRank with the hiopHessianLowRank state it drives.

    Reference call order per IPM iteration (src/Optimization/hiopAlgFilterIPM.cpp:1215-1226):
        Hess->update(...)  -> set_secant(l, sigma, St, Yt, L, D)
        kkt->update(iter, grad_f, Jac_c, Jac_d, Hess) -> set_jacobian(Jc, Jd); update(iterate blocks)
        kkt->computeDirections(resid, dir)  -> compute_directions(res) / solveCompressed(rx, ryc, ryd)
    """

    def __init__(self, ctx: Context, n_local: int, m_eq: int, m_ineq: int, l_max: int = 6):
        self.ctx, self.n, self.m_eq, self.m_ineq, self.l_max = ctx, n_local, m_eq, m_ineq, l_max
        self.h = ctypes.c_void_p()
        check(ctx.L.hb_lowrank_create(ctx.h, n_local, m_eq, m_ineq, l_max, ctypes.byref(self.h)), "hb_lowrank_create")
        self._keep = {}

    def close(self):
        if self.h:
            self.ctx.L.hb_lowrank_destroy(self.h)
            self.h = None

    def set_patterns(self, ixl, ixu, idl, idu):
        self._keep["pat"] = (ixl, ixu, idl, idu)
        check(self.ctx.L.hb_lowrank_set_patterns(self.h, _ptr(ixl), _ptr(ixu), _ptr(idl), _ptr(idu)), "hb_lowrank_set_patterns")

    def set_jacobian(self, Jc, Jd):
        self._keep["jac"] = (Jc, Jd)
        check(self.ctx.L.hb_lowrank_set_jacobian(self.h, _ptr(Jc), _ptr(Jd)), "hb_lowrank_set_jacobian")

    def set_secant(self, sigma: float, St, Yt, L: np.ndarray, D: np.ndarray):
        l = 0 if St is None else St.shape[0]
        self._keep["sec"] = (St, Yt)
        Lh = np.ascontiguousarray(L, dtype=np.float64)
        Dh = np.ascontiguousarray(D, dtype=np.float64)
        check(self.ctx.L.hb_lowrank_set_secant(self.h, l, float(sigma), _ptr(St) if l else None, _ptr(Yt) if l else None,
                                               Lh.ctypes.data_as(ctypes.c_void_p), Dh.ctypes.data_as(ctypes.c_void_p)),
              "hb_lowrank_set_secant")

    # ---- hiopHessianLowRank::update on the device: the engine owns S_t, Y_t, x_prev, grad_f_prev, J_prev ----
    def secant_reset(self, sigma0: float = 1.0, sigma_strategy: int = 1):
        check(self.ctx.L.hb_lowrank_secant_reset(self.h, float(sigma0), int(sigma_strategy)), "hb_lowrank_secant_reset")

    def secant_update(self, x, grad_f, yc, yd, jacobian_is_constant: bool = False) -> int:
        """Returns the status: 0 first iterate stored, 1 pair accepted, 2 / 3 skipped (see include/hiopb200.h)."""
        st = ctypes.c_int(0)
        check(self.ctx.L.hb_lowrank_secant_update(self.h, _ptr(x), _ptr(grad_f), _ptr(yc), _ptr(yd), int(jacobian_is_constant), ctypes.byref(st)),
              "hb_lowrank_secant_update")
        return st.value

    def secant_state(self):
        """(l, sigma, St, Yt, L, D) as numpy arrays (S_t, Y_t are downloaded)."""
        l, sg = ctypes.c_int(0), ctypes.c_double(0.0)
        pS, pY = ctypes.c_void_p(), ctypes.c_void_p()
        lm = max(self.l_max, 1)
        L, D = np.zeros(lm * lm), np.zeros(lm)
        check(self.ctx.L.hb_lowrank_secant_state(self.h, ctypes.byref(l), ctypes.byref(sg), ctypes.byref(pS), ctypes.byref(pY),
                                                 L.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), D.ctypes.data_as(ctypes.POINTER(ctypes.c_double))),
              "hb_lowrank_secant_state")
        ll = l.value
        St, Yt = np.zeros((ll, self.n)), np.zeros((ll, self.n))
        self.ctx.sync()
        if ll and self.n:
            nbytes = 8 * ll * self.n
            check(self.ctx.L.hb_memcpy_d2h(self.ctx.h, St.ctypes.data_as(ctypes.c_void_p), pS, nbytes), "d2h")
            check(self.ctx.L.hb_memcpy_d2h(self.ctx.h, Yt.ctypes.data_as(ctypes.c_void_p), pY, nbytes), "d2h")
            self.ctx.sync()
        return ll, sg.value, St, Yt, L[:ll * ll].reshape(ll, ll).copy(), D[:ll].copy()

    def residual_update(self, it: dict, c, d, grad_f, mu, kappa_d, xl, xu, dl, du, crhs, res: dict) -> dict:
        """hiopResidual::update: fills the 12 residual blocks (device tensors in `res`, keyed by RES_NAMES) from the iterate `it`
        (device tensors keyed by DIR_NAMES); returns the 11 norms as a dict (inf_nlp_optim ... inf_cons_violation, see include/hiopb200.h)."""
        I = (ctypes.c_void_p * 12)(*[_ptr(it[k]) for k in DIR_NAMES])
        R = (ctypes.c_void_p * 12)(*[_ptr(res[k]) for k in RES_NAMES])
        nrm = (ctypes.c_double * 11)()
        check(self.ctx.L.hb_lowrank_residual_update(self.h, I, _ptr(c), _ptr(d), _ptr(grad_f), float(mu), float(kappa_d), _ptr(xl), _ptr(xu),
                                                    _ptr(dl), _ptr(du), _ptr(crhs), R, nrm), "hb_lowrank_residual_update")
        names = ["inf_nlp_optim", "inf_nlp_feasib", "inf_nlp_complem", "inf_bar_optim", "inf_bar_feasib", "inf_bar_complem", "one_nlp_feasib",
                 "one_bar_feasib", "one_nlp_optim", "one_bar_optim", "inf_cons_violation"]
        return dict(zip(names, list(nrm)))

    # ---- hiopIterate / hiopLogBarProblem: the line-search side of an iteration ----
    def _blocks(self, d: dict):
        return (ctypes.c_void_p * 12)(*[_ptr(d[k]) for k in DIR_NAMES])

    def fraction_to_bdry(self, it: dict, direction: dict, tau: float):
        ap, ad = ctypes.c_double(0.0), ctypes.c_double(0.0)
        check(self.ctx.L.hb_iterate_fraction_to_bdry(self.h, self._blocks(it), self._blocks(direction), float(tau), ctypes.byref(ap), ctypes.byref(ad)),
              "hb_iterate_fraction_to_bdry")
        return ap.value, ad.value

    def take_step(self, it: dict, direction: dict, alpha_primal: float, alpha_dual: float, out: dict, which: int = 3):
        check(self.ctx.L.hb_iterate_take_step(self.h, self._blocks(it), self._blocks(direction), float(alpha_primal), float(alpha_dual), int(which),
                                              self._blocks(out)), "hb_iterate_take_step")

    def adjust_duals_plh(self, it: dict, mu: float, kappa_sigma: float):
        """hiopIterate::adjustDuals_primalLogHessian: clamps zl, zu, vl, vu of `it` in place."""
        check(self.ctx.L.hb_iterate_adjust_duals_plh(self.h, self._blocks(it), float(mu), float(kappa_sigma)), "hb_iterate_adjust_duals_plh")

    def adjust_small_slacks(self, it: dict, it_curr: dict, mu: float, xl, xu, dl, du) -> int:
        """hiopIterate::adjust_small_slacks: fixes the slacks of `it` in place; returns how many were adjusted."""
        num = ctypes.c_int(0)
        check(self.ctx.L.hb_iterate_adjust_small_slacks(self.h, self._blocks(it), self._blocks(it_curr), float(mu), _ptr(xl), _ptr(xu), _ptr(dl),
                                                        _ptr(du), ctypes.byref(num)), "hb_iterate_adjust_small_slacks")
        return num.value

    def logbar(self, it: dict, f: float, mu: float, kappa_d: float, grad_f=None, grad_x=None, grad_d=None) -> float:
        fl = ctypes.c_double(0.0)
        check(self.ctx.L.hb_iterate_logbar(self.h, self._blocks(it), float(f), float(mu), float(kappa_d), _ptr(grad_f), _ptr(grad_x), _ptr(grad_d),
                                           ctypes.byref(fl)), "hb_iterate_logbar")
        return fl.value

    def lsq_duals(self, grad_f, zl, zu, vl, vu, yc, yd) -> bool:
        """hiopDualsLsqUpdate: least-squares yc, yd for the registered Jacobian; False if J J^T + I is not numerically SPD."""
        rc = self.ctx.L.hb_lowrank_lsq_duals(self.h, _ptr(grad_f), _ptr(zl), _ptr(zu), _ptr(vl), _ptr(vu), _ptr(yc), _ptr(yd))
        if rc == -4:
            return False
        check(rc, "hb_lowrank_lsq_duals")
        return True

    def update(self, zl, sxl, zu, sxu, vl, sdl, vu, sdu) -> bool:
        self._keep["it"] = (zl, sxl, zu, sxu, vl, sdl, vu, sdu)
        check(self.ctx.L.hb_lowrank_update(self.h, *[_ptr(t) for t in (zl, sxl, zu, sxu, vl, sdl, vu, sdu)]), "hb_lowrank_update")
        return True

    def set_condense_mode(self, mode: int):
        """-1 = auto (default); 0 = exact FP64 on the DMMA pipe; 6/7/8 = INT8-slice emulation on tcgen05 with that many slices."""
        check(self.ctx.L.hb_lowrank_set_condense_mode(self.h, int(mode)), "hb_lowrank_set_condense_mode")

    def condense_mode_used(self) -> int:
        return int(self.ctx.L.hb_lowrank_get_condense_mode(self.h))

    def condense(self):
        """synchronous: raises on a breakdown (after the FP64 retry of the AUTO mode)"""
        check(self.ctx.L.hb_lowrank_condense(self.h), "hb_lowrank_condense")

    def condense_async(self):
        check(self.ctx.L.hb_lowrank_condense_async(self.h), "hb_lowrank_condense_async")

    def check(self):
        """synchronises and reports a breakdown of an asynchronous condensation"""
        check(self.ctx.L.hb_lowrank_check(self.h), "hb_lowrank_check")

    def fallback_count(self) -> int:
        return int(self.ctx.L.hb_lowrank_fallback_count(self.h))

    def condense_chunks(self) -> int:
        """column chunks of the last int8-slice condensation: 1 = unchunked, 0 = the FP64 kernel ran"""
        return int(self.ctx.L.hb_lowrank_last_condense_chunks(self.h))

    def solveCompressed(self, rx, ryc, ryd, dx, dyc, dyd) -> bool:
        """rx is clobbered, like in the reference (hiopKKTLinSys.cpp:1178)."""
        rc = self.ctx.L.hb_lowrank_solve_compressed(self.h, *[_ptr(t) for t in (rx, ryc, ryd, dx, dyc, dyd)])
        if rc == -4:
            return False
        check(rc, "hb_lowrank_solve_compressed")
        return True

    def computeDirections(self, res: dict, dirs: dict) -> bool:
        R = (ctypes.c_void_p * 12)(*[_ptr(res[k]) for k in RES_NAMES])
        Dp = (ctypes.c_void_p * 12)(*[_ptr(dirs[k]) for k in DIR_NAMES])
        rc = self.ctx.L.hb_lowrank_compute_directions(self.h, R, Dp)
        if rc == -4:
            return False
        check(rc, "hb_lowrank_compute_directions")
        return True

    def compute_directions_w_IR(self, res: dict, dirs: dict, mu: float, maxit: int = 8, tol_factor: float = 1e-2, tol_min: float = 1e-6):
        """hiopKKTLinSys::compute_directions_w_IR; tol = min(mu*ir_outer_tol_factor, ir_outer_tol_min) like the reference.
        Returns (ok, (flag, iterations, abs_resid, rel_resid))."""
        R = (ctypes.c_void_p * 12)(*[_ptr(res[k]) for k in RES_NAMES])
        Dp = (ctypes.c_void_p * 12)(*[_ptr(dirs[k]) for k in DIR_NAMES])
        info = (ctypes.c_double * 4)()
        rc = self.ctx.L.hb_lowrank_compute_directions_w_ir(self.h, R, Dp, min(mu * tol_factor, tol_min), int(maxit), info)
        if rc == -4:
            return False, tuple(info)
        check(rc, "hb_lowrank_compute_directions_w_ir")
        return True, (int(info[0]), info[1], info[2], info[3])

    def kkt_full_times_vec(self, x: dict, y: dict):
        """y = K x, hiopMatVecKKTFullOpr::times_vec; x keyed by DIR_NAMES, y by RES_NAMES."""
        X = (ctypes.c_void_p * 12)(*[_ptr(x[k]) for k in DIR_NAMES])
        Y = (ctypes.c_void_p * 12)(*[_ptr(y[k]) for k in RES_NAMES])
        check(self.ctx.L.hb_lowrank_kkt_full_times_vec(self.h, X, Y), "hb_lowrank_kkt_full_times_vec")

    def hess_solve(self, rhs, x):
        check(self.ctx.L.hb_lowrank_hess_solve(self.h, _ptr(rhs), _ptr(x)), "hb_lowrank_hess_solve")

    def hess_times_vec(self, beta, y, alpha, x, add_log_term=False):
        check(self.ctx.L.hb_lowrank_hess_times_vec(self.h, beta, _ptr(y), alpha, _ptr(x), int(add_log_term)), "hb_lowrank_hess_times_vec")

    def _readback(self, fn, count):
        p = getattr(self.ctx.L, fn)(self.h)
        out = np.empty(count, dtype=np.float64)
        check(self.ctx.L.hb_memcpy_d2h(self.ctx.h, out.ctypes.data_as(ctypes.c_void_p), ctypes.c_void_p(p), 8 * count), "memcpy")
        self.ctx.sync()
        return out

    def Dx(self): return self._readback("hb_lowrank_Dx", self.n)
    def DhInv(self): return self._readback("hb_lowrank_DhInv", self.n)
    def Dd_inv(self): return self._readback("hb_lowrank_Dd_inv", self.m_ineq)
    def N(self):
        m = self.m_eq + self.m_ineq
        return self._readback("hb_lowrank_N", m * m).reshape(m, m)

    def last_solve_stats(self):
        a, b = ctypes.c_int(), ctypes.c_double()
        check(self.ctx.L.hb_lowrank_last_solve_stats(self.h, ctypes.byref(a), ctypes.byref(b)), "hb_lowrank_last_solve_stats")
        return a.value, b.value

    def kkt_system_host(self, Jc, Jd, it: dict, rx, ryc, ryd, dx, dyc, dyd):
        """Whole system from HOST numpy buffers (pinned or pageable); Jc/Jd may be None to reuse the resident Jacobian."""
        def hp(a):
            if a is None:
                return None
            assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
            return a.ctypes.data_as(ctypes.c_void_p)
        args = [hp(Jc), hp(Jd)] + [hp(it[k]) for k in ("zl", "sxl", "zu", "sxu", "vl", "sdl", "vu", "sdu")] + \
               [hp(a) for a in (rx, ryc, ryd, dx, dyc, dyd)]
        check(self.ctx.L.hb_lowrank_kkt_system_host(self.h, *args), "hb_lowrank_kkt_system_host")


class KKTLinSysCompressedMDSXYcYd:
    """hiopKKTLinSysCompressedMDSXYcYd (src/Optimization/hiopKKTLinSysMDS.cpp:59-484) around a LinSolverSymDense.

    update(iterate blocks) -> build_kkt_matrix(blocks, deltas) -> factorizeWithCurvCheck() -> solveCompressed(...)."""

    def __init__(self, ctx: Context, nxs: int, nxd: int, neq: int, nineq: int, safe_mode: bool = True):
        self.ctx, self.nxs, self.nxd, self.neq, self.nineq = ctx, nxs, nxd, neq, nineq
        self.h = ctypes.c_void_p()
        check(ctx.L.hb_mds_create(ctx.h, nxs, nxd, neq, nineq, ctypes.byref(self.h)), "hb_mds_create")
        # determineAndCreateLinsys (:405-482): Bunch-Kaufman in safe mode, no-pivot LDL^T otherwise
        self.linSys = LinSolverSymDense(ctx, nxd + neq + nineq, LinSolverSymDense.BUNCH_KAUFMAN if safe_mode else LinSolverSymDense.NOPIV)
        self._keep = {}

    def close(self):
        if self.h:
            self.ctx.L.hb_mds_destroy(self.h)
            self.h = None
        self.linSys.close()

    def set_sparsity(self, iRow_c, jCol_c, iRow_d, jCol_d):
        a = [np.ascontiguousarray(v, dtype=np.int32) for v in (iRow_c, jCol_c, iRow_d, jCol_d)]
        p = [v.ctypes.data_as(ctypes.c_void_p) for v in a]
        check(self.ctx.L.hb_mds_set_sparsity(self.h, a[0].size, p[0], p[1], a[2].size, p[2], p[3]), "hb_mds_set_sparsity")

    def update(self, zl, sxl, zu, sxu, ixl, ixu):
        self._keep["it"] = (zl, sxl, zu, sxu, ixl, ixu)
        check(self.ctx.L.hb_mds_update(self.h, *[_ptr(t) for t in (zl, sxl, zu, sxu, ixl, ixu)]), "hb_mds_update")

    def build_kkt_matrix(self, Hd, Hs_diag, Jcd, Jdd, Jcs_vals, Jds_vals, vl, sdl, vu, sdu, idl, idu, delta_wx, delta_wd, delta_cc, delta_cd):
        args = (Hd, Hs_diag, Jcd, Jdd, Jcs_vals, Jds_vals, vl, sdl, vu, sdu, idl, idu, delta_wx, delta_wd, delta_cc, delta_cd)
        self._keep["blk"] = args
        check(self.ctx.L.hb_mds_build_kkt_matrix(self.h, *[_ptr(t) for t in args], ctypes.c_void_p(self.linSys._mptr)), "hb_mds_build_kkt_matrix")

    def factorizeWithCurvCheck(self) -> int:
        """Number of negative eigenvalues of the whole XYcYd system via Haynsworth additivity, or -1 (:78-110)."""
        n_neg = self.linSys.matrixChanged()
        if n_neg < 0:
            return -1
        a, b = ctypes.c_int(), ctypes.c_int()
        check(self.ctx.L.hb_mds_hxs_inertia(self.h, ctypes.byref(a), ctypes.byref(b)), "hb_mds_hxs_inertia")
        if b.value > 0:
            return -1
        return n_neg + a.value

    def solveCompressed(self, rx, ryc, ryd, dx, dyc, dyd) -> bool:
        rc = self.ctx.L.hb_mds_solve_compressed(self.h, self.linSys.h, *[_ptr(t) for t in (rx, ryc, ryd, dx, dyc, dyd)])
        if rc == -4:
            return False
        check(rc, "hb_mds_solve_compressed")
        return True

    def Msys(self) -> np.ndarray:
        N = self.nxd + self.neq + self.nineq
        out = np.empty(N * N, dtype=np.float64)
        check(self.ctx.L.hb_memcpy_d2h(self.ctx.h, out.ctypes.data_as(ctypes.c_void_p), ctypes.c_void_p(self.linSys._mptr), 8 * N * N), "memcpy")
        self.ctx.sync()
        return out.reshape(N, N)


class KKTLinSysDense:
    """hiopKKTLinSysDenseXYcYd (form="XYcYd") / hiopKKTLinSysDenseXDYcYd (form="XDYcYd"), src/Optimization/hiopKKTLinSysDense.hpp:
    the whole (nx + duals)^2 Newton KKT matrix assembled and factorized on the device (B1 solver)."""

    def __init__(self, ctx: Context, nx: int, neq: int, nineq: int, form: str = "XYcYd", mode: int = _lib.HB_FACT_BUNCH_KAUFMAN):
        assert form in ("XYcYd", "XDYcYd")
        self.ctx, self.nx, self.neq, self.nineq = ctx, nx, neq, nineq
        self.form = 0 if form == "XYcYd" else 1
        self.N = nx + neq + nineq + (nineq if self.form else 0)
        self.linSys = LinSolverSymDense(ctx, self.N, mode)          # owns sysMatrix(); build_kkt_matrix fills it in place
        self.Dx, self.Dd, self.work = ctx.zeros(nx), ctx.zeros(nineq), ctx.zeros(self.N)

    def close(self):
        self.linSys.close()

    def build_kkt_matrix(self, H, Jc, Jd, it: dict, pat: dict, deltas):
        dwx, dwd, dcc, dcd = deltas
        check(self.ctx.L.hb_densekkt_build(self.ctx.h, self.form, self.nx, self.neq, self.nineq, _ptr(H), _ptr(Jc), _ptr(Jd), _ptr(it["zl"]),
                                           _ptr(it["sxl"]), _ptr(it["zu"]), _ptr(it["sxu"]), _ptr(pat["ixl"]), _ptr(pat["ixu"]), _ptr(it["vl"]),
                                           _ptr(it["sdl"]), _ptr(it["vu"]), _ptr(it["sdu"]), _ptr(pat["idl"]), _ptr(pat["idu"]), _ptr(dwx), _ptr(dwd),
                                           _ptr(dcc), _ptr(dcd), _ptr(self.Dx), _ptr(self.Dd), ctypes.c_void_p(self.linSys._mptr)), "hb_densekkt_build")

    def Msys(self) -> np.ndarray:
        out = np.zeros((self.N, self.N))
        self.ctx.sync()
        check(self.ctx.L.hb_memcpy_d2h(self.ctx.h, out.ctypes.data_as(ctypes.c_void_p), ctypes.c_void_p(self.linSys._mptr), 8 * self.N * self.N), "memcpy")
        self.ctx.sync()
        return out

    def factorize(self) -> int:
        """matrixChanged(): number of negative eigenvalues, -1 if singular."""
        return self.linSys.matrixChanged()

    def solveCompressed(self, rx, rd, ryc, ryd, dx, dd, dyc, dyd) -> bool:
        rc = self.ctx.L.hb_densekkt_solve_compressed(self.ctx.h, self.linSys.h, self.form, self.nx, self.neq, self.nineq, _ptr(rx), _ptr(rd), _ptr(ryc),
                                                     _ptr(ryd), _ptr(dx), _ptr(dd), _ptr(dyc), _ptr(dyd), _ptr(self.work))
        if rc == -4:
            return False
        check(rc, "hb_densekkt_solve_compressed")
        return True
