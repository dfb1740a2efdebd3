#!/usr/bin/env python
"""bench.py -- KKT systems/sec (assemble + factor + solve) on the synthetic NlpDenseConsEx2 generalisation.

One "step" = one complete condensed KKT system of HiOp's quasi-Newton path, exactly the work of
hiopKKTLinSysLowRank::update + solveCompressed (src/Optimization/hiopKKTLinSys.cpp:1057-1190):
   D_x / DhInv build -> V (compact BFGS inner matrix) -> N = J (B_k+D_x)^{-1} J^T + D_d^{-1}  (one FP64 DMMA pass over J)
   -> equilibrated Cholesky of N -> rhs = J H^{-1} rx - [ryc;ryd] -> solve with residual refinement -> dx, dyc, dyd.
Nothing is cached across steps (the factor is recomputed every step like the reference does).

Workload (BASELINE.json configs[1]): n = 1e6, m = 1000 (500 eq + 500 ineq), l = 6, FP64, synthetic data of the
distributions in SURVEY.md 8(d). At N GPUs the n (column) dimension is sharded like the reference's MPI layout and the
condensed (m+2l)^2 block is all-reduced with NCCL: strong scaling (total work fixed).

  python bench.py [--gpus N] [--steps K] [--warmup W]            this repo's engine (one rank per GPU under torchrun)
  python bench.py --impl reference [...]                          the reference's own CPU path (oracle/_ref) on host cores
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_FULL, M_FULL, L_MEM = 1_000_000, 1000, 6
METRIC = "KKT systems/sec (assemble+factor+solve)"
UNIT = "systems/s"
FP64_DMMA_PEAK_TFLOPS = 37.15   # measured on this pool's B200 with tools/microbench_fp64.cu (profiles/microbench_fp64_r01.txt)


def flops_syrk(n, Ma):
    """algorithmic flops of the condensation: n*Ma*(Ma+1) (mul+add on the upper triangle incl. diagonal), SURVEY 8(d)"""
    return float(n) * Ma * (Ma + 1)


def algorithmic_bytes(n, m, l):
    """ideal bytes of one system, SURVEY 8(d)"""
    return 8.0 * (3.0 * m * n + 6.0 * l * n + 10.0 * n) + 8.0 * (3.0 * m * m + 4.0 * l * m)


# -----------------------------------------------------------------------------------------------------------------
# reference / CPU arm
# -----------------------------------------------------------------------------------------------------------------
def workload_string(n, m, l):
    m_ineq = m // 2
    return (f"synthetic NlpDenseConsEx2 generalisation n={n} m={m} (m_eq={m - m_ineq}, m_ineq={m_ineq}) l={l}: "
            "quasi-Newton condensed KKT, update+condense+Cholesky+solve every step")


def cpu_system_time_on(P, repeat: int = 1):
    """Times the reference's update + solveCompressed on the host problem P. Returns (seconds per system, kind)."""
    try:
        from oracle import ref
        use_ref = ref.available()
        if use_ref:
            ref.lib()
    except Exception:
        use_ref = False
    ts = []
    l = P.St.shape[0]
    if use_ref:
        q = ref.RefQn(P.n, P.m_eq, P.m_ineq, max(l, 1), P.ixl, P.ixu, P.idl, P.idu)
        q.set_jac(P.Jc, P.Jd)
        q.set_secant(P.sigma, P.St, P.Yt, P.L, P.D)
        for _ in range(repeat):
            q.set_iterate(P.sxl, P.sxu, P.zl, P.zu, P.sdl, P.sdu, P.vl, P.vu)
            t0 = time.perf_counter()
            q.update()
            q.solve_compressed(P.rx, P.ryc, P.ryd)
            ts.append(time.perf_counter() - t0)
        q.close()
        return min(ts), "reference"
    from oracle import kkt_oracle as ko
    for _ in range(repeat):
        t0 = time.perf_counter()
        Dx, DhInv, Dd, Dd_inv = ko.kkt_update(P.zl, P.sxl, P.zu, P.sxu, P.ixl, P.ixu, P.vl, P.sdl, P.vu, P.sdu, P.idl, P.idu, P.sigma)
        st = ko.QnState(P.Jc, P.Jd, DhInv, Dd_inv, P.St, P.Yt, P.L, P.D, P.sigma)
        ko.solve_compressed(st, P.rx, P.ryc, P.ryd)
        ts.append(time.perf_counter() - t0)
    return min(ts), "port"


def cpu_system_time(n_sample: int, m: int, l: int, repeat: int = 1):
    from hiop_b200 import synth
    return cpu_system_time_on(synth.make_qn_problem(n_sample, m, l, seed=1234), repeat)


def cpu_extrapolate(n1: int, n2: int, n_full: int = N_FULL, m: int = M_FULL, l: int = L_MEM):
    """Two sampled sizes -> t(n) = a + b*n (a: the m^3 factor/solve part, b: the n-linear condensation + gemv part);
    returns (t(n_full), t1, t2, kind)."""
    t1, kind = cpu_system_time(n1, m, l)
    t2, kind = cpu_system_time(n2, m, l)
    b = max((t2 - t1) / (n2 - n1), 0.0)
    a = max(t1 - b * n1, 0.0)
    return a + b * n_full, t1, t2, kind


def cpu_baseline(n_sample: int, n: int = N_FULL, m: int = M_FULL, l: int = L_MEM):
    """Bounded sample for the engine line (the full-size reference measurement is `bench.py --impl reference`)."""
    cores = os.cpu_count() or 1
    os.environ.setdefault("OPENBLAS_NUM_THREADS", str(cores))
    t_full, t1, t2, kind = cpu_extrapolate(n_sample // 2, n_sample, n, m, l)
    return {"value": 1.0 / t_full, "unit": UNIT, "cores": cores, "kind": kind, "extrapolated": True,
            "sample": f"the reference's update+solveCompressed on {n_sample // 2} and {n_sample} of {n} columns (all m={m} rows, "
                      f"l={l}): {t1:.2f} s and {t2:.2f} s measured, EXTRAPOLATED as a + b*n to n={n} (the condensation triple "
                      f"loop, >95% of the time, is single-threaded in the reference; BLAS/LAPACK parts use {cores} OpenBLAS threads); "
                      "`bench.py --impl reference` times one full-size system instead",
            "seconds_full_extrapolated": t_full}


def cpu_optimised_system(P, threads: int):
    """The same update + solveCompressed with an optimised CPU condensation: rows scaled by sqrt(DhInv), then DSYRK / DGEMM from the
    box's threaded OpenBLAS in column chunks, DPOSVX for the m x m system -- what SURVEY 8(d) / BASELINE.md ask for next to the naive
    triple loop. Returns (seconds, dx, dyc, dyd)."""
    import scipy.linalg.blas as blas
    from oracle import kkt_oracle as ko

    def syrk_blas(X, d, beta=0.0, W=None, alpha=1.0):
        X = np.ascontiguousarray(X)
        k, n = X.shape
        step = 131072
        if k <= 32 or (d < 0).any():          # small (V blocks) or indefinite weights: plain DGEMM
            out = np.zeros((k, k))
            for c0 in range(0, n, step):
                out += (X[:, c0:c0 + step] * d[c0:c0 + step]) @ X[:, c0:c0 + step].T
        else:
            out = np.zeros((k, k), order="F")
            sd = np.sqrt(d)
            for c0 in range(0, n, step):
                B = X[:, c0:c0 + step] * sd[c0:c0 + step]
                # B is C-ordered (k x w) = Fortran (w x k): a^T a = B B^T, upper triangle
                out = blas.dsyrk(1.0, B.T, beta=1.0, c=out, trans=1, lower=0, overwrite_c=1)
            out = np.triu(out) + np.triu(out, 1).T
        res = alpha * out
        if W is not None and beta != 0.0:
            res += beta * W
        return np.ascontiguousarray(res)

    def gemm_blas(S, d, X):
        S = np.ascontiguousarray(S)
        X = np.ascontiguousarray(X)
        n = S.shape[1]
        out = np.zeros((S.shape[0], X.shape[0]))
        step = 131072
        for c0 in range(0, n, step):
            out += (S[:, c0:c0 + step] * d[c0:c0 + step]) @ X[:, c0:c0 + step].T
        return out

    saved = (ko.symm_mat_diag_mat_trans, ko.mat_diag_mat_trans)
    ko.symm_mat_diag_mat_trans, ko.mat_diag_mat_trans = syrk_blas, gemm_blas
    try:
        t0 = time.perf_counter()
        Dx, DhInv, Dd, Dd_inv = ko.kkt_update(P.zl, P.sxl, P.zu, P.sxu, P.ixl, P.ixu, P.vl, P.sdl, P.vu, P.sdu, P.idl, P.idu, P.sigma)
        st = ko.QnState(P.Jc, P.Jd, DhInv, Dd_inv, P.St, P.Yt, P.L, P.D, P.sigma)
        dx, dyc, dyd, _ = ko.solve_compressed(st, P.rx, P.ryc, P.ryd)
        return time.perf_counter() - t0, dx, dyc, dyd
    finally:
        ko.symm_mat_diag_mat_trans, ko.mat_diag_mat_trans = saved


def run_reference(args):
    """The reference's own CPU path (oracle/_ref: hiopKKTLinSysLowRank::update + solveCompressed, unmodified) on the box's host cores.
    One step of this workload costs several minutes of CPU time (the condensation is a single-threaded triple loop), so whatever
    --steps/--warmup ask for, exactly ONE full-size system is timed and reported (steps = 1, warmup = 0); the quick two-sample fit of
    round 1 is kept as a cross-check field only. HB_REF_MAX_SECONDS (default 1500) bounds the run: if the fit predicts more, the
    sampled estimate is reported instead and marked as such."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    os.environ.setdefault("OPENBLAS_NUM_THREADS", str(cores))
    from hiop_b200 import synth
    n, m, l = args.n, args.m, args.l
    workload = workload_string(n, m, l)
    t_fit, t1, t2, kind = cpu_extrapolate(max(2000, n // 200), max(4000, n // 100), n, m, l)
    budget = float(os.environ.get("HB_REF_MAX_SECONDS", "1500"))
    line = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps_requested": args.steps, "warmup_requested": args.warmup,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic"}
    cross = {"seconds_full_from_two_samples": t_fit, "samples": [max(2000, n // 200), max(4000, n // 100)], "seconds": [t1, t2]}
    if t_fit <= budget and not args.ref_sampled:
        P = synth.make_qn_problem(n, m, l, seed=1234)
        t_full, kind = cpu_system_time_on(P)
        t_opt = None
        try:
            t_opt, dxo, _, _ = cpu_optimised_system(P, cores)
        except Exception as e:  # noqa: BLE001
            cross["optimised_error"] = repr(e)[:200]
        val = 1.0 / t_full
        sample = (f"ONE full-size system (n={n}, m={m}, l={l}) through the reference's own hiopKKTLinSysLowRank::update + solveCompressed "
                  f"({kind}): {t_full:.1f} s measured, nothing extrapolated; requested steps/warmup ({args.steps}/{args.warmup}) capped to 1/0")
        line.update({"value": val, "steps": 1, "warmup": 0, "ms_per_step": t_full * 1e3,
                     "config": {"workload": workload, "sampled": False},
                     "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
                     "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     "cross_check_sampled_fit": cross})
        if t_opt is not None:
            line["cpu_baseline_optimised"] = {"value": 1.0 / t_opt, "unit": UNIT, "cores": cores, "kind": "port",
                                              "seconds": t_opt, "sample": "the same full-size system with the condensation as row scaling + OpenBLAS DSYRK/DGEMM "
                                              f"({cores} threads) and DPOSVX; not the reference's code path"}
    else:
        val = 1.0 / t_fit
        line.update({"value": val, "steps": 1, "warmup": 0, "ms_per_step": t_fit * 1e3, "extrapolated": True,
                     "config": {"workload": workload, "sampled": True},
                     "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind,
                                      "sample": f"EXTRAPOLATED a + b*n from {cross['samples']} columns ({t1:.2f} s, {t2:.2f} s): a full-size system would exceed "
                                                f"HB_REF_MAX_SECONDS={budget:.0f}"},
                     "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     "cross_check_sampled_fit": cross})
    print(json.dumps(line))
    return 0


# -----------------------------------------------------------------------------------------------------------------
# GPU arm
# -----------------------------------------------------------------------------------------------------------------
DUMP_MAX_ENTRIES = 1 << 21     # per array: three float64 outputs stay within 48 MB


def dump_outputs(directory, arrays):
    """--dump-outputs: writes each array as <directory>/<name>.npy in float64. An array longer than DUMP_MAX_ENTRIES is written as its
    entries at DUMP_MAX_ENTRIES fixed positions (sorted, drawn with seed 0), the same positions for every run of the same size."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float64).reshape(-1)
        if a.size > DUMP_MAX_ENTRIES:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ENTRIES, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: NVML from a thread every 5 ms (an nvidia-smi
    subprocess needs >100 ms per sample, longer than a short timed region), nvidia-smi -lms as the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.idx = device_index
        self.p = None
        self.f = None
        self.thread = None
        self.samples = []
        self.smax = None
        self.reason_bits = 0
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES remaps cuda indices; resolve through the PCI bus id of the torch device
            import torch
            bus = getattr(torch.cuda.get_device_properties(device_index), "pci_bus_id", None)
            self.h = None
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    h = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if int(pynvml.nvmlDeviceGetPciInfo(h).bus) == int(bus):
                        self.h, self.idx = h, i
            if self.h is None:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _loop(self):
        nv = self.nvml
        while not self._stop:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                try:
                    self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                except Exception:
                    pass
            time.sleep(0.005)

    def start(self):
        if self.nvml is not None:
            import threading
            self._stop = False
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
            return
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.thread is not None:
            self._stop = True
            self.thread.join(timeout=2)
            nv = self.nvml
            names = (("hw_slowdown", getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8)),
                     ("hw_thermal_slowdown", getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)),
                     ("sw_thermal_slowdown", getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)),
                     ("sw_power_cap", getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)))
            reasons = sorted(n for n, bit in names if self.reason_bits & bit)
            sm_sorted = sorted(self.samples)
            load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
            return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": self.smax, "reasons": reasons,
                    "samples": len(self.samples), "source": "nvml"}
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, smax, reasons = [], None, set()
        for r in rows:
            try:
                r = [x.strip() for x in r]
                sm.append(float(r[1]))
                smax = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        # under load = upper half of the samples
        sm_sorted = sorted(sm)
        load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvidia-smi"}


def make_device_problem(ctx, torch, n_local, n_total, m, l, rank, world, dist):
    """Synthetic inputs generated directly in HBM (same distributions as hiop_b200.synth; torch RNG)."""
    dev = ctx.device
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    m_ineq = m // 2
    m_eq = m - m_ineq
    T = {}
    with torch.cuda.stream(ctx.stream):
        J = torch.empty((m, n_local), dtype=torch.float64, device=dev)
        rows_per = 50
        for r0 in range(0, m, rows_per):            # chunked: keeps the transient fp64 RNG buffers small
            r1 = min(m, r0 + rows_per)
            J[r0:r1].normal_(0.0, 1.0 / np.sqrt(n_total), generator=g)
        J[0].fill_(1.0)
        T["J"] = J

        def U(k):
            return torch.empty(k, dtype=torch.float64, device=dev).uniform_(1e-3, 1.0, generator=g)
        T["ixl"] = torch.ones(n_local, dtype=torch.float64, device=dev)
        T["ixu"] = (torch.rand(n_local, dtype=torch.float64, device=dev, generator=g) < 0.1).to(torch.float64)
        T["sxl"], T["zl"] = U(n_local), U(n_local)
        T["sxu"], T["zu"] = U(n_local) * T["ixu"], U(n_local) * T["ixu"]
        T["rx"] = torch.empty(n_local, dtype=torch.float64, device=dev).normal_(generator=g)
        St = torch.empty((l, n_local), dtype=torch.float64, device=dev).normal_(generator=g)
        Yt = St * torch.empty((l, n_local), dtype=torch.float64, device=dev).uniform_(0.5, 2.0, generator=g)
        T["St"], T["Yt"] = St, Yt
        # replicated (m-sized) data: same seed on every rank
        g2 = torch.Generator(device=dev)
        g2.manual_seed(99)

        def U2(k):
            return torch.empty(k, dtype=torch.float64, device=dev).uniform_(1e-3, 1.0, generator=g2)
        T["idl"] = torch.ones(m_ineq, dtype=torch.float64, device=dev)
        T["idu"] = (torch.rand(m_ineq, dtype=torch.float64, device=dev, generator=g2) < 0.1).to(torch.float64)
        T["sdl"], T["vl"] = U2(m_ineq), U2(m_ineq)
        T["sdu"], T["vu"] = U2(m_ineq) * T["idu"], U2(m_ineq) * T["idu"]
        T["ryc"] = torch.empty(m_eq, dtype=torch.float64, device=dev).normal_(generator=g2)
        T["ryd"] = torch.empty(m_ineq, dtype=torch.float64, device=dev).normal_(generator=g2)
        SY = St @ Yt.T                               # input generation only (L, D of the secant state)
        if world > 1:
            dist.all_reduce(SY)
        SY = SY.cpu().numpy()
    ctx.sync()
    T["L"], T["D"] = np.tril(SY, -1).copy(), np.diag(SY).copy()
    T["m_eq"], T["m_ineq"] = m_eq, m_ineq
    return T


def independent_kkt_residual(torch, dist, world, T, sigma, dx, dyc, dyd):
    """Parity gate of SURVEY 8(d), outside the timed region: relative residual of the 3-block compressed KKT system evaluated with
    operators that are NOT the engine's -- torch FP64 matmuls (cuBLAS) for J and the compact BFGS form of B assembled here from S, Y, L, D --
    so neither the condensed matrix, its factor nor any hiop_b200 kernel takes part. n-sharded: the l- and m-sized pieces are
    all-reduced with torch.distributed."""
    def allred(t, op=None):
        if world > 1:
            dist.all_reduce(t, op=op or dist.ReduceOp.SUM)
        return t
    J, St, Yt = T["J"], T["St"], T["Yt"]
    m_eq = T["m_eq"]
    l = St.shape[0]
    Dx = T["zl"] / T["sxl"] + torch.where(T["ixu"] == 1.0, T["zu"] / torch.where(T["ixu"] == 1.0, T["sxu"], torch.ones_like(T["sxu"])), torch.zeros_like(T["zu"]))
    Dd = T["vl"] / T["sdl"] + torch.where(T["idu"] == 1.0, T["vu"] / torch.where(T["idu"] == 1.0, T["sdu"], torch.ones_like(T["sdu"])), torch.zeros_like(T["vu"]))
    # B dx = sigma dx - [sigma S^T, Y^T] M^-1 [sigma S dx; Y dx],  M = [[sigma S S^T, L], [L^T, -D]]
    Bdx = sigma * dx
    if l:
        SS = allred(St @ St.T)
        Lm = torch.from_numpy(T["L"]).to(dx.device)
        Dm = torch.from_numpy(T["D"]).to(dx.device)
        M = torch.cat([torch.cat([sigma * SS, Lm], 1), torch.cat([Lm.T, -torch.diag(Dm)], 1)], 0)
        u = allred(torch.cat([sigma * (St @ dx), Yt @ dx]))
        p = torch.linalg.solve(M, u)
        Bdx = Bdx - (sigma * (St.T @ p[:l]) + Yt.T @ p[l:])
    dy = torch.cat([dyc, dyd])
    r1 = Bdx + Dx * dx + J.T @ dy - T["rx"]
    Jdx = allred(J @ dx)
    r2 = Jdx[:m_eq] - T["ryc"]
    r3 = Jdx[m_eq:] - dyd / Dd - T["ryd"]
    num = allred(r1.abs().max().reshape(1).clone(), dist.ReduceOp.MAX if world > 1 else None)
    den = allred(T["rx"].abs().max().reshape(1).clone(), dist.ReduceOp.MAX if world > 1 else None)
    num = max(float(num), float(r2.abs().max()) if r2.numel() else 0.0, float(r3.abs().max()) if r3.numel() else 0.0)
    den = max(float(den), float(T["ryc"].abs().max()) if m_eq else 0.0, float(T["ryd"].abs().max()) if T["m_ineq"] else 0.0)
    return num / den


def run_engine(args):
    import torch
    import torch.distributed as dist
    from hiop_b200.engine import Context, KKTLinSysLowRank

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
    ctx = Context(local_rank)
    if world > 1:
        uid = [ctx.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.init_comm(world, rank, uid[0])

    n, m, l = args.n, args.m, args.l
    n_local = n // world + (1 if rank < n % world else 0)
    T = make_device_problem(ctx, torch, n_local, n, m, l, rank, world, dist)
    m_eq, m_ineq = T["m_eq"], T["m_ineq"]
    k = KKTLinSysLowRank(ctx, n_local, m_eq, m_ineq, max(l, 1))
    k.set_patterns(T["ixl"], T["ixu"], T["idl"], T["idu"])
    k.set_jacobian(T["J"][:m_eq], T["J"][m_eq:])
    k.set_secant(1.0, T["St"] if l else None, T["Yt"] if l else None, T["L"], T["D"])
    ctx.enable_timing(True)
    rx_work = ctx.zeros(n_local)
    dx, dyc, dyd = ctx.zeros(n_local), ctx.zeros(m_eq), ctx.zeros(m_ineq)

    def set_mode(name):
        if name == "dmma":
            k.set_condense_mode(0)
        elif name == "auto":
            k.set_condense_mode(-1)
        else:
            k.set_condense_mode(int(name[2]))

    def step():
        # nothing here synchronises with the host: update + (implicit, asynchronous) condensation + solve are only enqueued;
        # a breakdown would be reported by k.check() after the timed region
        rx_work.copy_(T["rx"])                        # solveCompressed clobbers rx (like the reference)
        k.update(T["zl"], T["sxl"], T["zu"], T["sxu"], T["vl"], T["sdl"], T["vu"], T["sdu"])
        ok = k.solveCompressed(rx_work, T["ryc"], T["ryd"], dx, dyc, dyd)
        assert ok

    def barrier():
        if world > 1:
            dist.barrier()
        ctx.sync()
        torch.cuda.synchronize()

    def timed_loop(mode_name, steps, sample_clocks):
        set_mode(mode_name)
        for _ in range(max(args.warmup, 3)):
            step()
        k.check()
        barrier()
        sampler = ClockSampler(local_rank) if sample_clocks else None
        if sampler is not None and rank == 0:
            sampler.start()
        launches0 = ctx.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kernel_ms = []
        e0.record()
        for _ in range(steps):
            step()
            kernel_ms.append(ctx.last_syrk_ms())
        e1.record()
        barrier()
        k.check()
        launches = ctx.launch_count() - launches0
        clocks = sampler.stop() if (sampler is not None and rank == 0) else None
        ms_total = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms_total], dtype=torch.float64, device=ctx.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_total = float(t.item())
        nref, resid = k.last_solve_stats()
        return {"ms_step": ms_total / steps, "kernel_ms": statistics.mean(kernel_ms), "launches": launches, "clocks": clocks,
                "mode": k.condense_mode_used(), "nref": nref, "resid": resid}

    with ctx:                                          # engine stream is torch's current stream: events see the kernels
        # roofline denominators measured now, on this device (the driver's MEASURED_PEAKS.json has no FP64 / int8 tensor entry)
        peak_dmma = ctx.microbench_peak(0)
        peak_i8 = ctx.microbench_peak(1)
        main = timed_loop(args.condense, args.steps, True)
        ctx.sync()
        if args.dump_outputs:
            # what solveCompressed handed back in the last timed step; dx is column-sharded like J, dyc / dyd are replicated
            outputs = {"dx": dx.cpu().numpy().copy(), "dyc": dyc.cpu().numpy().copy(), "dyd": dyd.cpu().numpy().copy()}
            if world > 1:
                parts = [None] * world
                dist.all_gather_object(parts, outputs["dx"])
                outputs["dx"] = np.concatenate(parts)
        kkt_resid_rel = independent_kkt_residual(torch, dist, world, T, 1.0, dx, dyc, dyd)
        # the other condensation kernel on the same workload (both modes belong in the record)
        other_name = "dmma" if main["mode"] != 0 else "oz8"
        other = timed_loop(other_name, max(3, min(args.steps, 10)), False)
        ctx.sync()
        kkt_resid_other = independent_kkt_residual(torch, dist, world, T, 1.0, dx, dyc, dyd)
        set_mode(args.condense)
        # ---- per-rank phase timeline of ONE extra step (events recorded inside the library; outside the timed region) ----
        for _ in range(2):
            step()
        barrier()
        ctx.phase_timeline(True)
        step()
        tl = ctx.phase_timeline(False)
        timeline = [tl]
        if world > 1:
            timeline = [None] * world
            dist.all_gather_object(timeline, tl)

        # ---- phase split: the solve alone on the cached factor (second right-hand side of the same KKT matrix) ----
        def solve_only():
            rx_work.copy_(T["rx"])
            assert k.solveCompressed(rx_work, T["ryc"], T["ryd"], dx, dyc, dyd)
        for _ in range(3):
            solve_only()
        barrier()
        es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        es0.record()
        for _ in range(10):
            solve_only()
        es1.record()
        barrier()
        solve_only_ms = es0.elapsed_time(es1) / 10
        if world > 1:
            t = torch.tensor([solve_only_ms], dtype=torch.float64, device=ctx.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            solve_only_ms = float(t.item())

        # ---- end to end through the host-buffer entry point (public API a HiOp adapter calls when mem_space is host) ----
        e2e = None
        # N>1: every rank uploads its own column shard from pinned host memory (bounded to 4 GB of pinned J per rank)
        if not args.no_e2e and (world == 1 or 8.0 * m * n_local <= 4.0e9):
            host = {}
            for key in ("zl", "sxl", "zu", "sxu", "vl", "sdl", "vu", "sdu", "rx", "ryc", "ryd"):
                host[key] = torch.empty(T[key].shape, dtype=torch.float64, pin_memory=True)
                host[key].copy_(T[key])
            Jh = torch.empty((m, n_local), dtype=torch.float64, pin_memory=True)
            Jh.copy_(T["J"])
            hdx = torch.empty(n_local, dtype=torch.float64, pin_memory=True)
            hyc = torch.empty(m_eq, dtype=torch.float64, pin_memory=True)
            hyd = torch.empty(m_ineq, dtype=torch.float64, pin_memory=True)
            ctx.sync()
            it = {kk: host[kk].numpy() for kk in ("zl", "sxl", "zu", "sxu", "vl", "sdl", "vu", "sdu")}
            Jn = Jh.numpy()

            def e2e_step():
                k.kkt_system_host(Jn[:m_eq], Jn[m_eq:], it, host["rx"].numpy(), host["ryc"].numpy(), host["ryd"].numpy(),
                                  hdx.numpy(), hyc.numpy(), hyd.numpy())
            e2e_steps = max(2, min(args.steps, 5))
            h2d = 8 * (m * n_local + 5 * n_local + 4 * m_ineq + m)   # this rank's bytes; the line reports the sum over ranks
            d2h = 8 * (n_local + m)
            if world > 1:
                t = torch.tensor([h2d, d2h], dtype=torch.float64, device=ctx.device)
                dist.all_reduce(t)
                h2d, d2h = int(t[0].item()), int(t[1].item())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            res = {}
            for name in ("auto", "oz8"):
                set_mode(name)
                e2e_step()
                barrier()
                e0.record()
                for _ in range(e2e_steps):
                    e2e_step()
                e1.record()
                barrier()
                ms_e = e0.elapsed_time(e1) / e2e_steps
                if world > 1:
                    t = torch.tensor([ms_e], dtype=torch.float64, device=ctx.device)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    ms_e = float(t.item())
                res[name] = (ms_e, k.condense_mode_used())
            set_mode(args.condense)
            best = min(res, key=lambda q: res[q][0])
            e2e = {"value": 1e3 / res[best][0], "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": res[best][0],
                   "steps": e2e_steps, "condense_mode": "fp64_dmma" if res[best][1] == 0 else f"int8_slices_{res[best][1]}",
                   "by_mode": {"host_default(fp64_dmma, J uploaded in 16 column chunks overlapped with the condensation)": res["auto"][0],
                               "int8_slices_8 (whole J uploaded first: the row scaling needs all columns)": res["oz8"][0]},
                   "note": "hb_lowrank_kkt_system_host: J (8 m n bytes) + iterate + rhs copied from pinned host memory every step; PCIe bound"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    Ma = m + 2 * l
    fl = flops_syrk(n_local, Ma)

    def kernel_roofline(res):
        mode, ms = res["mode"], res["kernel_ms"]
        if mode == 0:
            ach = fl / (ms * 1e-3) / 1e12
            return {"kernel": "k_syrk_ws (FP64 DMMA.8x8x4 condensation [J;S;Y] DhInv [J;S;Y]^T)", "bound": "tensor", "achieved": ach, "peak": peak_dmma,
                    "unit": "TFLOP/s", "frac": ach / peak_dmma, "traffic": None, "kernel_ms": ms, "kernel_share_of_step": ms / res["ms_step"],
                    "flops_per_launch": fl,
                    "peak_source": "FP64 tensor (DMMA) rate measured in this run by hb_microbench_peak(0): mma.sync.m8n8k4.f64 back to back on all SMs "
                                   "(MEASURED_PEAKS.json holds only HBM and bf16 numbers; tcgen05 has no f64 kind)"}
        ops = 2.0 * (mode * (mode + 1) // 2) * (Ma * (Ma + 1) / 2) * n_local
        Mpad = (Ma + 127) // 128 * 128
        ntiles = sum(1 for bi in range(Mpad // 128) for bj in range(2 * bi, Mpad // 64) if bj * 64 < Ma)
        ops_executed = 2.0 * (mode * (mode + 1) // 2) * ntiles * 128 * 64 * ((n_local + 127) // 128 * 128)
        ach = ops / (ms * 1e-3) / 1e12
        return {"kernel": f"k_oz_gemm<{mode}> (tcgen05.mma.kind::i8, {mode} int8 slices, TMA SWIZZLE_128B, TMEM accumulators)", "bound": "tensor",
                "achieved": ach, "peak": peak_i8, "unit": "TFLOP/s", "frac": ach / peak_i8, "traffic": None, "kernel_ms": ms,
                "kernel_share_of_step": ms / res["ms_step"], "flops_per_launch": ops, "executed_ops_per_launch": ops_executed,
                "executed_rate": ops_executed / (ms * 1e-3) / 1e12, "peak_nominal": 4500.0,
                "peak_source": "int8 tcgen05 rate measured in this run by hb_microbench_peak(1): tcgen05.mma.kind::i8 M=128 N=256 K=32 back to back on "
                               "resident operands, one CTA per SM (nominal dense int8 rate of B200: 4.5 POP/s)",
                "note": "achieved/peak count int8 operations (2 per MAC); the FP64 work the kernel stands in for is fp64_equivalent_flops",
                "fp64_equivalent_flops": fl, "fp64_equivalent_tflops_gemm_only": fl / (ms * 1e-3) / 1e12}

    roofline = kernel_roofline(main)
    if main["mode"] == 8 and n_local == N_FULL and m == M_FULL and l == L_MEM:
        # dram bytes of this kernel at this workload from the committed ncu --set full capture (NOT measured in this run)
        try:
            unit = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
            tot = 0.0
            for row in open(os.path.join(ROOT, "profiles", "ozgemm_r01_ncu_full.csv")):
                parts = [q.strip().strip('"') for q in row.strip().split(",")]
                if len(parts) == 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tot += float(parts[2]) * unit[parts[1]]
            if tot > 0:
                roofline["traffic"] = tot
                roofline["traffic_source"] = ("profiles/ozgemm_r01_ncu_full.csv (ncu --set full of the same kernel and workload, one launch, committed; not "
                                              "re-measured in this run; algorithmic operand bytes: 8 slices x 1012 x 1e6 = 8.1e9)")
        except Exception:
            pass
    roofline["hbm_algorithmic_GBs_whole_step"] = algorithmic_bytes(n_local, m, l) / (main["ms_step"] * 1e-3) / 1e9
    roofline["condense_mode"] = "fp64_dmma" if main["mode"] == 0 else f"int8_slices_{main['mode']}"
    mode_tag = {0: "f64 (exact, DMMA)", 6: "f64-emulated(int8x6)", 7: "f64-emulated(int8x7)", 8: "f64-emulated(int8x8)"}
    line = {"metric": METRIC, "value": 1e3 / main["ms_step"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": main["ms_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64" if main["mode"] == 0 else mode_tag[main["mode"]], "data": "synthetic",
            "config": {"workload": workload_string(n, m, l),
                       "parallelism": f"column-sharded x{world}" if world > 1 else "single GPU",
                       "l2": f"J is {8e-9 * m * n_local:.1f} GB per GPU, far larger than the 126 MB L2; no flush needed",
                       "refinement_steps_last": main["nref"], "residual_inf_last": main["resid"],
                       "kkt_residual_rel_independent_operators": kkt_resid_rel,
                       "timeline_ms_per_rank": [{q: round(v, 4) for q, v in t.items()} for t in timeline],
                       "kkt_residual_note": "max-norm residual of the compressed 3-block KKT system over max-norm rhs, evaluated with torch FP64 matmuls and a "
                                            "compact-BFGS operator assembled in bench.py (no hiop_b200 kernel, not the condensed matrix); gate 1e-8"},
            "phase_split": {"assemble+factor_ms": main["ms_step"] - solve_only_ms, "solve_on_cached_factor_ms": solve_only_ms,
                            "note": "solve_on_cached_factor = solveCompressed with a valid condensation (two sweeps over J, SPD solve, two (H+Dx)^-1 "
                                    "applications), timed separately over 10 calls; assemble+factor = step - that"},
            "condensed_factor": {"kernel": "equilibrated Cholesky of the m x m condensed matrix N (replicated on every rank)", "N": m,
                                 "ms": max(t["Cholesky"] for t in timeline),
                                 "tflops": (m ** 3 / 3.0) / (max(t["Cholesky"] for t in timeline) * 1e-3) / 1e12 if m else 0.0},
            "clocks": main["clocks"], "gpu_launches": main["launches"], "roofline": roofline,
            "other_mode": {"condense_mode": "fp64_dmma" if other["mode"] == 0 else f"int8_slices_{other['mode']}", "value": 1e3 / other["ms_step"],
                           "ms_per_step": other["ms_step"], "kkt_residual_rel_independent_operators": kkt_resid_other, "roofline": kernel_roofline(other)},
            "measured_peaks_in_run": {"fp64_dmma_tflops": peak_dmma, "int8_tcgen05_tops": peak_i8}}
    assert kkt_resid_rel <= 1e-8 and kkt_resid_other <= 1e-8, (kkt_resid_rel, kkt_resid_other)
    if e2e is not None:
        line["e2e"] = e2e
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline(args.cpu_sample, n, m, l)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


# -----------------------------------------------------------------------------------------------------------------
# MDS workload (BASELINE configs[2], re-stated as 3b in SURVEY 8(d)): synthetic mixed dense-sparse Newton KKT system,
# n_s sparse variables (diagonal Hessian block, ~5 nnz per column of the sparse Jacobian), n_d dense variables, m constraints.
# One step = hiopKKTLinSysCompressedMDSXYcYd::update + build_kkt_matrix + factorizeWithCurvCheck + solveCompressed
# (src/Optimization/hiopKKTLinSysMDS.cpp:155-403): assemble the (n_d+m)^2 condensed matrix, Bunch-Kaufman factor + inertia, solve.
# -----------------------------------------------------------------------------------------------------------------
MDS_METRIC = "MDS KKT systems/sec (assemble + symmetric-indefinite factor + solve)"


def mds_workload_string(nxs, nxd, neq, nineq, nnz_row):
    return (f"synthetic NlpMdsEx1 generalisation n_s={nxs} (diagonal Hessian block, sparse Jacobian {nnz_row} nnz/row) n_d={nxd} m={neq + nineq} "
            f"(m_eq={neq}, m_ineq={nineq}): condensed dense KKT of order {nxd + neq + nineq}, update+build_kkt_matrix+factor+inertia+solve every step")


def make_mds_device_problem(torch, ctx, nxs, nxd, neq, nineq, nnz_row, seed=42):
    dev = ctx.device
    g = torch.Generator(device=dev).manual_seed(seed)
    r = np.random.default_rng(seed)
    n = nxs + nxd
    f64 = dict(dtype=torch.float64, device=dev)

    def U(k, lo=1e-3, hi=1.0):
        return torch.empty(k, **f64).uniform_(lo, hi, generator=g)
    T = {}
    A = torch.randn(nxd, nxd, generator=g, **f64) / np.sqrt(max(nxd, 1))
    T["Hd"] = A @ A.T + torch.diag(U(nxd, 1e-2, 1.0))
    del A
    T["Hs"] = U(nxs, 0.1, 2.0)
    T["Jcd"] = torch.randn(neq, nxd, generator=g, **f64) / np.sqrt(max(nxd, 1))
    T["Jdd"] = torch.randn(nineq, nxd, generator=g, **f64) / np.sqrt(max(nxd, 1))

    def triplets(m):
        # sorted (row, col) triplets, nnz_row distinct columns per row
        cols = np.empty((m, nnz_row), dtype=np.int32)
        for i in range(m):
            cols[i] = np.sort(r.choice(nxs, nnz_row, replace=False))
        rows = np.repeat(np.arange(m, dtype=np.int32), nnz_row)
        return rows, cols.reshape(-1)
    T["iRc"], T["jCc"] = triplets(neq)
    T["iRd"], T["jCd"] = triplets(nineq)
    T["Jcs"] = torch.randn(T["iRc"].size, generator=g, **f64)
    T["Jds"] = torch.randn(T["iRd"].size, generator=g, **f64)
    T["ixl"] = torch.ones(n, **f64)
    T["ixu"] = (torch.rand(n, generator=g, **f64) < 0.2).to(torch.float64)
    T["idl"] = torch.ones(nineq, **f64)
    T["idu"] = (torch.rand(nineq, generator=g, **f64) < 0.2).to(torch.float64)
    T["sxl"], T["zl"] = U(n), U(n)
    T["sxu"], T["zu"] = U(n) * T["ixu"], U(n) * T["ixu"]
    T["sdl"], T["vl"] = U(nineq), U(nineq)
    T["sdu"], T["vu"] = U(nineq) * T["idu"], U(nineq) * T["idu"]
    T["dwx"], T["dwd"], T["dcc"], T["dcd"] = (torch.zeros(n, **f64), torch.zeros(nineq, **f64), torch.zeros(neq, **f64), torch.zeros(nineq, **f64))
    T["rx"] = torch.randn(n, generator=g, **f64)
    T["ryc"] = torch.randn(neq, generator=g, **f64)
    T["ryd"] = torch.randn(nineq, generator=g, **f64)
    torch.cuda.synchronize()
    return T


def mds_independent_residual(torch, T, nxs, nxd, neq, nineq, dx, dyc, dyd):
    """residual of the UNcondensed XYcYd system with torch operators (sparse COO mat-vecs for J_s, matmuls for the dense blocks)"""
    dev = dx.device
    Dx = T["zl"] / T["sxl"] + torch.where(T["ixu"] == 1.0, T["zu"] / torch.where(T["ixu"] == 1.0, T["sxu"], torch.ones_like(T["sxu"])), torch.zeros_like(T["zu"]))
    Dd = T["vl"] / T["sdl"] + torch.where(T["idu"] == 1.0, T["vu"] / torch.where(T["idu"] == 1.0, T["sdu"], torch.ones_like(T["sdu"])), torch.zeros_like(T["vu"]))
    Jcs = torch.sparse_coo_tensor(torch.from_numpy(np.stack([T["iRc"], T["jCc"]]).astype(np.int64)).to(dev), T["Jcs"], (neq, nxs))
    Jds = torch.sparse_coo_tensor(torch.from_numpy(np.stack([T["iRd"], T["jCd"]]).astype(np.int64)).to(dev), T["Jds"], (nineq, nxs))
    xs, xd = dx[:nxs], dx[nxs:]
    r1s = (T["Hs"] + Dx[:nxs] + T["dwx"][:nxs]) * xs + torch.sparse.mm(Jcs.t(), dyc[:, None])[:, 0] + torch.sparse.mm(Jds.t(), dyd[:, None])[:, 0] - T["rx"][:nxs]
    r1d = T["Hd"] @ xd + (Dx[nxs:] + T["dwx"][nxs:]) * xd + T["Jcd"].T @ dyc + T["Jdd"].T @ dyd - T["rx"][nxs:]
    r2 = torch.sparse.mm(Jcs, xs[:, None])[:, 0] + T["Jcd"] @ xd - T["dcc"] * dyc - T["ryc"]
    r3 = torch.sparse.mm(Jds, xs[:, None])[:, 0] + T["Jdd"] @ xd - (1.0 / (Dd + T["dwd"]) + T["dcd"]) * dyd - T["ryd"]
    num = max(float(r1s.abs().max()), float(r1d.abs().max()), float(r2.abs().max()), float(r3.abs().max()))
    den = max(float(T["rx"].abs().max()), float(T["ryc"].abs().max()), float(T["ryd"].abs().max()))
    return num / den


def run_mds(args):
    import torch
    from hiop_b200.engine import Context, KKTLinSysCompressedMDSXYcYd
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        # the MDS path stays on one GPU (north star): replicas only -- rank 0 measures, the others leave
        if int(os.environ.get("RANK", "0")) != 0:
            return 0
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    ctx = Context(local_rank)
    nxs, nxd, m = args.mds_ns, args.mds_nd, args.mds_m
    nineq = m // 2
    neq = m - nineq
    nnz_row = max(1, int(round(5.0 * nxs / max(m, 1))))          # ~5 nonzeros per column of the sparse Jacobian
    N = nxd + m
    with ctx:
        peak_dmma = ctx.microbench_peak(0)
        T = make_mds_device_problem(torch, ctx, nxs, nxd, neq, nineq, nnz_row)
        dx, dyc, dyd = ctx.zeros(nxs + nxd), ctx.zeros(neq), ctx.zeros(nineq)

        def run_mode(safe_mode, steps, clocks):
            k = KKTLinSysCompressedMDSXYcYd(ctx, nxs, nxd, neq, nineq, safe_mode=safe_mode)
            k.set_sparsity(T["iRc"], T["jCc"], T["iRd"], T["jCd"])
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            phase = np.zeros(3)

            def step(timed):
                if timed:
                    ev[0].record()
                k.update(T["zl"], T["sxl"], T["zu"], T["sxu"], T["ixl"], T["ixu"])
                k.build_kkt_matrix(T["Hd"], T["Hs"], T["Jcd"], T["Jdd"], T["Jcs"], T["Jds"], T["vl"], T["sdl"], T["vu"], T["sdu"], T["idl"], T["idu"],
                                   T["dwx"], T["dwd"], T["dcc"], T["dcd"])
                if timed:
                    ev[1].record()
                nneg = k.factorizeWithCurvCheck()
                if timed:
                    ev[2].record()
                assert nneg == neq + nineq, (nneg, neq + nineq)     # inertia the Newton iteration requires (hiopAlgFilterIPM.cpp:2084-2096)
                assert k.solveCompressed(T["rx"], T["ryc"], T["ryd"], dx, dyc, dyd)
                if timed:
                    ev[3].record()
                    torch.cuda.synchronize()
                    for q in range(3):
                        phase[q] += ev[q].elapsed_time(ev[q + 1])
            for _ in range(max(args.warmup, 3)):
                step(False)
            ctx.sync()
            torch.cuda.synchronize()
            sampler = ClockSampler(local_rank) if clocks else None
            if sampler:
                sampler.start()
            launches0 = ctx.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step(False)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            launches = ctx.launch_count() - launches0
            ck = sampler.stop() if sampler else None
            outputs = {"dx": dx.cpu().numpy().copy(), "dyc": dyc.cpu().numpy().copy(), "dyd": dyd.cpu().numpy().copy()} if args.dump_outputs else None
            step(True)      # one extra, phase-stamped step (events between the phases; not part of the timed region)
            resid = mds_independent_residual(torch, T, nxs, nxd, neq, nineq, dx, dyc, dyd)
            k.close()
            return {"ms_step": ms, "launches": launches, "clocks": ck, "phase_ms": {"assemble": phase[0], "factor+inertia": phase[1], "solve": phase[2]},
                    "resid": resid, "outputs": outputs}

        bk = run_mode(True, args.steps, True)
        nopiv = run_mode(False, max(3, min(args.steps, 10)), False)
    fl = N ** 3 / 3.0

    def roof(res, name):
        t = res["phase_ms"]["factor+inertia"]
        ach = fl / (t * 1e-3) / 1e12
        return {"kernel": name, "bound": "tensor", "achieved": ach, "peak": peak_dmma, "unit": "TFLOP/s", "frac": ach / peak_dmma, "traffic": None,
                "kernel_ms": t, "kernel_share_of_step": t / res["ms_step"], "flops_per_launch": fl,
                "peak_source": "FP64 tensor (DMMA) rate measured in this run by hb_microbench_peak(0); flops counted as N^3/3 like the reference (FLOPS_DPOTRF, "
                               "hiopLinSolverSymDenseMagma.cpp:155)"}
    line = {"metric": MDS_METRIC, "value": 1e3 / bk["ms_step"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": bk["ms_step"], "higher_is_better": True, "scaling": "replicas only (the MDS path stays on one GPU)", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": mds_workload_string(nxs, nxd, neq, nineq, nnz_row), "parallelism": "single GPU",
                       "l2": f"condensed matrix {8e-9 * N * N:.1f} GB, H_d {8e-9 * nxd * nxd:.1f} GB: far larger than the 126 MB L2; no flush needed",
                       "linear_solver": "Bunch-Kaufman LDL^T (safe mode, hiopLinSolverSymDenseMagmaBuKa role)", "phase_ms": bk["phase_ms"],
                       "kkt_residual_rel_independent_operators": bk["resid"]},
            "clocks": bk["clocks"], "gpu_launches": bk["launches"],
            "roofline": roof(bk, "cluster Bunch-Kaufman: k_bk_panel (16-CTA cluster) + k_gemm_pq<64> trailing updates (FP64 DMMA)"),
            "other_mode": {"linear_solver": "LDL^T without pivoting (linsol_mode=speculative, hiopLinSolverSymDenseMagmaNopiv role)", "value": 1e3 / nopiv["ms_step"],
                           "ms_per_step": nopiv["ms_step"], "phase_ms": nopiv["phase_ms"], "kkt_residual_rel_independent_operators": nopiv["resid"],
                           "roofline": roof(nopiv, "look-ahead LDL^T: k_diag128 + k_trsm_panel + k_gemm_pq<64> (FP64 DMMA)")},
            "measured_peaks_in_run": {"fp64_dmma_tflops": peak_dmma}}
    assert bk["resid"] <= 1e-8 and nopiv["resid"] <= 1e-8, (bk["resid"], nopiv["resid"])
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, bk["outputs"])
    if not args.no_cpu:
        line["cpu_baseline"] = mds_cpu_baseline(args, nnz_row)
    print(json.dumps(line))
    ctx.close()
    return 0


def mds_cpu_baseline(args, nnz_row):
    """Bounded sample: the oracle's restatement of build_kkt_matrix + DSYTRF/inertia + solveCompressed (pinned to the compiled reference by
    tests/test_oracle_vs_ref.py) on a 1/4-scale instance of the workload (n_d and m divided by 4 -> N/4, n_s / 4), LAPACK through scipy."""
    from hiop_b200 import synth
    from oracle import kkt_oracle as ko
    cores = os.cpu_count() or 1
    sc = 4
    nxs, nxd, m = args.mds_ns // sc, args.mds_nd // sc, args.mds_m // sc
    nineq = m // 2
    neq = m - nineq
    P = synth.make_mds_problem(nxs, nxd, neq, nineq, nnz_per_row=max(1, nnz_row // sc), seed=42)
    t0 = time.perf_counter()
    M, _, Hxs, _ = ko.mds_build_kkt_matrix(P)
    t1 = time.perf_counter()
    ret, fac = ko.mds_factorize_with_curv_check(M, Hxs)
    t2 = time.perf_counter()
    ko.mds_solve_compressed(P, fac, Hxs, P.rx, P.ryc, P.ryd)
    t3 = time.perf_counter()
    t = t3 - t0
    N = nxd + m
    return {"value": 1.0 / t, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"1/{sc}-scale instance (n_s={nxs}, n_d={nxd}, m={m}: N={N}) through the oracle's build_kkt_matrix ({t1 - t0:.1f} s) + LAPACK DSYTRF/inertia "
                      f"({t2 - t1:.1f} s) + solveCompressed ({t3 - t2:.2f} s); the factor scales as N^3: x{sc ** 3} at full size",
            "seconds_sample": t, "seconds_full_extrapolated_cubic": (t2 - t1) * sc ** 3 + (t1 - t0) * sc ** 2 + (t3 - t2) * sc ** 2}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    # --kkt-n/--kkt-m/--kkt-l: under `python -m torch.distributed.run`, argparse rejects "--n"/"--m" as ambiguous launcher
    # abbreviations before it reaches the script's own arguments, so the long spellings are the ones to use there
    ap.add_argument("--n", "--kkt-n", dest="n", type=int, default=int(os.environ.get("HB_BENCH_N", N_FULL)))
    ap.add_argument("--m", "--kkt-m", dest="m", type=int, default=int(os.environ.get("HB_BENCH_M", M_FULL)))
    ap.add_argument("--l", "--kkt-l", dest="l", type=int, default=int(os.environ.get("HB_BENCH_L", L_MEM)))
    ap.add_argument("--condense", default="auto", choices=["auto", "dmma", "oz6", "oz7", "oz8"],
                    help="GEMM part of the condensation: auto (library default), exact FP64 DMMA, or INT8-slice tcgen05 with 6/7/8 slices")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=20000, help="columns of the workload the CPU baseline leg runs")
    ap.add_argument("--workload", default="qn", choices=["qn", "mds"], help="qn: quasi-Newton condensed KKT (BASELINE configs[1], the headline); "
                    "mds: mixed dense-sparse Newton KKT (configs[2], one GPU)")
    ap.add_argument("--mds-ns", type=int, default=500000)
    ap.add_argument("--mds-nd", type=int, default=20000)
    ap.add_argument("--mds-m", type=int, default=2000)
    ap.add_argument("--ref-sampled", action="store_true", help="--impl reference: report the two-sample extrapolation instead of one full-size system")
    ap.add_argument("--dump-outputs", metavar="DIR", help="engine arms: after the timed steps, write dx, dyc and dyd of the last timed step as DIR/<name>.npy "
                    "(float64; arrays over 2^21 entries as a fixed, seeded sample) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the engine arms")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "mds":
        return run_mds(args)
    return run_engine(args)


if __name__ == "__main__":
    sys.exit(main())
