"""Cost of condensing in column chunks under a bounded int8 slice buffer (hb_ctx_set_oz_workspace_limit), one JSON line per point.

  python tools/bench_oz_chunks.py [--steps 20] [--out FILE]

Bench size (n = 1e6, m = 1000, l = 6, the inputs of bench.py): for the budgets unlimited / 4 / 2 / 1 GiB / 512 MiB, in the default
condensation mode, the step time (update + solveCompressed, CUDA events over --steps steps), the summed device time of the int8 GEMM
(k_oz_gemm) and slicing (k_oz_slice) kernels per step (torch.profiler, mean over --prof-steps steps of their own), the chunk count and
the relative residual of the compressed KKT system evaluated with torch FP64 operators that never see N (bench.independent_kkt_residual).
The budgets are swept --rounds times, so the spread between rounds shows the noise.
Then one step of n = 4e6, m = 4000 on one GPU in the default mode when the device has the free memory for it (the Jacobian alone is
128 GB), otherwise a line that says it was not run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from hiop_b200.engine import Context, KKTLinSysLowRank  # noqa: E402

GIB = 1 << 30


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "unavailable"
    return info


def setup(ctx, n, m, l):
    T = bench.make_device_problem(ctx, torch, n, n, m, l, 0, 1, None)
    k = KKTLinSysLowRank(ctx, n, T["m_eq"], T["m_ineq"], max(l, 1))
    k.set_patterns(T["ixl"], T["ixu"], T["idl"], T["idu"])
    k.set_jacobian(T["J"][:T["m_eq"]], T["J"][T["m_eq"]:])
    k.set_secant(1.0, T["St"] if l else None, T["Yt"] if l else None, T["L"], T["D"])
    out = {"rx": ctx.zeros(n), "dx": ctx.zeros(n), "dyc": ctx.zeros(T["m_eq"]), "dyd": ctx.zeros(T["m_ineq"])}

    def step():
        out["rx"].copy_(T["rx"])
        k.update(T["zl"], T["sxl"], T["zu"], T["sxu"], T["vl"], T["sdl"], T["vu"], T["sdu"])
        assert k.solveCompressed(out["rx"], T["ryc"], T["ryd"], out["dx"], out["dyc"], out["dyd"])
    return T, k, out, step


def kernel_ms(step, nsteps):
    """mean device time per step of each kernel family, from profiled steps of their own"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(nsteps):
            step()
        torch.cuda.synchronize()
    sums = {"k_oz_gemm": 0.0, "k_oz_slice": 0.0}
    for ev in prof.key_averages():
        for name in sums:
            if name in ev.key:
                sums[name] += ev.device_time_total / 1e3 / nsteps      # us -> ms
    return sums


def bench_point(ctx, T, k, out, step, steps, prof_steps, tag, extra):
    for _ in range(3):
        step()
    k.check()
    ctx.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    ctx.sync()
    torch.cuda.synchronize()
    k.check()
    ms_step = e0.elapsed_time(e1) / steps
    resid = bench.independent_kkt_residual(torch, None, 1, T, 1.0, out["dx"], out["dyc"], out["dyd"])
    kms = kernel_ms(step, prof_steps)
    k.check()
    rec = {"point": tag, **extra, "chunks": k.condense_chunks(), "mode": k.condense_mode_used(), "fallbacks": k.fallback_count(),
           "ms_per_step": ms_step, "steps": steps, "gemm_ms": kms["k_oz_gemm"], "slice_ms": kms["k_oz_slice"], "profiled_steps": prof_steps,
           "kkt_residual_rel_independent_operators": resid}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--prof-steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2, help="sweeps over the budgets (their spread is the noise of the numbers)")
    ap.add_argument("--skip-large", action="store_true")
    args = ap.parse_args()
    fh = open(args.out, "w") if args.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if fh:
            fh.write(line + "\n")
            fh.flush()

    dev = device_info()
    ctx = Context(0)
    with ctx:
        n, m, l = 1_000_000, 1000, 6
        T, k, out, step = setup(ctx, n, m, l)
        for rnd in range(args.rounds):
            for name, b in (("unlimited", 0), ("4GiB", 4 * GIB), ("2GiB", 2 * GIB), ("1GiB", GIB), ("512MiB", GIB // 2)):
                ctx.set_oz_workspace_limit(b)
                emit(bench_point(ctx, T, k, out, step, args.steps, args.prof_steps, "bench_size",
                                 {"round": rnd, "n": n, "m": m, "l": l, "budget": name, "budget_bytes": b, **dev}))
        ctx.set_oz_workspace_limit(0)
        k.close()
        del T, out, step
        torch.cuda.empty_cache()
        ctx.sync()

        n, m, l = 4_000_000, 4000, 6
        free, _ = torch.cuda.mem_get_info(0)
        need = 8 * (m + 2 * l) * n + 40 * 8 * n + 4 * GIB      # J, S, Y + the n-vectors of the step and the residual + headroom
        if args.skip_large or free < need:
            emit({"point": "large_one_gpu", "n": n, "m": m, "l": l, **dev,
                  "not_run": f"{free / 1e9:.0f} GB free, about {need / 1e9:.0f} GB needed" if not args.skip_large else "skipped"})
        else:
            T, k, out, step = setup(ctx, n, m, l)
            emit(bench_point(ctx, T, k, out, step, 1, 1, "large_one_gpu", {"n": n, "m": m, "l": l, "budget": "auto", **dev}))
            k.close()
    ctx.close()
    if fh:
        fh.close()


if __name__ == "__main__":
    main()
