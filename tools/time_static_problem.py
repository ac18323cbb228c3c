"""Cost of the static problem entry points against the tip-load ones, on the same device-resident batch.

10^5 rods from sri_generate_rods (F_tip, M_tip ~ U(-1,1)^3 and its gravity fbar = (0, 0, -g), g ~ U(0,1)), H = (1, 1, 0.77),
ne = 4, zero initial guess, tol 1e-10, analytic Jacobian, at N = 16 and N = 32.  Three problems are solved and
differentiated (random cotangent, every gradient the problem has, refine_steps = 0 and 3):
    tip        sri_newton_static_shape / sri_static_shape_vjp (tip loads only)
    null       sri_newton_static_problem / sri_static_problem_vjp on the same rods, q0, Gamma, fbar, lbar NULL
    gravity    sri_newton_static_problem / sri_static_problem_vjp with the generator's fbar (and its gradient)
Each problem has its own handle, so that each keeps its Newton workspace and iteration graph (a handle reallocates them
when the set of optional inputs changes).  After a warm-up the nine timed operations alternate with CUDA events; best and
median over the repetitions are reported, with the Newton iteration count.  One JSON line per (N, problem, operation) on
stdout and, with --out, appended to that file; the card's name, power limit, maximum SM clock and the SM clock read right
after the timed loop are part of every line.

    python tools/time_static_problem.py [--out profiles/r06_static_problem.jsonl] [--reps 10]
"""
import argparse
import ctypes
import json
import statistics
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import SpectralRodIntegrator, _lib  # noqa: E402
from experimental_gpu_programming_for_a_spectral_numerical_integration_b200.api import _problem, _ptr, _report_dict  # noqa: E402
from time_vjp import event_ms  # noqa: E402

CONFIGS = [(16, 100_000), (32, 100_000)]
NE, H, TOL = 4, (1.0, 1.0, 0.77), 1e-10


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=30).stdout.strip()
    return {"card": torch.cuda.get_device_name(0), "power_limit_max_sm_clock_sm_clock": q}


def newton_null(h, F, Mt, qe, Hn):
    """sri_newton_static_problem with every optional input NULL (the Python method calls the tip-load entry point then)."""
    prob = _problem(F.shape[0], NE, Hn, F, Mt, None, None, None, None, None)
    rep = _lib.NewtonReport()
    _lib.check(h._lib.sri_newton_static_problem(h._h, ctypes.byref(prob), _ptr(qe, "qe"), TOL, 30, 0.0, 0, _lib.ALLREDUCE_FN(),
                                                None, ctypes.byref(rep)), "sri_newton_static_problem")
    return _report_dict(rep)


def vjp_null(h, F, Mt, qe, gqe, steps, out, info, Hn):
    prob = _problem(F.shape[0], NE, Hn, F, Mt, None, None, None, None, None)
    g = lambda k: _ptr(out.get(k), k)
    grads = _lib.StaticProblemGrad(gF_tip=g("F_tip"), gM_tip=g("M_tip"), gK0=g("K0"), gH=g("H"), resid=g("resid"),
                                   info=_ptr(info, "info", np.int32))
    _lib.check(h._lib.sri_static_problem_vjp(h._h, ctypes.byref(prob), _ptr(qe, "qe"), _ptr(gqe, "gqe"), steps,
                                             ctypes.byref(grads)), "sri_static_problem_vjp")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    Hn = np.ascontiguousarray(H, dtype=np.float64)
    lines = []
    for N, B in CONFIGS:
        hs = {p: SpectralRodIntegrator(N, 0) for p in ("tip", "null", "gravity")}
        for h in hs.values():
            h.set_stream(torch.cuda.current_stream())
        f64 = dict(dtype=torch.float64, device="cuda")
        F, Mt, fbar = torch.empty((B, 3), **f64), torch.empty((B, 3), **f64), torch.empty((B, 3, N), **f64)
        hs["tip"].generate_rods(0x5EED, 0, B, None, F, Mt, fbar)
        tip_want = ("F_tip", "M_tip", "K0", "H", "resid")
        qe = {p: torch.zeros((B, 3 * NE), **f64) for p in ("tip", "null", "gravity")}
        reports = {p: [] for p in qe}

        def forward(p):
            h = hs[p]
            qe[p].zero_()
            if p == "tip":
                rep = h.newton_static_shape(F, Mt, NE, H_diag=H, qe=qe[p], tol=TOL, max_iter=30, fd_step=0.0)[1]
            elif p == "null":
                rep = newton_null(h, F, Mt, qe[p], Hn)
            else:
                rep = h.newton_static_shape(F, Mt, NE, H_diag=H, qe=qe[p], tol=TOL, max_iter=30, fd_step=0.0, fbar=fbar)[1]
            reports[p].append(rep)

        for p in qe:
            forward(p)
        qstar = {p: v.clone() for p, v in qe.items()}
        gqe = torch.randn(qstar["tip"].shape, generator=torch.Generator(device="cuda").manual_seed(1), **f64)
        info_t = torch.empty((B,), dtype=torch.int32, device="cuda")
        outs = {}
        for s in (0, 3):
            outs["tip", s] = hs["tip"].static_shape_vjp(F, Mt, qstar["tip"], gqe, H_diag=H, refine_steps=s, want=tip_want)
            outs["null", s] = {k: torch.empty_like(v) for k, v in outs["tip", s].items()}
            outs["gravity", s] = hs["gravity"].static_shape_vjp(F, Mt, qstar["gravity"], gqe, H_diag=H, refine_steps=s,
                                                                fbar=fbar, want=tip_want + ("fbar",))

        def backward(p, s):
            h = hs[p]
            if p == "tip":
                h.static_shape_vjp(F, Mt, qstar[p], gqe, H_diag=H, refine_steps=s, info=info_t, want=tip_want, out=outs[p, s])
            elif p == "null":
                vjp_null(h, F, Mt, qstar[p], gqe, s, outs[p, s], info_t, Hn)
            else:
                h.static_shape_vjp(F, Mt, qstar[p], gqe, H_diag=H, refine_steps=s, info=info_t, want=tip_want + ("fbar",),
                                   out=outs[p, s], fbar=fbar)

        ops = {}
        for p in qe:
            ops[p, "newton"] = (lambda p=p: forward(p))
            for s in (0, 3):
                ops[p, f"vjp_refine{s}"] = (lambda p=p, s=s: backward(p, s))
        for fn in ops.values():  # warm-up of every shape the timed loop uses
            fn(); fn()
        torch.cuda.synchronize()
        times = {k: [] for k in ops}
        for _ in range(args.reps):
            for k, fn in ops.items():
                times[k].append(event_ms(fn))
                assert int((info_t != 0).sum()) == 0 or k[1] == "newton"
        info = card()
        assert all(r["converged"] for rs in reports.values() for r in rs)
        same = bool(torch.equal(qstar["tip"], qstar["null"])) and all(
            torch.equal(outs["tip", s][k], outs["null", s][k]) for s in (0, 3) for k in tip_want)
        for (p, op), ts in times.items():
            line = {"problem": p, "op": op, "N": N, "ne": NE, "rods": B, "ms_best": min(ts), "ms_median": statistics.median(ts),
                    "newton_iterations": reports[p][-1]["iterations"], "null_bitwise_equal_to_tip": same, **info}
            if op != "newton":
                line["max_resid"] = float(outs[p, int(op[-1])]["resid"].max())
            lines.append(line)
            print(json.dumps(line), flush=True)
        for h in hs.values():
            h.close()
        del F, Mt, fbar, qe, qstar, gqe, outs
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
