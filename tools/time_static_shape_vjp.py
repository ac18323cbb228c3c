"""Cost of differentiating the static shape solve: sri_static_shape_vjp (the implicit adjoint) against the forward solve
sri_newton_static_shape (analytic Jacobian) on the same device-resident batch.

10^5 tip-loaded rods (sri_generate_rods: F_tip, M_tip ~ U(-1,1)^3; H = (1, 1, 0.77); zero initial guess; tol 1e-10),
ne = 4, at N = 16 (bench config 5) and N = 32.  The backward runs at the forward's solution with a random cotangent, with
refine_steps = 0 (J_a alone) and 3 (the default), all four parameter gradients wanted.  After a warm-up the forward and the
two backward variants are timed alternately with CUDA events; the best and the median over the repetitions are reported.
One JSON line per (N, variant) on stdout and, with --out, appended to that file; the card's name, power limit and maximum
SM clock are part of every line.

    python tools/time_static_shape_vjp.py [--out profiles/r04_static_shape_vjp.jsonl] [--reps 10]
"""
import argparse
import json
import statistics
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import torch  # noqa: E402

from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import SpectralRodIntegrator  # noqa: E402
from time_vjp import card, event_ms  # noqa: E402

CONFIGS = [(16, 100_000), (32, 100_000)]
NE, H, TOL = 4, (1.0, 1.0, 0.77), 1e-10


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    info = card()
    lines = []
    for N, B in CONFIGS:
        h = SpectralRodIntegrator(N, 0)
        h.set_stream(torch.cuda.current_stream())
        f64 = dict(dtype=torch.float64, device="cuda")
        F, Mt = torch.empty((B, 3), **f64), torch.empty((B, 3), **f64)
        h.generate_rods(0x5EED, 0, B, None, F, Mt, None)
        qe = torch.zeros((B, 3 * NE), **f64)
        reports = []

        def forward():
            qe.zero_()
            reports.append(h.newton_static_shape(F, Mt, NE, H_diag=H, qe=qe, tol=TOL, max_iter=30, fd_step=0.0)[1])

        forward()
        qstar = qe.clone()
        gqe = torch.randn(qstar.shape, generator=torch.Generator(device="cuda").manual_seed(1), **f64)
        want = ("F_tip", "M_tip", "K0", "H", "resid")
        outs = {s: {k: torch.empty(v.shape, dtype=v.dtype, device="cuda") for k, v in
                    h.static_shape_vjp(F, Mt, qstar, gqe, H_diag=H, refine_steps=s, want=want).items()} for s in (0, 3)}
        info_t = torch.empty((B,), dtype=torch.int32, device="cuda")
        backward = lambda s: h.static_shape_vjp(F, Mt, qstar, gqe, H_diag=H, refine_steps=s, info=info_t, want=want, out=outs[s])
        variants = {"newton_static_shape": forward, "static_shape_vjp_refine0": lambda: backward(0),
                    "static_shape_vjp_refine3": lambda: backward(3)}
        for fn in variants.values():  # warm-up of every shape the timed loop uses
            fn(); fn()
        torch.cuda.synchronize()
        times = {k: [] for k in variants}
        for _ in range(args.reps):
            for k, fn in variants.items():
                times[k].append(event_ms(fn))
        assert all(r["converged"] for r in reports) and int((info_t != 0).sum()) == 0
        resid = {s: float(outs[s]["resid"].max()) for s in (0, 3)}
        for k in variants:
            line = {"op": k, "N": N, "ne": NE, "rods": B, "ms_best": min(times[k]), "ms_median": statistics.median(times[k]),
                    "ratio_to_forward": min(times[k]) / min(times["newton_static_shape"]), **info}
            if k == "newton_static_shape":
                line["newton_iterations"] = reports[-1]["iterations"]
            else:
                line["max_resid"] = resid[0 if k.endswith("0") else 3]
            lines.append(line)
            print(json.dumps(line), flush=True)
        h.close()
        del F, Mt, qe, qstar, gqe, outs
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
