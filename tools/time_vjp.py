"""Throughput of the reverse mode (sri_integrate_all_vjp) against the forward (sri_integrate_all) on the same batch.

Device-resident synthetic rods (sri_generate_rods), sizes well beyond the 126 MB L2 (10^6 rods at N = 16: ~5 GB of
inputs, outputs, cotangents and gradients).  After a warm-up the two calls are timed alternately with CUDA events, so
that both see the same clocks; the median over the repetitions is reported.  The VJP is timed twice: with all eight
gradients, and without the K / q0 gradients, which skips the transposed stage-1 solve (per-phase split: the difference
is the solve, the rest is stages 4 -> 2 and the pointwise terms).  One JSON line per (N, variant) on stdout and, with
--out, appended to that file; the card's name and power limit are part of every line.

    python tools/time_vjp.py [--out profiles/r03_vjp.jsonl] [--reps 20]
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch  # noqa: E402

from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import SpectralRodIntegrator  # noqa: E402

CONFIGS = [(16, 1_000_000), (32, 200_000), (64, 100_000)]
ALL = ("K", "q0", "r0", "Gamma", "fbar", "lbar", "F_tip", "M_tip")
NO_SOLVE = ("r0", "Gamma", "fbar", "lbar", "F_tip", "M_tip")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:  # pragma: no cover
        q = "unknown"
    return {"card": name, "power_limit_and_max_sm_clock": q}


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    info = card()
    lines = []
    for N, B in CONFIGS:
        M = N - 1
        h = SpectralRodIntegrator(N, 0)
        h.set_stream(torch.cuda.current_stream())
        f64 = dict(dtype=torch.float64, device="cuda")
        K, fb = torch.empty((B, 3, N), **f64), torch.empty((B, 3, N), **f64)
        F, Mt = torch.empty((B, 3), **f64), torch.empty((B, 3), **f64)
        h.generate_rods(0x5EED, 0, B, K, F, Mt, fb)
        fwd = {k: torch.empty((B, 4 if k == "Q" else 3, M), **f64) for k in "Qrnm"}
        gen = torch.Generator(device="cuda").manual_seed(1)
        cot = {"g" + k: torch.randn(v.shape, generator=gen, **f64) for k, v in fwd.items()}
        shapes = {"K": (B, 3, N), "q0": (B, 4), "r0": (B, 3), "Gamma": (B, 3, N), "fbar": (B, 3, N), "lbar": (B, 3, N),
                  "F_tip": (B, 3), "M_tip": (B, 3)}
        grads = {k: torch.empty(s, **f64) for k, s in shapes.items()}
        info_t = torch.empty((B,), dtype=torch.int32, device="cuda")
        run_fwd = lambda: h.integrate_all(K, F, Mt, fbar=fb, **fwd)
        run_fwd()
        run_vjp = lambda want: h.integrate_all_vjp(K, fwd["Q"], n=fwd["n"], **cot, info=info_t, want=want,
                                                   out={k: grads[k] for k in want})
        variants = {"forward": run_fwd, "vjp": lambda: run_vjp(ALL), "vjp_without_solve": lambda: run_vjp(NO_SOLVE)}
        for fn in variants.values():  # warm-up of every shape the timed loop uses
            fn(); fn()
        torch.cuda.synchronize()
        times = {k: [] for k in variants}
        for _ in range(args.reps):
            for k, fn in variants.items():
                times[k].append(event_ms(fn))
        assert int((info_t != 0).sum()) == 0
        med = {k: statistics.median(v) for k, v in times.items()}
        for k in variants:
            line = {"op": k, "N": N, "rods": B, "ms_median": med[k], "ms_min": min(times[k]), "ms_max": max(times[k]),
                    "rods_per_s": B / med[k] * 1e3, "ratio_to_forward": med[k] / med["forward"], **info}
            lines.append(line)
            print(json.dumps(line), flush=True)
        h.close()
        del K, fb, F, Mt, fwd, cot, grads
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
