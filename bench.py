#!/usr/bin/env python
"""bench.py -- headline benchmark: rod-integrations/sec (N=16, 4 stages, FP64) on N B200s.

  python bench.py --gpus 1 --steps 20 --warmup 3            # this repo's CUDA path (one JSON line)
  python bench.py --impl reference --steps 3 --warmup 1     # CPU arm: restated reference algorithm on host cores
  python bench.py --gpus 1 --steps 20 --dump-outputs DIR    # also write a sample of the last timed step's outputs as DIR/*.npy
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus 8 --steps 20 --warmup 3            # one rank per GPU, rods sharded by index, no collective

A "step" is one fused four-stage integration of `--rods` synthetic rods per GPU (SURVEY 8d inputs: constant+linear
curvature, random tip wrench, constant distributed load), inputs resident in HBM.  Weak scaling: every rank
integrates its own contiguous rod-index range [rank*rods, (rank+1)*rods).

Beside the headline the same run reports, under `other_configs`, the other BASELINE.json configurations:
  cfg2        10^4 rods on one GPU                                   (1 GPU only)
  stages      the four stages through their separate entry points, each against its roof (1 GPU only)
  cfg3_strong ONE batch of 10^6 rods sharded by rod index over the N GPUs (strong scaling; N > 1)
  cfg4        10^5 rods at N = 32 and N = 64                         (1 GPU only)
  cfg5        Newton static shape solve of 10^5 tip-loaded rods sharded over the N GPUs, residual norms reduced by NCCL on
              the handle's stream inside sri_newton_static_shape (every N)
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the tree this runs from may be read-only; it writes nothing there

import numpy as np  # noqa: E402

N_NODES = 16
SEED = 0x5EED
METRIC = "rod-integrations/sec (N=16, 4 stages, FP64)"
# SURVEY 8(d) / BASELINE.md section 2: algorithmic work of one rod-integration, dense real formulation
FLOPS_PER_ROD_DENSE = 155_700
DMMA_PER_ROD = 215  # tensor-core instructions the fused kernel issues per rod (csrc/sri_fused16_dmma.cuh)
KERNEL_NAME = "sri::fused16_dmma_kernel<15>"
EXECUTED_NOTE = ("215 DMMA m8n8k4 (512 flop each) per rod: 176 rank-4 updates, 23 pivot-row normalisations, 16 stage contractions "
                 "(position and force share one); dead columns and padding included")
PEAK_NOMINAL_TFLOPS = 37.2  # 148 SM x 64 FP64 FMA/clk x 2 x 1.965 GHz
BYTES_PER_ROD = 1_992 + 3 * N_NODES * 8  # compulsory HBM traffic incl. the nodal fbar this workload supplies
DUMP_RODS = 16_384  # rods in the --dump-outputs sample: 16384 x (Q, r, n, m, info) = 26 MB of float64


def _config(rods: int, world: int) -> dict:
    """The workload description shared by both arms."""
    return {"workload": f"cfg3: {rods} rods per GPU, N=16, constant+linear strain (Philox seed 0x5EED, counter = rod "
                        "index), random tip wrench, constant distributed load, all 4 stages fused",
            "N": N_NODES, "rods_per_gpu": rods, "parallelism": f"rod-index sharding x{world}, no collective",
            "l2": f"inputs+outputs {BYTES_PER_ROD * rods / 1e6:.0f} MB per step > 126 MB L2"}


def _parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--rods", type=int, default=1_000_000, help="rods per GPU per step (cfg3: 10^6 rods, N=16)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-side-configs", action="store_true", help="skip other_configs (cfg2, cfg3_strong, cfg4, cfg5)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write Q, r, n, m and info of the last step for a fixed, seeded sample of rank 0's "
                         f"rods (at most {DUMP_RODS}; rod_index names them) as DIR/<name>.npy in float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    return args


# ---------------------------------------------------------------------------------------------------------------
#  CPU arm (oracle = restated reference algorithm; Eigen/Boost are not in the image, see DESIGN.md)
# ---------------------------------------------------------------------------------------------------------------

def _native_oracle():
    """Oracle compiled -O3 -march=native on THIS host for timing (the portable build is used for checking)."""
    from oracle.oracle import Oracle, build_oracle
    try:
        build_oracle(native=True)
        return Oracle(N_NODES, native=True), "gcc -O3 -march=native -fopenmp"
    except Exception:  # no compiler on the box: fall back to the prebuilt portable oracle
        build_oracle()
        return Oracle(N_NODES), "gcc -O3 -fopenmp (prebuilt portable)"


def _time_oracle(o, rods: int, first_rod: int, explicit_inverse: bool, nthreads: int) -> float:
    K, F, Mt, fb = o.generate_rods(SEED, first_rod, rods)
    t0 = time.perf_counter()
    out = o.integrate_all(K, F, Mt, fbar=fb, explicit_inverse=explicit_inverse, nthreads=nthreads)
    dt = time.perf_counter() - t0
    assert out["bad"] == 0
    return dt


def _host_cores() -> int:
    """All host threads this process may use (torchrun exports OMP_NUM_THREADS=1, so do not ask OpenMP)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def _reference_own_code_rate():
    """Side figure: the reference's OWN main.cpp functions (integrateQuaternions() + integratePosition(), compiled verbatim in the
    build container against oracle/eigen_shim, oracle/_ref/libreference_harness.so) on one host core -- stages 1-2 only, the
    second quaternion solve of main.cpp:147 included, global qe => not thread-safe.  None when the prebuilt library is absent."""
    try:
        from oracle.build_reference import ReferenceHarness
        from oracle.oracle import Oracle
        h = ReferenceHarness()
        qe = Oracle(N_NODES).generate_modes(SEED, 0, 600)
        h.integrate(qe[:50])
        t0 = time.perf_counter()
        h.integrate(qe)
        dt = time.perf_counter() - t0
        return {"value": len(qe) / dt, "unit": "rods/s", "cores": 1, "kind": "reference",
                "sample": "600 rods, main.cpp's own integrateQuaternions() + integratePosition() per rod (stages 1-2 only; the "
                          "reference repeats the quaternion solve inside integratePosition), Eigen replaced by oracle/eigen_shim"}
    except Exception as exc:  # noqa: BLE001
        return {"unavailable": f"{type(exc).__name__}: {exc}"}


def cpu_baseline(target_seconds: float):
    o, how = _native_oracle()
    cores = _host_cores()
    probe = 1024 * cores
    _time_oracle(o, probe, 0, True, cores)  # warm up threads and caches
    dt = _time_oracle(o, probe, 0, True, cores)
    rate = probe / dt
    sample = int(min(max(rate * target_seconds, probe), 2_000_000))
    dt = _time_oracle(o, sample, 0, True, cores)
    value = sample / dt
    dt1 = _time_oracle(o, max(probe // cores, 64), 0, True, 1)
    dt_lu = _time_oracle(o, probe * 4, 0, False, cores)
    ref_own = _reference_own_code_rate()
    return {
        "value": value, "unit": "rods/s", "cores": cores, "kind": "port",
        "sample": f"{sample} rods of the same Philox stream (rods 0..{sample - 1}), all four stages, explicit 60x60 "
                  f"inverse as main.cpp:113, Dn cached, no redundant second quaternion solve; {how}",
        "value_1core": max(probe // cores, 64) / dt1,
        "value_lu_solve_variant": probe * 4 / dt_lu,
        "seconds": dt,
        "reference_own_code_1core": ref_own,
    }


def run_reference(args, rank: int):
    """CPU arm: the restated reference algorithm on all host cores of rank 0, EXACTLY `--rods` rods per step (the config of
    the GPU arm), steps over consecutive rod-index ranges of the same Philox stream.  Warm-up steps use a short range (they
    only start the threads and warm the caches; they are not timed)."""
    if rank != 0:
        return
    o, how = _native_oracle()
    cores = _host_cores()
    per_step = int(args.rods)
    warm = min(per_step, 4096 * cores)
    for _ in range(max(args.warmup, 1)):
        _time_oracle(o, warm, 0, True, cores)
    total = 0.0
    for s in range(args.steps):
        total += _time_oracle(o, per_step, s * per_step, True, cores)
    value = per_step * args.steps / total
    sample = (f"{per_step} rods per step = the GPU arm's rods per GPU per step, {args.steps} steps over consecutive rod ranges of the "
              f"same Philox stream, all four stages, explicit 60x60 inverse as main.cpp:113, Dn cached, no redundant second "
              f"quaternion solve; warm-up steps on {warm} rods; {how}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rods/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": _config(args.rods, args.gpus),
        "cpu_baseline": {"value": value, "unit": "rods/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "rods/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
#  clocks sampling during the timed region (NVML)
# ---------------------------------------------------------------------------------------------------------------

class ClockSampler:
    REASONS = {
        0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
        0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
        0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting",
    }

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._dev = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._dev, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _loop(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._dev, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._dev)
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self._nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------------------
#  GPU arm
# ---------------------------------------------------------------------------------------------------------------

def _bind_to_gpu_numa_node(torch, local_rank: int):
    """Multi-rank runs: pin this rank's CPU affinity to the NUMA node of its GPU before the pinned host buffers of the
    end-to-end leg are allocated (first touch), so that eight ranks do not stream their H2D/D2H traffic across sockets.
    Returns the node, or None when the topology cannot be read (then nothing is changed)."""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(Path(f"/sys/bus/pci/devices/{bdf}/numa_node").read_text())
        if node < 0:
            return None
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


def dump_outputs(out_dir: str, torch, outs: dict, first_rod: int) -> None:
    """Writes the rows of a fixed, seeded sample of the batch (all of it when it has at most DUMP_RODS rods) as
    out_dir/<name>.npy in float64, with rod_index = the global rod index of each row.  The sample depends on the batch
    size alone, so two builds run with the same arguments can be compared output for output."""
    any_out = next(iter(outs.values()))
    B = any_out.shape[0]
    rows = np.sort(np.random.default_rng(SEED).choice(B, size=min(B, DUMP_RODS), replace=False))
    sel = torch.from_numpy(rows).to(any_out.device)
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, t in outs.items():
        np.save(out / f"{name}.npy", t.index_select(0, sel).cpu().numpy().astype(np.float64))
    np.save(out / "rod_index.npy", (first_rod + rows).astype(np.float64))


def _max_over_ranks(torch, dist, world, dev, x: float) -> float:
    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_b200(args, rank: int, world: int, local_rank: int):
    import torch
    import torch.distributed as dist

    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import (
        SpectralRodIntegrator, kernel_launch_count, shard_range)

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl b200 needs a CUDA device: the integration path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = _bind_to_gpu_numa_node(torch, local_rank) if world > 1 else None
    B, N, M = args.rods, N_NODES, N_NODES - 1
    f64 = torch.float64
    warmup = max(args.warmup, 3)  # the timing rules ask for >= 3; the JSON line records what was run

    h = SpectralRodIntegrator(N, local_rank)
    stream = torch.cuda.current_stream(dev)
    h.set_stream(stream)

    # ---- inputs resident in HBM (generated on the device from the rod-index-keyed Philox stream)
    K = torch.empty((B, 3, N), dtype=f64, device=dev)
    F = torch.empty((B, 3), dtype=f64, device=dev)
    Mt = torch.empty((B, 3), dtype=f64, device=dev)
    fb = torch.empty((B, 3, N), dtype=f64, device=dev)
    first = rank * B
    h.generate_rods(SEED, first, B, K, F, Mt, fb)
    Q = torch.empty((B, 4, M), dtype=f64, device=dev)
    r = torch.empty((B, 3, M), dtype=f64, device=dev)
    n = torch.empty((B, 3, M), dtype=f64, device=dev)
    m = torch.empty((B, 3, M), dtype=f64, device=dev)
    info = torch.zeros((B,), dtype=torch.int32, device=dev)

    def step():
        h.integrate_all(K, F, Mt, fbar=fb, Q=Q, r=r, n=n, m=m, info=info)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def mx(x):
        return _max_over_ranks(torch, dist, world, dev, x)

    for _ in range(warmup):
        step()
    barrier()

    # live roofline denominators (MEASURED_PEAKS.json has no FP64 entry): scalar DFMA stream and DMMA m8n8k4 stream
    fp64_peak = h.measure_fp64_peak()
    dmma_peak = h.measure_dmma_peak()
    barrier()

    sampler = ClockSampler(local_rank)
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    launches0 = kernel_launch_count()
    barrier()
    sampler.start()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    launches = kernel_launch_count() - launches0
    ms_step = mx(e0.elapsed_time(e1)) / args.steps
    value = world * B / (ms_step * 1e-3)
    assert int(info.abs().sum().item()) == 0, "zero pivot reported on the synthetic workload"
    if args.dump_outputs is not None and rank == 0:  # before the legs below reuse Q, r, n, m
        dump_outputs(args.dump_outputs, torch, {"Q": Q, "r": r, "n": n, "m": m, "info": info}, first)

    # ---- end to end through the C ABI with HOST buffers (pinned), H2D + D2H inside the timed region, and beside it the bare
    #      concurrent copies of the very same buffers on all ranks (the ceiling the host platform allows this call)
    e2e = None
    if not args.no_e2e:
        hk = K.cpu().pin_memory(); hF = F.cpu().pin_memory(); hM = Mt.cpu().pin_memory(); hfb = fb.cpu().pin_memory()
        hQ = torch.empty((B, 4, M), dtype=f64).pin_memory(); hr = torch.empty((B, 3, M), dtype=f64).pin_memory()
        hn = torch.empty((B, 3, M), dtype=f64).pin_memory(); hm = torch.empty((B, 3, M), dtype=f64).pin_memory()
        he = max(3, min(args.steps, 10))

        def timed_host(fn, reps):
            for _ in range(2):
                fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()
            torch.cuda.synchronize(dev)
            return mx(time.perf_counter() - t0) / reps

        def host_step():
            h.integrate_all(hk, hF, hM, fbar=hfb, Q=hQ, r=hr, n=hn, m=hm)  # returns after the D2H copies complete

        dt = timed_host(host_step, he)
        h2d = (hk.numel() + hF.numel() + hM.numel() + hfb.numel()) * 8
        d2h = (hQ.numel() + hr.numel() + hn.numel() + hm.numel()) * 8
        assert torch.equal(hQ[:1000], Q[:1000].cpu()), "host-buffer path and device-buffer path disagree"

        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

        def bare_copies(outs):
            def run():
                with torch.cuda.stream(s_in):
                    K.copy_(hk, non_blocking=True); F.copy_(hF, non_blocking=True)
                    Mt.copy_(hM, non_blocking=True); fb.copy_(hfb, non_blocking=True)
                with torch.cuda.stream(s_out):
                    for hd, dd in outs:
                        hd.copy_(dd, non_blocking=True)
                s_in.synchronize(); s_out.synchronize()
            return run

        dt_copy = timed_host(bare_copies([(hQ, Q), (hr, r), (hn, n), (hm, m)]), he)
        # the variant the Newton driver's callers use: only Q and m come back (984 of 1 560 B per rod)
        def host_step_qm():
            h.integrate_all(hk, hF, hM, fbar=hfb, Q=hQ, m=hm, want=("Q", "m"))
        dt_qm = timed_host(host_step_qm, he)
        dt_copy_qm = timed_host(bare_copies([(hQ, Q), (hm, m)]), he)
        e2e = {"value": world * B / dt, "unit": "rods/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "steps": he, "ms_per_step": dt * 1e3, "rank0_numa_node": numa,
               "path": "sri_integrate_all() with pinned host buffers; per step: H2D of K,F_tip,M_tip,fbar, fused kernels, D2H of Q,r,n,m",
               "copy_ceiling_rods_per_s": world * B / dt_copy, "copy_ceiling_ms_per_step": dt_copy * 1e3,
               "frac_of_copy_ceiling": dt_copy / dt,
               "copy_ceiling_note": "bare cudaMemcpyAsync of the same pinned buffers, H2D and D2H on two streams, all ranks at once, "
                                    "same barrier / max-over-ranks timing: what the host's PCIe / memory fabric allows this call",
               "variant_Q_m_only": {"value": world * B / dt_qm, "ms_per_step": dt_qm * 1e3, "d2h_bytes_per_step": (hQ.numel() + hm.numel()) * 8,
                                    "copy_ceiling_rods_per_s": world * B / dt_copy_qm, "frac_of_copy_ceiling": dt_copy_qm / dt_qm}}
        h.generate_rods(SEED, first, B, K, F, Mt, fb)  # (the bare copies overwrote the inputs with themselves; keep them exact)
        del hk, hF, hM, hfb, hQ, hr, hn, hm
        barrier()

    other = {}
    side = not args.no_side_configs
    # ---- BASELINE configs[1] (10^4 rods on one GPU) timed beside the headline workload, device-resident ----------
    if side and world == 1:
        Bs = 10_000
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        small = lambda: h.integrate_all(K[:Bs], F[:Bs], Mt[:Bs], fbar=fb[:Bs], Q=Q[:Bs], r=r[:Bs], n=n[:Bs], m=m[:Bs])
        for _ in range(5):
            small()
        torch.cuda.synchronize(dev)
        e2.record(stream)
        for _ in range(50):
            small()
        e3.record(stream)
        torch.cuda.synchronize(dev)
        other["cfg2"] = {"workload": "cfg2: 10^4 rods, N=16, 1 GPU (a single 2.8-wave launch; L2-resident after the first pass)",
                         "rods_per_s": Bs / (e2.elapsed_time(e3) / 50 * 1e-3), "us_per_launch": e2.elapsed_time(e3) / 50 * 1e3}

    # ---- the four stages one by one (separate-stage entry points, device-resident), each against the roof that bounds it: stage 1
    #      FP64 tensor pipe, stages 2-4 HBM (SURVEY 8d); timed with the library's own per-call CUDA-event timer (sri_set_timing)
    if side and world == 1:
        try:
            hbm = 6650.0
            try:
                hbm = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()).get("hbm_gbs", hbm)
            except Exception:
                pass
            h.set_timing(True)

            def stage_ms(fn, reps=10):
                for _ in range(3):
                    fn()
                tot = 0.0
                for _ in range(reps):
                    fn()
                    tot += h.last_timing()[0]
                return tot / reps

            st = {}
            ms = stage_ms(lambda: h.integrate_quaternions(K, out=Q))
            st["quaternions"] = {"entry": "sri_integrate_quaternions", "ms": ms, "rods_per_s": B / ms * 1e3, "bound": "tensor",
                                 "dense_count_tflops": B / ms * 1e3 * 151_200 * 1e-12, "frac_of_dmma_peak_dense": B / ms * 1e3 * 151_200 * 1e-12 / dmma_peak}
            for name, fn, bytes_per_rod in (
                    ("position", lambda: h.integrate_position(Q, out=r), (4 * M + 3 * M) * 8),
                    ("stress", lambda: h.integrate_stress(F, fbar=fb, out=n), (3 * N + 3 + 3 * M) * 8),
                    ("couple", lambda: h.integrate_couple(Q, n, Mt, out=m), (4 * M + 3 * M + 3 + 3 * M) * 8)):
                ms = stage_ms(fn)
                gbs = B * bytes_per_rod / ms * 1e-6
                st[name] = {"entry": f"sri_integrate_{name}", "ms": ms, "rods_per_s": B / ms * 1e3, "bound": "hbm", "bytes_per_rod": bytes_per_rod,
                            "GBps": gbs, "frac_of_hbm_peak": gbs / hbm}
            h.set_timing(False)
            st["note"] = ("separate-stage entry points on the headline batch; the fused sri_integrate_all (the headline) does all four in "
                          "one launch and keeps Q on the SM; hbm peak = MEASURED_PEAKS.json copy bandwidth")
            other["stages"] = st
        except Exception as exc:  # noqa: BLE001
            other["stages"] = {"error": f"{type(exc).__name__}: {exc}"}

    # ---- BASELINE configs[2], the north-star target: ONE batch of 10^6 rods sharded by rod index over the GPUs (strong
    #      scaling), device-resident, same timing rules as the headline ------------------------------------------------
    if side and world > 1:
        total = 1_000_000
        lo, hi = shard_range(total, rank, world)
        Bs = hi - lo
        h.generate_rods(SEED, lo, Bs, K[:Bs], F[:Bs], Mt[:Bs], fb[:Bs])
        strong = lambda: h.integrate_all(K[:Bs], F[:Bs], Mt[:Bs], fbar=fb[:Bs], Q=Q[:Bs], r=r[:Bs], n=n[:Bs], m=m[:Bs], info=info[:Bs])
        for _ in range(warmup):
            strong()
        barrier()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record(stream)
        for _ in range(args.steps):
            strong()
        e3.record(stream)
        barrier()
        ms = mx(e2.elapsed_time(e3)) / args.steps
        rate = total / (ms * 1e-3)
        other["cfg3_strong"] = {
            "workload": f"cfg3 strong scaling: ONE batch of 10^6 rods, N=16, sharded by rod index over {world} GPUs "
                        f"({Bs} rods on rank 0), all 4 stages fused, device-resident, no collective",
            "rods_total": total, "rods_rank0": Bs, "steps": args.steps, "ms_per_step": ms, "rods_per_s": rate,
            "scaling": "strong", "dense_count_tflops_per_gpu": rate * FLOPS_PER_ROD_DENSE * 1e-12 / world,
            "frac_of_dmma_peak_dense": rate * FLOPS_PER_ROD_DENSE * 1e-12 / world / dmma_peak,
            "frac_of_dmma_peak_executed": rate * DMMA_PER_ROD * 512 * 1e-12 / world / dmma_peak,
            "l2": f"{BYTES_PER_ROD * Bs / 1e6:.0f} MB touched per GPU per step > 126 MB L2",
            "weak_headline_rods_per_s": value,
        }
        h.generate_rods(SEED, first, B, K, F, Mt, fb)

    # ---- BASELINE configs[3] (10^5 rods at N = 32 and N = 64), device-resident, beside the headline workload ---------
    if side and world == 1:
        cfg4 = {}
        for Nh, flops in ((32, 1_320_063), (64, 10_869_012)):
            Bh, Mh = 100_000, Nh - 1
            hh = SpectralRodIntegrator(Nh, local_rank)
            hh.set_stream(stream)
            Kh = torch.empty((Bh, 3, Nh), dtype=f64, device=dev); Fh = torch.empty((Bh, 3), dtype=f64, device=dev)
            Mh_t = torch.empty((Bh, 3), dtype=f64, device=dev); fbh = torch.empty((Bh, 3, Nh), dtype=f64, device=dev)
            hh.generate_rods(SEED, 0, Bh, Kh, Fh, Mh_t, fbh)
            outs = {k: torch.empty((Bh, c, Mh), dtype=f64, device=dev) for k, c in (("Q", 4), ("r", 3), ("n", 3), ("m", 3))}
            run = lambda: hh.integrate_all(Kh, Fh, Mh_t, fbar=fbh, **outs)
            for _ in range(2):
                run()
            torch.cuda.synchronize(dev)
            e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e4.record(stream)
            for _ in range(3):
                run()
            e5.record(stream)
            torch.cuda.synchronize(dev)
            ms = e4.elapsed_time(e5) / 3
            cfg4[f"N{Nh}"] = {"workload": f"cfg4: 10^5 rods, N={Nh}, 1 GPU, all 4 stages fused", "rods_per_s": Bh / (ms * 1e-3),
                              "ms_per_launch": ms, "dense_count_tflops": Bh / (ms * 1e-3) * flops * 1e-12}
            hh.close()
            del Kh, Fh, Mh_t, fbh, outs
        other["cfg4"] = cfg4

    # ---- BASELINE configs[4]: Newton static shape solve of 10^5 tip-loaded rods sharded over the GPUs, the loop inside the
    #      C ABI (sri_newton_static_shape), the residual norms all-gathered by NCCL on the handle's stream (sri_nccl_init)
    #      and tested on the device; wall-clock per solve between barriers, max over ranks.  Never fatal for the headline.
    if side:
        try:
            total, ne5, H5 = 100_000, 3, (1.0, 1.0, 0.77)
            lo, hi = shard_range(total, rank, world)
            Bn = hi - lo
            Fn = torch.empty((Bn, 3), dtype=f64, device=dev)
            h.generate_rods(SEED, lo, Bn, None, Fn, None, None)
            Fn[:, 2] = -(Fn[:, 2] + 1.0)
            Fn[:, :2] = 0.0
            Mn = torch.zeros((Bn, 3), dtype=f64, device=dev)
            if world > 1:
                h.nccl_init_from_torch()
            cfg5 = {"workload": f"cfg5: Newton static shape solve of 10^5 tip-loaded rods (F_tip = (0,0,-f), f ~ U(0,2)), N=16, ne=3, "
                                f"H = diag(1,1,0.77), rms tolerance 1e-10, sri_newton_static_shape, rods sharded over {world} GPU(s) "
                                f"({Bn} on rank 0)",
                    "reduction": ("ncclAllGather of the 16-byte norm pair on the handle's stream + device-side convergence flag, host test "
                                  "lagged by one iteration" if world > 1 else "single rank: device-side convergence flag, host test "
                                  "lagged by one iteration"),
                    "timing": "wall clock around the call, barrier + synchronize on both sides, max over ranks; best and median of 5 solves"}
            for name, fd_step in (("analytic_jacobian", 0.0), ("forward_difference_jacobian", 1e-6)):
                h.newton_static_shape(Fn, Mn, ne5, H5, fd_step=fd_step, total_dof=3 * ne5 * total)  # sizes the workspace of this mode
                times, rep5 = [], None
                for _ in range(5):
                    barrier()
                    t0 = time.perf_counter()
                    _, rep5 = h.newton_static_shape(Fn, Mn, ne5, H5, fd_step=fd_step, total_dof=3 * ne5 * total)
                    torch.cuda.synchronize(dev)
                    times.append(mx(time.perf_counter() - t0))
                best, med = min(times), sorted(times)[len(times) // 2]
                cfg5[name] = {"seconds": best, "seconds_median": med, "converged": rep5["converged"],
                              "newton_iterations": rep5["iterations"], "integrations_of_the_batch": rep5["integrations"],
                              "rod_solves_per_s": total / best, "rod_integrations_per_s": total * rep5["integrations"] / best,
                              "final_rms": rep5["rms"], "singular_solves": rep5["singular_solves"]}
            if world > 1:
                h.nccl_finalize()
            del Fn, Mn
        except Exception as exc:  # noqa: BLE001 -- a side leg must not take the headline measurement down
            cfg5 = {"error": f"{type(exc).__name__}: {exc}"}
        other["cfg5"] = cfg5

    if rank != 0:
        return

    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    traffic, traffic_src = None, None
    try:
        tj = json.loads((ROOT / "profiles" / "traffic.json").read_text())
        traffic = tj.get("fused16_dram_bytes_per_rod")
        traffic = traffic * B if traffic is not None else None
        traffic_src = tj.get("source", "profiles/traffic.json") + " -- per-rod DRAM bytes of one `ncu --set full` capture x rods per launch (not re-measured in this run: ncu cannot run inside it)"
    except Exception:
        pass
    # Two launches per step: fused16_dmma_kernel (all the work) and the row-pivoting second pass, whose CTAs exit at
    # once when no rod was handed back (always, on this workload); the events bracket both, so the step time is an
    # upper bound of the dominant kernel's duration (profiles/*launches.csv: the second pass is ~3 us).
    kernel_ms = ms_step
    tflops_dense = FLOPS_PER_ROD_DENSE * B / (kernel_ms * 1e-3) * 1e-12
    peak = max(fp64_peak, dmma_peak)
    executed = DMMA_PER_ROD * 512 * B / (kernel_ms * 1e-3) * 1e-12
    roofline = {
        "bound": "tensor", "kernel": KERNEL_NAME,
        "achieved": tflops_dense, "peak": peak, "unit": "TFLOP/s", "frac": tflops_dense / peak,
        "frac_executed": executed / peak, "peak_nominal": PEAK_NOMINAL_TFLOPS, "frac_of_nominal": tflops_dense / PEAK_NOMINAL_TFLOPS,
        "peak_source": "FP64 tensor-core (DMMA m8n8k4) stream measured live on this GPU in this run "
                       f"(sri_measure_dmma_peak: {dmma_peak:.1f}; scalar DFMA stream sri_measure_fp64_peak: {fp64_peak:.1f}); "
                       "nominal 148 SM x 64 FMA/clk x 1.965 GHz = 37.2; MEASURED_PEAKS.json holds no FP64 figure",
        "flops_per_rod": FLOPS_PER_ROD_DENSE,
        "flops_note": "`frac` uses the algorithmic count of SURVEY 8(d) (dense real 60x60 LU + 3 contractions); the kernel solves the "
                      "same system as a 15x15 quaternion system, which needs ~4x fewer flops, so `frac` may exceed 1; "
                      "`frac_executed` is what the tensor pipe actually does (DMMA instructions issued x 512 flop)",
        "executed": {"dmma_per_rod": DMMA_PER_ROD, "tflops": executed, "frac": executed / peak, "note": EXECUTED_NOTE},
        "traffic": traffic, "traffic_source": traffic_src,
        "hbm": {"achieved": BYTES_PER_ROD * B / (kernel_ms * 1e-3) * 1e-9, "peak": hbm_peak, "unit": "GB/s",
                "frac": BYTES_PER_ROD * B / (kernel_ms * 1e-3) * 1e-9 / hbm_peak, "peak_source": hbm_src,
                "bytes_per_rod": BYTES_PER_ROD},
    }
    line = {
        "metric": METRIC, "value": value, "unit": "rods/s", "n_gpus": world, "steps": args.steps,
        "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": _config(B, world),
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
    }
    if other:
        line["other_configs"] = other
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline(args.cpu_seconds)
    print(json.dumps(line), flush=True)


def main():
    args = _parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
