"""ctypes wrapper of oracle/sri_oracle.c (TEST INFRASTRUCTURE ONLY -- see the header of that file).

Build products go to oracle/_ref/ (git-ignored, shipped to the GPU box with the snapshot).
"""
from __future__ import annotations

import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile
from ctypes import c_double, c_int, c_long, c_void_p
from pathlib import Path

import numpy as np

ORACLE_DIR = Path(__file__).resolve().parent
REF_DIR = ORACLE_DIR / "_ref"
SRC = ORACLE_DIR / "sri_oracle.c"
_native_dir = None


def oracle_lib_path(native: bool = False) -> Path:
    if not native:
        return REF_DIR / "libsri_oracle.so"
    global _native_dir
    if _native_dir is None:
        _native_dir = Path(tempfile.mkdtemp(prefix="sri_oracle_native_"))
        atexit.register(shutil.rmtree, _native_dir, True)
    return _native_dir / "libsri_oracle_native.so"


def build_oracle(force: bool = False, native: bool = False) -> Path:
    """gcc on oracle/sri_oracle.c -> oracle/_ref/libsri_oracle.so.

    The default (checker) build is portable: generic x86-64, no FMA contraction, so its arithmetic is plain IEEE
    and identical on every x86-64 host.  native=True adds -march=native and is rebuilt on the host that runs it,
    in a temporary directory of this process (the tree it runs from may be read-only); bench.py uses it for the
    timed CPU baseline only.
    """
    out = oracle_lib_path(native)
    if not force and not native and out.exists() and out.stat().st_mtime >= SRC.stat().st_mtime:
        return out
    out.parent.mkdir(exist_ok=True)
    gcc = shutil.which("gcc") or "gcc"
    flags = ["-O3", "-march=native"] if native else ["-O3", "-ffp-contract=off"]
    cmd = [gcc, *flags, "-fopenmp", "-fPIC", "-shared", "-o", str(out), str(SRC), "-lm"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("gcc failed building the oracle:\n" + res.stdout + res.stderr)
    return out


def _p(a):
    if a is None:
        return None
    assert isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags["C_CONTIGUOUS"], "oracle wants C-contiguous float64"
    return a.ctypes.data


class Oracle:
    """Restated reference algorithm for N Chebyshev nodes."""

    def __init__(self, N: int = 16, native: bool = False):
        path = oracle_lib_path(native)
        if not path.exists():
            build_oracle(native=native)
        self.lib = ctypes.CDLL(str(path))
        self.N = int(N)
        self.M = self.N - 1
        L = self.lib
        L.sri_oracle_ops_create.restype = c_void_p
        L.sri_oracle_ops_create.argtypes = [c_int]
        L.sri_oracle_ops_destroy.argtypes = [c_void_p]
        L.sri_oracle_ops_get.restype = ctypes.POINTER(c_double)
        L.sri_oracle_ops_get.argtypes = [c_void_p, c_int]
        L.sri_oracle_legendre_p.restype = c_double
        L.sri_oracle_legendre_p.argtypes = [c_int, c_double]
        L.sri_oracle_chebyshev_points.argtypes = [c_int, c_double, c_void_p]
        L.sri_oracle_coefficients_c.argtypes = [c_int, c_void_p]
        L.sri_oracle_dn.argtypes = [c_int, c_void_p]
        L.sri_oracle_phi.argtypes = [c_int, c_int, c_double, c_double, c_double, c_void_p]
        L.sri_oracle_strain_from_modes.argtypes = [c_int, c_int, c_int, c_void_p, c_void_p]
        L.sri_oracle_assemble_A.argtypes = [c_void_p, c_void_p, c_void_p]
        L.sri_oracle_integrate_all_batch.restype = c_int
        L.sri_oracle_integrate_all_batch.argtypes = [c_int, c_long] + [c_void_p] * 12 + [c_int, c_int]
        L.sri_oracle_shape_residual.argtypes = [c_void_p] * 9
        L.sri_oracle_wrench_local.argtypes = [c_void_p] * 8
        L.sri_oracle_wrench_local_solve.restype = c_int
        L.sri_oracle_wrench_local_solve.argtypes = [c_void_p] * 10
        L.sri_oracle_max_threads.restype = c_int
        L.sri_oracle_generate_rods.argtypes = [c_int, ctypes.c_uint64, c_long, c_long, c_void_p, c_void_p, c_void_p, c_void_p]
        L.sri_oracle_generate_modes.argtypes = [ctypes.c_uint64, c_long, c_long, c_void_p]
        self._ops = L.sri_oracle_ops_create(self.N)

    def __del__(self):  # pragma: no cover
        try:
            self.lib.sri_oracle_ops_destroy(self._ops)
        except Exception:
            pass

    # -- operator pieces
    def chebyshev_points(self, L: float = 1.0) -> np.ndarray:
        x = np.empty(self.N)
        self.lib.sri_oracle_chebyshev_points(self.N, float(L), x.ctypes.data)
        return x

    def coefficients_c(self) -> np.ndarray:
        c = np.empty(self.N)
        self.lib.sri_oracle_coefficients_c(self.N, c.ctypes.data)
        return c

    def dn(self) -> np.ndarray:
        buf = np.empty(self.N * self.N)
        self.lib.sri_oracle_dn(self.N, buf.ctypes.data)
        return buf.reshape(self.N, self.N).T.copy()

    def operator(self, which: int) -> np.ndarray:
        M, N = self.M, self.N
        shape = {0: (N, N), 1: (M, M), 2: (M,), 3: (M, M), 4: (M, M), 5: (M,), 6: (M, M)}[which]
        ptr = self.lib.sri_oracle_ops_get(self._ops, which)
        buf = np.ctypeslib.as_array(ptr, shape=(int(np.prod(shape)),)).copy()
        return buf.reshape(shape[::-1]).T.copy() if len(shape) == 2 else buf

    def legendre_p(self, l: int, x: float) -> float:
        return float(self.lib.sri_oracle_legendre_p(int(l), float(x)))

    def phi(self, na: int, ne: int, X: float, begin: float = 0.0, end: float = 1.0) -> np.ndarray:
        buf = np.empty(na * na * ne)
        self.lib.sri_oracle_phi(na, ne, float(X), float(begin), float(end), buf.ctypes.data)
        return buf.reshape(na * ne, na).T.copy()

    def strain_from_modes(self, qe: np.ndarray, ne: int = 3) -> np.ndarray:
        qe = np.ascontiguousarray(qe, dtype=np.float64).reshape(-1, 3 * ne)
        K = np.empty((qe.shape[0], 3, self.N))
        for b in range(qe.shape[0]):
            self.lib.sri_oracle_strain_from_modes(self.N, 3, ne, qe[b].ctypes.data, K[b].ctypes.data)
        return K

    def assemble_A(self, K: np.ndarray) -> np.ndarray:
        n = 4 * self.M
        buf = np.empty(n * n)
        K = np.ascontiguousarray(K, dtype=np.float64)
        self.lib.sri_oracle_assemble_A(self._ops, K.ctypes.data, buf.ctypes.data)
        return buf.reshape(n, n).T.copy()

    # -- the four stages, batched
    def integrate_all(self, K, F_tip=None, M_tip=None, q0=None, r0=None, Gamma=None, fbar=None, lbar=None,
                      explicit_inverse: bool = True, nthreads: int = 0, want=("Q", "r", "n", "m")):
        K = np.ascontiguousarray(K, dtype=np.float64)
        B, M = K.shape[0], self.M
        out = {}
        if "Q" in want: out["Q"] = np.empty((B, 4, M))
        if "r" in want: out["r"] = np.empty((B, 3, M))
        if "n" in want: out["n"] = np.empty((B, 3, M))
        if "m" in want: out["m"] = np.empty((B, 3, M))
        if ("n" in want or "m" in want):
            assert F_tip is not None, "F_tip required for stages 3-4"
        if "m" in want:
            assert M_tip is not None, "M_tip required for stage 4"
        cz = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
        args = [cz(a) for a in (q0, r0, Gamma, fbar, lbar, F_tip, M_tip)]
        self._keep = args
        bad = self.lib.sri_oracle_integrate_all_batch(
            self.N, B, _p(K), *[_p(a) for a in args],
            _p(out.get("Q")), _p(out.get("r")), _p(out.get("n")), _p(out.get("m")),
            1 if explicit_inverse else 0, int(nthreads))
        out["bad"] = bad
        return out

    def shape_residual(self, K, H_diag, Q, m, M_tip, K0=None, q0=None) -> np.ndarray:
        K = np.ascontiguousarray(K, dtype=np.float64)
        B = K.shape[0]
        rho = np.empty((B, 3, self.N))
        H = np.ascontiguousarray(H_diag, dtype=np.float64)
        for b in range(B):
            self.lib.sri_oracle_shape_residual(
                self._ops, _p(K[b]), None if K0 is None else _p(np.ascontiguousarray(K0[b])), _p(H),
                _p(np.ascontiguousarray(Q[b])), None if q0 is None else _p(np.ascontiguousarray(q0[b])),
                _p(np.ascontiguousarray(m[b])), _p(np.ascontiguousarray(M_tip[b])), rho[b].ctypes.data)
        return rho

    def wrench_local(self, Q, n, m, F_tip, M_tip, q0=None) -> np.ndarray:
        B = Q.shape[0]
        lam = np.empty((B, 6, self.N))
        cz = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        for b in range(B):
            self.lib.sri_oracle_wrench_local(self._ops, _p(cz(Q[b])), None if q0 is None else _p(cz(q0[b])), _p(cz(n[b])),
                                             _p(cz(m[b])), _p(cz(F_tip[b])), _p(cz(M_tip[b])), lam[b].ctypes.data)
        return lam

    def wrench_local_solve(self, K, Q, F_tip, M_tip, q0=None, Gamma=None, fbar=None, lbar=None) -> np.ndarray:
        """Local-frame statics solved directly (strain-dependent collocation operator): Lambda [B][6][N], couple first."""
        B = K.shape[0]
        lam = np.empty((B, 6, self.N))
        cz = lambda a, b: None if a is None else _p(np.ascontiguousarray(a[b], dtype=np.float64))
        keep = []
        for b in range(B):
            args = [np.ascontiguousarray(x[b], dtype=np.float64) if x is not None else None
                    for x in (K, Q, q0, Gamma, fbar, lbar, F_tip, M_tip)]
            keep.append(args)
            bad = self.lib.sri_oracle_wrench_local_solve(self._ops, *[None if a is None else _p(a) for a in args], lam[b].ctypes.data)
            assert bad == 0
        return lam

    def generate_rods(self, seed: int, first_rod: int, batch: int):
        K = np.empty((batch, 3, self.N)); F = np.empty((batch, 3)); Mt = np.empty((batch, 3)); fb = np.empty((batch, 3, self.N))
        self.lib.sri_oracle_generate_rods(self.N, seed, first_rod, batch, K.ctypes.data, F.ctypes.data, Mt.ctypes.data, fb.ctypes.data)
        return K, F, Mt, fb

    def generate_modes(self, seed: int, first_rod: int, batch: int) -> np.ndarray:
        """qe [batch][9] of the rods generate_rods() samples: K_c = qe[3c] P_0 + qe[3c+1] P_1(2X-1)."""
        qe = np.empty((batch, 9))
        self.lib.sri_oracle_generate_modes(seed, first_rod, batch, qe.ctypes.data)
        return qe

    def max_threads(self) -> int:
        return int(self.lib.sri_oracle_max_threads())
