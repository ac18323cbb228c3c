"""Python host-side mirror of the reference's function surface on top of the C ABI (include/sri.h).

The reference is a single C++ translation unit (main.cpp + two headers); its C++ drop-in lives in
include/sri_reference_api.hpp.  This module is the same thin layer for Python callers (tests, bench.py, the Newton
driver): it owns no arithmetic, only pointer plumbing.  Buffers may be torch tensors (CUDA or CPU, float64,
contiguous) or numpy arrays; device tensors are passed through untouched, host arrays are staged by the library.

Reference names kept (file:line under /root/reference):
  ComputeChebyshevPoints  include/chebyshev_differentiation.h:19-30
  GetCoefficients_c       include/chebyshev_differentiation.h:37-52
  getDn                   include/chebyshev_differentiation.h:59-108
  Phi                     include/utilities.h:49-67
  integrateQuaternions    main.cpp:91-118   (the global `qe` becomes an argument)
  updatePositionb         main.cpp:121-140  (folded into integratePosition on the device)
  integratePosition       main.cpp:145-176
"""
from __future__ import annotations

import ctypes
from typing import Optional

import numpy as np

from . import _lib

try:  # torch is plumbing (device memory, streams); the library itself does not depend on it
    import torch
except Exception:  # pragma: no cover
    torch = None


def _is_torch(x) -> bool:
    return torch is not None and isinstance(x, torch.Tensor)


def _ptr(x, name: str = "buffer", dtype=np.float64) -> Optional[int]:
    """Raw address of a contiguous float64 (or int32) buffer; None stays None."""
    if x is None:
        return None
    if _is_torch(x):
        want = torch.float64 if dtype == np.float64 else torch.int32
        if x.dtype != want:
            raise TypeError(f"{name}: expected {want}, got {x.dtype}")
        if not x.is_contiguous():
            raise ValueError(f"{name}: tensor must be contiguous")
        return x.data_ptr()
    if isinstance(x, np.ndarray):
        if x.dtype != dtype:
            raise TypeError(f"{name}: expected {dtype}, got {x.dtype}")
        if not x.flags["C_CONTIGUOUS"]:
            raise ValueError(f"{name}: array must be C-contiguous")
        return x.ctypes.data
    raise TypeError(f"{name}: expected a torch tensor or numpy array, got {type(x)}")


def _empty_like_kind(ref, shape, dtype=np.float64):
    if _is_torch(ref):
        return torch.empty(shape, dtype=torch.float64 if dtype == np.float64 else torch.int32, device=ref.device)
    return np.empty(shape, dtype=dtype)


# ---- strain-independent operator ------------------------------------------------------------------------------

def ComputeChebyshevPoints(N: int, L: float = 1.0) -> np.ndarray:
    x = np.empty(N)
    _lib.check(_lib.load().sri_chebyshev_points(N, float(L), x.ctypes.data), "sri_chebyshev_points")
    return x


def GetCoefficients_c(N: int) -> np.ndarray:
    c = np.empty(N)
    _lib.check(_lib.load().sri_chebyshev_coefficients(N, c.ctypes.data), "sri_chebyshev_coefficients")
    return c


def getDn(N: int) -> np.ndarray:
    """N x N Chebyshev differentiation matrix on [0,1] (returned as a regular numpy matrix, Dn[i, j])."""
    buf = np.empty(N * N)
    _lib.check(_lib.load().sri_chebyshev_dn(N, buf.ctypes.data), "sri_chebyshev_dn")
    return buf.reshape(N, N).T.copy()  # the C ABI is column-major like Eigen


def Phi(na: int, ne: int, X: float, begin: float = 0.0, end: float = 1.0) -> np.ndarray:
    buf = np.empty(na * na * ne)
    _lib.check(_lib.load().sri_phi(na, ne, float(X), float(begin), float(end), buf.ctypes.data), "sri_phi")
    return buf.reshape(na * ne, na).T.copy()


# ---- handle -----------------------------------------------------------------------------------------------------

def skew(v) -> np.ndarray:
    """3x3 hat map, skew(v) w = v x w (include/utilities.h:16-24)."""
    v = np.asarray(v, dtype=np.float64).reshape(3)
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])


def ad(strain) -> np.ndarray:
    """6x6 se(3) adjoint of the strain twist [k; gamma]: [[k^, 0], [gamma^, k^]] (include/utilities.h:27-37)."""
    s = np.asarray(strain, dtype=np.float64).reshape(6)
    out = np.zeros((6, 6))
    out[:3, :3] = skew(s[:3]); out[3:, :3] = skew(s[3:]); out[3:, 3:] = skew(s[:3])
    return out


class SpectralRodIntegrator:
    """Owns an sri_handle: the cached operator set for N nodes on one CUDA device."""

    OPERATORS = {"Dn": 0, "Dn_NN": 1, "Dn_IN": 2, "Dn_NN_inv": 3, "D_TT": 4, "D_TI": 5, "D_TT_inv": 6}

    def __init__(self, N: int = 16, device: int = 0):
        self._lib = _lib.load()
        self._h = ctypes.c_void_p()
        _lib.check(self._lib.sri_create(int(N), int(device), ctypes.byref(self._h)), "sri_create")
        self.N = int(N)
        self.M = self.N - 1
        self.device = int(device)
        self._explicit_stream = False
        self._torch_stream = None

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.sri_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- plumbing
    def set_stream(self, stream) -> None:
        """Enqueue on a torch.cuda.Stream / raw cudaStream_t (None restores the handle's own stream)."""
        if stream is None:
            _lib.check(self._lib.sri_reset_stream(self._h), "sri_reset_stream")
            self._explicit_stream = False
            self._torch_stream = None
            return
        raw = int(getattr(stream, "cuda_stream", stream))
        _lib.check(self._lib.sri_set_stream(self._h, raw if raw else None), "sri_set_stream")
        self._explicit_stream = True

    def _follow_torch(self, *tensors) -> None:
        """Unless a stream was set explicitly, enqueue on torch's current stream whenever a CUDA tensor is passed, so
        that this library's kernels are ordered after the torch work that produced their inputs."""
        if self._explicit_stream or torch is None:
            return
        for x in tensors:
            if x is not None and _is_torch(x) and x.is_cuda:
                cur = torch.cuda.current_stream(x.device).cuda_stream
                if cur != self._torch_stream:
                    _lib.check(self._lib.sri_set_stream(self._h, cur if cur else None), "sri_set_stream")
                    self._torch_stream = cur
                return

    def use_current_torch_stream(self) -> None:
        self.set_stream(torch.cuda.current_stream(self.device))

    def synchronize(self) -> None:
        _lib.check(self._lib.sri_synchronize(self._h), "sri_synchronize")

    def operator(self, name: str) -> np.ndarray:
        which = self.OPERATORS[name]
        M, N = self.M, self.N
        shape = {0: (N, N), 1: (M, M), 2: (M,), 3: (M, M), 4: (M, M), 5: (M,), 6: (M, M)}[which]
        buf = np.empty(int(np.prod(shape)))
        _lib.check(self._lib.sri_get_operator(self._h, which, buf.ctypes.data), "sri_get_operator")
        return buf.reshape(shape[::-1]).T.copy() if len(shape) == 2 else buf

    # -- stages
    def strain_from_modes(self, qe, out=None):
        """qe [batch][3*ne] -> K [batch][3][N] (Phi<3,ne>(x_i)*qe, main.cpp:69)."""
        self._follow_torch(qe)
        batch = qe.shape[0]
        ne = qe.shape[1] // 3
        K = out if out is not None else _empty_like_kind(qe, (batch, 3, self.N))
        _lib.check(self._lib.sri_strain_from_modes(self._h, batch, ne, _ptr(qe, "qe"), _ptr(K, "K")), "sri_strain_from_modes")
        return K

    def strain_from_modes_transpose(self, gK, ne: int, out=None):
        """gK [batch][3][N] -> gqe [batch][3*ne] = sum_i P_k(2 x_i - 1) gK[b][c][i] (the transpose of strain_from_modes,
        no quadrature weights), 1 <= ne <= 8."""
        self._follow_torch(gK)
        batch = gK.shape[0]
        gqe = out if out is not None else _empty_like_kind(gK, (batch, 3 * int(ne)))
        _lib.check(self._lib.sri_strain_from_modes_transpose(self._h, batch, int(ne), _ptr(gK, "gK"), _ptr(gqe, "gqe")),
                   "sri_strain_from_modes_transpose")
        return gqe

    def scale_for_length_(self, length, K=None, Gamma=None, fbar=None, lbar=None) -> None:
        """sri_scale_for_length: scales the given [batch][3][N] arrays IN PLACE by the rod length (a float, or one value per rod as
        an array / tensor).  See scale_for_length() for the out-of-place convenience form."""
        ref = next(a for a in (K, Gamma, fbar, lbar) if a is not None)
        self._follow_torch(ref)
        batch = ref.shape[0]
        per_rod = np.ndim(length) > 0 or _is_torch(length)
        _lib.check(self._lib.sri_scale_for_length(self._h, batch, _ptr(length, "length") if per_rod else None,
                                                  1.0 if per_rod else float(length), _ptr(K, "K"), _ptr(Gamma, "Gamma"),
                                                  _ptr(fbar, "fbar"), _ptr(lbar, "lbar")), "sri_scale_for_length")

    def assemble_A(self, K, out=None):
        """A_NN [batch][4M][4M] of updateA (main.cpp:55-88), returned row/column indexed as A[b, row, col]."""
        self._follow_torch(K)
        batch, n = K.shape[0], 4 * self.M
        buf = out if out is not None else _empty_like_kind(K, (batch, n, n))
        _lib.check(self._lib.sri_assemble_A(self._h, batch, _ptr(K, "K"), _ptr(buf, "A_NN")), "sri_assemble_A")
        return buf.transpose(1, 2) if _is_torch(buf) else buf.transpose(0, 2, 1)  # the ABI is column-major like Eigen

    # -- NCCL residual-norm reduction of the Newton driver (one process per GPU)
    @staticmethod
    def nccl_unique_id() -> bytes:
        buf = ctypes.create_string_buffer(128)
        _lib.check(_lib.load().sri_nccl_unique_id(buf), "sri_nccl_unique_id")
        return buf.raw

    def nccl_init(self, nranks: int, rank: int, unique_id: bytes) -> None:
        """Collective over the ranks: attaches an NCCL communicator to this handle (sri_nccl_init)."""
        assert len(unique_id) == 128
        _lib.check(self._lib.sri_nccl_init(self._h, int(nranks), int(rank), ctypes.c_char_p(unique_id)), "sri_nccl_init")

    def nccl_init_from_torch(self, group=None) -> None:
        """nccl_init with the unique id broadcast from rank 0 over an initialised torch.distributed process group."""
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        box = [self.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0, group=group)
        self.nccl_init(world, rank, box[0])

    def nccl_finalize(self) -> None:
        _lib.check(self._lib.sri_nccl_finalize(self._h), "sri_nccl_finalize")

    def nccl_allreduce_norms(self, norm2_and_max) -> None:
        """In place on a 2-element CUDA tensor: (sum over ranks, max over ranks), asynchronous on the handle's stream."""
        self._follow_torch(norm2_and_max)
        _lib.check(self._lib.sri_nccl_allreduce_norms(self._h, _ptr(norm2_and_max, "norms")), "sri_nccl_allreduce_norms")

    def integrate_quaternions(self, K, q0=None, out=None, info=None):
        self._follow_torch(K)
        batch = K.shape[0]
        Q = out if out is not None else _empty_like_kind(K, (batch, 4, self.M))
        _lib.check(
            self._lib.sri_integrate_quaternions(self._h, batch, _ptr(K, "K"), _ptr(q0, "q0"), _ptr(Q, "Q"), _ptr(info, "info", np.int32)),
            "sri_integrate_quaternions",
        )
        return Q

    def integrate_position(self, Q, Gamma=None, r0=None, out=None):
        self._follow_torch(Q)
        batch = Q.shape[0]
        r = out if out is not None else _empty_like_kind(Q, (batch, 3, self.M))
        _lib.check(
            self._lib.sri_integrate_position(self._h, batch, _ptr(Q, "Q"), _ptr(Gamma, "Gamma"), _ptr(r0, "r0"), _ptr(r, "r")),
            "sri_integrate_position",
        )
        return r

    def integrate_stress(self, F_tip, fbar=None, out=None):
        self._follow_torch(F_tip)
        batch = F_tip.shape[0]
        n = out if out is not None else _empty_like_kind(F_tip, (batch, 3, self.M))
        _lib.check(
            self._lib.sri_integrate_stress(self._h, batch, _ptr(fbar, "fbar"), _ptr(F_tip, "F_tip"), _ptr(n, "n")),
            "sri_integrate_stress",
        )
        return n

    def integrate_couple(self, Q, n, M_tip, q0=None, Gamma=None, lbar=None, out=None):
        self._follow_torch(Q)
        batch = Q.shape[0]
        m = out if out is not None else _empty_like_kind(Q, (batch, 3, self.M))
        _lib.check(
            self._lib.sri_integrate_couple(
                self._h, batch, _ptr(Q, "Q"), _ptr(q0, "q0"), _ptr(Gamma, "Gamma"), _ptr(n, "n"), _ptr(lbar, "lbar"),
                _ptr(M_tip, "M_tip"), _ptr(m, "m")),
            "sri_integrate_couple",
        )
        return m

    def integrate_all(self, K, F_tip=None, M_tip=None, q0=None, r0=None, Gamma=None, fbar=None, lbar=None,
                      Q=None, r=None, n=None, m=None, info=None, want=("Q", "r", "n", "m")):
        """Fused four-stage integration.  Returns a dict with the requested outputs (allocated if not given)."""
        self._follow_torch(K)
        batch = K.shape[0]
        outs = {"Q": Q, "r": r, "n": n, "m": m}
        shapes = {"Q": (batch, 4, self.M), "r": (batch, 3, self.M), "n": (batch, 3, self.M), "m": (batch, 3, self.M)}
        for key in want:
            if outs[key] is None:
                outs[key] = _empty_like_kind(K, shapes[key])
        rb = _lib.RodBatch(
            batch=batch, K=_ptr(K, "K"), q0=_ptr(q0, "q0"), r0=_ptr(r0, "r0"), Gamma=_ptr(Gamma, "Gamma"),
            fbar=_ptr(fbar, "fbar"), lbar=_ptr(lbar, "lbar"), F_tip=_ptr(F_tip, "F_tip"), M_tip=_ptr(M_tip, "M_tip"),
            Q=_ptr(outs["Q"], "Q"), r=_ptr(outs["r"], "r"), n=_ptr(outs["n"], "n"), m=_ptr(outs["m"], "m"),
            info=_ptr(info, "info", np.int32),
        )
        _lib.check(self._lib.sri_integrate_all(self._h, ctypes.byref(rb)), "sri_integrate_all")
        return {k: v for k, v in outs.items() if v is not None}

    def integrate_all_vjp(self, K, Q, n=None, q0=None, Gamma=None, gQ=None, gr=None, gn=None, gm=None, info=None,
                          want=("K", "q0", "r0", "Gamma", "fbar", "lbar", "F_tip", "M_tip"), out=None):
        """sri_integrate_all_vjp: gradients of <gQ,Q> + <gr,r> + <gn,n> + <gm,m> with respect to the inputs named in `want`,
        from the forward's Q (and n, needed with gm).  Cotangents may be None (zero).  Returns a dict of the requested
        gradients (allocated unless given in the dict `out`)."""
        self._follow_torch(K)
        batch, N = K.shape[0], self.N
        shapes = {"K": (batch, 3, N), "q0": (batch, 4), "r0": (batch, 3), "Gamma": (batch, 3, N), "fbar": (batch, 3, N),
                  "lbar": (batch, 3, N), "F_tip": (batch, 3), "M_tip": (batch, 3)}
        given = out or {}
        grads = {key: given[key] if given.get(key) is not None else _empty_like_kind(K, shapes[key]) for key in want}
        rb = _lib.RodBatch(batch=batch, K=_ptr(K, "K"), q0=_ptr(q0, "q0"), Gamma=_ptr(Gamma, "Gamma"), Q=_ptr(Q, "Q"),
                           n=_ptr(n, "n"), info=_ptr(info, "info", np.int32))
        g = lambda key: _ptr(grads.get(key), "grad " + key)
        gb = _lib.RodBatchGrad(gQ=_ptr(gQ, "gQ"), gr=_ptr(gr, "gr"), gn=_ptr(gn, "gn"), gm=_ptr(gm, "gm"), gK=g("K"),
                               gq0=g("q0"), gr0=g("r0"), gGamma=g("Gamma"), gfbar=g("fbar"), glbar=g("lbar"),
                               gF_tip=g("F_tip"), gM_tip=g("M_tip"))
        _lib.check(self._lib.sri_integrate_all_vjp(self._h, ctypes.byref(rb), ctypes.byref(gb)), "sri_integrate_all_vjp")
        return {k: v for k, v in grads.items() if v is not None}

    def shape_residual(self, K, H_diag, Q, m, M_tip, K0=None, q0=None, rho=None, reduce=None):
        self._follow_torch(K)
        batch = K.shape[0]
        H = np.ascontiguousarray(np.asarray(H_diag, dtype=np.float64))
        if rho is None:
            rho = _empty_like_kind(K, (batch, 3, self.N))
        _lib.check(
            self._lib.sri_shape_residual(
                self._h, batch, _ptr(K, "K"), _ptr(K0, "K0"), H.ctypes.data, _ptr(Q, "Q"), _ptr(q0, "q0"), _ptr(m, "m"),
                _ptr(M_tip, "M_tip"), _ptr(rho, "rho"), _ptr(reduce, "reduce")),
            "sri_shape_residual",
        )
        return rho

    def wrench_local(self, Q, n, m, F_tip, M_tip, q0=None, out=None):
        """Local-frame wrench [R^T m; R^T n] at all N nodes, [batch][6][N] (rod_modeling.pdf eqs. 1.29, 2.18)."""
        self._follow_torch(Q)
        batch = Q.shape[0]
        if out is None:
            out = _empty_like_kind(Q, (batch, 6, self.N))
        _lib.check(
            self._lib.sri_wrench_local(self._h, batch, _ptr(Q, "Q"), _ptr(q0, "q0"), _ptr(n, "n"), _ptr(m, "m"),
                                       _ptr(F_tip, "F_tip"), _ptr(M_tip, "M_tip"), _ptr(out, "Lambda")),
            "sri_wrench_local",
        )
        return out

    def integrate_wrench_local(self, K, Q, F_tip, M_tip, q0=None, Gamma=None, fbar=None, lbar=None, out=None, info=None):
        """Local-frame wrench [C; N] by a direct collocation solve of the local-frame statics (N <= 16), [batch][6][N]."""
        self._follow_torch(K)
        batch = K.shape[0]
        if out is None:
            out = _empty_like_kind(K, (batch, 6, self.N))
        _lib.check(
            self._lib.sri_integrate_wrench_local(self._h, batch, _ptr(K, "K"), _ptr(Q, "Q"), _ptr(q0, "q0"), _ptr(Gamma, "Gamma"),
                                                 _ptr(fbar, "fbar"), _ptr(lbar, "lbar"), _ptr(F_tip, "F_tip"),
                                                 _ptr(M_tip, "M_tip"), _ptr(out, "Lambda"), _ptr(info, "info", np.int32)),
            "sri_integrate_wrench_local",
        )
        return out

    def project_onto_modes(self, f, ne: int, out=None):
        """Nodal field f [batch][3][N] -> modal coordinates [batch][3*ne] (Clenshaw-Curtis Galerkin projection)."""
        self._follow_torch(f)
        batch = f.shape[0]
        if out is None:
            out = _empty_like_kind(f, (batch, 3 * ne))
        _lib.check(self._lib.sri_project_onto_modes(self._h, batch, int(ne), _ptr(f, "f"), _ptr(out, "out")), "sri_project_onto_modes")
        return out

    def galerkin_residual(self, K, H_diag, Q, m, M_tip, ne: int, K0=None, q0=None, out=None, reduce=None):
        """g = int Phi^T (H (K - K0) - R(q)^T m) dX in one kernel (shape_residual + project_onto_modes, rho not stored);
        reduce (2 doubles, optional) receives sum g^2 and max |g|, summed in a fixed order."""
        self._follow_torch(K)
        batch = K.shape[0]
        H = np.ascontiguousarray(np.asarray(H_diag, dtype=np.float64))
        if out is None:
            out = _empty_like_kind(K, (batch, 3 * int(ne)))
        _lib.check(
            self._lib.sri_galerkin_residual(
                self._h, batch, int(ne), _ptr(K, "K"), _ptr(K0, "K0"), H.ctypes.data, _ptr(Q, "Q"), _ptr(q0, "q0"),
                _ptr(m, "m"), _ptr(M_tip, "M_tip"), _ptr(out, "g"), _ptr(reduce, "reduce")),
            "sri_galerkin_residual",
        )
        return out

    def galerkin_residual_vjp(self, K, H_diag, Q, m, M_tip, gg, K0=None, q0=None,
                              want=("K", "K0", "H", "Q", "q0", "m", "M_tip"), out=None):
        """sri_galerkin_residual_vjp: gradients of <gg, g> (g = galerkin_residual, gg [batch][3*ne]) with respect to the inputs
        named in `want`; "H" is per rod, [batch][3].  Returns a dict of the requested gradients (allocated unless given in the
        dict `out`)."""
        self._follow_torch(K)
        batch, N, M = K.shape[0], self.N, self.M
        ne = gg.shape[1] // 3
        H = np.ascontiguousarray(np.asarray(H_diag, dtype=np.float64))
        shapes = {"K": (batch, 3, N), "K0": (batch, 3, N), "H": (batch, 3), "Q": (batch, 4, M), "q0": (batch, 4),
                  "m": (batch, 3, M), "M_tip": (batch, 3)}
        given = out or {}
        grads = {key: given[key] if given.get(key) is not None else _empty_like_kind(K, shapes[key]) for key in want}
        g = lambda key: _ptr(grads.get(key), "grad " + key)
        _lib.check(self._lib.sri_galerkin_residual_vjp(
            self._h, batch, int(ne), _ptr(K, "K"), _ptr(K0, "K0"), H.ctypes.data, _ptr(Q, "Q"), _ptr(q0, "q0"), _ptr(m, "m"),
            _ptr(M_tip, "M_tip"), _ptr(gg, "gg"), g("K"), g("K0"), g("H"), g("Q"), g("q0"), g("m"), g("M_tip")),
            "sri_galerkin_residual_vjp")
        return grads

    def static_shape_vjp(self, F_tip, M_tip, qe, gqe, H_diag=(1.0, 1.0, 0.77), K0=None, refine_steps: int = 3, info=None,
                         want=("F_tip", "M_tip", "K0", "H"), out=None, q0=None, Gamma=None, fbar=None, lbar=None):
        """Gradients -(dg/dtheta)^T lam of the equilibrium qe [batch][3*ne] (the caller's converged newton_static_shape
        solution, with the same q0, Gamma, fbar, lbar) for the cotangent gqe, with respect to the parameters named in `want`
        among F_tip, M_tip, K0, H (per rod, [batch][3]), q0, Gamma, fbar, lbar; "lambda" ([batch][3*ne], the adjoint solution)
        and "resid" ([batch], its relative residual) may be requested too.  info: optional int32 [batch] pivot report.
        Returns a dict of the requested arrays (allocated unless given in the dict `out`).  sri_static_problem_vjp when a
        clamp rotation, Gamma or a distributed load is given or its gradient wanted, else sri_static_shape_vjp."""
        self._follow_torch(qe)
        batch, n, N = qe.shape[0], qe.shape[1], self.N
        H = np.ascontiguousarray(np.asarray(H_diag, dtype=np.float64))
        shapes = {"F_tip": (batch, 3), "M_tip": (batch, 3), "K0": (batch, 3, N), "H": (batch, 3), "lambda": (batch, n),
                  "resid": (batch,), "q0": (batch, 4), "Gamma": (batch, 3, N), "fbar": (batch, 3, N), "lbar": (batch, 3, N)}
        given = out or {}
        res = {key: given[key] if given.get(key) is not None else _empty_like_kind(qe, shapes[key]) for key in want}
        g = lambda key: _ptr(res.get(key), key)
        if all(a is None for a in (q0, Gamma, fbar, lbar)) and not set(want) & set(_PROBLEM_INPUTS):
            _lib.check(self._lib.sri_static_shape_vjp(
                self._h, batch, n // 3, H.ctypes.data, _ptr(F_tip, "F_tip"), _ptr(M_tip, "M_tip"), _ptr(K0, "K0"),
                _ptr(qe, "qe"), _ptr(gqe, "gqe"), int(refine_steps), g("F_tip"), g("M_tip"), g("K0"), g("H"), g("lambda"),
                g("resid"), _ptr(info, "info", np.int32)), "sri_static_shape_vjp")
            return res
        prob = _problem(batch, n // 3, H, F_tip, M_tip, K0, q0, Gamma, fbar, lbar)
        grads = _lib.StaticProblemGrad(gF_tip=g("F_tip"), gM_tip=g("M_tip"), gK0=g("K0"), gH=g("H"), gq0=g("q0"),
                                       gGamma=g("Gamma"), gfbar=g("fbar"), glbar=g("lbar"), lambda_=g("lambda"),
                                       resid=g("resid"), info=_ptr(info, "info", np.int32))
        _lib.check(self._lib.sri_static_problem_vjp(self._h, ctypes.byref(prob), _ptr(qe, "qe"), _ptr(gqe, "gqe"),
                                                    int(refine_steps), ctypes.byref(grads)), "sri_static_problem_vjp")
        return res

    def generalised_forces(self, Lambda, ne: int, out=None):
        """Q_ad = -int Phi^T (couple part of the local-frame wrench) dX  (rod_modeling.pdf eqs. 2.16, 2.20)."""
        self._follow_torch(Lambda)
        batch = Lambda.shape[0]
        if out is None:
            out = _empty_like_kind(Lambda, (batch, 3 * int(ne)))
        _lib.check(self._lib.sri_generalised_forces(self._h, batch, int(ne), _ptr(Lambda, "Lambda"), _ptr(out, "Qad")), "sri_generalised_forces")
        return out

    def shape_jacobian(self, Q, n, m, M_tip, ne: int, H_diag, q0=None, Gamma=None, out=None):
        """J[b][j][d] = d g_j / d qe_d of galerkin_residual, analytic and solve-free (sri_shape_jacobian); Q, n, m are the
        stage outputs at the current qe."""
        self._follow_torch(Q)
        batch = Q.shape[0]
        H = np.ascontiguousarray(np.asarray(H_diag, dtype=np.float64))
        nq = 3 * int(ne)
        if out is None:
            out = _empty_like_kind(Q, (batch, nq, nq))
        _lib.check(self._lib.sri_shape_jacobian(self._h, batch, int(ne), H.ctypes.data, _ptr(Q, "Q"), _ptr(q0, "q0"),
                                                _ptr(Gamma, "Gamma"), _ptr(n, "n"), _ptr(m, "m"), _ptr(M_tip, "M_tip"),
                                                _ptr(out, "J")), "sri_shape_jacobian")
        return out

    def newton_static_shape(self, F_tip, M_tip, ne: int, H_diag=(1.0, 1.0, 0.77), qe=None, K0=None, tol: float = 1e-10,
                            max_iter: int = 30, fd_step: float = 1e-6, total_dof: int = 0, allreduce=None, q0=None, Gamma=None,
                            fbar=None, lbar=None):
        """The Newton loop of the static shape problem inside the library: sri_newton_static_shape, or
        sri_newton_static_problem when a clamp rotation q0 [batch][4], Gamma or a global-frame distributed load fbar / lbar
        ([batch][3][N] each) is given.  qe (in/out, zeros when omitted) [batch][3*ne]; allreduce(norms) -- optional callable
        that replaces the 2-element float64 numpy array [sum g^2, max |g|] by its reduction over the ranks.  Returns
        (qe, dict report)."""
        self._follow_torch(F_tip)
        batch = F_tip.shape[0]
        if qe is None:
            qe = _empty_like_kind(F_tip, (batch, 3 * int(ne)))
            if isinstance(qe, np.ndarray):
                qe[...] = 0.0
            else:
                qe.zero_()
        H = np.ascontiguousarray(np.asarray(H_diag, dtype=np.float64))
        rep = _lib.NewtonReport()
        failure = []

        def _cb(ptr, _ctx):
            try:
                allreduce(np.ctypeslib.as_array(ptr, shape=(2,)))
                return 0
            except Exception as exc:  # never unwind through the C frames
                failure.append(exc)
                return 1

        cb = _lib.ALLREDUCE_FN(_cb) if allreduce is not None else _lib.ALLREDUCE_FN()
        if all(a is None for a in (q0, Gamma, fbar, lbar)):
            where = "sri_newton_static_shape"
            rc = self._lib.sri_newton_static_shape(self._h, batch, int(ne), H.ctypes.data, _ptr(F_tip, "F_tip"),
                                                   _ptr(M_tip, "M_tip"), _ptr(K0, "K0"), _ptr(qe, "qe"), float(tol), int(max_iter),
                                                   float(fd_step), int(total_dof), cb, None, ctypes.byref(rep))
        else:
            where = "sri_newton_static_problem"
            prob = _problem(batch, ne, H, F_tip, M_tip, K0, q0, Gamma, fbar, lbar)
            rc = self._lib.sri_newton_static_problem(self._h, ctypes.byref(prob), _ptr(qe, "qe"), float(tol), int(max_iter),
                                                     float(fd_step), int(total_dof), cb, None, ctypes.byref(rep))
        if failure:
            raise failure[0]
        _lib.check(rc, where)
        return qe, _report_dict(rep)

    def solve_small_batched(self, A, b, out=None, info=None):
        """A [batch][n][n] (row-major, destroyed), b [batch][n] -> x [batch][n]; CUDA tensors only."""
        self._follow_torch(A)
        batch, n = b.shape
        if out is None:
            out = _empty_like_kind(b, (batch, n))
        _lib.check(self._lib.sri_solve_small_batched(self._h, batch, n, _ptr(A, "A"), _ptr(b, "b"), _ptr(out, "x"),
                                                     _ptr(info, "info", np.int32)), "sri_solve_small_batched")
        return out

    def generate_rods(self, seed: int, first_rod: int, batch: int, K=None, F_tip=None, M_tip=None, fbar=None):
        self._follow_torch(K, F_tip, M_tip, fbar)
        _lib.check(
            self._lib.sri_generate_rods(self._h, seed, first_rod, batch, _ptr(K, "K"), _ptr(F_tip, "F_tip"),
                                        _ptr(M_tip, "M_tip"), _ptr(fbar, "fbar")),
            "sri_generate_rods",
        )

    def set_timing(self, enabled: bool = True) -> None:
        """CUDA-event timer around every following call on this handle (sri_set_timing)."""
        _lib.check(self._lib.sri_set_timing(self._h, 1 if enabled else 0), "sri_set_timing")

    def last_timing(self):
        """(milliseconds on the device, entry point name) of the most recent timed call."""
        ms = ctypes.c_float()
        name = ctypes.c_char_p()
        _lib.check(self._lib.sri_get_last_timing(self._h, ctypes.byref(ms), ctypes.byref(name)), "sri_get_last_timing")
        return float(ms.value), (name.value.decode() if name.value else "")

    def handback_count(self) -> int:
        """Rods of the last device-buffer call that the DMMA elimination handed back to the row-pivoting kernel."""
        v = ctypes.c_int64()
        _lib.check(self._lib.sri_get_handback_count(self._h, ctypes.byref(v)), "sri_get_handback_count")
        return int(v.value)

    def measure_fp64_peak(self) -> float:
        v = ctypes.c_double()
        _lib.check(self._lib.sri_measure_fp64_peak(self._h, ctypes.byref(v)), "sri_measure_fp64_peak")
        return v.value

    def measure_dmma_peak(self) -> float:
        v = ctypes.c_double()
        _lib.check(self._lib.sri_measure_dmma_peak(self._h, ctypes.byref(v)), "sri_measure_dmma_peak")
        return v.value


def scale_for_length(length, K, Gamma=None, fbar=None, lbar=None):
    """Inputs of a rod of length `length` (scalar, or one value per rod) for the unit-interval integrators.

    The reference integrates on X in [0, 1] with an implicit rod length of 1 (main.cpp:15 uses ComputeChebyshevPoints<N, 1>).
    For a rod of length l every ODE is multiplied by l (rod_modeling.pdf eq. 2.17): Q' = l/2 Q (x) (0,K), r' = l R Gamma,
    n' = -l fbar, m' = -(r' x n + l lbar), so the library is called with (l K, l Gamma, l fbar, l lbar); the tip loads and
    every output (Q, r, n, m at the nodes X_i = s_i / l) are unchanged.  Gamma = None means (1,0,0) and becomes (l,0,0).
    Returns (K, Gamma, fbar, lbar) scaled, same array kind as K; None stays None for the loads."""
    if _is_torch(K):
        ell = torch.as_tensor(length, dtype=K.dtype, device=K.device).reshape(-1, 1, 1)
    else:
        ell = np.asarray(length, dtype=np.float64).reshape(-1, 1, 1)
    if Gamma is None:
        e1 = (torch.zeros_like(K) if _is_torch(K) else np.zeros_like(K))
        e1[:, 0, :] = 1.0
        Gamma = e1
    sc = lambda a: None if a is None else (a * ell).contiguous() if _is_torch(a) else np.ascontiguousarray(a * ell)
    return sc(K), sc(Gamma), sc(fbar), sc(lbar)


_PROBLEM_INPUTS = ("q0", "Gamma", "fbar", "lbar")


def _problem(batch, ne, H, F_tip, M_tip, K0, q0, Gamma, fbar, lbar):
    """struct sri_static_problem over the given buffers (H: a contiguous numpy array the caller keeps alive)."""
    return _lib.StaticProblem(batch=batch, ne=int(ne), H_diag=H.ctypes.data, F_tip=_ptr(F_tip, "F_tip"),
                              M_tip=_ptr(M_tip, "M_tip"), K0=_ptr(K0, "K0"), q0=_ptr(q0, "q0"), Gamma=_ptr(Gamma, "Gamma"),
                              fbar=_ptr(fbar, "fbar"), lbar=_ptr(lbar, "lbar"))


def _report_dict(rep) -> dict:
    return {"iterations": rep.iterations, "converged": bool(rep.converged), "integrations": rep.integrations,
            "rms": rep.rms, "max_abs": rep.max_abs, "rms_history": list(rep.rms_history[:rep.history_len]),
            "singular_solves": rep.singular_solves}


def shard_range(total: int, rank: int, world: int):
    """sri_shard_range: [floor(rank*total/world), floor((rank+1)*total/world))."""
    a, b = ctypes.c_int64(), ctypes.c_int64()
    _lib.check(_lib.load().sri_shard_range(int(total), int(rank), int(world), ctypes.byref(a), ctypes.byref(b)), "sri_shard_range")
    return int(a.value), int(b.value)


class MultiDeviceIntegrator:
    """sri_multi_handle: one operator set per device, rods sharded by index, one host thread per device inside the library
    (the C/C++ host's multi-GPU path; bench.py uses one process per GPU instead)."""

    def __init__(self, N: int = 16, devices=None, ndev: int = None):
        self._lib = _lib.load()
        self._mh = ctypes.c_void_p()
        if devices is not None:
            arr = (ctypes.c_int * len(devices))(*devices)
            _lib.check(self._lib.sri_create_multi(int(N), arr, len(devices), ctypes.byref(self._mh)), "sri_create_multi")
        else:
            _lib.check(self._lib.sri_create_multi(int(N), None, int(ndev), ctypes.byref(self._mh)), "sri_create_multi")
        self.N, self.M = int(N), int(N) - 1

    def close(self) -> None:
        if getattr(self, "_mh", None) is not None and self._mh:
            self._lib.sri_destroy_multi(self._mh)
            self._mh = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @property
    def device_count(self) -> int:
        v = ctypes.c_int()
        _lib.check(self._lib.sri_multi_device_count(self._mh, ctypes.byref(v)), "sri_multi_device_count")
        return v.value

    def integrate_all(self, K, F_tip=None, M_tip=None, q0=None, r0=None, Gamma=None, fbar=None, lbar=None, info=None,
                      want=("Q", "r", "n", "m")):
        """Host (numpy / CPU torch) buffers, sharded over the devices; returns the requested outputs as numpy arrays."""
        batch = K.shape[0]
        shapes = {"Q": (batch, 4, self.M), "r": (batch, 3, self.M), "n": (batch, 3, self.M), "m": (batch, 3, self.M)}
        outs = {k: (np.empty(shapes[k]) if k in want else None) for k in "Qrnm"}
        rb = _lib.RodBatch(
            batch=batch, K=_ptr(K, "K"), q0=_ptr(q0, "q0"), r0=_ptr(r0, "r0"), Gamma=_ptr(Gamma, "Gamma"),
            fbar=_ptr(fbar, "fbar"), lbar=_ptr(lbar, "lbar"), F_tip=_ptr(F_tip, "F_tip"), M_tip=_ptr(M_tip, "M_tip"),
            Q=_ptr(outs["Q"], "Q"), r=_ptr(outs["r"], "r"), n=_ptr(outs["n"], "n"), m=_ptr(outs["m"], "m"),
            info=_ptr(info, "info", np.int32))
        _lib.check(self._lib.sri_integrate_all_sharded(self._mh, ctypes.byref(rb)), "sri_integrate_all_sharded")
        return {k: v for k, v in outs.items() if v is not None}

    def newton_static_shape(self, F_tip, M_tip, ne: int, H_diag=(1.0, 1.0, 0.77), qe=None, K0=None, tol: float = 1e-10,
                            max_iter: int = 30, fd_step: float = 0.0, q0=None, Gamma=None, fbar=None, lbar=None):
        """Host buffers, rods sharded over the devices: sri_newton_static_shape_sharded, or sri_newton_static_problem_sharded
        when q0, Gamma, fbar or lbar is given."""
        batch = F_tip.shape[0]
        if qe is None:
            qe = np.zeros((batch, 3 * int(ne)))
        H = np.ascontiguousarray(np.asarray(H_diag, dtype=np.float64))
        rep = _lib.NewtonReport()
        if all(a is None for a in (q0, Gamma, fbar, lbar)):
            _lib.check(self._lib.sri_newton_static_shape_sharded(
                self._mh, batch, int(ne), H.ctypes.data, _ptr(F_tip, "F_tip"), _ptr(M_tip, "M_tip"), _ptr(K0, "K0"),
                _ptr(qe, "qe"), float(tol), int(max_iter), float(fd_step), ctypes.byref(rep)), "sri_newton_static_shape_sharded")
        else:
            prob = _problem(batch, ne, H, F_tip, M_tip, K0, q0, Gamma, fbar, lbar)
            _lib.check(self._lib.sri_newton_static_problem_sharded(
                self._mh, ctypes.byref(prob), _ptr(qe, "qe"), float(tol), int(max_iter), float(fd_step), ctypes.byref(rep)),
                "sri_newton_static_problem_sharded")
        return qe, _report_dict(rep)


def kernel_launch_count() -> int:
    return int(_lib.load().sri_kernel_launch_count())


# ---- the reference's stage functions, single rod, modal strain input (main.cpp:181-205) -----------------------

def integrateQuaternions(qe, N: int = 16, device: int = 0) -> np.ndarray:
    """Q_stack (4*(N-1),) for one rod with modal strain coordinates qe (9,), as main.cpp:197 prints it."""
    qe = np.ascontiguousarray(np.asarray(qe, dtype=np.float64).reshape(1, -1))
    with SpectralRodIntegrator(N, device) as h:
        K = h.strain_from_modes(qe)
        return h.integrate_quaternions(K).reshape(-1)


def integratePosition(qe, N: int = 16, device: int = 0) -> np.ndarray:
    """r_stack ((N-1), 3) for one rod, as main.cpp:201 prints it (row i = node i)."""
    qe = np.ascontiguousarray(np.asarray(qe, dtype=np.float64).reshape(1, -1))
    with SpectralRodIntegrator(N, device) as h:
        K = h.strain_from_modes(qe)
        out = h.integrate_all(K, want=("Q", "r"))
        return out["r"].reshape(3, N - 1).T.copy()
