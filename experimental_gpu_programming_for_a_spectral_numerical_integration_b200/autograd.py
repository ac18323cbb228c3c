"""torch.autograd bindings of the four-stage integration and of the modal strain adapter.

    Q, r, n, m = integrate_all(integ, K, F_tip, M_tip, q0=..., r0=..., Gamma=..., fbar=..., lbar=...)
    K = strain_from_modes(integ, qe, ne)
    g = galerkin_residual(integ, K, Q, m, M_tip, ne, H_diag, K0=..., q0=...)
    qe = static_shape(integ, F_tip, M_tip, ne, H_diag, K0=..., qe0=..., q0=..., Gamma=..., fbar=..., lbar=...)
                                                                           (the equilibrium, differentiated implicitly)

are differentiable with respect to every tensor argument: the backward pass is one sri_integrate_all_vjp launch (resp.
sri_strain_from_modes_transpose, sri_galerkin_residual_vjp, sri_static_shape_vjp / sri_static_problem_vjp), enqueued on torch's current stream like the forward.  Only what the backward needs is
saved (K, Q, n, and q0 / Gamma when given), not the graph of the forward.  Gradients are computed for the inputs that
require them only, and outputs that receive no cotangent pass none to the library.  Tensors are CUDA float64 on the
integrator's device; H_diag may be a 3-tensor (on any device) that requires grad, or a sequence of 3 floats.
SpectralRodIntegrator.integrate_all itself stays a plain (non-differentiable) call.

static_shape's backward is the implicit-function theorem, not an unrolled Newton loop: one sri_static_shape_vjp at the
forward's solution (DESIGN section 5e).  Its gradients are those of the equilibrium, so its forward raises when the Newton
solve did not converge.
"""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable

_INPUTS = ("K", "F_tip", "M_tip", "q0", "r0", "Gamma", "fbar", "lbar")


def _c(x):
    return None if x is None else x.contiguous()


class _IntegrateAll(torch.autograd.Function):
    @staticmethod
    def forward(ctx, integ, K, F_tip, M_tip, q0, r0, Gamma, fbar, lbar):
        out = integ.integrate_all(K, F_tip, M_tip, q0=q0, r0=r0, Gamma=Gamma, fbar=fbar, lbar=lbar)
        ctx.integ = integ
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(K, out["Q"], out["n"], q0, Gamma)
        return out["Q"], out["r"], out["n"], out["m"]

    @staticmethod
    @once_differentiable
    def backward(ctx, gQ, gr, gn, gm):
        K, Q, n, q0, Gamma = ctx.saved_tensors
        want = [name for name, need in zip(_INPUTS, ctx.needs_input_grad[1:]) if need]
        grads = {}
        if want:
            grads = ctx.integ.integrate_all_vjp(K, Q, n=n if gm is not None else None, q0=q0, Gamma=Gamma, gQ=_c(gQ),
                                                gr=_c(gr), gn=_c(gn), gm=_c(gm), want=want)
        return (None,) + tuple(grads.get(name) for name in _INPUTS)


class _StrainFromModes(torch.autograd.Function):
    @staticmethod
    def forward(ctx, integ, qe, ne):
        ctx.integ, ctx.ne = integ, ne
        return integ.strain_from_modes(qe)

    @staticmethod
    @once_differentiable
    def backward(ctx, gK):
        return None, ctx.integ.strain_from_modes_transpose(gK.contiguous(), ctx.ne), None


def integrate_all(integ, K, F_tip=None, M_tip=None, q0=None, r0=None, Gamma=None, fbar=None, lbar=None):
    """Differentiable four-stage integration on the SpectralRodIntegrator `integ`: returns (Q, r, n, m).  F_tip / M_tip
    None mean no tip load (zeros); the other optional inputs take the library's defaults (q0 identity, r0 = 0,
    Gamma = e1, no distributed loads)."""
    B = K.shape[0]
    if F_tip is None:
        F_tip = K.new_zeros((B, 3))
    if M_tip is None:
        M_tip = K.new_zeros((B, 3))
    return _IntegrateAll.apply(integ, _c(K), _c(F_tip), _c(M_tip), _c(q0), _c(r0), _c(Gamma), _c(fbar), _c(lbar))


def strain_from_modes(integ, qe, ne: int):
    """Differentiable modal strain adapter: qe [batch][3*ne] -> K [batch][3][N] (its backward needs 1 <= ne <= 8)."""
    if qe.shape[-1] != 3 * int(ne):
        raise ValueError(f"qe has {qe.shape[-1]} coordinates per rod, expected 3*ne = {3 * int(ne)}")
    return _StrainFromModes.apply(integ, _c(qe), int(ne))


def _H(H_diag):
    """(tensor or None, tuple of 3 floats) of a stiffness given as a tensor or as a sequence."""
    if isinstance(H_diag, torch.Tensor):
        return H_diag, tuple(float(v) for v in H_diag.detach().to("cpu", torch.float64).reshape(3))
    return None, tuple(float(v) for v in H_diag)


class _GalerkinResidual(torch.autograd.Function):
    @staticmethod
    def forward(ctx, integ, ne, Hv, K, Q, m, M_tip, H_t, K0, q0):
        ctx.integ, ctx.Hv = integ, Hv
        ctx.save_for_backward(K, Q, m, M_tip, K0, q0)
        return integ.galerkin_residual(K, Hv, Q, m, M_tip, ne, K0=K0, q0=q0)

    @staticmethod
    @once_differentiable
    def backward(ctx, gg):
        K, Q, m, M_tip, K0, q0 = ctx.saved_tensors
        names = ("K", "Q", "m", "M_tip", "H", "K0", "q0")
        want = [name for name, need in zip(names, ctx.needs_input_grad[3:]) if need]
        grads = {}
        if want:
            grads = ctx.integ.galerkin_residual_vjp(K, ctx.Hv, Q, m, M_tip, gg.contiguous(), K0=K0, q0=q0, want=want)
            if "H" in grads:
                grads["H"] = grads["H"].sum(0)
        return (None, None, None) + tuple(grads.get(name) for name in names)


class _StaticShape(torch.autograd.Function):
    @staticmethod
    def forward(ctx, integ, ne, Hv, tol, max_iter, refine_steps, F_tip, M_tip, H_t, K0, qe0, q0, Gamma, fbar, lbar):
        qe = None if qe0 is None else qe0.detach().clone()
        qe, rep = integ.newton_static_shape(F_tip, M_tip, ne, H_diag=Hv, qe=qe, K0=K0, tol=tol, max_iter=max_iter, fd_step=0.0,
                                            q0=q0, Gamma=Gamma, fbar=fbar, lbar=lbar)
        if not rep["converged"]:
            raise RuntimeError(f"static_shape: the Newton solve did not converge (rms {rep['rms']:.3e} after "
                               f"{rep['iterations']} iterations, tol {tol:.1e}); its gradient would not be that of an equilibrium")
        ctx.integ, ctx.Hv, ctx.refine_steps = integ, Hv, refine_steps
        ctx.save_for_backward(F_tip, M_tip, K0, qe, q0, Gamma, fbar, lbar)
        return qe

    @staticmethod
    @once_differentiable
    def backward(ctx, gqe):
        F_tip, M_tip, K0, qe, q0, Gamma, fbar, lbar = ctx.saved_tensors
        names = ("F_tip", "M_tip", "H", "K0", "qe0", "q0", "Gamma", "fbar", "lbar")
        want = [name for name, need in zip(names, ctx.needs_input_grad[6:]) if need and name != "qe0"]
        grads = {}
        if want:
            info = torch.empty(qe.shape[0], dtype=torch.int32, device=qe.device)
            grads = ctx.integ.static_shape_vjp(F_tip, M_tip, qe, gqe.contiguous(), H_diag=ctx.Hv, K0=K0,
                                               refine_steps=ctx.refine_steps, info=info, want=want, q0=q0, Gamma=Gamma,
                                               fbar=fbar, lbar=lbar)
            bad = int((info != 0).sum())
            if bad:
                raise RuntimeError(f"static_shape backward: {bad} rod(s) met a zero or non-finite pivot in the adjoint solve")
            if "H" in grads:
                grads["H"] = grads["H"].sum(0)
        return (None,) * 6 + tuple(grads.get(name) for name in names)


def galerkin_residual(integ, K, Q, m, M_tip, ne: int, H_diag, K0=None, q0=None):
    """Differentiable Galerkin residual g [batch][3*ne] of the static shape problem (sri_galerkin_residual; backward: one
    sri_galerkin_residual_vjp) with respect to K, Q, m, M_tip, H_diag (when a tensor), K0 and q0."""
    H_t, Hv = _H(H_diag)
    return _GalerkinResidual.apply(integ, int(ne), Hv, _c(K), _c(Q), _c(m), _c(M_tip), H_t, _c(K0), _c(q0))


def static_shape(integ, F_tip, M_tip, ne: int, H_diag, K0=None, qe0=None, tol: float = 1e-12, max_iter: int = 30,
                 refine_steps: int = 3, q0=None, Gamma=None, fbar=None, lbar=None):
    """Differentiable equilibrium qe* [batch][3*ne] of rods under tip loads, a clamp rotation q0 [batch][4], Gamma and the
    global-frame distributed loads fbar, lbar ([batch][3][N] each; None: identity, e1, 0): the forward is newton_static_shape
    with the analytic Jacobian (raises unless it converges), the backward one static_shape_vjp with `refine_steps` refinement
    steps, differentiating with respect to F_tip, M_tip, H_diag (when a tensor), K0, q0, Gamma, fbar and lbar -- not qe0,
    the starting point."""
    H_t, Hv = _H(H_diag)
    return _StaticShape.apply(integ, int(ne), Hv, float(tol), int(max_iter), int(refine_steps), _c(F_tip), _c(M_tip), H_t,
                              _c(K0), _c(qe0), _c(q0), _c(Gamma), _c(fbar), _c(lbar))
