"""torch.autograd bindings of the four-stage integration and of the modal strain adapter.

    Q, r, n, m = integrate_all(integ, K, F_tip, M_tip, q0=..., r0=..., Gamma=..., fbar=..., lbar=...)
    K = strain_from_modes(integ, qe, ne)

are differentiable with respect to every tensor argument: the backward pass is one sri_integrate_all_vjp launch (resp.
sri_strain_from_modes_transpose), enqueued on torch's current stream like the forward.  Only what the backward needs is
saved (K, Q, n, and q0 / Gamma when given), not the graph of the forward.  Gradients are computed for the inputs that
require them only, and outputs that receive no cotangent pass none to the library.  Tensors are CUDA float64 on the
integrator's device.  SpectralRodIntegrator.integrate_all itself stays a plain (non-differentiable) call.
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
