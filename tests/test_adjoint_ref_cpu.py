"""The extended-precision reverse-mode reference of tests/adjoint_ref.py, pinned on the CPU before the GPU tests rely on it.

For every node count 2..64: the transposed system is the oracle's operator; the reference agrees with oracle/adjoint.py and
its refinement has converged; the stage bounds admit the oracle's plain float64 gradients and see a perturbation of 1e-13
of the rod's largest entry placed on the nodal entry with the smallest bound; and the adjoint passes an exact dot-product test against a long-double
tangent of the same discrete map, at 1e-15 of the sum of the terms instead of the 1e-7 of central differences.
"""
import numpy as np
import pytest

from adjoint_ref import (INPUTS, _cross, _rot, excess, integrate_all_vjp, norm_inf, reverse_stages, stage1_grads,
                         transposed_system)
from elimination_ref import LD, U, Tables, refine_step, refined_solve

B = 6
STAGE_GRADS = ("lbar", "M_tip", "fbar", "F_tip", "r0", "Gamma")


def _inputs(o, N, seed, B=B):
    """Generator rods with every optional input (as tests/test_elimination_ref_cpu.py) and four random cotangents."""
    rng = np.random.default_rng(seed)
    K, F, Mt, fb = o.generate_rods(0x5EED, 1000 * N + 7, B)
    q0 = rng.normal(size=(B, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    Gamma = np.concatenate([1 + 0.1 * rng.normal(size=(B, 1, N)), 0.1 * rng.normal(size=(B, 2, N))], axis=1)
    a = dict(K=K, F_tip=F, M_tip=Mt, q0=q0, r0=rng.normal(size=(B, 3)), Gamma=Gamma, fbar=fb, lbar=rng.normal(size=(B, 3, N)))
    M = N - 1
    cot = {"gQ": rng.normal(size=(B, 4, M)), "gr": rng.normal(size=(B, 3, M)), "gn": rng.normal(size=(B, 3, M)),
           "gm": rng.normal(size=(B, 3, M))}
    return a, cot


def _rod_rel(x, ref):
    x = np.asarray(x, dtype=np.float64).reshape(x.shape[0], -1)
    ref = np.asarray(ref, dtype=np.float64).reshape(ref.shape[0], -1)
    return np.abs(x - ref).max(axis=1) / np.maximum(np.abs(ref).max(axis=1), 1e-300)


def _node_major_A(o, K, M):
    perm = np.array([c * M + j for j in range(M) for c in range(4)])  # node-major index -> the oracle's block order
    return np.stack([o.assemble_A(k)[np.ix_(perm, perm)] for k in K])


@pytest.mark.parametrize("N", range(2, 65))
def test_reference_against_oracle_adjoint(make_oracle, N):
    from oracle.adjoint import integrate_all_vjp as oracle_vjp
    o = make_oracle(N)
    tab = Tables.from_oracle(o)
    a, cot = _inputs(o, N, N)
    fwd = o.integrate_all(a["K"], a["F_tip"], a["M_tip"], q0=a["q0"], r0=a["r0"], Gamma=a["Gamma"], fbar=a["fbar"],
                          lbar=a["lbar"], explicit_inverse=False)
    assert fwd["bad"] == 0
    ref = integrate_all_vjp(tab, a["K"], fwd["Q"], fwd["n"], a["q0"], a["Gamma"], **cot)
    orc = oracle_vjp(o, a["K"], fwd["Q"], n=fwd["n"], q0=a["q0"], Gamma=a["Gamma"], **cot)
    assert orc["bad"] == 0
    level = {k: float(_rod_rel(orc[k], ref.value[k]).max()) for k in INPUTS}
    print(f"[adjoint_ref] N={N}: oracle/adjoint.py vs long double, worst rod per gradient: "
          + ", ".join(f"{k} {v:.1e}" for k, v in level.items()))
    assert max(level.values()) <= 5e-14, level

    # converged: one more refinement step moves lam' by less than 1e-17 relative
    _, rel = refine_step(ref.C, ref.lam.reshape(B, -1), ref.b)
    assert rel.max() < 1e-17

    # the stage bounds admit a plain float64 evaluation (the oracle's own gradients, numpy's summation order) ...
    for k in STAGE_GRADS:
        assert excess(orc[k], ref, k).max() <= 1.0, k
    # ... and are not blind: 1e-13 of the rod's largest entry, added to the nodal entry with the smallest non-zero bound
    # (the tip gradients are three sums each, whose bound is set by their cancellation, up to 3e-12 of the entry at N = 64)
    for k in ("lbar", "fbar", "Gamma"):
        bound = ref.bound[k].reshape(B, -1)
        pert = np.asarray(orc[k], dtype=np.float64).reshape(B, -1).copy()
        idx = np.where(bound > 0, bound, np.inf).argmin(axis=1)
        pert[np.arange(B), idx] += 1e-13 * np.abs(pert).max(axis=1)
        assert (excess(pert.reshape(orc[k].shape), ref, k) > 1.0).all(), k


@pytest.mark.parametrize("N", [2, 3, 9, 16, 17, 33, 64])
def test_transposed_system_is_the_oracle_operator(make_oracle, N):
    """C' = (S^T x I4) A_NN^T in node-major order, up to the rounding of S (|Dn_NN S - I|) and of the entries fl(1/2 S_ji K_j)."""
    o = make_oracle(N)
    M = N - 1
    tab = Tables.from_oracle(o)
    K, _, _, _ = o.generate_rods(3, N, 2)
    C = transposed_system(tab, K)
    A = _node_major_A(o, K, M)
    Dn = _node_major_A(o, np.zeros((1, 3, N)), M)[0][::4, ::4]  # A_NN(0) = Dn_NN x I4
    SAT = np.einsum("ki,bkj->bij", np.kron(tab.S, np.eye(4)).astype(LD), np.swapaxes(A, 1, 2).astype(LD))
    dS = np.abs(Dn.astype(LD) @ tab.S.astype(LD) - np.eye(M)).T.astype(np.float64)  # |(Dn S - I)_ji|
    bound = np.kron(dS, np.eye(4))[None] * (1 + 1e-6) + 2 * U * np.abs(C) + 1e-25
    err = np.abs(SAT - C).astype(np.float64)
    assert (err <= bound).all(), float((err / bound).max())


def _forward_ld(tab, A, x):
    """The discrete four-stage map in long double with A_NN given (float64, node-major): Q, qn, b, r, n, m."""
    Bn, M, N = A.shape[0], tab.M, tab.N
    S, ST, dti, dnin = (np.asarray(t).astype(LD) for t in (tab.S, tab.ST, tab.D_TI, tab.Dn_IN))
    q0 = x["q0"].astype(LD)
    rhs = (-dnin[None, :, None] * q0[:, None, :]).reshape(Bn, 4 * M)
    Qx = refined_solve(A, rhs).reshape(Bn, M, 4)
    qn = np.concatenate([Qx, q0[:, None, :]], axis=1)
    gam = np.swapaxes(x["Gamma"], 1, 2).astype(LD)
    b, _ = _rot(qn, gam)
    r = np.einsum("ij,bjc->bic", S, b[:, :M] - dnin[None, :, None] * x["r0"].astype(LD)[:, None, :])
    f, lb = (np.swapaxes(x[k], 1, 2).astype(LD)[:, 1:] for k in ("fbar", "lbar"))
    n = np.einsum("ij,bjc->bic", ST, -f - dti[None, :, None] * x["F_tip"].astype(LD)[:, None, :])
    m = np.einsum("ij,bjc->bic", ST, -(_cross(b[:, 1:], n) + lb) - dti[None, :, None] * x["M_tip"].astype(LD)[:, None, :])
    return {"Q": Qx, "qn": qn, "b": b, "r": r, "n": n, "m": m}


def _tangent_ld(tab, A, A0, Ad, x, fw, d):
    """The exact tangent of _forward_ld at x in the direction d (every input of d; A0 = A_NN(0), Ad = A_NN(dK)).  R is
    quadratic in q, so the polarisation identity R(q+dq) - R(q) - R(dq) + I makes dR exact."""
    Bn, M = A.shape[0], tab.M
    S, ST, dti, dnin = (np.asarray(t).astype(LD) for t in (tab.S, tab.ST, tab.D_TI, tab.Dn_IN))
    dq0 = d["q0"].astype(LD)
    drhs = (-dnin[None, :, None] * dq0[:, None, :]).reshape(Bn, 4 * M)
    dAQ = np.matmul((Ad - A0).astype(LD), fw["Q"].reshape(Bn, 4 * M, 1))[..., 0]   # dA = A(dK) - A(0), exact
    v = drhs - dAQ
    dQ = (refined_solve(A, v) if v.any() else v).reshape(Bn, M, 4)  # (a zero direction has no relative correction)
    dqn = np.concatenate([dQ, dq0[:, None, :]], axis=1)
    gam = np.swapaxes(x["Gamma"], 1, 2).astype(LD)
    dgam = np.swapaxes(d["Gamma"], 1, 2).astype(LD)
    qn = fw["qn"]
    db = _rot(qn + dqn, gam)[0] - _rot(qn, gam)[0] - _rot(dqn, gam)[0] + gam + _rot(qn, dgam)[0]
    dr = np.einsum("ij,bjc->bic", S, db[:, :M] - dnin[None, :, None] * d["r0"].astype(LD)[:, None, :])
    df, dl = (np.swapaxes(d[k], 1, 2).astype(LD)[:, 1:] for k in ("fbar", "lbar"))
    dn = np.einsum("ij,bjc->bic", ST, -df - dti[None, :, None] * d["F_tip"].astype(LD)[:, None, :])
    dcr = _cross(db[:, 1:], fw["n"]) + _cross(fw["b"][:, 1:], dn)
    dm = np.einsum("ij,bjc->bic", ST, -(dcr + dl) - dti[None, :, None] * d["M_tip"].astype(LD)[:, None, :])
    return {"Q": dQ, "r": dr, "n": dn, "m": dm}


@pytest.mark.parametrize("N", range(2, 65))
def test_dot_product_exact(make_oracle, N):
    """<gbar, J dtheta> = <J^T gbar, dtheta> in long double for each of the eight inputs alone and all together, with the
    adjoint's stage 1 solved as A_NN^T lam = r; then lam against lam' of the preconditioned C' (the reference the GPU
    tests use), whose difference is the rounding of S: C'(lam' - lam) = (S^T A_NN^T - C') lam."""
    o = make_oracle(N)
    M = N - 1
    tab = Tables.from_oracle(o)
    Bn = 2
    x, cot = _inputs(o, N, 500 + N, B=Bn)
    rng = np.random.default_rng(N)
    d = {k: rng.normal(size=v.shape) for k, v in x.items()}
    A = _node_major_A(o, x["K"], M)
    A0 = _node_major_A(o, np.zeros_like(x["K"]), M)
    fw = _forward_ld(tab, A, x)
    st = reverse_stages(tab, np.swapaxes(fw["Q"], 1, 2), np.swapaxes(fw["n"], 1, 2), x["q0"], x["Gamma"], **cot)
    lam = refined_solve(np.swapaxes(A, 1, 2), st["r"].reshape(Bn, 4 * M)).reshape(Bn, M, 4)
    gK, gq0 = stage1_grads(st["qn"], lam, st["gq"], tab.Dn_IN)
    grad = {"K": gK, "q0": gq0, **{k: v for k, (v, _) in st["out"].items()}}
    cotl = {s: np.swapaxes(cot["g" + s], 1, 2).astype(LD) for s in "Qrnm"}  # [B][M][k]
    worst = 0.0
    for keys in [(k,) for k in INPUTS] + [INPUTS]:
        dk = {k: (d[k] if k in keys else np.zeros_like(d[k])) for k in INPUTS}
        Ad = _node_major_A(o, dk["K"], M)
        t = _tangent_ld(tab, A, A0, Ad, x, fw, dk)
        lhs = sum((cotl[s] * t[s]).sum() for s in "Qrnm")
        terms = [grad[k] * np.asarray(dk[k]).astype(LD) for k in keys]
        rhs = sum(tm.sum() for tm in terms)
        scale = sum(np.abs(tm).sum() for tm in terms)
        worst = max(worst, float(abs(lhs - rhs) / scale))
        assert abs(lhs - rhs) <= 1e-15 * scale, (keys, float(lhs), float(rhs), float(scale))

    # lam' of C' (what the kernels solve) against lam of A_NN^T: the rounding of S, bounded through C'^-1
    C = transposed_system(tab, x["K"])
    bp = np.einsum("ji,bjc->bic", tab.S.astype(LD), st["r"]).reshape(Bn, 4 * M)
    lamp = refined_solve(C, bp)
    lv = lam.reshape(Bn, 4 * M)
    SAl = np.einsum("ji,bjc->bic", tab.S.astype(LD), np.matmul(np.swapaxes(A, 1, 2).astype(LD), lv[..., None])[..., 0]
                    .reshape(Bn, M, 4)).reshape(Bn, 4 * M)
    rho = SAl - np.matmul(C.astype(LD), lv[..., None])[..., 0]
    diff = np.abs(lamp - lv).max(axis=1).astype(np.float64)
    lnorm = np.abs(lv).max(axis=1).astype(np.float64)
    bound = norm_inf(np.linalg.inv(C)) * np.abs(rho).max(axis=1).astype(np.float64) * 1.01 + 1e-17 * lnorm
    print(f"[adjoint_ref] N={N}: dot product worst |lhs - rhs| / sum|terms| {worst:.1e}; "
          f"|lam' - lam| / |lam| {float((diff / lnorm).max()):.1e} (bound {float((bound / lnorm).max()):.1e})")
    assert (diff <= bound).all(), (diff / bound).max()
    assert (diff / lnorm).max() <= 1e-13
