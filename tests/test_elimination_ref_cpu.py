"""The extended-precision reference of tests/elimination_ref.py, pinned on the CPU before the GPU tests rely on it.

For every node count 2..64, on generator rods with every optional input: the refined solution of the preconditioned system
and the long-double stages 2-4 agree with the float64 oracle; the refinement has converged; LAPACK's plain float64 solve
has the backward error a backward-stable solver must have; and the backward error does see a perturbation of 1e-13.
"""
import numpy as np
import pytest

from elimination_ref import (U, Tables, backward_error, q_to_x, refine_step, refined_solve, stage_bound, stage_excess,
                             stage_m, stage_n, stage_r, system, x_to_q)

B = 16


def _inputs(o, N, seed):
    rng = np.random.default_rng(seed)
    K, F, Mt, fb = o.generate_rods(0x5EED, 1000 * N, B)
    q0 = rng.normal(size=(B, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    r0 = rng.normal(size=(B, 3))
    Gamma = np.concatenate([1 + 0.1 * rng.normal(size=(B, 1, N)), 0.1 * rng.normal(size=(B, 2, N))], axis=1)
    lbar = rng.normal(size=(B, 3, N))
    return dict(K=K, F_tip=F, M_tip=Mt, q0=q0, r0=r0, Gamma=Gamma, fbar=fb, lbar=lbar)


def _rod_rel(x, ref):
    x = np.asarray(x, dtype=np.float64).reshape(x.shape[0], -1)
    ref = np.asarray(ref, dtype=np.float64).reshape(ref.shape[0], -1)
    return np.abs(x - ref).max(axis=1) / np.abs(ref).max(axis=1)


@pytest.mark.parametrize("N", range(2, 65))
def test_reference_against_oracle(make_oracle, N):
    o = make_oracle(N)
    tab = Tables.from_oracle(o)
    M = N - 1
    a = _inputs(o, N, N)
    ref = o.integrate_all(a["K"], a["F_tip"], a["M_tip"], q0=a["q0"], r0=a["r0"], Gamma=a["Gamma"], fbar=a["fbar"],
                          lbar=a["lbar"], explicit_inverse=False)
    assert ref["bad"] == 0
    C, b = system(tab, a["K"], a["q0"])
    x = refined_solve(C, b)
    Q = x_to_q(x, M)
    assert _rod_rel(Q, ref["Q"]).max() <= 5e-14
    r, _ = stage_r(tab, Q, a["Gamma"], a["r0"])
    n, _ = stage_n(tab, B, a["F_tip"], a["fbar"])
    m, _ = stage_m(tab, Q, n, a["q0"], a["Gamma"], a["lbar"], a["M_tip"])
    for name, val in (("r", r), ("n", n), ("m", m)):
        assert _rod_rel(val, ref[name]).max() <= 5e-14, name

    # converged: one more step moves x by less than 1e-17 relative
    _, rel = refine_step(C, x, b)
    assert rel.max() < 1e-17

    # a backward-stable float64 solve (LAPACK, partial pivoting) has eta of a few u; 8u bounds it at every N
    x64 = np.linalg.solve(C, b[..., None])[..., 0]
    eta = backward_error(C, x64, b)
    assert eta.max() <= 8 * U, eta.max() / U
    # ...and eta is not blind: one entry of the exact solution off by 1e-13 relative is seen far above 8u
    xp = x.astype(np.float64).copy()
    k = np.abs(xp).argmax(axis=1)
    xp[np.arange(B), k] *= 1 + 1e-13
    assert backward_error(C, xp, b).min() >= 10 * 8 * U

    # the stage bounds admit a plain float64 evaluation: the oracle's own r, n, m from its own Q and n
    for name, (val, mag) in (("r", stage_r(tab, ref["Q"], a["Gamma"], a["r0"])), ("n", stage_n(tab, B, a["F_tip"], a["fbar"])),
                             ("m", stage_m(tab, ref["Q"], ref["n"], a["q0"], a["Gamma"], a["lbar"], a["M_tip"]))):
        assert stage_excess(ref[name], val, stage_bound(tab, mag)).max() <= 1.0, name


def test_system_is_the_oracle_operator():
    """C is the preconditioned A_NN: S A_NN (row/column permuted to node-major order) equals C up to the rounding of S."""
    from oracle import Oracle, build_oracle
    build_oracle()
    N, M = 9, 8
    o = Oracle(N)
    tab = Tables.from_oracle(o)
    K, _, _, _ = o.generate_rods(3, 0, 2)
    C, b = system(tab, K)
    perm = np.array([c * M + j for j in range(M) for c in range(4)])  # node-major index -> the oracle's block order
    for r in range(2):
        A = o.assemble_A(K[r])[np.ix_(perm, perm)]
        SA = np.kron(tab.S, np.eye(4)) @ A
        assert np.abs(SA - C[r]).max() <= 1e-13
        rhs = -np.kron(tab.Dn_IN, [1.0, 0.0, 0.0, 0.0])
        assert np.abs(np.kron(tab.S, np.eye(4)) @ rhs - b[r]).max() <= 1e-13
    Q = np.random.default_rng(0).normal(size=(2, 4, M))
    assert np.array_equal(x_to_q(q_to_x(Q), M), Q) and q_to_x(Q)[0, 4 * 3 + 2] == Q[0, 2, 3]
