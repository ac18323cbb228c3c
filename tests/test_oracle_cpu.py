"""CPU tests that pin the oracle: the reference's own main() (compiled verbatim against a stand-in for Eigen/Boost),
analytic known-answer tests (SURVEY section 4, T1-T13), numpy/LAPACK and 40-digit mpmath restatements."""
import ctypes
import json
from pathlib import Path

import numpy as np
import pytest

from conftest import DEFAULT_QE, rel_err

GOLDEN = Path(__file__).resolve().parent / "golden"


def _A_of_K(k):
    k0, k1, k2 = k
    return np.array([[0, -k0, -k1, -k2], [k0, 0, k2, -k1], [k1, -k2, 0, k0], [k2, k1, -k0, 0]], dtype=float)


def _numpy_stage12(o, K, q0=(1.0, 0, 0, 0), r0=(0.0, 0, 0)):
    """Independent numpy/LAPACK restatement of SURVEY Appendix A.2-A.3 (solve, not inverse)."""
    N, M = o.N, o.M
    Dn = o.dn()
    DNN, DIN = Dn[:M, :M], Dn[:M, M]
    A = np.kron(np.eye(4), DNN)
    for i in range(M):
        Ak = _A_of_K(K[:, i])
        for r in range(4):
            for c in range(4):
                A[r * M + i, c * M + i] = (DNN[i, i] if r == c else 0.0) - 0.5 * Ak[r, c]
    rhs = -np.kron(np.asarray(q0, dtype=float), DIN)
    Q = np.linalg.solve(A, rhs)
    w, x, y, z = Q[:M], Q[M:2 * M], Q[2 * M:3 * M], Q[3 * M:]
    b = np.stack([1 - 2 * (y * y + z * z), 2 * (x * y + w * z), 2 * (x * z - w * y)], axis=1)
    r = np.linalg.solve(DNN, b - np.outer(DIN, r0))
    return Q, r


# ---- pin 1: the reference's own main() -----------------------------------------------------------------------

def test_oracle_reproduces_reference_main_golden(oracle16):
    g = json.loads((GOLDEN / "reference_main_default.json").read_text())
    Qref = np.array([float(v) for v in g["Q_stack"]])
    rref = np.array([[float(v) for v in row] for row in g["r_stack_rows"]])  # (15, 3), row i = node i
    K = oracle16.strain_from_modes(DEFAULT_QE)
    out = oracle16.integrate_all(K, want=("Q", "r"))
    assert np.abs(out["Q"].reshape(-1) - Qref).max() <= 2e-15
    assert np.abs(out["r"][0].T - rref).max() <= 2e-15


def test_reference_stdout_first_lines():
    """What a user of the reference sees (6 significant digits, SURVEY Appendix B)."""
    g = json.loads((GOLDEN / "reference_main_default.json").read_text())
    lines = g["stdout_native_precision"].split("\n")
    assert lines[0] == "Q_stack : "
    assert [s.strip() for s in lines[1:5]] == ["0.79977", "0.800067", "0.801102", "0.803372"]
    r0 = lines[lines.index("r_stack : ") + 1].split()
    assert r0 == ["0.562673", "0", "-0.745914"]


# ---- pin 1b: the reference's own integrateQuaternions()/integratePosition()/updateA on 512 random benchmark rods -----

def test_oracle_matches_reference_functions_on_random_rods(oracle16):
    """tests/golden/reference_random_rods.npz holds what the reference main.cpp's OWN functions return (compiled through
    oracle/reference_harness.cpp, global qe set per rod) for rods 0..511 of the benchmark's Philox stream.  The oracle must
    reproduce them: bound 5e-14 relative per rod (measured: bit-identical for the explicit-inverse form the reference uses,
    4e-15 for the LU-solve variant)."""
    g = np.load(GOLDEN / "reference_random_rods.npz")
    n = g["qe"].shape[0]
    assert n == 512 and int(g["seed"]) == 0x5EED
    assert np.array_equal(oracle16.generate_modes(0x5EED, 0, n), g["qe"])  # the fixture is the benchmark's own stream
    Kgen = oracle16.generate_rods(0x5EED, 0, n)[0]
    assert np.abs(Kgen - g["K"]).max() <= 1e-15  # reference's Phi*qe against the generator's fma(beta, 2x-1, alpha)
    assert np.abs(oracle16.strain_from_modes(g["qe"]) - g["K"]).max() <= 1e-15
    out = oracle16.integrate_all(g["K"], want=("Q", "r"))
    assert rel_err(out["Q"], g["Q"]) <= 5e-14 and rel_err(out["r"], g["r"]) <= 5e-14
    lu = oracle16.integrate_all(g["K"], want=("Q", "r"), explicit_inverse=False)
    assert rel_err(lu["Q"], g["Q"]) <= 5e-14 and rel_err(lu["r"], g["r"]) <= 5e-14
    for b in range(g["A_NN"].shape[0]):  # updateA main.cpp:55-88
        assert np.array_equal(oracle16.assemble_A(g["K"][b]), g["A_NN"][b])


def test_oracle_stages34_golden(oracle16):
    g = json.loads((GOLDEN / "oracle_default_stages34.json").read_text())
    K = np.array([[float(v) for v in row] for row in g["K"]])[None]
    out = oracle16.integrate_all(K, np.array([[0.0, 0.0, -1.0]]), np.zeros((1, 3)))
    assert np.abs(out["n"][0] - np.array([[float(v) for v in r] for r in g["n"]])).max() <= 1e-15
    assert np.abs(out["m"][0] - np.array([[float(v) for v in r] for r in g["m"]])).max() <= 1e-15
    # SURVEY Appendix B spot values
    assert abs(out["m"][0][1, 14] - 0.562672557482171) < 1e-13
    assert abs(out["m"][0][1, 0] - 0.00305642152055519) < 1e-13


# ---- operator known answers (T1-T3, T11) -----------------------------------------------------------------------

def test_T1_tiny_differentiation_matrices(make_oracle):
    assert np.allclose(make_oracle(2).dn(), [[1, -1], [1, -1]], atol=1e-15)
    assert np.allclose(make_oracle(3).dn(), [[3, -4, 1], [1, 0, -1], [-1, 4, -3]], atol=1e-14)


@pytest.mark.parametrize("N,tol", [(16, 1e-14), (32, 1e-13), (64, 1e-12)])
def test_T2_corner_entries(make_oracle, N, tol):
    Dn = make_oracle(N).dn()
    corner = 2 * (2 * (N - 1) ** 2 + 1) / 6
    assert abs(Dn[0, 0] / corner - 1) < tol and abs(-Dn[-1, -1] / corner - 1) < tol


@pytest.mark.parametrize("N,tol", [(16, 1e-12), (32, 1e-11), (64, 1e-10)])
def test_T3_polynomial_exactness(make_oracle, N, tol):
    o = make_oracle(N)
    Dn, x = o.dn(), o.chebyshev_points()
    assert x[0] == 1.0 and abs(x[-1]) < 1e-16 and np.all(np.diff(x) < 0)
    assert np.abs(Dn @ np.ones(N)).max() < tol
    assert np.abs(Dn @ x - 1).max() < tol
    assert np.abs(Dn @ x ** 3 - 3 * x ** 2).max() < tol


def test_T11_centro_antisymmetry_and_operator_slices(oracle16):
    Dn = oracle16.dn()
    assert np.abs(Dn + Dn[::-1, ::-1]).max() < 1e-12
    assert np.array_equal(oracle16.operator(1), Dn[:15, :15]) and np.array_equal(oracle16.operator(2), Dn[:15, 15])
    assert np.array_equal(oracle16.operator(4), Dn[1:, 1:]) and np.array_equal(oracle16.operator(5), Dn[1:, 0])
    assert np.abs(oracle16.operator(3) @ Dn[:15, :15] - np.eye(15)).max() < 1e-12
    assert np.abs(oracle16.operator(6) @ Dn[1:, 1:] - np.eye(15)).max() < 1e-12


def test_coefficients_and_phi(oracle16):
    c = oracle16.coefficients_c()
    assert c[0] == 2 and c[-1] == -2 and list(c[1:4]) == [-1, 1, -1]
    from numpy.polynomial import legendre as L
    for X in (0.0, 0.3, 1.0):
        P = oracle16.phi(3, 3, X)
        assert P.shape == (3, 9)
        row = [L.legval(2 * X - 1, [0] * k + [1]) for k in range(3)]
        assert np.allclose(P, np.kron(np.eye(3), row), atol=1e-15)
    assert abs(oracle16.legendre_p(5, 0.37) - L.legval(0.37, [0, 0, 0, 0, 0, 1])) < 1e-15


def test_assembly_matches_index_map(oracle16):
    """main.cpp:72-82: only the 16*M node-diagonal entries differ from I4 (x) Dn_NN."""
    rng = np.random.default_rng(0)
    K = rng.normal(size=(3, 16))
    A = oracle16.assemble_A(K)
    M = 15
    DNN = oracle16.operator(1)
    ref = np.kron(np.eye(4), DNN)
    for i in range(M):
        Ak = _A_of_K(K[:, i])
        for r in range(4):
            for c in range(4):
                ref[r * M + i, c * M + i] = (DNN[i, i] if r == c else 0.0) - 0.5 * Ak[r, c]
    assert np.array_equal(A, ref)


# ---- stage known answers (T4-T8) ---------------------------------------------------------------------------------

@pytest.mark.parametrize("N", [16, 32, 64])
def test_T4_straight_rod(make_oracle, N):
    o = make_oracle(N)
    out = o.integrate_all(np.zeros((1, 3, N)), want=("Q", "r"))
    x = o.chebyshev_points()[:-1]
    assert np.abs(out["Q"][0] - np.array([[1.0], [0], [0], [0]])).max() < 1e-13
    assert np.abs(out["r"][0] - np.stack([x, 0 * x, 0 * x])).max() < 1e-13


@pytest.mark.parametrize("N", [16, 32, 64])
def test_T5_circular_arc(make_oracle, N):
    o = make_oracle(N)
    k = 1.2877691307032
    K = np.zeros((1, 3, N)); K[0, 1] = k
    out = o.integrate_all(K, want=("Q", "r"))
    X = o.chebyshev_points()[:-1]
    Q = np.stack([np.cos(k * X / 2), 0 * X, np.sin(k * X / 2), 0 * X])
    r = np.stack([np.sin(k * X) / k, 0 * X, -(1 - np.cos(k * X)) / k])
    assert np.abs(out["Q"][0] - Q).max() < 2e-13 and np.abs(out["r"][0] - r).max() < 2e-13


def test_T6_default_configuration_analytic(oracle16):
    a, b, c = DEFAULT_QE[3:6]
    X = oracle16.chebyshev_points()[:-1]
    theta = a * X + b * (X ** 2 - X) + c * (2 * X ** 3 - 3 * X ** 2 + X)
    out = oracle16.integrate_all(oracle16.strain_from_modes(DEFAULT_QE), want=("Q",))
    Q = np.stack([np.cos(theta / 2), 0 * X, np.sin(theta / 2), 0 * X])
    assert np.abs(out["Q"][0] - Q).max() < 1e-10  # spectral discretisation error at N=16 (SURVEY T6: 4.3e-12)


def test_T8_quaternion_norm_is_discretisation_error(oracle16, make_oracle):
    K, F, Mt, fb = oracle16.generate_rods(0x5EED, 0, 200)
    Q = oracle16.integrate_all(K, want=("Q",))["Q"]
    assert np.abs((Q ** 2).sum(axis=1) - 1).max() < 1e-8
    o32 = make_oracle(32)
    K32 = o32.generate_rods(0x5EED, 0, 20)[0]
    Q32 = o32.integrate_all(K32, want=("Q",))["Q"]
    assert np.abs((Q32 ** 2).sum(axis=1) - 1).max() < 1e-13


# ---- stages 3-4 known answers (T9, T13) ----------------------------------------------------------------------------

def test_T9_stress_polynomial_exactness(oracle16):
    """n' = -fbar with polynomial fbar of degree < N-1 is integrated exactly: n(X) = F_tip + int_X^1 fbar."""
    x = oracle16.chebyshev_points()
    fbar = np.stack([1 + 0 * x, x, 3 * x ** 2])[None]
    F = np.array([[0.3, -0.2, 0.5]])
    n = oracle16.integrate_all(np.zeros((1, 3, 16)), F, np.zeros((1, 3)), fbar=fbar, want=("n",))["n"][0]
    X = x[1:]
    exact = np.stack([F[0, 0] + (1 - X), F[0, 1] + (1 - X ** 2) / 2, F[0, 2] + (1 - X ** 3)])
    assert np.abs(n - exact).max() < 1e-13


@pytest.mark.parametrize("N,tol", [(16, 1e-9), (32, 1e-13)])
def test_T13_dead_load_couple(make_oracle, N, tol):
    """fbar = lbar = 0  =>  n == F_tip and m(X) = M_tip + (r_tip - r(X)) x F_tip."""
    o = make_oracle(N)
    K = o.strain_from_modes(DEFAULT_QE)
    F = np.array([[0.0, 0.0, -1.0]]); Mt = np.array([[0.1, -0.2, 0.05]])
    out = o.integrate_all(K, F, Mt)
    assert np.abs(out["n"][0] - F[0][:, None]).max() < 1e-13
    r_nodes = np.concatenate([out["r"][0], np.zeros((3, 1))], axis=1)  # nodes 0..N-1 (base r = 0)
    m_exact = Mt[0][:, None] + np.cross((r_nodes[:, :1] - r_nodes[:, 1:]).T, F[0]).T
    assert np.abs(out["m"][0] - m_exact).max() < tol


@pytest.mark.parametrize("N,tol", [(16, 1e-7), (32, 1e-12), (48, 1e-12)])  # observed: 1e-8, 1e-13, 1e-13
def test_T10_global_vs_local_frame_statics(make_oracle, N, tol):
    """SURVEY T10: the global-frame stages 3-4 (rod_modeling.pdf 1.17-1.18), rotated into the body frame, must solve the
    local-frame statics Lambda' = ad^T_xi Lambda - Fbar (eq. 1.29 / 2.18), i.e. N' = -K^ N - R^T fbar and
    C' = -K^ C - Gamma^ N - R^T lbar.  The local ODE is collocated here independently (numpy, strain-dependent 3M x 3M
    operator with the tip node eliminated); agreement is to discretisation error, which pins the sign conventions of
    stages 3-4 and of the wrench_local output."""
    o = make_oracle(N)
    M = N - 1
    rng = np.random.default_rng(N)
    K, F, Mt, fb = o.generate_rods(0x5EED, 3, 3)
    x = o.chebyshev_points()
    fbar = fb + 0.3 * rng.normal(size=(3, 3, 1)) * np.sin(2 * x)[None, None, :] + 0.2 * rng.normal(size=(3, 3, 1)) * x[None, None, :]
    lbar = 0.2 * rng.normal(size=(3, 3, 1)) * np.cos(x)[None, None, :]
    q0 = rng.normal(size=(3, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    out = o.integrate_all(K, F, Mt, q0=q0, fbar=fbar, lbar=lbar)
    lam = o.wrench_local(out["Q"], out["n"], out["m"], F, Mt, q0=q0)     # [B][6][N], couple first
    Dn = o.operator(0)
    D_TT, D_TI = Dn[1:, 1:], Dn[1:, 0]

    def rot(q):
        w, x, y, z = q
        return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                         [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                         [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])

    def skew(v):
        return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])

    for b in range(3):
        R = [rot(out["Q"][b][:, i]) if i < M else rot(q0[b]) for i in range(N)]
        A = np.kron(D_TT, np.eye(3))
        for i in range(1, N):
            A[3 * (i - 1):3 * i, 3 * (i - 1):3 * i] += skew(K[b][:, i])
        # internal force
        N0 = R[0].T @ F[b]
        rhs = np.concatenate([-R[i].T @ fbar[b][:, i] for i in range(1, N)]) - np.kron(D_TI, N0)
        Nloc = np.linalg.solve(A, rhs).reshape(M, 3)
        # internal couple (Gamma = e1)
        C0 = R[0].T @ Mt[b]
        G = skew(np.array([1.0, 0.0, 0.0]))
        rhs = np.concatenate([-G @ Nloc[i - 1] - R[i].T @ lbar[b][:, i] for i in range(1, N)]) - np.kron(D_TI, C0)
        Cloc = np.linalg.solve(A, rhs).reshape(M, 3)
        scale = max(np.abs(Nloc).max(), np.abs(Cloc).max())
        assert np.abs(lam[b][3:, 1:].T - Nloc).max() <= tol * scale, (N, "N")
        assert np.abs(lam[b][:3, 1:].T - Cloc).max() <= tol * scale, (N, "C")
        assert np.abs(lam[b][3:, 0] - N0).max() <= 1e-15 and np.abs(lam[b][:3, 0] - C0).max() <= 1e-15


@pytest.mark.parametrize("N,tol", [(16, 1e-7), (32, 1e-12)])
def test_wrench_local_solve_vs_pointwise_and_numpy(make_oracle, N, tol):
    """The oracle's direct local-frame solve (one LU of the strain-dependent operator, two solves) against (a) the
    pointwise form [R^T m; R^T n] of the global-frame stages -- equal to discretisation error -- and (b) numpy/LAPACK on
    the same collocation system -- equal to rounding."""
    o = make_oracle(N)
    M = N - 1
    rng = np.random.default_rng(7 * N)
    x = o.chebyshev_points()
    K, F, Mt, fb = o.generate_rods(0x5EED, 11, 3)
    fbar = fb + 0.3 * rng.normal(size=(3, 3, 1)) * np.sin(2 * x)[None, None, :]
    lbar = 0.2 * rng.normal(size=(3, 3, 1)) * np.cos(x)[None, None, :]
    Gamma = np.stack([1 + 0.05 * np.sin(x), 0.03 * x, 0.02 * np.cos(x)])[None].repeat(3, axis=0)
    q0 = rng.normal(size=(3, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    out = o.integrate_all(K, F, Mt, q0=q0, Gamma=Gamma, fbar=fbar, lbar=lbar)
    lam_pw = o.wrench_local(out["Q"], out["n"], out["m"], F, Mt, q0=q0)
    lam = o.wrench_local_solve(K, out["Q"], F, Mt, q0=q0, Gamma=Gamma, fbar=fbar, lbar=lbar)
    scale = np.abs(lam_pw).max()
    assert np.abs(lam - lam_pw).max() <= tol * scale
    # numpy on the same system
    Dn = o.operator(0); D_TT, D_TI = Dn[1:, 1:], Dn[1:, 0]
    skew = lambda v: np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])

    def rot(q):
        w, a, b, c = q
        return np.array([[1 - 2 * (b * b + c * c), 2 * (a * b - w * c), 2 * (a * c + w * b)],
                         [2 * (a * b + w * c), 1 - 2 * (a * a + c * c), 2 * (b * c - w * a)],
                         [2 * (a * c - w * b), 2 * (b * c + w * a), 1 - 2 * (a * a + b * b)]])

    for b in range(3):
        R = [rot(out["Q"][b][:, i]) if i < M else rot(q0[b]) for i in range(N)]
        A = np.kron(D_TT, np.eye(3))
        for i in range(1, N):
            A[3 * (i - 1):3 * i, 3 * (i - 1):3 * i] += skew(K[b][:, i])
        N0, C0 = R[0].T @ F[b], R[0].T @ Mt[b]
        Nl = np.linalg.solve(A, np.concatenate([-R[i].T @ fbar[b][:, i] for i in range(1, N)]) - np.kron(D_TI, N0)).reshape(M, 3)
        rhs = np.concatenate([-np.cross(Gamma[b][:, i], Nl[i - 1]) - R[i].T @ lbar[b][:, i] for i in range(1, N)]) - np.kron(D_TI, C0)
        Cl = np.linalg.solve(A, rhs).reshape(M, 3)
        assert np.abs(lam[b][3:, 1:].T - Nl).max() <= 1e-12 * scale and np.abs(lam[b][:3, 1:].T - Cl).max() <= 1e-12 * scale


# ---- independent restatements -----------------------------------------------------------------------------------

@pytest.mark.parametrize("N", [8, 16, 32])
def test_numpy_lapack_restatement(make_oracle, N):
    o = make_oracle(N)
    rng = np.random.default_rng(N)
    K, F, Mt, fb = o.generate_rods(1, 0, 6)
    q0 = rng.normal(size=(6, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    r0 = rng.normal(size=(6, 3))
    for explicit in (True, False):
        out = o.integrate_all(K, q0=q0, r0=r0, explicit_inverse=explicit, want=("Q", "r"))
        for b in range(6):
            Q, r = _numpy_stage12(o, K[b], q0[b], r0[b])
            assert np.abs(out["Q"][b].reshape(-1) - Q).max() < 2e-13
            assert np.abs(out["r"][b].T - r).max() < 2e-13


def test_mpmath_40_digits_default_configuration(oracle16):
    mp = pytest.importorskip("mpmath")
    mp.mp.dps = 40
    N, M = 16, 15
    x = [mp.mpf(1) / 2 * (1 + mp.cos(mp.pi * j / (N - 1))) for j in range(N)]
    c = [(-1) ** j * (2 if j in (0, N - 1) else 1) for j in range(N)]
    D = mp.matrix(N, N)
    for i in range(N):
        for j in range(N):
            if i != j:
                D[i, j] = mp.mpf(c[i]) / c[j] / (x[i] - x[j])
    for i in range(N):
        D[i, i] = -sum(D[i, j] for j in range(N) if j != i)
    qe = [mp.mpf(repr(float(v))) for v in DEFAULT_QE]
    Ky = [qe[3] + qe[4] * (2 * x[i] - 1) + qe[5] * (3 * (2 * x[i] - 1) ** 2 - 1) / 2 for i in range(N)]
    A = mp.matrix(4 * M, 4 * M)
    for blk in range(4):
        for i in range(M):
            for j in range(M):
                A[blk * M + i, blk * M + j] = D[i, j]
    for i in range(M):
        Ak = [[0, 0, -Ky[i], 0], [0, 0, 0, -Ky[i]], [Ky[i], 0, 0, 0], [0, Ky[i], 0, 0]]
        for r in range(4):
            for cc in range(4):
                A[r * M + i, cc * M + i] -= mp.mpf(Ak[r][cc]) / 2
    rhs = mp.matrix(4 * M, 1)
    for i in range(M):
        rhs[i] = -D[i, M]
    Q = mp.lu_solve(A, rhs)
    out = oracle16.integrate_all(oracle16.strain_from_modes(DEFAULT_QE), want=("Q",))["Q"].reshape(-1)
    err = max(abs(float(Q[i]) - out[i]) for i in range(4 * M))
    assert err < 5e-14  # FP64 Dn differs from the 40-digit Dn by rounding; cond(A_NN) ~ 190


def test_explicit_inverse_and_lu_solve_variants_agree(oracle16):
    K, F, Mt, fb = oracle16.generate_rods(3, 0, 64)
    a = oracle16.integrate_all(K, F, Mt, fbar=fb, explicit_inverse=True)
    b = oracle16.integrate_all(K, F, Mt, fbar=fb, explicit_inverse=False)
    for s in "Qrnm":
        assert rel_err(a[s], b[s]) < 1e-13


def test_oracle_threads_give_identical_results(oracle16):
    K, F, Mt, fb = oracle16.generate_rods(3, 0, 257)
    a = oracle16.integrate_all(K, F, Mt, fbar=fb, nthreads=1)
    b = oracle16.integrate_all(K, F, Mt, fbar=fb, nthreads=0)
    for s in "Qrnm":
        assert np.array_equal(a[s], b[s])


# ---- synthetic input generator -----------------------------------------------------------------------------------

def test_philox4x32_10_known_answers(oracle16):
    """Random123 known-answer vectors for Philox4x32-10."""
    f = oracle16.lib.sri_oracle_philox4x32_10
    U4, U2 = ctypes.c_uint32 * 4, ctypes.c_uint32 * 2
    for ctr, key, want in (
        ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
        ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
        ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
    ):
        out = U4()
        f(U4(*ctr), U2(*key), out)
        assert tuple(out) == want


def test_generator_is_sharding_invariant_and_in_range(oracle16):
    K, F, Mt, fb = oracle16.generate_rods(0x5EED, 0, 1000)
    K2, F2, M2, fb2 = oracle16.generate_rods(0x5EED, 400, 300)
    assert np.array_equal(K[400:700], K2) and np.array_equal(F[400:700], F2)
    assert np.array_equal(Mt[400:700], M2) and np.array_equal(fb[400:700], fb2)
    assert np.abs(K).max() <= 4.0 and np.abs(F).max() <= 1.0 and np.abs(Mt).max() <= 1.0
    assert (fb[:, 2] <= 0).all() and (fb[:, 2] >= -1).all() and not fb[:, :2].any()
    t = 2 * oracle16.chebyshev_points() - 1                       # K_c is constant + linear in X
    assert np.abs(K[:, :, 0] + K[:, :, -1] - 2 * K[:, :, 5] + (K[:, :, 0] - K[:, :, -1]) * t[5]).max() < 1e-14


def test_analytic_jacobian_of_the_discrete_static_shape_residual(oracle16):
    """oracle/tangent.py: the exact tangent of the discrete four-stage map (stage-1 operator shared by all directions) gives
    the Newton Jacobian of the Galerkin residual; pinned here against central differences of the oracle's own residual
    (with and without a reference curvature K0).  Groundwork for the multi-right-hand-side elimination of DESIGN section 7."""
    from numpy.polynomial import legendre as L
    from oracle.tangent import cc_weights, galerkin_residual_and_jacobian
    o = oracle16
    B, ne = 3, 3
    n = 3 * ne
    rng = np.random.default_rng(0)
    qe = 0.8 * rng.normal(size=(B, n))
    F = rng.uniform(-1, 1, size=(B, 3)); Mt = rng.uniform(-0.5, 0.5, size=(B, 3))
    K0 = 0.2 * rng.normal(size=(B, 3, 16))
    H = np.array([1.0, 0.9, 0.77])
    x = o.chebyshev_points(); w = cc_weights(16)
    P = np.stack([L.legval(2 * x - 1, [0] * k + [1]) for k in range(ne)])

    for k0 in (None, K0):
        def g_of(q):
            K = o.strain_from_modes(q, ne)
            out = o.integrate_all(K, F, Mt, explicit_inverse=False, want=("Q", "m", "n"))
            rho = o.shape_residual(K, H, out["Q"], out["m"], Mt, K0=k0)
            return np.einsum("bci,ki,i->bck", rho, P, w).reshape(B, n)

        g, J = galerkin_residual_and_jacobian(o, qe, F, Mt, H, ne, K0=k0)
        assert np.abs(g - g_of(qe)).max() <= 1e-14
        Jfd = np.empty_like(J)
        h = 1e-6
        for d in range(n):
            e = np.zeros(n); e[d] = h
            Jfd[:, :, d] = (g_of(qe + e) - g_of(qe - e)) / (2 * h)
        assert np.abs(J - Jfd).max() <= 1e-8 * np.abs(Jfd).max()


@pytest.mark.parametrize("N,tol", [(16, 1e-9), (32, 1e-13)])
def test_jacobian_by_quadrature_agrees_with_the_exact_tangent(make_oracle, N, tol):
    """The solve-free Jacobian of sri_shape_jacobian (left-trivialised rotation variation: two contractions per direction)
    against the exact tangent of the discrete map: equal to the discretisation error."""
    from oracle.tangent import galerkin_residual_and_jacobian, jacobian_by_quadrature
    o = make_oracle(N)
    B, ne = 3, 3
    rng = np.random.default_rng(1)
    qe = 0.8 * rng.normal(size=(B, 3 * ne))
    F = rng.uniform(-1, 1, size=(B, 3)); Mt = rng.uniform(-0.5, 0.5, size=(B, 3))
    H = np.array([1.0, 0.9, 0.77])
    _, J_exact = galerkin_residual_and_jacobian(o, qe, F, Mt, H, ne)
    J = jacobian_by_quadrature(o, qe, F, Mt, H, ne)
    assert np.abs(J - J_exact).max() <= tol * np.abs(J_exact).max()


# ---- rod length (SURVEY 8 f3; rod_modeling.pdf eq. 2.17) ---------------------------------------------------------------

@pytest.mark.parametrize("N,ell", [(16, 0.4), (24, 3.0)])
def test_rod_length_is_an_input_scaling(make_oracle, N, ell):
    """Integrating a rod of length ell on the physical interval [0, ell] (differentiation matrix Dn / ell, nodes
    ComputeChebyshevPoints<N, ell>) equals the unit-interval integration of (ell K, ell Gamma, ell fbar, ell lbar): the
    equivalence the package's scale_for_length() helper relies on.  Independent numpy collocation vs the oracle."""
    o = make_oracle(N)
    M = N - 1
    rng = np.random.default_rng(7)
    x = o.chebyshev_points(1.0)
    assert np.allclose(o.chebyshev_points(ell), ell * x, rtol=0, atol=1e-15 * ell)
    K = (rng.uniform(-1.5, 1.5, size=(3, 1)) + rng.uniform(-1, 1, size=(3, 1)) * (2 * x - 1))[None]
    Gam = np.array([1.0, 0.04, -0.03])[None, :, None] * np.ones((1, 3, N))
    fb = rng.normal(size=(1, 3, 1)) * np.ones((1, 1, N)); lb = 0.2 * rng.normal(size=(1, 3, 1)) * np.ones((1, 1, N))
    F = rng.uniform(-1, 1, size=(1, 3)); Mt = rng.uniform(-1, 1, size=(1, 3))
    out = o.integrate_all(ell * K, F, Mt, Gamma=ell * Gam, fbar=ell * fb, lbar=ell * lb, explicit_inverse=False)
    D = o.dn() / ell
    A = np.kron(np.eye(4), D[:M, :M])
    for i in range(M):
        Ak = _A_of_K(K[0, :, i])
        for r in range(4):
            for c in range(4):
                A[r * M + i, c * M + i] -= 0.5 * Ak[r, c]
    Q = np.linalg.solve(A, -np.kron(np.array([1.0, 0, 0, 0]), D[:M, M]))
    assert np.abs(Q - out["Q"][0].reshape(-1)).max() <= 1e-12
    w, xq, y, z = np.concatenate([Q.reshape(4, M), np.array([[1.0], [0], [0], [0]])], axis=1)
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (xq * y - w * z), 2 * (xq * z + w * y)],
                  [2 * (xq * y + w * z), 1 - 2 * (xq * xq + z * z), 2 * (y * z - w * xq)],
                  [2 * (xq * z - w * y), 2 * (y * z + w * xq), 1 - 2 * (xq * xq + y * y)]])
    rp = np.einsum("ijn,jn->in", R, Gam[0])
    r = np.linalg.solve(D[:M, :M], rp[:, :M].T)
    n = np.linalg.solve(D[1:, 1:], -fb[0][:, 1:].T - np.outer(D[1:, 0], F[0]))
    m = np.linalg.solve(D[1:, 1:], -(np.cross(rp[:, 1:].T, n) + lb[0][:, 1:].T) - np.outer(D[1:, 0], Mt[0]))
    assert np.abs(r.T - out["r"][0]).max() <= 1e-12
    assert np.abs(n.T - out["n"][0]).max() <= 1e-12 * max(1.0, np.abs(n).max())
    assert np.abs(m.T - out["m"][0]).max() <= 1e-11 * max(1.0, np.abs(m).max())
