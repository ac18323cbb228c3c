"""GPU tests of the static shape problem under distributed loads, a rotated clamp and a given Gamma: sri_shape_jacobian at a
loaded state, sri_newton_static_problem and sri_static_problem_vjp against the numpy restatement (static_loads_ref.py) and
known answers, the unchanged tip-load entry points, the sharded solve, and autograd.static_shape with the new inputs."""
import ctypes

import numpy as np
import pytest

from conftest import rel_err
from static_loads_ref import INPUTS, loaded_problem, unit_quaternion

pytestmark = pytest.mark.gpu

H0 = np.array([1.0, 1.0, 0.77])
OPTIONAL = ("K0",) + INPUTS
ALL_GRADS = ("F_tip", "M_tip", "K0", "H") + INPUTS + ("lambda", "resid")


@pytest.fixture(scope="module")
def integ():
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import SpectralRodIntegrator
    cache = {}

    def get(N):
        if N not in cache:
            cache[N] = SpectralRodIntegrator(N, 0)
        return cache[N]

    yield get
    for h in cache.values():
        h.close()


def _cuda(a):
    import torch
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def _launches():
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import kernel_launch_count
    return kernel_launch_count()


def _on(conv, t, keys=OPTIONAL):
    return {k: conv(t[k]) for k in keys if t.get(k) is not None}


def _solve(h, t, ne, conv=_cuda, fd_step=0.0, tol=1e-13, max_iter=40, **kw):
    """newton_static_shape with every optional input of t; returns (qe as numpy, report)."""
    qe, rep = h.newton_static_shape(conv(t["F_tip"]), conv(t["M_tip"]), ne, H_diag=H0, tol=tol, max_iter=max_iter,
                                    fd_step=fd_step, **_on(conv, t), **kw)
    return _np(qe), rep


def _newton_problem_null(h, F, Mt, ne, K0, qe, fd_step, tol, max_iter, callback):
    """sri_newton_static_problem with q0, Gamma, fbar, lbar NULL, called directly."""
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import _lib
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200.api import _problem, _ptr, _report_dict
    H = np.ascontiguousarray(H0)
    prob = _problem(F.shape[0], ne, H, F, Mt, K0, None, None, None, None)
    rep = _lib.NewtonReport()
    cb = _lib.ALLREDUCE_FN(lambda p, c: 0) if callback else _lib.ALLREDUCE_FN()
    h._follow_torch(F)
    _lib.check(h._lib.sri_newton_static_problem(h._h, ctypes.byref(prob), _ptr(qe, "qe"), tol, max_iter, fd_step, 0, cb, None,
                                                ctypes.byref(rep)), "sri_newton_static_problem")
    return qe, _report_dict(rep)


def _vjp_problem_null(h, F, Mt, K0, qe, gqe, steps, out, info):
    """sri_static_problem_vjp with q0, Gamma, fbar, lbar NULL and the tip-load outputs, called directly."""
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import _lib
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200.api import _problem, _ptr
    H = np.ascontiguousarray(H0)
    prob = _problem(F.shape[0], qe.shape[1] // 3, H, F, Mt, K0, None, None, None, None)
    g = lambda k: _ptr(out.get(k), k)
    grads = _lib.StaticProblemGrad(gF_tip=g("F_tip"), gM_tip=g("M_tip"), gK0=g("K0"), gH=g("H"), lambda_=g("lambda"),
                                   resid=g("resid"), info=_ptr(info, "info", np.int32))
    h._follow_torch(qe)
    _lib.check(h._lib.sri_static_problem_vjp(h._h, ctypes.byref(prob), _ptr(qe, "qe"), _ptr(gqe, "gqe"), steps,
                                             ctypes.byref(grads)), "sri_static_problem_vjp")
    return out


def _quat_mul(a, b):
    """Hamilton product (w, x, y, z), row-wise: R(a * b) = R(a) R(b)."""
    w1, v1, w2, v2 = a[..., :1], a[..., 1:], b[..., :1], b[..., 1:]
    return np.concatenate([w1 * w2 - np.sum(v1 * v2, -1, keepdims=True), w1 * v2 + w2 * v1 + np.cross(v1, v2)], -1)


# ---- 1. the analytic Jacobian under loads -------------------------------------------------------------------------------

@pytest.mark.parametrize("N", [16, 24, 33])
def test_shape_jacobian_under_loads_matches_reference(make_oracle, integ, N):
    """N = 16: the DMMA kernel; 24, 33: the scalar kernel.  The reference is evaluated on the GPU's own stages."""
    from oracle.tangent import cc_weights, jacobian_by_quadrature_from_state
    from static_adjoint_ref import legendre_table
    rng = np.random.default_rng(3000 + N)
    B, ne = 9, 4
    t = loaded_problem(rng, B, N)
    qe = rng.uniform(-0.6, 0.6, size=(B, 3 * ne))
    h = integ(N)
    K = h.strain_from_modes(_cuda(qe))
    st = h.integrate_all(K, _cuda(t["F_tip"]), _cuda(t["M_tip"]), want=("Q", "n", "m"), **_on(_cuda, t, INPUTS))
    J = h.shape_jacobian(st["Q"], st["n"], st["m"], _cuda(t["M_tip"]), ne, H0, q0=_cuda(t["q0"]), Gamma=_cuda(t["Gamma"]))
    o = make_oracle(N)
    Dn, M = o.dn(), o.M
    want = jacobian_by_quadrature_from_state(_np(st["Q"]), _np(st["n"]), _np(st["m"]), t["M_tip"], H0, ne,
                                             legendre_table(o, ne), cc_weights(N), np.linalg.inv(Dn[:M, :M]),
                                             np.linalg.inv(Dn[1:, 1:]), q0=t["q0"], Gamma=t["Gamma"])
    assert np.ptp(_np(st["n"]), axis=2).max() > 0.5   # n varies along the rod
    assert rel_err(_np(J), want) <= 1e-12


# ---- 2. nothing changes without loads ---------------------------------------------------------------------------------

@pytest.mark.parametrize("fd_step", [0.0, 1e-6])
@pytest.mark.parametrize("host", [False, True])
@pytest.mark.parametrize("callback", [False, True])
def test_null_loads_newton_is_the_tip_load_entry_point(integ, fd_step, host, callback):
    N, ne, B = 16, 3, 301
    rng = np.random.default_rng(11)
    F, Mt = rng.uniform(-0.6, 0.6, size=(B, 3)), rng.uniform(-0.6, 0.6, size=(B, 3))
    K0 = rng.uniform(-0.3, 0.3, size=(B, 3, N))
    conv = np.ascontiguousarray if host else _cuda
    h = integ(N)
    allreduce = (lambda norms: None) if callback else None
    runs = []
    for new in (False, True, False, True):
        qe = conv(np.zeros((B, 3 * ne)))
        before = _launches()
        if new:
            q, rep = _newton_problem_null(h, conv(F), conv(Mt), ne, conv(K0), qe, fd_step, 1e-12, 30, callback)
        else:
            q, rep = h.newton_static_shape(conv(F), conv(Mt), ne, H_diag=H0, qe=qe, K0=conv(K0), tol=1e-12, max_iter=30,
                                           fd_step=fd_step, allreduce=allreduce)
        runs.append((_np(q).copy(), rep, _launches() - before))
    assert runs[0][1]["converged"]
    for q, rep, launches in runs[1:]:
        assert np.array_equal(q, runs[0][0]) and rep == runs[0][1] and launches == runs[0][2]


@pytest.mark.parametrize("host", [False, True])
def test_null_loads_vjp_is_the_tip_load_entry_point(integ, host):
    N, ne, B = 16, 4, 57
    rng = np.random.default_rng(12)
    F, Mt = rng.uniform(-0.6, 0.6, size=(B, 3)), rng.uniform(-0.6, 0.6, size=(B, 3))
    K0 = rng.uniform(-0.3, 0.3, size=(B, 3, N))
    h = integ(N)
    qe, _ = h.newton_static_shape(_cuda(F), _cuda(Mt), ne, H_diag=H0, K0=_cuda(K0), tol=1e-13, max_iter=40, fd_step=0.0)
    gqe = rng.normal(size=(B, 3 * ne))
    conv = np.ascontiguousarray if host else _cuda
    want = ("F_tip", "M_tip", "K0", "H", "lambda", "resid")
    shapes = {"F_tip": (B, 3), "M_tip": (B, 3), "K0": (B, 3, N), "H": (B, 3), "lambda": (B, 3 * ne), "resid": (B,)}
    for steps in (0, 3):
        b0 = _launches()
        info_old = conv(np.full(B, -1, dtype=np.int32))
        old = h.static_shape_vjp(conv(F), conv(Mt), conv(_np(qe)), conv(gqe), H_diag=H0, K0=conv(K0), refine_steps=steps,
                                 info=info_old, want=want)
        b1 = _launches()
        info_new = conv(np.full(B, -1, dtype=np.int32))
        new = _vjp_problem_null(h, conv(F), conv(Mt), conv(K0), conv(_np(qe)), conv(gqe), steps,
                                {k: conv(np.empty(shapes[k])) for k in want}, info_new)
        b2 = _launches()
        assert b2 - b1 == b1 - b0
        assert np.array_equal(_np(info_old), _np(info_new)) and not _np(info_new).any()
        for k in want:
            assert np.array_equal(_np(old[k]), _np(new[k])), (steps, k)


@pytest.mark.parametrize("fd_step", [0.0, 1e-6])
def test_loads_launch_the_same_kernels_per_iteration(integ, fd_step):
    """One Newton iteration under loads launches what one without loads does (lagged mode, eager and graph iterations), and
    a handle that alternates between the two keeps giving the results of a fresh one."""
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import SpectralRodIntegrator
    N, ne, B = 16, 3, 513
    rng = np.random.default_rng(13)
    t = loaded_problem(rng, B, N)
    tip = {"F_tip": t["F_tip"], "M_tip": t["M_tip"], "K0": t["K0"]}
    h = integ(N)
    counts = {}
    for name, prob in (("tip", tip), ("loaded", t)):
        for iters in (1, 3):
            before = _launches()
            _, rep = _solve(h, prob, ne, fd_step=fd_step, tol=0.0, max_iter=iters)
            assert rep["iterations"] == iters
            counts[name, iters] = _launches() - before
    assert counts["tip", 1] == counts["loaded", 1] and counts["tip", 3] == counts["loaded", 3]
    with SpectralRodIntegrator(N, 0) as fresh:
        q_fresh, rep_fresh = _solve(fresh, t, ne, fd_step=fd_step)
    for prob in (tip, t, tip, t):
        q, rep = _solve(h, prob, ne, fd_step=fd_step)
    assert np.array_equal(q, q_fresh) and rep == rep_fresh


# ---- 3. the solve against the reference ---------------------------------------------------------------------------------

@pytest.mark.parametrize("N", [5, 9, 16, 33])
@pytest.mark.parametrize("ne", [2, 4])
def test_newton_under_loads_matches_reference(make_oracle, integ, N, ne):
    from static_loads_ref import newton
    rng = np.random.default_rng(4000 + 10 * N + ne)
    B = 3
    t = loaded_problem(rng, B, N)
    h = integ(N)
    qa, rep_a = _solve(h, t, ne)
    assert rep_a["converged"] and rep_a["max_abs"] < 1e-13, rep_a
    want, gmax = newton(make_oracle(N), t["F_tip"], t["M_tip"], H0, ne, **{k: t[k] for k in OPTIONAL})
    assert gmax < 1e-13 and np.abs(want).max() > 0.3
    assert rel_err(qa, want) <= 1e-10, (N, ne)
    qf, rep_f = _solve(h, t, ne, fd_step=1e-6, tol=1e-12)
    assert rep_f["converged"] and rel_err(qf, qa) <= 1e-10
    if N == 16:   # quadratic convergence of the analytic-Jacobian solve
        hist = rep_a["rms_history"]
        pairs = [(a, b) for a, b in zip(hist, hist[1:]) if 1e-9 < a < 1e-2 and b > 1e-15]
        assert pairs and all(b <= 10.0 * a * a for a, b in pairs), hist


# ---- 4. known answers ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("ne", [2, 4])
def test_known_answer_uniform_distributed_couple(integ, ne):
    """lbar = c e_z, M_tip = M e_z: K_z = (M + c (1 - X)) / H_z exactly, i.e. qe[2ne] = (M + c/2) / H_z, qe[2ne+1] = -c / (2 H_z)."""
    N, B, c, M = 16, 1, 0.4, 0.3
    h = integ(N)
    lbar = np.zeros((B, 3, N)); lbar[:, 2] = c
    t = {"F_tip": np.zeros((B, 3)), "M_tip": np.array([[0.0, 0.0, M]]), "lbar": lbar}
    qe, rep = _solve(h, t, ne)
    want = np.zeros((B, 3 * ne)); want[0, 2 * ne] = (M + c / 2) / H0[2]; want[0, 2 * ne + 1] = -c / (2 * H0[2])
    assert np.abs(qe - want).max() <= 1e-13, qe
    gqe = np.zeros((B, 3 * ne)); gqe[0, 2 * ne] = 1.0
    g = h.static_shape_vjp(_cuda(t["F_tip"]), _cuda(t["M_tip"]), _cuda(qe), _cuda(gqe), H_diag=H0, lbar=_cuda(lbar),
                           want=("lbar", "M_tip", "H"))
    assert abs(float(_np(g["lbar"])[0, 2].sum()) - 1 / (2 * H0[2])) <= 1e-12
    assert abs(float(_np(g["M_tip"])[0, 2]) - 1 / H0[2]) <= 1e-12
    assert abs(float(_np(g["H"])[0, 2]) + (M + c / 2) / H0[2] ** 2) <= 1e-12


def test_known_answer_cantilever_under_self_weight(integ):
    """fbar = (0, 0, -w): the tip deflects by w / (8 H_y), Euler-Bernoulli w L^4 / (8 EI) with L = 1, to O(w^2) relative."""
    N, B, ne, w = 16, 1, 3, 1e-4
    h = integ(N)
    fbar = np.zeros((B, 3, N)); fbar[:, 2] = -w
    t = {"F_tip": np.zeros((B, 3)), "M_tip": np.zeros((B, 3)), "fbar": fbar}
    qe, rep = _solve(h, t, ne)
    assert rep["converged"]
    r = h.integrate_all(h.strain_from_modes(_cuda(qe)), want=("r",))["r"]
    tip_z = float(_np(r)[0, 2, 0])
    assert abs(tip_z / (-w / (8 * H0[1])) - 1) <= 10 * w, tip_z


def test_frame_invariance(integ):
    """Rotating the clamp and every global-frame load by one rotation leaves qe* unchanged; the load gradients rotate.  (The
    rotation of a node is Eigen's un-normalised toRotationMatrix, and R(q_g q) = R(q_g) R(q) only for |q| = 1: the discrete
    map is invariant to the drift of |Q| from 1, 5e-11 in qe* at N = 16 with these loads, round-off at N = 32.)"""
    N, ne, B = 32, 4, 6
    rng = np.random.default_rng(14)
    t = loaded_problem(rng, B, N)
    qg = unit_quaternion(rng, 1)[0]
    w, v = qg[0], qg[1:]
    Rg = (w * w - v @ v) * np.eye(3) + 2 * np.outer(v, v) + 2 * w * np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])
    rot = dict(t, q0=_quat_mul(np.tile(qg, (B, 1)), t["q0"]), F_tip=t["F_tip"] @ Rg.T, M_tip=t["M_tip"] @ Rg.T,
               fbar=np.einsum("kc,bcn->bkn", Rg, t["fbar"]), lbar=np.einsum("kc,bcn->bkn", Rg, t["lbar"]))
    h = integ(N)
    q1, _ = _solve(h, t, ne, tol=1e-14)
    q2, _ = _solve(h, rot, ne, tol=1e-14)
    assert np.abs(q1 - q2).max() <= 1e-12
    gqe = rng.normal(size=(B, 3 * ne))
    want = ("F_tip", "M_tip", "fbar", "lbar")
    g1 = h.static_shape_vjp(t["F_tip"], t["M_tip"], q1, gqe, H_diag=H0, want=want, **_on(np.ascontiguousarray, t))
    g2 = h.static_shape_vjp(rot["F_tip"], rot["M_tip"], q1, gqe, H_diag=H0, want=want, **_on(np.ascontiguousarray, rot))
    assert np.abs(g1["F_tip"] @ Rg.T - g2["F_tip"]).max() <= 1e-12 * np.abs(g1["F_tip"]).max()
    assert np.abs(g1["M_tip"] @ Rg.T - g2["M_tip"]).max() <= 1e-12 * np.abs(g1["M_tip"]).max()
    for k in ("fbar", "lbar"):
        assert np.abs(np.einsum("kc,bcn->bkn", Rg, g1[k]) - g2[k]).max() <= 1e-12 * np.abs(g1[k]).max(), k


# ---- 5. gradients -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("N,steps", [(5, 12), (9, 3), (16, 3), (32, 3)])
def test_static_problem_vjp_matches_reference_at_the_gpu_equilibrium(make_oracle, integ, N, steps):
    from static_loads_ref import adjoint
    rng = np.random.default_rng(5000 + N)
    B, ne = 4, 3
    t = loaded_problem(rng, B, N)
    h = integ(N)
    qe, rep = _solve(h, t, ne)
    assert rep["max_abs"] < 1e-12
    gqe = rng.normal(size=(B, 3 * ne))
    info = _cuda(np.full(B, -1, dtype=np.int32))
    got = h.static_shape_vjp(_cuda(t["F_tip"]), _cuda(t["M_tip"]), _cuda(qe), _cuda(gqe), H_diag=H0, refine_steps=steps,
                             info=info, want=ALL_GRADS, **_on(_cuda, t))
    assert not _np(info).any()
    assert float(_np(got["resid"]).max()) <= 1e-12, _np(got["resid"])
    ref = adjoint(make_oracle(N), qe, t["F_tip"], t["M_tip"], H0, ne, gqe, **{k: t[k] for k in OPTIONAL})
    for k in ALL_GRADS[:-1]:
        assert rel_err(_np(got[k]), ref[k]) <= 1e-10, (N, k)


def test_static_problem_vjp_against_central_differences_of_the_gpu_newton_solve(integ):
    N, ne, B, hstep = 16, 4, 8, 1e-5
    rng = np.random.default_rng(15)
    t = loaded_problem(rng, B, N)
    h = integ(N)
    qe, _ = _solve(h, t, ne, tol=1e-14)
    gqe = rng.normal(size=(B, 3 * ne))
    g = {k: _np(v) for k, v in h.static_shape_vjp(_cuda(t["F_tip"]), _cuda(t["M_tip"]), _cuda(qe), _cuda(gqe), H_diag=H0,
                                                  want=INPUTS, **_on(_cuda, t)).items()}
    for k in INPUTS:
        d = rng.normal(size=t[k].shape)
        qp, rp = _solve(h, dict(t, **{k: t[k] + hstep * d}), ne, tol=1e-14)
        qm, rm = _solve(h, dict(t, **{k: t[k] - hstep * d}), ne, tol=1e-14)
        assert rp["max_abs"] < 1e-13 and rm["max_abs"] < 1e-13
        fd = float(np.sum(gqe * (qp - qm))) / (2 * hstep)
        terms = g[k] * d
        assert abs(fd - float(terms.sum())) <= 1e-6 * max(abs(float(terms.sum())), float(np.abs(terms).sum())), (k, fd)


def test_static_problem_vjp_outputs_alone_and_host_buffers_are_bitwise_identical(integ):
    N, ne, B = 16, 4, 37
    rng = np.random.default_rng(16)
    t = loaded_problem(rng, B, N)
    h = integ(N)
    qe, _ = _solve(h, t, ne)
    gqe = rng.normal(size=(B, 3 * ne))
    call = lambda conv, want: h.static_shape_vjp(conv(t["F_tip"]), conv(t["M_tip"]), conv(qe), conv(gqe), H_diag=H0,
                                                 want=want, **_on(conv, t))
    full = {k: _np(v) for k, v in call(_cuda, ALL_GRADS).items()}
    for k in ALL_GRADS:
        alone = call(_cuda, (k,))
        assert set(alone) == {k} and np.array_equal(_np(alone[k]), full[k]), k
    host = call(np.ascontiguousarray, ALL_GRADS)
    for k in ALL_GRADS:
        assert np.array_equal(host[k], full[k]), k


def test_static_problem_vjp_non_finite_load_is_reported_alone(integ):
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import SriError
    N, ne, B = 16, 4, 6
    rng = np.random.default_rng(17)
    t = loaded_problem(rng, B, N)
    h = integ(N)
    qe, _ = _solve(h, t, ne)
    gqe = rng.normal(size=(B, 3 * ne))
    want = ALL_GRADS
    ref = h.static_shape_vjp(_cuda(t["F_tip"]), _cuda(t["M_tip"]), _cuda(qe), _cuda(gqe), H_diag=H0, want=want, **_on(_cuda, t))
    bad = dict(t, fbar=t["fbar"].copy()); bad["fbar"][2, 1, 5] = np.nan
    info = np.full(B, -7, dtype=np.int32)
    with pytest.raises(SriError) as e:
        h.static_shape_vjp(bad["F_tip"], bad["M_tip"], qe, gqe, H_diag=H0, info=info, want=want, **_on(np.ascontiguousarray, bad))
    assert e.value.code == -5
    assert info[2] != 0 and not np.delete(info, 2).any()
    dinfo = _cuda(np.zeros(B, dtype=np.int32))
    dev = h.static_shape_vjp(_cuda(bad["F_tip"]), _cuda(bad["M_tip"]), _cuda(qe), _cuda(gqe), H_diag=H0, info=dinfo, want=want,
                             **_on(_cuda, bad))
    assert np.array_equal(_np(dinfo), info)
    keep = [b for b in range(B) if b != 2]
    for k in want:
        assert np.array_equal(_np(dev[k])[keep], _np(ref[k])[keep]), k


def test_empty_batches_and_argument_errors(integ):
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import _lib
    import torch
    N, ne = 9, 2
    h = integ(N)
    lib, hh = h._lib, h._h
    H = (ctypes.c_double * 3)(1.0, 1.0, 0.77)
    buf = (ctypes.c_double * 4096)()
    rep = _lib.NewtonReport()
    grads = _lib.StaticProblemGrad()
    P = lambda **kw: _lib.StaticProblem(**dict(dict(batch=1, ne=ne, H_diag=ctypes.addressof(H), F_tip=ctypes.addressof(buf),
                                                    M_tip=ctypes.addressof(buf), fbar=ctypes.addressof(buf)), **kw))
    newton = lambda p, qe=buf, max_iter=30, fd=0.0: lib.sri_newton_static_problem(
        hh, p if p is None else ctypes.byref(p), qe, 1e-10, max_iter, fd, 0, _lib.ALLREDUCE_FN(), None, ctypes.byref(rep))
    vjp = lambda p, qe=buf, gqe=buf, steps=3, g=grads: lib.sri_static_problem_vjp(
        hh, p if p is None else ctypes.byref(p), qe, gqe, steps, g if g is None else ctypes.byref(g))
    for p in (P(ne=0), P(ne=9), P(batch=-1), P(H_diag=None), P(F_tip=None)):
        assert newton(p) == -1 and vjp(p) == -1
    assert newton(None) == -1 and vjp(None) == -1 and vjp(P(), g=None) == -1
    assert newton(P(), qe=None) == -1 and newton(P(), max_iter=63) == -1 and newton(P(), fd=-1.0) == -1
    assert vjp(P(), qe=None) == -1 and vjp(P(), gqe=None) == -1 and vjp(P(), steps=-1) == -1
    assert newton(P(batch=0)) == 0 and vjp(P(batch=0)) == 0
    e3, eN = torch.zeros((0, 3), dtype=torch.float64, device="cuda"), torch.zeros((0, 3, N), dtype=torch.float64, device="cuda")
    qe, r = h.newton_static_shape(e3, e3, ne, H_diag=H0, fbar=eN, fd_step=0.0)
    assert qe.shape == (0, 3 * ne) and r["iterations"] == 0
    g = h.static_shape_vjp(e3, e3, qe, qe, H_diag=H0, fbar=eN, want=("fbar", "q0"))
    assert g["fbar"].shape == (0, 3, N) and g["q0"].shape == (0, 4)


# ---- 6. the sharded solve -----------------------------------------------------------------------------------------------

def test_sharded_static_problem_is_bit_identical_to_one_device(integ):
    """On a one-GPU box the shards are three handles on device 0, which runs the same code."""
    import torch
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import MultiDeviceIntegrator
    ndev = torch.cuda.device_count()
    devices = list(range(ndev)) if ndev > 1 else [0, 0, 0]
    N, ne, B = 16, 3, 2003
    t = loaded_problem(np.random.default_rng(18), B, N)
    q1, rep1 = _solve(integ(N), t, ne, conv=np.ascontiguousarray, tol=1e-12)
    with MultiDeviceIntegrator(N, devices=devices) as mh:
        qm, repm = mh.newton_static_shape(t["F_tip"], t["M_tip"], ne, H0, tol=1e-12, max_iter=40, **_on(np.ascontiguousarray, t))
    assert repm["converged"] and repm["iterations"] == rep1["iterations"]
    assert np.allclose(repm["rms_history"], rep1["rms_history"], rtol=1e-9, atol=1e-16)
    assert np.array_equal(qm, q1)


# ---- 7. autograd --------------------------------------------------------------------------------------------------------

def test_static_shape_gradcheck_with_loads_and_only_required_gradients(integ, monkeypatch):
    import torch
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200.autograd import static_shape
    N, ne, B = 9, 2, 2
    rng = np.random.default_rng(19)
    t = loaded_problem(rng, B, N)
    h = integ(N)
    F, Mt, K0 = _cuda(t["F_tip"]), _cuda(t["M_tip"]), _cuda(t["K0"])
    x = {k: _cuda(t[k]).requires_grad_() for k in INPUTS}
    f = lambda q0, G, fb, lb: static_shape(h, F, Mt, ne, tuple(H0), K0=K0, refine_steps=6, q0=q0, Gamma=G, fbar=fb, lbar=lb)
    assert torch.autograd.gradcheck(f, tuple(x[k] for k in INPUTS))
    asked = []
    real = h.static_shape_vjp
    monkeypatch.setattr(h, "static_shape_vjp", lambda *a, **kw: (asked.append(tuple(kw["want"])), real(*a, **kw))[1])
    fb = x["fbar"].detach().clone().requires_grad_()
    lb = x["lbar"].detach().clone()
    qe = static_shape(h, F, Mt, ne, tuple(H0), K0=K0, q0=x["q0"].detach(), Gamma=x["Gamma"].detach(), fbar=fb, lbar=lb)
    qe.sum().backward()
    assert asked == [("fbar",)] and fb.grad is not None and lb.grad is None


def test_inverse_problem_recovers_self_weight(integ):
    """L-BFGS over the weight g_b of 64 rods, fbar = (0, 0, -g_b), through static_shape -> strain_from_modes -> integrate_all,
    so that every node's position matches targets made from known weights (clamp rotated, tip loads known)."""
    import torch
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import autograd as ag
    N, ne, B = 16, 4, 64
    h = integ(N)
    rng = np.random.default_rng(20)
    F, Mt = (_cuda(rng.uniform(-0.3, 0.3, size=(B, 3))) for _ in range(2))
    q0 = _cuda(unit_quaternion(rng, B))
    g_true = _cuda(rng.uniform(0.2, 1.0, size=B))

    def observe(g):
        zero = torch.zeros((B, N), dtype=torch.float64, device="cuda")
        fbar = torch.stack([zero, zero, -g[:, None].expand(B, N)], dim=1)
        qe = ag.static_shape(h, F, Mt, ne, tuple(H0), q0=q0, fbar=fbar)
        _, r, _, _ = ag.integrate_all(h, ag.strain_from_modes(h, qe, ne), F, Mt, q0=q0, fbar=fbar)
        return r

    with torch.no_grad():
        target = observe(g_true)
    g = torch.full_like(g_true, 0.5).requires_grad_()
    opt = torch.optim.LBFGS([g], lr=1.0, max_iter=200, history_size=50, tolerance_grad=1e-15, tolerance_change=1e-30,
                            line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        loss = 0.5 * ((observe(g) - target) ** 2).sum()
        loss.backward()
        return loss

    for _ in range(3):
        opt.step(closure)
    err = float((g.detach() - g_true).abs().max())
    assert err <= 1e-6, err
