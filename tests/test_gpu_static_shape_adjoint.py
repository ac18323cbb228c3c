"""GPU tests of the reverse mode of the static shape problem: sri_galerkin_residual_vjp and sri_static_shape_vjp against
the numpy restatement (static_adjoint_ref.py), against central differences of the GPU's own Newton solve and a known
closed-form answer, and the torch.autograd bindings galerkin_residual / static_shape (gradcheck, an inverse problem)."""
import ctypes

import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu

H0 = np.array([1.0, 1.0, 0.77])
RES_OUTPUTS = ("K", "K0", "H", "Q", "q0", "m", "M_tip")


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
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(x):
    return x.cpu().numpy()


def _state(rng, B, N):
    M = N - 1
    return {"K": rng.uniform(-2, 2, size=(B, 3, N)), "K0": rng.uniform(-1, 1, size=(B, 3, N)), "Q": rng.normal(size=(B, 4, M)),
            "q0": rng.normal(size=(B, 4)), "m": rng.normal(size=(B, 3, M)), "M_tip": rng.normal(size=(B, 3))}


# ---- sri_galerkin_residual_vjp ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("N", [2, 5, 9, 16, 17, 32, 33, 64])
@pytest.mark.parametrize("ne", [1, 4, 8])
@pytest.mark.parametrize("optional", [False, True])
def test_residual_vjp_matches_reference(make_oracle, integ, N, ne, optional):
    from static_adjoint_ref import galerkin_residual_vjp
    rng = np.random.default_rng(1000 + 10 * N + ne)
    B = 5
    x = _state(rng, B, N)
    K0, q0 = (x["K0"], x["q0"]) if optional else (None, None)
    gg = rng.normal(size=(B, 3 * ne))
    want = galerkin_residual_vjp(make_oracle(N), x["K"], H0, x["Q"], x["m"], x["M_tip"], gg, K0=K0, q0=q0)
    c = lambda a: None if a is None else _cuda(a)
    got = integ(N).galerkin_residual_vjp(_cuda(x["K"]), H0, _cuda(x["Q"]), _cuda(x["m"]), _cuda(x["M_tip"]), _cuda(gg),
                                         K0=c(K0), q0=c(q0))
    for k in RES_OUTPUTS:
        assert rel_err(_np(got[k]), want[k]) <= 1e-12, (N, ne, k)


@pytest.mark.parametrize("N", [16, 33])
def test_residual_vjp_outputs_alone_and_host_buffers_are_bitwise_identical(integ, N):
    rng = np.random.default_rng(7 + N)
    B, ne = 37, 4
    x = _state(rng, B, N)
    gg = rng.normal(size=(B, 3 * ne))
    h = integ(N)
    args = lambda conv: [conv(x["K"]), H0, conv(x["Q"]), conv(x["m"]), conv(x["M_tip"]), conv(gg)]
    kw = lambda conv: {"K0": conv(x["K0"]), "q0": conv(x["q0"])}
    full = {k: _np(v) for k, v in h.galerkin_residual_vjp(*args(_cuda), **kw(_cuda)).items()}
    for k in RES_OUTPUTS:
        alone = h.galerkin_residual_vjp(*args(_cuda), **kw(_cuda), want=(k,))
        assert set(alone) == {k} and np.array_equal(_np(alone[k]), full[k]), k
    host = h.galerkin_residual_vjp(*args(np.ascontiguousarray), **kw(np.ascontiguousarray))
    for k in RES_OUTPUTS:
        assert np.array_equal(host[k], full[k]), k
    again = h.galerkin_residual_vjp(*args(_cuda), **kw(_cuda), want=("H",))
    assert np.array_equal(_np(again["H"]), full["H"])   # the per-rod reduction is reproducible


@pytest.mark.parametrize("B", [0, 1, 3, 129, 1000])
def test_residual_vjp_batches(make_oracle, integ, B):
    from static_adjoint_ref import galerkin_residual_vjp
    N, ne = 16, 3
    rng = np.random.default_rng(50 + B)
    x = _state(rng, B, N)
    gg = rng.normal(size=(B, 3 * ne))
    got = integ(N).galerkin_residual_vjp(_cuda(x["K"]), H0, _cuda(x["Q"]), _cuda(x["m"]), _cuda(x["M_tip"]), _cuda(gg),
                                         K0=_cuda(x["K0"]), q0=_cuda(x["q0"]))
    if B == 0:
        return
    want = galerkin_residual_vjp(make_oracle(N), x["K"], H0, x["Q"], x["m"], x["M_tip"], gg, K0=x["K0"], q0=x["q0"])
    for k in RES_OUTPUTS:
        assert rel_err(_np(got[k]), want[k]) <= 1e-12, (B, k)


# ---- sri_static_shape_vjp --------------------------------------------------------------------------------------------

def _loads(rng, B, scale=0.6):
    return rng.uniform(-scale, scale, size=(B, 3)), rng.uniform(-scale, scale, size=(B, 3))


def _equilibrium(h, F, Mt, ne, K0=None, tol=1e-13):
    qe, rep = h.newton_static_shape(_cuda(F), _cuda(Mt), ne, H_diag=H0, K0=None if K0 is None else _cuda(K0), tol=tol,
                                    max_iter=40, fd_step=0.0)
    assert rep["rms"] < 1e-12, rep
    return qe


@pytest.mark.parametrize("N,steps", [(5, 12), (9, 3), (16, 3), (32, 3)])
@pytest.mark.parametrize("ne", [2, 4])
def test_static_shape_vjp_matches_reference_at_the_gpu_equilibrium(make_oracle, integ, N, steps, ne):
    from static_adjoint_ref import static_shape_vjp
    rng = np.random.default_rng(2000 + 10 * N + ne)
    B = 4
    F, Mt = _loads(rng, B)
    K0 = rng.uniform(-0.3, 0.3, size=(B, 3, N))
    h = integ(N)
    qe = _equilibrium(h, F, Mt, ne, K0)
    gqe = rng.normal(size=(B, 3 * ne))
    info = _cuda(np.zeros(B, dtype=np.int32))
    got = h.static_shape_vjp(_cuda(F), _cuda(Mt), qe, _cuda(gqe), H_diag=H0, K0=_cuda(K0), refine_steps=steps, info=info,
                             want=("F_tip", "M_tip", "K0", "H", "lambda", "resid"))
    assert not _np(info).any()
    assert float(_np(got["resid"]).max()) <= 1e-12, _np(got["resid"])
    want = static_shape_vjp(make_oracle(N), _np(qe), F, Mt, H0, ne, gqe, K0=K0)
    for k in ("F_tip", "M_tip", "K0", "H", "lambda"):
        assert rel_err(_np(got[k]), want[k]) <= 1e-10, (N, ne, k)
    if N == 16:   # J_a alone is exact to 5e-12 there
        zero = h.static_shape_vjp(_cuda(F), _cuda(Mt), qe, _cuda(gqe), H_diag=H0, K0=_cuda(K0), refine_steps=0)
        for k in ("F_tip", "M_tip", "K0", "H"):
            assert rel_err(_np(zero[k]), _np(got[k])) <= 1e-10, k


def test_static_shape_vjp_against_central_differences_of_the_gpu_newton_solve(integ):
    N, ne, B, hstep = 16, 4, 8, 1e-5
    rng = np.random.default_rng(77)
    F, Mt = _loads(rng, B)
    K0 = rng.uniform(-0.3, 0.3, size=(B, 3, N))
    h = integ(N)
    theta = {"F_tip": F, "M_tip": Mt, "K0": K0}
    gqe = rng.normal(size=(B, 3 * ne))

    def solve(t, H=H0):
        qe, rep = h.newton_static_shape(_cuda(t["F_tip"]), _cuda(t["M_tip"]), ne, H_diag=H, K0=_cuda(t["K0"]), tol=1e-14,
                                        max_iter=40, fd_step=0.0)
        assert rep["max_abs"] < 1e-13, rep
        return _np(qe)

    qe = solve(theta)
    g = {k: _np(v) for k, v in h.static_shape_vjp(_cuda(F), _cuda(Mt), _cuda(qe), _cuda(gqe), H_diag=H0, K0=_cuda(K0)).items()}
    for k in ("F_tip", "M_tip", "K0", "H"):
        d = rng.normal(size=(3,) if k == "H" else theta[k].shape)
        if k == "H":
            fd = float(np.sum(gqe * (solve(theta, H0 + hstep * d) - solve(theta, H0 - hstep * d)))) / (2 * hstep)
            terms = g["H"].sum(0) * d
        else:
            fd = float(np.sum(gqe * (solve(dict(theta, **{k: theta[k] + hstep * d})) -
                                     solve(dict(theta, **{k: theta[k] - hstep * d}))))) / (2 * hstep)
            terms = g[k] * d
        ad = float(terms.sum())
        assert abs(fd - ad) <= 1e-6 * max(abs(ad), float(np.abs(terms).sum())), (k, fd, ad)


@pytest.mark.parametrize("c", [0, 1, 2])
def test_static_shape_vjp_known_answer_pure_tip_moment(integ, c):
    """M_tip = M_c e_c, F = 0: the equilibrium is the constant K = M_c / H_c e_c, so qe*[c*ne] = M_c / H_c."""
    N, ne, B, Mc = 16, 3, 1, 0.7
    h = integ(N)
    F = np.zeros((B, 3))
    Mt = np.zeros((B, 3)); Mt[0, c] = Mc
    qe = _equilibrium(h, F, Mt, ne)
    assert abs(float(_np(qe)[0, c * ne]) - Mc / H0[c]) <= 1e-12
    gqe = np.zeros((B, 3 * ne)); gqe[0, c * ne] = 1.0
    g = h.static_shape_vjp(_cuda(F), _cuda(Mt), qe, _cuda(gqe), H_diag=H0, want=("M_tip", "H"))
    assert abs(float(_np(g["M_tip"])[0, c]) - 1.0 / H0[c]) <= 1e-10 / H0[c]
    assert abs(float(_np(g["H"])[0, c]) + Mc / H0[c] ** 2) <= 1e-10 * Mc / H0[c] ** 2


def test_static_shape_vjp_non_finite_rod_is_reported_alone(integ):
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import SriError
    N, ne, B = 16, 4, 6
    rng = np.random.default_rng(5)
    F, Mt = _loads(rng, B)
    h = integ(N)
    qe = _np(_equilibrium(h, F, Mt, ne))
    gqe = rng.normal(size=(B, 3 * ne))
    want = ("F_tip", "M_tip", "H", "lambda", "resid")
    ref = h.static_shape_vjp(F, Mt, qe, gqe, H_diag=H0, want=want)
    Fbad = F.copy(); Fbad[2, 1] = np.nan
    info = np.full(B, -7, dtype=np.int32)
    h.set_timing(True)
    with pytest.raises(SriError) as e:
        h.static_shape_vjp(Fbad, Mt, qe, gqe, H_diag=H0, info=info, want=want)
    assert e.value.code == -5
    assert info[2] != 0 and (info[2] & 0xff) >= 1 and not np.delete(info, 2).any()
    ms, name = h.last_timing()
    h.set_timing(False)
    assert name == "sri_static_shape_vjp" and ms > 0
    # the other rods' results with device buffers are those of the call without the bad rod, bit for bit
    dinfo = _cuda(np.zeros(B, dtype=np.int32))
    dev = h.static_shape_vjp(_cuda(Fbad), _cuda(Mt), _cuda(qe), _cuda(gqe), H_diag=H0, info=dinfo, want=want)
    assert np.array_equal(_np(dinfo), info)
    keep = [b for b in range(B) if b != 2]
    for k in want:
        assert np.array_equal(_np(dev[k])[keep], ref[k][keep]), k


def test_static_shape_vjp_argument_errors(integ):
    h = integ(9)
    lib, hh = h._lib, h._h
    H = (ctypes.c_double * 3)(1.0, 1.0, 0.77)
    buf = (ctypes.c_double * 64)()
    assert lib.sri_static_shape_vjp(hh, 1, 0, H, buf, buf, None, buf, buf, 3, *[None] * 7) == -1
    assert lib.sri_static_shape_vjp(hh, 1, 2, H, buf, buf, None, buf, buf, -1, *[None] * 7) == -1
    assert lib.sri_static_shape_vjp(hh, 1, 2, H, buf, buf, None, buf, None, 3, *[None] * 7) == -1
    assert lib.sri_static_shape_vjp(hh, -1, 2, H, *[None] * 5, 3, *[None] * 7) == -1
    assert lib.sri_static_shape_vjp(hh, 0, 2, H, *[None] * 5, 3, *[None] * 7) == 0
    assert lib.sri_galerkin_residual_vjp(hh, 1, 9, buf, None, H, buf, None, buf, buf, buf, *[None] * 7) == -1
    assert lib.sri_galerkin_residual_vjp(hh, 1, 2, None, None, H, buf, None, buf, buf, buf, *[None] * 7) == -1


# ---- torch.autograd ----------------------------------------------------------------------------------------------------

def test_galerkin_residual_gradcheck(integ):
    import torch
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200.autograd import galerkin_residual
    N, ne, B = 5, 2, 2
    rng = np.random.default_rng(9)
    x = {k: _cuda(v).requires_grad_() for k, v in _state(rng, B, N).items()}
    H = _cuda(H0).requires_grad_()
    f = lambda K, Q, m, Mt, H, K0, q0: galerkin_residual(integ(N), K, Q, m, Mt, ne, H, K0=K0, q0=q0)
    assert torch.autograd.gradcheck(f, (x["K"], x["Q"], x["m"], x["M_tip"], H, x["K0"], x["q0"]))


def test_static_shape_gradcheck_and_only_required_gradients(integ):
    import torch
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200.autograd import static_shape
    N, ne, B = 9, 2, 2
    rng = np.random.default_rng(11)
    F, Mt = (_cuda(a).requires_grad_() for a in _loads(rng, B))
    K0 = _cuda(rng.uniform(-0.3, 0.3, size=(B, 3, N))).requires_grad_()
    H = _cuda(H0).requires_grad_()
    f = lambda F, Mt, K0, H: static_shape(integ(N), F, Mt, ne, H, K0=K0)
    assert torch.autograd.gradcheck(f, (F, Mt, K0, H))
    Fo, Mo = F.detach().clone().requires_grad_(), Mt.detach().clone()
    qe = static_shape(integ(N), Fo, Mo, ne, tuple(H0))
    qe.sum().backward()
    assert Fo.grad is not None and Mo.grad is None
    with pytest.raises(RuntimeError, match="did not converge"):
        static_shape(integ(N), Fo, Mo, ne, tuple(H0), max_iter=1)


def test_inverse_problem_recovers_tip_loads(integ):
    """L-BFGS over the tip loads of 64 rods, through static_shape -> strain_from_modes -> integrate_all, so that the shape (every
    node's position) and the wrench at the clamped base match targets made from known loads.  (The shape alone hardly sees the
    axial part of the tip force of an inextensible rod; the base wrench, what a load cell at the clamp reads, pins it.)"""
    import torch
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import autograd as ag
    N, ne, B = 16, 4, 64
    h = integ(N)
    rng = np.random.default_rng(21)
    F_true, M_true = (_cuda(a) for a in _loads(rng, B, 0.5))

    def observe(F, Mt):
        qe = ag.static_shape(h, F, Mt, ne, tuple(H0))
        _, r, n, m = ag.integrate_all(h, ag.strain_from_modes(h, qe, ne), F, Mt)
        return r, n[:, :, -1], m[:, :, -1]

    with torch.no_grad():
        target = observe(F_true, M_true)
    F = torch.zeros_like(F_true, requires_grad=True)
    Mt = torch.zeros_like(M_true, requires_grad=True)
    opt = torch.optim.LBFGS([F, Mt], lr=1.0, max_iter=200, history_size=50, tolerance_grad=1e-15, tolerance_change=1e-30,
                            line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        loss = 0.5 * sum(((o - t) ** 2).sum() for o, t in zip(observe(F, Mt), target))
        loss.backward()
        return loss

    for _ in range(3):
        opt.step(closure)
    err = max(float((F.detach() - F_true).abs().max()), float((Mt.detach() - M_true).abs().max()))
    assert err <= 1e-6, err
