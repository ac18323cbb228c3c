"""GPU tests of the reverse mode: sri_integrate_all_vjp against the numpy restatement oracle/adjoint.py, its argument and
failure handling, the transpose of the modal strain adapter, and the torch.autograd binding (gradcheck and a shape fit)."""
import ctypes

import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-12
INPUTS = ("K", "q0", "r0", "Gamma", "fbar", "lbar", "F_tip", "M_tip")
COTS = ("gQ", "gr", "gn", "gm")


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    return torch


def _integrator(N):
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import SpectralRodIntegrator
    return SpectralRodIntegrator(N, 0)


def _rods(rng, B, N, optional=True):
    K = rng.uniform(-2, 2, size=(B, 3, N))
    F, Mt = rng.normal(size=(B, 3)), rng.normal(size=(B, 3))
    if not optional:
        return K, F, Mt, {}
    q0 = rng.normal(size=(B, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    Gam = rng.normal(scale=0.3, size=(B, 3, N)); Gam[:, 0] += 1.0
    return K, F, Mt, {"q0": q0, "r0": rng.normal(size=(B, 3)), "Gamma": Gam, "fbar": rng.normal(size=(B, 3, N)),
                      "lbar": rng.normal(size=(B, 3, N))}


def _cotangents(rng, B, M):
    return {"gQ": rng.normal(size=(B, 4, M)), "gr": rng.normal(size=(B, 3, M)), "gn": rng.normal(size=(B, 3, M)),
            "gm": rng.normal(size=(B, 3, M))}


def _reference(o, K, F, Mt, opt, cot):
    fwd = o.integrate_all(K, F, Mt, explicit_inverse=False, **opt)
    from oracle.adjoint import integrate_all_vjp
    ref = integrate_all_vjp(o, K, fwd["Q"], n=fwd["n"], q0=opt.get("q0"), Gamma=opt.get("Gamma"), **cot)
    return fwd, ref


def _gpu_vjp(h, torch, K, Q, n, q0, Gamma, cot, want=INPUTS, host=False):
    """sri_integrate_all_vjp through the Python wrapper; device tensors unless host=True (numpy in, numpy out)."""
    B = K.shape[0]
    conv = (lambda a: None if a is None else np.ascontiguousarray(a)) if host else \
        (lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda())
    info = np.full(B, -1, dtype=np.int32) if host else torch.full((B,), -1, dtype=torch.int32, device="cuda")
    g = h.integrate_all_vjp(conv(K), conv(Q), n=conv(n), q0=conv(q0), Gamma=conv(Gamma),
                            **{k: conv(v) for k, v in cot.items()}, info=info, want=want)
    h.synchronize()
    res = {k: (v if host else v.cpu().numpy()) for k, v in g.items()}
    res["info"] = info if host else info.cpu().numpy()
    return res


@pytest.mark.parametrize("optional", [True, False], ids=["all_inputs", "defaults"])
@pytest.mark.parametrize("N", [2, 3, 5, 11, 16, 17, 24, 32, 33, 48, 64])
def test_vjp_matches_oracle(make_oracle, torch_mod, N, optional):
    o = make_oracle(N)
    rng = np.random.default_rng(7 * N + optional)
    B = 37  # odd: the N <= 16 kernel's last warp holds one rod
    K, F, Mt, opt = _rods(rng, B, N, optional)
    cot = _cotangents(rng, B, N - 1)
    fwd, ref = _reference(o, K, F, Mt, opt, cot)
    with _integrator(N) as h:
        got = _gpu_vjp(h, torch_mod, K, fwd["Q"], fwd["n"], opt.get("q0"), opt.get("Gamma"), cot)
    assert (got["info"] == 0).all()
    for k in INPUTS:
        assert rel_err(got[k], ref[k]) <= TOL, (N, k, rel_err(got[k], ref[k]))


@pytest.mark.parametrize("N", [16, 33])
@pytest.mark.parametrize("B", [0, 1, 2, 3, 129, 1000])
def test_vjp_ragged_and_empty_batches(make_oracle, torch_mod, N, B):
    rng = np.random.default_rng(B + N)
    K, F, Mt, opt = _rods(rng, B, N)
    cot = _cotangents(rng, B, N - 1)
    with _integrator(N) as h:
        if B == 0:
            got = _gpu_vjp(h, torch_mod, K, np.zeros((0, 4, N - 1)), np.zeros((0, 3, N - 1)), opt["q0"], opt["Gamma"], cot)
            assert all(got[k].shape[0] == 0 for k in INPUTS)
            return
        o = make_oracle(N)
        sel = np.unique(np.r_[0, B - 1, rng.integers(0, B, size=min(B, 40))])  # the oracle on a sample incl. both ends
        fwd, ref = _reference(o, K[sel], F[sel], Mt[sel], {k: v[sel] for k, v in opt.items()}, {k: v[sel] for k, v in cot.items()})
        full = o.integrate_all(K, F, Mt, explicit_inverse=False, **opt)
        got = _gpu_vjp(h, torch_mod, K, full["Q"], full["n"], opt["q0"], opt["Gamma"], cot)
    for k in INPUTS:
        assert rel_err(got[k][sel], ref[k]) <= TOL, (N, B, k)


@pytest.mark.parametrize("N", [16, 33])
def test_vjp_host_and_device_buffers_agree_bitwise(make_oracle, torch_mod, N):
    rng = np.random.default_rng(11)
    B = 300
    K, F, Mt, opt = _rods(rng, B, N)
    cot = _cotangents(rng, B, N - 1)
    fwd = make_oracle(N).integrate_all(K, F, Mt, explicit_inverse=False, **opt)
    with _integrator(N) as h:
        dev = _gpu_vjp(h, torch_mod, K, fwd["Q"], fwd["n"], opt["q0"], opt["Gamma"], cot)
        host = _gpu_vjp(h, torch_mod, K, fwd["Q"], fwd["n"], opt["q0"], opt["Gamma"], cot, host=True)
    for k in INPUTS + ("info",):
        assert np.array_equal(dev[k], host[k]), k


@pytest.mark.parametrize("N", [5, 16, 33])
def test_vjp_each_cotangent_alone_and_each_gradient_alone(make_oracle, torch_mod, N):
    o = make_oracle(N)
    rng = np.random.default_rng(3 * N)
    B = 20
    K, F, Mt, opt = _rods(rng, B, N)
    cot = _cotangents(rng, B, N - 1)
    fwd = o.integrate_all(K, F, Mt, explicit_inverse=False, **opt)
    from oracle.adjoint import integrate_all_vjp
    with _integrator(N) as h:
        for c in COTS:
            ref = integrate_all_vjp(o, K, fwd["Q"], n=fwd["n"], q0=opt["q0"], Gamma=opt["Gamma"], **{c: cot[c]})
            n = fwd["n"] if c == "gm" else None  # n is read only with gm
            got = _gpu_vjp(h, torch_mod, K, fwd["Q"], n, opt["q0"], opt["Gamma"], {c: cot[c]})
            for k in INPUTS:
                if np.abs(ref[k]).max() == 0.0:
                    assert not got[k].any(), (c, k)
                else:
                    assert rel_err(got[k], ref[k]) <= TOL, (N, c, k)
        every = _gpu_vjp(h, torch_mod, K, fwd["Q"], fwd["n"], opt["q0"], opt["Gamma"], cot)
        for k in INPUTS:
            alone = _gpu_vjp(h, torch_mod, K, fwd["Q"], fwd["n"], opt["q0"], opt["Gamma"], cot, want=(k,))
            assert set(alone) == {k, "info"}
            assert np.array_equal(alone[k], every[k]), k


def test_vjp_large_curvature_needs_pivoting(make_oracle, torch_mod):
    """The rods of test_large_curvature_needs_pivoting (gpu parity suite): the transposed stage-1 operator has the
    forward's conditioning, so the CPU LU is only good to ~cond*eps there as well; compare at 1e-10 like that test."""
    o = make_oracle(16)
    rng = np.random.default_rng(5)
    B = 2000
    K = rng.uniform(-40, 40, size=(B, 3, 1)) + rng.uniform(-40, 40, size=(B, 3, 1)) * np.linspace(1, -1, 16)[None, None, :]
    F = rng.uniform(-1, 1, size=(B, 3)); Mt = rng.uniform(-1, 1, size=(B, 3))
    sel = np.arange(0, B, 10)
    cot = _cotangents(np.random.default_rng(6), B, 15)
    fwd = o.integrate_all(K, F, Mt, explicit_inverse=False)
    from oracle.adjoint import integrate_all_vjp
    ref = integrate_all_vjp(o, K[sel], fwd["Q"][sel], n=fwd["n"][sel], **{k: v[sel] for k, v in cot.items()})
    with _integrator(16) as h:
        got = _gpu_vjp(h, torch_mod, K, fwd["Q"], fwd["n"], None, None, cot)
    assert (got["info"] == 0).all()
    for k in INPUTS:
        assert rel_err(got[k][sel], ref[k]) <= 1e-10, k


@pytest.mark.parametrize("N", [16, 32])
def test_vjp_non_finite_rod_is_reported_not_fatal(make_oracle, torch_mod, N):
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import SriError
    o = make_oracle(N)
    rng = np.random.default_rng(9)
    B = 50
    K, F, Mt, opt = _rods(rng, B, N)
    cot = _cotangents(rng, B, N - 1)
    fwd, ref = _reference(o, K, F, Mt, opt, cot)
    Kbad = K.copy()
    Kbad[7, 1, 2] = np.nan
    Kbad[30, 0, 0] = np.inf
    good = np.setdiff1d(np.arange(B), [7, 30])
    with _integrator(N) as h:
        got = _gpu_vjp(h, torch_mod, Kbad, fwd["Q"], fwd["n"], opt["q0"], opt["Gamma"], cot)
        assert got["info"][7] != 0 and got["info"][30] != 0
        assert (got["info"][good] == 0).all()
        for k in INPUTS:
            assert rel_err(got[k][good], ref[k][good]) <= TOL, k
        with pytest.raises(SriError) as e:  # host buffers: the call reports the singular rods after writing every output
            _gpu_vjp(h, torch_mod, Kbad, fwd["Q"], fwd["n"], opt["q0"], opt["Gamma"], cot, host=True)
        assert e.value.code == -5


def test_vjp_argument_errors_are_reported_not_thrown(sri_lib, torch_mod):
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import _lib
    rb, gb = _lib.RodBatch(), _lib.RodBatchGrad()
    assert sri_lib.sri_integrate_all_vjp(None, ctypes.byref(rb), ctypes.byref(gb)) == -1
    assert b"handle" in sri_lib.sri_last_error_string().lower()
    assert sri_lib.sri_strain_from_modes_transpose(None, 1, 3, None, None) == -1
    N, B = 16, 4
    with _integrator(N) as h:
        K = torch_mod.zeros((B, 3, N), dtype=torch_mod.float64, device="cuda")
        Q = torch_mod.zeros((B, 4, N - 1), dtype=torch_mod.float64, device="cuda")
        gm = torch_mod.zeros((B, 3, N - 1), dtype=torch_mod.float64, device="cuda")
        gK = torch_mod.zeros_like(K)
        call = lambda r, g: sri_lib.sri_integrate_all_vjp(h._h, r, g)
        assert call(None, ctypes.byref(gb)) == -1
        assert call(ctypes.byref(rb), None) == -1
        assert call(ctypes.byref(_lib.RodBatch(batch=-1)), ctypes.byref(gb)) == -1
        assert b"negative batch" in sri_lib.sri_last_error_string()
        assert call(ctypes.byref(_lib.RodBatch(batch=0)), ctypes.byref(gb)) == 0  # empty batch: nothing to do
        assert call(ctypes.byref(_lib.RodBatch(batch=B, Q=Q.data_ptr())), ctypes.byref(_lib.RodBatchGrad(gK=gK.data_ptr()))) == -1
        assert b"K is required" in sri_lib.sri_last_error_string()
        assert call(ctypes.byref(_lib.RodBatch(batch=B, K=K.data_ptr())), ctypes.byref(_lib.RodBatchGrad(gK=gK.data_ptr()))) == -1
        assert b"Q" in sri_lib.sri_last_error_string()
        assert call(ctypes.byref(_lib.RodBatch(batch=B, K=K.data_ptr(), Q=Q.data_ptr())),
                    ctypes.byref(_lib.RodBatchGrad(gm=gm.data_ptr(), gK=gK.data_ptr()))) == -1
        assert b"n" in sri_lib.sri_last_error_string()
        for ne in (0, 9):
            assert sri_lib.sri_strain_from_modes_transpose(h._h, B, ne, K.data_ptr(), gK.data_ptr()) == -1
        assert sri_lib.sri_strain_from_modes_transpose(h._h, -1, 3, K.data_ptr(), gK.data_ptr()) == -1


def test_vjp_is_timed_as_its_own_entry_point(make_oracle, torch_mod):
    rng = np.random.default_rng(2)
    K, F, Mt, opt = _rods(rng, 64, 16)
    fwd = make_oracle(16).integrate_all(K, F, Mt, explicit_inverse=False, **opt)
    t = lambda a: torch_mod.from_numpy(np.ascontiguousarray(a)).cuda()
    with _integrator(16) as h:
        h.set_timing(True)
        h.integrate_all_vjp(t(K), t(fwd["Q"]), n=t(fwd["n"]), **{k: t(v) for k, v in _cotangents(rng, 64, 15).items()})
        ms, name = h.last_timing()  # (waits for the call)
    assert name == "sri_integrate_all_vjp" and ms > 0.0


@pytest.mark.parametrize("N", [16, 33])
def test_strain_from_modes_transpose(make_oracle, torch_mod, N):
    """<gK, Phi qe> = <Phi^T gK, qe>: the adapter's transpose against the oracle's Phi at the nodes."""
    o = make_oracle(N)
    rng = np.random.default_rng(N)
    B = 33
    x = o.chebyshev_points()
    with _integrator(N) as h:
        for ne in (1, 3, 8):
            gK = rng.normal(size=(B, 3, N))
            P = np.stack([o.phi(3, ne, xi) for xi in x])                 # [N][3][3 ne]
            ref = np.einsum("bci,icd->bd", gK, P)
            got = h.strain_from_modes_transpose(torch_mod.from_numpy(gK).cuda(), ne).cpu().numpy()
            assert rel_err(got, ref) <= TOL, ne


@pytest.mark.parametrize("N", [5, 16, 33])
def test_autograd_gradcheck(make_oracle, torch_mod, N):
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import autograd
    torch = torch_mod
    rng = np.random.default_rng(N)
    K, F, Mt, opt = _rods(rng, 4, N)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda().requires_grad_(True)
    args = [t(K), t(F), t(Mt), t(opt["q0"]), t(opt["r0"]), t(opt["Gamma"]), t(opt["fbar"]), t(opt["lbar"])]
    with _integrator(N) as h:
        fn = lambda K, F, Mt, q0, r0, G, fb, lb: autograd.integrate_all(h, K, F, Mt, q0=q0, r0=r0, Gamma=G, fbar=fb, lbar=lb)
        assert torch.autograd.gradcheck(fn, args, eps=1e-6, atol=1e-7, rtol=1e-6)
        qe = t(rng.normal(size=(4, 9)))
        assert torch.autograd.gradcheck(lambda q: autograd.strain_from_modes(h, q, 3), [qe], eps=1e-6, atol=1e-8, rtol=1e-7)


def test_autograd_gradients_only_where_required(torch_mod):
    """Inputs without requires_grad get no gradient, an output without a cotangent contributes none."""
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import autograd
    torch = torch_mod
    rng = np.random.default_rng(4)
    K, F, Mt, _ = _rods(rng, 8, 16, optional=False)
    t = lambda a, g: torch.from_numpy(a).cuda().requires_grad_(g)
    Kt, Ft, Mtt = t(K, True), t(F, False), t(Mt, True)
    with _integrator(16) as h:
        Q, r, n, m = autograd.integrate_all(h, Kt, Ft, Mtt)
        r.square().sum().backward()
        assert Ft.grad is None and Kt.grad is not None
        assert not Mtt.grad.any()  # m received no cotangent: M_tip does not reach r
        g_r = h.integrate_all_vjp(Kt.detach(), Q.detach(), gr=(2 * r).detach(), want=("K",))["K"]
        assert torch.equal(Kt.grad, g_r)


def test_autograd_fits_modal_strain_from_positions_and_orientations(torch_mod):
    """256 rods, N = 16: recover qe* from the r and Q it produces, by L-BFGS through strain_from_modes -> integrate_all.
    Q is needed too: with Gamma = e1, r does not see the twist about the tangent."""
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import autograd
    torch = torch_mod
    rng = np.random.default_rng(12)
    B, ne = 256, 3
    qe_star = torch.from_numpy(rng.uniform(-1, 1, size=(B, 3 * ne))).cuda()
    with _integrator(16) as h:
        Q_star, r_star, _, _ = autograd.integrate_all(h, autograd.strain_from_modes(h, qe_star, ne))
        qe = (qe_star + 0.2 * torch.from_numpy(rng.normal(size=(B, 3 * ne))).cuda()).requires_grad_(True)

        def closure():
            opt.zero_grad()
            Q, r, _, _ = autograd.integrate_all(h, autograd.strain_from_modes(h, qe, ne))
            loss = (r - r_star).square().sum() + (Q - Q_star).square().sum()
            loss.backward()
            return loss

        for _ in range(40):  # a fresh history now and then: one line search serves all 256 rods at once
            opt = torch.optim.LBFGS([qe], lr=1.0, max_iter=300, history_size=50, tolerance_grad=1e-15,
                                    tolerance_change=1e-30, line_search_fn="strong_wolfe")
            opt.step(closure)
            if (qe.detach() - qe_star).abs().max().item() <= 1e-10:
                break
        err = (qe.detach() - qe_star).abs().max().item()
    assert err <= 1e-8, err
