"""CPU tests of the reverse-mode restatement oracle/adjoint.py: the dot-product test against central differences of the
oracle's four-stage integration, for all eight inputs at once and for each input alone."""
import numpy as np
import pytest

INPUTS = ("K", "q0", "r0", "Gamma", "fbar", "lbar", "F_tip", "M_tip")


def _rods(rng, B, N):
    K = rng.uniform(-2, 2, size=(B, 3, N))
    q0 = rng.normal(size=(B, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    return {"K": K, "q0": q0, "r0": rng.normal(size=(B, 3)), "Gamma": rng.normal(size=(B, 3, N)),
            "fbar": rng.normal(size=(B, 3, N)), "lbar": rng.normal(size=(B, 3, N)),
            "F_tip": rng.normal(size=(B, 3)), "M_tip": rng.normal(size=(B, 3))}


def _loss(o, x, cot):
    out = o.integrate_all(explicit_inverse=False, **x)
    return sum(float(np.sum(cot[s] * out[s])) for s in "Qrnm")


@pytest.mark.parametrize("N", [2, 5, 16, 33, 64])
def test_adjoint_dot_product_against_central_differences(make_oracle, N):
    from oracle.adjoint import integrate_all_vjp
    o = make_oracle(N)
    rng = np.random.default_rng(100 + N)
    B, M, h = 3, N - 1, 1e-6
    x = _rods(rng, B, N)
    cot = {"Q": rng.normal(size=(B, 4, M)), "r": rng.normal(size=(B, 3, M)), "n": rng.normal(size=(B, 3, M)),
           "m": rng.normal(size=(B, 3, M))}
    fwd = o.integrate_all(explicit_inverse=False, **x)
    g = integrate_all_vjp(o, x["K"], fwd["Q"], n=fwd["n"], q0=x["q0"], Gamma=x["Gamma"],
                          gQ=cot["Q"], gr=cot["r"], gn=cot["n"], gm=cot["m"])
    assert g["bad"] == 0
    dirs = {k: rng.normal(size=v.shape) for k, v in x.items()}

    def directional(keys):
        xp = {k: v + h * dirs[k] if k in keys else v for k, v in x.items()}
        xm = {k: v - h * dirs[k] if k in keys else v for k, v in x.items()}
        fd = (_loss(o, xp, cot) - _loss(o, xm, cot)) / (2 * h)
        ad = sum(float(np.sum(g[k] * dirs[k])) for k in keys)
        return fd, ad

    fd, ad = directional(INPUTS)
    assert abs(fd - ad) <= 1e-7 * abs(ad), (N, fd, ad)
    for k in INPUTS:  # each input alone, so that an error in one gradient cannot hide behind a larger one
        fd, ad = directional((k,))
        scale = max(abs(ad), float(np.abs(g[k] * dirs[k]).sum()))  # (a sum that cancels is compared with its terms)
        assert abs(fd - ad) <= 1e-7 * scale, (N, k, fd, ad)


def test_adjoint_defaults_match_explicit_identity_and_e1(make_oracle):
    """q0 = None / Gamma = None are the identity and e1, as in the forward; absent cotangents are zero."""
    from oracle.adjoint import integrate_all_vjp
    N, B = 7, 2
    o = make_oracle(N)
    rng = np.random.default_rng(1)
    K = rng.uniform(-2, 2, size=(B, 3, N))
    F, Mt = rng.normal(size=(B, 3)), rng.normal(size=(B, 3))
    fwd = o.integrate_all(K, F, Mt, explicit_inverse=False)
    gm = rng.normal(size=(B, 3, N - 1))
    a = integrate_all_vjp(o, K, fwd["Q"], n=fwd["n"], gm=gm)
    q0 = np.tile([1.0, 0, 0, 0], (B, 1))
    Gam = np.zeros((B, 3, N)); Gam[:, 0] = 1.0
    b = integrate_all_vjp(o, K, fwd["Q"], n=fwd["n"], q0=q0, Gamma=Gam, gQ=np.zeros((B, 4, N - 1)), gr=None, gn=None, gm=gm)
    for k in INPUTS:
        assert np.array_equal(a[k], b[k]), k
    assert not a["K"][:, :, -1].any() and not a["fbar"][:, :, 0].any() and not a["lbar"][:, :, 0].any()
