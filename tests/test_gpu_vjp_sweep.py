"""The reverse-mode kernels at every node count, cotangent, pivot pattern and batch size, against the long-double adjoint
of tests/adjoint_ref.py.

vjp16_kernel<15> (N = 16), vjp16_kernel<0> (N <= 15) and vjp_tiled_kernel (17 <= N <= 64) are given the same float64 Q and
n as the reference.  Every stage gradient (fbar, lbar, F_tip, M_tip, r0, Gamma) is checked entry by entry against
(depth M + C_OPS) u |T| |x|; the K- and q0-gradients, which carry the stage-1 solve, against the forward-error bound of a
solve with backward error C_ETA u (adjoint_ref.py).  A zero bound demands an exact zero: the base node's gK, fbar- and
lbar-gradient at node 0, and every gradient a cotangent cannot reach.  Outputs are pre-filled with NaN and info with a
sentinel, so an unwritten entry fails.

C_ETA = 64 u is the allowance of the forward solve's tests (tests/test_gpu_handback.py), whose kernels measured below 14 u;
the reverse kernels eliminate the same kind of system with the same pivot rules.  Each test prints the largest ratio of
error to bound per kernel, for the solve (gK, gq0) and for the stages.  On a B200 (1000 W power limit) this file measured at
most 0.020 of the gK/gq0 bound (vjp16<0>, generator rods; 0.003 on the |K| ~ 300 rods) and 0.112 of the stage bound.
"""
import numpy as np
import pytest

from adjoint_ref import INPUTS, excess, integrate_all_vjp, pivot_order
from conftest import rel_err
from elimination_ref import Tables

pytestmark = pytest.mark.gpu

INFO_SENTINEL = -12345
COTS = ("gQ", "gr", "gn", "gm")
SOLVE = ("K", "q0")
STAGES = ("lbar", "M_tip", "fbar", "F_tip", "r0", "Gamma")
# the gradients each cotangent reaches (gn: n does not depend on K, Q or Gamma; gm: through b x nu also fbar and F_tip)
REACH = {"gQ": {"K", "q0"}, "gr": {"K", "q0", "r0", "Gamma"}, "gn": {"fbar", "F_tip"},
         "gm": {"K", "q0", "Gamma", "lbar", "M_tip", "fbar", "F_tip"}}
SLOTS = {16: (128, 8), 9: (128, 8), 17: (256, 1), 64: (256, 1)}  # (threads per CTA, rods per CTA), sri_api.cu launch_vjp
_WORST = {}


def _kernel(N):
    return "vjp16<15>" if N == 16 else "vjp16<0>" if N < 16 else "vjp_tiled N<=32" if N <= 32 else "vjp_tiled N>32"


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for (kern, kind), (s, g) in sorted(_WORST.items()):
        print(f"[vjp sweep] {kern:16s} {kind:10s}: gK/gq0 error / bound {s:.3f}, stage gradients error / bound {g:.3f}")


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    return torch


@pytest.fixture
def handle(sri_lib):
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import SpectralRodIntegrator
    made = []

    def make(N):
        made.append(SpectralRodIntegrator(N, 0))
        return made[-1]

    yield make
    for h in made:
        h.close()


def _rods(o, N, B, seed, full=True, first_rod=0):
    """Generator rods (tip loads always, for the forward's n); with full=True every optional input too."""
    rng = np.random.default_rng(seed)
    K, F, Mt, fb = o.generate_rods(0x5EED, first_rod, B)
    a = {"K": K, "F_tip": F, "M_tip": Mt}
    if full:
        q0 = rng.normal(size=(B, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
        Gamma = np.concatenate([1 + 0.1 * rng.normal(size=(B, 1, N)), 0.1 * rng.normal(size=(B, 2, N))], axis=1)
        a.update(q0=q0, r0=rng.normal(size=(B, 3)), Gamma=Gamma, fbar=fb, lbar=rng.normal(size=(B, 3, N)))
    return a


def _large_curvature(N, B, seed, scale=300.0):
    """|K| up to ~scale, in the shape of the forward's large-curvature tests: the pivots move."""
    rng = np.random.default_rng(seed)
    lin = np.linspace(1, -1, N)[None, None, :]
    return rng.uniform(-scale, scale, size=(B, 3, 1)) + rng.uniform(-2 * scale / 3, 2 * scale / 3, size=(B, 3, 1)) * lin


def _cotangents(rng, B, M):
    return {"gQ": rng.normal(size=(B, 4, M)), "gr": rng.normal(size=(B, 3, M)), "gn": rng.normal(size=(B, 3, M)),
            "gm": rng.normal(size=(B, 3, M))}


def _forward(o, a):
    f = o.integrate_all(a["K"], a["F_tip"], a["M_tip"], q0=a.get("q0"), r0=a.get("r0"), Gamma=a.get("Gamma"),
                        fbar=a.get("fbar"), lbar=a.get("lbar"), explicit_inverse=False)
    return f["Q"], f["n"]


def _vjp(h, torch, K, Q, n, q0, Gamma, cot, want=INPUTS):
    """One device-buffer sri_integrate_all_vjp with every output pre-filled with NaN and info with a sentinel.  Inputs are
    numpy arrays or device tensors; returns numpy arrays."""
    B, N = K.shape[0], h.N
    dev = lambda x: None if x is None else (x if torch.is_tensor(x) else torch.from_numpy(np.ascontiguousarray(x)).cuda())
    shapes = {"K": (B, 3, N), "q0": (B, 4), "r0": (B, 3), "Gamma": (B, 3, N), "fbar": (B, 3, N), "lbar": (B, 3, N),
              "F_tip": (B, 3), "M_tip": (B, 3)}
    out = {k: torch.full(shapes[k], float("nan"), dtype=torch.float64, device="cuda") for k in want}
    info = torch.full((B,), INFO_SENTINEL, dtype=torch.int32, device="cuda")
    h.integrate_all_vjp(dev(K), dev(Q), n=dev(n), q0=dev(q0), Gamma=dev(Gamma), **{k: dev(v) for k, v in cot.items()},
                        info=info, want=want, out=out)
    h.synchronize()
    res = {k: v.cpu().numpy() for k, v in out.items()}
    res["info"] = info.cpu().numpy()
    return res


def _check(h, K, Q, n, q0, Gamma, cot, got, kind, rods=None):
    """Asserts info == 0 and every gradient of `got` (rows `rods`, all by default) within its bound; returns the reference."""
    sel = np.arange(K.shape[0]) if rods is None else np.asarray(rods)
    pick = lambda x: None if x is None else np.asarray(x)[sel]
    tab = Tables.from_handle(h)
    ref = integrate_all_vjp(tab, K[sel], pick(Q), pick(n), pick(q0), pick(Gamma), **{k: pick(v) for k, v in cot.items()})
    assert (got["info"][sel] == 0).all(), np.nonzero(got["info"][sel])[0][:8]
    ratio = {k: excess(got[k][sel], ref, k) for k in INPUTS if k in got}
    for k, r in ratio.items():
        assert (r <= 1.0).all(), (h.N, kind, k, float(r.max()), int(sel[r.argmax()]))
    M = h.M
    if "K" in got:
        assert not got["K"][:, :, M].any()             # the base node's strain sample does not enter the forward
    for k in ("fbar", "lbar"):
        if k in got:
            assert not got[k][:, :, 0].any()
    s = max([float(ratio[k].max()) for k in SOLVE if k in ratio] + [0.0])
    g = max([float(ratio[k].max()) for k in STAGES if k in ratio] + [0.0])
    key = (_kernel(h.N), kind)
    w = _WORST.get(key, (0.0, 0.0))
    _WORST[key] = (max(w[0], s), max(w[1], g))
    print(f"[vjp sweep] N={h.N} {kind}: gK/gq0 {s:.3f}, stages {g:.3f} of the bound")
    return ref


# ---- every node count, with all optional inputs and with none ----------------------------------------------------------

@pytest.mark.parametrize("N", range(2, 65))
def test_every_node_count(handle, make_oracle, torch_mod, N):
    from oracle.adjoint import integrate_all_vjp as oracle_vjp
    o, h = make_oracle(N), handle(N)
    B = 37  # odd: the last warp of vjp16 holds one rod
    for full in (True, False):
        a = _rods(o, N, B, seed=N + 1000 * full, full=full, first_rod=313 * N)
        rng = np.random.default_rng(N + 77 * full)
        cot = _cotangents(rng, B, N - 1)
        Q, n = _forward(o, a)
        got = _vjp(h, torch_mod, a["K"], Q, n, a.get("q0"), a.get("Gamma"), cot)
        _check(h, a["K"], Q, n, a.get("q0"), a.get("Gamma"), cot, got, "generator")
        orc = oracle_vjp(o, a["K"], Q, n=n, q0=a.get("q0"), Gamma=a.get("Gamma"), **cot)
        for k in INPUTS:
            assert rel_err(got[k], orc[k]) <= 1e-12, (N, full, k, rel_err(got[k], orc[k]))


# ---- each cotangent alone, and the call without the solve --------------------------------------------------------------

@pytest.mark.parametrize("N", [16, 9, 17, 33, 64])
def test_each_cotangent_alone(handle, make_oracle, torch_mod, N):
    o, h = make_oracle(N), handle(N)
    B = 37
    a = _rods(o, N, B, seed=5 * N, first_rod=11)
    cot = _cotangents(np.random.default_rng(N), B, N - 1)
    Q, n = _forward(o, a)
    q0, Gam = a["q0"], a["Gamma"]
    for c in COTS:
        nc = n if c == "gm" else None  # n is read only with gm
        got = _vjp(h, torch_mod, a["K"], Q, nc, q0, Gam, {c: cot[c]})
        _check(h, a["K"], Q, nc, q0, Gam, {c: cot[c]}, got, "generator")
        assert {k for k in INPUTS if got[k].any()} == REACH[c], c   # the rest exactly zero (the bound demands it too)
    every = _vjp(h, torch_mod, a["K"], Q, n, q0, Gam, cot)
    rest = tuple(k for k in INPUTS if k not in SOLVE)
    nosolve = _vjp(h, torch_mod, a["K"], Q, n, q0, Gam, cot, want=rest)
    assert set(nosolve) == set(rest) | {"info"}
    assert (nosolve["info"] == 0).all()
    for k in rest:
        assert np.array_equal(nosolve[k], every[k]), k


# ---- pivots that move ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("N", [9, 16, 17, 24, 33, 48, 64])
def test_pivots_that_move(handle, make_oracle, torch_mod, N):
    """|K| up to ~300: the transposed operator is far from diagonally dominant and the row search leaves the identity
    order on most rods (shown by a numpy restatement of the kernels' pivot rule on C')."""
    o, h = make_oracle(N), handle(N)
    B = 64
    a = _rods(o, N, B, seed=900 + N, first_rod=3)
    a["K"] = _large_curvature(N, B, seed=N)
    cot = _cotangents(np.random.default_rng(40 + N), B, N - 1)
    Q, n = _forward(o, a)
    got = _vjp(h, torch_mod, a["K"], Q, n, a["q0"], a["Gamma"], cot)
    ref = _check(h, a["K"], Q, n, a["q0"], a["Gamma"], cot, got, "|K|~300")
    perm = pivot_order(ref.C, quantized=N <= 16)
    moved = (perm != np.arange(N - 1)).any(axis=1).mean()
    print(f"[vjp sweep] N={N}: {moved:.0%} of the |K|~300 rods leave the identity pivot order")
    assert moved >= 0.5, moved


# ---- more than two waves: every warp / CTA takes several turns of its grid-stride loop -----------------------------------

@pytest.mark.parametrize("N", [16, 9, 17, 64])
def test_more_than_two_waves(handle, make_oracle, torch_mod, N):
    """More rods than 2 x SMs x (CTAs per SM at the thread limit) x (rods per CTA), which no occupancy can cover in two
    waves, bit-identical to the same rods sent in chunks of SMs x (rods per CTA), which one wave covers at any occupancy."""
    torch = torch_mod
    threads, per_cta = SLOTS[N]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 2 * sms * (2048 // threads) * per_cta + 3
    o, h = make_oracle(N), handle(N)
    a = _rods(o, N, B, seed=N, first_rod=17)
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    fwd = h.integrate_all(t(a["K"]), t(a["F_tip"]), t(a["M_tip"]), q0=t(a["q0"]), r0=t(a["r0"]), Gamma=t(a["Gamma"]),
                          fbar=t(a["fbar"]), lbar=t(a["lbar"]), want=("Q", "n"))
    dK, dQ, dn, dq0, dG = t(a["K"]), fwd["Q"], fwd["n"], t(a["q0"]), t(a["Gamma"])
    cot = _cotangents(np.random.default_rng(N), B, N - 1)
    dcot = {k: t(v) for k, v in cot.items()}
    full = _vjp(h, torch, dK, dQ, dn, dq0, dG, dcot)
    chunk = sms * per_cta
    parts = [_vjp(h, torch, dK[s:s + chunk], dQ[s:s + chunk], dn[s:s + chunk], dq0[s:s + chunk], dG[s:s + chunk],
                  {k: v[s:s + chunk] for k, v in dcot.items()}) for s in range(0, B, chunk)]
    for k in INPUTS + ("info",):
        assert np.array_equal(full[k], np.concatenate([p[k] for p in parts])), k
    rng = np.random.default_rng(N)
    sample = np.unique(np.concatenate([np.arange(16), np.arange(B - 16, B), rng.choice(B, 64, replace=False)]))
    _check(h, a["K"], fwd["Q"].cpu().numpy(), fwd["n"].cpu().numpy(), a["q0"], a["Gamma"], cot, full, "generator",
           rods=sample)


# ---- non-unit quaternions -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("N", [5, 16, 24, 64])
def test_non_unit_quaternions(handle, make_oracle, torch_mod, N):
    """The adjoint is exact for any Q and q0 (R is the un-normalised rotation), so nothing may assume |q| = 1."""
    from oracle.adjoint import integrate_all_vjp as oracle_vjp
    o, h = make_oracle(N), handle(N)
    B, M = 37, N - 1
    rng = np.random.default_rng(60 + N)
    a = _rods(o, N, B, seed=N, first_rod=29)
    Q = rng.normal(size=(B, 4, M)) * rng.uniform(0.2, 3.0, size=(B, 1, M))
    q0 = rng.normal(size=(B, 4)) * 1.7
    n = rng.normal(size=(B, 3, M))
    cot = _cotangents(rng, B, M)
    got = _vjp(h, torch_mod, a["K"], Q, n, q0, a["Gamma"], cot)
    _check(h, a["K"], Q, n, q0, a["Gamma"], cot, got, "non-unit Q")
    orc = oracle_vjp(o, a["K"], Q, n=n, q0=q0, Gamma=a["Gamma"], **cot)
    for k in INPUTS:
        assert rel_err(got[k], orc[k]) <= 1e-12, (k, rel_err(got[k], orc[k]))


# ---- a non-finite rod leaves its neighbours untouched -------------------------------------------------------------------

@pytest.mark.parametrize("N", [16, 9, 17, 64])
def test_non_finite_rod_leaves_neighbours_bit_identical(handle, make_oracle, torch_mod, N):
    """NaN in rod 7 (odd slot: vjp16's half-warp partner is rod 6) and Inf in rod 30 (even slot, partner 31): info reports
    them, and every other rod's gradients and info are bit-identical to the batch without them."""
    o, h = make_oracle(N), handle(N)
    B = 50
    a = _rods(o, N, B, seed=70 + N, first_rod=41)
    cot = _cotangents(np.random.default_rng(N), B, N - 1)
    Q, n = _forward(o, a)
    clean = _vjp(h, torch_mod, a["K"], Q, n, a["q0"], a["Gamma"], cot)
    Kbad = a["K"].copy()
    Kbad[7, 1, 2] = np.nan
    Kbad[30, 0, 0] = np.inf
    bad = _vjp(h, torch_mod, Kbad, Q, n, a["q0"], a["Gamma"], cot)
    assert bad["info"][7] != 0 and bad["info"][30] != 0
    good = np.setdiff1d(np.arange(B), [7, 30])
    for k in INPUTS + ("info",):
        assert np.array_equal(bad[k][good], clean[k][good]), k
    _check(h, a["K"], Q, n, a["q0"], a["Gamma"], cot, clean, "generator")
