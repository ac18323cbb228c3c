"""Both passes of the fused integration at every node count, with every input, through every call path.

Pass 1 eliminates on the FP64 tensor cores in a fixed pivot order (fused16_dmma_kernel<15|0>, tiled_dmma_kernel<4,4,4> /
<2,8,16>) and hands back every rod whose sub-diagonal growth exceeds G (SRI_DMMA_GROWTH, default 4) or whose pivot is zero
or non-finite; pass 2 (fused16_kernel<15|0>, tiled_kernel<16,4> / <32,8>) re-solves the listed rods with row pivoting.
SRI_DMMA_GROWTH=0 hands back every rod with a non-zero sub-diagonal entry (all but straight rods and N = 2),
SRI_FUSED16_IMPL=scalar runs pass 2 alone over the batch.

Stage 1 is checked by its backward error with respect to the system the handle's own tables define (tests/elimination_ref.py):
eta <= C_ETA u per rod, whatever the conditioning, and the forward error against the refined solution x is within what
that backward error allows: ||x^ - x|| = ||C^-1 (C x^ - b)|| <= kappa_inf(C) eta (||x^|| + ||b|| / ||C||), and ||b|| <= ||C|| ||x||,
so ||x^ - x|| / ||x|| <= C_ETA u kappa_inf(C) (1 + ||x^|| / ||x||), about 2 C_ETA u kappa_inf(C) (and <= 1e-12 on generator
rods).  Stages 2-4 are checked entry by entry against the long-double evaluation
from the kernel's own Q (and n, for m), within (M + 4) u |T| |x|.

C_ETA: both passes compute each entry of the eliminated system by at most M rank-one updates of quaternion products (four
FMAs deep) on entries whose growth is bounded (by G = 4 in pass 1, by the pivoting in pass 2), and back-substitute or
normalise with a reciprocal accurate to ~1 u; that bounds eta by a small multiple of 4 u, far from 64 u at every M <= 63.
LAPACK's pivoted solve of the same systems stays below 4.9 u (tests/test_elimination_ref_cpu.py); on a B200 the six
kernels stayed below 14 u over this file (largest: the N <= 64 kernels).
"""
import numpy as np
import pytest

from elimination_ref import (U, Tables, backward_error, cond_inf, q_to_x, refined_solve, stage_bound, stage_excess, stage_m,
                             stage_n, stage_n_dmma16_extra, stage_r, system)

pytestmark = pytest.mark.gpu

C_ETA = 64
SWEEP_B = 97
INSTANTIATIONS = (16, 9, 24, 50)   # fused16 <15>, <0>; tiled <16,4>; tiled <32,8> (and their first-pass twins)
INFO_SENTINEL = -12345
OPTIONAL = ("q0", "r0", "Gamma", "fbar", "lbar", "F_tip", "M_tip")


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    return torch


@pytest.fixture
def handle(monkeypatch, sri_lib):
    """handle(N, **env): a handle created with the given kernel-selection variables set (they are read by sri_create);
    closed at the end of the test."""
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import SpectralRodIntegrator
    made = []

    def make(N, **env):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        h = SpectralRodIntegrator(N, 0)
        for k in env:
            monkeypatch.delenv(k)
        made.append(h)
        return h

    yield make
    for h in made:
        h.close()


def _rods(o, N, B, seed, full=True, first_rod=0):
    """Generator rods; with full=True every optional input too (unit q0, r0, nodal Gamma near e1, fbar, lbar)."""
    rng = np.random.default_rng(seed)
    K, F, Mt, fb = o.generate_rods(0x5EED, first_rod, B)
    if not full:
        return {"K": K}
    q0 = rng.normal(size=(B, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    Gamma = np.concatenate([1 + 0.1 * rng.normal(size=(B, 1, N)), 0.1 * rng.normal(size=(B, 2, N))], axis=1)
    return {"K": K, "F_tip": F, "M_tip": Mt, "q0": q0, "r0": rng.normal(size=(B, 3)), "Gamma": Gamma, "fbar": fb,
            "lbar": rng.normal(size=(B, 3, N))}


def _large_curvature(N, B, seed, scale=300.0):
    """|K| up to ~scale (as in the large-curvature tests of test_gpu_parity.py): pass 1 hands these back."""
    rng = np.random.default_rng(seed)
    lin = np.linspace(1, -1, N)[None, None, :]
    return rng.uniform(-scale, scale, size=(B, 3, 1)) + rng.uniform(-2 * scale / 3, 2 * scale / 3, size=(B, 3, 1)) * lin


def _run(h, torch, a, want=None, quaternions_only=False):
    """One device-buffer call with every output pre-filled with NaN and info with a sentinel (by default every output the
    inputs allow: n and m need F_tip).  Returns numpy arrays and the hand-back count."""
    B, M = a["K"].shape[0], h.M
    if want is None:
        want = ("Q", "r", "n", "m") if a.get("F_tip") is not None else ("Q", "r")
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    shapes = {"Q": (B, 4, M), "r": (B, 3, M), "n": (B, 3, M), "m": (B, 3, M)}
    outs = {k: torch.full(shapes[k], float("nan"), dtype=torch.float64, device="cuda") for k in want}
    info = torch.full((B,), INFO_SENTINEL, dtype=torch.int32, device="cuda")
    if quaternions_only:
        h.integrate_quaternions(t(a["K"]), q0=None if a.get("q0") is None else t(a["q0"]), out=outs["Q"], info=info)
    else:
        h.integrate_all(t(a["K"]), info=info, want=want, **{k: (None if a.get(k) is None else t(a[k])) for k in OPTIONAL},
                        **outs)
    h.synchronize()
    res = {k: v.cpu().numpy() for k, v in outs.items()}
    res["info"] = info.cpu().numpy()
    res["count"] = h.handback_count()
    return res


def _assert_complete(res, ok=None):
    """Every requested element written (finite) and info == 0 on the rods `ok` (all by default)."""
    ok = slice(None) if ok is None else ok
    assert (res["info"][ok] == 0).all(), np.nonzero(res["info"][ok])[0][:8]
    for s in "Qrnm":
        if s in res:
            assert np.isfinite(res[s][ok]).all(), s


def _assert_identical(a, b, what):
    for k in ("Q", "r", "n", "m", "info"):
        if k in a or k in b:
            assert np.array_equal(a[k], b[k]), (what, k)


class Reference:
    """The handle's own system for the rods `a`, solved once with refinement."""

    def __init__(self, h, a, tol=1e-17):
        self.tab = Tables.from_handle(h)
        self.a = a
        self.C, self.b = system(self.tab, a["K"], a.get("q0"))
        self.kappa = cond_inf(self.C)
        # the reference must be far more accurate than the bound it checks: correction <= 1e-4 C_ETA u kappa
        self.x = refined_solve(self.C, self.b, steps=4, tol=np.maximum(tol, 1e-4 * C_ETA * U * self.kappa))

    def check(self, res, label, rods=None, dmma16=False, benchmark=True):
        """Asserts the stage-1 backward and forward error bounds and the componentwise stage 2-4 bounds on `res` (rows
        `rods` of the reference).  dmma16: the rods may have been solved by the N <= 16 tensor-core kernel, whose stress
        operator differs from D_TT^-1 by the float64 table difference.  Returns (max eta / u, max forward error)."""
        sel = np.arange(self.C.shape[0]) if rods is None else np.asarray(rods)
        a = {k: (None if v is None else v[sel]) for k, v in self.a.items()}
        tab, B = self.tab, len(sel)
        xg = q_to_x(res["Q"])
        eta = backward_error(self.C[sel], xg, self.b[sel])
        assert (eta <= C_ETA * U).all(), (float(eta.max() / U), int(sel[eta.argmax()]))
        x = self.x[sel]
        fwd = (np.abs(xg.astype(np.longdouble) - x).max(axis=1) / np.abs(x).max(axis=1)).astype(np.float64)
        fwd_bound = C_ETA * U * self.kappa[sel] * (1.0 + (np.abs(xg).max(axis=1) / np.abs(x).max(axis=1)).astype(np.float64))
        assert (fwd <= fwd_bound).all(), float((fwd / fwd_bound).max())
        if benchmark:
            assert fwd.max() <= 1e-12, float(fwd.max())
        checks = []
        if "r" in res:
            checks.append(("r", res["r"], stage_r(tab, res["Q"], a.get("Gamma"), a.get("r0")), None))
        if "n" in res:
            extra = stage_n_dmma16_extra(tab, B, a.get("F_tip"), a.get("fbar")) if dmma16 else None
            checks.append(("n", res["n"], stage_n(tab, B, a.get("F_tip"), a.get("fbar")), extra))
        if "m" in res:
            checks.append(("m", res["m"], stage_m(tab, res["Q"], res["n"], a.get("q0"), a.get("Gamma"), a.get("lbar"),
                                                  a.get("M_tip")), None))
        for name, got, (val, mag), extra in checks:
            bound = stage_bound(tab, mag) + (0.0 if extra is None else extra.astype(np.float64))
            worst = stage_excess(got, val, bound)
            assert (worst <= 1.0).all(), (name, float(worst.max()), int(sel[worst.argmax()]))
        print(f"[elimination] {self.tab.N} {label}: max eta/u {eta.max() / U:.2f}, max forward error {fwd.max():.2e}")
        return float(eta.max() / U), float(fwd.max())


def _oracle(o, a):
    """The float64 oracle (LU solve) on the rods `a`; absent tip loads are zero."""
    B = a["K"].shape[0]
    tips = {k: (np.zeros((B, 3)) if a.get(k) is None else a[k]) for k in ("F_tip", "M_tip")}
    return o.integrate_all(a["K"], tips["F_tip"], tips["M_tip"], q0=a.get("q0"), r0=a.get("r0"), Gamma=a.get("Gamma"),
                           fbar=a.get("fbar"), lbar=a.get("lbar"), explicit_inverse=False)


def _assert_oracle(ref, res, rods=None):
    """The oracle's result `ref` agrees to 1e-12 per rod and stage, normalised by the rod's largest entry."""
    from conftest import rel_err
    sel = slice(None) if rods is None else rods
    for s in "Qrnm":
        if s in res:
            assert rel_err(res[s][sel], ref[s][sel]) <= 1e-12, s


def _sub(res, rods):
    return {k: (v[rods] if k != "count" else v) for k, v in res.items()}


# ---- every node count, both passes, both input sets --------------------------------------------------------------

@pytest.mark.parametrize("N", range(2, 65))
def test_both_passes_every_node_count(handle, make_oracle, torch_mod, N):
    hd, hb, hs = handle(N), handle(N, SRI_DMMA_GROWTH="0"), handle(N, SRI_FUSED16_IMPL="scalar")
    o = make_oracle(N)
    for full in (True, False):
        a = _rods(o, N, SWEEP_B, seed=N, full=full, first_rod=977 * N)
        ref = Reference(hd, a)
        d, b1, s, b2 = _run(hd, torch_mod, a), _run(hb, torch_mod, a), _run(hs, torch_mod, a), _run(hb, torch_mod, a)
        for res in (d, b1, s):
            _assert_complete(res)
        # G = 0 hands back the rods with a non-zero sub-diagonal entry: all of them, except at N = 2, whose 1 x 1 quaternion
        # system has none, so that pass 1 solves it alone
        handed = SWEEP_B if N > 2 else 0
        assert d["count"] == 0 and b1["count"] == handed and b2["count"] == handed and s["count"] == 0
        _assert_identical(b1, s if N > 2 else d, "G = 0 vs the pass that solves the rods")
        _assert_identical(b1, b2, "G = 0 twice")
        ref.check(d, "default", dmma16=N <= 16)
        ref.check(b1, "G=0", dmma16=N == 2)
        ref.check(s, "pass 2 alone")
        oracle = _oracle(o, a)
        for res in (d, b1, s):
            _assert_oracle(oracle, res)


# ---- partial hand-back: kept and handed-back rods side by side --------------------------------------------------

@pytest.mark.parametrize("N", INSTANTIATIONS)
def test_partial_handback(handle, make_oracle, torch_mod, N):
    """Nearly straight rods (kept by pass 1 at G = 0.01), generator rods and |K| ~ 300 rods (handed back), interleaved.
    The backward-error bound holds for every rod whichever pass solved it; it replaces the conditioning-dependent
    tolerances of the large-curvature tests."""
    B = 201
    o = make_oracle(N)
    a = _rods(o, N, B, seed=100 + N, first_rod=31)
    kind = np.arange(B) % 3
    a["K"][kind == 0] *= 1e-3
    a["K"][kind == 2] = _large_curvature(N, int((kind == 2).sum()), seed=N)
    hp, hs = handle(N, SRI_DMMA_GROWTH="0.01"), handle(N, SRI_FUSED16_IMPL="scalar")
    got, scalar = _run(hp, torch_mod, a), _run(hs, torch_mod, a)
    assert 0 < got["count"] < B, got["count"]
    _assert_complete(got); _assert_complete(scalar)
    ref = Reference(hp, a)
    ref.check(got, "G=0.01 mixed", dmma16=N <= 16, benchmark=False)
    ref.check(scalar, "pass 2 alone, mixed", benchmark=False)
    bench = np.nonzero(kind != 2)[0]
    ref.check(_sub(got, bench), "G=0.01 generator rods", rods=bench, dmma16=N <= 16)
    _assert_oracle(_oracle(o, a), got, rods=bench)


# ---- pass 2 over a list longer than one wave ------------------------------------------------------------------------

# (threads per CTA, rods per CTA) of the pass-2 kernel of each instantiation (sri_api.cu, fused_second_pass)
_PASS2 = {16: (128, 8), 9: (128, 8), 24: (128, 2), 50: (256, 1)}


@pytest.mark.parametrize("N", INSTANTIATIONS)
def test_handback_list_longer_than_one_wave(handle, make_oracle, torch_mod, N):
    """More listed rods than 2 x (resident CTAs at full occupancy) x (rods per CTA): every warp of pass 2 takes at least
    two turns of its grid-stride loop, with the next listed rod's strain samples prefetched."""
    threads, per_cta = _PASS2[N]
    sms = torch_mod.cuda.get_device_properties(0).multi_processor_count
    B = 2 * sms * (2048 // threads) * per_cta + 3
    o = make_oracle(N)
    a = _rods(o, N, B, seed=7 + N, first_rod=5)
    hb, hs = handle(N, SRI_DMMA_GROWTH="0"), handle(N, SRI_FUSED16_IMPL="scalar")
    got, scalar = _run(hb, torch_mod, a), _run(hs, torch_mod, a)
    assert got["count"] == B
    _assert_complete(got)
    _assert_identical(got, scalar, "listed vs pass 2 alone")
    rng = np.random.default_rng(N)
    sample = np.unique(np.concatenate([np.arange(16), np.arange(B - 16, B), rng.choice(B, 64, replace=False)]))
    ref = Reference(hb, {k: v[sample] for k, v in a.items()})
    ref.check(_sub(got, sample), "G=0 grid-stride sample")


# ---- batches smaller than a warp's pair -------------------------------------------------------------------------------

@pytest.mark.parametrize("N", (9, 16))
@pytest.mark.parametrize("B", (1, 2, 3))
def test_tiny_handback_batches(handle, make_oracle, torch_mod, N, B):
    """B = 1, 2, 3 handed back: the half-warp without a rod writes nothing (outputs are views into NaN-filled buffers one
    rod longer; info into a sentinel-filled one)."""
    o = make_oracle(N)
    a = _rods(o, N, B, seed=B, first_rod=11)
    hb, hs = handle(N, SRI_DMMA_GROWTH="0"), handle(N, SRI_FUSED16_IMPL="scalar")
    t = lambda x: torch_mod.from_numpy(np.ascontiguousarray(x)).cuda()
    M = N - 1
    res = {}
    for name, h in (("b", hb), ("s", hs)):
        bufs = {k: torch_mod.full((B + 1, 4 if k == "Q" else 3, M), float("nan"), dtype=torch_mod.float64, device="cuda")
                for k in "Qrnm"}
        info = torch_mod.full((B + 1,), INFO_SENTINEL, dtype=torch_mod.int32, device="cuda")
        h.integrate_all(t(a["K"]), info=info[:B], **{k: t(a[k]) for k in OPTIONAL}, **{k: v[:B] for k, v in bufs.items()})
        h.synchronize()
        r = {k: v.cpu().numpy() for k, v in bufs.items()}
        r["info"] = info.cpu().numpy()
        for k in "Qrnm":
            assert np.isnan(r[k][B]).all(), (name, k)
        assert r["info"][B] == INFO_SENTINEL
        res[name] = {k: v[:B] for k, v in r.items()}
        _assert_complete(res[name])
    assert hb.handback_count() == B
    _assert_identical(res["b"], res["s"], "tiny batch")
    Reference(hb, a).check(res["b"], f"G=0 B={B}")


# ---- non-finite rods among finite ones --------------------------------------------------------------------------------

@pytest.mark.parametrize("N", INSTANTIATIONS)
@pytest.mark.parametrize("growth", (None, "0"))
def test_non_finite_rods_do_not_touch_their_neighbours(handle, make_oracle, torch_mod, N, growth):
    """NaN, Inf and 1e200 strain samples, next to finite rods that share their warp (pairs 2p, 2p+1 of pass 2): the bad
    rods report info != 0 or non-finite outputs, every other rod is bit-identical to the run without the bad rods, and the
    host-buffer call raises SRI_ERR_SINGULAR naming the first rod with a non-zero info."""
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import SriError
    B = SWEEP_B
    o = make_oracle(N)
    a = _rods(o, N, B, seed=3 * N, first_rod=1234)
    h = handle(N) if growth is None else handle(N, SRI_DMMA_GROWTH=growth)
    clean = _run(h, torch_mod, a)
    bad = {10: np.nan, 41: np.inf, 42: 1e200, 77: np.nan}
    abad = dict(a, K=a["K"].copy())
    abad["K"][10, 1, 2] = np.nan
    abad["K"][41, 0, 0] = np.inf
    abad["K"][42] = 1e200
    abad["K"][77, 2, N - 2] = np.nan
    got = _run(h, torch_mod, abad)
    assert got["count"] == (len(bad) if growth is None else B)
    good = np.setdiff1d(np.arange(B), list(bad))
    _assert_identical(_sub(got, good), _sub(clean, good), "neighbours of non-finite rods")
    for b in bad:
        assert got["info"][b] != 0 or not np.isfinite(got["Q"][b]).all(), b
    flagged = np.nonzero(got["info"])[0]
    assert flagged.size > 0
    info = np.full(B, INFO_SENTINEL, dtype=np.int32)
    with pytest.raises(SriError) as exc:
        h.integrate_all(abad["K"], info=info, **{k: abad[k] for k in OPTIONAL})
    assert exc.value.code == -5  # SRI_ERR_SINGULAR
    assert f"first: rod {flagged[0]}," in str(exc.value)
    assert np.array_equal(info, got["info"])


# ---- the call paths that run pass 2 ------------------------------------------------------------------------------------

@pytest.mark.parametrize("N", INSTANTIATIONS)
def test_quaternions_only_and_output_subsets(handle, make_oracle, torch_mod, N):
    o = make_oracle(N)
    a = _rods(o, N, SWEEP_B, seed=N + 5)
    hb, hs = handle(N, SRI_DMMA_GROWTH="0"), handle(N, SRI_FUSED16_IMPL="scalar")
    full = _run(hb, torch_mod, a)
    assert np.array_equal(full["Q"], _run(hs, torch_mod, a)["Q"])
    q = _run(hb, torch_mod, a, want=("Q",), quaternions_only=True)
    assert q["count"] == SWEEP_B
    assert np.array_equal(q["Q"], full["Q"]) and np.array_equal(q["info"], full["info"])
    for want in (("m",), ("r",), ("Q",), ("n", "m")):
        sub = _run(hb, torch_mod, a, want=want)
        for k in want:
            assert np.array_equal(sub[k], full[k]), (want, k)


@pytest.mark.parametrize("N,B", [(16, 8192 + 3 * 65536 + 4097), (40, 512 + 3 * 4096 + 1025)])
def test_host_pipeline_reuses_every_handback_slot(handle, torch_mod, N, B):
    """Host numpy buffers, five pipeline chunks (the three hand-back lists each used, two of them twice), every rod handed
    back: bit-identical to the device-buffer call."""
    hb = handle(N, SRI_DMMA_GROWTH="0")
    t = torch_mod
    K = t.empty((B, 3, N), dtype=t.float64, device="cuda")
    F = t.empty((B, 3), dtype=t.float64, device="cuda"); Mt = t.empty_like(F); fb = t.empty_like(K)
    hb.generate_rods(0x5EED, 99, B, K, F, Mt, fb)
    hb.synchronize()
    rng = np.random.default_rng(N)
    q0 = rng.normal(size=(B, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    a = {"K": K.cpu().numpy(), "F_tip": F.cpu().numpy(), "M_tip": Mt.cpu().numpy(), "fbar": fb.cpu().numpy(), "q0": q0,
         "r0": rng.normal(size=(B, 3)), "Gamma": None, "lbar": 0.1 * rng.normal(size=(B, 3, N))}
    dev = _run(hb, torch_mod, a)
    assert dev["count"] == B
    info = np.full(B, INFO_SENTINEL, dtype=np.int32)
    host = hb.integrate_all(a["K"], info=info, **{k: a[k] for k in OPTIONAL})
    host["info"] = info
    _assert_identical(host, dev, "host pipeline vs device buffers")


def test_multi_device_path_hands_back(handle, make_oracle, torch_mod, monkeypatch):
    """The sharded host path (three shards on device 0) under G = 0: bit-identical to one handle."""
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200 import MultiDeviceIntegrator
    N, B = 16, 20001
    o = make_oracle(N)
    a = _rods(o, N, B, seed=21, first_rod=3)
    one = handle(N, SRI_FUSED16_IMPL="scalar")
    info1 = np.full(B, INFO_SENTINEL, dtype=np.int32)
    want = one.integrate_all(a["K"], info=info1, **{k: a[k] for k in OPTIONAL})
    monkeypatch.setenv("SRI_DMMA_GROWTH", "0")
    with MultiDeviceIntegrator(N, devices=[0, 0, 0]) as mh:
        info = np.full(B, INFO_SENTINEL, dtype=np.int32)
        got = mh.integrate_all(a["K"], info=info, **{k: a[k] for k in OPTIONAL})
    monkeypatch.delenv("SRI_DMMA_GROWTH")
    got["info"], want["info"] = info, info1
    _assert_identical(got, want, "multi-device vs one handle")


# ---- Newton: pass 2 inside the captured iteration graph ----------------------------------------------------------------

def _newton_case(N, B, seed, ne=3):
    """Tip loads and a curved start: G = 0 hands back every rod with a non-zero sub-diagonal entry, and a straight rod
    (qe = 0, the default start) has none, so pass 1 would keep it and the comparison with pass 2 alone would not hold."""
    rng = np.random.default_rng(seed)
    F = np.zeros((B, 3)); F[:, 2] = -rng.uniform(0.1, 2.0, size=B); F[:, 1] = rng.uniform(-0.3, 0.3, size=B)
    Mt = rng.uniform(-0.1, 0.1, size=(B, 3))
    return F, Mt, rng.uniform(-0.05, 0.05, size=(B, 3 * ne))


@pytest.mark.parametrize("N", (16, 9, 24, 40))
def test_newton_through_pass_two(handle, torch_mod, monkeypatch, N):
    """newton_static_shape (finite-difference and analytic Jacobian, graph-captured and eager) and StaticShapeSolver with
    every rod handed back: same iterations, rms history and bit-identical qe as with pass 2 alone."""
    from experimental_gpu_programming_for_a_spectral_numerical_integration_b200.newton import StaticShapeSolver
    B, ne = 301, 3
    F, Mt, qe0 = _newton_case(N, B, N, ne)
    tF, tM = (torch_mod.from_numpy(x).cuda() for x in (F, Mt))
    start = lambda: torch_mod.from_numpy(qe0.copy()).cuda()
    for graph in ("1", "0"):
        monkeypatch.setenv("SRI_NEWTON_GRAPH", graph)
        hb, hs = handle(N, SRI_DMMA_GROWTH="0"), handle(N, SRI_FUSED16_IMPL="scalar")
        for fd in (0.0, 1e-6):
            qb, rb = hb.newton_static_shape(tF, tM, ne, qe=start(), fd_step=fd)
            qs, rs = hs.newton_static_shape(tF, tM, ne, qe=start(), fd_step=fd)
            assert rb["converged"] and rb["iterations"] >= 3, (graph, fd, rb)
            assert rb["iterations"] == rs["iterations"] and rb["rms_history"] == rs["rms_history"], (graph, fd)
            assert torch_mod.equal(qb, qs), (graph, fd)
    monkeypatch.delenv("SRI_NEWTON_GRAPH")
    hb, hs = handle(N, SRI_DMMA_GROWTH="0"), handle(N, SRI_FUSED16_IMPL="scalar")
    qb, rb = StaticShapeSolver(hb, ne=ne).solve(tF, tM, qe0=start())
    qs, rs = StaticShapeSolver(hs, ne=ne).solve(tF, tM, qe0=start())
    assert rb.converged and rb.iterations == rs.iterations and rb.rms_history == rs.rms_history
    assert torch_mod.equal(qb, qs)


def test_newton_static_problem_through_pass_two(handle, torch_mod):
    """sri_newton_static_problem with a rotated clamp and a distributed load, N = 9, every rod handed back."""
    N, B, ne = 9, 257, 3
    F, Mt, qe0 = _newton_case(N, B, 5, ne)
    rng = np.random.default_rng(6)
    q0 = rng.normal(size=(B, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    fbar = np.zeros((B, 3, N)); fbar[:, 2, :] = -rng.uniform(0.1, 1.0, size=(B, 1))
    t = lambda x: torch_mod.from_numpy(x).cuda()
    hb, hs = handle(N, SRI_DMMA_GROWTH="0"), handle(N, SRI_FUSED16_IMPL="scalar")
    qb, rb = hb.newton_static_shape(t(F), t(Mt), ne, qe=t(qe0.copy()), fd_step=0.0, q0=t(q0), fbar=t(fbar))
    qs, rs = hs.newton_static_shape(t(F), t(Mt), ne, qe=t(qe0.copy()), fd_step=0.0, q0=t(q0), fbar=t(fbar))
    assert rb["converged"] and rb["iterations"] == rs["iterations"] and rb["rms_history"] == rs["rms_history"]
    assert torch_mod.equal(qb, qs)
