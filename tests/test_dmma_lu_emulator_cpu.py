"""The lane-exact model of the shipped N <= 16 schedule (tools/dmma_gj_emulator.py: solve_rod_lu): elimination below
the pivot only, -U' kept in shared memory, back-substitution with the solved quaternion as the DMMA A operand.  Pins
its index algebra (tile rows per step, store addresses, back-substitution fragments, shuffle sources and signs)
against the oracle, its growth check against the Gauss-Jordan model's, and its DMMA count."""
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tools"))
import dmma_gj_emulator as emu  # noqa: E402


def _system(o, N):
    S = o.operator(3)
    return emu.tables(S, -S @ o.operator(2), N - 1)


@pytest.mark.parametrize("N", [16, 11, 3])
def test_lu_schedule_matches_oracle(make_oracle, N):
    o = make_oracle(N)
    Stx = _system(o, N)
    K, _, _, _ = o.generate_rods(0x5EED, 42, 5)
    rng = np.random.default_rng(N)
    q0 = rng.normal(size=(5, 4)); q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    ref = o.integrate_all(K, q0=q0, want=("Q",))["Q"]
    for b in range(5):
        Q, flagged = emu.solve_rod_lu(Stx, K[b], q0[b], N - 1, growth=4.0)
        assert not flagged
        assert np.abs(Q.T - ref[b]).max() <= 1e-12 * np.abs(ref[b]).max()


@pytest.mark.parametrize("growth", [4.0, 0.5])
def test_lu_schedule_flags_the_same_rods_as_gauss_jordan(make_oracle, growth):
    """The rows below the pivot see the same operations in both schedules, so the growth check fires on the same rods;
    at G = 4 (the kernel's default) none of this |K| <= 70 sample is handed back, at G = 0.5 most are."""
    o = make_oracle(16)
    Stx = _system(o, 16)
    x = o.chebyshev_points()
    rng = np.random.default_rng(3)
    q0 = np.array([1.0, 0, 0, 0])
    lu, gj = [], []
    for _ in range(20):
        K = rng.uniform(-70, 70, (3, 1)) + rng.uniform(-30, 30, (3, 1)) * (2 * x[None, :] - 1)
        lu.append(emu.solve_rod_lu(Stx, K, q0, 15, growth=growth)[1])
        gj.append(emu.solve_rod(Stx, K, q0, 15, growth=growth)[1])
    assert lu == gj
    assert (sum(lu) == 0) if growth == 4.0 else (sum(lu) > 10)


def test_lu_schedule_issues_166_dmmas_per_rod(make_oracle):
    o = make_oracle(16)
    K, _, _, _ = o.generate_rods(0x5EED, 42, 1)
    stats = {}
    emu.solve_rod_lu(_system(o, 16), K[0], np.array([1.0, 0, 0, 0]), 15, stats=stats)
    assert stats == {"update": 107, "normalise": 23, "backsub": 20}
    assert sum(stats.values()) + emu.STAGE_DMMAS == 166
