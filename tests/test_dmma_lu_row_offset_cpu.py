"""The N = 16 tile layout of the shipped schedule (tools/dmma_gj_emulator.py: solve_rod_lu with row_offset=1, as in
fused16_dmma_kernel<15>): the padding row sits above row 0, so every elimination step updates only the tile rows
that hold live rows.  Moving a row to another tile position changes which lane computes it, not the operands of
any FMA, so Q and the growth check must be bit-for-bit those of the row_offset=0 layout (the emulator's DMMA is a
sequential elementwise FMA chain, hence exact equality)."""
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tools"))
import dmma_gj_emulator as emu  # noqa: E402


def _system(o):
    S = o.operator(3)
    return emu.tables(S, -S @ o.operator(2), 15)


def _both(Stx, K, q0, growth):
    a = emu.solve_rod_lu(Stx, K, q0, 15, growth=growth, row_offset=0)
    b = emu.solve_rod_lu(Stx, K, q0, 15, growth=growth, row_offset=1)
    return a, b


def test_padding_on_top_issues_155_dmmas_per_rod(make_oracle):
    o = make_oracle(16)
    K, _, _, _ = o.generate_rods(0x5EED, 0, 1)
    stats = {}
    emu.solve_rod_lu(_system(o), K[0], np.array([1.0, 0, 0, 0]), 15, stats=stats, row_offset=1)
    assert stats == {"update": 96, "normalise": 23, "backsub": 20}
    assert sum(stats.values()) + emu.STAGE_DMMAS == 155


@pytest.mark.parametrize("random_q0", [False, True])
def test_padding_on_top_is_bit_identical_on_benchmark_rods(make_oracle, random_q0):
    """The benchmark's Philox rods (seed 0x5EED, counter = rod index), with q0 = 1 as in bench.py or random."""
    o = make_oracle(16)
    Stx = _system(o)
    B = 24
    K, _, _, _ = o.generate_rods(0x5EED, 0, B)
    if random_q0:
        q0 = np.random.default_rng(1).normal(size=(B, 4))
        q0 /= np.linalg.norm(q0, axis=1, keepdims=True)
    else:
        q0 = np.tile([1.0, 0, 0, 0], (B, 1))
    ref = o.integrate_all(K, q0=q0, want=("Q",))["Q"]
    for b in range(B):
        (Qa, fa), (Qb, fb) = _both(Stx, K[b], q0[b], 4.0)
        assert np.array_equal(Qa, Qb) and fa == fb
        assert not fb
        assert np.abs(Qb.T - ref[b]).max() <= 1e-12 * np.abs(ref[b]).max()


@pytest.mark.parametrize("growth", [4.0, 0.5])
def test_padding_on_top_flags_the_same_rods(make_oracle, growth):
    """|K| <= 70: none handed back at G = 4 (the kernel's default), most at G = 0.5; flagged rods included, Q and the
    flag match the row_offset=0 layout exactly."""
    o = make_oracle(16)
    Stx = _system(o)
    x = o.chebyshev_points()
    rng = np.random.default_rng(3)
    q0 = np.array([1.0, 0, 0, 0])
    flags = []
    for _ in range(20):
        K = rng.uniform(-70, 70, (3, 1)) + rng.uniform(-30, 30, (3, 1)) * (2 * x[None, :] - 1)
        (Qa, fa), (Qb, fb) = _both(Stx, K, q0, growth)
        assert np.array_equal(Qa, Qb) and fa == fb
        flags.append(fb)
    assert (sum(flags) == 0) if growth == 4.0 else (sum(flags) > 10)
