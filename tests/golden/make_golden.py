"""Regenerates the committed golden fixtures.  Run in the build container (needs /root/reference):

    python tests/golden/make_golden.py

reference_main_default.json  -- output of the reference's own main() (compiled verbatim against oracle/eigen_shim),
                                at its native 6 significant digits and at 17.
oracle_default_stages34.json -- stages 3-4 for the same rod (F_tip=(0,0,-1), M_tip=0); the reference does not
                                implement them, so this file is produced by the oracle and pinned by the analytic
                                known-answer tests in tests/test_oracle_cpu.py.
reference_random_rods.npz    -- 512 rods of the benchmark's Philox stream (seed 0x5EED, rods 0..511) through the reference's
                                OWN integrateQuaternions() / integratePosition() (oracle/reference_harness.cpp #includes
                                the reference's main.cpp): qe [512][9], the reference's strain samples K [512][3][16],
                                Q [512][4][15], r [512][3][15], and A_NN of updateA (main.cpp:55-88) for rods 0..3; exact FP64
                                (512 rods keep the file under 1 MB).
"""
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle.build_reference import run_reference  # noqa: E402
from oracle.oracle import Oracle, build_oracle  # noqa: E402

HERE = Path(__file__).resolve().parent
QE = [0, 0, 0, 1.2877691307032, -1.63807499160786, 0.437406679142598, 0, 0, 0]

full = run_reference(17)
native = run_reference(None)
(HERE / "reference_main_default.json").write_text(json.dumps({
    "source": "/root/reference/main.cpp compiled verbatim against oracle/eigen_shim; qe of main.cpp:187-195; N=16",
    "qe": QE,
    "stdout_native_precision": native["stdout"],
    "Q_stack": [repr(float(v)) for v in full["Q_stack"]],
    "r_stack_rows": [[repr(float(v)) for v in row] for row in full["r_stack"]],
}, indent=1))

build_oracle()
o = Oracle(16)
K = o.strain_from_modes(np.array(QE, dtype=np.float64))
F = np.array([[0.0, 0.0, -1.0]]); Mt = np.zeros((1, 3))
out = o.integrate_all(K, F, Mt)
(HERE / "oracle_default_stages34.json").write_text(json.dumps({
    "source": "oracle/sri_oracle.c (SURVEY Appendix A.4-A.5); qe of main.cpp:187-195; F_tip=(0,0,-1), M_tip=0; N=16",
    "K": [[repr(float(v)) for v in row] for row in K[0]],
    "n": [[repr(float(v)) for v in row] for row in out["n"][0]],
    "m": [[repr(float(v)) for v in row] for row in out["m"][0]],
}, indent=1))
from oracle.build_reference import ReferenceHarness  # noqa: E402

NR = 512
qe = o.generate_modes(0x5EED, 0, NR)
harness = ReferenceHarness()
ref = harness.integrate(qe)
A = np.stack([harness.update_A(qe[b]) for b in range(4)])
np.savez_compressed(HERE / "reference_random_rods.npz", qe=qe, K=ref["K"], Q=ref["Q"], r=ref["r"], A_NN=A,
                    seed=np.uint64(0x5EED), first_rod=np.int64(0))
print("golden fixtures written to", HERE)
