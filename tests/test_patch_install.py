"""`symmer_b200.patch.install()` executed against the REAL reference (INTEGRATION.md section 2, the S2 seam): the
names that `symmer/operators/base.py:7-11` and `independent_op.py:6` import from `symmer/operators/utils.py` are
re-bound to this engine, and the reference's own PauliwordOp / IndependentOp then run H*H, adjacency_matrix and
symmetry_generators through them. The reference is not part of this repository: the test runs when
SYMMER_REFERENCE names a source checkout of UCL-CCS/symmer (imported through oracle/shim for its uninstalled
third-party packages) and skips otherwise; the kernels behind the seams are the NumPy test double
(tests/_host_double.py), so this checks the seam and the host logic, not the CUDA code."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
REF = os.environ.get("SYMMER_REFERENCE", "")

SCRIPT = r'''
import json, os, sys, warnings
import numpy as np
warnings.simplefilter("ignore")
ROOT, REF = sys.argv[1], sys.argv[2]
sys.path[:0] = [os.path.join(ROOT, "oracle", "shim"), REF, ROOT, os.path.join(ROOT, "tests")]
import symmer
from symmer import PauliwordOp
from symmer.operators import IndependentOp
import symmer.operators.base as ref_base, symmer.operators.utils as ref_utils, symmer.operators.independent_op as ref_ind

with open(os.path.join(REF, "tests", "hamiltonian_data", "H2O_STO-3G_SINGLET_JW.json")) as f:
    ham = {k: complex(v[0], v[1]) for k, v in json.load(f)["hamiltonian"].items()}

def run():
    H = PauliwordOp.from_dictionary(ham)
    HH = (H * H).sort("lex")
    np.random.seed(5)
    P, Q = PauliwordOp.random(40, 60), PauliwordOp.random(40, 45)
    PQ = (P * Q + P).sort("lex")
    gens = IndependentOp.symmetry_generators(H)
    recon = H.generator_reconstruction(H.generators if hasattr(H, "generators") else gens)
    return dict(hh_s=HH.symp_matrix.copy(), hh_c=HH.coeff_vec.copy(), adj=H.adjacency_matrix.copy(), pq_s=PQ.symp_matrix.copy(),
                pq_c=PQ.coeff_vec.copy(), gen_s=gens.symp_matrix.copy(), gen_c=np.asarray(gens.coeff_vec).copy(),
                comm=P.commutes_termwise(Q).copy(), rec=np.asarray(recon[0]).copy())

before = run()
from _host_double import host_double
from symmer_b200 import patch
originals = {n: getattr(ref_base, n) for n in ("symplectic_cleanup", "matmul_GF2", "cref_binary", "check_independent")}
with host_double():
    done = patch.install()
    assert ("symmer.operators.base", "symplectic_cleanup") in done and ("symmer.operators.utils", "matmul_GF2") in done
    assert ("symmer.operators.independent_op", "_rref_binary") in done
    for n, fn in originals.items():
        assert getattr(ref_base, n) is not fn, n                # re-bound inside base.py's own namespace
    assert ref_base.symplectic_cleanup.__module__.startswith("symmer_b200")
    assert ref_ind._rref_binary.__module__.startswith("symmer_b200")
    assert symmer.process.method == "single_thread"
    calls = {"n": 0}
    import symmer_b200.ops as ops
    real_cleanup, real_commute = ops.cleanup, ops.commute
    def counted_cleanup(*a, **k):
        calls["n"] += 1
        return real_cleanup(*a, **k)
    def counted_commute(*a, **k):
        calls["n"] += 1
        return real_commute(*a, **k)
    ops.cleanup, ops.commute = counted_cleanup, counted_commute
    after = run()
    ops.cleanup, ops.commute = real_cleanup, real_commute
    patch.uninstall()
assert calls["n"] > 5, calls                                     # the engine really was on the path
for n, fn in originals.items():
    assert getattr(ref_base, n) is fn, n                         # uninstall restores the reference's own functions
for k in before:
    a, b = before[k], after[k]
    assert a.shape == b.shape, (k, a.shape, b.shape)
    if a.dtype == bool:
        assert np.array_equal(a, b), k
    else:
        assert np.allclose(a, b, rtol=1e-12, atol=1e-12), k
print("patch ok", len(done), calls["n"])
'''


@pytest.mark.skipif(not os.path.isdir(REF), reason="SYMMER_REFERENCE does not name a UCL-CCS/symmer checkout")
@pytest.mark.timeout(300)
def test_patch_install_runs_the_reference_on_this_engine():
    res = subprocess.run([sys.executable, "-c", SCRIPT, ROOT, REF], capture_output=True, text=True, timeout=280)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert "patch ok" in res.stdout
