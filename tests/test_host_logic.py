"""Host logic of the reference-facing classes on the CPU box: the kernels behind `symmer_b200.ops` are swapped for
the NumPy test double of tests/_host_double.py (test infrastructure; the product itself has no CPU path), and
the same golden-vector cases that `-m gpu` runs against the CUDA kernels are run here."""
import numpy as np
import pytest

from _host_double import host_double
from api_cases import CASES, load_api_golden


@pytest.fixture(scope="module")
def api_golden():
    return load_api_golden()


@pytest.fixture()
def host_ops():
    with host_double():
        yield


@pytest.mark.parametrize("case", CASES, ids=lambda f: f.__name__)
def test_api_case_on_host_double(case, api_golden, host_ops):
    import symmer_b200
    case(symmer_b200, api_golden)


def test_double_is_gone_after_the_block():
    import torch
    from symmer_b200 import ops
    real_device = ops.device
    with host_double():
        assert ops.device().type == "cpu"
    assert ops.device is real_device
    if torch.cuda.is_available():
        assert ops.device().type == "cuda"
    else:
        with pytest.raises(RuntimeError):
            ops.device()                  # no CUDA device: the product path refuses to run


def test_double_matches_the_oracle_on_core_paths(golden, host_ops):
    """The double itself is held to the reference vectors through the host classes (multiply, cleanup, commute,
    rotations, GF(2)), so a host-logic failure above cannot hide behind a wrong stand-in."""
    from oracle import pauli_oracle as po
    from symmer_b200 import PauliwordOp
    from symmer_b200.utils import rref_binary
    seen = 0
    for name, g in golden.items():
        if name.startswith("mul_") and "a_symp" in g and "out_symp" in g:
            A, B = PauliwordOp(g["a_symp"], g["a_coeff"]), PauliwordOp(g["b_symp"], g["b_coeff"])
            C = A * B
            ok, why = po.compare_term_sets(C.symp_matrix, C.coeff_vec, g["out_symp"], g["out_coeff"])
            assert ok, (name, why)
            seen += 1
        if seen >= 12:
            break
    assert seen >= 9
    P = PauliwordOp.from_list(["XXX", "YYY", "XXX", "YYY"], [1, 1, -1, 1]).cleanup()
    assert P.n_terms == 1 and P.to_dictionary == {"YYY": 2}
    m = np.array([[1, 1, 0], [0, 1, 1], [1, 0, 1]], dtype=bool)
    assert np.array_equal(rref_binary(m), po.rref_binary(m))


def test_compat_serves_import_symmer(host_ops):
    """`symmer_b200.compat.install_as_symmer()`: code written against the reference's package names runs on this
    engine (scripts/run_reference_tests.py drives the reference's own test files through the same alias)."""
    import sys
    from symmer_b200 import compat
    assert "symmer" not in sys.modules
    compat.install_as_symmer()
    try:
        from symmer import PauliwordOp, QuantumState, QubitTapering, process
        from symmer.operators import IndependentOp, single_term_expval
        from symmer.operators.utils import check_independent, symplectic_cleanup
        from symmer.evolution import trotter
        from symmer.evolution.gate_library import Had, CX
        from symmer.evolution.circuit_symmerlator import CircuitSymmerlator
        from symmer.utils import exact_gs_energy, tensor_list
        import symmer.operators.utils as ref_utils
        import symmer_b200
        assert PauliwordOp is symmer_b200.PauliwordOp and process.method == 'single_thread'
        assert ref_utils.check_independent is check_independent
        H = PauliwordOp.from_list(['XX', 'ZZ'], [1, 1])
        assert (H * H).to_dictionary == {'II': 2, 'YY': -2}
        assert check_independent(IndependentOp.from_list(['ZI', 'IZ']))
        assert np.isclose(exact_gs_energy(H.to_sparse_matrix)[0], -2)
        assert CX(2, 0, 1).n_terms == 4 and Had(1, 0).n_terms == 2 and callable(trotter) and callable(tensor_list)
        assert isinstance(QuantumState.zero(2), QuantumState) and callable(single_term_expval) and callable(symplectic_cleanup)
        assert CircuitSymmerlator(2).n_qubits == 2 and QubitTapering.__name__ == 'QubitTapering'
    finally:
        compat.uninstall()
    assert "symmer" not in sys.modules and "symmer.operators.utils" not in sys.modules


def test_replay_of_the_reference_on_host_double(host_ops):
    """tests/replay_cases.py: the API script recorded on the REAL reference, replayed on this engine (host logic here;
    tests/test_gpu_replay.py replays it on the CUDA kernels)."""
    import os
    import types
    import replay_cases
    import symmer_b200
    stored = dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "replay_vectors.npz")))
    api = types.SimpleNamespace(PauliwordOp=symmer_b200.PauliwordOp, QuantumState=symmer_b200.QuantumState,
                                IndependentOp=symmer_b200.IndependentOp, QubitTapering=symmer_b200.QubitTapering)
    check = replay_cases.Checker(stored)
    replay_cases.run(api, check)
    assert check.checked == sum(1 for k in stored if k.endswith("/kind") and not k.endswith("stab_input/kind"))
    assert check.checked > 700
