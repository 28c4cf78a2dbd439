"""symmer_b200 — B200-native (sm_100a) engine for symmer's symplectic Pauli algebra.

Drop-in for the hot path behind UCL-CCS/symmer's PauliwordOp / QuantumState / IndependentOp API.
Operators live in CUDA memory as bit-packed uint64 X|Z rows + complex128 coefficients (PyTorch
owns the memory) and every kernel is reached through the C ABI of include/symmer_b200.h.
"""
from . import _cabi  # noqa: F401  (raises if the CUDA library is missing and cannot be built)

__all__ = ["PauliwordOp", "QuantumState", "IndependentOp", "QubitTapering", "S3Projection", "single_term_expval",
           "get_PauliwordOp_projector", "get_ij_operator", "change_of_basis_XY_to_Z", "CircuitSymmerlator",
           "exact_gs_energy", "trotter", "NoncontextualOp"]
_BASE_NAMES = ("PauliwordOp", "QuantumState", "single_term_expval", "get_PauliwordOp_projector", "get_ij_operator",
               "change_of_basis_XY_to_Z")


def __getattr__(name):
    if name in _BASE_NAMES:
        from . import base
        return getattr(base, name)
    if name == "IndependentOp":
        from .independent_op import IndependentOp
        return IndependentOp
    if name == "NoncontextualOp":
        from .noncontextual_op import NoncontextualOp
        return NoncontextualOp
    if name in ("QubitTapering", "S3Projection"):
        from . import projection
        return getattr(projection, name)
    if name == "CircuitSymmerlator":
        from .circuit_symmerlator import CircuitSymmerlator
        return CircuitSymmerlator
    if name in ("exact_gs_energy", "trotter"):
        from . import evolution, symmer_utils
        return getattr(symmer_utils if name == "exact_gs_energy" else evolution, name)
    raise AttributeError(name)
