"""`import symmer` served by this engine: `install_as_symmer()` registers module objects named like the reference's
packages (`symmer`, `symmer.operators`, `symmer.operators.utils`, `symmer.operators.base`,
`symmer.operators.independent_op`, `symmer.operators.noncontextual_op`, `symmer.projection`, `symmer.evolution[.gate_library|.exponentiation|.circuit_symmerlator]`, `symmer.utils`) whose attributes are the
device-resident classes and functions of `symmer_b200`, so code written against UCL-CCS/symmer — including the
reference's own test files — runs unmodified on the B200 engine. Only what this repository implements is exposed
(INTEGRATION.md §3); anything else raises AttributeError / ImportError as usual.

It refuses to shadow a real `symmer` that is already imported; for patching the array seams of a real install see
`symmer_b200.patch`.
"""
import sys
import types

_NAMES = ["symmer", "symmer.operators", "symmer.operators.utils", "symmer.operators.base",
          "symmer.operators.independent_op", "symmer.operators.noncontextual_op", "symmer.projection",
          "symmer.projection.qubit_tapering", "symmer.projection.base", "symmer.evolution", "symmer.evolution.gate_library",
          "symmer.evolution.exponentiation", "symmer.evolution.circuit_symmerlator", "symmer.utils"]


class _Process:
    """Stand-in for symmer.process (process_handler.py): the engine never forks, every method runs on the device."""
    method = 'single_thread'


def _public(module):
    return {k: v for k, v in vars(module).items() if not k.startswith('__')}


def install_as_symmer():
    """Register the alias modules; returns the top-level `symmer` module object."""
    if "symmer" in sys.modules and not getattr(sys.modules["symmer"], "__symmer_b200_alias__", False):
        raise ImportError("a real `symmer` package is already imported; use symmer_b200.patch.install() instead")
    from . import base, circuit_symmerlator, evolution, independent_op, noncontextual_op, projection, symmer_utils, utils
    mods = {name: types.ModuleType(name) for name in _NAMES}
    for m in mods.values():
        m.__symmer_b200_alias__ = True
    mods["symmer.operators.utils"].__dict__.update(_public(utils))
    mods["symmer.operators.base"].__dict__.update(_public(base))
    mods["symmer.operators.independent_op"].__dict__.update(IndependentOp=independent_op.IndependentOp)
    mods["symmer.operators.noncontextual_op"].__dict__.update(NoncontextualOp=noncontextual_op.NoncontextualOp)
    ops_ns = mods["symmer.operators"].__dict__
    ops_ns.update(_public(utils))
    ops_ns.update(_public(base))
    ops_ns.update(IndependentOp=independent_op.IndependentOp, NoncontextualOp=noncontextual_op.NoncontextualOp)
    mods["symmer.projection"].__dict__.update(QubitTapering=projection.QubitTapering, S3Projection=projection.S3Projection)
    mods["symmer.projection.qubit_tapering"].__dict__.update(QubitTapering=projection.QubitTapering)
    mods["symmer.projection.base"].__dict__.update(S3Projection=projection.S3Projection)
    mods["symmer.evolution"].__dict__.update(trotter=evolution.trotter, exponentiate_single_Pop=evolution.exponentiate_single_Pop,
                                             truncated_exponential=evolution.truncated_exponential)
    mods["symmer.evolution.gate_library"].__dict__.update(_public(evolution))
    mods["symmer.evolution.exponentiation"].__dict__.update(_public(evolution))
    mods["symmer.evolution.circuit_symmerlator"].__dict__.update(CircuitSymmerlator=circuit_symmerlator.CircuitSymmerlator)
    mods["symmer.utils"].__dict__.update(_public(symmer_utils))
    mods["symmer"].__dict__.update(PauliwordOp=base.PauliwordOp, QuantumState=base.QuantumState,
                                   QubitTapering=projection.QubitTapering, process=_Process())
    for name, m in mods.items():
        if "." in name:
            parent, child = name.rsplit(".", 1)
            setattr(mods[parent], child, m)
        if name in ("symmer", "symmer.operators", "symmer.projection", "symmer.evolution"):
            m.__path__ = []                                   # packages: allow `import symmer.operators.utils`
    sys.modules.update(mods)
    return mods["symmer"]


def uninstall():
    for name in _NAMES:
        if getattr(sys.modules.get(name), "__symmer_b200_alias__", False):
            del sys.modules[name]
