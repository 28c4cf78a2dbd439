"""NoncontextualOp and its brute-force ground-state kernel (sym_nc_signs, sym_nc_min).

The oracle is the identity min_nu E(nu) = lowest eigenvalue of a noncontextual operator (Kirby & Love): random
noncontextual operators and the noncontextual parts of the bundled Hamiltonians are checked against dense and
matrix-free eigensolvers, and the 24-qubit cases against an independent NumPy fast Walsh-Hadamard minimum written
here. The kernel is also checked on its own against a NumPy direct evaluation on every dispatch edge."""
import ctypes
import sys

import numpy as np
import pytest

NC_LO = 12      # low assignment bits of one kernel tile (noncontextual.cu)


# ------------------------------------------------------------------------------------------ NumPy oracles
def _direct_energies(J, v, clique, N, f):
    """E(m) for every m < 2^f by direct sign evaluation."""
    m = np.arange(1 << f, dtype=np.uint64)
    sign = 1.0 - 2.0 * (np.bitwise_count(m[:, None] & np.asarray(J, dtype=np.uint64)[None, :]) & 1)
    terms = sign * np.asarray(v)[None, :]
    a = terms[:, clique < 0].sum(axis=1)
    w2 = sum(terms[:, clique == i].sum(axis=1) ** 2 for i in range(N)) if N else 0.0
    return a - np.sqrt(w2)


def _fwht(g):
    """In-place fast Walsh-Hadamard transform: F(m) = sum_j g(j) (-1)^{|j & m|}."""
    h = 1
    while h < g.size:
        view = g.reshape(-1, 2, h)
        lo = view[:, 0, :].copy()
        view[:, 0, :] += view[:, 1, :]
        view[:, 1, :] = lo - view[:, 1, :]
        h *= 2
    return g


def _wht_minimum(J, v, clique, N, f):
    J = np.asarray(J, dtype=np.int64)
    a = np.zeros(1 << f)
    np.add.at(a, J[clique < 0], v[clique < 0])
    _fwht(a)
    w2 = np.zeros(1 << f)
    for i in range(N):
        g = np.zeros(1 << f)
        np.add.at(g, J[clique == i], v[clique == i])
        w2 += _fwht(g) ** 2
    return float(np.min(a - np.sqrt(w2)))


def _pack_free(J_bool):
    out = np.zeros(J_bool.shape[0], dtype=np.uint64)
    for q in range(J_bool.shape[1]):
        out |= J_bool[:, q].astype(np.uint64) << np.uint64(q)
    return out


# ------------------------------------------------------------------------------------------ operators
def _random_noncontextual(n, N, n_terms, seed, n_rotations=6):
    """Symmetry terms are Z strings on the first n - ceil(N/2) qubits; clique i multiplies them with the i-th
    Jordan-Wigner string (X_q, Y_q with Z on the qubits before, q past the symmetry qubits), so the cliques pairwise
    anticommute. Random Clifford rotations then hide the structure."""
    from symmer_b200 import PauliwordOp
    rng = np.random.default_rng(seed)
    n_sym = n - (N + 1) // 2
    reps = np.zeros((N, 2 * n), dtype=bool)
    for i in range(N):
        q = n_sym + i // 2
        reps[i, n + n_sym:n + q] = True                      # Z before
        reps[i, q] = True                                    # X ...
        reps[i, n + q] = bool(i % 2)                         # ... or Y
    symp = np.zeros((n_terms, 2 * n), dtype=bool)
    symp[:, n:n + n_sym] = rng.random((n_terms, n_sym)) < 0.4
    clique = rng.integers(-1, N, size=n_terms) if N else np.full(n_terms, -1)
    clique[:N] = np.arange(N)
    symp[clique >= 0] ^= reps[clique[clique >= 0]]
    op = PauliwordOp(symp, rng.normal(size=n_terms))
    rotations = []
    for _ in range(n_rotations):
        row = rng.random(2 * n) < 0.3
        row[rng.integers(2 * n)] = True
        rotations.append((PauliwordOp(row, [1]), None))
    return op.perform_rotations(rotations)


def _ground(op):
    return float(np.linalg.eigvalsh(op.to_sparse_matrix.toarray())[0])


def _scale(op):
    return float(np.sum(np.abs(op.coeff_vec)))


def _hamiltonian(load, tag):
    from symmer_b200 import PauliwordOp
    symp, coeff, d = load(tag)
    return PauliwordOp(symp, coeff), d


# ------------------------------------------------------------------------------------------ the ground state
@pytest.mark.gpu
@pytest.mark.parametrize("N", [0, 2, 3, 5])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_noncontextual_ground_energy(N, seed):
    from symmer_b200 import NoncontextualOp
    n = 5 + seed + (N + 1) // 2
    op = _random_noncontextual(n, N, 40 + 10 * seed, seed)
    nc = NoncontextualOp.from_PauliwordOp(op)
    assert nc.clique_operator.n_terms == N
    nc.solve()
    assert abs(nc.energy - _ground(nc)) <= 1e-10 * _scale(nc)
    assert nc.energy == nc.get_energy(nc.symmetry_generators.coeff_vec.real)


@pytest.mark.gpu
@pytest.mark.parametrize("strategy", ["diag", "SingleSweep_magnitude"])
def test_be_matches_dense_eigensolver(strategy, hamiltonians):
    from symmer_b200 import NoncontextualOp
    H, _ = _hamiltonian(hamiltonians, "Be_STO3G")
    nc = NoncontextualOp.from_hamiltonian(H, strategy=strategy)
    nc.solve()
    assert abs(nc.energy - _ground(nc)) <= 1e-10 * _scale(nc)
    r = nc.clique_operator.coeff_vec
    assert r.size == 0 or abs(np.linalg.norm(r) - 1) < 1e-12


@pytest.mark.gpu
def test_nh3_sweep_matches_matrix_free_eigensolver(hamiltonians):
    from symmer_b200 import NoncontextualOp, exact_gs_energy
    H, _ = _hamiltonian(hamiltonians, "NH3_STO3G")
    nc = NoncontextualOp.from_hamiltonian(H, strategy="SingleSweep_magnitude")
    nc.solve()
    e0, _ = exact_gs_energy(nc)
    assert abs(nc.energy - e0) <= 1e-8 * _scale(nc)


@pytest.mark.gpu
@pytest.mark.parametrize("strategy,f", [("diag", 24), ("SingleSweep_magnitude", 23)])
def test_hooh_matches_numpy_walsh_hadamard_minimum(strategy, f, hamiltonians):
    from symmer_b200 import NoncontextualOp
    H, _ = _hamiltonian(hamiltonians, "HOOH_STO3G")
    nc = NoncontextualOp.from_hamiltonian(H, strategy=strategy)
    assert nc.symmetry_generators.n_terms == f
    nc.solve()
    v = nc.coeff_vec.real * nc._signs
    ref = _wht_minimum(_pack_free(nc._J), v, nc._clique, nc.clique_operator.n_terms, f)
    assert abs(nc.energy - ref) <= 1e-10 * _scale(nc)
    nu, energy = nc.symmetry_generators.coeff_vec.copy(), nc.energy
    nc.solve()                                          # deterministic: same bits twice
    assert np.array_equal(nu, nc.symmetry_generators.coeff_vec) and energy == nc.energy


@pytest.mark.gpu
def test_current_order_sweep(hamiltonians):
    from symmer_b200 import NoncontextualOp
    from symmer_b200.utils import perform_noncontextual_sweep
    H, _ = _hamiltonian(hamiltonians, "Be_STO3G")
    nc = NoncontextualOp.from_hamiltonian(H, strategy="SingleSweep_CurrentOrder")
    assert nc == perform_noncontextual_sweep(H)
    nc.solve()
    assert abs(nc.energy - _ground(nc)) <= 1e-10 * _scale(nc)


# ------------------------------------------------------------------------------------------ decomposition
def _check_decomposition(nc):
    from symmer_b200 import PauliwordOp
    from symmer_b200.utils import check_independent
    G, C = nc.symmetry_generators, nc.clique_operator
    n = nc.n_qubits
    if G.n_terms:
        assert check_independent(G) and np.all(G.adjacency_matrix)
    if C.n_terms:
        assert np.array_equal(C.adjacency_matrix, np.eye(C.n_terms, dtype=bool))
        if G.n_terms:
            assert np.all(C.commutes_termwise(G))
    for t in range(nc.n_terms):
        prod = PauliwordOp(np.zeros(2 * n, dtype=bool), [1])
        for j in np.flatnonzero(nc._J[t]):
            prod = prod * PauliwordOp(G.symp_matrix[j], [1])
        if nc._clique[t] >= 0:
            prod = prod * PauliwordOp(C.symp_matrix[nc._clique[t]], [1])
        assert np.array_equal(prod.symp_matrix[0], nc.symp_matrix[t])
        assert prod.coeff_vec[0] == nc._signs[t]


@pytest.mark.gpu
def test_decomposition_invariants(hamiltonians):
    from symmer_b200 import NoncontextualOp
    H, _ = _hamiltonian(hamiltonians, "Be_STO3G")
    _check_decomposition(NoncontextualOp.from_hamiltonian(H, strategy="SingleSweep_magnitude"))
    _check_decomposition(NoncontextualOp.from_PauliwordOp(_random_noncontextual(9, 3, 50, 7)))


# ------------------------------------------------------------------------------------------ reference state
@pytest.mark.gpu
def test_reference_state_fixes_generators(hamiltonians):
    from symmer_b200 import NoncontextualOp, QuantumState
    from symmer_b200.independent_op import assign_value
    H, d = _hamiltonian(hamiltonians, "Be_STO3G")
    nc = NoncontextualOp.from_hamiltonian(H, strategy="SingleSweep_magnitude")
    hf = QuantumState(d["hf_array"].astype(int))
    fixed = np.array(assign_value(nc.symmetry_generators, hf))
    assert np.any(fixed != 0)
    nc.solve(ref_state=hf)
    nu = nc.symmetry_generators.coeff_vec.real.astype(int)
    assert np.array_equal(nu[fixed != 0], fixed[fixed != 0])
    free = np.flatnonzero(fixed == 0)
    best = np.inf
    for m in range(1 << free.size):
        trial = fixed.copy()
        trial[free] = 1 - 2 * ((m >> np.arange(free.size)) & 1)
        best = min(best, nc.get_energy(trial))
    assert abs(nc.energy - best) <= 1e-12 * _scale(nc)
    nc.solve()
    assert nc.energy <= best + 1e-12 * _scale(nc)


# ------------------------------------------------------------------------------------------ kernel edges
@pytest.mark.gpu
@pytest.mark.parametrize("f", [0, 1, NC_LO - 1, NC_LO, NC_LO + 1, NC_LO + 3])
@pytest.mark.parametrize("N", [0, 3])
def test_kernel_against_direct_evaluation(f, N):
    import torch
    from symmer_b200 import ops
    rng = np.random.default_rng(100 * f + N)
    M = 60
    J = rng.integers(0, 1 << max(f, 1), size=M, dtype=np.uint64) if f else np.zeros(M, dtype=np.uint64)
    v = rng.normal(size=M)
    clique = rng.integers(-1, N, size=M).astype(np.int32) if N else np.full(M, -1, dtype=np.int32)
    dev = ops.device()
    args = (torch.from_numpy(J.view(np.int64)).to(dev), torch.from_numpy(v).to(dev), torch.from_numpy(clique).to(dev), N, f)
    e, m = ops.nc_min(*args)
    E = _direct_energies(J, v, clique, N, f)
    assert 0 <= m < (1 << f) or (f == 0 and m == 0)
    assert abs(e - E.min()) <= 1e-12 * np.abs(v).sum()
    assert abs(E[m] - E.min()) <= 1e-12 * np.abs(v).sum()
    assert ops.nc_min(*args) == (e, m)


@pytest.mark.gpu
def test_small_operators():
    from symmer_b200 import NoncontextualOp, PauliwordOp
    single = NoncontextualOp.from_PauliwordOp(PauliwordOp.from_list(["XZY"], [0.7]))
    single.solve()
    assert single.symmetry_generators.n_terms == 1 and single.energy == -0.7
    ident = NoncontextualOp.from_PauliwordOp(PauliwordOp.from_list(["III"], [1.3]))
    ident.solve()
    assert ident.symmetry_generators.n_terms == 0 and ident.energy == 1.3
    diag = NoncontextualOp.from_PauliwordOp(PauliwordOp.from_list(["ZZI", "IZZ", "ZIZ", "ZII"], [1, 0.5, -0.25, 0.3]))
    diag.solve()
    assert diag.clique_operator.n_terms == 0 and abs(diag.energy - _ground(diag)) < 1e-12


# ------------------------------------------------------------------------------------------ errors
@pytest.mark.gpu
def test_errors():
    from symmer_b200 import NoncontextualOp, PauliwordOp
    from symmer_b200.noncontextual_op import MAX_FREE_GENERATORS
    with pytest.raises(AssertionError, match="Specified operator is contextual."):
        NoncontextualOp.from_PauliwordOp(PauliwordOp.from_list(["IX", "IZ", "XI", "ZI", "XX", "ZZ"], np.ones(6)))
    cplx = NoncontextualOp.from_PauliwordOp(PauliwordOp.from_list(["ZI", "XZ"], [1, 0.5j]))
    with pytest.raises(ValueError, match="real coefficients"):
        cplx.solve()
    n = MAX_FREE_GENERATORS + 1
    big = NoncontextualOp(np.hstack([np.zeros((n, n), dtype=bool), np.eye(n, dtype=bool)]), np.linspace(1, 2, n))
    with pytest.raises(ValueError, match="brute-force limit"):
        big.solve()
    with pytest.raises(NotImplementedError):
        big.solve(strategy="binary_relaxation")
    with pytest.raises(ValueError, match="SingleSweep_magnitude"):
        NoncontextualOp.from_hamiltonian(big, strategy="DFS_magnitude")


# ------------------------------------------------------------------------------------------ without a GPU
def test_abi_rejects_bad_sizes():
    from symmer_b200 import _cabi
    lib = _cabi.load()
    assert lib.sym_nc_signs(None, -1, 1, None, 0, None, 0, None, 1, None, None, None) == -1
    assert lib.sym_nc_signs(None, 4, 0, None, 0, None, 0, None, 1, None, None, None) == -1
    assert lib.sym_nc_signs(None, 4, 1, None, 65, None, 0, None, 1, None, None, None) == -1
    assert lib.sym_nc_min_ws_bytes(500, 3) > 0 and lib.sym_nc_min_ws_bytes(500, 5000) == 0
    best = ctypes.create_string_buffer(16)
    for M, N, f in [(-1, 0, 4), (10, -1, 4), (10, 5000, 4), (10, 2, -1), (10, 2, 63)]:
        assert lib.sym_nc_min(None, None, None, M, N, f, best, None, None, 0, None) == -1, (M, N, f)
    assert lib.sym_nc_min(None, None, None, 10, 2, 4, None, None, None, 0, None) == -1
    assert lib.sym_nc_min(None, None, None, 10, 2, 4, best, None, None, 0, None) == -3


def test_compat_exports_noncontextual_op():
    from symmer_b200 import compat
    import symmer_b200
    assert "symmer" not in sys.modules
    compat.install_as_symmer()
    try:
        from symmer.operators import NoncontextualOp
        from symmer.operators.noncontextual_op import NoncontextualOp as nc_from_module
        assert NoncontextualOp is nc_from_module is symmer_b200.NoncontextualOp
    finally:
        compat.uninstall()
