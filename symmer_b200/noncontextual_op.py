"""NoncontextualOp with the reference's API (symmer/operators/noncontextual_op.py): the noncontextual part of CS-VQE
and its exact ground-state search on the device.

A noncontextual operator splits into symmetry terms Z (they commute with every term) and cliques 1..N of the other
terms (commutation is an equivalence relation on them; terms of different cliques anticommute). With C_i the first
term of clique i, the group spanned by Z and {P * C_i : P in clique i} is abelian; its independent generators G_1..G_k
(`symmetry_generators`) and the C_i (`clique_operator`) reconstruct every term exactly as

    P_t = s_t * G^{J_t} * C_{i_t}          (no C for a symmetry term, s_t = +-1).

Fixing the generators to nu in {+-1}^k and minimising over the unit vector r of clique weights gives the quasi-quantized
energy E(nu) = a(nu) - ||w(nu)||, and min_nu E(nu) is the lowest eigenvalue of the operator (Kirby & Love). `solve`
enumerates all 2^f assignments of the free generators with one device kernel (`sym_nc_min`: tiled Walsh-Hadamard
transforms of a and of every w_i).
"""
from typing import Optional

import numpy as np
import torch

from . import ops
from .base import PauliwordOp, QuantumState
from .independent_op import IndependentOp, assign_value
from .utils import perform_noncontextual_sweep

# Largest number of free generators `solve` enumerates (2^f assignments): 8.9e10 assignments/s were measured at
# f = 36 with 500 terms and 3 cliques (scripts/bench_noncontextual.py, one B200 at 1000 W), so f = 42 takes ~50 s.
MAX_FREE_GENERATORS = 42

_STRATEGIES = ('diag', 'SingleSweep_magnitude', 'SingleSweep_CurrentOrder')


class NoncontextualOp(PauliwordOp):
    """noncontextual_op.py:16. The operator is cleaned on construction; `symmetry_generators` (IndependentOp of G) and
    `clique_operator` (PauliwordOp of the clique representatives C_i) are built at once, and `solve` sets their
    coefficients to the minimising nu and r and `energy` to E(nu)."""

    def __init__(self, symp_matrix, coeff_vec) -> None:
        self._adopt(PauliwordOp(symp_matrix, coeff_vec).cleanup())

    @classmethod
    def from_PauliwordOp(cls, PwordOp: PauliwordOp) -> "NoncontextualOp":
        self = cls.__new__(cls)
        self._adopt(PwordOp.cleanup())
        return self

    @classmethod
    def from_hamiltonian(cls, H: PauliwordOp, strategy: str = 'diag') -> "NoncontextualOp":
        """A noncontextual sub-Hamiltonian of H: 'diag' keeps the terms without X or Y; 'SingleSweep_magnitude' sweeps
        the terms by decreasing |coefficient| and 'SingleSweep_CurrentOrder' in the given order, keeping every term
        that leaves the kept set noncontextual (`perform_noncontextual_sweep`)."""
        if strategy == 'diag':
            op = H[np.flatnonzero(~np.any(H.X_block, axis=1))]
        elif strategy == 'SingleSweep_magnitude':
            op = perform_noncontextual_sweep(H.sort(by='magnitude'))
        elif strategy == 'SingleSweep_CurrentOrder':
            op = perform_noncontextual_sweep(H)
        else:
            raise ValueError(f'Unrecognised strategy {strategy!r}; supported strategies are {", ".join(_STRATEGIES)}')
        return cls.from_PauliwordOp(op)

    # ------------------------------------------------------------------ decomposition
    def _adopt(self, op: PauliwordOp) -> None:
        self.n_qubits, self.n_terms = op.n_qubits, op.n_terms
        self._xz, self._c = op.device_rows, op.device_coeffs
        self._symp_host = self._c_host = self._c_snapshot = None
        self._cache = {}
        assert self.is_noncontextual, 'Specified operator is contextual.'
        self.energy = None
        self._decompose()

    def _decompose(self) -> None:
        n, M, dev = self.n_qubits, self.n_terms, self._xz.device
        adj = self.adjacency_matrix
        sym = adj.all(axis=1)
        others = np.flatnonzero(~sym)
        # cliques: equal commutation rows among the non-symmetry terms, numbered by first occurrence
        label = np.full(M, -1, dtype=np.int64)
        if others.size:
            _, first, inverse = np.unique(adj[np.ix_(others, others)], axis=0, return_index=True, return_inverse=True)
            rank = np.empty(first.size, dtype=np.int64)
            rank[np.argsort(first)] = np.arange(first.size)
            label[others] = rank[inverse.reshape(-1)]
        N = int(label.max()) + 1 if others.size else 0
        reps = np.array([np.flatnonzero(label == i)[0] for i in range(N)], dtype=np.int64)
        # the abelian group: symmetry terms and P * C_i for the other members of clique i (rows XOR; phases irrelevant)
        members = np.flatnonzero((label >= 0) & ~np.isin(np.arange(M), reps))
        idx = lambda a: torch.as_tensor(np.asarray(a, dtype=np.int64), device=dev)
        span_rows = torch.cat([self._xz.index_select(0, idx(np.flatnonzero(sym))),
                               self._xz.index_select(0, idx(members)) ^ self._xz.index_select(0, idx(reps[label[members]]))])
        G = PauliwordOp._from_device(span_rows.contiguous(), torch.ones(span_rows.shape[0], dtype=torch.complex128, device=dev),
                                     n).generators if span_rows.shape[0] else None
        k = G.n_terms if G is not None else 0
        gen_xz = G.device_rows if k else torch.zeros((0, self._xz.shape[1]), dtype=torch.int64, device=dev)
        rep_xz = self._xz.index_select(0, idx(reps)).contiguous()
        self.symmetry_generators = IndependentOp._from_independent_rows(gen_xz, n)
        self.clique_operator = PauliwordOp._from_device(rep_xz, torch.ones(N, dtype=torch.complex128, device=dev), n)
        # J_t and i_t from the Jordan reconstruction over G followed by C
        if k + N:
            basis = PauliwordOp._from_device(torch.cat([gen_xz, rep_xz]).contiguous(),
                                             torch.ones(k + N, dtype=torch.complex128, device=dev), n)
            recon, ok = self.jordan_generator_reconstruction(basis)
            if not np.all(ok):
                raise RuntimeError('noncontextual reconstruction failed for some terms')
        else:
            recon = np.zeros((M, 0), dtype=int)
        J = recon[:, :k].astype(bool)
        C_part = recon[:, k:].astype(bool)
        if np.any(C_part.sum(axis=1) > 1):
            raise RuntimeError('a term reconstructs with more than one clique representative')
        clique = (np.where(C_part.any(axis=1), C_part.argmax(axis=1), -1) if N else np.full(M, -1)).astype(np.int32)
        Jw = max(1, (k + 63) // 64)
        packed = np.zeros((M, 8 * Jw), dtype=np.uint8)
        packed[:, :(k + 7) // 8] = np.packbits(J, axis=1, bitorder='little')
        signs = ops.nc_signs(self._xz, gen_xz, rep_xz, torch.from_numpy(packed.view(np.int64).copy()).to(dev),
                             torch.from_numpy(clique).to(dev)).cpu().numpy()
        if np.any(signs == 0):
            raise RuntimeError('noncontextual reconstruction gives a term that is not +-s * G^J * C')
        self._J, self._clique, self._signs, self._n_cliques = J, clique, signs, N

    # ------------------------------------------------------------------ energies
    def _real_coeffs(self) -> np.ndarray:
        c = self.coeff_vec
        scale = float(np.max(np.abs(c))) if c.size else 0.0
        if np.any(np.abs(c.imag) > 1e-12 * scale):
            raise ValueError('NoncontextualOp needs real coefficients (a Hermitian operator)')
        return c.real

    def _weights(self, nu: np.ndarray):
        """(a, w) for the assignment nu, every sum over terms in stored order."""
        flips = (self._J.astype(np.int64) @ (np.asarray(nu) < 0).astype(np.int64)) % 2
        v = self._real_coeffs() * self._signs * (1 - 2 * flips)
        a = float(np.sum(v[self._clique < 0]))
        w = np.array([np.sum(v[self._clique == i]) for i in range(self._n_cliques)], dtype=float)
        return a, w

    def get_energy(self, nu) -> float:
        """Quasi-quantized energy a(nu) - ||w(nu)|| of the generator assignment nu in {+-1}^k."""
        nu = np.asarray(nu).real
        assert nu.shape == (self.symmetry_generators.n_terms,) and set(np.unique(nu)).issubset({-1, 1}), \
            'nu must assign +1 or -1 to every symmetry generator'
        a, w = self._weights(nu)
        return a - float(np.sqrt(np.sum(w * w)))

    def solve(self, strategy: str = 'brute_force', ref_state: Optional[QuantumState] = None) -> None:
        """Exact minimum of the quasi-quantized energy over every assignment of the free generators. With `ref_state`
        the generators that `assign_value` gives +-1 on it are fixed to that value; the others stay free. Sets
        `symmetry_generators.coeff_vec` = nu, `clique_operator.coeff_vec` = r and `energy` = get_energy(nu)."""
        if strategy != 'brute_force':
            raise NotImplementedError(f'solver strategy {strategy!r} is not implemented; use brute_force')
        h = self._real_coeffs()
        k, N = self.symmetry_generators.n_terms, self._n_cliques
        fixed = np.zeros(k, dtype=int)
        if ref_state is not None and k:
            if not isinstance(ref_state, QuantumState):
                ref_state = QuantumState(ref_state)
            fixed = np.array(assign_value(self.symmetry_generators, ref_state), dtype=int)
        free = np.flatnonzero(fixed == 0)
        f = int(free.size)
        if f > MAX_FREE_GENERATORS:
            raise ValueError(f'{f} free generators: 2^{f} assignments exceed the brute-force limit of '
                             f'{MAX_FREE_GENERATORS} free generators')
        # fixed generators fold into the coefficients; the kernel enumerates the free bits only
        fold = 1 - 2 * ((self._J[:, fixed < 0].sum(axis=1)) % 2)
        v = h * self._signs * fold
        J_free = np.zeros(self.n_terms, dtype=np.uint64)
        for q, j in enumerate(free):
            J_free |= self._J[:, j].astype(np.uint64) << np.uint64(q)
        dev = self._xz.device
        _, m = ops.nc_min(torch.from_numpy(J_free.view(np.int64)).to(dev), torch.from_numpy(v).to(dev),
                          torch.from_numpy(self._clique).to(dev), N, f)
        nu = fixed.copy()
        nu[free] = 1 - 2 * ((np.int64(m) >> np.arange(f, dtype=np.int64)) & 1)
        _, w = self._weights(nu)
        norm = float(np.sqrt(np.sum(w * w)))
        if N:
            r = -w / norm if norm > 0 else np.eye(N)[0]
            self.clique_operator.coeff_vec = r.astype(complex)
        self.symmetry_generators.coeff_vec = nu.astype(complex)
        self.energy = self.get_energy(nu)
