"""Exact tests of the matrix-free kernels of symmer_b200/csrc/spmv.cu (sym_apply, sym_expval, the symmetric
expectation-value table of sym_expval_prepare_sym, sym_to_csr) and of their dispatch in symmer_b200.ops.

Every kernel here forms signed sums of c'_t * psi[r ^ x_t] in FP64 and flips signs on the sign bit. With small
Gaussian-integer coefficients and amplitudes every product and partial sum is an integer below 2^53, so the device
result is exact whatever the summation order (the atomic adds included) and must equal an int64 reference bit for
bit: one term dropped, doubled or given the wrong sign anywhere fails, which a float tolerance would not catch."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import pauli_oracle as po

gpu = pytest.mark.gpu

TILE = 512              # APPLY_TERMS: terms per shared-memory tile of the kernels
SPAN = 2048             # rows per CTA of the 16-row (real) and 8-row (complex) kernels; symmetric-mode alignment
SYM_MIN_BIT = 11        # symmetric mode: groups whose x has its top bit h >= 11 run on one half of the rows
LEN_CAP = 0xffff        # symmetric table: group length field (a longer group is skipped in several hops)
WIN = 14                # row window of the 64-bit sign tests
CMAX = 3                # |Re c'|, |Im c'| <= CMAX
PMAX = 3                # |Re psi|, |Im psi| <= PMAX
PARTIAL0 = (7.0, -3.0)  # sym_expval adds into partial: it starts from this pair
GUARD = 37              # elements after y that sym_apply must leave alone


# ------------------------------------------------------------------------------------------- exact reference
def parity(v):
    v = np.array(v, dtype=np.int64).view(np.uint64)
    for s in (32, 16, 8, 4, 2, 1):
        v = v ^ (v >> np.uint64(s))
    return (v & np.uint64(1)).astype(np.int64)


def top_bit(x):
    """Index of the highest set bit of each x (-1 for x = 0)."""
    x = np.asarray(x, dtype=np.int64)
    h = np.full(x.shape, -1, dtype=np.int64)
    for b in range(63):
        h[((x >> b) & 1) == 1] = b
    return h


def mix64(x):
    """murmur3 fmix64 (common.cuh)."""
    x = np.array(x, dtype=np.uint64)
    x ^= x >> np.uint64(33)
    x *= np.uint64(0xff51afd7ed558ccd)
    x ^= x >> np.uint64(33)
    x *= np.uint64(0xc4ceb9fe1a85ec53)
    x ^= x >> np.uint64(33)
    return x


def sym_side(x):
    """The half of the rows (bit h clear or set) that evaluates the group with mask x in symmetric mode."""
    return ((mix64(x) >> np.uint64(17)) & np.uint64(1)).astype(np.int64)


def x_with_side(h, side):
    """The smallest x > 2^h with top bit h whose group is evaluated by the given half of the rows."""
    x = np.arange((1 << h) + 1, 1 << (h + 1), dtype=np.int64)
    return int(x[sym_side(x) == side][0])


def check_exact(rows, M, cr, ci, pr, pi, sym=False):
    """Every partial sum the kernels form stays an integer below 2^53 (symmetric mode doubles c')."""
    cmax = max([1] + [int(np.abs(a).max()) for a in (cr, ci) if a.size])
    pmax = max([1] + [int(np.abs(a).max()) for a in (pr, pi) if a.size])
    assert rows * max(M, 1) * cmax * pmax ** 2 * 8 * (2 if sym else 1) < 2 ** 53, "inputs outside the exact range"


def wht_(w):
    """In place, along axis 1: w[g, r] <- sum_z w[g, z] (-1)^popcount(r & z) (unnormalised, natural order, int64)."""
    G, side = w.shape
    h = 1
    while h < side:
        v = w.reshape(G, side // (2 * h), 2, h)
        a = v[:, :, 0, :].copy()
        b = v[:, :, 1, :]
        v[:, :, 0, :] += b
        np.subtract(a, b, out=b)
        h *= 2


def exact_apply(n, xm, zm, cr, ci, pr, pi, sym=False):
    """y[r] = sum_t c'_t (-1)^popcount(r & z_t) psi[r ^ x_t] over all 2^n rows, as int64 (yr, yi).

    Terms are grouped by x; a group's coefficients are scattered at their z (repeated (x, z) pairs add up) and one
    Walsh-Hadamard transform gives its row weights w_g(r), which multiply psi[r ^ x_g] as Gaussian integers.
    sym=True restates the symmetric expectation-value mode instead: a group whose x has its top bit h >= 11
    contributes with doubled weights on the rows whose bit h equals the group's side bit, and not at all on the
    others."""
    side = 1 << n
    xm, zm = np.asarray(xm, np.int64), np.asarray(zm, np.int64)
    cr, ci = np.asarray(cr, np.int64), np.asarray(ci, np.int64)
    check_exact(side, xm.size, cr, ci, pr, pi, sym)
    assert pr.size == side and pi.size == side
    yr = np.zeros(side, np.int64)
    yi = np.zeros(side, np.int64)
    if xm.size == 0:
        return yr, yi
    assert 0 <= zm.min() and zm.max() < side and 0 <= xm.min() and xm.max() < side
    ux, g = np.unique(xm, return_inverse=True)
    rows = np.arange(side, dtype=np.int64)
    chunk = max(1, (1 << 21) // side)
    has_im = bool(ci.any())
    for g0 in range(0, ux.size, chunk):
        xs = ux[g0:g0 + chunk]
        sel = (g >= g0) & (g < g0 + xs.size)
        wr = np.zeros((xs.size, side), np.int64)
        np.add.at(wr, (g[sel] - g0, zm[sel]), cr[sel])
        wht_(wr)
        wi = np.zeros_like(wr)
        if has_im:
            np.add.at(wi, (g[sel] - g0, zm[sel]), ci[sel])
            wht_(wi)
        if sym:
            h = top_bit(xs)
            own = ((rows[None, :] >> np.maximum(h, 0)[:, None]) & 1) == sym_side(xs)[:, None]
            mult = np.where((h >= SYM_MIN_BIT)[:, None], 2 * own, 1)
            wr *= mult
            wi *= mult
        cols = rows[None, :] ^ xs[:, None]
        qr, qi = pr[cols], pi[cols]
        yr += (wr * qr - wi * qi).sum(axis=0)
        yi += (wr * qi + wi * qr).sum(axis=0)
    return yr, yi


def exact_expval(pr, pi, y, lo=0, hi=None):
    """sum_{lo <= r < hi} conj(psi[r]) * y[r] as a pair of Python ints."""
    yr, yi = y
    hi = pr.size if hi is None else hi
    a, b, c, d = pr[lo:hi], pi[lo:hi], yr[lo:hi], yi[lo:hi]
    return int((a * c + b * d).sum()), int((a * d - b * c).sum())


def exact_apply_window(B, wbits, xm, zm, cr, ci, pr, pi, sym=False):
    """Rows [B, B + 2^wbits) of exact_apply from that window of psi alone, for terms with x < 2^wbits and B a
    multiple of 2^wbits: row r = B | l has the sign parity(B & z) ^ parity(l & z), and r ^ x = B | (l ^ x)."""
    assert B % (1 << wbits) == 0 and np.asarray(xm).max(initial=0) < (1 << wbits)
    s = 1 - 2 * parity(np.int64(B) & np.asarray(zm, np.int64))
    return exact_apply(wbits, xm, np.asarray(zm, np.int64) & ((1 << wbits) - 1), s * cr, s * ci, pr, pi, sym)


def prepare_sym_ref(xm, zm, cr, ci):
    """prepare_sym_kernel restated: for the terms of a group whose x has its top bit h >= 11,
    z |= side << 63 | (h+1) << 56 | min(terms left in the group, 0xffff) << 40 and c' *= 2."""
    xm = np.asarray(xm, np.int64)
    M = xm.size
    new = np.r_[True, xm[1:] != xm[:-1]]
    ends = np.r_[np.flatnonzero(new)[1:], M]
    left = ends[np.cumsum(new) - 1] - np.arange(M)
    h = top_bit(xm)
    on = h >= SYM_MIN_BIT
    z = np.asarray(zm, np.int64).astype(np.uint64)
    meta = ((sym_side(xm).astype(np.uint64) << np.uint64(63)) | ((h + 1).astype(np.uint64) << np.uint64(56))
            | (np.minimum(left, LEN_CAP).astype(np.uint64) << np.uint64(40)))
    z[on] |= meta[on]
    return z, np.where(on, 2 * cr, cr), np.where(on, 2 * ci, ci)


def masks_from_symp(symp, coeff_re, coeff_im):
    """Basis-index masks (qubit 0 = most significant bit) and c' = c * (-i)^popcount(x & z) of packed rows."""
    n = symp.shape[1] // 2
    w = np.int64(1) << np.arange(n - 1, -1, -1, dtype=np.int64)
    xb, zb = symp[:, :n].astype(np.int64), symp[:, n:].astype(np.int64)
    k = np.count_nonzero(xb & zb, axis=1) & 3
    re, im = np.asarray(coeff_re, np.int64), np.asarray(coeff_im, np.int64)
    cr = np.choose(k, [re, im, -re, -im])
    ci = np.choose(k, [im, -re, -im, re])
    return (xb * w).sum(axis=1), (zb * w).sum(axis=1), cr, ci


# ------------------------------------------------------------------------------------------- operators and states
def nonzero_ints(rng, size):
    v = rng.integers(1, CMAX + 1, size=size)
    return np.where(rng.random(size) < 0.5, -v, v).astype(np.int64)


def make_terms(n, xs, lengths, rng):
    """Masks sorted by x: group k has x = xs[k] (strictly ascending) and lengths[k] terms. z has popcount(x & z)
    even, so a real c' is a Hermitian term; for n > 32 every z has a bit at or above 32; about one term in eight
    repeats the z of the term before it."""
    xs = np.asarray(xs, np.int64)
    assert (np.diff(xs) > 0).all()
    xm = np.repeat(xs, lengths)
    M = xm.size
    zm = rng.integers(0, 1 << n, size=M, dtype=np.int64)
    if n > 32:
        zm |= rng.integers(1, 1 << (n - 32), size=M, dtype=np.int64) << 32
    odd = parity(xm & zm) == 1
    zm[odd] ^= (xm & -xm)[odd]
    rep = np.flatnonzero((rng.random(M) < 0.125) & np.r_[False, xm[1:] == xm[:-1]])
    zm[rep] = zm[rep - 1]
    return xm, zm


def random_groups(n, n_groups, M, rng):
    """x = 0 first, 2^n - 1 last, some groups with top bit below 11, lengths from 1 to several tiles."""
    side = 1 << n
    xs = np.unique(np.concatenate([[0, side - 1], rng.integers(0, min(side, 1 << SYM_MIN_BIT), n_groups // 4 + 1),
                                   rng.integers(0, side, n_groups)]))
    lengths = 1 + rng.multinomial(max(M, xs.size) - xs.size, rng.dirichlet(np.full(xs.size, 0.5)))
    return make_terms(n, xs, lengths, rng)


def _dev(a, dtype=torch.int64):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype).cuda()


def _cplx(re, im):
    return torch.from_numpy(np.asarray(re, np.float64) + 1j * np.asarray(im, np.float64)).cuda()


def _vp(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class Op:
    """Sorted masks with two coefficient sets: real c' (Hermitian with these masks) and complex c' with the same
    real parts. `d_c[real_coeffs]` holds the one that real_coeffs = 1 or 0 expects."""

    def __init__(self, n, xm, zm, rng):
        self.n, self.xm, self.zm, self.M = n, np.asarray(xm, np.int64), np.asarray(zm, np.int64), len(xm)
        self.cr, self.ci = nonzero_ints(rng, self.M), nonzero_ints(rng, self.M)
        self.d_xm, self.d_zm = _dev(self.xm), _dev(self.zm)
        self.d_c = {1: _cplx(self.cr, 0 * self.ci), 0: _cplx(self.cr, self.ci)}
        self._sym = None

    def coeffs(self, real):
        return self.cr, (0 * self.ci if real else self.ci)

    def sym_table(self, ops):
        """The device table of sym_expval_prepare_sym for the real set, checked bit for bit against its restatement."""
        if self._sym is None:
            z_sym = torch.empty_like(self.d_zm)
            c_sym = torch.empty_like(self.d_c[1])
            if self.M:
                _check(ops.lib().sym_expval_prepare_sym(_vp(self.d_xm), _vp(self.d_zm), _vp(self.d_c[1]), self.M,
                                                        _vp(z_sym), _vp(c_sym), _stream()))
            z_ref, cr_ref, _ = prepare_sym_ref(self.xm, self.zm, self.cr, 0 * self.ci)
            assert np.array_equal(z_sym.cpu().numpy().view(np.uint64), z_ref)
            c = c_sym.cpu().numpy()
            assert np.array_equal(c.real, cr_ref) and np.array_equal(c.imag, np.zeros(self.M))
            self._sym = (z_sym, c_sym)
        return self._sym


def host_state(rows, rng):
    return (rng.integers(-PMAX, PMAX + 1, size=rows, dtype=np.int64),
            rng.integers(-PMAX, PMAX + 1, size=rows, dtype=np.int64))


def state(rows, rng):
    pr, pi = host_state(rows, rng)
    return pr, pi, _cplx(pr, pi)


def _check(rc):
    from symmer_b200 import _cabi
    _cabi.check(rc)


# ------------------------------------------------------------------------------------------- C ABI calls
def branch(n, rb, re, real, knob, sym=False):
    """Which kernel apply_common runs (for failure messages)."""
    rows = re - rb
    wide = "" if n <= 32 else "-wide"
    if rows == 0:
        return "empty"
    if sym:
        return "applyw-sym" + wide
    if knob == 1 and rows % SPAN == 0 and rb % SPAN == 0:
        return ("applyw-real" if real else "applyw-complex") + wide
    if rows % 1024 == 0 and rb % 1024 == 0:
        return "apply4-real" if real else "apply4-complex"
    return "apply"


def call_apply(ops, op, n, psi_ptr, rb, re, real, d_xm=None, d_zm=None):
    """sym_apply into a NaN-filled buffer with a guard region: returns the rows it wrote, and checks that every
    row was written and nothing after them."""
    rows = re - rb
    y = torch.full((rows + GUARD,), complex(float("nan"), float("nan")), dtype=torch.complex128, device="cuda")
    d_xm = op.d_xm if d_xm is None else d_xm
    d_zm = op.d_zm if d_zm is None else d_zm
    _check(ops.lib().sym_apply(_vp(d_xm), _vp(d_zm), _vp(op.d_c[real]), op.M, n, psi_ptr, _vp(y), rb, re, real,
                               _stream()))
    y = y.cpu().numpy()
    assert np.isnan(y[rows:].real).all() and np.isnan(y[rows:].imag).all(), "sym_apply wrote past row_end - row_begin"
    return y[:rows]


def call_expval(ops, op, n, psi_ptr, rb, re, mode):
    """sym_expval with real_coeffs = mode into a partial that already holds PARTIAL0; returns what was added."""
    partial = torch.tensor(PARTIAL0, dtype=torch.float64, device="cuda")
    if mode == 2:
        z, c = op.sym_table(ops)
    else:
        z, c = op.d_zm, op.d_c[mode]
    _check(ops.lib().sym_expval(_vp(op.d_xm), _vp(z), _vp(c), op.M, n, psi_ptr, _vp(partial), rb, re, mode,
                                _stream()))
    got = partial.cpu().numpy()
    return got[0] - PARTIAL0[0], got[1] - PARTIAL0[1]


def assert_rows(y, ref, lo, hi, what):
    yr, yi = ref
    bad = np.flatnonzero((y.real != yr[lo:hi]) | (y.imag != yi[lo:hi]))
    assert bad.size == 0, (what, f"{bad.size} wrong rows, first {lo + bad[0]}: {y[bad[0]]} vs {yr[lo + bad[0]]}"
                                 f"{yi[lo + bad[0]]:+d}j")


def run_plain(ops, op, pr, pi, d_psi, ranges, knobs=(1, 0), refs=None):
    """apply and expval through every (range, knob, real_coeffs) against the exact reference."""
    n = op.n
    refs = refs or {real: exact_apply(n, op.xm, op.zm, *op.coeffs(real), pr, pi) for real in (1, 0)}
    try:
        for knob in knobs:
            ops.set_tuning(4, knob)
            for rb, re in ranges:
                for real in (1, 0):
                    what = (n, rb, re, knob, branch(n, rb, re, real, knob))
                    assert_rows(call_apply(ops, op, n, _vp(d_psi), rb, re, real), refs[real], rb, re, what)
                    e = call_expval(ops, op, n, _vp(d_psi), rb, re, real)
                    assert e == exact_expval(pr, pi, refs[real], rb, re), what
    finally:
        ops.set_tuning(4, 1)
    return refs


def run_sym(ops, op, pr, pi, d_psi, cuts):
    """Symmetric mode over [cuts[0], cuts[-1]) and over the shards between consecutive cuts: each shard equals the
    restated symmetric partial sum, partial[1] is never touched, and the shards add up to the exact expectation
    value when they cover the whole basis."""
    n = op.n
    ysym = exact_apply(n, op.xm, op.zm, *op.coeffs(1), pr, pi, sym=True)
    full = call_expval(ops, op, n, _vp(d_psi), cuts[0], cuts[-1], 2)
    assert full == (exact_expval(pr, pi, ysym, cuts[0], cuts[-1])[0], 0.0), (n, cuts[0], cuts[-1], "applyw-sym")
    total = 0
    for rb, re in zip(cuts[:-1], cuts[1:]):
        e = call_expval(ops, op, n, _vp(d_psi), rb, re, 2)
        assert e == (exact_expval(pr, pi, ysym, rb, re)[0], 0.0), (n, rb, re, "applyw-sym")
        total += e[0]
    assert total == full[0]
    if (cuts[0], cuts[-1]) == (0, 1 << n):
        e_full = exact_expval(pr, pi, exact_apply(n, op.xm, op.zm, *op.coeffs(1), pr, pi))
        assert e_full[1] == 0 and full[0] == e_full[0]


@pytest.fixture(scope="module")
def ops():
    import symmer_b200.ops as o
    o.device()
    return o


# ------------------------------------------------------------------------------------------- 1. the reference
@pytest.mark.parametrize("n", [1, 2, 5, 8])
def test_exact_reference_matches_oracle(n):
    """The int64 reference against the oracle's matrix-free apply and its sparse matrix (qiskit semantics), with
    masks taken from packed rows that include Y (the (-i)^Y folding), repeated Paulis and Gaussian-integer
    coefficients; and the windowed and symmetric forms against the full one."""
    rng = np.random.default_rng(100 + n)
    M = 6 * n + 3
    symp = rng.random((M, 2 * n)) < 0.5
    symp[1] = symp[0]
    symp[2] = False
    symp[2, 0] = symp[2, n] = True                      # Y on qubit 0
    symp[3, :] = True                                   # Y everywhere
    re, im = nonzero_ints(rng, M), nonzero_ints(rng, M)
    pr, pi = host_state(1 << n, rng)
    xm, zm, cr, ci = masks_from_symp(symp, re, im)
    order = np.argsort(xm, kind="stable")
    y = exact_apply(n, xm[order], zm[order], cr[order], ci[order], pr, pi)
    psi = pr + 1j * pi
    ref = po.pauli_apply_dense(symp, re + 1j * im, psi)
    assert np.array_equal(y[0], ref.real) and np.array_equal(y[1], ref.imag)
    ref = po.to_sparse_matrix(symp, re + 1j * im) @ psi
    assert np.array_equal(y[0], ref.real) and np.array_equal(y[1], ref.imag)
    e = exact_expval(pr, pi, y)
    assert complex(*e) == np.vdot(psi, ref)
    if n >= 5:
        wbits, B = 3, (1 << n) - 8
        small = xm < (1 << wbits)
        yw = exact_apply_window(B, wbits, xm[small], zm[small], cr[small], ci[small], pr[B:B + 8], pi[B:B + 8])
        yf = exact_apply(n, xm[small], zm[small], cr[small], ci[small], pr, pi)
        assert np.array_equal(yw[0], yf[0][B:B + 8]) and np.array_equal(yw[1], yf[1][B:B + 8])


def test_symmetric_restatement_sums_to_the_expectation_value():
    """The restated symmetric mode: over the whole basis it gives the exact real expectation value of a Hermitian
    operator, while a single 2048-row shard differs from the plain partial sum over its rows."""
    rng = np.random.default_rng(7)
    n = 13
    xm, zm = random_groups(n, 30, 900, rng)
    cr = nonzero_ints(rng, xm.size)
    pr, pi = host_state(1 << n, rng)
    zero = 0 * cr
    y = exact_apply(n, xm, zm, cr, zero, pr, pi)
    ys = exact_apply(n, xm, zm, cr, zero, pr, pi, sym=True)
    e = exact_expval(pr, pi, y)
    assert e[1] == 0 and exact_expval(pr, pi, ys)[0] == e[0]
    assert exact_expval(pr, pi, ys, 2048, 4096)[0] != exact_expval(pr, pi, y, 2048, 4096)[0]
    z_sym, c_sym, _ = prepare_sym_ref(xm, zm, cr, zero)
    hi = top_bit(xm) >= SYM_MIN_BIT
    assert np.array_equal(c_sym[hi], 2 * cr[hi]) and np.array_equal(c_sym[~hi], cr[~hi])
    assert np.array_equal(z_sym[~hi], zm[~hi].astype(np.uint64))
    assert np.array_equal((z_sym[hi] >> np.uint64(56)) & np.uint64(0x7f), (top_bit(xm[hi]) + 1).astype(np.uint64))


# ------------------------------------------------------------------------------------------- 2. dispatch branches
def dispatch_ranges(side):
    rs = [(0, side)]
    if side >= 2 * SPAN:
        rs += [(SPAN, side), (1024, 3072)]          # applyw with row_begin > 0; 1024- but not 2048-aligned: apply4
    elif side == SPAN:
        rs += [(1024, SPAN)]
    rs += [(3, side - 5)] if side > 8 else [(1, side - 1)]
    rs += [(side - 1, side), (side // 3, side // 3 + 1)]
    if side >= 1024:
        rs += [(256, side - 100)]                   # ends inside the last CTA
    rs += [(side // 2, side // 2)]                  # empty range: nothing written, nothing added
    return rs


@gpu
@pytest.mark.parametrize("n", [1, 3, 10, 11, 12, 13, 16, 20])
def test_every_dispatch_branch_is_exact(ops, n):
    """sym_apply / sym_expval through the C ABI on every kernel family apply_common can pick: the 16-row (real) and
    8-row (complex) static-sign kernels (knob 4 = 1, 2048-aligned ranges), the 4-row kernel (knob 4 = 0, or ranges
    aligned to 1024 only), the one-row kernel (unaligned ranges, one row, a range ending inside its last CTA), the
    symmetric mode, M = 0 and empty ranges. y must be written exactly up to row_end - row_begin and no further,
    partial must be added into, and symmetric mode must leave partial[1] alone."""
    rng = np.random.default_rng(n)
    side = 1 << n
    groups, M = {1: (2, 5), 3: (6, 40)}.get(n, (6 if n == 20 else 40, 1100))
    op = Op(n, *random_groups(n, groups, M, rng), rng)
    assert op.M > TILE or n <= 3
    pr, pi, d_psi = state(side, rng)
    run_plain(ops, op, pr, pi, d_psi, dispatch_ranges(side))
    if side % SPAN == 0:
        run_sym(ops, op, pr, pi, d_psi, sorted({0, SPAN, side // 2 // SPAN * SPAN, side}))
    # M = 0: y is all zeros and partial does not move, on every branch
    empty = Op(n, np.zeros(0, np.int64), np.zeros(0, np.int64), rng)
    run_plain(ops, empty, pr, pi, d_psi, dispatch_ranges(side))
    if side % SPAN == 0:
        assert call_expval(ops, empty, n, _vp(d_psi), 0, side, 2) == (0.0, 0.0)


# ------------------------------------------------------------------------------------------- 3. tile boundaries
def _mixed_shape(rng):
    """~5000 terms: the diagonal group first, singletons with top bit < 11, a skip that ends exactly at a tile's end
    (375 terms ending at 511), a group that fills tile 1, a group that starts at the last slot of tile 2 and runs
    into tile 3, a group of 1100 terms across three tiles, hundreds of singletons, a group straddling 3583/3584,
    and 2^13 - 1 last."""
    head = [37] + [1] * 100
    hi = [375, 512, 511, 3, 1100] + [1] * 400 + [34, 429, 200]
    tail = list(rng.integers(1, 30, size=40)) + [1] * 300
    hi += tail + [5001 - sum(head) - sum(hi) - sum(tail)]
    assert hi[-1] > 0
    lo_x = np.sort(rng.choice(np.arange(1, 1 << SYM_MIN_BIT), size=100, replace=False))
    hi_x = np.r_[np.sort(rng.choice(np.arange(1 << SYM_MIN_BIT, (1 << 13) - 1), size=len(hi) - 1, replace=False)),
                 (1 << 13) - 1]
    return np.r_[0, lo_x, hi_x], head + hi


SHAPES = {
    "M1": lambda rng: ([6000], [1]),
    "M511": lambda rng: ([0, 3000, 8191], [1, 199, 311]),
    "M512_one_tile": lambda rng: ([x_with_side(12, 1)], [512]),
    "M513_straddle": lambda rng: ([x_with_side(11, 1), 5000], [500, 13]),
    "M1024_last_slot_then_full_tile": lambda rng: ([0, 2050, 7000], [511, 1, 512]),
    "M1031_three_tiles": lambda rng: ([3333, 8191], [1030, 1]),
    "M5001_mixed": _mixed_shape,
}


@gpu
@pytest.mark.parametrize("shape", list(SHAPES))
def test_term_stream_tile_boundaries(ops, shape):
    """Groups placed on purpose against the 512-term tiles, through every branch at n = 13. In symmetric mode half
    of the CTAs skip each group with top bit >= 11, so the same placements skip from the last slot of a tile, up
    to exactly a tile's end, and across tiles."""
    rng = np.random.default_rng(len(shape))
    n, side = 13, 1 << 13
    xs, lengths = SHAPES[shape](rng)
    op = Op(n, *make_terms(n, xs, lengths, rng), rng)
    pr, pi, d_psi = state(side, rng)
    run_plain(ops, op, pr, pi, d_psi, [(0, side), (1024, 3072), (3, side - 5)])
    run_sym(ops, op, pr, pi, d_psi, [0, SPAN, 3 * SPAN, side])


# ------------------------------------------------------------------------------------------- 4. symmetric table
@gpu
def test_symmetric_table_and_capped_groups(ops):
    """sym_expval_prepare_sym bit for bit against its restatement on groups of 1, 2, 65535, 65536 and 2*65535 + 3
    terms (the length field caps at 65535, so the longer groups are skipped in several hops), then symmetric
    expectation values over the whole basis and over 2048-aligned shards. The groups alternate between the two
    halves of the rows, so each half skips some of them."""
    rng = np.random.default_rng(17)
    n, side = 17, 1 << 17
    xs = [0, 5, x_with_side(11, 0), x_with_side(12, 1), x_with_side(14, 1), x_with_side(15, 0), x_with_side(16, 1)]
    lengths = [3, 4, 1, 2, LEN_CAP, LEN_CAP + 1, 2 * LEN_CAP + 3]
    op = Op(n, *make_terms(n, xs, lengths, rng), rng)
    op.sym_table(ops)
    pr, pi, d_psi = state(side, rng)
    run_sym(ops, op, pr, pi, d_psi, [0, SPAN, 4 * SPAN, side // 2, side])
    y = exact_apply(n, op.xm, op.zm, *op.coeffs(1), pr, pi)
    assert call_expval(ops, op, n, _vp(d_psi), 0, side, 1) == exact_expval(pr, pi, y)


# ------------------------------------------------------------------------------------------- 5. 64-bit signs
WINDOWS = [(20, (1 << 19) + 3 * (1 << WIN)), (32, 1 << 31), (32, (1 << 32) - (1 << WIN)),
           (34, (1 << 33) - (1 << WIN)), (34, (1 << 33) + 5 * (1 << WIN)), (40, (1 << 40) - (1 << WIN))]


@gpu
@pytest.mark.parametrize("n,B", WINDOWS)
def test_row_window_of_a_wide_state(ops, n, B):
    """Rows [B, B + 2^14) of an n-qubit operator without the 2^n state, so the 64-bit sign instantiations
    (n = 33..40) run. The terms have x < 2^14, so every psi[r ^ x] the kernels read lies in the window, and psi is
    passed as a 2^14-entry buffer minus B elements: every address the kernels form, psi + (r ^ x) and psi + r,
    lands in the buffer. z masks have bits at or above 32, so a 32-bit popcount of r & z would give wrong signs.

    The harness itself is checked where a full state fits: at n = 20 the windowed call on a copy of the window must
    equal the call on the full state, and the windowed reference must equal the full reference's rows. n = 32 runs
    the same windows on the 32-bit instantiations at the top rows of the index range."""
    rng = np.random.default_rng(n + B % 1000)
    xs = np.unique(np.r_[0, rng.integers(1, 1 << SYM_MIN_BIT, 4), rng.integers(1 << SYM_MIN_BIT, 1 << WIN, 16)])
    lengths = 1 + rng.multinomial(700 - xs.size, rng.dirichlet(np.full(xs.size, 0.5)))
    op = Op(n, *make_terms(n, xs, lengths, rng), rng)
    rows = 1 << WIN
    pr, pi, d_win = state(rows, rng)
    psi_ptr = ctypes.c_void_p((d_win.data_ptr() - B * 16) % (1 << 64))
    refs = {real: exact_apply_window(B, WIN, op.xm, op.zm, *op.coeffs(real), pr, pi) for real in (1, 0)}
    if n == 20:
        side = 1 << n
        fr, fi, d_full = state(side, rng)
        fr[B:B + rows], fi[B:B + rows] = pr, pi
        d_full[B:B + rows] = d_win
        for real in (1, 0):
            yf = exact_apply(n, op.xm, op.zm, *op.coeffs(real), fr, fi)
            assert np.array_equal(yf[0][B:B + rows], refs[real][0]) and np.array_equal(yf[1][B:B + rows], refs[real][1])
            full = call_apply(ops, op, n, _vp(d_full), B, B + rows, real)
            assert np.array_equal(call_apply(ops, op, n, psi_ptr, B, B + rows, real), full)
            assert call_expval(ops, op, n, psi_ptr, B, B + rows, real) == call_expval(ops, op, n, _vp(d_full), B,
                                                                                      B + rows, real)
    try:
        for knob in (1, 0):
            ops.set_tuning(4, knob)
            for real in (1, 0):
                what = (n, B, knob, branch(n, B, B + rows, real, knob))
                assert_rows(call_apply(ops, op, n, psi_ptr, B, B + rows, real), refs[real], 0, rows, what)
                assert call_expval(ops, op, n, psi_ptr, B, B + rows, real) == exact_expval(pr, pi, refs[real]), what
    finally:
        ops.set_tuning(4, 1)
    ysym = exact_apply_window(B, WIN, op.xm, op.zm, *op.coeffs(1), pr, pi, sym=True)
    total = 0
    for lo, hi in [(0, SPAN), (SPAN, 3 * SPAN), (3 * SPAN, rows)]:
        e = call_expval(ops, op, n, psi_ptr, B + lo, B + hi, 2)
        assert e == (exact_expval(pr, pi, ysym, lo, hi)[0], 0.0), (n, B, lo, hi, "applyw-sym")
        total += e[0]
    assert total == exact_expval(pr, pi, refs[1])[0]
    assert call_expval(ops, op, n, psi_ptr, B, B + rows, 2) == (total, 0.0)


# ------------------------------------------------------------------------------------------- 6. CSR
def exact_csr(n, xm, zm, cr, ci):
    """G entries per row, sorted by column, explicit zeros kept: (data_re, data_im, indices, indptr)."""
    side = 1 << n
    ux, g = np.unique(xm, return_inverse=True)
    G = ux.size
    w = []
    for c in (cr, ci):
        a = np.zeros((G, side), np.int64)
        np.add.at(a, (g, zm), c)
        wht_(a)
        w.append(a.T)
    cols = np.arange(side, dtype=np.int64)[:, None] ^ ux[None, :]
    order = np.argsort(cols, axis=1)
    take = lambda a: np.take_along_axis(a, order, axis=1).ravel()    # noqa: E731
    return take(w[0]), take(w[1]), take(cols), np.arange(side + 1, dtype=np.int64) * G


@gpu
@pytest.mark.parametrize("n,G", [(1, 1), (1, 2), (5, 1), (5, 32), (12, 300), (14, 300)])
def test_csr_is_exact(ops, n, G):
    """ops.to_csr and sym_to_csr against the exact CSR (G entries per row sorted by column, zeros kept), csr @ psi
    against the exact apply, and every output slot written (buffers pre-filled with sentinels)."""
    import scipy.sparse as sps
    rng = np.random.default_rng(1000 * n + G)
    side = 1 << n
    xs = np.sort(rng.choice(side, size=G, replace=False))
    lengths = rng.integers(1, 6, size=G)
    xm, zm = make_terms(n, xs, lengths, rng)
    if lengths[0] >= 2:
        zm[1] = zm[0]                                   # a repeated (x, z) pair
    op = Op(n, xm, zm, rng)
    cr, ci = op.coeffs(0)
    ci[rng.random(op.M) < 0.1] = 0
    op.d_c[0] = _cplx(cr, ci)
    ref = exact_csr(n, xm, zm, cr, ci)
    data, indices, indptr = (t.cpu().numpy() for t in ops.to_csr(op.d_xm, op.d_zm, op.d_c[0], n))
    assert np.array_equal(data.real, ref[0]) and np.array_equal(data.imag, ref[1])
    assert np.array_equal(indices, ref[2]) and np.array_equal(indptr, ref[3])
    pr, pi, _ = state(side, rng)
    y = sps.csr_matrix((data, indices, indptr), shape=(side, side)) @ (pr + 1j * pi)
    yr, yi = exact_apply(n, xm, zm, cr, ci, pr, pi)
    assert np.array_equal(y.real, yr) and np.array_equal(y.imag, yi)
    # direct call with sentinel-filled outputs
    d_xg = _dev(xs)
    d_start = _dev(np.r_[0, np.cumsum(lengths)], torch.int32)
    d_data = torch.full((side * G,), complex(float("nan"), float("nan")), dtype=torch.complex128, device="cuda")
    d_idx = torch.full((side * G,), -1, dtype=torch.int64, device="cuda")
    d_ptr = torch.full((side + 1,), -1, dtype=torch.int64, device="cuda")
    _check(ops.lib().sym_to_csr(_vp(op.d_zm), _vp(op.d_c[0]), op.M, n, _vp(d_xg), G, _vp(d_start),
                                _vp(d_data), _vp(d_idx), _vp(d_ptr), _stream()))
    data = d_data.cpu().numpy()
    assert np.array_equal(data.real, ref[0]) and np.array_equal(data.imag, ref[1])
    assert np.array_equal(d_idx.cpu().numpy(), ref[2]) and np.array_equal(d_ptr.cpu().numpy(), ref[3])


# ------------------------------------------------------------------------------------------- 7. masks and dispatch
def _flavoured_coeffs(symp, rng, flavour):
    """Integer coefficients: 'hermitian' real c on even-Y rows only; 'real' real c with odd-Y rows present (c' is
    not real); 'phased' c = a * i^Y, so c' = a is real but c is not; 'complex' Gaussian integers."""
    y = po.y_count(symp)
    M = symp.shape[0]
    a, b = nonzero_ints(rng, M), nonzero_ints(rng, M)
    if flavour == "hermitian":
        keep = y % 2 == 0
        return symp[keep], a[keep], 0 * a[keep]
    if flavour == "real":
        assert (y % 2 == 1).any()
        return symp, a, 0 * a
    if flavour == "phased":
        k = y & 3
        return symp, np.choose(k, [a, 0 * a, -a, 0 * a]), np.choose(k, [0 * a, a, 0 * a, -a])
    return symp, a, b


FLAGS = {"hermitian": (True, True), "real": (False, False), "phased": (True, False), "complex": (False, False)}


@gpu
@pytest.mark.parametrize("n", [1, 31, 32, 33, 62])
@pytest.mark.parametrize("M", [32, 33, 300])
def test_term_masks_sorted_is_exact(ops, n, M):
    """Bit-reversed masks, c' = c * (-i)^popcount(x & z) exactly, stable ascending x order, and the real/Hermitian
    flags on both sides of the 32-term cut (32 terms and fewer never take the fast paths)."""
    for k, flavour in enumerate(FLAGS):
        rng = np.random.default_rng(10 * n + M + k)
        symp = rng.random((3 * M, 2 * n)) < 0.5
        symp[0] = False
        symp[0, 0] = symp[0, n] = True                      # one Y: odd
        symp[M // 2:M] = symp[:M - M // 2]                  # repeated rows: the sort must keep their order
        symp, re, im = _flavoured_coeffs(symp, rng, flavour)
        symp, re, im = symp[:M], re[:M], im[:M]
        assert symp.shape[0] == M
        assert flavour == "hermitian" or (po.y_count(symp) % 2 == 1).any()
        xz = ops.pack(torch.from_numpy(np.ascontiguousarray(symp)), n)
        xm, zm, cp = ops.term_masks_sorted(xz, _cplx(re, im), n)
        rx, rz, rcr, rci = masks_from_symp(symp, re, im)
        order = np.argsort(rx, kind="stable")
        assert np.array_equal(xm.cpu().numpy(), rx[order]) and np.array_equal(zm.cpu().numpy(), rz[order])
        c = cp.cpu().numpy()
        assert np.array_equal(c.real, rcr[order]) and np.array_equal(c.imag, rci[order]), flavour
        want = FLAGS[flavour] if M > 32 else (False, False)
        assert (cp._sym_real, cp._sym_hermitian) == want, flavour
        assert cp._sym_table is None


@gpu
def test_public_dispatch_picks_the_symmetric_mode_exactly_when_allowed(ops):
    """ops.apply_dense / ops.expval_dense with the attributes term_masks_sorted computes: the symmetric mode runs
    exactly when the operator is Hermitian with real c', side, row_begin and row_end are multiples of 2048 and
    use_symmetric_expval is on (a symmetric shard sum differs from the plain one, which tells them apart); both
    give the exact value over the whole basis, and the table is built once and reused."""
    def setup(n, flavour, seed):
        rng = np.random.default_rng(seed)
        symp = rng.random((900, 2 * n)) < 0.5
        symp[:, :n] &= rng.random((900, 1)) < 0.9             # some diagonal terms
        symp, re, im = _flavoured_coeffs(symp, rng, flavour)
        symp, re, im = symp[:400], re[:400], im[:400]
        xz = ops.pack(torch.from_numpy(np.ascontiguousarray(symp)), n)
        xm, zm, cp = ops.term_masks_sorted(xz, _cplx(re, im), n)
        hx, hz = xm.cpu().numpy(), zm.cpu().numpy()
        c = cp.cpu().numpy()
        hcr, hci = c.real.astype(np.int64), c.imag.astype(np.int64)
        pr, pi, d_psi = state(1 << n, rng)
        y = exact_apply(n, hx, hz, hcr, hci, pr, pi)
        ysym = exact_apply(n, hx, hz, hcr, hci, pr, pi, sym=True) if flavour == "hermitian" else None
        return (xm, zm, cp), (hx, hz, hcr, hci), (pr, pi, d_psi), y, ysym

    def ev(dev_op, n, d_psi, rb, re):
        e = complex(ops.expval_dense(*dev_op, n, d_psi, rb, re).cpu().numpy())
        return e.real, e.imag

    n = 12
    side = 1 << n
    dev_op, host, (pr, pi, d_psi), y, ysym = setup(n, "hermitian", 1)
    cp = dev_op[2]
    assert cp._sym_hermitian
    for rb, re in [(0, side), (SPAN, side), (3, 100)]:
        got = ops.apply_dense(*dev_op, n, d_psi, rb, re).cpu().numpy()
        assert_rows(got, y, rb, re, ("apply_dense", rb, re))
    full = exact_expval(pr, pi, y)
    assert full[1] == 0
    shard_sym = exact_expval(pr, pi, ysym, SPAN, 2 * SPAN)
    shard_plain = exact_expval(pr, pi, y, SPAN, 2 * SPAN)
    assert shard_sym[0] != shard_plain[0]
    assert ev(dev_op, n, d_psi, 0, side) == full                        # symmetric
    table = cp._sym_table
    assert table is not None
    z_ref, c_ref, _ = prepare_sym_ref(host[0], host[1], host[2], host[3])
    assert np.array_equal(table[0].cpu().numpy().view(np.uint64), z_ref)
    assert np.array_equal(table[1].cpu().numpy().real, c_ref)
    assert ev(dev_op, n, d_psi, SPAN, 2 * SPAN) == (shard_sym[0], 0.0)  # symmetric, table reused
    assert cp._sym_table is table
    assert ev(dev_op, n, d_psi, 1024, 3072) == exact_expval(pr, pi, y, 1024, 3072)   # unaligned: plain
    try:
        ops.use_symmetric_expval = False
        assert ev(dev_op, n, d_psi, SPAN, 2 * SPAN) == shard_plain
        assert ev(dev_op, n, d_psi, 0, side) == full
    finally:
        ops.use_symmetric_expval = True
    assert cp._sym_table is table

    # side not a multiple of 2048 (n = 10), and operators that are not Hermitian with real c': always plain
    for n, flavour in [(10, "hermitian"), (12, "phased"), (12, "complex"), (11, "hermitian")]:
        dev_op, host, (pr, pi, d_psi), y, ysym = setup(n, flavour, n)
        side = 1 << n
        got = ops.apply_dense(*dev_op, n, d_psi).cpu().numpy()
        assert_rows(got, y, 0, side, ("apply_dense", n, flavour))
        assert ev(dev_op, n, d_psi, 0, side) == exact_expval(pr, pi, y), (n, flavour)
        assert (dev_op[2]._sym_table is not None) == (side % SPAN == 0 and flavour == "hermitian"), (n, flavour)
