"""Class-local duplicate detection (csrc/class_dedup.cu) when duplicates are rare: the presence filter releases almost
every record and only a few survivors reach the compact list, the table rounds and the counting sort. Duplicates are
planted between different rows of A and different rows of B (B[j] = B[i] ^ A[p] ^ A[p'] makes cross term (p, j) equal
to (p', i)), as pairs and triples in several classes, plus one anticommuting pair whose coefficients cancel exactly."""
import numpy as np
import pytest
import torch

from oracle import pauli_oracle as po

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    import symmer_b200.ops as o
    o.device()
    return o


def anticommute(r1, r2, n):
    return bool((np.count_nonzero(r1[:n] & r2[n:]) + np.count_nonzero(r1[n:] & r2[:n])) & 1)


def planted_operators(n, m1, m2, seed, pairs=40, triples=12):
    """Random A (m1 terms) and B (m2 terms) with planted equal cross terms. Every planted group has its own row i of B,
    so groups cannot meet: a pair plant merges 2 cross terms into others ((p, j) = (p', i) and (p', j) = (p, i)), a
    triple plant 5 ((p, j) = (p3, i) = (p2, j2), (p3, j) = (p, i), (p3, j2) = (p2, i), (p, j2) = (p2, j)), and the
    cancelling pair removes 3 (P*Q and Q*P vanish, the two identity terms P*P and Q*Q merge). Returns the operators,
    the cancelled row and the number of cross terms that leave no row of their own."""
    a_s, a_c = po.random_operator(n, m1, seed=seed)
    b_s, b_c = po.random_operator(n, m2, seed=seed + 1)
    rng = np.random.default_rng(seed)
    js = rng.choice(np.arange(m2 // 2, m2), size=pairs + 2 * triples + 2, replace=False)
    iss = rng.choice(m2 // 2, size=pairs + triples, replace=False)
    for t in range(pairs):                        # (p, j) == (p', i)
        i = int(iss[t])
        p, p2 = rng.choice(m1, size=2, replace=False)
        b_s[js[t]] = b_s[i] ^ a_s[p] ^ a_s[p2]
    for t in range(triples):                      # (p, j) == (p2, j2) == (p3, i)
        i = int(iss[pairs + t])
        p, p2, p3 = rng.choice(m1, size=3, replace=False)
        b_s[js[pairs + 2 * t]] = b_s[i] ^ a_s[p] ^ a_s[p3]
        b_s[js[pairs + 2 * t + 1]] = b_s[i] ^ a_s[p2] ^ a_s[p3]
    # P = A[p1], Q = A[p2] anticommute; B[j1] = Q, B[j2] = P with the same coefficients: P*Q + Q*P = 0 exactly
    p1 = 0
    p2 = next(p for p in range(1, m1) if anticommute(a_s[p1], a_s[p], n))
    j1, j2 = int(js[-2]), int(js[-1])
    b_s[j1], b_c[j1] = a_s[p2], a_c[p2]
    b_s[j2], b_c[j2] = a_s[p1], a_c[p1]
    return a_s, a_c, b_s, b_c, a_s[p1] ^ a_s[p2], 2 * pairs + 5 * triples + 3


def products(ops, a_s, a_c, b_s, b_c, thr=1e-15):
    """Ordered-tile product through the class kernel (knob 11 = 2, and the unfiltered form 3) and the record sort
    (knob 10 = 0); device tensors (xz, c) per (knob 10, knob 11)."""
    n = a_s.shape[1] // 2
    dev = lambda s, c: (ops.pack(torch.from_numpy(np.ascontiguousarray(s)), n), torch.from_numpy(np.asarray(c, dtype=complex)).cuda())
    a, ac = dev(a_s, a_c)
    b, bc = dev(b_s, b_c)
    out = {}
    try:
        ops.set_tuning(0, 0)                      # force the large-product (ordered-tile) path
        for knob in ((1, 2), (1, 3), (0, 2)):
            ops.set_tuning(10, knob[0])
            ops.set_tuning(11, knob[1])
            out[knob] = ops.mul_cleanup(a, ac, b, bc, thr)
    finally:
        ops.set_tuning(10, 1)
        ops.set_tuning(11, 2)
        ops.set_tuning(0, 1 << 22)
    return out


def check_against_record_sort(out, scale):
    base_xz, base_c = out[(0, 2)]
    for knob in ((1, 2), (1, 3)):
        xz, c = out[knob]
        assert torch.equal(xz, base_xz), knob                    # same rows, same (first-occurrence) order
        assert torch.allclose(c, base_c, rtol=1e-12, atol=1e-12 * scale), knob


def check_planted(ops, out, cancelled, T, merged):
    xz, _ = out[(1, 2)]
    n = cancelled.shape[0] // 2
    assert xz.shape[0] == T - merged                             # every planted duplicate merged, nothing else
    row = ops.pack(torch.from_numpy(cancelled[None, :].copy()), n).to(xz.device)
    assert not bool((xz == row).all(dim=1).any())                # the cancelling pair left nothing


@pytest.mark.parametrize("n", [1000, 64])
def test_sparse_duplicates_small_against_oracle(ops, n):
    a_s, a_c, b_s, b_c, cancelled, merged = planted_operators(n, 700, 300, seed=5 + n)
    out = products(ops, a_s, a_c, b_s, b_c)
    scale = float(np.abs(a_c).max() * np.abs(b_c).max())
    check_against_record_sort(out, scale)
    check_planted(ops, out, cancelled, 700 * 300, merged)
    ref_s, ref_c = po.multiply_by_operator(a_s, a_c, b_s, b_c, 1e-15)
    xz, c = out[(1, 2)]
    s, cc = ops.unpack(xz, n).cpu().numpy(), c.cpu().numpy()
    ok, why = po.compare_term_sets(s, cc, ref_s, ref_c, scale=scale)
    assert ok, why
    assert np.array_equal(s, ref_s)                              # first-occurrence order


@pytest.mark.parametrize("n", [1000, 64])
def test_sparse_duplicates_6e6_cross_terms(ops, n):
    """3000 x 2000 terms: 1024 classes of ~5900 records, about a hundred survivors of the filter per class."""
    a_s, a_c, b_s, b_c, cancelled, merged = planted_operators(n, 3000, 2000, seed=17 + n, pairs=150, triples=50)
    out = products(ops, a_s, a_c, b_s, b_c)
    check_against_record_sort(out, float(np.abs(a_c).max() * np.abs(b_c).max()))
    check_planted(ops, out, cancelled, 3000 * 2000, merged)


@pytest.mark.parametrize("rows_a", [2000, 4000, 8000, 16000])
def test_many_survivors_per_class(ops, rows_a):
    """The other end: the last third of A repeats the first, so two thirds of the cross terms have a twin. 1024 classes
    of 2000-16000 records whose survivor lists take 2, 3, 6 and 11 entries per thread; with a threshold that drops
    unique rows (released by the filter, or survivors without a mate) and group sums too."""
    n = 64
    a_s, a_c = po.random_operator(n, rows_a, seed=rows_a)
    b_s, b_c = po.random_operator(n, 1000, seed=rows_a + 1)
    third = rows_a // 3
    a_s[2 * third:3 * third] = a_s[:third]
    scale = float(np.abs(a_c).max() * np.abs(b_c).max())
    for thr in (1e-15, 0.7):
        out = products(ops, a_s, a_c, b_s, b_c, thr)
        check_against_record_sort(out, scale)
        assert out[(1, 2)][0].shape[0] < rows_a * 1000 - third * 1000 // 2
