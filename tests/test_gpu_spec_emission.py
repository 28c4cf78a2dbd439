"""Speculative row emission of class-mode products (csrc/dedup.cu, dedup_product_spec_classes). The class kernel first
runs one wave of classes, one per SM. When that sample finds no duplicate candidate, no class overflow and no
coefficient that can fail the threshold, the output is allocated at T rows and every cross term is written at its
no-drop slot while the rest of the detection runs; the rows are kept iff nothing was dropped (U == T), and otherwise
rewritten by the plain emission.

Every product is compared with the record-sort path (knob 10 = 0). Which path ran is read from the output's storage
(a speculating product allocates T rows) and from the launch count: against a kept speculation, a refused one runs one
launch more (the first wave and the rest are two class-kernel launches, the plain emission adds its fix-up) and a
fallback two more (the plain emission and its fix-up)."""
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


def n_sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def class_bits(T):
    """class_job_plan (csrc/class_dedup.cu) for the default class kernel: 2^k classes."""
    target = int(0.85 * 18432)
    if T // 1024 < target:
        target = max(T // 1024, 256)
    k = 0
    while k < 22 and (T >> k) > target:
        k += 1
    return k


def cd_class(sk, k):
    """cd_class_of (csrc/class_dedup.cu) of uint64 sketches."""
    sk = np.asarray(sk, dtype=np.uint64)
    y = sk ^ (sk >> np.uint64(21)) ^ (sk >> np.uint64(43))
    return ((y >> np.uint64(5)) & np.uint64((1 << k) - 1)).astype(np.int64)


def dev_op(ops, s, c):
    n = s.shape[1] // 2
    return (ops.pack(torch.from_numpy(np.ascontiguousarray(s)), n),
            torch.from_numpy(np.asarray(c, dtype=complex)).cuda())


def sketches(ops, s):
    xz, _ = dev_op(ops, s, np.ones(len(s)))
    return ops.sketch(xz).cpu().numpy().view(np.uint64)


def unit_phase(a_row, b_row):
    """Coefficient of the cross term a_row * b_row with unit coefficients: one of 1, -1, i, -i."""
    c = complex(po.cross_terms(a_row[None], [1.0], b_row[None], [1.0])[1][0])
    return complex(round(c.real), round(c.imag))


def plant(ops, a_s, a_c, b_s, b_c, seed, cancel):
    """B[j] = B[i] ^ A[p] ^ A[p2] makes (p, j) == (p2, i) and (p2, j) == (p, i). Both rows are in classes at or above the
    SM count, which the sampled wave does not see. cancel: unit coefficients chosen so that both pairs sum to exactly 0.
    Returns the two planted rows."""
    M, N = len(a_s), len(b_s)
    k = class_bits(M * N)
    assert (1 << k) > n_sms()
    ska, skb = sketches(ops, a_s), sketches(ops, b_s)
    rng = np.random.default_rng(seed)
    for _ in range(10000):
        p, p2 = (int(x) for x in rng.choice(M, 2, replace=False))
        i, j = (int(x) for x in rng.choice(N, 2, replace=False))
        if min(cd_class(ska[p2] ^ skb[i], k), cd_class(ska[p] ^ skb[i], k)) < n_sms():
            continue
        bj = b_s[i] ^ a_s[p] ^ a_s[p2]
        if cancel:
            # c_A[p] = c_B[i] = 1, c_A[p2] = v, c_B[j] = u: v f1 + u f2 = 0 and f3 + u v f4 = 0
            f1, f2 = unit_phase(a_s[p2], b_s[i]), unit_phase(a_s[p], bj)
            f3, f4 = unit_phase(a_s[p], b_s[i]), unit_phase(a_s[p2], bj)
            sol = [v for v in (1, -1, 1j, -1j) if f3 - v * v * f1 * f4 / f2 == 0]
            if not sol:
                continue
            v = sol[0]
            u = -v * f1 / f2
            a_c[p], b_c[i], a_c[p2], b_c[j] = 1, 1, v, complex(round(u.real), round(u.imag))
        b_s[j] = bj
        return a_s[p2] ^ b_s[i], a_s[p] ^ b_s[i]
    raise AssertionError("no plant outside the sampled wave")


def counted(ops, fn):
    torch.cuda.synchronize()
    l0 = ops.launch_count()
    out = fn()
    torch.cuda.synchronize()
    return out, ops.launch_count() - l0


def record_sort(ops, fn):
    try:
        ops.set_tuning(10, 0)
        return fn()
    finally:
        ops.set_tuning(10, 1)


def rows_allocated(xz):
    return xz.untyped_storage().nbytes() // (xz.shape[1] * 8)


def check_same(out, ref, scale, n_groups=0):
    """Same rows in the same order; coefficients bit-identical except at the heads of summed groups (rtol 1e-12)."""
    (xz, c), (rxz, rc) = out, ref
    assert torch.equal(xz, rxz)
    diff = c != rc
    assert int(diff.sum()) <= n_groups
    assert torch.allclose(c[diff], rc[diff], rtol=1e-12, atol=1e-12 * scale)


def has_row(ops, xz, row):
    r = ops.pack(torch.from_numpy(row[None, :].copy()), row.shape[0] // 2).to(xz.device)
    return bool((xz == r).all(dim=1).any())


def mul(ops, a_s, a_c, b_s, b_c, thr=1e-15):
    a, ac = dev_op(ops, a_s, a_c)
    b, bc = dev_op(ops, b_s, b_c)
    return lambda: ops.mul_cleanup(a, ac, b, bc, thr)


def kept_launches(ops, n, m1, m2, seed):
    a_s, a_c = po.random_operator(n, m1, seed=seed)
    b_s, b_c = po.random_operator(n, m2, seed=seed + 1)
    (xz, _), launches = counted(ops, mul(ops, a_s, a_c, b_s, b_c))
    assert xz.shape[0] == m1 * m2
    return launches


@pytest.mark.parametrize("n", [1000, 64])
def test_random_operators_keep_the_speculation(ops, n):
    a_s, a_c = po.random_operator(n, 2100, seed=3)
    b_s, b_c = po.random_operator(n, 2100, seed=4)
    fn = mul(ops, a_s, a_c, b_s, b_c)
    (xz, c), launches = counted(ops, fn)
    T = 2100 * 2100
    assert xz.shape[0] == T and rows_allocated(xz) == T
    check_same((xz, c), record_sort(ops, fn), 1.0)
    # the same product with one coefficient below the threshold is refused at the gate: one launch more
    a_c2 = a_c.copy()
    a_c2[11] = 1e-17
    fn2 = mul(ops, a_s, a_c2, b_s, b_c)
    (xz2, c2), launches2 = counted(ops, fn2)
    assert launches2 == launches + 1
    assert xz2.shape[0] == T - 2100 and rows_allocated(xz2) == T - 2100
    check_same((xz2, c2), record_sort(ops, fn2), 1.0)


@pytest.mark.parametrize("n", [1000, 64])
@pytest.mark.parametrize("cancel", [False, True])
def test_duplicates_outside_the_sample_fall_back(ops, n, cancel):
    """A duplicate pair (or two pairs that cancel to exactly zero, so that their rows leave through the threshold) in
    classes the first wave does not see: the speculation is taken and the plain emission rewrites the output."""
    kept = kept_launches(ops, n, 2100, 2100, seed=20)
    a_s, a_c = po.random_operator(n, 2100, seed=20)
    b_s, b_c = po.random_operator(n, 2100, seed=21)
    r1, r2 = plant(ops, a_s, a_c, b_s, b_c, seed=n + int(cancel), cancel=cancel)
    fn = mul(ops, a_s, a_c, b_s, b_c)
    (xz, c), launches = counted(ops, fn)
    T = 2100 * 2100
    assert launches == kept + 2
    assert rows_allocated(xz) == T
    assert xz.shape[0] == (T - 4 if cancel else T - 2)
    assert has_row(ops, xz, r1) != cancel and has_row(ops, xz, r2) != cancel
    check_same((xz, c), record_sort(ops, fn), 1.0, n_groups=0 if cancel else 2)


def test_small_products_against_oracle(ops):
    """700 x 300 terms through the ordered-tile path (knob 0 = 0): kept, fallback on a pair, fallback on a cancellation."""
    n = 64
    T = 700 * 300
    try:
        ops.set_tuning(0, 0)
        kept = kept_launches(ops, n, 700, 300, seed=30)
        for case in ("random", "pair", "cancel"):
            a_s, a_c = po.random_operator(n, 700, seed=30)
            b_s, b_c = po.random_operator(n, 300, seed=31)
            if case != "random":
                plant(ops, a_s, a_c, b_s, b_c, seed=7, cancel=case == "cancel")
            fn = mul(ops, a_s, a_c, b_s, b_c)
            (xz, c), launches = counted(ops, fn)
            assert launches == kept + (0 if case == "random" else 2), case
            assert rows_allocated(xz) == T
            check_same((xz, c), record_sort(ops, fn), 1.0, n_groups=2 if case == "pair" else 0)
            ref_s, ref_c = po.multiply_by_operator(a_s, a_c, b_s, b_c, 1e-15)
            s, cc = ops.unpack(xz, n).cpu().numpy(), c.cpu().numpy()
            ok, why = po.compare_term_sets(s, cc, ref_s, ref_c)
            assert ok, (case, why)
            assert np.array_equal(s, ref_s), case                  # first-occurrence order
    finally:
        ops.set_tuning(0, 1 << 22)


def test_span_operands_take_the_plain_path(ops):
    """Both operands from the span of 20 generators: the sample is full of duplicates, no output is allocated at T."""
    n = 64
    rng = np.random.default_rng(5)
    gens = rng.random((20, 2 * n)) < 0.3

    def span(rows):
        pick = rng.random((rows, gens.shape[0])) < 0.5
        return ((pick.astype(np.uint8) @ gens.astype(np.uint8)) % 2).astype(bool), rng.standard_normal(rows) + 1j * rng.standard_normal(rows)

    (a_s, a_c), (b_s, b_c) = span(2100), span(2100)
    fn = mul(ops, a_s, a_c, b_s, b_c)
    xz, c = fn()
    U = xz.shape[0]
    assert U < 2100 * 2100 and rows_allocated(xz) == U
    rxz, rc = record_sort(ops, fn)
    assert torch.equal(xz, rxz)
    assert torch.allclose(c, rc, rtol=1e-12, atol=1e-12 * float(np.abs(a_c).max() * np.abs(b_c).max()))


def test_rotation_block_list(ops):
    """rotate_dedup: commuting rows x [I] and anticommuting rows x [cos I, -i sin Q], two blocks of unequal shape."""
    n = 1000
    s, cf = po.random_operator(n, 60000, seed=40)
    q_s, _ = po.random_operator(n, 1, seed=41)
    q = ops.pack(torch.from_numpy(q_s), n)[0].contiguous()

    def rot(coeffs):
        xz, c = dev_op(ops, s, coeffs)
        return lambda: ops.rotate_dedup(xz, c, q, np.cos(0.37), np.sin(0.37))

    (xz, c), launches = counted(ops, rot(cf))
    n_comm = int(po.commutes_termwise(s, q_s).sum())
    assert xz.shape[0] == n_comm + 2 * (60000 - n_comm)
    assert rows_allocated(xz) == xz.shape[0]
    check_same((xz, c), record_sort(ops, rot(cf)), 1.0)
    cf2 = cf.copy()
    cf2[5] = 1e-17
    (xz2, _), launches2 = counted(ops, rot(cf2))
    assert launches2 == launches + 1                             # refused at the gate: the first product speculated


def test_owner_block_list(ops):
    """One owner's part of the product (dist.owned_product, 8 owner classes): 8 blocks of unequal size, as every rank
    of the sharded product and every pass of c5_streamed run them. Checks the per-block output bases."""
    from symmer_b200 import dist as sdist
    n = 1000
    a_s, a_c = po.random_operator(n, 2100, seed=50)
    b_s, b_c = po.random_operator(n, 2100, seed=51)
    a, ac = dev_op(ops, a_s, a_c)
    b, bc = dev_op(ops, b_s, b_c)
    for owner in (0, 5):
        fn = lambda: sdist.owned_product(a, ac, b, bc, 3, owner)[:2]
        (xz, c), launches = counted(ops, fn)
        blocks = sdist.owned_product(a, ac, b, bc, 3, owner)[2]["blocks"]
        sizes = [(p1 - p0) * (q1 - q0) for p0, p1, q0, q1 in blocks]
        assert len(blocks) == 8 and len(set(sizes)) > 1
        assert xz.shape[0] == sum(sizes) and rows_allocated(xz) == sum(sizes)
        check_same((xz, c), record_sort(ops, fn), 1.0)
        ac2 = ac.clone()
        ac2[0] = 1e-17
        _, launches2 = counted(ops, lambda: sdist.owned_product(a, ac2, b, bc, 3, owner)[:2])
        assert launches2 == launches + 1                         # refused at the gate: the first product speculated


def test_result_is_used_on_the_callers_stream(ops):
    """The caller reduces the result on its stream right after the call, with no synchronisation: the library stream
    that wrote the rows must have been joined into it."""
    n = 1000
    a_s, a_c = po.random_operator(n, 2100, seed=60)
    b_s, b_c = po.random_operator(n, 2100, seed=61)
    fn = mul(ops, a_s, a_c, b_s, b_c)
    rxz, rc = record_sort(ops, fn)
    ref = (rc.sum().item(), rxz[-1].clone(), rxz[len(rxz) // 2].clone())
    for _ in range(3):
        xz, c = fn()
        total, last, mid = c.sum(), xz[-1].clone(), xz[len(xz) // 2].clone()
        assert rows_allocated(xz) == 2100 * 2100
        assert total.item() == ref[0]
        assert torch.equal(last, ref[1]) and torch.equal(mid, ref[2])
        del xz, c
