"""GPU parity tests of the C-ABI kernels (through symmer_b200.ops) against the CPU oracle."""
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


def dev_op(ops, symp, coeff):
    n = symp.shape[1] // 2
    xz = ops.pack(torch.from_numpy(np.ascontiguousarray(symp)), n)
    c = torch.from_numpy(np.asarray(coeff, dtype=complex)).cuda()
    return xz, c


def host_op(ops, xz, c, n):
    return ops.unpack(xz, n).cpu().numpy(), c.cpu().numpy()


@pytest.mark.parametrize("n", [1, 5, 63, 64, 65, 130, 1000, 1100])
def test_pack_unpack_ycount(ops, n):
    rng = np.random.default_rng(n)
    symp = rng.random((37, 2 * n)) < 0.3
    xz = ops.pack(torch.from_numpy(symp), n)
    assert np.array_equal(xz.cpu().numpy().view(np.uint64), po.pack_bits(symp))
    assert np.array_equal(ops.unpack(xz, n).cpu().numpy(), symp)
    assert np.array_equal(ops.ycount(xz).cpu().numpy(), po.y_count(symp))


def test_sketch_is_linear(ops):
    rng = np.random.default_rng(0)
    for n in [3, 64, 200, 1000, 3000]:
        a = rng.random((50, 2 * n)) < 0.3
        b = rng.random((50, 2 * n)) < 0.3
        ha = ops.sketch(ops.pack(torch.from_numpy(a), n))
        hb = ops.sketch(ops.pack(torch.from_numpy(b), n))
        hab = ops.sketch(ops.pack(torch.from_numpy(a ^ b), n))
        assert torch.equal(ha ^ hb, hab)
        assert len(set(ha.cpu().tolist())) == len(np.unique(a, axis=0))   # no sketch collisions


def test_sort_pairs(ops):
    """Both pass forms (knob 8), nonzero begin_bit with an even and an odd (13: 7 passes, copied back) pass
    count, and a size above 1024 tiles, where the one-sweep passes share one look-back state."""
    try:
        for onesweep in [1, 0]:
            ops.set_tuning(8, onesweep)
            rng = np.random.default_rng(1)
            for T in [1, 31, 4096, 4097, 100003, 5_000_000]:
                keys = rng.integers(0, 2**63 - 1, size=T, dtype=np.int64) * 2 + rng.integers(0, 2, size=T)
                keys[::5] = keys[0]                       # many duplicates: checks stability
                vals = np.arange(T, dtype=np.int32)
                for begin_bit in [0, 4, 13]:
                    k = torch.from_numpy(keys.copy()).cuda()
                    v = torch.from_numpy(vals.copy()).cuda()
                    ops.sort_pairs(k, v, begin_bit)
                    order = np.argsort(keys.view(np.uint64) >> np.uint64(begin_bit), kind="stable")
                    assert np.array_equal(k.cpu().numpy(), keys[order]), (onesweep, T, begin_bit)
                    assert np.array_equal(v.cpu().numpy(), vals[order]), (onesweep, T, begin_bit)
    finally:
        ops.set_tuning(8, 1)


@pytest.mark.parametrize("n,m1,m2", [(1, 3, 2), (5, 20, 7), (63, 12, 9), (64, 10, 13), (65, 9, 11), (130, 16, 5),
                                     (1000, 40, 30), (1100, 7, 5)])
def test_cross_terms_bit_exact(ops, n, m1, m2):
    a_s, a_c = po.random_operator(n, m1, seed=n + m1)
    b_s, b_c = po.random_operator(n, m2, seed=n + m2 + 1)
    ref_rows, ref_c = po.cross_terms(a_s, a_c, b_s, b_c)
    xz, c = ops.cross_mul(*dev_op(ops, a_s, a_c), *dev_op(ops, b_s, b_c))
    rows, cc = host_op(ops, xz, c, n)
    assert np.array_equal(rows, ref_rows)               # rows and order: bit-exact
    assert np.allclose(cc, ref_c, rtol=1e-14, atol=0)   # one complex multiply of rounding


def _check_product(ops, a_s, a_c, b_s, b_c, thr=1e-15):
    n = a_s.shape[1] // 2
    ref_s, ref_c = po.multiply_by_operator(a_s, a_c, b_s, b_c, thr)
    xz, c = ops.mul_cleanup(*dev_op(ops, a_s, a_c), *dev_op(ops, b_s, b_c), thr)
    s, cc = host_op(ops, xz, c, n)
    scale = max(1e-300, np.abs(a_c).max() * np.abs(b_c).max())
    ok, why = po.compare_term_sets(s, cc, ref_s, ref_c, scale=scale)
    assert ok, why
    return s, cc, ref_s, ref_c


@pytest.mark.parametrize("n,m1,m2", [(1, 3, 2), (2, 4, 4), (5, 20, 7), (8, 30, 30), (64, 10, 13), (65, 9, 11),
                                     (130, 16, 5), (1000, 60, 45), (1100, 6, 9), (4, 1, 1), (6, 1, 17), (6, 17, 1)])
def test_mul_cleanup_matches_oracle(ops, n, m1, m2):
    a_s, a_c = po.random_operator(n, m1, seed=10 * n + m1)
    b_s, b_c = po.random_operator(n, m2, seed=10 * n + m2 + 3)
    s, cc, ref_s, ref_c = _check_product(ops, a_s, a_c, b_s, b_c)
    if len(ref_c) == len(cc):
        # first-occurrence order, like the reference
        assert np.array_equal(s, ref_s)


def test_square_cancels_anticommuting_pairs_exactly(ops):
    a_s, a_c = po.random_operator(1000, 120, seed=1)
    s, cc, ref_s, ref_c = _check_product(ops, a_s, a_c, a_s, a_c)
    comm = po.commutes_termwise(a_s, a_s)
    n_comm_pairs = (np.count_nonzero(comm) - 120) // 2
    assert len(cc) == n_comm_pairs + 1                  # commuting pairs + identity, residues are exact zeros


def test_mul_cleanup_golden(ops, golden):
    for nm in sorted(k for k in golden if k.startswith(("mul_rand_", "mul_single_"))):
        g = golden[nm]
        a_s, a_c, b_s, b_c = g["a_symp"], g["a_coeff"], g["b_symp"], g["b_coeff"]
        n = a_s.shape[1] // 2
        if a_s.shape[0] < b_s.shape[0]:                 # the reference's dagger swap (base.py:846-851)
            xz, c = ops.mul_cleanup(*dev_op(ops, b_s, b_c.conj()), *dev_op(ops, a_s, a_c.conj()))
            c = c.conj()
        else:
            xz, c = ops.mul_cleanup(*dev_op(ops, a_s, a_c), *dev_op(ops, b_s, b_c))
        s, cc = host_op(ops, xz, c, n)
        ok, why = po.compare_term_sets(s, cc, g["out_symp"], g["out_coeff"],
                                       scale=np.abs(a_c).max() * np.abs(b_c).max())
        assert ok, (nm, why)


def test_forced_key_collisions_still_exact(ops):
    """Mask the dedup keys down to a few bits so that distinct rows share keys: exercises the
    irregular (linked) path; results must not change."""
    a_s, a_c = po.random_operator(70, 40, seed=5)
    b_s, b_c = po.random_operator(70, 35, seed=6)
    b_s[:10] = a_s[:10]
    try:
        for mask in [0xFF00000000000000, 0xF000000000000000, 0x0]:
            ops.set_debug_key_mask(mask)
            _check_product(ops, a_s, a_c, b_s, b_c)
            _check_product(ops, a_s, a_c, a_s, a_c)
            symp = np.vstack([a_s, b_s, a_s[::-1]])
            coeff = np.hstack([a_c, b_c, a_c])
            xz, c = ops.cleanup(*dev_op(ops, symp, coeff))
            s, cc = host_op(ops, xz, c, 70)
            ref_s, ref_c = po.cleanup(symp, coeff)
            ok, why = po.compare_term_sets(s, cc, ref_s, ref_c, scale=np.abs(coeff).max())
            assert ok, why
    finally:
        ops.set_debug_key_mask(0xFFFFFFFFFFFFFFFF)


def test_cleanup_golden_and_order(ops, golden):
    for nm in sorted(k for k in golden if k.startswith("cleanup_")):
        g = golden[nm]
        n = g["symp"].shape[1] // 2
        xz, c = ops.cleanup(*dev_op(ops, g["symp"], g["coeff"]))
        s, cc = host_op(ops, xz, c, n)
        assert s.shape == g["out_symp"].shape, nm
        assert np.array_equal(s, g["out_symp"]), nm      # same first-occurrence order as the reference
        assert np.allclose(cc, g["out_coeff"], rtol=1e-12, atol=1e-15), nm


def test_cleanup_threshold_none_keeps_zeros(ops):
    symp, coeff = po.from_strings(["XX", "YY", "XX"], [1, 0, -1])
    xz, c = ops.cleanup(*dev_op(ops, symp, coeff), zero_threshold=None)
    assert xz.shape[0] == 2
    xz, c = ops.cleanup(*dev_op(ops, symp, coeff), zero_threshold=1e-15)
    assert xz.shape[0] == 0


def test_commute_golden(ops, golden):
    for nm in sorted(k for k in golden if k.startswith("commute_")):
        g = golden[nm]
        n = g["a_symp"].shape[1] // 2
        a = ops.pack(torch.from_numpy(g["a_symp"]), n)
        b = ops.pack(torch.from_numpy(g["b_symp"]), n)
        assert np.array_equal(ops.commute(a, b).cpu().numpy(), g["out"]), nm
        assert np.array_equal(ops.commute_mma(a, b).cpu().numpy(), g["out"]), nm
        bits = ops.commute_bits(a, b).cpu().numpy().view(np.uint32)
        N = g["b_symp"].shape[0]
        unp = ((bits[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(bits.shape[0], -1)[:, :N].astype(bool)
        assert np.array_equal(unp, g["out"]), nm
    for nm in sorted(k for k in golden if k.startswith("adj_ref_")):
        g = golden[nm]
        a = ops.pack(torch.from_numpy(g["symp"]), g["symp"].shape[1] // 2)
        assert np.array_equal(ops.commute(a, a).cpu().numpy(), g["adj"]), nm


@pytest.mark.parametrize("n,m1,m2", [(1, 5, 7), (36, 700, 513), (64, 128, 256), (100, 130, 300), (1000, 300, 257),
                                     (1100, 70, 50), (1500, 40, 33), (2100, 129, 257)])
def test_commute_random_both_kernels(ops, n, m1, m2):
    """Bit-packed kernel and tcgen05 int8 tensor-core kernel against the oracle, bit-exact."""
    a_s, _ = po.random_operator(n, m1, seed=n)
    b_s, _ = po.random_operator(n, m2, seed=n + 1)
    a = ops.pack(torch.from_numpy(a_s), n)
    b = ops.pack(torch.from_numpy(b_s), n)
    ref = po.commutes_termwise(a_s, b_s)
    assert np.array_equal(ops.commute_packed(a, b).cpu().numpy(), ref)
    assert np.array_equal(ops.commute_mma(a, b).cpu().numpy(), ref)
    assert np.array_equal(ops.commute(a, b).cpu().numpy(), ref)


def test_commute_mma_unpitched_abi_ragged(ops):
    """sym_commute_mma with the natural pitch N (odd: rows unaligned, per-byte epilogue) must equal the pitched call."""
    import ctypes
    from symmer_b200 import _cabi
    n, m1, m2 = 36, 300, 2599
    a_s, _ = po.random_operator(n, m1, seed=4)
    b_s, _ = po.random_operator(n, m2, seed=5)
    a = ops.pack(torch.from_numpy(a_s), n)
    b = ops.pack(torch.from_numpy(b_s), n)
    out = torch.empty((m1, m2), dtype=torch.uint8, device=a.device)
    L = ops.lib()
    ws = ops.workspace(L.sym_commute_mma_ws_bytes(m1, m2, 1))
    _cabi.check(L.sym_commute_mma(ctypes.c_void_p(a.data_ptr()), m1, ctypes.c_void_p(b.data_ptr()), m2, 1,
                                  ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(ws.data_ptr()), ws.numel(),
                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    ref = po.commutes_termwise(a_s, b_s)
    assert np.array_equal(out.cpu().numpy().astype(bool), ref)
    assert np.array_equal(ops.commute_mma(a, b).cpu().numpy(), ref)


def test_commute_large_dispatches_to_tensor_cores(ops):
    n, M = 200, 3000                                   # 9e6 pairs > MMA_MIN_PAIRS
    a_s, _ = po.random_operator(n, M, seed=9)
    a = ops.pack(torch.from_numpy(a_s), n)
    adj = ops.commute(a, a).cpu().numpy()
    assert np.array_equal(adj, po.commutes_termwise(a_s, a_s))
    assert np.array_equal(adj, adj.T) and adj.diagonal().all()


def test_gf2_golden(ops, golden):
    for nm in sorted(k for k in golden if k.startswith("gf2_rand_")):
        g = golden[nm]
        m = g["matrix"]
        bits = ops.pack_matrix(torch.from_numpy(m))
        piv = ops.rref_packed(bits, m.shape[1])
        red = ops.unpack_matrix(bits, m.shape[1]).cpu().numpy()
        assert np.array_equal(red, g["rref_norows"]), nm
        exp_piv = np.array([np.flatnonzero(r)[0] if r.any() else -1 for r in g["rref_norows"]])
        assert np.array_equal(piv.cpu().numpy(), exp_piv), nm


def _rref_check(ops, m):
    bits = ops.pack_matrix(torch.from_numpy(m))
    piv = ops.rref_packed(bits, m.shape[1]).cpu().numpy()
    ref = po._rref_binary(m)
    assert np.array_equal(ops.unpack_matrix(bits, m.shape[1]).cpu().numpy(), ref)
    assert np.array_equal(piv, np.array([np.flatnonzero(r)[0] if r.any() else -1 for r in ref]))


@pytest.mark.parametrize("variant", [1, 0])
def test_gf2_large_path(ops, variant):
    """Matrices beyond one CTA's shared memory: blocked panels (variant 1, default) and the
    one-pivot-per-sweep form (variant 0), both bit-exact with the row-driven rule of _rref_binary."""
    rng = np.random.default_rng(3)
    try:
        ops.set_tuning(5, variant)
        _rref_check(ops, rng.random((300, 9000)) < 0.02)          # wide, sparse: 300 x 141 words
        _rref_check(ops, rng.random((131, 20000)) < 0.5)          # wide, dense, rows not a multiple of the panel
        tall = rng.random((3000, 700)) < 0.3                      # tall: rank 700, most rows reduce to zero
        tall[50:60] = 0                                           # zero rows inside a panel
        tall[100] = tall[7]                                       # duplicate rows
        _rref_check(ops, tall)
        low = (rng.random((400, 12)) < 0.5).astype(np.uint8) @ (rng.random((12, 8000)) < 0.5).astype(np.uint8) % 2
        _rref_check(ops, low.astype(bool))                        # rank <= 12: panels full of dependent rows
        _rref_check(ops, rng.random((40, 50000)) < 0.001)         # panels of fewer rows (4 per panel at 782 words)
    finally:
        ops.set_tuning(5, 1)


def test_apply_expval_csr(ops, golden):
    for nm in sorted(k for k in golden if k.startswith("matrix_rand_")):
        g = golden[nm]
        n = g["symp"].shape[1] // 2
        xz, c = dev_op(ops, g["symp"], g["coeff"])
        xm, zm, cp = ops.term_masks_sorted(xz, c, n)
        psi = torch.from_numpy(g["psi"]).cuda()
        y = ops.apply_dense(xm, zm, cp, n, psi).cpu().numpy()
        assert np.allclose(y, g["Hpsi"], rtol=1e-12, atol=1e-13), nm
        e = complex(ops.expval_dense(xm, zm, cp, n, psi).cpu().numpy())
        assert np.isclose(e, g["expval"][0], rtol=1e-12), nm
        half = (1 << n) // 2
        if half:
            e2 = ops.expval_dense(xm, zm, cp, n, psi, 0, half) + ops.expval_dense(xm, zm, cp, n, psi, half, 1 << n)
            assert np.isclose(complex(e2.cpu().numpy()), g["expval"][0], rtol=1e-12), nm
        if g["dense"].size:
            import scipy.sparse as sps
            data, indices, indptr = [t.cpu().numpy() for t in ops.to_csr(xm, zm, cp, n)]
            M = sps.csr_matrix((data, indices, indptr), shape=(1 << n, 1 << n))
            assert M.has_canonical_format
            assert np.allclose(M.toarray(), g["dense"], rtol=1e-13, atol=1e-13), nm


def _rotate_dev(ops, symp, coeff, q_symp, angle):
    """host logic of _rotate_by_single_Pword + cleanup, on device tensors (mirrors symmer_b200.base)."""
    n = symp.shape[1] // 2
    xz, c = dev_op(ops, symp, coeff)
    q = ops.pack(torch.from_numpy(q_symp.reshape(1, -1)), n)
    if angle is None:
        angle = np.pi / 2
    multiple = angle * 2 / np.pi
    int_part = round(multiple)
    if abs(int_part - multiple) <= 1e-18:
        sign = -1.0 if int_part in [2, 3] else 1.0
        oxz, oc = ops.rotate(xz, c, q, 0.0, 0.0, 1 if int_part % 2 else 2, sign)
    else:
        oxz, oc = ops.rotate(xz, c, q, np.cos(angle), np.sin(angle), 0)
    oxz, oc = ops.cleanup(oxz, oc)
    return host_op(ops, oxz, oc, n)


def test_rotations_golden(ops, golden):
    names = sorted(k for k in golden if k.startswith("rot_single_"))
    assert len(names) >= 40
    for nm in names:
        g = golden[nm]
        ang = None if np.isnan(g["angle"][0]) else float(g["angle"][0])
        s, cc = _rotate_dev(ops, g["symp"], g["coeff"], g["q_symp"][0], ang)
        ok, why = po.compare_term_sets(s, cc, g["out_symp"], g["out_coeff"], scale=np.abs(g["coeff"]).max())
        assert ok, (nm, why)


@pytest.mark.parametrize("n", [3, 64, 100, 700, 1000, 1100, 2100])
def test_rotate_split_tables_and_fused_rotation(ops, n):
    """sym_rotate_split: stable (commuting | anticommuting) partition whose sketch / Y-count tables equal
    sym_sketch_rows / sym_ycount of the partitioned rows; then the fused rotation + dedup against the oracle."""
    M = 777
    s, c = po.random_operator(n, M, seed=n)
    s[500:] = s[:277]                                        # duplicate rows
    q, _ = po.random_operator(n, 1, seed=n + 5)
    xz, cc = dev_op(ops, s, c)
    qxz = ops.pack(torch.from_numpy(q), n)
    sxz, sc, sk, yc, n_comm = ops.rotate_split(xz, cc, qxz)
    comm = po.commutes_termwise(s, q)[:, 0]
    order = np.concatenate([np.flatnonzero(comm), np.flatnonzero(~comm)])
    assert n_comm == int(comm.sum())
    assert np.array_equal(ops.unpack(sxz, n).cpu().numpy(), s[order])
    assert np.array_equal(sc.cpu().numpy(), c[order])
    assert torch.equal(sk, ops.sketch(sxz))
    assert torch.equal(yc, ops.ycount(sxz))
    for angle in [0.37, -2.2]:
        oxz, oc = ops.rotate_dedup(xz, cc, qxz, np.cos(angle), np.sin(angle))
        ref_s, ref_c = po.perform_rotations(s, c, [(q[0], angle)])
        ok, why = po.compare_term_sets(*host_op(ops, oxz, oc, n), ref_s, ref_c, scale=np.abs(c).max() * 2)
        assert ok, (angle, why)


@pytest.mark.parametrize("n,m1,m2", [(5, 300, 7), (64, 130, 13), (100, 257, 9), (200, 129, 20), (500, 140, 33),
                                     (1000, 260, 45), (1000, 100, 3), (1000, 128, 128), (1100, 30, 9), (40, 1, 50)])
def test_ordered_tile_mode_first_occurrence_order(ops, n, m1, m2):
    """Force the large-product path on small inputs: the ordered-tile mode must give the reference's
    first-occurrence order (rows bit-exact IN ORDER), whatever the tile raggedness; widths it does
    not cover (W = 18 here) fall back to sorted-hash order and still match as a term set."""
    try:
        ops.set_tuning(0, 0)
        tiled = n != 1100 and m1 >= 32      # a one-row A would be > 75 % tile padding: sorted-hash order instead
        a_s, a_c = po.random_operator(n, m1, seed=5 * n + m1)
        b_s, b_c = po.random_operator(n, m2, seed=5 * n + m2 + 1)
        k = min(m1, m2) // 2
        b_s[:k] = a_s[:k]                              # duplicates: identity terms + repeated products
        a_s[m1 // 2:] = a_s[: m1 - m1 // 2]            # and duplicated rows inside A
        for q in (16, 1, 5):
            ops.set_tuning(7, q)
            s, cc, ref_s, ref_c = _check_product(ops, a_s, a_c, b_s, b_c)
            if tiled and len(ref_c) == len(cc):
                assert np.array_equal(s, ref_s)
        # a threshold that drops some singletons and some group sums
        s, cc, ref_s, ref_c = _check_product(ops, a_s, a_c, b_s, b_c, thr=0.8)
        s, cc, ref_s, ref_c = _check_product(ops, a_s, a_c, b_s, b_c, thr=None)
        if tiled:
            assert np.array_equal(s, ref_s)
    finally:
        ops.set_tuning(7, 16)
        ops.set_tuning(0, 1 << 22)


def test_ordered_tile_mode_squares_and_forced_collisions(ops):
    try:
        ops.set_tuning(0, 0)
        a_s, a_c = po.random_operator(1000, 150, seed=1)
        s, cc, ref_s, ref_c = _check_product(ops, a_s, a_c, a_s, a_c)
        comm = po.commutes_termwise(a_s, a_s)
        assert len(cc) == (np.count_nonzero(comm) - 150) // 2 + 1     # anticommuting pairs cancel exactly
        a_s, a_c = po.random_operator(100, 90, seed=11)
        for mask in [0xFFFFFFFFFFFFFFFF, 0xFF00000000000000, 0x0]:
            ops.set_debug_key_mask(mask)
            s, cc, ref_s, ref_c = _check_product(ops, a_s, a_c, a_s, a_c)
            if len(ref_c) == len(cc):
                assert np.array_equal(s, ref_s)
    finally:
        ops.set_debug_key_mask(0xFFFFFFFFFFFFFFFF)
        ops.set_tuning(0, 1 << 22)


def test_mul_blocks_cleanup_matches_block_products(ops):
    """sym_mul_blocks_*: disjoint rectangles of the cross-term grid, survivors block by block in
    (q, p) order; equal rows in different blocks must merge. Checked against the oracle product of
    the same set of cross terms."""
    n, M, N = 1000, 300, 70
    a_s, a_c = po.random_operator(n, M, seed=31)
    b_s, b_c = po.random_operator(n, N, seed=32)
    b_s[:30] = a_s[:30]
    b_s[30:60] = a_s[150:180]
    a, ac = dev_op(ops, a_s, a_c)
    b, bc = dev_op(ops, b_s, b_c)
    blocks = [(0, 130, 40, 70), (130, 131, 0, 40), (131, 300, 0, 35), (0, 100, 0, 40)]
    rows, coeffs = [], []
    for p0, p1, q0, q1 in blocks:          # the same cross terms, in the same order, on the CPU
        r, c = po.cross_terms(a_s[p0:p1], a_c[p0:p1], b_s[q0:q1], b_c[q0:q1])
        rows.append(r)
        coeffs.append(c)
    ref_s, ref_c = po.symplectic_cleanup(np.vstack(rows), np.hstack(coeffs), 1e-15)
    try:
        for limit in (0, 1 << 22):
            for knob6 in (1, 0):
                ops.set_tuning(0, limit)
                ops.set_tuning(6, knob6)
                xz, c, T = ops.mul_blocks_cleanup(a, ac, b, bc, blocks)
                assert T == sum((p1 - p0) * (q1 - q0) for p0, p1, q0, q1 in blocks)
                s, cc = host_op(ops, xz, c, n)
                ok, why = po.compare_term_sets(s, cc, ref_s, ref_c, scale=np.abs(a_c).max() * np.abs(b_c).max())
                assert ok, (limit, knob6, why)
                if knob6 == 1 and len(cc) == len(ref_c):
                    assert np.array_equal(s, ref_s)            # block-by-block first-occurrence order
        with pytest.raises(Exception):
            ops.mul_blocks_cleanup(a, ac, b, bc, [(0, 10, 0, 10), (5, 15, 5, 15)])   # overlapping blocks
    finally:
        ops.set_tuning(0, 1 << 22)
        ops.set_tuning(6, 1)


@pytest.mark.parametrize("onesweep", [1, 0])
def test_record_sort_variants_agree(ops, onesweep):
    """One-sweep passes (decoupled look-back over hundreds of tiles) must give exactly what the
    histogram + scan + scatter form gives: term sets against the oracle, and first-occurrence order
    (a stable sort) in ordered-tile mode. Also through plain cleanup and the block-list product."""
    try:
        ops.set_tuning(8, onesweep)
        ops.set_tuning(0, 0)
        n, m1, m2 = 40, 2500, 420                       # 1.05e6 cross terms = 257 sort tiles, one word per block
        a_s, a_c = po.random_operator(n, m1, seed=77)
        b_s, b_c = po.random_operator(n, m2, seed=78)
        b_s[:200] = a_s[:200]
        a_s[1250:] = a_s[:1250]
        s, cc, ref_s, ref_c = _check_product(ops, a_s, a_c, b_s, b_c)
        if len(ref_c) == len(cc):
            assert np.array_equal(s, ref_s)
        a_s, a_c = po.random_operator(1000, 300, seed=79)
        b_s, b_c = po.random_operator(1000, 200, seed=80)
        b_s[:50] = a_s[:50]
        s, cc, ref_s, ref_c = _check_product(ops, a_s, a_c, b_s, b_c)
        if len(ref_c) == len(cc):
            assert np.array_equal(s, ref_s)
        # block list of 8 and of 9 blocks
        a, ac = dev_op(ops, a_s, a_c)
        b, bc = dev_op(ops, b_s, b_c)
        for nb in (8, 9):
            pb = np.linspace(0, 300, nb + 1).astype(int)
            blocks = [(int(pb[i]), int(pb[i + 1]), 0 if i % 2 else 100, 100 if i % 2 else 200) for i in range(nb)]
            rows, coeffs = [], []
            for p0, p1, q0, q1 in blocks:
                r, c = po.cross_terms(a_s[p0:p1], a_c[p0:p1], b_s[q0:q1], b_c[q0:q1])
                rows.append(r)
                coeffs.append(c)
            ref_s, ref_c = po.symplectic_cleanup(np.vstack(rows), np.hstack(coeffs), 1e-15)
            xz, c, T = ops.mul_blocks_cleanup(a, ac, b, bc, blocks)
            s, cc = host_op(ops, xz, c, 1000)
            ok, why = po.compare_term_sets(s, cc, ref_s, ref_c, scale=np.abs(a_c).max() * np.abs(b_c).max())
            assert ok, (nb, why)
            if len(cc) == len(ref_c):
                assert np.array_equal(s, ref_s)
        # plain cleanup of 2e5 stored rows with many duplicates: first-occurrence order
        rng = np.random.default_rng(5)
        base_s, base_c = po.random_operator(200, 50000, seed=81)
        idx = rng.integers(0, 50000, size=200000)
        big_s, big_c = base_s[idx], rng.standard_normal(200000) + 1j * rng.standard_normal(200000)
        ref_s, ref_c = po.symplectic_cleanup(big_s, big_c, 1e-15)
        xz, c = ops.cleanup(*dev_op(ops, big_s, big_c))
        s, cc = host_op(ops, xz, c, 200)
        assert np.array_equal(s, ref_s)
        assert np.allclose(cc, ref_c, rtol=1e-12, atol=1e-12)
    finally:
        ops.set_tuning(8, 1)
        ops.set_tuning(0, 1 << 22)


def test_bench_size_product_properties(ops):
    """BASELINE config C5/8 at FULL size (1000 q, 12 500 x 10 000 terms = 1.25e8 cross terms, 34 GB of output),
    checked through size-independent properties: random 1000-qubit rows never collide, so every cross term
    survives and — first-occurrence order — output row t = q*M + p must be A[p] ^ B[q] bit for bit; a block of
    64 rows of A against all of B is compared with the materialised cross terms (rows bit-exact, coefficients
    1e-14), and 2e6 random rows with the XOR of their operands."""
    free, _ = torch.cuda.mem_get_info()
    if free < 60 * 2 ** 30:
        pytest.skip("needs 60 GB of free device memory")
    n, M, N = 1000, 12500, 10000
    a_s, a_c = po.random_operator(n, M, seed=100)
    b_s, b_c = po.random_operator(n, N, seed=7)
    a, ac = dev_op(ops, a_s, a_c)
    b, bc = dev_op(ops, b_s, b_c)
    xz, c = ops.mul_cleanup(a, ac, b, bc)
    assert xz.shape[0] == M * N and c.shape[0] == M * N
    # (1) a 64-row block of A against all of B, against the materialised cross terms of the same block
    p0 = 4321
    blk_xz, blk_c = ops.cross_mul(a[p0:p0 + 64].contiguous(), ac[p0:p0 + 64].contiguous(), b, bc)   # t' = q*64 + p'
    t = (torch.arange(N, device=a.device).repeat_interleave(64) * M + p0 + torch.arange(64, device=a.device).repeat(N))
    assert torch.equal(xz[t], blk_xz)
    assert torch.allclose(c[t], blk_c, rtol=1e-14, atol=0)
    # ... and that block against the oracle on a slice small enough for the CPU
    ref_rows, ref_c = po.cross_terms(a_s[p0:p0 + 64], a_c[p0:p0 + 64], b_s[:50], b_c[:50])
    assert np.array_equal(ops.unpack(blk_xz[:3200].contiguous(), n).cpu().numpy(), ref_rows)
    assert np.allclose(blk_c[:3200].cpu().numpy(), ref_c, rtol=1e-14, atol=0)
    # (2) 2e6 random output rows equal the XOR of their operands
    g = torch.Generator(device=a.device)
    g.manual_seed(0)
    ts = torch.randint(0, M * N, (2_000_000,), device=a.device, generator=g)
    assert torch.equal(xz[ts], a[ts % M] ^ b[ts // M])
    # (3) |coefficient| of every output term = |a_p| |b_q| (phases are powers of i): a checksum over all 1.25e8 terms
    mag = (ac.abs()[None, :] * bc.abs()[:, None]).reshape(-1)
    assert torch.allclose(c.abs(), mag, rtol=1e-13, atol=0)
    del xz, c, mag
    ops.release_workspace()
    torch.cuda.empty_cache()


def test_sorted_hash_order_path(ops):
    """Force the large-product path (output in sorted-hash order) on small inputs."""
    try:
        ops.set_tuning(0, 0)
        ops.set_tuning(6, 0)
        for n, m1, m2 in [(5, 20, 7), (64, 30, 13), (1000, 60, 45)]:
            a_s, a_c = po.random_operator(n, m1, seed=3 * n + m1)
            b_s, b_c = po.random_operator(n, m2, seed=3 * n + m2 + 7)
            _check_product(ops, a_s, a_c, b_s, b_c)
        a_s, a_c = po.random_operator(100, 90, seed=11)
        _check_product(ops, a_s, a_c, a_s, a_c)
        for mask in [0xFF00000000000000, 0x0]:
            ops.set_debug_key_mask(mask)
            _check_product(ops, a_s, a_c, a_s, a_c)
    finally:
        ops.set_debug_key_mask(0xFFFFFFFFFFFFFFFF)
        ops.set_tuning(0, 1 << 22)
        ops.set_tuning(6, 1)


@pytest.mark.parametrize("log2g", [0, 1, 2, 3])
def test_record_exchange_blocks_single_gpu(ops, log2g):
    """The multi-GPU product path on one device: block-wise records, partition by owner, per-owner
    dedup. The union over owners must equal the oracle product, and owners must be disjoint."""
    n, M, N = 70, 96, 41
    a_s, a_c = po.random_operator(n, M, seed=21)
    b_s, b_c = po.random_operator(n, N, seed=22)
    b_s[:20] = a_s[:20]                                   # force duplicates across blocks
    ref_s, ref_c = po.multiply_by_operator(a_s, a_c, b_s, b_c)
    a, ac = dev_op(ops, a_s, a_c)
    b, bc = dev_op(ops, b_s, b_c)
    G = 1 << log2g
    bounds = np.linspace(0, M, G + 1).astype(int)
    per_owner = [[] for _ in range(G)]
    for r in range(G):                                    # "rank r" generates its block
        recs = ops.pair_records(a, int(bounds[r]), int(bounds[r + 1]), b)
        part, counts = ops.partition_records(recs, log2g)
        counts = counts.cpu().numpy()
        assert counts.sum() == recs.numel()
        offs = np.concatenate([[0], np.cumsum(counts)])
        for o in range(G):
            per_owner[o].append(part[offs[o]:offs[o + 1]])
    rows, coeffs = [], []
    for o in range(G):                                    # "rank o" dedups what it owns
        mine = torch.cat(per_owner[o]).contiguous()
        if log2g:
            assert bool(((mine.view(torch.int64) >> (64 - log2g)) & (G - 1) == o).all())
        xz, c = ops.dedup_records(mine, a, ac, b, bc)
        s, cc = host_op(ops, xz, c, n)
        rows.append(s)
        coeffs.append(cc)
    s = np.vstack(rows)
    cc = np.hstack(coeffs)
    assert len(np.unique(s, axis=0)) == len(s)            # owners hold disjoint rows
    ok, why = po.compare_term_sets(s, cc, ref_s, ref_c, scale=np.abs(a_c).max() * np.abs(b_c).max())
    assert ok, why


def test_owner_classes_are_linear_and_partition_is_stable(ops):
    """Ownership must be GF(2)-linear in the row (class(a^b) = class(a)^class(b)) and the class
    grouping a stable permutation with the right counts."""
    rng = np.random.default_rng(5)
    for n, m in [(3, 300), (64, 300), (200, 300), (1000, 300), (2100, 300), (64, 10000), (1000, 10000)]:   # 10 000: 3 tiles
        a = rng.random((m, 2 * n)) < 0.3
        b = rng.random((m, 2 * n)) < 0.3
        for lg in [0, 1, 3, 8]:
            ca = ops.owner_classes(ops.pack(torch.from_numpy(a), n), lg).cpu().numpy()
            cb = ops.owner_classes(ops.pack(torch.from_numpy(b), n), lg).cpu().numpy()
            cab = ops.owner_classes(ops.pack(torch.from_numpy(a ^ b), n), lg).cpu().numpy()
            assert np.array_equal(ca ^ cb, cab)
            assert ca.max(initial=0) < (1 << lg)
        if n >= 64:
            assert len(np.unique(ca)) > 100                           # 8 bits of 300 random rows: well spread
        coeff = rng.standard_normal(m) + 1j * rng.standard_normal(m)
        xz, c = dev_op(ops, a, coeff)
        cls = ops.owner_classes(xz, 3).cpu().numpy()
        p_xz, p_c, perm, counts = ops.class_partition(xz, c, 3)
        order = np.argsort(cls, kind="stable")
        assert np.array_equal(perm.cpu().numpy(), order)
        assert np.array_equal(counts.cpu().numpy(), np.bincount(cls, minlength=8))
        assert np.array_equal(ops.unpack(p_xz, n).cpu().numpy(), a[order])
        assert np.array_equal(p_c.cpu().numpy(), coeff[order])


@pytest.mark.parametrize("log2g", [0, 1, 2, 3])
def test_exchange_free_owner_product_single_gpu(ops, log2g):
    """The default multi-GPU product path on one device: every "rank" computes the part of the
    product it owns from the full operands, with no exchange. The union over owners must equal the
    oracle product, every cross term must be generated exactly once, and owners must be disjoint."""
    from symmer_b200 import dist as sdist
    for n, M, N in [(70, 96, 41), (1000, 130, 77), (4, 40, 40)]:
        a_s, a_c = po.random_operator(n, M, seed=21)
        b_s, b_c = po.random_operator(n, N, seed=22)
        b_s[:20] = a_s[:20]                                   # duplicates across class blocks
        ref_s, ref_c = po.multiply_by_operator(a_s, a_c, b_s, b_c)
        a, ac = dev_op(ops, a_s, a_c)
        b, bc = dev_op(ops, b_s, b_c)
        rows, coeffs, generated = [], [], 0
        for r in range(1 << log2g):
            xz, c, info = sdist.owned_product(a, ac, b, bc, log2g, r)
            generated += info["cross_terms_generated"]
            if xz.shape[0]:
                assert bool((ops.owner_classes(xz, log2g) == r).all())
            s, cc = host_op(ops, xz, c, n)
            rows.append(s)
            coeffs.append(cc)
        assert generated == M * N
        s = np.vstack(rows)
        cc = np.hstack(coeffs)
        assert len(np.unique(s, axis=0)) == len(s)
        ok, why = po.compare_term_sets(s, cc, ref_s, ref_c, scale=np.abs(a_c).max() * np.abs(b_c).max())
        assert ok, (n, why)


@pytest.mark.parametrize("n,real", [(11, True), (12, False), (13, True), (14, False), (15, True)])
def test_binned_apply_kernel_matches_oracle_and_4row_kernel(ops, n, real):
    """The Walsh-Hadamard binned kernel (16 / 8 basis rows per thread) against the oracle and against
    the 4-row kernel, on operators whose x groups hold 1..many terms (molecular-like structure)."""
    rng = np.random.default_rng(n)
    n_groups, M = 37, 400
    xs = rng.random((n_groups, n)) < 0.4
    xs[0] = False                                               # a diagonal group
    grp = np.concatenate([np.arange(n_groups), rng.integers(0, n_groups, size=M - n_groups)])
    symp = np.hstack([xs[grp], rng.random((M, n)) < 0.5])
    symp = np.unique(symp, axis=0)
    M = symp.shape[0]
    if real:   # real phased coefficients: only terms with an even number of Y survive, like a real Hamiltonian
        symp = symp[(po.y_count(symp) % 2) == 0]
        M = symp.shape[0]
        coeff = rng.standard_normal(M).astype(complex)
    else:
        coeff = rng.standard_normal(M) + 1j * rng.standard_normal(M)
    psi = rng.standard_normal(1 << n) + 1j * rng.standard_normal(1 << n)
    psi /= np.linalg.norm(psi)
    ref = po.pauli_apply_dense(symp, coeff, psi)
    xz, c = dev_op(ops, symp, coeff)
    xm, zm, cp = ops.term_masks_sorted(xz, c, n)
    assert bool(ops._is_real(cp)) == real
    psi_d = torch.from_numpy(psi).cuda()
    out = {}
    try:
        for variant in (1, 0):
            ops.set_tuning(4, variant)
            y = ops.apply_dense(xm, zm, cp, n, psi_d).cpu().numpy()
            assert np.allclose(y, ref, rtol=1e-12, atol=1e-13), variant
            e = complex(ops.expval_dense(xm, zm, cp, n, psi_d).cpu().numpy())
            assert np.isclose(e, np.vdot(psi, ref), rtol=1e-12, atol=1e-14), variant
            quarter = (1 << n) // 4                             # sharded row ranges (multi-GPU expval)
            parts = sum(complex(ops.expval_dense(xm, zm, cp, n, psi_d, k * quarter, (k + 1) * quarter).cpu().numpy())
                        for k in range(4))
            assert np.isclose(parts, e, rtol=1e-12, atol=1e-14), variant
            out[variant] = y
    finally:
        ops.set_tuning(4, 1)
    assert np.allclose(out[0], out[1], rtol=1e-13, atol=1e-14)
    # symmetric (Hermitian, real phased coefficients) expectation-value mode: on for `real`, never for complex
    assert bool(getattr(cp, "_sym_hermitian", False)) == real
    if real:
        e_ref = np.vdot(psi, ref)
        assert abs(e_ref.imag) < 1e-12
        try:
            ops.use_symmetric_expval = False
            e_plain = complex(ops.expval_dense(xm, zm, cp, n, psi_d).cpu().numpy())
        finally:
            ops.use_symmetric_expval = True
        e_sym = complex(ops.expval_dense(xm, zm, cp, n, psi_d).cpu().numpy())
        assert cp._sym_table is not None and e_sym.imag == 0.0
        assert np.isclose(e_sym.real, e_ref.real, rtol=1e-12, atol=1e-14)
        assert np.isclose(e_plain, e_ref, rtol=1e-12, atol=1e-14)
        n_parts = max(1, (1 << n) // 2048)
        step = (1 << n) // n_parts
        parts = sum(complex(ops.expval_dense(xm, zm, cp, n, psi_d, k * step, (k + 1) * step).cpu().numpy())
                    for k in range(n_parts))
        assert np.isclose(parts.real, e_ref.real, rtol=1e-12, atol=1e-14)      # shards still add up to the total
