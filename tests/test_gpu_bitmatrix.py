"""Exact tests of the bit-matrix kernels: the packed commutation kernels of symmer_b200/csrc/commute.cu (sym_commute,
sym_commute_bits, sym_commute_qwc, sym_mirror_upper), the tensor-core kernel of commute_mma.cu
(sym_commute_mma_pitched) and the GF(2) kernels of gf2.cu (sym_rref, sym_bit_transpose, sym_or_rows), and their
dispatch in symmer_b200.ops.

Every result is a bit or a byte, so every comparison is exact against a NumPy restatement. Every output the C ABI
writes lies inside a device buffer filled with a sentinel byte, with guard bytes before and after it and the pitch
slack of its rows kept: a test fails when a kernel writes a byte it was not meant to, and a wrong write still lands in
memory the test allocated."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import pauli_oracle as po

gpu = pytest.mark.gpu

SENT = 0xA5          # sentinel byte of every guarded output
PRE = 256            # guard bytes before an output
POST = 4096          # guard bytes after an output
COM_ICH = 64         # A rows per CTA of the packed kernels (commute.cu)
MMA_M = 128          # A rows per CTA of the tensor-core kernel (commute_mma.cu)
GRID_Y = 65535       # grid.y limit: the packed and tensor-core entries loop over slabs of A beyond it
PANEL_CAP = 200 * 1024   # shared-memory budget of the one-CTA and panel rref kernels (gf2.cu)
SYM_E_INVALID = -1
SYM_E_WORKSPACE = -3


# ------------------------------------------------------------------------------------------- NumPy restatements
def ceil32(n):
    return (n + 31) // 32 * 32


def words_for(n):
    return max(1, (n + 63) // 64)


def rand_words(rng, shape):
    return rng.integers(0, np.iinfo(np.uint64).max, size=shape, dtype=np.uint64, endpoint=True)


def pack_bits(m, Cw):
    """bool[R, C] -> uint64[R, Cw]: column j is bit j % 64 of word j // 64 (the packed row layout)."""
    R, C = m.shape
    full = np.zeros((R, 64 * Cw), dtype=np.uint8)
    full[:, :C] = m
    return np.ascontiguousarray(np.packbits(full, axis=1, bitorder="little")).view("<u8").reshape(R, Cw)


def unpack_bits(w):
    """uint64[R, Cw] -> bool[R, 64 * Cw]."""
    w = np.ascontiguousarray(w, dtype="<u8")
    return np.unpackbits(w.view(np.uint8).reshape(w.shape[0], -1), axis=1, bitorder="little").astype(bool)


def pack_symp(symp):
    """bool[M, 2n] symplectic rows -> uint64[M, 2W] packed rows (X words, then Z words)."""
    n = symp.shape[1] // 2
    W = words_for(n)
    return np.concatenate([pack_bits(symp[:, :n], W), pack_bits(symp[:, n:], W)], axis=1)


def random_rows(rng, M, n):
    """M packed rows over n qubits, uniform on the Paulis; the bits past n are 0."""
    W = words_for(n)
    w = rand_words(rng, (M, 2 * W))
    if n % 64:
        keep = np.uint64((1 << (n % 64)) - 1)
        w[:, W - 1] &= keep
        w[:, 2 * W - 1] &= keep
    return w


def structured_b(rng, a, N, n):
    """N rows: copies of A's rows (which commute with them), A's rows with one bit of one qubit flipped (one Pauli
    apart: they commute with the original iff its other bit on that qubit is 0), then random rows."""
    W = a.shape[1] // 2
    k = min(a.shape[0], N // 3)
    b = random_rows(rng, N, n)
    b[:k] = a[:k]
    b[k:2 * k] = a[:k]
    q = rng.integers(0, n, size=k)
    half = rng.integers(0, 2, size=k)
    b[k + np.arange(k), half * W + q // 64] ^= np.uint64(1) << (q % 64).astype(np.uint64)
    return b


def commute_ref(a, b):
    """uint8[M, N]: 1 where the symplectic product of A[i] and B[j] is even, i.e. the parity of popcount(A & swap(B))
    over the 2W words (swap exchanges B's X and Z words)."""
    M, N, W = a.shape[0], b.shape[0], a.shape[1] // 2
    swap = np.concatenate([b[:, W:], b[:, :W]], axis=1)
    out = np.empty((M, N), dtype=np.uint8)
    step = max(1, (1 << 22) // max(1, N * 2 * W))
    for i0 in range(0, M, step):
        cnt = np.bitwise_count(a[i0:i0 + step, None, :] & swap[None, :, :]).sum(axis=2, dtype=np.int64)
        out[i0:i0 + step] = (cnt & 1) == 0
    return out


def qwc_ref(a, b):
    """uint8[M, N]: the oracle's qubit-wise rule on packed words. On the qubits where both rows are not the identity
    (non_I) the X bits and the Z bits must agree."""
    M, N, W = a.shape[0], b.shape[0], a.shape[1] // 2
    out = np.empty((M, N), dtype=np.uint8)
    step = max(1, (1 << 22) // max(1, N * W))
    for i0 in range(0, M, step):
        ax, az = a[i0:i0 + step, None, :W], a[i0:i0 + step, None, W:]
        bx, bz = b[None, :, :W], b[None, :, W:]
        non_i = (ax | az) & (bx | bz)
        out[i0:i0 + step] = ~(((ax ^ bx) | (az ^ bz)) & non_i).any(axis=2)
    return out


def bits_ref(byte_ref):
    """The bit-packed output of sym_commute_bits: row stride ceil(N/32) uint32, bit j % 32 of word j // 32, bits
    past N zero."""
    M, N = byte_ref.shape
    stride = (N + 31) // 32
    full = np.zeros((M, 32 * stride), dtype=np.uint8)
    full[:, :N] = byte_ref
    return np.ascontiguousarray(np.packbits(full, axis=1, bitorder="little")).view("<u4").reshape(M, stride)


def mirror_ref(m, M, blk):
    """mirror_upper_kernel restated on a byte matrix with any pitch: for every 32 x 32 tile (ti, tj) whose block
    column is right of its block row's (bj > bi), or inside a diagonal block strictly above the diagonal tile
    (bj == bi and tj > ti), element (r, c) is copied to (c, r). Diagonal tiles, the tiles it writes and the
    padding columns are left as they are."""
    out = m.copy()
    r, c = np.meshgrid(np.arange(M), np.arange(M), indexing="ij")
    ti, tj = r // 32, c // 32
    bi, bj = ti * 32 // blk, tj * 32 // blk
    src = (bj > bi) | ((bj == bi) & (tj > ti))
    out[c[src], r[src]] = m[r[src], c[src]]
    return out


def rref_ref(words, C):
    """po._rref_binary on the first C columns: (reduced packed rows, pivot column per row or -1)."""
    R, Cw = words.shape
    red = po._rref_binary(unpack_bits(words)[:, :C])
    piv = np.array([np.flatnonzero(row)[0] if row.any() else -1 for row in red], dtype=np.int32)
    return pack_bits(red, Cw), piv


def transpose_ref(words, R, Cw_out):
    """sym_bit_transpose restated: rows [0, R) of an uint64[., Cw_in] matrix -> uint64[Cw_in * 64, Cw_out]."""
    m = unpack_bits(words[:R])
    return pack_bits(np.ascontiguousarray(m.T), Cw_out)


def gf2_matrix(rng, R, Cw, C, density=0.5):
    """R packed rows of C columns: row 1 duplicates row 0, the last row has bits in the last word only (its pivot
    is there), and with enough rows row 2 is zero and row 3 has only the last column set; the bits past C are 0."""
    m = rng.random((R, C)) < density
    if R >= 3:
        m[1] = m[0]
        lo = 64 * (Cw - 1)
        m[R - 1] = False
        m[R - 1, lo:C] = rng.random(C - lo) < 0.5
        m[R - 1, C - 1] = True
    if R >= 5:
        m[2] = False
    if R >= 6:
        m[3] = False
        m[3, C - 1] = True
    return pack_bits(m, Cw)


# ------------------------------------------------------------------------------------------- device helpers
def _vp(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check(rc):
    from symmer_b200 import _cabi
    _cabi.check(rc)


def _dev(a):
    a = np.ascontiguousarray(a)
    return torch.from_numpy(a.view(np.int64) if a.dtype == np.uint64 else a).cuda()


class Guarded:
    """nbytes of output `offset` bytes after a 256-byte aligned point of a sentinel-filled device buffer, with PRE
    guard bytes before (plus the offset) and POST after."""

    def __init__(self, nbytes, offset=0, fill=None):
        self.n, self.off = int(nbytes), PRE + offset
        self.buf = torch.full((self.off + self.n + POST,), SENT, dtype=torch.uint8, device="cuda")
        if fill is not None:
            self.buf[self.off:self.off + self.n] = torch.from_numpy(np.ascontiguousarray(fill).view(np.uint8).ravel())

    @property
    def ptr(self):
        return ctypes.c_void_p(self.buf.data_ptr() + self.off)

    def host(self, what=""):
        """The output bytes, after checking that no guard byte changed."""
        h = self.buf.cpu().numpy()
        bad = np.flatnonzero(h[:self.off] != SENT)
        assert bad.size == 0, (f"{what}: {bad.size} guard bytes before the output written, "
                               f"first {self.off - bad[0]} B before it")
        bad = np.flatnonzero(h[self.off + self.n:] != SENT)
        assert bad.size == 0, (f"{what}: {bad.size} guard bytes after the output written, "
                               f"bytes {bad[0]}..{bad[-1]} past its end")
        return h[self.off:self.off + self.n]


def assert_equal(got, ref, what):
    bad = np.argwhere(got != ref)
    if bad.size:
        at = tuple(bad[0])
        raise AssertionError(f"{what}: {len(bad)} wrong entries, first at {at}: {got[at]} vs {ref[at]}")


@pytest.fixture(scope="module")
def ops():
    import symmer_b200.ops as o
    o.device()
    return o


# ------------------------------------------------------------------------------------------- 1. the references
@pytest.mark.parametrize("n", [1, 3, 63, 64, 65, 130])
def test_commute_references_match_the_oracle(n):
    """The packed restatements of commutes_termwise and qubitwise_commutes_termwise against the oracle on random
    and structured rows (copies, one Pauli apart, identities), and the bit-packed layout against the byte matrix."""
    rng = np.random.default_rng(n)
    M, N = 9, 23
    a_symp = rng.random((M, 2 * n)) < 0.5
    a_symp[1] = False
    b_symp = rng.random((N, 2 * n)) < 0.5
    b_symp[:M] = a_symp
    b_symp[M:2 * M] = a_symp
    b_symp[M + np.arange(M), rng.integers(0, 2 * n, M)] ^= True
    a, b = pack_symp(a_symp), pack_symp(b_symp)
    assert np.array_equal(unpack_bits(a[:, :words_for(n)])[:, :n], a_symp[:, :n])
    ref = commute_ref(a, b)
    assert np.array_equal(ref.astype(bool), po.commutes_termwise(a_symp, b_symp))
    assert ref[:, :M].diagonal().all() and 0 < ref.sum() < ref.size
    assert np.array_equal(qwc_ref(a, b).astype(bool), po.qubitwise_commutes_termwise(a_symp, b_symp))
    sb = structured_b(rng, a, N, n)
    k = N // 3
    assert np.array_equal(sb[:k], a[:k]) and (np.bitwise_count(sb[k:2 * k] ^ a[:k]).sum(axis=1) == 1).all()
    bits = bits_ref(ref)
    assert bits.shape == (M, 1)
    unpacked = np.unpackbits(bits.view(np.uint8).reshape(M, -1), axis=1, bitorder="little")
    assert np.array_equal(unpacked[:, :N], ref) and not unpacked[:, N:].any()


@pytest.mark.parametrize("M,blk", [(1, 32), (33, 32), (100, 64), (300, 64), (300, 2048)])
def test_mirror_reference_recovers_a_symmetric_matrix(M, blk):
    """The restated tile rule: it leaves a symmetric matrix unchanged, and when everything below the block diagonal
    (and below the diagonal tiles inside it) is junk, it rebuilds the symmetric matrix from the rest."""
    rng = np.random.default_rng(M + blk)
    s = rng.integers(0, 2, size=(M, M), dtype=np.uint8)
    s = s | s.T
    assert np.array_equal(mirror_ref(s, M, blk), s)
    r, c = np.meshgrid(np.arange(M), np.arange(M), indexing="ij")
    ti, tj = r // 32, c // 32
    kept = (tj * 32 // blk > ti * 32 // blk) | ((tj * 32 // blk == ti * 32 // blk) & (tj >= ti))
    junk = np.where(kept, s, rng.integers(2, 255, size=(M, M), dtype=np.uint8))
    assert np.array_equal(mirror_ref(junk, M, blk), s)


@pytest.mark.parametrize("R,Cw,C", [(1, 1, 1), (6, 1, 64), (12, 2, 100), (40, 3, 150)])
def test_gf2_references_are_consistent(R, Cw, C):
    """The rref restatement: each nonzero row's pivot is its first set column and a unit column of the result,
    zero rows have pivot -1, the duplicate row reduces to zero; transposing twice gives the rows back; the OR of
    rows equals NumPy's reduction."""
    rng = np.random.default_rng(R)
    w = gf2_matrix(rng, R, Cw, C)
    red, piv = rref_ref(w, C)
    m, mr = unpack_bits(w)[:, :C], unpack_bits(red)
    assert not mr[:, C:].any()
    for i, p in enumerate(piv):
        if p >= 0:
            assert not mr[i, :p].any() and mr[:, p].sum() == 1 and mr[i, p]
        else:
            assert not mr[i].any()
    if R >= 3:
        assert piv[1] == -1 and piv[R - 1] >= 64 * (Cw - 1)
    t = transpose_ref(w, R, words_for(R) + 1)
    assert t.shape == (64 * Cw, words_for(R) + 1)
    back = transpose_ref(t, 64 * Cw, Cw)
    assert np.array_equal(back[:R], w) and not back[R:].any()
    assert np.array_equal(np.bitwise_or.reduce(w, axis=0), pack_bits(m.any(axis=0)[None], Cw)[0])


# ------------------------------------------------------------------------------------------- 2. packed kernels
WIDTHS = [1, 2, 3, 4, 5, 8, 9, 15, 16, 17, 32]          # every width template (W < WT inside one), the generic kernel
PACKED_M = [1, 63, 64, 65, 129]
PACKED_N = [1, 31, 32, 33, 255, 256, 257]


def run_packed(ops, d_a, d_b, M, N, W, entry):
    """One packed entry into a guarded buffer: the byte matrix (sym_commute, sym_commute_qwc) or the bit rows
    (sym_commute_bits), after checking that nothing was written outside it."""
    L = ops.lib()
    if entry == "bits":
        stride = (N + 31) // 32
        g = Guarded(4 * M * stride)
        _check(L.sym_commute_bits(_vp(d_a), M, _vp(d_b), N, W, g.ptr, _stream()))
        return g.host(f"sym_commute_bits M={M} N={N} W={W}").view("<u4").reshape(M, stride)
    g = Guarded(M * N)
    fn = L.sym_commute if entry == "bytes" else L.sym_commute_qwc
    _check(fn(_vp(d_a), M, _vp(d_b), N, W, g.ptr, _stream()))
    return g.host(f"sym_commute_{entry} M={M} N={N} W={W}").reshape(M, N)


@gpu
@pytest.mark.parametrize("W", WIDTHS)
def test_packed_kernels_are_exact_on_every_template(ops, W):
    """sym_commute, sym_commute_bits and sym_commute_qwc at every width template and the generic kernel, on row
    counts around the 64-row CTA chunk and column counts around the 32-bit words and the 256-thread CTA: every
    byte and bit exact, the bits past N in each row's last word zero, nothing written past the output."""
    rng = np.random.default_rng(W)
    n = 64 * W - (W % 3) * 7
    a = random_rows(rng, max(PACKED_M), n)
    b = structured_b(rng, a, max(PACKED_N), n)
    refs = {"bytes": commute_ref(a, b), "qwc": qwc_ref(a, b)}
    assert 0 < refs["bytes"].sum() < refs["bytes"].size
    d_a, d_b = _dev(a), _dev(b)
    for M in PACKED_M:
        for N in PACKED_N:
            for entry in ("bytes", "qwc"):
                assert_equal(run_packed(ops, d_a, d_b, M, N, W, entry), refs[entry][:M, :N], (entry, M, N, W))
            assert_equal(run_packed(ops, d_a, d_b, M, N, W, "bits"), bits_ref(refs["bytes"][:M, :N]), ("bits", M, N, W))


@gpu
@pytest.mark.parametrize("M,N,W", [(GRID_Y * COM_ICH + 1, 3, 1), (GRID_Y + 2, 40, 17)])
def test_packed_kernels_loop_over_slabs_of_a(ops, M, N, W):
    """Past the grid.y limit (65535 chunks of 64 rows for W <= 16, 65535 rows for the generic kernel) every entry
    runs A in slabs: the rows of the last slab must land at their own offset in the output."""
    rng = np.random.default_rng(M)
    n = 64 * W
    a = random_rows(rng, M, n)
    b = structured_b(rng, a[-N:].copy(), N, n)
    refs = {"bytes": commute_ref(a, b), "qwc": qwc_ref(a, b)}
    d_a, d_b = _dev(a), _dev(b)
    for entry in ("bytes", "qwc"):
        assert_equal(run_packed(ops, d_a, d_b, M, N, W, entry), refs[entry], (entry, M, N, W))
    assert_equal(run_packed(ops, d_a, d_b, M, N, W, "bits"), bits_ref(refs["bytes"]), ("bits", M, N, W))


@gpu
def test_packed_kernels_write_nothing_for_empty_operands(ops):
    rng = np.random.default_rng(0)
    for W in (1, 17):
        d = _dev(random_rows(rng, 4, 64 * W))
        for M, N in [(0, 4), (4, 0), (0, 0)]:
            for entry in ("bytes", "qwc", "bits"):
                assert run_packed(ops, d, d, M, N, W, entry).size == 0


# ------------------------------------------------------------------------------------------- 3. tensor-core kernel
MMA_WIDTHS = [1, 2, 3, 4, 16, 17, 40]     # stages of 2 words: no reuse, a full ring, reuse with a phase flip, odd/even
MMA_M_LIST = [1, 127, 128, 129, 383]
MMA_N_LIST = [1, 31, 32, 33, 255, 256, 257, 600]


def call_mma(ops, d_a, d_b, M, N, W, pitch, offset=0):
    """sym_commute_mma_pitched into M rows of `pitch` bytes `offset` bytes past a 256-byte boundary: returns the
    rows, after checking the guards and that bytes [ceil32(N), pitch) of every row kept the sentinel."""
    L = ops.lib()
    g = Guarded(M * pitch, offset)
    ws = ops.workspace(L.sym_commute_mma_ws_bytes(M, N, W))
    _check(L.sym_commute_mma_pitched(_vp(d_a), M, _vp(d_b), N, W, g.ptr, pitch, _vp(ws), ws.numel(), _stream()))
    what = f"sym_commute_mma_pitched M={M} N={N} W={W} pitch={pitch} offset={offset}"
    out = g.host(what).reshape(M, pitch)
    slack = out[:, min(pitch, ceil32(N)):]
    bad = np.argwhere(slack != SENT)
    assert bad.size == 0, (f"{what}: {len(bad)} slack bytes written, first row {bad[0][0]} byte "
                           f"{min(pitch, ceil32(N)) + bad[0][1]}")
    return out


@gpu
@pytest.mark.parametrize("W", MMA_WIDTHS)
def test_tensor_core_kernel_is_exact_and_keeps_the_pitch_slack(ops, W):
    """The tcgen05 kernel on row counts around its 128-row tile, column counts around its 32-byte store chunks and
    256-column tile, and widths that cover its two-stage ring; rows of pitch N (unaligned: per-byte stores),
    ceil32(N), ceil32(N) + 64, and a base 16 bytes off a 32-byte boundary. A call may write bytes
    [0, min(pitch, ceil32(N))) of each row and nothing else."""
    rng = np.random.default_rng(100 + W)
    n = 64 * W - (W % 2) * 5
    a = random_rows(rng, max(MMA_M_LIST), n)
    b = structured_b(rng, a, max(MMA_N_LIST), n)
    ref = commute_ref(a, b)
    d_a, d_b = _dev(a), _dev(b)
    for M in MMA_M_LIST:
        for N in MMA_N_LIST:
            for pitch, offset in [(N, 0), (ceil32(N), 0), (ceil32(N) + 64, 0), (ceil32(N), 16)]:
                out = call_mma(ops, d_a, d_b, M, N, W, pitch, offset)
                assert_equal(out[:, :N], ref[:M, :N], (M, N, W, pitch, offset))


@gpu
def test_tensor_core_refusals_come_before_any_write(ops):
    """A workspace one byte short is refused and nothing is written."""
    rng = np.random.default_rng(1)
    M, N, W = 300, 70, 3
    d_a, d_b = _dev(random_rows(rng, M, 64 * W)), _dev(random_rows(rng, N, 64 * W))
    L = ops.lib()
    need = L.sym_commute_mma_ws_bytes(M, N, W)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    g = Guarded(M * ceil32(N))
    rc = L.sym_commute_mma_pitched(_vp(d_a), M, _vp(d_b), N, W, g.ptr, ceil32(N), _vp(ws), need - 1, _stream())
    assert rc == SYM_E_WORKSPACE
    assert (g.host("refused call") == SENT).all()


def self_blocks(M):
    """The default block size of ops.commute_self."""
    return max(2048, ((M + 31) // 32 + 31) // 32 * 32)


def check_adjacency(ops, a, d_a, got, what, samples=300):
    """got (device, [M, M]) against ops.commute_packed on the device, and sampled rows against the reference."""
    M = a.shape[0]
    full = ops.commute_packed(d_a, d_a).view(torch.uint8)
    eq = got.view(torch.uint8) == full
    if not bool(eq.all()):
        i, j = (int(v) for v in torch.nonzero(~eq)[0])
        raise AssertionError(f"{what}: {int((~eq).sum())} entries differ from commute_packed, first at ({i}, {j})")
    rows = np.unique(np.r_[0, M - 1, np.random.default_rng(M).integers(0, M, samples)])
    assert_equal(full[torch.from_numpy(rows).cuda()].cpu().numpy(), commute_ref(a[rows], a), what)


@gpu
@pytest.mark.parametrize("M,blk", [(8200, 4096), (9001, 2048), (10000, None)])
def test_upper_block_pattern_stays_inside_the_matrix(ops, M, blk):
    """commute_self's call pattern through the ABI: for every block row, sym_commute_mma_pitched on the sub-view
    out + i0 * (pitch + 1) with N = M - i0, then sym_mirror_upper. The last block row's tile runs up to 224 bytes
    past ceil32(N); none of it may reach the guard after the matrix, and the mirrored matrix must be exact."""
    rng = np.random.default_rng(M)
    W = 2
    blk = blk or self_blocks(M)
    a = random_rows(rng, M, 100)
    d_a = _dev(a)
    pitch = ceil32(M)
    L = ops.lib()
    g = Guarded(M * pitch)
    base = g.buf.data_ptr() + g.off
    for i0 in range(0, M, blk):
        i1 = min(M, i0 + blk)
        ws = ops.workspace(L.sym_commute_mma_ws_bytes(i1 - i0, M - i0, W))
        _check(L.sym_commute_mma_pitched(ctypes.c_void_p(d_a.data_ptr() + i0 * 16 * W), i1 - i0,
                                         ctypes.c_void_p(d_a.data_ptr() + i0 * 16 * W), M - i0, W,
                                         ctypes.c_void_p(base + i0 * pitch + i0), pitch, _vp(ws), ws.numel(),
                                         _stream()))
    _check(L.sym_mirror_upper(g.ptr, M, pitch, blk, _stream()))
    out = g.host(f"upper blocks M={M} block_rows={blk}")
    got = torch.from_numpy(out.reshape(M, pitch)[:, :M].copy()).cuda()
    check_adjacency(ops, a, d_a, got, f"upper blocks M={M} block_rows={blk}")


@gpu
@pytest.mark.parametrize("M,W", [(8191, 2), (8192, 2), (10000, 2), (9000, 1)])
def test_commute_self_matches_the_packed_kernel(ops, M, W):
    """ops.commute_self on both sides of SELF_COMMUTE_MIN_ROWS, and at W = 1, which never takes the block path."""
    assert ops.SELF_COMMUTE_MIN_ROWS == 8192
    rng = np.random.default_rng(M + W)
    a = random_rows(rng, M, 64 * W - 3)
    a[M // 2:M // 2 + 50] = a[:50]
    d_a = _dev(a)
    check_adjacency(ops, a, d_a, ops.commute_self(d_a), f"commute_self M={M} W={W}")


@gpu
def test_commute_of_a_tall_operand(ops):
    """ops.commute sends M * N >= 2^22 to the tensor-core kernel: one row more than 65535 tiles of 128 rows runs in
    two slabs of A."""
    M = GRID_Y * MMA_M + 1
    rng = np.random.default_rng(5)
    a = random_rows(rng, M, 64)
    b = a[M - 1:M].copy()
    b[0, 0] ^= np.uint64(1)
    got = ops.commute(_dev(a), _dev(b)).cpu().numpy().astype(np.uint8)
    ref = commute_ref(a, b)
    assert 0 < ref.sum() < M
    assert_equal(got, ref, f"commute M={M} N=1")


@gpu
@pytest.mark.parametrize("n", [20000, 40000])
def test_wide_rows_keep_exact_parity(ops, n):
    """Widths above 16 words always take the tensor-core kernel. Its operand bytes are up to 227, so the int32
    dot product of two all-Y rows of 40 000 qubits passes 2^31: the parity must survive it. All-Y rows against
    all-Y rows (even), against all-Y but one qubit (odd), and dense random rows."""
    rng = np.random.default_rng(n)
    W = words_for(n)
    ones = pack_symp(np.ones((1, 2 * n), dtype=bool))
    a = np.vstack([ones, ones, random_rows(rng, 3, n)])
    a[1, 0] ^= np.uint64(1)                           # qubit 0: Z instead of Y
    b = np.vstack([ones, ones, random_rows(rng, 3, n)])
    b[1, 2 * W - 1] ^= np.uint64(1) << np.uint64((n - 1) % 64)   # last qubit: X instead of Y
    ref = commute_ref(a, b)
    assert ref[0, 0] == 1 and ref[0, 1] == 0 and ref[1, 0] == 0
    d_a, d_b = _dev(a), _dev(b)
    assert_equal(ops.commute(d_a, d_b).cpu().numpy().astype(np.uint8), ref, f"commute n={n}")
    assert_equal(call_mma(ops, d_a, d_b, 5, 5, W, 32)[:, :5], ref, f"sym_commute_mma_pitched n={n}")
    assert_equal(ops.commute_packed(d_a, d_b).cpu().numpy().astype(np.uint8), ref, f"commute_packed n={n}")


@gpu
def test_dispatch_boundary_gives_the_same_answer(ops):
    """M * N = 2^22 - 1 (packed kernel) and 2^22 (tensor-core kernel) on the same rows."""
    rng = np.random.default_rng(22)
    a = random_rows(rng, 2049, 100)
    d = _dev(a)
    ref = commute_ref(a, a)
    lo = ops.commute(d[:2047], d).cpu().numpy().astype(np.uint8)
    hi = ops.commute(d[:2048], d[:2048]).cpu().numpy().astype(np.uint8)
    assert 2047 * 2049 == (1 << 22) - 1
    assert_equal(lo, ref[:2047], "commute 2047 x 2049")
    assert_equal(hi, ref[:2048, :2048], "commute 2048 x 2048")


# ------------------------------------------------------------------------------------------- 4. mirror
@gpu
@pytest.mark.parametrize("M", [1, 31, 33, 100, 1000])
def test_mirror_follows_the_tile_rule(ops, M):
    """sym_mirror_upper on a random non-symmetric byte matrix, padding columns included, for blocks of 32, 64 and
    2048 rows: the result equals the restated tile rule byte for byte; bad block sizes are refused."""
    rng = np.random.default_rng(M)
    L = ops.lib()
    for pitch in (M, ceil32(M) + 32):
        for blk in (32, 64, 2048):
            m = rng.integers(0, 256, size=(M, pitch), dtype=np.uint8)
            g = Guarded(M * pitch, fill=m)
            _check(L.sym_mirror_upper(g.ptr, M, pitch, blk, _stream()))
            got = g.host(f"mirror M={M} pitch={pitch} block_rows={blk}").reshape(M, pitch)
            assert_equal(got, mirror_ref(m, M, blk), f"mirror M={M} pitch={pitch} block_rows={blk}")
    m = rng.integers(0, 256, size=(M, M), dtype=np.uint8)
    for blk in (0, 16, 48, 2047):
        g = Guarded(M * M, fill=m)
        assert L.sym_mirror_upper(g.ptr, M, M, blk, _stream()) == SYM_E_INVALID, blk
        assert np.array_equal(g.host("refused mirror"), m.ravel())


# ------------------------------------------------------------------------------------------- 5. GF(2)
RREF_CASES = {
    # name: (R, Cw, C)
    "small": (12, 2, 100),
    "smem_boundary": (100, 256, 256 * 64 - 13),      # R * Cw * 8 = 204 800 B: one CTA
    "panels_past_boundary": (101, 256, 256 * 64),    # one row more: panels of 16
    "panels16_r_1_mod_16": (33, 1000, 1000 * 64 - 1),
    "panels2": (5, 12800, 12800 * 64 - 40),
    "panels1": (5, 25600, 25600 * 64),
    "one_pivot_sweep": (3, 25601, 25601 * 64 - 5),   # no panel fits: the one-pivot sweep, whatever knob 5 says
}


def run_rref(ops, w, R, Cw, C):
    L = ops.lib()
    g = Guarded(R * Cw * 8, fill=w)
    piv = Guarded(4 * R)
    ws = ops.workspace(L.sym_rref_ws_bytes(R))
    _check(L.sym_rref(g.ptr, R, C, Cw, piv.ptr, _vp(ws), ws.numel(), _stream()))
    return (g.host(f"rref bits R={R} Cw={Cw}").view("<u8").reshape(R, Cw),
            piv.host(f"rref pivots R={R} Cw={Cw}").view("<i4"))


@gpu
@pytest.mark.parametrize("case", list(RREF_CASES))
def test_rref_is_exact_on_every_path(ops, case):
    """sym_rref in the one-CTA shared-memory kernel, in panels of 16, 2 and 1 rows, and in the one-pivot sweep,
    under both values of tuning knob 5, bit for bit and pivot for pivot against _rref_binary."""
    R, Cw, C = RREF_CASES[case]
    assert (R * Cw * 8 <= PANEL_CAP) == (case in ("small", "smem_boundary"))
    rng = np.random.default_rng(R * Cw)
    w = gf2_matrix(rng, R, Cw, C, density=0.5 if Cw < 1000 else 0.02)
    red, piv = rref_ref(w, C)
    try:
        for knob in (1, 0):
            ops.set_tuning(5, knob)
            got, gpiv = run_rref(ops, w, R, Cw, C)
            assert_equal(got, red, (case, knob))
            assert_equal(gpiv, piv, (case, knob, "pivots"))
    finally:
        ops.set_tuning(5, 1)


@gpu
def test_rref_empty_shapes(ops):
    """C = 0 with Cw = 0: every pivot is -1; R = 0: nothing is written."""
    L = ops.lib()
    ws = ops.workspace(L.sym_rref_ws_bytes(4))
    piv = Guarded(16)
    dummy = Guarded(0)
    _check(L.sym_rref(dummy.ptr, 4, 0, 0, piv.ptr, _vp(ws), ws.numel(), _stream()))
    assert (piv.host("rref C=0").view("<i4") == -1).all()
    dummy.host("rref C=0 bits")
    piv = Guarded(0)
    bits = Guarded(0)
    _check(L.sym_rref(bits.ptr, 0, 64, 1, piv.ptr, _vp(ws), ws.numel(), _stream()))
    piv.host("rref R=0 pivots")
    bits.host("rref R=0 bits")


def run_transpose(ops, w_rows, R, Cw_in, Cw_out):
    """sym_bit_transpose of the first R rows of w_rows (uint64[rows, Cw_in]; the rows past R are junk) into a
    guarded uint64[Cw_in * 64, Cw_out]."""
    g = Guarded(Cw_in * 64 * Cw_out * 8)
    d_in = _dev(w_rows)
    _check(ops.lib().sym_bit_transpose(_vp(d_in), R, Cw_in, g.ptr, Cw_out, _stream()))
    return g.host(f"bit_transpose R={R} Cw_in={Cw_in} Cw_out={Cw_out}").view("<u8").reshape(Cw_in * 64, Cw_out)


@gpu
def test_bit_transpose_is_exact(ops):
    """sym_bit_transpose at row counts around the 32-row groups, several input widths and output widths of
    ceil(R/64) and one more, with nonzero junk rows after row R that must not be read; transposing twice gives
    the rows back; 2 * Cw_out > 65535 is refused."""
    rng = np.random.default_rng(3)
    for R in (1, 31, 32, 33, 63, 64, 65, 1000):
        for Cw_in in (1, 2, 3, 17):
            for Cw_out in (words_for(R), words_for(R) + 1):
                rows = 64 * Cw_out
                w = rand_words(rng, (rows, Cw_in))
                w[R:] |= np.uint64(1)                     # junk: every row past R has bits
                t = run_transpose(ops, w, R, Cw_in, Cw_out)
                assert_equal(t, transpose_ref(w, R, Cw_out), ("transpose", R, Cw_in, Cw_out))
                back = run_transpose(ops, t, Cw_in * 64, Cw_out, Cw_in)
                assert_equal(back[:R], w[:R], ("round trip", R, Cw_in, Cw_out))
                assert not back[R:].any(), ("round trip rows past R", R, Cw_in, Cw_out)
    Cw_out = 32768
    g = Guarded(64 * Cw_out * 8)
    d_in = torch.zeros(64 * Cw_out, dtype=torch.int64, device="cuda")
    assert ops.lib().sym_bit_transpose(_vp(d_in), 5, 1, g.ptr, Cw_out, _stream()) == SYM_E_INVALID
    assert (g.host("refused transpose") == SENT).all()


@gpu
@pytest.mark.parametrize("Cw", [1, 255, 256, 257])
def test_or_rows_is_exact(ops, Cw):
    """sym_or_rows over all rows (rows = NULL), over an unordered index list with repeats, and over no rows."""
    rng = np.random.default_rng(Cw)
    R = 40
    w = rand_words(rng, (R, Cw)) & rand_words(rng, (R, Cw)) & rand_words(rng, (R, Cw))
    d_w = _dev(w)
    L = ops.lib()
    sel = np.array([17, 3, 3, 39, 0, 17, 22], dtype=np.int32)
    d_sel = _dev(sel)
    for rows, n_rows, ref in [(None, R, np.bitwise_or.reduce(w, axis=0)),
                              (d_sel, sel.size, np.bitwise_or.reduce(w[sel], axis=0)),
                              (None, 0, np.zeros(Cw, np.uint64)), (d_sel, 0, np.zeros(Cw, np.uint64))]:
        g = Guarded(8 * Cw)
        _check(L.sym_or_rows(_vp(d_w), Cw, ctypes.c_void_p(0) if rows is None else _vp(rows), n_rows, g.ptr,
                             _stream()))
        assert_equal(g.host(f"or_rows Cw={Cw} n_rows={n_rows}").view("<u8"), ref, ("or_rows", Cw, n_rows))
    assert not np.array_equal(np.bitwise_or.reduce(w[sel], axis=0), np.bitwise_or.reduce(w[:sel.size], axis=0))


# ------------------------------------------------------------------------------------------- 6. second device
def wht_ref(d):
    """c'[k, z] = 2^-n sum_r (-1)^popcount(r & z) d[k, r] for integer d, exactly."""
    w = np.array(d, dtype=np.int64)
    K, side = w.shape
    h = 1
    while h < side:
        v = w.reshape(K, side // (2 * h), 2, h)
        a, b = v[:, :, 0, :].copy(), v[:, :, 1, :].copy()
        v[:, :, 0, :] = a + b
        v[:, :, 1, :] = a - b
        h *= 2
    return w / side


@gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_large_shared_memory_kernels_on_a_second_device(ops):
    """The kernels that need more than 48 KB of dynamic shared memory (the one-CTA and panel rref, the Walsh-Hadamard
    tile of the Pauli decomposition) run on device 0 and then on device 1 in the same process."""
    rng = np.random.default_rng(2)
    cases = [(20, 4, 250), (33, 1000, 64000)]
    mats = [gf2_matrix(rng, R, Cw, C, density=0.1) for R, Cw, C in cases]
    n = 13
    diag = rng.integers(-3, 4, size=(2, 1 << n)) + 1j * rng.integers(-3, 4, size=(2, 1 << n))
    ref = wht_ref(diag.real) + 1j * wht_ref(diag.imag)
    for dev in (0, 1):
        with torch.cuda.device(dev):
            ops.device()
            for (R, Cw, C), w in zip(cases, mats):
                bits = _dev(w).to(f"cuda:{dev}")
                piv = ops.rref_packed(bits, C).cpu().numpy()
                red, rpiv = rref_ref(w, C)
                assert_equal(bits.cpu().numpy().view("<u8"), red, ("rref", dev, R, Cw))
                assert_equal(piv, rpiv, ("rref pivots", dev, R, Cw))
            d = torch.from_numpy(diag.copy()).to(f"cuda:{dev}")
            got = ops.pauli_decompose_diagonals(d, n).cpu().numpy()
            assert_equal(got, ref, ("pauli_decompose_diagonals", dev))
