"""Device-level operators: thin torch plumbing (memory, streams) around the C ABI.

Every function takes and returns CUDA tensors. Packed rows are `torch.int64[M, 2W]` (the bit
pattern of the uint64 words of include/symmer_b200.h), coefficients `torch.complex128[M]`.
There is no CPU path: without a CUDA device these raise.
"""
import ctypes
import math

import numpy as np

import torch

from . import _cabi

_ws_cache = {}
# bench.py sets this to a list to collect (start, end) CUDA events around every row-emission launch
emit_events = None


# (start, end) events recorded INSIDE the library around the row-emission kernel alone
emit_kernel_events = None


def _emit_begin():
    if emit_events is None:
        return None
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    if emit_kernel_events is not None:
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()          # instantiates the cudaEvent_t handles; the library re-records them
        k1.record()
        _cabi.check(lib().sym_set_emit_events(ctypes.c_void_p(k0.cuda_event), ctypes.c_void_p(k1.cuda_event)))
        emit_kernel_events.append((k0, k1))
    return e


def _emit_end(start):
    if start is not None:
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        emit_events.append((start, e))
        if emit_kernel_events is not None:
            _cabi.check(lib().sym_set_emit_events(None, None))


def lib():
    return _cabi.load()


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("symmer_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


_checked = set()


def device():
    require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device())
    if dev.index not in _checked:
        _cabi.check(lib().sym_check_device(None, None, None))
        _checked.add(dev.index)
    return dev


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream():
    # the raw handle of torch's current stream; the private accessor skips building a Stream object (this runs once
    # per library call, and a tapering makes hundreds of microsecond-sized calls)
    if _raw_stream is not None:
        return ctypes.c_void_p(_raw_stream(torch.cuda.current_device()))
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def workspace(nbytes):
    """Grow-only scratch buffer per device (torch owns the memory; the C ABI never allocates)."""
    dev = device()
    buf = _ws_cache.get(dev.index)
    if buf is None or buf.numel() < nbytes:
        if buf is not None:
            del _ws_cache[dev.index]
            del buf
        buf = torch.empty(int(nbytes * 1.1) + 4096, dtype=torch.uint8, device=dev)
        _ws_cache[dev.index] = buf
    return buf


def release_workspace():
    _ws_cache.clear()


def to_host(t):
    """Device tensor -> NumPy array. Large results land in page-locked memory by DMA (torch caches the pinned block,
    so repeated downloads do not pay the allocation again); `.cpu()` would stage them through pageable memory."""
    if not t.is_cuda or t.numel() * t.element_size() < (1 << 20):
        return t.cpu().numpy()
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    host.copy_(t, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return host.numpy()


def words_for(n_qubits):
    return max(1, (int(n_qubits) + 63) // 64)


def _rows(xz):
    assert xz.is_cuda and xz.dtype == torch.int64 and xz.dim() == 2 and xz.is_contiguous()
    return xz.shape[0], xz.shape[1] // 2


def _coeff(c):
    assert c.is_cuda and c.dtype == torch.complex128 and c.is_contiguous()
    return c


# ------------------------------------------------------------------------------------------ layout
def pack(symp, n_qubits):
    """bool/uint8[M, 2n] (device) -> int64[M, 2W]."""
    dev = device()
    symp = symp.to(device=dev)
    if symp.dtype == torch.bool:
        symp = symp.view(torch.uint8)
    symp = symp.contiguous()
    M = symp.shape[0]
    W = words_for(n_qubits)
    xz = torch.empty((M, 2 * W), dtype=torch.int64, device=dev)
    _cabi.check(lib().sym_pack(_p(symp), M, int(n_qubits), _p(xz), _stream()))
    return xz


def unpack(xz, n_qubits):
    M, W = _rows(xz)
    out = torch.empty((M, 2 * int(n_qubits)), dtype=torch.uint8, device=xz.device)
    _cabi.check(lib().sym_unpack(_p(xz), M, int(n_qubits), _p(out), _stream()))
    return out.view(torch.bool)


def ycount(xz):
    M, W = _rows(xz)
    y = torch.empty(M, dtype=torch.int32, device=xz.device)
    _cabi.check(lib().sym_ycount(_p(xz), M, W, _p(y), _stream()))
    return y


def sketch(xz):
    M, W = _rows(xz)
    h = torch.empty(M, dtype=torch.int64, device=xz.device)
    _cabi.check(lib().sym_sketch_rows(_p(xz), M, W, _p(h), _stream()))
    return h


# ---------------------------------------------------------------------------------------- multiply
def cross_mul(a_xz, a_c, b_xz, b_c):
    """Materialised cross terms in the reference's order t = q*M + p."""
    M, W = _rows(a_xz)
    N, W2 = _rows(b_xz)
    assert W == W2
    out_xz = torch.empty((M * N, 2 * W), dtype=torch.int64, device=a_xz.device)
    out_c = torch.empty(M * N, dtype=torch.complex128, device=a_xz.device)
    _cabi.check(lib().sym_cross_mul(_p(a_xz), _p(_coeff(a_c)), M, _p(b_xz), _p(_coeff(b_c)), N, W, _p(out_xz),
                                    _p(out_c), _stream()))
    return out_xz, out_c


def _thr(zero_threshold):
    return -1.0 if zero_threshold is None else float(zero_threshold)


def _mul_blocks(a_xz, a_c, b_xz, b_c, flat, nblk, ws, zero_threshold, a_sketch=None, a_ycount=None):
    """Count + emission of a block-list product; returns (xz[U,2W], c[U]). When the count offers the speculative
    emission (a large product whose sampled classes showed no duplicate), the output is allocated at T rows and the
    rows are written while the duplicate detection finishes; a product that turns out to have duplicates after all
    comes back as the first U rows of that buffer."""
    M, W = _rows(a_xz)
    N, _ = _rows(b_xz)
    L = lib()
    U = ctypes.c_int64(0)
    spec = ctypes.c_int32(0)
    _cabi.check(L.sym_mul_blocks_count_tables(_p(a_xz), _p(_coeff(a_c)), _p(a_sketch), _p(a_ycount), M, _p(b_xz),
                                              _p(_coeff(b_c)), N, W, flat, nblk, _thr(zero_threshold), None,
                                              ctypes.byref(U), ctypes.byref(spec), _p(ws), ws.numel(), _stream()))
    U = U.value
    out_xz = torch.empty((U, 2 * W), dtype=torch.int64, device=a_xz.device)
    out_c = torch.empty(U, dtype=torch.complex128, device=a_xz.device)
    ev = _emit_begin()
    if spec.value:
        n = ctypes.c_int64(0)
        _cabi.check(L.sym_mul_blocks_emit_spec(_p(a_xz), _p(a_c), M, _p(b_xz), _p(b_c), N, W, flat, nblk,
                                               _thr(zero_threshold), _p(out_xz), _p(out_c), ctypes.byref(n), _p(ws),
                                               ws.numel(), _stream()))
        if n.value < U:
            out_xz, out_c = out_xz[:n.value], out_c[:n.value]
    else:
        _cabi.check(L.sym_mul_blocks_emit(_p(a_xz), _p(a_c), M, _p(b_xz), _p(b_c), N, W, flat, nblk, U, _p(out_xz),
                                          _p(out_c), _p(ws), ws.numel(), _stream()))
    _emit_end(ev)
    return out_xz, out_c


def mul_cleanup(a_xz, a_c, b_xz, b_c, zero_threshold=1e-15):
    """Fused A*B + cleanup; returns (xz[U,2W], c[U]) in first-occurrence order of t = q*M + p."""
    M, W = _rows(a_xz)
    N, W2 = _rows(b_xz)
    assert W == W2
    dev = a_xz.device
    if M * N == 0:
        return (torch.empty((0, 2 * W), dtype=torch.int64, device=dev),
                torch.empty(0, dtype=torch.complex128, device=dev))
    ws = workspace(lib().sym_mul_cleanup_ws_bytes(M, N, W))
    return _mul_blocks(a_xz, a_c, b_xz, b_c, (ctypes.c_int64 * 4)(0, M, 0, N), 1, ws, zero_threshold)


def mul_blocks_cleanup(a_xz, a_c, b_xz, b_c, blocks, zero_threshold=1e-15, a_sketch=None, a_ycount=None):
    """Product + cleanup restricted to disjoint rectangular blocks [(p0, p1, q0, q1), ...] of the
    cross-term grid A x B (the exchange-free sharded product: rank r passes the blocks it owns).
    Survivors leave block by block in (q, p) order. Returns (xz[U,2W], c[U], n_cross_terms)."""
    M, W = _rows(a_xz)
    N, W2 = _rows(b_xz)
    assert W == W2
    dev = a_xz.device
    blocks = [tuple(int(v) for v in blk) for blk in blocks]
    T = sum((p1 - p0) * (q1 - q0) for p0, p1, q0, q1 in blocks)
    if T == 0:
        return (torch.empty((0, 2 * W), dtype=torch.int64, device=dev),
                torch.empty(0, dtype=torch.complex128, device=dev), 0)
    flat = (ctypes.c_int64 * (4 * len(blocks)))(*[v for blk in blocks for v in blk])
    nbytes = lib().sym_mul_blocks_ws_bytes(M, N, W, flat, len(blocks))
    if nbytes == 0:
        _cabi.check(-1)
    ws = workspace(nbytes)
    out_xz, out_c = _mul_blocks(a_xz, a_c, b_xz, b_c, flat, len(blocks), ws, zero_threshold, a_sketch, a_ycount)
    return out_xz, out_c, T


def cleanup(xz, c, zero_threshold=1e-15):
    T, W = _rows(xz)
    dev = xz.device
    if T == 0:
        return xz.clone(), c.clone()
    L = lib()
    ws = workspace(L.sym_cleanup_ws_bytes(T, W))
    U = ctypes.c_int64(0)
    _cabi.check(L.sym_cleanup_count(_p(xz), _p(_coeff(c)), T, W, _thr(zero_threshold), None, ctypes.byref(U), _p(ws),
                                    ws.numel(), _stream()))
    U = U.value
    out_xz = torch.empty((U, 2 * W), dtype=torch.int64, device=dev)
    out_c = torch.empty(U, dtype=torch.complex128, device=dev)
    _cabi.check(L.sym_cleanup_emit(_p(xz), _p(c), T, W, U, _p(out_xz), _p(out_c), _p(ws), ws.numel(), _stream()))
    return out_xz, out_c


# ----------------------------------------------------------------------------------------- commute
# Measured on B200 (scripts/probe_commute_cross.py, profiles/r01_commute.md): the tcgen05 int8 kernel
# beats the bit-packed one at every width once the output is large enough to amortise its two
# operand transposes; the bit-packed kernel keeps the small (launch-bound) cases.
MMA_MIN_PAIRS = 1 << 22


def commute(a_xz, b_xz):
    """bool[M, N], True where A[i] commutes with B[j] (dispatches to the kernel ncu shows winning)."""
    M, W = _rows(a_xz)
    N, _ = _rows(b_xz)
    if M * N >= MMA_MIN_PAIRS or W > 16:
        return commute_mma(a_xz, b_xz)
    return commute_packed(a_xz, b_xz)


def commute_packed(a_xz, b_xz):
    """Bit-packed AND/XOR + popcount-parity kernel."""
    M, W = _rows(a_xz)
    N, W2 = _rows(b_xz)
    assert W == W2
    out = torch.empty((M, N), dtype=torch.uint8, device=a_xz.device)
    _cabi.check(lib().sym_commute(_p(a_xz), M, _p(b_xz), N, W, _p(out), _stream()))
    return out.view(torch.bool)


def commute_mma(a_xz, b_xz):
    """Tensor-core (tcgen05 int8) variant of `commute`; identical output."""
    M, W = _rows(a_xz)
    N, W2 = _rows(b_xz)
    assert W == W2
    # rows padded to a multiple of 32 bytes: every row stays 16-byte aligned and the kernel keeps its 32-byte
    # vector stores for ragged N; the caller gets the [M, N] view of the padded buffer
    pitch = (N + 31) // 32 * 32
    out = torch.empty((M, pitch), dtype=torch.uint8, device=a_xz.device)
    L = lib()
    ws = workspace(L.sym_commute_mma_ws_bytes(M, N, W))
    _cabi.check(L.sym_commute_mma_pitched(_p(a_xz), M, _p(b_xz), N, W, _p(out), pitch, _p(ws), ws.numel(), _stream()))
    return out.view(torch.bool)[:, :N]


# self-commutation of at least this many rows computes the upper block triangle only and mirrors it (the matrix is
# symmetric); below, one full launch is cheaper than several block launches plus the mirror pass
SELF_COMMUTE_MIN_ROWS = 8192


def commute_self(a_xz, row_begin=0, row_end=None, block_rows=None):
    """adjacency_matrix (base.py:1054-1062): bool[M, M], True where A[i] commutes with A[j]. Symmetric, so for large
    operators only the blocks on and above the block diagonal are computed (sym_commute* on A[i0:i1) x A[i0:M)) and
    one pass mirrors them into the lower triangle. row_begin / row_end / block_rows: internal (multi-GPU shares)."""
    M, W = _rows(a_xz)
    if M < SELF_COMMUTE_MIN_ROWS or W < 2:
        return commute(a_xz, a_xz)
    blk = block_rows or max(2048, ((M + 31) // 32 + 31) // 32 * 32)      # at most ~32 block rows, multiples of 32
    pitch = (M + 31) // 32 * 32
    out = torch.empty((M, pitch), dtype=torch.uint8, device=a_xz.device)
    L = lib()
    for i0 in range(0, M, blk):
        i1 = min(M, i0 + blk)
        a_blk, b_blk = a_xz[i0:i1], a_xz[i0:]
        ws = workspace(L.sym_commute_mma_ws_bytes(i1 - i0, M - i0, W))
        sub = out[i0:i1, i0:]                                            # starts on a 32-byte boundary of its row
        _cabi.check(L.sym_commute_mma_pitched(_p(a_blk), i1 - i0, _p(b_blk), M - i0, W, _p(sub), pitch, _p(ws), ws.numel(),
                                              _stream()))
    _cabi.check(L.sym_mirror_upper(_p(out), M, pitch, blk, _stream()))
    return out.view(torch.bool)[:, :M]


def commute_bits(a_xz, b_xz):
    M, W = _rows(a_xz)
    N, _ = _rows(b_xz)
    out = torch.zeros((M, (N + 31) // 32), dtype=torch.int32, device=a_xz.device)
    _cabi.check(lib().sym_commute_bits(_p(a_xz), M, _p(b_xz), N, W, _p(out), _stream()))
    return out


def commute_qwc(a_xz, b_xz):
    """bool[M, N], True where A[i] and B[j] commute qubit by qubit (base.py:985-1009)."""
    M, W = _rows(a_xz)
    N, W2 = _rows(b_xz)
    assert W == W2
    out = torch.empty((M, N), dtype=torch.uint8, device=a_xz.device)
    _cabi.check(lib().sym_commute_qwc(_p(a_xz), M, _p(b_xz), N, W, _p(out), _stream()))
    return out.view(torch.bool)


def gather_qubits(xz, src, n_in):
    """Rows over len(src) qubits: output qubit k takes input qubit src[k] (identity where src[k] < 0).
    Reindexing (a permutation) and the embedding of a tensor factor into a wider register."""
    M, W = _rows(xz)
    src = np.ascontiguousarray(src, dtype=np.int32)
    assert src.ndim == 1 and (src.size == 0 or int(src.max()) < int(n_in)), 'source qubit out of range'
    n_out = int(src.size)
    out = torch.empty((M, 2 * words_for(n_out)), dtype=torch.int64, device=xz.device)
    src_dev = torch.from_numpy(src).to(xz.device)
    _cabi.check(lib().sym_gather_qubits(_p(xz), M, W, _p(src_dev), n_out, _p(out), _stream()))
    return out


# ------------------------------------------------------------------------------- ordering / joins
def gather_rows(xz, c, perm):
    """Rows (and coefficients, if given) in the order of the int32 device permutation `perm`."""
    M, W = _rows(xz)
    n = int(perm.numel())
    assert perm.dtype == torch.int32 and perm.is_contiguous()
    out_xz = torch.empty((n, 2 * W), dtype=torch.int64, device=xz.device)
    out_c = torch.empty(n, dtype=torch.complex128, device=xz.device) if c is not None else None
    _cabi.check(lib().sym_gather_rows(_p(xz), _p(_coeff(c)) if c is not None else _p(None), _p(perm), n, W, _p(out_xz), _p(out_c),
                                      _stream()))
    return out_xz, out_c


def lex_order(xz):
    """int32 device permutation that sorts the packed rows like `np.lexsort(symp_matrix.T)` (base.py:469-470: the LAST
    column is the primary key, i.e. rows ordered as integers whose most significant bits are the Z block's highest
    qubits). Stable LSD radix sort word by word: X words from the lowest up, then Z words; all-zero word columns
    (padding, sparse registers) are skipped. No host unpack, only 2W words of OR come back."""
    M, W = _rows(xz)
    perm = torch.arange(M, dtype=torch.int32, device=xz.device)
    if M <= 1:
        return perm
    used = or_rows(xz).cpu().numpy()
    keys = torch.empty(M, dtype=torch.int64, device=xz.device)
    L = lib()
    first = True
    for col in range(2 * W):                       # least significant word first
        w = int(used[col]) & 0xFFFFFFFFFFFFFFFF
        if w == 0:
            continue
        _cabi.check(L.sym_gather_column(_p(xz), M, 2 * W, col, _p(None) if first else _p(perm), _p(keys), _stream()))
        begin_bit = (w & -w).bit_length() - 1      # bits below the lowest used bit are zero in every row
        sort_pairs(keys, perm, begin_bit=begin_bit)
        first = False
    return perm


def join_rows(keys_l, rows_l, keys_r, rows_r):
    """int32[M]: for every left row the index of the equal right row, or -1 (exact: sketches only locate candidates)."""
    M, N = int(keys_l.numel()), int(keys_r.numel())
    words = int(rows_l.shape[1])
    match = torch.full((M,), -1, dtype=torch.int32, device=keys_l.device)
    if M == 0 or N == 0:
        return match
    kr = keys_r.clone()                                  # sorted as uint64, like the kernel compares them
    perm = torch.arange(N, dtype=torch.int32, device=keys_r.device)
    sort_pairs(kr, perm)
    _cabi.check(lib().sym_join_rows(_p(keys_l.contiguous()), _p(rows_l.contiguous()), M, _p(kr), _p(perm), _p(rows_r.contiguous()),
                                    N, words, _p(match), _stream()))
    return match


# --------------------------------------------------------------------------------------- rotations
ROTATE_PADDED_MAX_ROWS = 1 << 19


def rotate(xz, c, q_xz, cos_a, sin_a, mode, sign=1.0, padded_ok=False):
    """One rotation step (no dedup). mode 0 general (returns M + M_ac rows), 1/2 Clifford. padded_ok: the caller
    runs a cleanup next, so a general rotation of a config-size operator may return its padded form (2M rows,
    the second row of a commuting term a zero-coefficient copy: see sym_rotate mode 4) and skip the flag scan
    and the host round trip for the row count."""
    M, W = _rows(xz)
    dev = xz.device
    if mode == 0 and padded_ok and 0 < M <= ROTATE_PADDED_MAX_ROWS and ((W % 2 == 0 and W <= 16) or W == 1):
        out_xz = torch.empty((2 * M, 2 * W), dtype=torch.int64, device=dev)
        out_c = torch.empty(2 * M, dtype=torch.complex128, device=dev)
        n_out = torch.empty(1, dtype=torch.int64, device=dev)
        _cabi.check(lib().sym_rotate(_p(xz), _p(_coeff(c)), M, W, _p(q_xz), float(cos_a), float(sin_a), 4, float(sign),
                                     _p(out_xz), _p(out_c), _p(n_out), None, 0, _stream()))
        return out_xz, out_c
    cap = 2 * M if mode == 0 else M
    out_xz = torch.empty((cap, 2 * W), dtype=torch.int64, device=dev)
    out_c = torch.empty(cap, dtype=torch.complex128, device=dev)
    n_out = torch.empty(1, dtype=torch.int64, device=dev)      # always written by the library
    L = lib()
    ws = workspace(L.sym_rotate_ws_bytes(M))
    _cabi.check(L.sym_rotate(_p(xz), _p(_coeff(c)), M, W, _p(q_xz), float(cos_a), float(sin_a), int(mode), float(sign),
                             _p(out_xz), _p(out_c), _p(n_out), _p(ws), ws.numel(), _stream()))
    if mode == 0:
        n = int(n_out.item())
        return out_xz[:n], out_c[:n]
    return out_xz, out_c


def rotate_split(xz, c, q_xz):
    """Stable split of the rows into (commuting with Q | anticommuting with Q) with the sketch and Y-count
    tables of the split rows: (xz', c', sketch int64[M], ycount int32[M], n_commuting)."""
    M, W = _rows(xz)
    dev = xz.device
    out_xz = torch.empty_like(xz)
    out_c = torch.empty_like(c)
    sk = torch.empty(M, dtype=torch.int64, device=dev)
    yc = torch.empty(M, dtype=torch.int32, device=dev)
    n_out = torch.zeros(1, dtype=torch.int64, device=dev)
    if M == 0:
        return out_xz, out_c, sk, yc, 0
    L = lib()
    ws = workspace(L.sym_rotate_split_ws_bytes(M))
    _cabi.check(L.sym_rotate_split(_p(xz), _p(_coeff(c)), M, W, _p(q_xz), _p(out_xz), _p(out_c), _p(sk), _p(yc), _p(n_out),
                                   _p(ws), ws.numel(), _stream()))
    return out_xz, out_c, sk, yc, int(n_out.item())


def rotate_dedup(xz, c, q_xz, cos_a, sin_a, zero_threshold=1e-15):
    """General rotation R P R^dagger, R = exp(i*angle/2*Q), INCLUDING its dedup, as one block-list product
    (base.py:1090-1161 = base.py:764-794 applied to blocks): commuting rows x [I], anticommuting rows x
    [cos I, -i sin Q]. The rotated rows are never materialised before the dedup; survivors leave with the
    commuting rows first. Returns (xz', c')."""
    M, W = _rows(xz)
    sxz, sc, sk, yc, n_comm = rotate_split(xz, c, q_xz)
    b_xz = torch.zeros((3, 2 * W), dtype=torch.int64, device=xz.device)
    b_xz[2] = q_xz.reshape(-1)
    b_c = torch.tensor([1.0, float(cos_a), -1j * float(sin_a)], dtype=torch.complex128, device=xz.device)
    out_xz, out_c, _ = mul_blocks_cleanup(sxz, sc, b_xz, b_c, [(0, n_comm, 0, 1), (n_comm, M, 1, 3)], zero_threshold,
                                          a_sketch=sk, a_ycount=yc)
    return out_xz, out_c


# -------------------------------------------------------------------------------------- projection
def project(xz, c, n_qubits, stab_cols, stab_eigs, free_qubits):
    """Stabilizer-subspace projection of rotated rows (no duplicate merge): returns (xz', c') over the
    free qubits, rows that anticommute with a single-qubit stabilizer dropped, signs fixed."""
    M, W = _rows(xz)
    dev = xz.device
    cols = torch.as_tensor(stab_cols, dtype=torch.int32, device=dev).contiguous()
    eigs = torch.as_tensor(stab_eigs, dtype=torch.float64, device=dev).contiguous()
    free = torch.as_tensor(free_qubits, dtype=torch.int32, device=dev).contiguous()
    n_free = int(free.numel())
    Wo = max(1, (n_free + 63) // 64)
    out_xz = torch.empty((M, 2 * Wo), dtype=torch.int64, device=dev)
    out_c = torch.empty(M, dtype=torch.complex128, device=dev)
    if M == 0:
        return out_xz, out_c
    L = lib()
    ws = workspace(L.sym_project_ws_bytes(M, n_free))
    U = ctypes.c_int64(0)
    _cabi.check(L.sym_project(_p(xz), _p(_coeff(c)), M, W, int(n_qubits), _p(cols), _p(eigs), int(cols.numel()), _p(free),
                              n_free, _p(out_xz), _p(out_c), None, ctypes.byref(U), _p(ws), ws.numel(), _stream()))
    return out_xz[:U.value], out_c[:U.value]


# ------------------------------------------------------------------------------------- matrix-free
def term_masks_sorted(xz, c, n_qubits):
    """Basis-index masks and phased coefficients of every term, sorted by x mask. The returned
    coefficient tensor carries two Python attributes used by the kernels' fast paths:
    `_sym_real` (every phased coefficient is real) and `_sym_hermitian` (additionally every original
    coefficient is real, i.e. a Hermitian operator whose terms all have an even number of Y)."""
    M, W = _rows(xz)
    assert W == 1 and n_qubits <= 62
    dev = xz.device
    xm = torch.empty(M, dtype=torch.int64, device=dev)
    zm = torch.empty(M, dtype=torch.int64, device=dev)
    cp = torch.empty(M, dtype=torch.complex128, device=dev)
    L = lib()
    _cabi.check(L.sym_term_masks(_p(xz), _p(_coeff(c)), M, int(n_qubits), _p(xm), _p(zm), _p(cp), _stream()))
    if M > 1:
        order = sort_pairs(xm.clone(), torch.arange(M, dtype=torch.int32, device=dev), begin_bit=0)[1].to(torch.int64)
        xm, zm, cp = xm[order].contiguous(), zm[order].contiguous(), cp[order].contiguous()
    if M <= 32:
        # a handful of terms (stabilizers measured one at a time): the fast paths would save nothing, and reading
        # the flags back costs a stream synchronise per operator
        flags = [False, False]
    else:
        flags = torch.stack([(cp.imag == 0).all(), (c.imag == 0).all()]).cpu().tolist()    # one sync, once per operator
    cp._sym_real = bool(flags[0])
    cp._sym_hermitian = bool(flags[0] and flags[1])
    cp._sym_table = None
    return xm, zm, cp


def _is_real(cp):
    return 1 if getattr(cp, "_sym_real", False) else 0


def apply_dense(xm, zm, cp, n_qubits, psi, row_begin=0, row_end=None):
    side = 1 << int(n_qubits)
    row_end = side if row_end is None else row_end
    psi = psi.contiguous()
    assert psi.dtype == torch.complex128 and psi.numel() == side
    y = torch.empty(row_end - row_begin, dtype=torch.complex128, device=psi.device)
    _cabi.check(lib().sym_apply(_p(xm), _p(zm), _p(cp), xm.numel(), int(n_qubits), _p(psi), _p(y), row_begin, row_end,
                                _is_real(cp), _stream()))
    return y


SYM_ALIGN = 2048      # row-range alignment of the symmetric expectation-value mode
use_symmetric_expval = True


def expval_dense(xm, zm, cp, n_qubits, psi, row_begin=0, row_end=None):
    """Partial <psi|H|psi> over basis rows [row_begin, row_end) as a complex128 device scalar. For a
    Hermitian operator with real phased coefficients (see term_masks_sorted) and 2048-aligned row
    ranges the symmetric mode halves the work: the partial sums of the row ranges then only add up
    to the total when every range is evaluated this way (they are, for a given operator)."""
    side = 1 << int(n_qubits)
    row_end = side if row_end is None else row_end
    psi = psi.contiguous()
    assert psi.dtype == torch.complex128 and psi.numel() == side
    partial = torch.zeros(2, dtype=torch.float64, device=psi.device)
    L = lib()
    M = xm.numel()
    if (use_symmetric_expval and getattr(cp, "_sym_hermitian", False) and side % SYM_ALIGN == 0
            and row_begin % SYM_ALIGN == 0 and row_end % SYM_ALIGN == 0 and M > 0):
        if cp._sym_table is None:
            z_sym = torch.empty_like(zm)
            c_sym = torch.empty_like(cp)
            _cabi.check(L.sym_expval_prepare_sym(_p(xm), _p(zm), _p(cp), M, _p(z_sym), _p(c_sym), _stream()))
            cp._sym_table = (z_sym, c_sym)
        z_sym, c_sym = cp._sym_table
        _cabi.check(L.sym_expval(_p(xm), _p(z_sym), _p(c_sym), M, int(n_qubits), _p(psi), _p(partial), row_begin, row_end, 2,
                                 _stream()))
    else:
        _cabi.check(L.sym_expval(_p(xm), _p(zm), _p(cp), M, int(n_qubits), _p(psi), _p(partial), row_begin, row_end,
                                 _is_real(cp), _stream()))
    return torch.view_as_complex(partial)


def to_csr(xm, zm, cp, n_qubits):
    """(data, indices, indptr) device tensors; every row has G = #distinct x entries sorted by column."""
    dev = xm.device
    # group boundaries of the sorted x masks: a few thousand terms, found on the host (one small copy each way)
    xh = xm.cpu().numpy()
    first = np.flatnonzero(np.concatenate([[True], xh[1:] != xh[:-1]])) if xh.size else np.zeros(0, dtype=np.int64)
    G = int(first.size)
    xg = torch.from_numpy(np.ascontiguousarray(xh[first])).to(dev)
    start = torch.from_numpy(np.concatenate([first, [xh.size]]).astype(np.int32)).to(dev)
    side = 1 << int(n_qubits)
    data = torch.empty(side * G, dtype=torch.complex128, device=dev)
    indices = torch.empty(side * G, dtype=torch.int64, device=dev)
    indptr = torch.empty(side + 1, dtype=torch.int64, device=dev)
    _cabi.check(lib().sym_to_csr(_p(zm), _p(cp), xm.numel(), int(n_qubits), _p(xg.contiguous()), G, _p(start), _p(data),
                                 _p(indices), _p(indptr), _stream()))
    return data, indices, indptr


def pauli_decompose_dense(matrix, n_qubits):
    """complex128[2^n, 2^n] device matrix -> c'[x, z] (see include/symmer_b200.h): one Walsh-Hadamard transform
    per XOR-diagonal. The Pauli with masks (x, z) has coefficient c' * i^popcount(x&z)."""
    side = 1 << int(n_qubits)
    matrix = matrix.contiguous()
    assert matrix.is_cuda and matrix.dtype == torch.complex128 and tuple(matrix.shape) == (side, side)
    out = torch.empty_like(matrix)
    _cabi.check(lib().sym_pauli_decompose_dense(_p(matrix), int(n_qubits), _p(out), _stream()))
    return out


def pauli_decompose_diagonals(diag, n_qubits):
    """In place: complex128[K, 2^n] XOR-diagonals d_x[r] = M[r, r^x] -> c'[k, z]."""
    assert diag.is_cuda and diag.dtype == torch.complex128 and diag.is_contiguous() and diag.shape[1] == 1 << int(n_qubits)
    _cabi.check(lib().sym_pauli_decompose_diagonals(_p(diag), diag.shape[0], int(n_qubits), _stream()))
    return diag


def rows_from_masks(xm, zm, cp, n_qubits):
    """Inverse of term masks: (x, z) basis-index masks + phased coefficients -> (packed rows [M, 2], coefficients)."""
    M = xm.numel()
    xz = torch.empty((M, 2), dtype=torch.int64, device=xm.device)
    c = torch.empty(M, dtype=torch.complex128, device=xm.device)
    _cabi.check(lib().sym_rows_from_masks(_p(xm.contiguous()), _p(zm.contiguous()), _p(_coeff(cp.contiguous())), M,
                                          int(n_qubits), _p(xz), _p(c), _stream()))
    return xz, c


# ------------------------------------------------------------------------------------------- GF(2)
def pack_matrix(m):
    """bool[R, C] (device) -> int64[R, Cw]."""
    dev = device()
    m = m.to(device=dev)
    if m.dtype == torch.bool:
        m = m.view(torch.uint8)
    m = m.contiguous()
    R, C = m.shape
    Cw = max(1, (C + 63) // 64)
    bits = torch.zeros((R, Cw), dtype=torch.int64, device=dev)
    _cabi.check(lib().sym_pack_matrix(_p(m), R, C, _p(bits), Cw, _stream()))
    return bits


def unpack_matrix(bits, C):
    R, Cw = bits.shape
    out = torch.empty((R, C), dtype=torch.uint8, device=bits.device)
    _cabi.check(lib().sym_unpack_matrix(_p(bits), R, C, Cw, _p(out), _stream()))
    return out.view(torch.bool)


def rref_packed(bits, C):
    """In-place _rref_binary on packed rows; returns the pivot column per row (-1 = zero row)."""
    R, Cw = bits.shape
    piv = torch.empty(R, dtype=torch.int32, device=bits.device)
    L = lib()
    ws = workspace(L.sym_rref_ws_bytes(R))
    _cabi.check(L.sym_rref(_p(bits), R, C, Cw, _p(piv), _p(ws), ws.numel(), _stream()))
    return piv


def bit_transpose(bits):
    """int64[R, Cw] bit matrix (Cw*64 columns) -> int64[Cw*64, ceil(R/64)]."""
    assert bits.is_cuda and bits.dtype == torch.int64 and bits.dim() == 2 and bits.is_contiguous()
    R, Cw = bits.shape
    Cw_out = max(1, (R + 63) // 64)
    out = torch.empty((Cw * 64, Cw_out), dtype=torch.int64, device=bits.device)
    _cabi.check(lib().sym_bit_transpose(_p(bits), R, Cw, _p(out), Cw_out, _stream()))
    return out


def or_rows(bits, rows=None):
    """int64[Cw]: bitwise OR of the selected rows (int32 device indices; None = all rows)."""
    R, Cw = bits.shape
    out = torch.empty(Cw, dtype=torch.int64, device=bits.device)
    n = R if rows is None else int(rows.numel())
    _cabi.check(lib().sym_or_rows(_p(bits), Cw, _p(rows), n, _p(out), _stream()))
    return out


# ---------------------------------------------------------------------------------- noncontextual
def nc_signs(xz, gen_xz, rep_xz, J, clique):
    """float64[M] device: s_t of P_t = s_t * G^{J_t} * C_{clique[t]} (0 where the product is not +-P_t).
    J: int64[M, Jw] device bit rows over the k generators; clique: int32[M] device, -1 for symmetry terms."""
    M, W = _rows(xz)
    k, N = int(gen_xz.shape[0]), int(rep_xz.shape[0])
    assert J.dtype == torch.int64 and J.dim() == 2 and J.shape[0] == M and J.is_contiguous()
    assert clique.dtype == torch.int32 and clique.numel() == M and clique.is_contiguous()
    signs = torch.empty(M, dtype=torch.float64, device=xz.device)
    _cabi.check(lib().sym_nc_signs(_p(xz), M, W, _p(gen_xz.contiguous()), k, _p(rep_xz.contiguous()), N, _p(J),
                                   int(J.shape[1]), _p(clique), _p(signs), _stream()))
    return signs


def nc_min(J, v, clique, n_cliques, f):
    """(E, m): the minimum over the 2^f assignments m of a(m) - ||w(m)|| (see sym_nc_min), ties to the smaller m.
    J: int64[M] free-bit masks, v: float64[M], clique: int32[M] (device). One 16-byte copy back."""
    M = int(J.numel())
    assert J.dtype == torch.int64 and v.dtype == torch.float64 and clique.dtype == torch.int32
    assert v.numel() == M and clique.numel() == M
    L = lib()
    nbytes = L.sym_nc_min_ws_bytes(M, int(n_cliques))
    if nbytes == 0:
        _cabi.check(-1)
    ws = workspace(nbytes)
    best = torch.empty(2, dtype=torch.int64, device=ws.device)
    host = (ctypes.c_uint64 * 2)()
    _cabi.check(L.sym_nc_min(_p(J.contiguous()), _p(v.contiguous()), _p(clique.contiguous()), M, int(n_cliques), int(f),
                             _p(best), ctypes.cast(host, ctypes.c_void_p), _p(ws), ws.numel(), _stream()))
    return float(np.frombuffer(bytes(host), dtype=np.float64)[0]), int(host[1])


# ---------------------------------------------------------------------------------- sort / records
def sort_pairs(keys, vals, begin_bit=0):
    """Stable sort of (int64-as-uint64 keys, int32-as-uint32 vals) in place; returns (keys, vals)."""
    T = keys.numel()
    assert keys.dtype == torch.int64 and vals.dtype == torch.int32 and vals.numel() == T
    if T == 0:
        return keys, vals
    L = lib()
    ws = workspace(L.sym_sort_pairs_ws_bytes(T))
    _cabi.check(L.sym_sort_pairs(_p(keys), _p(vals), T, int(begin_bit), _p(ws), ws.numel(), _stream()))
    return keys, vals


def pair_records(a_xz, p_begin, p_end, b_xz):
    """int64[T] records of the block A[p_begin:p_end) x B, T = (p_end-p_begin)*N."""
    M, W = _rows(a_xz)
    N, _ = _rows(b_xz)
    T = (p_end - p_begin) * N
    recs = torch.empty(T, dtype=torch.int64, device=a_xz.device)
    if T == 0:
        return recs
    L = lib()
    ws = workspace(L.sym_pair_records_ws_bytes(M, N, W))
    _cabi.check(L.sym_pair_records(_p(a_xz), M, p_begin, p_end, _p(b_xz), N, W, _p(recs), _p(ws), ws.numel(),
                                   _stream()))
    return recs


def pair_records_blocks(a_xz, b_xz, blocks):
    """Records of the rectangular blocks [(p0, p1, q0, q1), ...] of A x B, back to back in block order."""
    M, W = _rows(a_xz)
    N, _ = _rows(b_xz)
    blocks = [tuple(int(v) for v in blk) for blk in blocks]
    T = sum((p1 - p0) * (q1 - q0) for p0, p1, q0, q1 in blocks)
    recs = torch.empty(T, dtype=torch.int64, device=a_xz.device)
    if T == 0:
        return recs
    flat = (ctypes.c_int64 * (4 * len(blocks)))(*[v for blk in blocks for v in blk])
    L = lib()
    ws = workspace(L.sym_pair_records_ws_bytes(M, N, W))
    _cabi.check(L.sym_pair_records_blocks(_p(a_xz), M, _p(b_xz), N, W, flat, len(blocks), _p(recs), _p(ws), ws.numel(),
                                          _stream()))
    return recs


def owner_classes(xz, log2_parts):
    """uint8[M]: owner class of every row (GF(2)-linear in the row, so class(a^b) = class(a)^class(b))."""
    M, W = _rows(xz)
    cls = torch.empty(M, dtype=torch.uint8, device=xz.device)
    if M:
        ws = workspace(8 * M + 512)
        _cabi.check(lib().sym_owner_classes(_p(xz), M, W, int(log2_parts), _p(cls), _p(ws), ws.numel(), _stream()))
    return cls


def class_partition(xz, c, log2_parts):
    """Stable grouping of an operator by owner class: (xz', c', perm int32[M], counts int64[parts])."""
    M, W = _rows(xz)
    dev = xz.device
    out_xz = torch.empty_like(xz)
    out_c = torch.empty_like(c) if c is not None else None
    perm = torch.empty(M, dtype=torch.int32, device=dev)
    counts = torch.zeros(1 << int(log2_parts), dtype=torch.int64, device=dev)
    L = lib()
    ws = workspace(L.sym_class_partition_ws_bytes(M))
    _cabi.check(L.sym_class_partition(_p(xz), _p(_coeff(c)) if c is not None else _p(None), M, W, int(log2_parts),
                                      _p(out_xz), _p(out_c), _p(perm), _p(counts), _p(ws), ws.numel(), _stream()))
    return out_xz, out_c, perm, counts


def partition_records(recs, log2_parts):
    """Stable partition by owner (top log2_parts bits); returns (recs_by_owner, counts int64[parts])."""
    T = recs.numel()
    out = torch.empty_like(recs)
    counts = torch.zeros(1 << log2_parts, dtype=torch.int64, device=recs.device)
    L = lib()
    ws = workspace(L.sym_partition_ws_bytes(T))
    _cabi.check(L.sym_partition_records(_p(recs), T, int(log2_parts), _p(out), _p(counts), _p(ws), ws.numel(),
                                        _stream()))
    return out, counts


def dedup_records(recs, a_xz, a_c, b_xz, b_c, zero_threshold=1e-15):
    """Dedup + reduce + emit for records whose rows are A[p]^B[q]; recs is clobbered."""
    T = recs.numel()
    M, W = _rows(a_xz)
    N, _ = _rows(b_xz)
    dev = a_xz.device
    if T == 0:
        return (torch.empty((0, 2 * W), dtype=torch.int64, device=dev),
                torch.empty(0, dtype=torch.complex128, device=dev))
    L = lib()
    ws = workspace(L.sym_dedup_records_ws_bytes(T, W))
    U = ctypes.c_int64(0)
    _cabi.check(L.sym_dedup_records_count(_p(recs), T, _p(a_xz), _p(_coeff(a_c)), M, _p(b_xz), _p(_coeff(b_c)), N, W,
                                          _thr(zero_threshold), None, ctypes.byref(U), _p(ws), ws.numel(), _stream()))
    U = U.value
    out_xz = torch.empty((U, 2 * W), dtype=torch.int64, device=dev)
    out_c = torch.empty(U, dtype=torch.complex128, device=dev)
    ev = _emit_begin()
    _cabi.check(L.sym_dedup_records_emit(_p(recs), T, _p(a_xz), _p(a_c), M, _p(b_xz), _p(b_c), N, W, U, _p(out_xz),
                                         _p(out_c), _p(ws), ws.numel(), _stream()))
    _emit_end(ev)
    return out_xz, out_c


def set_tuning(which, value):
    _cabi.check(lib().sym_set_tuning(int(which), int(value)))


def launch_count():
    return int(lib().sym_launch_count())


def set_debug_key_mask(mask):
    _cabi.check(lib().sym_debug_set_key_mask(ctypes.c_uint64(mask & 0xFFFFFFFFFFFFFFFF)))
