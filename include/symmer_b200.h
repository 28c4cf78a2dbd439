/* symmer_b200 — C ABI of the B200 (sm_100a) engine for symmer's symplectic Pauli algebra.
 *
 * The reference (UCL-CCS/symmer) is pure Python and has no FFI of its own; its de-facto seams for the
 * hot path are the array kernels of symmer/operators/utils.py and the PauliwordOp methods of
 * symmer/operators/base.py (SURVEY.md §8b). Each entry point below replaces one of those; the
 * reference-side binding (ctypes) a maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch tensors in the Python host) unless
 *     the parameter name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls are
 *     asynchronous on that stream unless stated otherwise;
 *   - return value: 0 = ok, <0 = error (SYM_E_*); sym_last_error() gives a message; no C++
 *     exceptions cross the boundary; nothing is allocated inside — scratch memory comes from the
 *     caller through (`ws`, `ws_bytes`), sized by the matching *_ws_bytes() query;
 *   - packed operator layout: row-major uint64[M][2*W], W = ceil(n_qubits/64) (W >= 1); words
 *     [0,W) are the X block, [W,2W) the Z block; qubit q is bit (q % 64) of word (q / 64) of its
 *     block; padding bits are zero. Coefficients: complex128 as interleaved double[M][2].
 */
#ifndef SYMMER_B200_H
#define SYMMER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SYM_ABI_VERSION 1

#define SYM_OK 0
#define SYM_E_INVALID (-1)   /* bad argument */
#define SYM_E_CUDA (-2)      /* a CUDA runtime call failed */
#define SYM_E_WORKSPACE (-3) /* ws_bytes smaller than the *_ws_bytes() query */
#define SYM_E_CAPACITY (-4)  /* output capacity too small (n_out holds the required size) */
#define SYM_E_UNSUPPORTED (-5)

int sym_abi_version(void);
const char *sym_last_error(void);
/* Fails with SYM_E_UNSUPPORTED unless the current device is compute capability 10.x. */
int sym_check_device(int *sm_count_host, int *cc_major_host, int *cc_minor_host);

/* ---- a1 layout: PauliwordOp.__init__ (base.py:42-74) holds bool[M,2n]; the engine holds packed rows */
int sym_pack(const uint8_t *symp, int64_t M, int32_t n_qubits, uint64_t *xz, void *stream);
int sym_unpack(const uint64_t *xz, int64_t M, int32_t n_qubits, uint8_t *symp, void *stream);
/* a3 Y_count (base.py:604-615): y[i] = popcount(X_i & Z_i) */
int sym_ycount(const uint64_t *xz, int64_t M, int32_t W, int32_t *y, void *stream);
/* GF(2)-linear 64-bit sketch of each row: L(r1 ^ r2) == L(r1) ^ L(r2). Dedup key of a row is
 * a bijective 64-bit finaliser of L(row), so equal sketches <=> equal keys. */
int sym_sketch_rows(const uint64_t *xz, int64_t M, int32_t W, uint64_t *sketch, void *stream);

/* ---- a4 multiply: PauliwordOp._multiply_by_operator (base.py:764-794)
 * Materialised cross terms in the reference's flattened order t = q*M + p (p indexes A, q indexes B):
 *   out_xz[t] = A[p] ^ B[q];  out_c[t] = A.c[p]*B.c[q]*(-1)^{|A.x[p]&B.z[q]|}*i^{(3(Y_p+Y_q)+Y_out) mod 4}
 * out_xz: uint64[M*N][2W], out_c: double[M*N][2]. For parity checks and small products. */
int sym_cross_mul(const uint64_t *a_xz, const double *a_c, int64_t M, const uint64_t *b_xz,
                  const double *b_c, int64_t N, int32_t W, uint64_t *out_xz, double *out_c, void *stream);

/* Fused product + cleanup (base.py:764-794 followed by utils.py:230-279) that never materialises
 * the M*N cross terms: dedup runs on 64-bit keys derived from the row sketches, rows are only
 * written for the survivors. zero_threshold < 0 disables the |c| > threshold filter (the
 * reference's `None`). Output rows are unique and leave in first-occurrence order of the
 * reference's flattened cross-term index t = q*M + p (base.py:783-792) at every size: small
 * products scatter by t, large ones (> 2^22 cross terms) run the ordered-tile mode (drop bit per
 * cross term, survivors streamed tile by tile); only rows wider than 1024 qubits or with a word
 * count that is not a power of two fall back to sorted-hash order above 2^22 cross terms (parity
 * is defined on canonically sorted term sets, SURVEY.md §8c).
 * n_out: device int64[1], receives the number of surviving terms. out_capacity: rows available in
 * out_xz/out_c; on overflow returns SYM_E_CAPACITY after a stream synchronise.
 * This call synchronises the stream once (it needs the survivor count to size the emit launch). */
size_t sym_mul_cleanup_ws_bytes(int64_t M, int64_t N, int32_t W);
/* Two-phase form so the caller can allocate exact-size outputs: _count runs everything up to the
 * survivor count U (one stream synchronise, plan left in ws); _emit writes the U rows (async) and
 * must be given the same operands and the untouched ws. */
int sym_mul_cleanup_count(const uint64_t *a_xz, const double *a_c, int64_t M, const uint64_t *b_xz,
                          const double *b_c, int64_t N, int32_t W, double zero_threshold,
                          int64_t *n_out, int64_t *n_out_host, void *ws, size_t ws_bytes, void *stream);
int sym_mul_cleanup_emit(const uint64_t *a_xz, const double *a_c, int64_t M, const uint64_t *b_xz,
                         const double *b_c, int64_t N, int32_t W, int64_t U, uint64_t *out_xz,
                         double *out_c, void *ws, size_t ws_bytes, void *stream);
int sym_mul_cleanup(const uint64_t *a_xz, const double *a_c, int64_t M, const uint64_t *b_xz,
                    const double *b_c, int64_t N, int32_t W, double zero_threshold, uint64_t *out_xz,
                    double *out_c, int64_t out_capacity, int64_t *n_out, int64_t *n_out_host,
                    void *ws, size_t ws_bytes, void *stream);

/* Same product + cleanup restricted to nblk disjoint rectangular blocks A[p0:p1) x B[q0:q1) of the
 * cross-term grid (blocks_host: HOST int64[nblk][4] = {p0, p1, q0, q1}, nblk <= 256); one block
 * {0, M_total, 0, N} is sym_mul_cleanup. This is the exchange-free sharded product of SURVEY.md
 * §8e: with both operands grouped by owner class (sym_class_partition) rank r passes the blocks
 * A_a x B_{a^r} and gets exactly the part of (A*B).cleanup() it owns. Survivors leave block by
 * block, in (q, p) order inside a block. Same two-phase contract as sym_mul_cleanup_count/_emit. */
size_t sym_mul_blocks_ws_bytes(int64_t M_total, int64_t N, int32_t W, const int64_t *blocks_host, int32_t nblk);
int sym_mul_blocks_count(const uint64_t *a_xz, const double *a_c, int64_t M_total, const uint64_t *b_xz,
                         const double *b_c, int64_t N, int32_t W, const int64_t *blocks_host, int32_t nblk,
                         double zero_threshold, int64_t *n_out, int64_t *n_out_host, void *ws,
                         size_t ws_bytes, void *stream);
/* sym_mul_blocks_count with the sketch and Y-count tables of A supplied by the caller (what
 * sym_sketch_rows / sym_ycount would compute; both NULL = computed here). */
int sym_mul_blocks_count_tables(const uint64_t *a_xz, const double *a_c, const uint64_t *a_sketch,
                                const int32_t *a_ycount, int64_t M_total, const uint64_t *b_xz,
                                const double *b_c, int64_t N, int32_t W, const int64_t *blocks_host,
                                int32_t nblk, double zero_threshold, int64_t *n_out, int64_t *n_out_host,
                                void *ws, size_t ws_bytes, void *stream);
int sym_mul_blocks_emit(const uint64_t *a_xz, const double *a_c, int64_t M_total, const uint64_t *b_xz,
                        const double *b_c, int64_t N, int32_t W, const int64_t *blocks_host, int32_t nblk,
                        int64_t U, uint64_t *out_xz, double *out_c, void *ws, size_t ws_bytes, void *stream);

/* ---- a5 cleanup: symplectic_cleanup (utils.py:230-279) / PauliwordOp.cleanup (base.py:617-638)
 * Unique rows with duplicates' coefficients summed in input order, then |c| > zero_threshold.
 * Output order: first occurrence (same as the reference). */
size_t sym_cleanup_ws_bytes(int64_t T, int32_t W);
int sym_cleanup_count(const uint64_t *xz, const double *c, int64_t T, int32_t W, double zero_threshold,
                      int64_t *n_out, int64_t *n_out_host, void *ws, size_t ws_bytes, void *stream);
int sym_cleanup_emit(const uint64_t *xz, const double *c, int64_t T, int32_t W, int64_t U,
                     uint64_t *out_xz, double *out_c, void *ws, size_t ws_bytes, void *stream);
int sym_cleanup(const uint64_t *xz, const double *c, int64_t T, int32_t W, double zero_threshold,
                uint64_t *out_xz, double *out_c, int64_t out_capacity, int64_t *n_out,
                int64_t *n_out_host, void *ws, size_t ws_bytes, void *stream);

/* ---- a7 commute: PauliwordOp.commutes_termwise (base.py:938-971) -> matmul_GF2 (utils.py:9-78)
 * out[i*N + j] = 1 if A[i] commutes with B[j] else 0 (uint8, the reference's bool[M,N]). */
int sym_commute(const uint64_t *a_xz, int64_t M, const uint64_t *b_xz, int64_t N, int32_t W,
                uint8_t *out, void *stream);
/* Tensor-core variant of sym_commute (same output): int8 tcgen05.mma on bits unpacked on the fly in
 * shared memory, int32 accumulators in TMEM, parity epilogue — the reference's own "integer GEMM,
 * then mod 2" formulation (utils.py:63-78). Wins over the bit-packed kernel for wide operators. */
size_t sym_commute_mma_ws_bytes(int64_t M, int64_t N, int32_t W);
int sym_commute_mma(const uint64_t *a_xz, int64_t M, const uint64_t *b_xz, int64_t N, int32_t W,
                    uint8_t *out, void *ws, size_t ws_bytes, void *stream);
/* Same with out_pitch bytes between output rows (out_pitch >= N). A pitch that is a multiple of 32
 * keeps every row 16-byte aligned, so ragged N (NaCl: 42 599 terms) takes the 32-byte vector stores
 * instead of per-byte stores (measured 10x at 36 qubits); bytes N..out_pitch-1 of a row are scratch. */
int sym_commute_mma_pitched(const uint64_t *a_xz, int64_t M, const uint64_t *b_xz, int64_t N, int32_t W,
                            uint8_t *out, int64_t out_pitch, void *ws, size_t ws_bytes, void *stream);
/* Mirrors the blocks on and above the block diagonal (square blocks of `block_rows` rows, a multiple of 32) of a
 * symmetric byte matrix into its lower triangle, in place. With it `adjacency_matrix`
 * (symmer/operators/base.py:1054-1062: commutes_termwise of an operator with itself) computes only the upper block
 * triangle: sym_commute* on A[i0:i1) x A[i0:M) for every block row, then one mirror pass. */
int sym_mirror_upper(uint8_t *matrix, int64_t M, int64_t pitch, int64_t block_rows, void *stream);

/* Same symplectic inner product, bit-packed output: out_bits[i][j/32] bit j%32 (row stride
 * ceil(N/32) uint32). Used when the matrix is consumed on the device (masks, graph colouring). */
int sym_commute_bits(const uint64_t *a_xz, int64_t M, const uint64_t *b_xz, int64_t N, int32_t W,
                     uint32_t *out_bits, void *stream);

/* Qubit-wise commutation: PauliwordOp.qubitwise_commutes_termwise / adjacency_matrix_qwc
 * (base.py:985-1009, 1065-1072). out[i*N + j] = 1 iff on every qubit where A[i] and B[j] both act
 * non-trivially they carry the same Pauli (uint8, the reference's bool[M,N]). */
int sym_commute_qwc(const uint64_t *a_xz, int64_t M, const uint64_t *b_xz, int64_t N, int32_t W,
                    uint8_t *out, void *stream);

/* ---- a8 rotations: PauliwordOp._rotate_by_single_Pword (base.py:1090-1161)
 * One rotation R P R^dagger, R = exp(i*angle/2*Q), Q = q_xz (a single packed row, coefficient 1).
 * mode 0: general angle: writes M + M_ac rows (row i keeps slot i with cos*c for anticommuting P;
 *         the new terms -i*sin*P*Q are appended from slot M in row order) WITHOUT dedup; follow
 *         with sym_cleanup (the one dedup the algebra needs; the reference runs four).
 *         out_xz/out_c capacity must be 2*M rows.
 * mode 1: Clifford, odd multiple of pi/2: anticommuting rows become (-i)*P*Q*sign; M rows out.
 * mode 2: Clifford, even multiple: anticommuting rows * sign; M rows out.
 * mode 4: general angle, padded: exactly 2*M rows out, no flag scan and no count to read back. Row M+i is
 *         the -i*sin*P*Q term of an anticommuting row i and, for a commuting row, a copy of row i with
 *         coefficient 0, which the sym_cleanup that follows merges into row i (same survivors, same order,
 *         same sums as mode 0). Takes no workspace.
 * `sign` is +1 or -1 (the reference's `int_part in [2,3]` rule, base.py:1148-1149).
 * n_out: device int64[1]. Fully asynchronous. */
size_t sym_rotate_ws_bytes(int64_t M);
int sym_rotate(const uint64_t *xz, const double *c, int64_t M, int32_t W, const uint64_t *q_xz,
               double cos_a, double sin_a, int32_t mode, double sign, uint64_t *out_xz, double *out_c,
               int64_t *n_out, void *ws, size_t ws_bytes, void *stream);

/* Fused form of the general rotation INCLUDING its dedup (large operators). sym_rotate_split leaves
 * the M rows stably partitioned into (commuting with Q | anticommuting with Q), coefficients
 * untouched, together with the row sketches and Y counts of the partitioned rows (computed in the
 * same read as the commutation test); n_commuting: device int64[1]. The rotation is then ONE
 * block-list product of the split operator with the three-row operator [I, cos*I, -i*sin*Q]
 * (sym_mul_blocks_count_tables / sym_mul_blocks_emit with blocks {0,nc,0,1} and {nc,M,1,3}):
 * base.py:1090-1161 expressed through base.py:764-794, the rotated rows are never materialised
 * before the dedup. out_sketch: uint64[M], out_ycount: int32[M]. */
size_t sym_rotate_split_ws_bytes(int64_t M);
int sym_rotate_split(const uint64_t *xz, const double *c, int64_t M, int32_t W, const uint64_t *q_xz,
                     uint64_t *out_xz, double *out_c, uint64_t *out_sketch, int32_t *out_ycount,
                     int64_t *n_commuting, void *ws, size_t ws_bytes, void *stream);

/* ---- a9/a10 matrix-free operator application: to_sparse_matrix (base.py:1458-1510) semantics,
 * qubit 0 = most significant bit of the basis index.
 * sym_term_masks: per term, basis-index masks x, z (int64, n_qubits <= 62) and the coefficient with
 * (-i)^Y folded in. The apply/expval/CSR kernels take the terms SORTED BY x MASK (the host sorts
 * with sym_sort_pairs) so that terms sharing a column offset share one gather of psi. */
int sym_term_masks(const uint64_t *xz, const double *c, int64_t M, int32_t n_qubits, int64_t *x_masks,
                   int64_t *z_masks, double *c_phased, void *stream);
/*   y[r - row_begin] = sum_t c'_t (-1)^{popcount(r & z_t)} psi[r ^ x_t]   for r in [row_begin, row_end)
 * psi: complex128[2^n]; y: complex128[row_end-row_begin]; n_qubits <= 40. real_coeffs != 0 promises
 * that every c' has zero imaginary part (halves the FP64 work; molecular Hamiltonians). */
int sym_apply(const int64_t *x_masks, const int64_t *z_masks, const double *c_phased, int64_t M,
              int32_t n_qubits, const double *psi, double *y, int64_t row_begin, int64_t row_end,
              int32_t real_coeffs, void *stream);
/* partial[0..1] += sum_{r in [row_begin,row_end)} conj(psi[r]) * (H psi)[r]  (device double[2],
 * zero it first). The 2^n basis shards over ranks by row range; all-reduce the two doubles.
 * real_coeffs: 0 complex, 1 all phased coefficients real, 2 symmetric mode (see sym_expval_prepare_sym). */
int sym_expval(const int64_t *x_masks, const int64_t *z_masks, const double *c_phased, int64_t M,
               int32_t n_qubits, const double *psi, double *partial, int64_t row_begin, int64_t row_end,
               int32_t real_coeffs, void *stream);
/* Symmetric expectation-value mode for Hermitian operators whose phased coefficients are all real
 * (every term has an even number of Y and a real coefficient: molecular Hamiltonians). The pair of
 * basis rows (r, r ^ x) contributes a complex-conjugate pair, so a group of terms whose x mask has
 * its highest set bit h >= 11 is evaluated only on one half of the rows (bit h clear or set, a
 * pseudo-random choice per group that keeps CTAs and row shards balanced), with doubled
 * coefficients: half the work. sym_expval_prepare_sym builds that table once per operator
 * (z_sym = z | side << 63 | (h+1) << 56 | group_length << 40, c_sym = 2c for those groups, copies
 * otherwise; x_masks unchanged); pass
 * it to sym_expval with real_coeffs = 2 and row ranges aligned to 2048. partial[0] receives the
 * (real) expectation value, partial[1] is left untouched (exactly zero for a Hermitian operator).
 * Row-range partial sums are no longer the sums over those rows, but they still add up to the total
 * when every range uses this mode (the 2^n basis shards over ranks as before). */
int sym_expval_prepare_sym(const int64_t *x_masks, const int64_t *z_masks, const double *c_phased,
                           int64_t M, int64_t *z_sym, double *c_sym, void *stream);
/* CSR emitter for small n (parity with to_sparse_matrix): G distinct x masks (x_groups, ascending),
 * terms sorted by x with group g spanning [group_start[g], group_start[g+1]). Every row gets exactly
 * G entries sorted by column (explicit zeros kept). data: double[2^n*G][2], indices: int64[2^n*G],
 * indptr: int64[2^n+1]. */
int sym_to_csr(const int64_t *z_masks, const double *c_phased, int64_t M, int32_t n_qubits,
               const int64_t *x_groups, int64_t G, const int32_t *group_start, double *data,
               int64_t *indices, int64_t *indptr, void *stream);

/* ---- inverse of a9: PauliwordOp.from_matrix (base.py:238-425), get_ij_operator (base.py:2354-2436).
 * Pauli decomposition by Walsh-Hadamard transforms of the XOR-diagonals d_x[r] = M[r, r^x] (basis index r
 * with qubit 0 = most significant bit):  c'_{x,z} = 2^-n sum_r (-1)^{popcount(r & z)} M[r, r^x], and the
 * coefficient of the Pauli with masks (x, z) is c' * i^{popcount(x & z)}.
 * sym_pauli_decompose_dense: matrix = complex128[2^n][2^n] row-major (n_qubits <= 15), out[x][z] = c'.
 * sym_pauli_decompose_diagonals: diag = complex128[K][2^n], the K populated diagonals of a sparse matrix,
 *   transformed in place (diag[k][z] = c' for the k-th x).
 * sym_rows_from_masks: inverse of sym_term_masks — masks + c' -> packed single-word rows and coefficients
 *   with the i^{popcount(x&z)} factor applied (1 <= n_qubits <= 62). */
int sym_pauli_decompose_dense(const double *matrix, int32_t n_qubits, double *out, void *stream);
int sym_pauli_decompose_diagonals(double *diag, int64_t K, int32_t n_qubits, void *stream);
int sym_rows_from_masks(const int64_t *x_masks, const int64_t *z_masks, const double *c_phased, int64_t M,
                        int32_t n_qubits, uint64_t *xz, double *c, void *stream);

/* ---- a11 GF(2): _rref_binary (utils.py:292-315), row-driven pivot rule, no row swaps.
 * bits: uint64[R][Cw] bit-packed rows (column j = bit j%64 of word j/64), reduced in place.
 * pivots: device int32[R], pivot column of each row after reduction or -1 for a zero row. */
size_t sym_rref_ws_bytes(int64_t R);
int sym_rref(uint64_t *bits, int64_t R, int64_t C, int64_t Cw, int32_t *pivots, void *ws,
             size_t ws_bytes, void *stream);
/* Column reduction (_cref_binary / cref_binary, utils.py:337-359; generator_reconstruction,
 * base.py:523-560) works on the transpose. sym_bit_transpose: in uint64[R][Cw_in] (R rows of
 * Cw_in*64 bit columns) -> out uint64[Cw_in*64][Cw_out], Cw_out >= ceil(R/64); bits beyond R are 0.
 * sym_or_rows: out[k] = OR_i bits[rows[i]][k] over n_rows selected rows (rows == NULL: rows 0..n_rows-1)
 * — the "all remaining columns are zero" test of generator_reconstruction. */
int sym_bit_transpose(const uint64_t *in, int64_t R, int64_t Cw_in, uint64_t *out, int64_t Cw_out,
                      void *stream);
int sym_or_rows(const uint64_t *bits, int64_t Cw, const int32_t *rows, int64_t n_rows, uint64_t *out,
                void *stream);
/* bool[R][C] <-> packed uint64[R][Cw] helpers for the GF(2) matrices (any C). */
int sym_pack_matrix(const uint8_t *m, int64_t R, int64_t C, uint64_t *bits, int64_t Cw, void *stream);
int sym_unpack_matrix(const uint64_t *bits, int64_t R, int64_t C, int64_t Cw, uint8_t *m, void *stream);

/* ---- SURVEY §8f-2: S3Projection._perform_projection (symmer/projection/base.py:44-84) on packed rows.
 * The S stabilizers are single-qubit Paulis: stab_cols[j] (device int32) is the column of stabilizer
 * j's single set bit in the [X | Z] symplectic layout (q < n: X_q, n + q: Z_q), stab_eigs[j] (device
 * double) its +/-1 eigenvalue. Rows anticommuting with any stabilizer are dropped; the coefficient
 * of a kept row is multiplied by the eigenvalue of every stabilizer whose Pauli appears in it; the
 * kept rows are written over the n_free free qubits only (free_qubits: device int32, ascending;
 * output layout uint64[*][2*W'], W' = max(1, ceil(n_free/64))) in input order. out_xz / out_c must
 * hold M rows. n_out (device int64, may be NULL) / n_out_host (may be NULL; forces one stream
 * synchronise) receive the number of kept rows. Duplicates are NOT merged: follow with sym_cleanup. */
size_t sym_project_ws_bytes(int64_t M, int32_t n_free);
int sym_project(const uint64_t *xz, const double *c, int64_t M, int32_t W, int32_t n_qubits,
                const int32_t *stab_cols, const double *stab_eigs, int32_t S, const int32_t *free_qubits,
                int32_t n_free, uint64_t *out_xz, double *out_c, int64_t *n_out, int64_t *n_out_host,
                void *ws, size_t ws_bytes, void *stream);

/* out[i] = words[perm[i] * pitch_words + column] (perm NULL = identity): one 64-bit word column of a row-major matrix
 * in a given row order. Key of one pass of the word-by-word lexicographic sort that replaces
 * `np.lexsort(symp_matrix.T)` (symmer/operators/base.py:469-470) and of `__eq__` (base.py:640-662). */
int sym_gather_column(const uint64_t *words, int64_t M, int64_t pitch_words, int64_t column, const uint32_t *perm,
                      uint64_t *out, void *stream);

/* out row i = row perm[i] of (xz, c) (c / out_c may be NULL): reorders an operator on the device
 * (`PauliwordOp.sort`, `__getitem__`: base.py:453-489). */
int sym_gather_rows(const uint64_t *xz, const double *c, const uint32_t *perm, int64_t M_out, int32_t W, uint64_t *out_xz,
                    double *out_c, void *stream);

/* Exact join of two row sets (`words` uint64 per row) on equal rows: match[i] = index of the right row equal to left
 * row i, or -1. keys_* are 64-bit row sketches; the right keys are sorted and perm_r maps sorted position -> row.
 * Replaces the Python dict join of `QuantumState.__mul__` (bra * ket, base.py:1781-1830). */
int sym_join_rows(const uint64_t *keys_l, const uint64_t *rows_l, int64_t M, const uint64_t *keys_r_sorted,
                  const uint32_t *perm_r, const uint64_t *rows_r, int64_t N, int32_t words, int32_t *match, void *stream);

/* ---- qubit relabelling / embedding: PauliwordOp.reindex (base.py:493-521), PauliwordOp.tensor
 * (base.py:1188-1204), QuantumState.reindex (base.py:1910-1936).
 * Output rows have n_out qubits (uint64[M][2*W'], W' = max(1, ceil(n_out/64))); bit k of the output
 * X (Z) block = bit src[k] of the input X (Z) block, 0 where src[k] < 0 (src: device int32[n_out],
 * every entry < 64*W_in). Coefficients are untouched. */
int sym_gather_qubits(const uint64_t *xz, int64_t M, int32_t W_in, const int32_t *src, int32_t n_out,
                      uint64_t *out_xz, void *stream);

/* ---- multi-GPU building blocks (SURVEY.md §8e): the product path split at its exchange point.
 * A record is one 64-bit word  [ hash : 62-tb bits | t : tb bits | e : 2 bits ]  with
 * hash = top bits of mix64(sketch(A[p]) ^ sketch(B[q])), t = global flattened cross-term index
 * q*M_total + p, e = phase exponent of the pair, tb = ceil(log2(M_total*N)) (M_total*N < 4e9).
 * Equal rows have equal hash fields, so the owner of a row is a function of its top hash bits and
 * only these 8-byte records (never rows) cross NVLink; the owner rebuilds rows from its replicas of
 * A and B.
 * sym_pair_records: records of the block A[p_begin:p_end) x B, written in (q, p) order. */
size_t sym_pair_records_ws_bytes(int64_t M_total, int64_t N, int32_t W);
int sym_pair_records(const uint64_t *a_xz, int64_t M_total, int64_t p_begin, int64_t p_end,
                     const uint64_t *b_xz, int64_t N, int32_t W, uint64_t *recs, void *ws,
                     size_t ws_bytes, void *stream);
/* Records of nblk rectangular blocks A[p0:p1) x B[q0:q1), written back to back in block order
 * ((q, p) order inside a block); blocks_host: HOST int64[nblk][4] = {p0, p1, q0, q1}. t = q*M_total + p
 * with the global row indices. `recs` must hold the sum of the block sizes. */
int sym_pair_records_blocks(const uint64_t *a_xz, int64_t M_total, const uint64_t *b_xz, int64_t N,
                            int32_t W, const int64_t *blocks_host, int32_t nblk, uint64_t *recs,
                            void *ws, size_t ws_bytes, void *stream);
/* Exchange-free ownership for sharded products. owner(row) = log2_parts parity bits of the row's
 * GF(2)-linear sketch, hence owner(A[p] ^ B[q]) = owner(A[p]) ^ owner(B[q]): with both operands
 * grouped by owner class, rank r generates exactly the cross terms it owns (blocks A_a x B_{a^r},
 * sym_pair_records_blocks) and no record crosses NVLink.
 * sym_owner_classes: cls[i] = owner class of row i (ws >= 8*M bytes, rounded up to 256).
 * sym_class_partition: stable grouping of an operator by class: out rows/coefficients in class
 * order (input order inside a class), perm[i] = source row of output row i (may be NULL),
 * counts: device int64[1 << log2_parts] class sizes. c/out_c may be NULL. */
int sym_owner_classes(const uint64_t *xz, int64_t M, int32_t W, int32_t log2_parts, uint8_t *cls,
                      void *ws, size_t ws_bytes, void *stream);
size_t sym_class_partition_ws_bytes(int64_t M);
int sym_class_partition(const uint64_t *xz, const double *c, int64_t M, int32_t W, int32_t log2_parts,
                        uint64_t *out_xz, double *out_c, int32_t *perm, int64_t *counts, void *ws,
                        size_t ws_bytes, void *stream);
/* Stable partition of records by owner = rec >> (64 - log2_parts); counts: device int64[parts]. */
size_t sym_partition_ws_bytes(int64_t T);
int sym_partition_records(const uint64_t *recs, int64_t T, int32_t log2_parts, uint64_t *out_recs,
                          int64_t *counts, void *ws, size_t ws_bytes, void *stream);
/* Dedup + coefficient reduction + row emission for T records whose rows are A[p] ^ B[q] (A, B
 * fully resident, M_total rows in A). recs is clobbered; pass the same buffer to _emit. Output in
 * sorted-hash order. Same two-phase contract as sym_mul_cleanup_count/_emit. */
size_t sym_dedup_records_ws_bytes(int64_t T, int32_t W);
int sym_dedup_records_count(uint64_t *recs, int64_t T, const uint64_t *a_xz, const double *a_c,
                            int64_t M_total, const uint64_t *b_xz, const double *b_c, int64_t N,
                            int32_t W, double zero_threshold, int64_t *n_out, int64_t *n_out_host,
                            void *ws, size_t ws_bytes, void *stream);
int sym_dedup_records_emit(const uint64_t *recs, int64_t T, const uint64_t *a_xz, const double *a_c,
                           int64_t M_total, const uint64_t *b_xz, const double *b_c, int64_t N, int32_t W,
                           int64_t U, uint64_t *out_xz, double *out_c, void *ws, size_t ws_bytes,
                           void *stream);
int sym_dedup_records(uint64_t *recs, int64_t T, const uint64_t *a_xz, const double *a_c,
                      int64_t M_total, const uint64_t *b_xz, const double *b_c, int64_t N, int32_t W,
                      double zero_threshold, uint64_t *out_xz, double *out_c, int64_t out_capacity,
                      int64_t *n_out, int64_t *n_out_host, void *ws, size_t ws_bytes, void *stream);

/* ---- primitives exported for tests and reuse */
/* Stable LSD radix sort of (key, val) pairs on key bits [begin_bit, 64). Result in keys/vals. */
size_t sym_sort_pairs_ws_bytes(int64_t T);
int sym_sort_pairs(uint64_t *keys, uint32_t *vals, int64_t T, int32_t begin_bit, void *ws,
                   size_t ws_bytes, void *stream);
/* Tuning knobs (A/B switches kept for measurement). which = 0: cross-term count up to which
 * sym_mul_cleanup scatters by t (above it: knob 6; default 2^22); 4: apply/expval kernel (1 binned,
 * 0 four-row); 5: GF(2) large path (1 blocked panels, 0 one pivot per sweep); 6: large products in
 * ordered-tile mode (1, default) or sorted-hash order (0); 7: B rows per CTA of the tiled row emission
 * (default 16); 8: record sort as one-sweep passes with decoupled look-back (1, default) or histogram +
 * scan + scatter per pass (0); 10: duplicate detection of ordered-tile products by class-local
 * enumeration (1, default) or by the global record sort (0); 11: class kernel shape (2, default: compact
 * 4-byte entries with the presence filter; 3: the same without the filter, 128 KB table; 1: 8-byte entries,
 * 9216 records per class; 0: 512-thread CTAs, 4096 records). Any other number is SYM_E_INVALID. */
int sym_set_tuning(int32_t which, int64_t value);
/* Measurement hook: two cudaEvent_t (as void*, NULL to disable) recorded on the stream immediately
 * before and after the row-emission kernel (emit_kernel) of the next *_emit calls, so that a
 * benchmark can time the dominant kernel alone with CUDA events. */
int sym_set_emit_events(void *before_event, void *after_event);
/* Test hook: AND every dedup key with this mask (default ~0) to force sketch collisions. */
int sym_debug_set_key_mask(uint64_t mask);
/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
int64_t sym_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SYMMER_B200_H */
