// PauliwordOp multiplication (symmer/operators/base.py:764-794): all-pairs cross terms as XOR of
// packed rows with the i-phase from popcounts of X&Z overlaps.
//
// Two forms:
//   * sym_cross_mul     — materialises the M*N cross terms (parity checks, small products);
//   * pair records      — never materialises rows: for every pair (p, q) emit one 64-bit record
//                         key = (mix64(sketch(A[p]) ^ sketch(B[q])) & ~3) | phase_exponent(p, q)
//                         which is all the dedup needs; rows are rebuilt only for survivors.
// Integer/bit work bound by the LOP3 pipe and by the 8 B/pair store; no tensor cores.
#include "rows.cuh"
#include "sort.cuh"

namespace symb {

// phase exponent e with coefficient factor i^e = (-1)^{|xa&zb|} * i^{(3(Ya+Yb)+Yout) mod 4}  (base.py:785-788)
__device__ __forceinline__ int finish_phase(int ya, int yb, uint64_t s, uint64_t c0, uint64_t c1) {
    int yout = __popcll(c0) + 2 * __popcll(c1);
    int sgn = __popcll(s) & 1;
    return (3 * (ya + yb) + yout + 2 * sgn) & 3;
}

// ---------------------------------------------------------------------------------------------
// tiled pair kernel: thread = one A row held in registers, CTA streams QCH B rows through smem
// ---------------------------------------------------------------------------------------------
constexpr int PAIR_THREADS = 256;
constexpr int PAIR_QCH = 64;

template <int WT>
__global__ void __launch_bounds__(PAIR_THREADS) pair_records_kernel(
    const uint64_t *__restrict__ a_xz, const uint64_t *__restrict__ a_sk, const int32_t *__restrict__ a_y, uint32_t M_total,
    uint32_t p_begin, uint32_t p_end, const uint64_t *__restrict__ b_xz, const uint64_t *__restrict__ b_sk,
    const int32_t *__restrict__ b_y, uint32_t N, uint32_t q_off, int W, uint64_t key_mask, RecFmt fmt,
    uint64_t *__restrict__ recs, uint32_t qch) {
    // B tile: qch <= QCH rows (fewer for small products, so that the grid still covers the SMs),
    // (x_w, z_w) interleaved so one 16-byte shared load feeds a word step
    __shared__ ulonglong2 sb[PAIR_QCH][WT];
    __shared__ uint64_t sb_sk[PAIR_QCH];
    __shared__ int sb_y[PAIR_QCH];

    const uint32_t q0 = blockIdx.y * qch;
    const uint32_t nq = min(qch, N - q0);
    for (int i = threadIdx.x; i < (int)qch * WT; i += blockDim.x) {
        int qi = i / WT, w = i % WT;
        ulonglong2 v = make_ulonglong2(0ull, 0ull);
        if ((uint32_t)qi < nq && w < W) {
            const uint64_t *row = b_xz + (size_t)(q0 + qi) * 2 * W;
            v.x = row[w];
            v.y = row[W + w];
        }
        sb[qi][w] = v;
    }
    for (int i = threadIdx.x; i < (int)qch; i += blockDim.x) {
        sb_sk[i] = ((uint32_t)i < nq) ? b_sk[q0 + i] : 0ull;
        sb_y[i] = ((uint32_t)i < nq) ? b_y[q0 + i] : 0;
    }

    const uint32_t p = p_begin + blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = p < p_end;
    uint64_t xa[WT], za[WT];
    uint64_t ska = 0;
    int ya = 0;
    if (active) {
        const uint64_t *row = a_xz + (size_t)p * 2 * W;
        if (WT >= 2 && (W & 1) == 0) {   // 16-byte loads: a thread's row is strided against its neighbours' either way
            const uint4 *row4 = reinterpret_cast<const uint4 *>(row);
#pragma unroll
            for (int w = 0; w < WT; w += 2) {
                uint4 xv = make_uint4(0u, 0u, 0u, 0u), zv = make_uint4(0u, 0u, 0u, 0u);
                if (w < W) {
                    xv = row4[w >> 1];
                    zv = row4[(W + w) >> 1];
                }
                xa[w] = ((uint64_t)xv.y << 32) | xv.x;
                za[w] = ((uint64_t)zv.y << 32) | zv.x;
                if (w + 1 < WT) {
                    xa[w + 1] = ((uint64_t)xv.w << 32) | xv.z;
                    za[w + 1] = ((uint64_t)zv.w << 32) | zv.z;
                }
            }
        } else {
#pragma unroll
            for (int w = 0; w < WT; ++w) {
                xa[w] = (w < W) ? row[w] : 0ull;
                za[w] = (w < W) ? row[W + w] : 0ull;
            }
        }
        ska = a_sk[p];
        ya = a_y[p];
    } else {
#pragma unroll
        for (int w = 0; w < WT; ++w) xa[w] = za[w] = 0ull;
    }
    __syncthreads();
    if (!active) return;

    const uint32_t m_blk = p_end - p_begin;
    const uint32_t p_local = p - p_begin;
    for (uint32_t qi = 0; qi < nq; ++qi) {
        uint64_t s = 0, c0 = 0, c1 = 0;
#pragma unroll
        for (int w = 0; w < WT; ++w) {
            const ulonglong2 b = sb[qi][w];  // broadcast read
            s ^= xa[w] & b.y;
            const uint64_t v = (xa[w] ^ b.x) & (za[w] ^ b.y);
            c1 ^= c0 & v;
            c0 ^= v;
        }
        const int e = finish_phase(ya, sb_y[qi], s, c0, c1);
        const size_t j = (size_t)(q0 + qi) * m_blk + p_local;
        recs[j] = fmt.make(mix64(ska ^ sb_sk[qi]) & key_mask, (uint64_t)(q_off + q0 + qi) * M_total + p, e);
    }
}

// Ordered-tile mode: records without the phase exponent (the tiled emission computes it from the rows it
// holds in registers), so a record is just the mixed XOR of two sketches: 8 B store per pair, HBM-write bound.
constexpr int KEYS_QCH = 64;
__global__ void __launch_bounds__(256) pair_keys_kernel(const uint64_t *__restrict__ a_sk, uint32_t M_total, uint32_t p_begin,
                                                         uint32_t m_blk, const uint64_t *__restrict__ b_sk, uint32_t nq,
                                                         uint32_t q_off, uint64_t key_mask, RecFmt fmt,
                                                         uint64_t *__restrict__ recs) {
    const uint32_t p_local = blockIdx.x * blockDim.x + threadIdx.x;
    if (p_local >= m_blk) return;
    const uint32_t p = p_begin + p_local;
    const uint64_t ska = a_sk[p];
    const uint32_t q_lo = blockIdx.y * KEYS_QCH, q_hi = min(nq, q_lo + KEYS_QCH);
#pragma unroll 4
    for (uint32_t q = q_lo; q < q_hi; ++q)
        recs[(size_t)q * m_blk + p_local] = fmt.make(mix64(ska ^ b_sk[q]) & key_mask, (uint64_t)(q_off + q) * M_total + p, 0);
}

// generic fallback for W > 16: one thread per pair, rows read through L1/L2
__global__ void __launch_bounds__(256) pair_records_generic_kernel(
    const uint64_t *__restrict__ a_xz, const uint64_t *__restrict__ a_sk, const int32_t *__restrict__ a_y, uint32_t M_total,
    uint32_t p_begin, uint32_t p_end, const uint64_t *__restrict__ b_xz, const uint64_t *__restrict__ b_sk,
    const int32_t *__restrict__ b_y, uint32_t N, uint32_t q_off, int W, uint64_t key_mask, RecFmt fmt,
    uint64_t *__restrict__ recs) {
    const uint32_t m_blk = p_end - p_begin;
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= (size_t)m_blk * N) return;
    uint32_t q = (uint32_t)(j / m_blk);
    uint32_t p = p_begin + (uint32_t)(j - (size_t)q * m_blk);
    const uint64_t *ra = a_xz + (size_t)p * 2 * W, *rb = b_xz + (size_t)q * 2 * W;
    uint64_t s = 0, c0 = 0, c1 = 0;
    for (int w = 0; w < W; ++w) {
        uint64_t xa = ra[w], za = ra[W + w], xb = rb[w], zb = rb[W + w];
        s ^= xa & zb;
        uint64_t v = (xa ^ xb) & (za ^ zb);
        c1 ^= c0 & v;
        c0 ^= v;
    }
    int e = finish_phase(a_y[p], b_y[q], s, c0, c1);
    recs[j] = fmt.make(mix64(a_sk[p] ^ b_sk[q]) & key_mask, (uint64_t)(q_off + q) * M_total + p, e);
}

static int launch_pair_records(const uint64_t *a_xz, const uint64_t *a_sk, const int32_t *a_y, int64_t M_total,
                               int64_t p_begin, int64_t p_end, const uint64_t *b_xz, const uint64_t *b_sk,
                               const int32_t *b_y, int64_t N, int W, RecFmt fmt, uint64_t *recs, cudaStream_t st,
                               int64_t q_off = 0) {
    // b_xz / b_sk / b_y point at B row q_off; N rows from there. t uses the global index q_off + q.
    const int64_t m_blk = p_end - p_begin;
    if (m_blk <= 0 || N <= 0) return SYM_OK;
    // CTA shape: 256 A rows x 64 B rows; a small product (C1: 500 x 500 terms would be 2 x 8 CTAs) takes 64-row CTAs and
    // fewer B rows per CTA until the grid covers the SMs. Every CTA column re-reads the A rows with one 32-byte sector
    // per load (a thread's row is strided against its neighbours'), so the B tile is not shrunk further than needed.
    int threads = PAIR_THREADS;
    uint32_t qch = PAIR_QCH;
    if (((m_blk + PAIR_THREADS - 1) / PAIR_THREADS) * ((N + PAIR_QCH - 1) / PAIR_QCH) < 2 * 148) {
        threads = 64;
        while (qch > 8 && ((m_blk + 63) / 64) * ((N + qch - 1) / qch) < 256) qch >>= 1;
    }
    dim3 grid((unsigned)((m_blk + threads - 1) / threads), (unsigned)((N + qch - 1) / qch));
#define PAIR_CASE(WT)                                                                                               \
    pair_records_kernel<WT><<<grid, threads, 0, st>>>(a_xz, a_sk, a_y, (uint32_t)M_total, (uint32_t)p_begin,   \
                                                           (uint32_t)p_end, b_xz, b_sk, b_y, (uint32_t)N,           \
                                                           (uint32_t)q_off, W, g_key_mask, fmt, recs, qch)
    if (grid.y > 65535) {
        set_error("too many B rows for one launch (N=%lld)", (long long)N);
        return SYM_E_UNSUPPORTED;
    }
    if (W <= 1) PAIR_CASE(1);
    else if (W <= 2) PAIR_CASE(2);
    else if (W <= 4) PAIR_CASE(4);
    else if (W <= 8) PAIR_CASE(8);
    else if (W <= 16) PAIR_CASE(16);
    else {
        int64_t total = m_blk * N;
        pair_records_generic_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
            a_xz, a_sk, a_y, (uint32_t)M_total, (uint32_t)p_begin, (uint32_t)p_end, b_xz, b_sk, b_y, (uint32_t)N,
            (uint32_t)q_off, W, g_key_mask, fmt, recs);
    }
#undef PAIR_CASE
    SYM_LAUNCH_OK();
    return SYM_OK;
}

// ---------------------------------------------------------------------------------------------
// materialised cross terms
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cross_rows_kernel(const uint64_t *__restrict__ a, uint32_t M, const uint64_t *__restrict__ b,
                                                          int64_t total_words, int words, uint64_t *__restrict__ out) {
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total_words) return;
    int64_t t = g / words;
    int k = (int)(g - t * words);
    uint32_t q = (uint32_t)(t / M), p = (uint32_t)(t - (int64_t)q * M);
    out[g] = a[(size_t)p * words + k] ^ b[(size_t)q * words + k];
}

__global__ void __launch_bounds__(256) cross_coeff_kernel(const uint64_t *__restrict__ a, const double *__restrict__ ac, uint32_t M,
                                                           const uint64_t *__restrict__ b, const double *__restrict__ bc,
                                                           int64_t T, int W, double2 *__restrict__ out_c) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    uint32_t q = (uint32_t)(t / M), p = (uint32_t)(t - (int64_t)q * M);
    const uint64_t *ra = a + (size_t)p * 2 * W, *rb = b + (size_t)q * 2 * W;
    uint64_t s = 0, c0 = 0, c1 = 0;
    int ya = 0, yb = 0;
    for (int w = 0; w < W; ++w) {
        uint64_t xa = ra[w], za = ra[W + w], xb = rb[w], zb = rb[W + w];
        ya += __popcll(xa & za);
        yb += __popcll(xb & zb);
        s ^= xa & zb;
        uint64_t v = (xa ^ xb) & (za ^ zb);
        c1 ^= c0 & v;
        c0 ^= v;
    }
    int e = finish_phase(ya, yb, s, c0, c1);
    double re, im;
    cmul(ac[2 * (size_t)p], ac[2 * (size_t)p + 1], bc[2 * (size_t)q], bc[2 * (size_t)q + 1], re, im);
    mul_i_pow(re, im, e);
    out_c[t] = make_double2(re, im);
}

}  // namespace symb

using namespace symb;

extern "C" int sym_cross_mul(const uint64_t *a_xz, const double *a_c, int64_t M, const uint64_t *b_xz, const double *b_c,
                             int64_t N, int32_t W, uint64_t *out_xz, double *out_c, void *stream) {
    SYM_REQUIRE(M >= 0 && N >= 0 && W >= 1, "bad size");
    SYM_REQUIRE(M < (int64_t)1 << 31 && N < (int64_t)1 << 31, "operand too large");
    int64_t T = M * N;
    if (T == 0) return SYM_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int64_t total_words = T * 2 * W;
    cross_rows_kernel<<<(unsigned)((total_words + 255) / 256), 256, 0, st>>>(a_xz, (uint32_t)M, b_xz, total_words, 2 * W,
                                                                            out_xz);
    SYM_LAUNCH_OK();
    cross_coeff_kernel<<<(unsigned)((T + 255) / 256), 256, 0, st>>>(a_xz, a_c, (uint32_t)M, b_xz, b_c, T, W,
                                                                   reinterpret_cast<double2 *>(out_c));
    SYM_LAUNCH_OK();
    return SYM_OK;
}

extern "C" size_t sym_pair_records_ws_bytes(int64_t M_total, int64_t N, int32_t W) {
    (void)W;
    return arena_need((size_t)(M_total > 0 ? M_total : 1), 8) + arena_need((size_t)(N > 0 ? N : 1), 8) +
           arena_need((size_t)(M_total > 0 ? M_total : 1), 4) + arena_need((size_t)(N > 0 ? N : 1), 4) + 1024;
}

static int prepare_operand_tables(const uint64_t *a_xz, int64_t M, const uint64_t *b_xz, int64_t N, int W, Arena &ar,
                                  uint64_t *&a_sk, uint64_t *&b_sk, int32_t *&a_y, int32_t *&b_y, cudaStream_t st) {
    a_sk = ar.take<uint64_t>((size_t)(M > 0 ? M : 1));
    b_sk = ar.take<uint64_t>((size_t)(N > 0 ? N : 1));
    a_y = ar.take<int32_t>((size_t)(M > 0 ? M : 1));
    b_y = ar.take<int32_t>((size_t)(N > 0 ? N : 1));
    if (!b_y) {
        set_error("workspace arena exhausted");
        return SYM_E_WORKSPACE;
    }
    return operand_tables(a_xz, M, b_xz, N, W, a_sk, a_y, b_sk, b_y, st);
}

extern "C" int sym_pair_records(const uint64_t *a_xz, int64_t M_total, int64_t p_begin, int64_t p_end,
                                const uint64_t *b_xz, int64_t N, int32_t W, uint64_t *recs, void *ws, size_t ws_bytes,
                                void *stream) {
    SYM_REQUIRE(M_total >= 0 && N >= 0 && W >= 1, "bad size");
    SYM_REQUIRE(0 <= p_begin && p_begin <= p_end && p_end <= M_total, "bad row block");
    SYM_REQUIRE(M_total * N < (int64_t)4000000000LL, "M_total*N must be < 4e9");
    if (ws_bytes < sym_pair_records_ws_bytes(M_total, N, W)) {
        set_error("workspace too small");
        return SYM_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    Arena ar(ws, ws_bytes);
    uint64_t *a_sk, *b_sk;
    int32_t *a_y, *b_y;
    SYM_TRY(prepare_operand_tables(a_xz, M_total, b_xz, N, W, ar, a_sk, b_sk, a_y, b_y, st));
    RecFmt fmt{t_bits_for(M_total * N)};
    return launch_pair_records(a_xz, a_sk, a_y, M_total, p_begin, p_end, b_xz, b_sk, b_y, N, W, fmt, recs, st);
}

extern "C" int sym_pair_records_blocks(const uint64_t *a_xz, int64_t M_total, const uint64_t *b_xz, int64_t N, int32_t W,
                                       const int64_t *blocks_host, int32_t nblk, uint64_t *recs, void *ws,
                                       size_t ws_bytes, void *stream) {
    SYM_REQUIRE(M_total >= 0 && N >= 0 && W >= 1 && nblk >= 0, "bad size");
    SYM_REQUIRE(M_total * N < (int64_t)4000000000LL, "M_total*N must be < 4e9");
    for (int b = 0; b < nblk; ++b) {
        const int64_t *q = blocks_host + 4 * b;
        SYM_REQUIRE(0 <= q[0] && q[0] <= q[1] && q[1] <= M_total, "bad A row block");
        SYM_REQUIRE(0 <= q[2] && q[2] <= q[3] && q[3] <= N, "bad B row block");
    }
    if (ws_bytes < sym_pair_records_ws_bytes(M_total, N, W)) {
        set_error("workspace too small");
        return SYM_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    Arena ar(ws, ws_bytes);
    uint64_t *a_sk, *b_sk;
    int32_t *a_y, *b_y;
    SYM_TRY(prepare_operand_tables(a_xz, M_total, b_xz, N, W, ar, a_sk, b_sk, a_y, b_y, st));
    RecFmt fmt{t_bits_for(M_total * N)};
    size_t off = 0;
    for (int b = 0; b < nblk; ++b) {
        const int64_t p0 = blocks_host[4 * b], p1 = blocks_host[4 * b + 1], q0 = blocks_host[4 * b + 2],
                      q1 = blocks_host[4 * b + 3];
        SYM_TRY(launch_pair_records(a_xz, a_sk, a_y, M_total, p0, p1, b_xz + (size_t)q0 * 2 * W, b_sk + q0, b_y + q0,
                                    q1 - q0, W, fmt, recs + off, st, q0));
        off += (size_t)(p1 - p0) * (size_t)(q1 - q0);
    }
    return SYM_OK;
}

extern "C" size_t sym_partition_ws_bytes(int64_t T) {
    if (T < 1) T = 1;
    return arena_need(record_hist_elems(T), 4) + 1024;
}

extern "C" int sym_partition_records(const uint64_t *recs, int64_t T, int32_t log2_parts, uint64_t *out_recs,
                                     int64_t *counts, void *ws, size_t ws_bytes, void *stream) {
    SYM_REQUIRE(T >= 0 && T < (int64_t)4000000000LL, "T out of range");
    SYM_REQUIRE(log2_parts >= 0 && log2_parts <= 8, "log2_parts must be in [0,8]");
    if (ws_bytes < sym_partition_ws_bytes(T)) {
        set_error("workspace too small");
        return SYM_E_WORKSPACE;
    }
    Arena ar(ws, ws_bytes);
    uint32_t *hist = ar.take<uint32_t>(record_hist_elems(T));
    return radix_partition(recs, nullptr, out_recs, nullptr, T, log2_parts, counts, hist, (cudaStream_t)stream);
}

extern "C" size_t sym_dedup_records_ws_bytes(int64_t T, int32_t W) {
    (void)W;
    return dedup_ws_bytes(T);
}

extern "C" int sym_dedup_records_count(uint64_t *recs, int64_t T, const uint64_t *a_xz, const double *a_c,
                                       int64_t M_total, const uint64_t *b_xz, const double *b_c, int64_t N, int32_t W,
                                       double zero_threshold, int64_t *n_out, int64_t *n_out_host, void *ws,
                                       size_t ws_bytes, void *stream) {
    SYM_REQUIRE(T >= 0 && T < (int64_t)4000000000LL, "T out of range");
    SYM_REQUIRE(M_total >= 1 && N >= 1 && W >= 1, "bad size");
    SYM_REQUIRE(M_total * N < (int64_t)4000000000LL, "M_total*N must be < 4e9");
    ProductRows rows{a_xz, b_xz, a_c, b_c, (uint32_t)M_total, 2 * W, (uint32_t)N};
    RecFmt fmt{t_bits_for(M_total * N)};
    return dedup_product_plan(Path::SORTED, recs, T, fmt, rows, zero_threshold, n_out, n_out_host, ws, ws_bytes,
                              (cudaStream_t)stream);
}

extern "C" int sym_dedup_records_emit(const uint64_t *recs, int64_t T, const uint64_t *a_xz, const double *a_c,
                                      int64_t M_total, const uint64_t *b_xz, const double *b_c, int64_t N, int32_t W,
                                      int64_t U, uint64_t *out_xz, double *out_c, void *ws, size_t ws_bytes, void *stream) {
    SYM_REQUIRE(T >= 0 && U >= 0 && U <= T, "bad counts");
    SYM_REQUIRE(M_total >= 1 && N >= 1 && W >= 1, "bad size");
    ProductRows rows{a_xz, b_xz, a_c, b_c, (uint32_t)M_total, 2 * W, (uint32_t)N};
    RecFmt fmt{t_bits_for(M_total * N)};
    return dedup_product_emit(Path::SORTED, recs, T, fmt, rows, U, out_xz, out_c, ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int sym_dedup_records(uint64_t *recs, int64_t T, const uint64_t *a_xz, const double *a_c, int64_t M_total,
                                 const uint64_t *b_xz, const double *b_c, int64_t N, int32_t W, double zero_threshold,
                                 uint64_t *out_xz, double *out_c, int64_t out_capacity, int64_t *n_out,
                                 int64_t *n_out_host, void *ws, size_t ws_bytes, void *stream) {
    int64_t U = 0;
    SYM_TRY(sym_dedup_records_count(recs, T, a_xz, a_c, M_total, b_xz, b_c, N, W, zero_threshold, n_out, &U, ws, ws_bytes,
                                    stream));
    if (n_out_host) *n_out_host = U;
    if (U > out_capacity) {
        set_error("output capacity %lld < %lld surviving terms", (long long)out_capacity, (long long)U);
        return SYM_E_CAPACITY;
    }
    return sym_dedup_records_emit(recs, T, a_xz, a_c, M_total, b_xz, b_c, N, W, U, out_xz, out_c, ws, ws_bytes, stream);
}

// Tuning knobs that select the path of a product (mul_blocks_plan reads them, nothing else does):
//   0  by_t_limit: below this many cross terms a whole product is emitted in first-occurrence (reference) order by t;
//      above, in the ordered-tile mode or in sorted-hash order, which keeps every pass of the dedup streaming (no
//      T-sized scatters)
//   6  ordered_tiles: 1 (default) = products above the limit use the ordered-tile mode (first-occurrence order at every
//      size, streaming tiled row emission); 0 = the sorted-hash order path
//   10 class_dedup: 1 (default) = class-local duplicate detection for ordered-tile products, 0 = global record sort
//   11 class_variant: class kernel (0: 512 threads x 2 CTAs/SM, 4096 records; 1: 1024 threads, 9216 records;
//      2 (default): compact 4-byte entries, 1024 threads, 18432 records per class, presence filter;
//      3: the same without the filter and with a 32768-slot table)
struct PathKnobs { int64_t by_t_limit; int ordered_tiles, class_dedup, class_variant; };
static PathKnobs g_path_knobs = {(int64_t)1 << 22, 1, 1, 2};
namespace symb { extern int g_apply_variant; extern int g_rref_variant; extern int g_tile_qgroup; extern int g_onesweep; }

extern "C" int sym_set_tuning(int32_t which, int64_t value) {
    if (which == 0) {
        g_path_knobs.by_t_limit = value;
        return SYM_OK;
    }
    if (which == 4) {
        symb::g_apply_variant = (int)value;
        return SYM_OK;
    }
    if (which == 5) {
        symb::g_rref_variant = (int)value;
        return SYM_OK;
    }
    if (which == 6) {
        g_path_knobs.ordered_tiles = (int)value;
        return SYM_OK;
    }
    if (which == 7) {
        symb::g_tile_qgroup = (int)value;
        return SYM_OK;
    }
    if (which == 8) {
        symb::g_onesweep = (int)value;
        return SYM_OK;
    }
    if (which == 10) {
        g_path_knobs.class_dedup = (int)value;
        return SYM_OK;
    }
    if (which == 11) {
        g_path_knobs.class_variant = (int)value;
        return SYM_OK;
    }
    set_error("unknown tuning knob %d", which);
    return SYM_E_INVALID;
}

extern "C" int sym_set_emit_events(void *before_event, void *after_event) {
    symb::set_emit_events((cudaEvent_t)before_event, (cudaEvent_t)after_event);
    return SYM_OK;
}

// ---------------------------------------------------------------------------------------------
// product + cleanup of a list of rectangular blocks of A x B (one block = the whole product)
// ---------------------------------------------------------------------------------------------
struct MulBlocksPlan {
    Path path;
    int64_t T;
    RecFmt fmt;
    int nblk;
    uint32_t n_seg;
    TileBlock blocks[256];
    // workspace slices
    uint64_t *a_sk, *b_sk;
    int32_t *a_y, *b_y;
    uint64_t *recs;
    TileBlock *d_blocks;   // ordered-tile paths
    uint32_t *drop;
    uint32_t *segoff;
    ClassJob job;          // TILES_CLASS
    void *class_ws;
    size_t class_ws_bytes;
    void *rest;
    size_t rest_bytes;
    size_t need;

    bool tiles() const { return path == Path::TILES_SORT || path == Path::TILES_CLASS; }
};

static int mul_blocks_plan(int64_t M_total, int64_t N, int32_t W, const int64_t *blocks_host, int32_t nblk, void *ws,
                           size_t ws_bytes, MulBlocksPlan &P, const PathKnobs &knobs = g_path_knobs) {
    SYM_REQUIRE(M_total >= 0 && N >= 0 && W >= 1, "bad size");
    SYM_REQUIRE(nblk >= 0 && nblk <= 256, "at most 256 blocks");
    SYM_REQUIRE(M_total * N < (int64_t)4000000000LL, "M_total*N must be < 4e9 cross terms per call");
    SYM_REQUIRE(nblk == 0 || blocks_host != nullptr, "blocks_host is NULL");
    P.nblk = nblk;
    P.T = 0;
    P.fmt = RecFmt{t_bits_for(M_total * N)};
    int64_t segs = 0;
    for (int b = 0; b < nblk; ++b) {
        const int64_t *q = blocks_host + 4 * b;
        SYM_REQUIRE(0 <= q[0] && q[0] <= q[1] && q[1] <= M_total, "bad A row block");
        SYM_REQUIRE(0 <= q[2] && q[2] <= q[3] && q[3] <= N, "bad B row block");
        for (int o = 0; o < b; ++o) {   // rectangles must not overlap: every cross term is generated once
            const int64_t *r = blocks_host + 4 * o;
            const bool disjoint = q[1] <= r[0] || r[1] <= q[0] || q[3] <= r[2] || r[3] <= q[2] || q[0] == q[1] ||
                                  q[2] == q[3] || r[0] == r[1] || r[2] == r[3];
            SYM_REQUIRE(disjoint, "blocks overlap");
        }
        TileBlock &tb = P.blocks[b];
        tb.p0 = (uint32_t)q[0];
        tb.m_blk = (uint32_t)(q[1] - q[0]);
        tb.q0 = (uint32_t)q[2];
        tb.nq = (uint32_t)(q[3] - q[2]);
        tb.ptiles = (tb.m_blk + TILE_ROWS - 1) / TILE_ROWS;
        tb.seg_base = (uint32_t)segs;
        tb.t_base = (uint32_t)P.T;
        segs += (int64_t)tb.nq * tb.ptiles;
        P.T += (int64_t)tb.m_blk * tb.nq;
    }
    const bool whole = nblk == 1 && P.blocks[0].p0 == 0 && P.blocks[0].q0 == 0 && P.blocks[0].m_blk == M_total &&
                       P.blocks[0].nq == N;
    const bool tiles_ok = knobs.ordered_tiles != 0 && (W == 1 || W == 2 || W == 4 || W == 8 || W == 16) &&
                          segs * TILE_ROWS <= 4 * P.T + 4096 && segs < (int64_t)1 << 31;
    if (whole && P.T <= knobs.by_t_limit) P.path = Path::BY_T;
    else if (!tiles_ok) P.path = Path::SORTED;
    else if (knobs.class_dedup != 0 && class_job_plan(M_total, P.blocks, nblk, P.T, P.fmt.tb, g_key_mask,
                                                      knobs.class_variant, P.job))
        P.path = Path::TILES_CLASS;
    else P.path = Path::TILES_SORT;
    P.n_seg = P.tiles() ? (uint32_t)segs : 0u;

    Arena ar(ws, ws ? ws_bytes : 0);
    const size_t m = (size_t)(M_total > 0 ? M_total : 1), n = (size_t)(N > 0 ? N : 1), t = (size_t)(P.T > 0 ? P.T : 1);
    size_t need = arena_need(m, 8) + arena_need(n, 8) + arena_need(m, 4) + arena_need(n, 4) + arena_need(t, 8);
    P.a_sk = ar.take<uint64_t>(m);
    P.b_sk = ar.take<uint64_t>(n);
    P.a_y = ar.take<int32_t>(m);
    P.b_y = ar.take<int32_t>(n);
    P.recs = ar.take<uint64_t>(t);
    P.d_blocks = nullptr;
    P.drop = nullptr;
    P.segoff = nullptr;
    P.class_ws = nullptr;
    P.class_ws_bytes = 0;
    if (P.tiles()) {
        const size_t sg = (size_t)P.n_seg;
        need += arena_need(256, sizeof(TileBlock)) + arena_need(4 * sg, 4) + arena_need(sg + 1, 4);
        P.d_blocks = ar.take<TileBlock>(256);
        P.drop = ar.take<uint32_t>(4 * sg);
        P.segoff = ar.take<uint32_t>(sg + 1);
    }
    if (P.path == Path::TILES_CLASS) {
        P.class_ws_bytes = class_job_ws_bytes(P.job);
        need += arena_need(P.class_ws_bytes, 1);
        P.class_ws = ar.take<unsigned char>(P.class_ws_bytes);
    }
    P.rest = ws ? (void *)(ar.base + ar.off) : nullptr;
    P.rest_bytes = (ws && ws_bytes > ar.off) ? ws_bytes - ar.off : 0;
    P.need = need + dedup_ws_bytes(P.T) + 1024;
    return SYM_OK;
}

static TileMap tile_map_of(const MulBlocksPlan &P, int64_t M_total) {
    TileMap tm;
    tm.first = P.blocks[0];
    tm.blocks = P.d_blocks;
    tm.nblk = P.nblk;
    tm.M = (uint32_t)M_total;
    tm.Minv = fastdiv_magic((uint32_t)M_total);
    tm.n_seg = P.n_seg;
    tm.drop = P.drop;
    tm.segoff = P.segoff;
    return tm;
}

static int check_ws(const MulBlocksPlan &P, const void *ws, size_t ws_bytes) {
    if (ws == nullptr || ws_bytes < P.need) {
        set_error("workspace too small: need %zu bytes, got %zu", P.need, ws_bytes);
        return SYM_E_WORKSPACE;
    }
    return SYM_OK;
}

extern "C" size_t sym_mul_blocks_ws_bytes(int64_t M_total, int64_t N, int32_t W, const int64_t *blocks_host, int32_t nblk) {
    MulBlocksPlan P;
    if (mul_blocks_plan(M_total, N, W, blocks_host, nblk, nullptr, 0, P) != SYM_OK) return 0;
    return P.need;
}

extern "C" int sym_mul_blocks_count(const uint64_t *a_xz, const double *a_c, int64_t M_total, const uint64_t *b_xz,
                                    const double *b_c, int64_t N, int32_t W, const int64_t *blocks_host, int32_t nblk,
                                    double zero_threshold, int64_t *n_out, int64_t *n_out_host, void *ws, size_t ws_bytes,
                                    void *stream) {
    return sym_mul_blocks_count_tables(a_xz, a_c, nullptr, nullptr, M_total, b_xz, b_c, N, W, blocks_host, nblk,
                                       zero_threshold, n_out, n_out_host, nullptr, ws, ws_bytes, stream);
}

extern "C" int sym_mul_blocks_count_tables(const uint64_t *a_xz, const double *a_c, const uint64_t *a_sketch,
                                           const int32_t *a_ycount, int64_t M_total, const uint64_t *b_xz, const double *b_c,
                                           int64_t N, int32_t W, const int64_t *blocks_host, int32_t nblk,
                                           double zero_threshold, int64_t *n_out, int64_t *n_out_host, int32_t *speculate,
                                           void *ws, size_t ws_bytes, void *stream) {
    SYM_REQUIRE((a_sketch == nullptr) == (a_ycount == nullptr), "a_sketch and a_ycount come together");
    SYM_REQUIRE(speculate == nullptr || n_out == nullptr, "a speculating count leaves no device count");
    if (speculate) *speculate = 0;
    MulBlocksPlan P;
    SYM_TRY(mul_blocks_plan(M_total, N, W, blocks_host, nblk, ws, ws_bytes, P));
    cudaStream_t st = (cudaStream_t)stream;
    if (P.T == 0) {
        if (n_out) SYM_CUDA_OK(cudaMemsetAsync(n_out, 0, sizeof(int64_t), st));
        if (n_out_host) *n_out_host = 0;
        return SYM_OK;
    }
    SYM_TRY(check_ws(P, ws, ws_bytes));
    if (a_sketch) {   // the caller already has A's tables (sym_rotate_split): two reads of A saved
        SYM_CUDA_OK(cudaMemcpyAsync(P.a_sk, a_sketch, sizeof(uint64_t) * (size_t)M_total, cudaMemcpyDeviceToDevice, st));
        SYM_CUDA_OK(cudaMemcpyAsync(P.a_y, a_ycount, sizeof(int32_t) * (size_t)M_total, cudaMemcpyDeviceToDevice, st));
        SYM_TRY(sym_sketch_rows(b_xz, N, W, P.b_sk, st));
        SYM_TRY(sym_ycount(b_xz, N, W, P.b_y, st));
    } else {
        SYM_TRY(operand_tables(a_xz, M_total, b_xz, N, W, P.a_sk, P.a_y, P.b_sk, P.b_y, st));
    }
    if (P.tiles()) {
        if (P.nblk > 1)   // block 0 travels inside the TileMap kernel argument
            SYM_CUDA_OK(cudaMemcpyAsync(P.d_blocks, P.blocks, sizeof(TileBlock) * (size_t)P.nblk, cudaMemcpyHostToDevice, st));
        SYM_CUDA_OK(cudaMemsetAsync(P.drop, 0, sizeof(uint32_t) * 4 * (size_t)P.n_seg, st));
    }
    const RecFmt fmt = P.fmt;
    size_t off = 0;
    for (int b = 0; b < P.nblk && P.path != Path::TILES_CLASS; ++b) {
        const TileBlock &tb = P.blocks[b];
        if (P.path == Path::TILES_SORT) {
            // a separate kernel writes the records before the sort: generating them inside the first radix pass
            // measured slower on B200 (10.06 vs 9.65 ms per 1.25e8 cross terms: a key costs two 64-bit multiplies
            // and is generated twice, in the histogram and in pass 0, against 0.15 ms for writing 1 GB once)
            if (tb.m_blk > 0 && tb.nq > 0) {
                dim3 grid((tb.m_blk + 255) / 256, (tb.nq + KEYS_QCH - 1) / KEYS_QCH);
                if (grid.y > 65535) {
                    set_error("too many B rows for one launch (N=%u)", tb.nq);
                    return SYM_E_UNSUPPORTED;
                }
                pair_keys_kernel<<<grid, 256, 0, st>>>(P.a_sk, (uint32_t)M_total, tb.p0, tb.m_blk, P.b_sk + tb.q0, tb.nq, tb.q0,
                                                       g_key_mask, fmt, P.recs + off);
                SYM_LAUNCH_OK();
            }
        } else {
            SYM_TRY(launch_pair_records(a_xz, P.a_sk, P.a_y, M_total, tb.p0, (int64_t)tb.p0 + tb.m_blk,
                                        b_xz + (size_t)tb.q0 * 2 * W, P.b_sk + tb.q0, P.b_y + tb.q0, tb.nq, W, fmt,
                                        P.recs + off, st, tb.q0));
        }
        off += (size_t)tb.m_blk * tb.nq;
    }
    ProductRows rows{a_xz, b_xz, a_c, b_c, (uint32_t)M_total, 2 * W, (uint32_t)N};
    rows.Minv = fastdiv_magic((uint32_t)M_total);
    switch (P.path) {
        case Path::BY_T:
        case Path::SORTED:
            return dedup_product_plan(P.path, P.recs, P.T, fmt, rows, zero_threshold, n_out, n_out_host, P.rest, P.rest_bytes, st);
        case Path::TILES_SORT:
            return dedup_product_plan_tiles(P.recs, P.T, fmt, rows, tile_map_of(P, M_total), zero_threshold, n_out, n_out_host,
                                            P.rest, P.rest_bytes, st);
        case Path::TILES_CLASS: {
            bool spec = false;
            SYM_TRY(dedup_product_plan_classes(P.recs, P.T, fmt, rows, tile_map_of(P, M_total), P.job, P.a_sk, P.b_sk, P.a_y,
                                               P.b_y, P.class_ws, P.class_ws_bytes, zero_threshold, n_out, n_out_host,
                                               speculate ? &spec : nullptr, P.rest, P.rest_bytes, st));
            if (speculate) *speculate = spec ? 1 : 0;
            return SYM_OK;
        }
    }
    return SYM_E_INVALID;
}

extern "C" int sym_mul_blocks_emit(const uint64_t *a_xz, const double *a_c, int64_t M_total, const uint64_t *b_xz,
                                   const double *b_c, int64_t N, int32_t W, const int64_t *blocks_host, int32_t nblk,
                                   int64_t U, uint64_t *out_xz, double *out_c, void *ws, size_t ws_bytes, void *stream) {
    MulBlocksPlan P;
    SYM_TRY(mul_blocks_plan(M_total, N, W, blocks_host, nblk, ws, ws_bytes, P));
    if (P.T == 0 || U == 0) return SYM_OK;
    SYM_REQUIRE(U >= 0 && U <= P.T, "bad survivor count");
    SYM_TRY(check_ws(P, ws, ws_bytes));
    ProductRows rows{a_xz, b_xz, a_c, b_c, (uint32_t)M_total, 2 * W, (uint32_t)N};
    rows.Minv = fastdiv_magic((uint32_t)M_total);
    cudaStream_t st = (cudaStream_t)stream;
    switch (P.path) {
        case Path::BY_T:
        case Path::SORTED:
            return dedup_product_emit(P.path, P.recs, P.T, P.fmt, rows, U, out_xz, out_c, P.rest, P.rest_bytes, st);
        case Path::TILES_SORT:
        case Path::TILES_CLASS:
            return dedup_product_emit_tiles(P.path, P.recs, P.T, P.fmt, rows, tile_map_of(P, M_total), P.blocks, P.a_y, P.b_y, U,
                                            out_xz, out_c, P.rest, P.rest_bytes, st);
    }
    return SYM_E_INVALID;
}

extern "C" int sym_mul_blocks_emit_spec(const uint64_t *a_xz, const double *a_c, int64_t M_total, const uint64_t *b_xz,
                                        const double *b_c, int64_t N, int32_t W, const int64_t *blocks_host, int32_t nblk,
                                        double zero_threshold, uint64_t *out_xz, double *out_c, int64_t *n_out_host, void *ws,
                                        size_t ws_bytes, void *stream) {
    MulBlocksPlan P;
    SYM_TRY(mul_blocks_plan(M_total, N, W, blocks_host, nblk, ws, ws_bytes, P));
    SYM_REQUIRE(P.path == Path::TILES_CLASS && P.T > 0, "this product takes no speculative emission");
    SYM_TRY(check_ws(P, ws, ws_bytes));
    ProductRows rows{a_xz, b_xz, a_c, b_c, (uint32_t)M_total, 2 * W, (uint32_t)N};
    rows.Minv = fastdiv_magic((uint32_t)M_total);
    return dedup_product_spec_classes(P.recs, P.T, P.fmt, rows, tile_map_of(P, M_total), P.blocks, P.job, P.b_sk, P.a_y, P.b_y,
                                      P.class_ws, P.class_ws_bytes, zero_threshold, out_xz, out_c, n_out_host, P.rest,
                                      P.rest_bytes, (cudaStream_t)stream);
}

// The whole product = one block. Sized for every path a tuning-knob change can select for the shape (BY_T needs what
// SORTED needs, the class tables grow with the class count of knob 11's shape), so that a knob change between calls
// never invalidates a workspace.
extern "C" size_t sym_mul_cleanup_ws_bytes(int64_t M, int64_t N, int32_t W) {
    const int64_t blk[4] = {0, M, 0, N};
    size_t need = 0;
    for (int tiles = 0; tiles <= 1; ++tiles) {
        for (int variant = -1; variant <= 3; ++variant) {   // -1: knob 10 = 0
            const PathKnobs knobs{-1, tiles, variant >= 0, variant >= 0 ? variant : 0};
            MulBlocksPlan P;
            if (mul_blocks_plan(M, N, W, blk, 1, nullptr, 0, P, knobs) == SYM_OK && P.need > need) need = P.need;
        }
    }
    return need;
}

extern "C" int sym_mul_cleanup_count(const uint64_t *a_xz, const double *a_c, int64_t M, const uint64_t *b_xz,
                                     const double *b_c, int64_t N, int32_t W, double zero_threshold, int64_t *n_out,
                                     int64_t *n_out_host, void *ws, size_t ws_bytes, void *stream) {
    const int64_t blk[4] = {0, M, 0, N};
    return sym_mul_blocks_count(a_xz, a_c, M, b_xz, b_c, N, W, blk, 1, zero_threshold, n_out, n_out_host, ws, ws_bytes, stream);
}

extern "C" int sym_mul_cleanup_emit(const uint64_t *a_xz, const double *a_c, int64_t M, const uint64_t *b_xz,
                                    const double *b_c, int64_t N, int32_t W, int64_t U, uint64_t *out_xz, double *out_c,
                                    void *ws, size_t ws_bytes, void *stream) {
    const int64_t blk[4] = {0, M, 0, N};
    return sym_mul_blocks_emit(a_xz, a_c, M, b_xz, b_c, N, W, blk, 1, U, out_xz, out_c, ws, ws_bytes, stream);
}

extern "C" int sym_mul_cleanup(const uint64_t *a_xz, const double *a_c, int64_t M, const uint64_t *b_xz, const double *b_c,
                               int64_t N, int32_t W, double zero_threshold, uint64_t *out_xz, double *out_c,
                               int64_t out_capacity, int64_t *n_out, int64_t *n_out_host, void *ws, size_t ws_bytes,
                               void *stream) {
    int64_t U = 0;
    SYM_TRY(sym_mul_cleanup_count(a_xz, a_c, M, b_xz, b_c, N, W, zero_threshold, n_out, &U, ws, ws_bytes, stream));
    if (n_out_host) *n_out_host = U;
    if (U > out_capacity) {
        set_error("output capacity %lld < %lld surviving terms", (long long)out_capacity, (long long)U);
        return SYM_E_CAPACITY;
    }
    return sym_mul_cleanup_emit(a_xz, a_c, M, b_xz, b_c, N, W, U, out_xz, out_c, ws, ws_bytes, stream);
}
