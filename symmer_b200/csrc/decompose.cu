// Pauli decomposition of a matrix: the inverse of to_sparse_matrix (symmer/operators/base.py:1458-1510) and the
// engine behind PauliwordOp.from_matrix (base.py:238-425; the reference loops over matrix entries building
// |i><j| projectors, O(nnz * 2^n) in Python, or over all 4^n basis operators).
//
// With basis index r (qubit 0 = most significant bit) and c' = c * (-i)^{popc(x&z)}:
//     M[r, r^x] = sum_z c'_{x,z} (-1)^{popc(r&z)}    =>    c'_{x,z} = 2^-n sum_r (-1)^{popc(r&z)} M[r, r^x]
// i.e. ONE Walsh-Hadamard transform of every XOR-diagonal d_x[r] = M[r, r^x]. The low WHT_SMEM_BITS stages of a
// diagonal run in shared memory (one CTA per 4096-entry tile), the remaining stages are in-place butterflies in
// global memory (coalesced runs of >= 4096 entries). HBM-bound: 32 B per matrix entry per pass.
#include "common.cuh"

namespace symb {

constexpr int WHT_SMEM_BITS = 12;     // 4096 complex128 = 64 KB of shared memory per CTA
constexpr int WHT_THREADS = 256;

// One CTA = one tile of 2^L consecutive r of diagonal k. FROM_DENSE: gather the diagonal from the row-major matrix
// (x = k); otherwise transform diag[k][.] in place. The 2^-n scale is folded into the store.
template <bool FROM_DENSE>
__global__ void __launch_bounds__(WHT_THREADS) wht_tile_kernel(const double2 *src, double2 *dst,
                                                                int n, int L, double scale) {
    extern __shared__ double2 tile[];
    const int64_t side = (int64_t)1 << n;
    const int64_t tiles_per_diag = side >> L;
    const int64_t k = blockIdx.x / tiles_per_diag;
    const int64_t r0 = (blockIdx.x - k * tiles_per_diag) << L;
    const int len = 1 << L;
    for (int i = threadIdx.x; i < len; i += WHT_THREADS) {
        const int64_t r = r0 + i;
        tile[i] = FROM_DENSE ? src[r * side + (r ^ k)] : src[k * side + r];
    }
    __syncthreads();
    for (int s = 0; s < L; ++s) {
        const int h = 1 << s;
        for (int p = threadIdx.x; p < (len >> 1); p += WHT_THREADS) {
            const int lo = p & (h - 1);
            const int i0 = ((p >> s) << (s + 1)) | lo, i1 = i0 | h;
            const double2 a = tile[i0], b = tile[i1];
            tile[i0] = make_double2(a.x + b.x, a.y + b.y);
            tile[i1] = make_double2(a.x - b.x, a.y - b.y);
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < len; i += WHT_THREADS) {
        const double2 v = tile[i];
        dst[k * side + r0 + i] = make_double2(v.x * scale, v.y * scale);
    }
}

// Butterfly stage `bit` (>= WHT_SMEM_BITS) of every diagonal, in place. thread = one pair (r, r | 1 << bit).
__global__ void __launch_bounds__(256) wht_stage_kernel(double2 *__restrict__ d, int64_t pairs_total, int n, int bit) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= pairs_total) return;
    const int64_t half = (int64_t)1 << (n - 1);
    const int64_t k = t / half, p = t - k * half;
    const int64_t lo = p & (((int64_t)1 << bit) - 1);
    const int64_t i0 = (k << n) + (((p >> bit) << (bit + 1)) | lo), i1 = i0 + ((int64_t)1 << bit);
    const double2 a = d[i0], b = d[i1];
    d[i0] = make_double2(a.x + b.x, a.y + b.y);
    d[i1] = make_double2(a.x - b.x, a.y - b.y);
}

// Inverse of term_masks_kernel (layout.cu): basis-index masks (qubit 0 = most significant bit) and phased
// coefficients c' -> packed single-word rows and c = c' * i^{popc(x&z)}.
__global__ void __launch_bounds__(256) rows_from_masks_kernel(const int64_t *__restrict__ xm, const int64_t *__restrict__ zm,
                                                               const double2 *__restrict__ cp, int64_t M, int n,
                                                               uint64_t *__restrict__ xz, double2 *__restrict__ c) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= M) return;
    const uint64_t x = __brevll((uint64_t)xm[t] << (64 - n)), z = __brevll((uint64_t)zm[t] << (64 - n));
    xz[2 * t] = x;
    xz[2 * t + 1] = z;
    const double2 v = cp[t];
    double2 o;
    switch (__popcll(x & z) & 3) {
        case 0: o = v; break;
        case 1: o = make_double2(-v.y, v.x); break;       // * i
        case 2: o = make_double2(-v.x, -v.y); break;      // * -1
        default: o = make_double2(v.y, -v.x); break;      // * -i
    }
    c[t] = o;
}

template <bool FROM_DENSE>
static int wht_run(const double2 *src, double2 *dst, int64_t K, int n, cudaStream_t st) {
    const int L = n < WHT_SMEM_BITS ? n : WHT_SMEM_BITS;
    const size_t smem = sizeof(double2) << L;
    static bool attr_done[64] = {};   // per device (one array per instantiation)
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !attr_done[dev]) {
        SYM_CUDA_OK(cudaFuncSetAttribute(wht_tile_kernel<FROM_DENSE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)(sizeof(double2) << WHT_SMEM_BITS)));
        attr_done[dev] = true;
    }
    const int64_t side = (int64_t)1 << n;
    const int64_t ctas = K * (side >> L);
    SYM_REQUIRE(ctas < ((int64_t)1 << 31), "too many tiles for one launch");
    wht_tile_kernel<FROM_DENSE><<<(unsigned)ctas, WHT_THREADS, smem, st>>>(src, dst, n, L, 1.0 / (double)side);
    SYM_LAUNCH_OK();
    const int64_t pairs = K * (side >> 1);
    for (int bit = L; bit < n; ++bit) {
        wht_stage_kernel<<<(unsigned)((pairs + 255) / 256), 256, 0, st>>>(dst, pairs, n, bit);
        SYM_LAUNCH_OK();
    }
    return SYM_OK;
}

}  // namespace symb

using namespace symb;

extern "C" int sym_pauli_decompose_dense(const double *matrix, int32_t n_qubits, double *out, void *stream) {
    SYM_REQUIRE(n_qubits >= 0 && n_qubits <= 15, "dense decomposition needs n_qubits <= 15");
    SYM_REQUIRE(matrix != out, "the dense decomposition is not in place");
    return wht_run<true>(reinterpret_cast<const double2 *>(matrix), reinterpret_cast<double2 *>(out),
                         (int64_t)1 << n_qubits, n_qubits, (cudaStream_t)stream);
}

extern "C" int sym_pauli_decompose_diagonals(double *diag, int64_t K, int32_t n_qubits, void *stream) {
    SYM_REQUIRE(K >= 0 && n_qubits >= 0 && n_qubits <= 40, "bad size");
    if (K == 0) return SYM_OK;
    SYM_REQUIRE(K <= (((int64_t)1 << 38) >> n_qubits), "diagonal table too large");
    return wht_run<false>(reinterpret_cast<const double2 *>(diag), reinterpret_cast<double2 *>(diag), K, n_qubits,
                          (cudaStream_t)stream);
}

extern "C" int sym_rows_from_masks(const int64_t *x_masks, const int64_t *z_masks, const double *c_phased, int64_t M,
                                   int32_t n_qubits, uint64_t *xz, double *c, void *stream) {
    SYM_REQUIRE(M >= 0 && n_qubits >= 1 && n_qubits <= 62, "rows from masks need 1 <= n_qubits <= 62");
    if (M == 0) return SYM_OK;
    rows_from_masks_kernel<<<(unsigned)((M + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        x_masks, z_masks, reinterpret_cast<const double2 *>(c_phased), M, n_qubits, xz, reinterpret_cast<double2 *>(c));
    SYM_LAUNCH_OK();
    return SYM_OK;
}
