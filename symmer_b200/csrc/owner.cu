// Exchange-free hash partition of a sharded product (SURVEY.md §8e, multiply + cleanup).
//
// The owner of a row is a GF(2)-LINEAR function of its sketch: owner bit k = parity(sketch & R_k).
// Linearity gives owner(A[p] ^ B[q]) = owner(A[p]) ^ owner(B[q]), so with both operands grouped by
// owner class, rank r generates exactly the cross terms it owns — the blocks A_a x B_{a^r} — and
// equal rows (wherever they come from) meet on one rank without any record or row crossing NVLink.
// Kernels here: class of every row + stable grouping of an operator by class (rows, coefficients,
// permutation, class sizes). Byte/integer work, HBM/L2-bound and tiny next to the product itself.
#include "rows.cuh"
#include "sort.cuh"

namespace symb {

// fixed odd-looking 64-bit masks; any set of linearly independent functionals would do
__constant__ uint64_t OWNER_MASKS[8] = {0x9e3779b97f4a7c15ULL, 0xc2b2ae3d27d4eb4fULL, 0x165667b19e3779f9ULL,
                                        0xd6e8feb86659fd93ULL, 0xa0761d6478bd642fULL, 0xe7037ed1a0b428dbULL,
                                        0x8ebc6af09c88c6e3ULL, 0x589965cc75374cc3ULL};

__device__ __forceinline__ uint32_t owner_of_sketch(uint64_t sk, int lg) {
    uint32_t cls = 0;
    for (int k = 0; k < lg; ++k) cls |= (uint32_t)(__popcll(sk & OWNER_MASKS[k]) & 1) << k;
    return cls;
}

// keys[row] = class << (64 - lg) (radix_partition splits on the top lg bits), vals[row] = row
__global__ void __launch_bounds__(256) owner_keys_kernel(const uint64_t *__restrict__ sk, int64_t M, int lg,
                                                          uint64_t *__restrict__ keys, uint32_t *__restrict__ vals,
                                                          uint8_t *__restrict__ cls_out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const uint32_t cls = owner_of_sketch(sk[i], lg);
    if (keys) keys[i] = lg > 0 ? ((uint64_t)cls << (64 - lg)) : 0ull;
    if (vals) vals[i] = (uint32_t)i;
    if (cls_out) cls_out[i] = (uint8_t)cls;
}

// out row i = in row perm[i]; thread = (row, 16-byte chunk); the coefficient rides on chunk 0
__global__ void __launch_bounds__(256) gather_rows_kernel(const uint4 *__restrict__ xz, const double2 *__restrict__ c,
                                                           const uint32_t *__restrict__ perm, int64_t M, int chunks,
                                                           uint4 *__restrict__ out_xz, double2 *__restrict__ out_c,
                                                           int32_t *__restrict__ perm_out) {
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= M * chunks) return;
    const int64_t i = g / chunks;
    const int k = (int)(g - i * chunks);
    const uint32_t src = perm[i];
    out_xz[g] = xz[(size_t)src * chunks + k];
    if (k == 0) {
        if (c && out_c) out_c[i] = c[src];
        if (perm_out) perm_out[i] = (int32_t)src;
    }
}

}  // namespace symb

using namespace symb;

extern "C" int sym_owner_classes(const uint64_t *xz, int64_t M, int32_t W, int32_t log2_parts, uint8_t *cls, void *ws,
                                 size_t ws_bytes, void *stream) {
    SYM_REQUIRE(M >= 0 && W >= 1, "bad size");
    SYM_REQUIRE(log2_parts >= 0 && log2_parts <= 8, "log2_parts must be in [0,8]");
    if (M == 0) return SYM_OK;
    if (ws_bytes < arena_need((size_t)M, 8)) {
        set_error("workspace too small");
        return SYM_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    uint64_t *sk = static_cast<uint64_t *>(ws);
    SYM_TRY(sym_sketch_rows(xz, M, W, sk, st));
    owner_keys_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(sk, M, log2_parts, nullptr, nullptr, cls);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

extern "C" int sym_gather_rows(const uint64_t *xz, const double *c, const uint32_t *perm, int64_t M_out, int32_t W, uint64_t *out_xz,
                               double *out_c, void *stream) {
    SYM_REQUIRE(M_out >= 0 && M_out < ((int64_t)1 << 31) && W >= 1, "bad size");
    if (M_out == 0) return SYM_OK;
    const int chunks = W;
    gather_rows_kernel<<<(unsigned)((M_out * chunks + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint4 *>(xz), reinterpret_cast<const double2 *>(c), perm, M_out, chunks,
        reinterpret_cast<uint4 *>(out_xz), reinterpret_cast<double2 *>(out_c), nullptr);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

extern "C" size_t sym_class_partition_ws_bytes(int64_t M) {
    if (M < 1) M = 1;
    return arena_need((size_t)M, 8) * 3 + arena_need((size_t)M, 4) * 2 + arena_need(record_hist_elems(M), 4) + 2048;
}

extern "C" int sym_class_partition(const uint64_t *xz, const double *c, int64_t M, int32_t W, int32_t log2_parts,
                                   uint64_t *out_xz, double *out_c, int32_t *perm, int64_t *counts, void *ws,
                                   size_t ws_bytes, void *stream) {
    SYM_REQUIRE(M >= 0 && M < ((int64_t)1 << 31) && W >= 1, "bad size");
    SYM_REQUIRE(log2_parts >= 0 && log2_parts <= 8, "log2_parts must be in [0,8]");
    cudaStream_t st = (cudaStream_t)stream;
    const int parts = 1 << log2_parts;
    if (M == 0) {
        SYM_CUDA_OK(cudaMemsetAsync(counts, 0, sizeof(int64_t) * parts, st));
        return SYM_OK;
    }
    if (ws_bytes < sym_class_partition_ws_bytes(M)) {
        set_error("workspace too small");
        return SYM_E_WORKSPACE;
    }
    Arena ar(ws, ws_bytes);
    uint64_t *sk = ar.take<uint64_t>((size_t)M);
    uint64_t *keys = ar.take<uint64_t>((size_t)M);
    uint64_t *keys2 = ar.take<uint64_t>((size_t)M);
    uint32_t *vals = ar.take<uint32_t>((size_t)M);
    uint32_t *vals2 = ar.take<uint32_t>((size_t)M);
    uint32_t *hist = ar.take<uint32_t>(record_hist_elems(M));
    if (!hist) {
        set_error("workspace arena exhausted");
        return SYM_E_WORKSPACE;
    }
    SYM_TRY(sym_sketch_rows(xz, M, W, sk, st));
    owner_keys_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(sk, M, log2_parts, keys, vals, nullptr);
    SYM_LAUNCH_OK();
    const uint32_t *order = vals;
    if (log2_parts > 0) {
        SYM_TRY(radix_partition(keys, vals, keys2, vals2, M, log2_parts, counts, hist, st));
        order = vals2;
    } else {
        int64_t m = M;
        SYM_CUDA_OK(cudaMemcpyAsync(counts, &m, sizeof(int64_t), cudaMemcpyHostToDevice, st));
        SYM_CUDA_OK(cudaStreamSynchronize(st));
    }
    const int chunks = W;  // 2W words = W 16-byte chunks
    gather_rows_kernel<<<(unsigned)((M * chunks + 255) / 256), 256, 0, st>>>(
        reinterpret_cast<const uint4 *>(xz), reinterpret_cast<const double2 *>(c), order, M, chunks,
        reinterpret_cast<uint4 *>(out_xz), reinterpret_cast<double2 *>(out_c), perm);
    SYM_LAUNCH_OK();
    return SYM_OK;
}
