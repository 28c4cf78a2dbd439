// _rref_binary (symmer/operators/utils.py:292-315) on bit-packed rows: GF(2) row reduction with the
// reference's row-driven pivot rule — for each row i in order, the pivot is the first set column of
// the CURRENT row i, and row i is XORed into every other row with a 1 in that column; rows are
// never swapped. Results are bit-exact with the reference.
//
// Small matrices (the symmetry-generator search: 2n rows x (M+2n) columns) run in ONE CTA with the
// whole matrix in shared memory, one warp-parallel step per pivot row. Large matrices run one
// pivot step per pair of launches over the whole GPU (HBM-bound XOR sweep).
#include "common.cuh"

namespace symb {

constexpr int RREF_THREADS = 1024;

__device__ __forceinline__ int first_set_column(const uint64_t *row, int64_t Cw, int tid, int nthreads, int *s_min) {
    // block-wide: smallest set bit index of `row` (or INT_MAX). s_min must be initialised to INT_MAX.
    int best = 0x7fffffff;
    for (int64_t k = tid; k < Cw; k += nthreads) {
        uint64_t w = row[k];
        if (w) {
            int col = (int)(k * 64 + (__ffsll((long long)w) - 1));
            best = min(best, col);
            break;  // columns grow with k for this thread
        }
    }
    if (best != 0x7fffffff) atomicMin(s_min, best);
    return 0;
}

__global__ void __launch_bounds__(RREF_THREADS) rref_smem_kernel(uint64_t *__restrict__ bits, int R, int64_t Cw,
                                                                  int32_t *__restrict__ pivots) {
    extern __shared__ uint64_t sm[];  // R*Cw words
    __shared__ int s_piv;
    const int tid = threadIdx.x, nt = blockDim.x;
    const int64_t total = (int64_t)R * Cw;
    for (int64_t i = tid; i < total; i += nt) sm[i] = bits[i];
    __syncthreads();
    for (int i = 0; i < R; ++i) {
        if (tid == 0) s_piv = 0x7fffffff;
        __syncthreads();
        first_set_column(sm + (int64_t)i * Cw, Cw, tid, nt, &s_piv);
        __syncthreads();
        const int piv = s_piv;
        if (piv != 0x7fffffff) {
            const int64_t pw = piv >> 6;
            const uint64_t pm = 1ull << (piv & 63);
            // each thread owns whole (row, word) cells; the pivot-column test reads word pw of row r,
            // which is itself updated in this step, so handle it last: first all other words.
            for (int64_t c = tid; c < total; c += nt) {
                const int r = (int)(c / Cw);
                const int64_t k = c - (int64_t)r * Cw;
                if (r == i || k == pw) continue;
                if (sm[(int64_t)r * Cw + pw] & pm) sm[c] ^= sm[(int64_t)i * Cw + k];
            }
            __syncthreads();
            for (int r = tid; r < R; r += nt) {
                if (r == i) continue;
                uint64_t w = sm[(int64_t)r * Cw + pw];
                if (w & pm) sm[(int64_t)r * Cw + pw] = w ^ sm[(int64_t)i * Cw + pw];
            }
        }
        __syncthreads();
    }
    for (int64_t i = tid; i < total; i += nt) bits[i] = sm[i];
    // final pivot column of every row
    for (int r = tid; r < R; r += nt) {
        int p = -1;
        for (int64_t k = 0; k < Cw; ++k) {
            uint64_t w = sm[(int64_t)r * Cw + k];
            if (w) {
                p = (int)(k * 64 + (__ffsll((long long)w) - 1));
                break;
            }
        }
        pivots[r] = p;
    }
}

// ---- large path: one pivot step = (pivot + hit flags) kernel, then a grid-wide XOR sweep
__global__ void __launch_bounds__(RREF_THREADS) rref_pivot_kernel(const uint64_t *__restrict__ bits, int64_t R, int64_t Cw,
                                                                   int64_t i, int *__restrict__ piv_out) {
    __shared__ int s_piv;
    if (threadIdx.x == 0) s_piv = 0x7fffffff;
    __syncthreads();
    first_set_column(bits + i * Cw, Cw, threadIdx.x, blockDim.x, &s_piv);
    __syncthreads();
    if (threadIdx.x == 0) *piv_out = s_piv;
}

__global__ void __launch_bounds__(256) rref_hit_kernel(const uint64_t *__restrict__ bits, int64_t R, int64_t Cw, int64_t i,
                                                        const int *__restrict__ piv_in, uint8_t *__restrict__ hit) {
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const int piv = *piv_in;
    uint8_t h = 0;
    if (piv != 0x7fffffff && r != i) h = (bits[r * Cw + (piv >> 6)] >> (piv & 63)) & 1ull;
    hit[r] = h;
}

__global__ void __launch_bounds__(256) rref_xor_kernel(uint64_t *__restrict__ bits, int64_t R, int64_t Cw, int64_t i,
                                                        const uint8_t *__restrict__ hit) {
    int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= R * Cw) return;
    int64_t r = c / Cw, k = c - r * Cw;
    if (hit[r]) bits[c] ^= bits[i * Cw + k];
}

// ---- blocked large path (method-of-four-Russians style panels, bit-exact with the row-driven rule)
// A panel is kk consecutive rows. (1) panel kernel: the kk rows are reduced among themselves in
// shared memory with the sequential rule (pivot = first set column of the current row, XOR into the
// other panel rows with a 1 there); afterwards panel row j has a 1 in its pivot column p_j and the
// other panel rows a 0. (2) mask kernel: for every row r outside the panel, m(r) = its bits at the
// panel's pivot columns, read BEFORE any update. (3) sweep: r ^= XOR of the panel rows selected by
// m(r). This equals the result of the kk sequential steps: the sequential result for r is the unique
// element of r + span(panel) with zeros in every panel pivot column, and the panel rows are a basis
// of that span that is the identity on those columns. One sweep of the matrix per kk pivots instead
// of one per pivot: kk x less HBM/L2 traffic and 3 launches per panel instead of 3 per row.
constexpr int PANEL_MAX = 16;
constexpr int SWEEP_WORDS = 128;   // column strip of a sweep CTA (1 KB per row)
constexpr int SWEEP_ROWS = 32;     // rows per sweep CTA

__global__ void __launch_bounds__(RREF_THREADS) rref_panel_kernel(uint64_t *__restrict__ bits, int64_t Cw, int64_t i0, int kk,
                                                                   int *__restrict__ piv_out) {
    extern __shared__ uint64_t sm[];  // kk*Cw words
    __shared__ int s_piv;
    __shared__ uint8_t s_hit[PANEL_MAX];
    const int tid = threadIdx.x, nt = blockDim.x;
    const int64_t total = (int64_t)kk * Cw;
    uint64_t *g = bits + i0 * Cw;
    for (int64_t c = tid; c < total; c += nt) sm[c] = g[c];
    __syncthreads();
    for (int j = 0; j < kk; ++j) {
        if (tid == 0) s_piv = 0x7fffffff;
        __syncthreads();
        first_set_column(sm + (int64_t)j * Cw, Cw, tid, nt, &s_piv);
        __syncthreads();
        const int piv = s_piv;
        if (tid == 0) piv_out[j] = piv;
        if (piv != 0x7fffffff) {
            if (tid < kk) s_hit[tid] = (tid != j) && ((sm[(int64_t)tid * Cw + (piv >> 6)] >> (piv & 63)) & 1ull);
            __syncthreads();
            const uint64_t *src = sm + (int64_t)j * Cw;
            for (int r = 0; r < kk; ++r) {          // uniform over the CTA: no per-cell division
                if (!s_hit[r]) continue;
                uint64_t *dst = sm + (int64_t)r * Cw;
                for (int64_t k = tid; k < Cw; k += nt) dst[k] ^= src[k];
            }
        }
        __syncthreads();
    }
    for (int64_t c = tid; c < total; c += nt) g[c] = sm[c];
}

__global__ void __launch_bounds__(256) rref_mask_kernel(const uint64_t *__restrict__ bits, int64_t R, int64_t Cw, int64_t i0,
                                                         int kk, const int *__restrict__ piv, uint32_t *__restrict__ mask) {
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    uint32_t m = 0;
    if (r < i0 || r >= i0 + kk) {
        for (int j = 0; j < kk; ++j) {
            const int p = piv[j];
            if (p != 0x7fffffff) m |= (uint32_t)((bits[r * Cw + (p >> 6)] >> (p & 63)) & 1ull) << j;
        }
    }
    mask[r] = m;
}

__global__ void __launch_bounds__(256) rref_sweep_kernel(uint64_t *__restrict__ bits, int64_t R, int64_t Cw, int64_t i0, int kk,
                                                          const uint32_t *__restrict__ mask) {
    __shared__ uint64_t sB[PANEL_MAX][SWEEP_WORDS];
    const int64_t k0 = (int64_t)blockIdx.x * SWEEP_WORDS;
    for (int i = threadIdx.x; i < kk * SWEEP_WORDS; i += 256) {
        const int j = i / SWEEP_WORDS, t = i % SWEEP_WORDS;
        sB[j][t] = (k0 + t < Cw) ? bits[(i0 + j) * Cw + k0 + t] : 0ull;
    }
    __syncthreads();
    const int t = threadIdx.x & (SWEEP_WORDS - 1);
    if (k0 + t >= Cw) return;
    const int64_t r_base = (int64_t)blockIdx.y * SWEEP_ROWS;
    for (int rr = threadIdx.x / SWEEP_WORDS; rr < SWEEP_ROWS; rr += 256 / SWEEP_WORDS) {
        const int64_t r = r_base + rr;
        if (r >= R) break;
        uint32_t m = mask[r];
        if (m == 0u) continue;
        uint64_t w = bits[r * Cw + k0 + t];
        while (m) {
            const int j = __ffs(m) - 1;
            m &= m - 1;
            w ^= sB[j][t];
        }
        bits[r * Cw + k0 + t] = w;
    }
}

__global__ void __launch_bounds__(256) rref_final_pivots_kernel(const uint64_t *__restrict__ bits, int64_t R, int64_t Cw,
                                                                 int32_t *__restrict__ pivots) {
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    int p = -1;
    for (int64_t k = 0; k < Cw; ++k) {
        uint64_t w = bits[r * Cw + k];
        if (w) {
            p = (int)(k * 64 + (__ffsll((long long)w) - 1));
            break;
        }
    }
    pivots[r] = p;
}

// Bit-matrix transpose on 32 x 32 bit tiles: lane l holds 32 bits of row (rb*32 + l); 32 ballots turn
// them into the 32 transposed words, lane b keeps word b. Consecutive warps of a CTA take consecutive
// 32-bit column words so a CTA reads 32 contiguous bytes per row.
__global__ void __launch_bounds__(256) bit_transpose_kernel(const uint32_t *__restrict__ in32, int64_t R, int64_t in_words32,
                                                             uint32_t *__restrict__ out32, int64_t out_words32) {
    const int lane = threadIdx.x & 31;
    const int64_t cb = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);   // 32-bit column word of the input
    const int64_t rb = blockIdx.y;                                     // 32-row group of the input
    if (cb >= in_words32) return;
    const int64_t row = rb * 32 + lane;
    const uint32_t w = row < R ? in32[row * in_words32 + cb] : 0u;
    uint32_t mine = 0;
#pragma unroll
    for (int b = 0; b < 32; ++b) {
        const uint32_t v = __ballot_sync(0xffffffffu, (w >> b) & 1u);
        if (lane == b) mine = v;
    }
    out32[(cb * 32 + lane) * out_words32 + rb] = mine;
}

// out[k] = OR over the selected rows of bits[row][k]
__global__ void __launch_bounds__(256) or_rows_kernel(const uint64_t *__restrict__ bits, int64_t Cw, const int32_t *__restrict__ rows,
                                                       int64_t n_rows, uint64_t *__restrict__ out) {
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= Cw) return;
    uint64_t acc = 0;
    for (int64_t i = 0; i < n_rows; ++i) acc |= bits[(int64_t)(rows ? rows[i] : (int32_t)i) * Cw + k];
    out[k] = acc;
}

}  // namespace symb

using namespace symb;

extern "C" int sym_bit_transpose(const uint64_t *in, int64_t R, int64_t Cw_in, uint64_t *out, int64_t Cw_out, void *stream) {
    SYM_REQUIRE(R >= 0 && Cw_in >= 0 && Cw_out * 64 >= R, "bad shape");
    if (Cw_in == 0 || Cw_out == 0) return SYM_OK;
    SYM_REQUIRE(2 * Cw_out <= 65535, "too many input rows for one launch");
    const dim3 grid((unsigned)((2 * Cw_in + 7) / 8), (unsigned)(2 * Cw_out));
    bit_transpose_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint32_t *>(in), R, 2 * Cw_in,
                                                                reinterpret_cast<uint32_t *>(out), 2 * Cw_out);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

extern "C" int sym_or_rows(const uint64_t *bits, int64_t Cw, const int32_t *rows, int64_t n_rows, uint64_t *out, void *stream) {
    SYM_REQUIRE(Cw >= 0 && n_rows >= 0, "bad shape");
    if (Cw == 0) return SYM_OK;
    or_rows_kernel<<<(unsigned)((Cw + 255) / 256), 256, 0, (cudaStream_t)stream>>>(bits, Cw, rows, n_rows, out);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

extern "C" size_t sym_rref_ws_bytes(int64_t R) { return arena_need((size_t)(R > 0 ? R : 1), 4) + 1024; }

namespace symb { int g_rref_variant = 1; }  // tuning knob 5: 1 = blocked panels (default), 0 = one pivot per sweep

extern "C" int sym_rref(uint64_t *bits, int64_t R, int64_t C, int64_t Cw, int32_t *pivots, void *ws, size_t ws_bytes,
                        void *stream) {
    SYM_REQUIRE(R >= 0 && C >= 0 && Cw * 64 >= C, "bad matrix shape");
    SYM_REQUIRE(C < ((int64_t)1 << 31) && R < ((int64_t)1 << 31), "matrix too large");
    cudaStream_t st = (cudaStream_t)stream;
    if (R == 0) return SYM_OK;
    if (Cw == 0) {
        SYM_CUDA_OK(cudaMemsetAsync(pivots, 0xff, sizeof(int32_t) * (size_t)R, st));
        return SYM_OK;
    }
    const size_t smem = (size_t)R * (size_t)Cw * 8;
    int dev = 0;
    cudaGetDevice(&dev);
    if (smem <= 200 * 1024) {
        static bool attr_done[64] = {};   // per device
        if (dev >= 0 && dev < 64 && !attr_done[dev]) {
            SYM_CUDA_OK(cudaFuncSetAttribute(rref_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            attr_done[dev] = true;
        }
        rref_smem_kernel<<<1, RREF_THREADS, smem, st>>>(bits, (int)R, Cw, pivots);
        SYM_LAUNCH_OK();
        return SYM_OK;
    }
    if (ws_bytes < sym_rref_ws_bytes(R)) {
        set_error("workspace too small");
        return SYM_E_WORKSPACE;
    }
    Arena ar(ws, ws_bytes);
    const size_t panel_cap = 200 * 1024;
    int kk = (int)(panel_cap / ((size_t)Cw * 8));
    if (kk > PANEL_MAX) kk = PANEL_MAX;
    if (g_rref_variant == 1 && kk >= 1) {
        uint32_t *mask = ar.take<uint32_t>((size_t)R);
        int *pv = ar.take<int>(PANEL_MAX);
        static bool attr_done[64] = {};   // per device
        if (dev >= 0 && dev < 64 && !attr_done[dev]) {
            SYM_CUDA_OK(cudaFuncSetAttribute(rref_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)panel_cap));
            attr_done[dev] = true;
        }
        const dim3 sweep_grid((unsigned)((Cw + SWEEP_WORDS - 1) / SWEEP_WORDS), (unsigned)((R + SWEEP_ROWS - 1) / SWEEP_ROWS));
        for (int64_t i0 = 0; i0 < R; i0 += kk) {
            const int k = (int)((R - i0) < kk ? (R - i0) : kk);
            rref_panel_kernel<<<1, RREF_THREADS, (size_t)k * (size_t)Cw * 8, st>>>(bits, Cw, i0, k, pv);
            SYM_LAUNCH_OK();
            rref_mask_kernel<<<(unsigned)((R + 255) / 256), 256, 0, st>>>(bits, R, Cw, i0, k, pv, mask);
            SYM_LAUNCH_OK();
            rref_sweep_kernel<<<sweep_grid, 256, 0, st>>>(bits, R, Cw, i0, k, mask);
            SYM_LAUNCH_OK();
        }
        rref_final_pivots_kernel<<<(unsigned)((R + 255) / 256), 256, 0, st>>>(bits, R, Cw, pivots);
        SYM_LAUNCH_OK();
        return SYM_OK;
    }
    uint8_t *hit = ar.take<uint8_t>((size_t)R);
    int *piv = reinterpret_cast<int *>(ar.take<int>(4));
    const int64_t cells = R * Cw;
    for (int64_t i = 0; i < R; ++i) {
        rref_pivot_kernel<<<1, RREF_THREADS, 0, st>>>(bits, R, Cw, i, piv);
        SYM_LAUNCH_OK();
        rref_hit_kernel<<<(unsigned)((R + 255) / 256), 256, 0, st>>>(bits, R, Cw, i, piv, hit);
        SYM_LAUNCH_OK();
        rref_xor_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(bits, R, Cw, i, hit);
        SYM_LAUNCH_OK();
    }
    rref_final_pivots_kernel<<<(unsigned)((R + 255) / 256), 256, 0, st>>>(bits, R, Cw, pivots);
    SYM_LAUNCH_OK();
    return SYM_OK;
}
