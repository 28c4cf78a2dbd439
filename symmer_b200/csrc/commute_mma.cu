// commutes_termwise (symmer/operators/base.py:938-971) on the 5th-generation tensor cores:
// the symplectic inner product  A.x . B.z^T + A.z . B.x^T  as an int8 tcgen05.mma on UNPACKED bits,
// followed by a parity step (commute <=> even), i.e. the reference's own formulation
// (`matmul_GF2`: integer GEMM then mod 2, utils.py:63-78) with exact int32 accumulation in TMEM.
//
// One CTA computes a 128 (A rows) x 256 (B rows) tile of the output. The packed operands (16 B of
// bits per row and stage) are read from L2 and expanded on the fly to operand bytes in shared memory in
// the canonical K-major no-swizzle UMMA layout (8-row x 16-byte core matrices). The kernel is
// warp-specialised: EXPANDER warps turn packed bits into operand bytes, one ISSUER warp feeds the tensor
// core (4 x tcgen05.mma kind::i8, M=128 N=256 K=32 per stage); they meet only through mbarriers
// (full[s]: every expander has written stage s; empty[s]: the MMAs that read stage s have completed,
// signalled by tcgen05.commit), so there is no block-wide barrier in the main loop and the tensor core
// works on stage s while the next stage is being expanded. Epilogue: tcgen05.ld of the int32
// accumulators, parity, byte stores. Never pre-unpacks the operands in HBM (8x the bytes).
//
// Shape: 2 stages of 48 KB, 8 expander warps, two CTAs per SM (256 TMEM columns each). Measured on B200
// at 1000 qubits: 5.7e11 pairs/s, against 4.4e11 for a form where all warps expand and meet the MMAs at
// a block barrier, and 4.0e11 for one CTA per SM with 3-4 stages and 8 or 16 expander warps: the
// expansion (ALU) needs the second CTA's warps to hide its latency.
#include "common.cuh"

namespace symb {

constexpr int MMA_M = 128;
constexpr int MMA_N = 256;
constexpr int MMA_THREADS = 256;
constexpr int STAGE_WORDS = 2;                      // 64-bit words of packed bits per row and stage
constexpr int STAGE_KBYTES = STAGE_WORDS * 64;      // 128 unpacked bytes of K per stage
constexpr int A_STAGE_BYTES = MMA_M * STAGE_KBYTES; // 16 KB
constexpr int B_STAGE_BYTES = MMA_N * STAGE_KBYTES; // 32 KB
constexpr int MMA_STAGES = 2;
constexpr int TMEM_COLS = 256;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major, no swizzle: core matrix = 8 rows x 16 B contiguous (128 B); SBO = stride between 8-row
// groups, LBO = stride between 16-byte K chunks (both in bytes, encoded >> 4). version = 1 (sm_100).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;  // descriptor version for Blackwell
    return d;                // base_offset = 0, lbo_mode = 0, layout_type = SWIZZLE_NONE (0)
}

// instruction descriptor, kind::i8: D = S32, A/B = unsigned 8-bit, both K-major, dense
__device__ __forceinline__ uint32_t make_idesc_i8(int m, int n) {
    return (2u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    }
}

__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u)
        : "memory");
}

// 16 packed bits -> 16 operand bytes: nibble * 0x00204081 puts bit k of the nibble at the LEAST SIGNIFICANT bit of byte k
// (the copies n, n<<7, n<<14, n<<21 do not overlap, so no carries). The higher bits of every byte are left as they
// fall: only the PARITY of the int32 dot product is used, and the parity of sum(a_i * b_i) depends on the low bits of
// a_i and b_i alone (bytes are unsigned and <= 227, so the sum stays below 2^31 up to ~20 000 qubits). Dropping
// the `& 0x01010101` of the 0/1 encoding saves a third of the expansion's ALU work, which is what limits the kernel.
__device__ __forceinline__ uint4 expand16(uint32_t bits) {
    uint4 v;
    v.x = (bits & 0xFu) * 0x00204081u;
    v.y = ((bits >> 4) & 0xFu) * 0x00204081u;
    v.z = ((bits >> 8) & 0xFu) * 0x00204081u;
    v.w = ((bits >> 12) & 0xFu) * 0x00204081u;
    return v;
}

// Word-major copies of the operands: t[k][row] = word k of row `row` (for B with the X and Z halves
// swapped, so that A'.B'^T is the symplectic form). With this layout the per-stage reads of a tile
// are coalesced (consecutive rows -> consecutive 8-byte words).
__global__ void __launch_bounds__(256) transpose_words_kernel(const uint64_t *__restrict__ xz, uint32_t rows, int words,
                                                               int swap_halves, uint64_t *__restrict__ t) {
    __shared__ uint64_t tile[32][33];
    const uint32_t r0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    for (int j = ty; j < 32; j += 8) {
        const uint32_t r = r0 + j, k = k0 + tx;
        tile[j][tx] = (r < rows && k < (uint32_t)words) ? xz[(size_t)r * words + k] : 0ull;
    }
    __syncthreads();
    const int W = words / 2;
    for (int j = ty; j < 32; j += 8) {
        const uint32_t k = k0 + j, r = r0 + tx;
        if (k < (uint32_t)words && r < rows) {
            const uint32_t kd = swap_halves ? (k + W) % words : k;   // B' word kd = B row word k
            t[(size_t)kd * rows + r] = tile[tx][j];
        }
    }
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// one packed word (64 bits) of row r -> 4 chunks of 16 bytes starting at K chunk `c0`
__device__ __forceinline__ void expand_word(unsigned char *stage, int rows, int r, int c0, uint64_t w) {
    unsigned char *base = stage + (r >> 3) * 128 + (r & 7) * 16;
    const uint32_t lbo = (uint32_t)rows * 16u;
#pragma unroll
    for (int c = 0; c < 4; ++c) *reinterpret_cast<uint4 *>(base + (c0 + c) * lbo) = expand16((uint32_t)(w >> (16 * c)) & 0xFFFFu);
}

// MMA_STAGES x 48 KB of operand bytes; 8 expander warps, a thread expands both words of its rows
__global__ void __launch_bounds__(MMA_THREADS + 32, 2) commute_mma_ws_kernel(const uint64_t *__restrict__ a_t, uint32_t M,
                                                                             const uint64_t *__restrict__ b_t, uint32_t N, int W,
                                                                             uint8_t *__restrict__ out, size_t pitch) {
    constexpr int EXPANDERS = MMA_THREADS;
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + MMA_STAGES * (A_STAGE_BYTES + B_STAGE_BYTES));
    uint64_t *empty = full + MMA_STAGES;
    uint64_t *done = empty + MMA_STAGES;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(done + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t i0 = blockIdx.y * MMA_M, j0 = blockIdx.x * MMA_N;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < MMA_STAGES; ++s) {
            mbar_init(&full[s], EXPANDERS);
            mbar_init(&empty[s], 1);
        }
        mbar_init(done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    const int iters = (2 * W) / STAGE_WORDS;

    if (warp == EXPANDERS / 32) {
        // ---- issuer warp: one elected lane
        if (lane == 0) {
            const uint32_t idesc = make_idesc_i8(MMA_M, MMA_N);
            int s = 0;
            uint32_t ph = 0;
            for (int it = 0; it < iters; ++it) {
                mbar_wait(&full[s], ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_addr = smem_u32(smem + s * (A_STAGE_BYTES + B_STAGE_BYTES)), b_addr = a_addr + A_STAGE_BYTES;
#pragma unroll
                for (int kk = 0; kk < STAGE_KBYTES / 32; ++kk) {
                    const uint64_t da = make_smem_desc(a_addr + kk * 2 * (MMA_M * 16), MMA_M * 16, 128);
                    const uint64_t db = make_smem_desc(b_addr + kk * 2 * (MMA_N * 16), MMA_N * 16, 128);
                    umma_i8(tmem_base, da, db, idesc, (it > 0 || kk > 0) ? 1u : 0u);
                }
                umma_commit(&empty[s]);
                if (it == iters - 1) umma_commit(done);
                if (++s == MMA_STAGES) {
                    s = 0;
                    ph ^= 1u;
                }
            }
        }
    } else {
        // ---- expander warps: thread = B row and, for rows < 128, an A row
        const int r = tid;
        const uint32_t jb = j0 + r;
        const bool b_ok = jb < N;
        const uint32_t ia = i0 + r;
        const bool a_ok = r < MMA_M && ia < M;
        uint64_t bw[2], aw[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const size_t k = (size_t)h;
            bw[h] = b_ok ? b_t[k * N + jb] : 0ull;
            aw[h] = a_ok ? a_t[k * M + ia] : 0ull;
        }
        int s = 0;
        uint32_t ph = 0;
        for (int it = 0; it < iters; ++it) {
            uint64_t nb[2] = {0ull, 0ull}, na[2] = {0ull, 0ull};
            if (it + 1 < iters) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const size_t k = (size_t)(it + 1) * STAGE_WORDS + h;
                    nb[h] = b_ok ? b_t[k * N + jb] : 0ull;
                    na[h] = a_ok ? a_t[k * M + ia] : 0ull;
                }
            }
            if (it >= MMA_STAGES) mbar_wait(&empty[s], ph ^ 1u);
            unsigned char *stA = smem + s * (A_STAGE_BYTES + B_STAGE_BYTES), *stB = stA + A_STAGE_BYTES;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int c0 = 4 * h;
                expand_word(stB, MMA_N, r, c0, bw[h]);
                if (r < MMA_M) expand_word(stA, MMA_M, r, c0, aw[h]);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core
            mbar_arrive(&full[s]);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                bw[h] = nb[h];
                aw[h] = na[h];
            }
            if (++s == MMA_STAGES) {
                s = 0;
                ph ^= 1u;
            }
        }
        mbar_wait(done, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (warp < 8) {
            // epilogue: warp w reads TMEM lanes 32*(w%4).., columns 128*(w/4)..; thread = one output row
            const uint32_t row = i0 + (warp & 3) * 32 + lane;
            const uint32_t col_half = (warp >> 2) * 128;
#pragma unroll 1
            for (int cb = 0; cb < 128; cb += 32) {
                uint32_t v[32];
                const uint32_t taddr = tmem_base + (((uint32_t)(warp & 3) * 32u) << 16) + col_half + cb;
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                      "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
                      "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
                      "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                    : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (row < M) {
                    const uint32_t jbase = j0 + col_half + cb;
                    uint8_t *dst = out + (size_t)row * pitch + jbase;
                    if (jbase + 32 <= pitch && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
                        uint32_t p[8];
#pragma unroll
                        for (int q = 0; q < 8; ++q)
                            p[q] = ((v[4 * q] & 1u) ^ 1u) | (((v[4 * q + 1] & 1u) ^ 1u) << 8) | (((v[4 * q + 2] & 1u) ^ 1u) << 16) |
                                   (((v[4 * q + 3] & 1u) ^ 1u) << 24);
                        reinterpret_cast<uint4 *>(dst)[0] = make_uint4(p[0], p[1], p[2], p[3]);
                        reinterpret_cast<uint4 *>(dst)[1] = make_uint4(p[4], p[5], p[6], p[7]);
                    } else {
#pragma unroll
                        for (int q = 0; q < 32; ++q)
                            if (jbase + q < N) dst[q] = (uint8_t)((v[q] & 1u) ^ 1u);
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

}  // namespace symb

using namespace symb;

extern "C" size_t sym_commute_mma_ws_bytes(int64_t M, int64_t N, int32_t W) {
    return arena_need((size_t)(M > 0 ? M : 1) * 2 * W, 8) + arena_need((size_t)(N > 0 ? N : 1) * 2 * W, 8) + 1024;
}

extern "C" int sym_commute_mma(const uint64_t *a_xz, int64_t M, const uint64_t *b_xz, int64_t N, int32_t W, uint8_t *out,
                               void *ws, size_t ws_bytes, void *stream) {
    return sym_commute_mma_pitched(a_xz, M, b_xz, N, W, out, N, ws, ws_bytes, stream);
}

extern "C" int sym_commute_mma_pitched(const uint64_t *a_xz, int64_t M, const uint64_t *b_xz, int64_t N, int32_t W,
                                       uint8_t *out, int64_t out_pitch, void *ws, size_t ws_bytes, void *stream) {
    SYM_REQUIRE(M >= 0 && N >= 0 && W >= 1, "bad size");
    SYM_REQUIRE(out_pitch >= N, "out_pitch must be >= N");
    SYM_REQUIRE(M < ((int64_t)1 << 31) && N < ((int64_t)1 << 31), "operand too large");
    if (M == 0 || N == 0) return SYM_OK;
    if (ws_bytes < sym_commute_mma_ws_bytes(M, N, W)) {
        set_error("workspace too small");
        return SYM_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    Arena ar(ws, ws_bytes);
    uint64_t *a_t = ar.take<uint64_t>((size_t)M * 2 * W);
    uint64_t *b_t = ar.take<uint64_t>((size_t)N * 2 * W);
    const int words = 2 * W;
    transpose_words_kernel<<<dim3((unsigned)((M + 31) / 32), (unsigned)((words + 31) / 32)), 256, 0, st>>>(a_xz, (uint32_t)M,
                                                                                                        words, 0, a_t);
    SYM_LAUNCH_OK();
    transpose_words_kernel<<<dim3((unsigned)((N + 31) / 32), (unsigned)((words + 31) / 32)), 256, 0, st>>>(b_xz, (uint32_t)N,
                                                                                                        words, 1, b_t);
    SYM_LAUNCH_OK();
    constexpr size_t smem = MMA_STAGES * (A_STAGE_BYTES + B_STAGE_BYTES) + 128;
    static bool attr_done[64] = {};   // per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !attr_done[dev]) {
        SYM_CUDA_OK(cudaFuncSetAttribute(commute_mma_ws_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev] = true;
    }
    const int64_t tiles_m = (M + MMA_M - 1) / MMA_M;
    SYM_REQUIRE(tiles_m <= 65535, "too many A rows for one launch (slice A)");
    dim3 grid((unsigned)((N + MMA_N - 1) / MMA_N), (unsigned)tiles_m);
    commute_mma_ws_kernel<<<grid, MMA_THREADS + 32, smem, st>>>(a_t, (uint32_t)M, b_t, (uint32_t)N, W, out, (size_t)out_pitch);
    SYM_LAUNCH_OK();
    return SYM_OK;
}
