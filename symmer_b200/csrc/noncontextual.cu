// Ground state of a noncontextual Hamiltonian (CS-VQE; symmer/operators/noncontextual_op.py).
//
// A noncontextual H decomposes as P_t = s_t * G^{J_t} * C_{i_t}: k commuting generators G, N pairwise anticommuting
// clique representatives C (left out for the symmetry terms, i_t = -1) and a sign s_t = +-1. For an assignment
// nu in {+-1}^k, encoded as the bitmask m (bit j set <=> nu_j = -1), the quasi-quantized energy minimised over the
// unit vector r is
//     E(m) = a(m) - ||w(m)||,   a(m) = sum_{t sym} v_t (-1)^{|J_t & m|},   w_i(m) = sum_{t in clique i} v_t (-1)^{|J_t & m|}
// with v_t = h_t s_t, and min_m E(m) is the lowest eigenvalue of H (Kirby & Love).
//
// a and every w_i are Walsh-Hadamard transforms of sparse functions of J, so the 2^f assignments are enumerated as
// tiles: m = (hi << NC_LO) | lo. One CTA per high pattern hi builds g_hi(J_lo) = sum_t v_t (-1)^{|J_t^hi & hi|} in
// shared memory and transforms it over the NC_LO low bits; the 4096 values of a and of sum_i w_i^2 that come out
// are the tile's energies. Cost per assignment: (N+1) * NC_LO butterflies + M / 2^NC_LO term reads, against M sign
// evaluations for the direct form.
#include "common.cuh"
#include "sort.cuh"

namespace symb {

constexpr int NC_LO = 12;                 // low assignment bits per tile: 4096 doubles = 32 KB of shared memory
constexpr int NC_TILE = 1 << NC_LO;
constexpr int NC_THREADS = 256;           // 16 tile entries per thread
constexpr int NC_PER = NC_TILE / NC_THREADS;
constexpr int NC_MAX_CTAS = 2048;
constexpr int NC_KEY_SHIFT = 52;          // sort key: (clique + 1) << 52 | J_lo << 40
constexpr int NC_MAX_CLIQUES = 4094;

// s_t of P_t = s_t * G^{J_t} * C_{i_t}: the factors are multiplied in order with the phase rule of rows.cuh
// (sigma(x, z) = i^{|x&z|} X^x Z^z, so sigma(a) sigma(b) = i^{Y_a + Y_b - Y_ab} (-1)^{|z_a & x_b|} sigma(a ^ b)), word by
// word since the exponents only add. 0 marks a term whose product is not +-P_t.
__global__ void __launch_bounds__(256) nc_signs_kernel(const uint64_t *__restrict__ xz, int64_t M, int W,
                                                       const uint64_t *__restrict__ gen, int k,
                                                       const uint64_t *__restrict__ rep, int N,
                                                       const uint64_t *__restrict__ J, int Jw,
                                                       const int32_t *__restrict__ clique, double *__restrict__ signs) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= M) return;
    const int cl = clique[t];
    bool ok = cl >= -1 && cl < N;
    int e = 0;
    for (int w = 0; ok && w < W; ++w) {
        uint64_t x = 0, z = 0;
        for (int jw = 0; jw < Jw; ++jw) {
            uint64_t bits = J[t * Jw + jw];
            while (bits) {
                const int j = 64 * jw + __ffsll((long long)bits) - 1;
                bits &= bits - 1;
                if (j >= k) { ok = false; break; }
                const uint64_t gx = gen[(size_t)j * 2 * W + w], gz = gen[(size_t)j * 2 * W + W + w];
                e += __popcll(gx & gz) + 2 * __popcll(z & gx);
                x ^= gx;
                z ^= gz;
            }
        }
        if (ok && cl >= 0) {
            const uint64_t cx = rep[(size_t)cl * 2 * W + w], cz = rep[(size_t)cl * 2 * W + W + w];
            e += __popcll(cx & cz) + 2 * __popcll(z & cx);
            x ^= cx;
            z ^= cz;
        }
        e -= __popcll(x & z);
        ok = ok && x == xz[t * 2 * W + w] && z == xz[t * 2 * W + W + w];
    }
    e &= 3;
    signs[t] = !ok || (e & 1) ? 0.0 : (e == 0 ? 1.0 : -1.0);
}

__global__ void __launch_bounds__(256) nc_keys_kernel(const uint64_t *__restrict__ J, const int32_t *__restrict__ clique,
                                                      int64_t M, uint64_t *__restrict__ keys, uint32_t *__restrict__ idx) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= M) return;
    keys[t] = ((uint64_t)(uint32_t)(clique[t] + 1) << NC_KEY_SHIFT) | ((J[t] & (NC_TILE - 1)) << 40);
    idx[t] = (uint32_t)t;
}

// Terms in (clique, J_lo) order; fn_start[phi] = first term of function phi (0: symmetry terms, 1 + i: clique i).
// Keys of an out-of-range clique sort outside [fn_start[0], fn_start[N + 1]) and are never read.
__global__ void __launch_bounds__(256) nc_gather_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ idx,
                                                        const uint64_t *__restrict__ J, const double *__restrict__ v,
                                                        int64_t M, int N, uint64_t *__restrict__ Js, double *__restrict__ vs,
                                                        int64_t *__restrict__ fn_start) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < M) {
        Js[t] = J[idx[t]];
        vs[t] = v[idx[t]];
    }
    if (t <= N + 1) {
        const uint64_t target = (uint64_t)t << NC_KEY_SHIFT;
        int64_t lo = 0, hi = M;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (keys[mid] < target) lo = mid + 1; else hi = mid;
        }
        fn_start[t] = lo;
    }
}

__device__ __forceinline__ bool nc_better(double e1, uint64_t m1, double e2, uint64_t m2) {
    return e1 < e2 || (e1 == e2 && m1 < m2);
}

// (E, m) minimum of the CTA, ties to the smaller m; thread 0 returns it
__device__ __forceinline__ void nc_block_min(double &be, uint64_t &bm) {
    __shared__ double se[NC_THREADS / 32];
    __shared__ uint64_t sm[NC_THREADS / 32];
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const double oe = __shfl_xor_sync(0xffffffffu, be, s);
        const uint64_t om = __shfl_xor_sync(0xffffffffu, bm, s);
        if (nc_better(oe, om, be, bm)) { be = oe; bm = om; }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { se[warp] = be; sm[warp] = bm; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < NC_THREADS / 32; ++i)
            if (nc_better(se[i], sm[i], be, bm)) { be = se[i]; bm = sm[i]; }
    }
    __syncthreads();
}

// One CTA per high pattern (grid-stride). Tile entry e = lo is held in two layouts:
//   A: e = tid + 256 r       (r = bits 8..11: butterflies in registers; lane = bits 0..4: butterflies by shuffles)
//   B: e = lane | (r & 7) << 5 | (r >> 3) << 8 | warp << 9   (r & 7 = bits 5..7: butterflies in registers)
// so every one of the 12 stages runs in registers or shuffles and the tile crosses shared memory twice per function.
__global__ void __launch_bounds__(NC_THREADS) nc_min_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ Js,
                                                            const double *__restrict__ vs, const int64_t *__restrict__ fn_start,
                                                            int N, int f, int64_t n_hi, double *__restrict__ cta_e,
                                                            uint64_t *__restrict__ cta_m) {
    __shared__ double tile[NC_TILE];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t lo_count = f < NC_LO ? (1u << f) : (uint32_t)NC_TILE;
    double best_e = __longlong_as_double(0x7ff0000000000000LL);     // +inf
    uint64_t best_m = ~0ull;
    for (int64_t h = blockIdx.x; h < n_hi; h += gridDim.x) {
        double acc_a[NC_PER], acc_w[NC_PER];
#pragma unroll
        for (int r = 0; r < NC_PER; ++r) { acc_a[r] = 0.0; acc_w[r] = 0.0; }
        for (int phi = 0; phi <= N; ++phi) {
            const int64_t s = fn_start[phi], end = fn_start[phi + 1];
            if (s == end) continue;                                   // uniform over the CTA
#pragma unroll
            for (int r = 0; r < NC_PER; ++r) tile[tid + NC_THREADS * r] = 0.0;
            __syncthreads();
            // one thread per run of equal J_lo, summed sequentially in the sorted order
            for (int64_t i = s + tid; i < end; i += NC_THREADS) {
                if (i != s && keys[i] == keys[i - 1]) continue;
                double g = 0.0;
                int64_t j = i;
                do {
                    const double v = vs[j];
                    g += (__popcll((Js[j] >> NC_LO) & (uint64_t)h) & 1) ? -v : v;
                    ++j;
                } while (j < end && keys[j] == keys[i]);
                tile[Js[i] & (NC_TILE - 1)] = g;
            }
            __syncthreads();
            double x[NC_PER];
#pragma unroll
            for (int r = 0; r < NC_PER; ++r) x[r] = tile[tid + NC_THREADS * r];
#pragma unroll
            for (int b = 1; b < NC_PER; b <<= 1)
#pragma unroll
                for (int r = 0; r < NC_PER; ++r)
                    if (!(r & b)) {
                        const double p = x[r], q = x[r | b];
                        x[r] = p + q;
                        x[r | b] = p - q;
                    }
#pragma unroll
            for (int b = 1; b < 32; b <<= 1)
#pragma unroll
                for (int r = 0; r < NC_PER; ++r) {
                    const double o = __shfl_xor_sync(0xffffffffu, x[r], b);
                    x[r] = (lane & b) ? o - x[r] : x[r] + o;
                }
#pragma unroll
            for (int r = 0; r < NC_PER; ++r) tile[tid + NC_THREADS * r] = x[r];
            __syncthreads();
#pragma unroll
            for (int r = 0; r < NC_PER; ++r) x[r] = tile[lane | ((r & 7) << 5) | ((r >> 3) << 8) | (warp << 9)];
#pragma unroll
            for (int b = 1; b < 8; b <<= 1)
#pragma unroll
                for (int r = 0; r < NC_PER; ++r)
                    if (!(r & b)) {
                        const double p = x[r], q = x[r | b];
                        x[r] = p + q;
                        x[r | b] = p - q;
                    }
            __syncthreads();                                          // the next function overwrites the tile
            if (phi == 0) {
#pragma unroll
                for (int r = 0; r < NC_PER; ++r) acc_a[r] = x[r];
            } else {
#pragma unroll
                for (int r = 0; r < NC_PER; ++r) acc_w[r] = fma(x[r], x[r], acc_w[r]);
            }
        }
#pragma unroll
        for (int r = 0; r < NC_PER; ++r) {
            const uint32_t lo = lane | ((r & 7) << 5) | ((r >> 3) << 8) | (warp << 9);
            const double e = acc_a[r] - sqrt(acc_w[r]);
            const uint64_t m = ((uint64_t)h << NC_LO) | lo;
            if (lo < lo_count && nc_better(e, m, best_e, best_m)) { best_e = e; best_m = m; }
        }
    }
    nc_block_min(best_e, best_m);
    if (tid == 0) {
        cta_e[blockIdx.x] = best_e;
        cta_m[blockIdx.x] = best_m;
    }
}

// Ordered final reduction of the per-CTA minima into best = {double E; uint64 m}
__global__ void __launch_bounds__(NC_THREADS) nc_final_kernel(const double *__restrict__ cta_e, const uint64_t *__restrict__ cta_m,
                                                              int n, uint64_t *__restrict__ best) {
    double be = __longlong_as_double(0x7ff0000000000000LL);
    uint64_t bm = ~0ull;
    for (int i = threadIdx.x; i < n; i += NC_THREADS)
        if (nc_better(cta_e[i], cta_m[i], be, bm)) { be = cta_e[i]; bm = cta_m[i]; }
    nc_block_min(be, bm);
    if (threadIdx.x == 0) {
        best[0] = (uint64_t)__double_as_longlong(be);
        best[1] = bm;
    }
}

struct NcWorkspace {
    uint64_t *keys, *keys_alt, *Js;
    uint32_t *idx, *idx_alt, *hist;
    double *vs, *cta_e;
    uint64_t *cta_m;
    int64_t *fn_start;
};

static size_t nc_ws_layout(int64_t M, int32_t N, NcWorkspace *out, void *ws, size_t ws_bytes) {
    const size_t m = (size_t)(M < 1 ? 1 : M);
    const size_t need = 4 * arena_need(m, 8) + 2 * arena_need(m, 4) + arena_need(record_hist_elems((int64_t)m), 4) +
                        2 * arena_need(NC_MAX_CTAS, 8) + arena_need((size_t)N + 2, 8);
    if (out) {
        Arena ar(ws, ws_bytes);
        out->keys = ar.take<uint64_t>(m);
        out->keys_alt = ar.take<uint64_t>(m);
        out->Js = ar.take<uint64_t>(m);
        out->idx = ar.take<uint32_t>(m);
        out->idx_alt = ar.take<uint32_t>(m);
        out->hist = ar.take<uint32_t>(record_hist_elems((int64_t)m));
        out->vs = ar.take<double>(m);
        out->cta_e = ar.take<double>(NC_MAX_CTAS);
        out->cta_m = ar.take<uint64_t>(NC_MAX_CTAS);
        out->fn_start = ar.take<int64_t>((size_t)N + 2);
    }
    return need;
}

}  // namespace symb

using namespace symb;

extern "C" int sym_nc_signs(const uint64_t *xz, int64_t M, int32_t W, const uint64_t *gen_xz, int32_t k,
                            const uint64_t *rep_xz, int32_t N, const uint64_t *J, int32_t Jw, const int32_t *clique,
                            double *signs, void *stream) {
    SYM_REQUIRE(M >= 0 && M < ((int64_t)1 << 40) && W >= 1, "bad operator size");
    SYM_REQUIRE(k >= 0 && N >= 0 && Jw >= 0 && (int64_t)k <= 64 * (int64_t)Jw, "bad generator or J size");
    if (M == 0) return SYM_OK;
    nc_signs_kernel<<<(unsigned)((M + 255) / 256), 256, 0, (cudaStream_t)stream>>>(xz, M, W, gen_xz, k, rep_xz, N, J, Jw,
                                                                                   clique, signs);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

extern "C" size_t sym_nc_min_ws_bytes(int64_t M, int32_t N) {
    if (M < 0 || N < 0 || N > NC_MAX_CLIQUES) return 0;
    return nc_ws_layout(M, N, nullptr, nullptr, 0);
}

extern "C" int sym_nc_min(const uint64_t *J, const double *v, const int32_t *clique, int64_t M, int32_t N, int32_t f,
                          void *best, void *best_host, void *ws, size_t ws_bytes, void *stream) {
    SYM_REQUIRE(M >= 0 && M < (int64_t)4000000000LL, "M out of range");
    SYM_REQUIRE(N >= 0 && N <= NC_MAX_CLIQUES, "N out of range");
    SYM_REQUIRE(f >= 0 && f <= 62, "need 0 <= f <= 62 free generators");
    SYM_REQUIRE(best != nullptr, "best is required");
    if (ws_bytes < sym_nc_min_ws_bytes(M, N)) {
        set_error("workspace too small");
        return SYM_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    NcWorkspace w;
    nc_ws_layout(M, N, &w, ws, ws_bytes);
    const int64_t prep = M > N + 2 ? M : N + 2;
    if (M > 0) {
        nc_keys_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(J, clique, M, w.keys, w.idx);
        SYM_LAUNCH_OK();
        uint64_t *sorted = w.keys;
        SYM_TRY(radix_sort(w.keys, w.idx, w.keys_alt, w.idx_alt, M, 40, w.hist, &sorted, st));
        const uint32_t *idx = sorted == w.keys ? w.idx : w.idx_alt;
        if (sorted != w.keys) w.keys = sorted;
        nc_gather_kernel<<<(unsigned)((prep + 255) / 256), 256, 0, st>>>(w.keys, idx, J, v, M, N, w.Js, w.vs, w.fn_start);
    } else {
        nc_gather_kernel<<<(unsigned)((prep + 255) / 256), 256, 0, st>>>(w.keys, w.idx, J, v, 0, N, w.Js, w.vs, w.fn_start);
    }
    SYM_LAUNCH_OK();
    const int64_t n_hi = f > NC_LO ? ((int64_t)1 << (f - NC_LO)) : 1;
    const int64_t cap = (int64_t)num_sms() * 8 < NC_MAX_CTAS ? (int64_t)num_sms() * 8 : NC_MAX_CTAS;
    const int grid = (int)(n_hi < cap ? n_hi : cap);
    nc_min_kernel<<<grid, NC_THREADS, 0, st>>>(w.keys, w.Js, w.vs, w.fn_start, N, f, n_hi, w.cta_e, w.cta_m);
    SYM_LAUNCH_OK();
    nc_final_kernel<<<1, NC_THREADS, 0, st>>>(w.cta_e, w.cta_m, grid, static_cast<uint64_t *>(best));
    SYM_LAUNCH_OK();
    if (best_host) {
        SYM_CUDA_OK(cudaMemcpyAsync(best_host, best, 16, cudaMemcpyDeviceToHost, st));
        SYM_CUDA_OK(cudaStreamSynchronize(st));
    }
    return SYM_OK;
}
