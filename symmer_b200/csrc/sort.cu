// Exclusive scan, hand-written for sm_100a, and the C ABI of the pair sort (record_sort.cu).
// HBM-bound integer work: coalesced 16-byte accesses, grids sized by the data (thousands of CTAs >> 148 SMs).
#include "sort.cuh"

namespace symb {

// ---------------------------------------------------------------------------------------------
// scan
// ---------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 16;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

template <typename T>
__device__ __forceinline__ void load_items(const T *__restrict__ in, int64_t base, int64_t n, uint32_t (&v)[SCAN_ITEMS]) {
    if (base + SCAN_ITEMS <= n) {
        if constexpr (sizeof(T) == 1) {
            uint4 q = *reinterpret_cast<const uint4 *>(in + base);
            uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = (w[j >> 2] >> ((j & 3) * 8)) & 0xffu;
        } else {
            const uint4 *p = reinterpret_cast<const uint4 *>(in + base);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                uint4 q = p[j];
                v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w;
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < SCAN_ITEMS; ++j) v[j] = (base + j < n) ? static_cast<uint32_t>(in[base + j]) : 0u;
    }
}

template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS) scan_reduce_kernel(const T *__restrict__ in, int64_t n,
                                                                    uint32_t *__restrict__ sums) {
    __shared__ uint32_t warp_sum[SCAN_THREADS / 32];
    int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    load_items(in, base, n, v);
    uint32_t s = 0;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) s += v[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
#pragma unroll
        for (int w = 0; w < SCAN_THREADS / 32; ++w) t += warp_sum[w];
        sums[blockIdx.x] = t;
    }
}

// single block: exclusive scan of sums[0..nb) in place, total -> *total
__global__ void __launch_bounds__(1024) scan_sums_kernel(uint32_t *__restrict__ sums, int64_t nb,
                                                         uint32_t *__restrict__ total) {
    __shared__ uint32_t warp_tot[32];
    __shared__ uint32_t carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int64_t base = 0; base < nb; base += 1024) {
        int64_t i = base + threadIdx.x;
        uint32_t x = (i < nb) ? sums[i] : 0u;
        uint32_t inc = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        if (lane == 31) warp_tot[wid] = inc;
        __syncthreads();
        if (wid == 0) {
            uint32_t t = warp_tot[lane];
            uint32_t ti = t;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                uint32_t y = __shfl_up_sync(0xffffffffu, ti, o);
                if (lane >= o) ti += y;
            }
            warp_tot[lane] = ti - t;  // exclusive warp offsets
        }
        __syncthreads();
        uint32_t excl = carry_s + warp_tot[wid] + inc - x;
        if (i < nb) sums[i] = excl;
        __syncthreads();  // every thread has consumed carry_s and warp_tot
        if (threadIdx.x == 1023) carry_s = excl + x;
        __syncthreads();
    }
    if (threadIdx.x == 0 && total != nullptr) *total = carry_s;
}

template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS) scan_apply_kernel(const T *in, uint32_t *out,
                                                                   int64_t n, const uint32_t *__restrict__ sums) {
    __shared__ uint32_t warp_tot[SCAN_THREADS / 32];
    int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    load_items(in, base, n, v);
    uint32_t s = 0;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) {
        uint32_t t = v[j];
        v[j] = s;
        s += t;
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    uint32_t woff = 0;
#pragma unroll
    for (int w = 0; w < SCAN_THREADS / 32; ++w)
        if (w < wid) woff += warp_tot[w];
    uint32_t off = sums[blockIdx.x] + woff + inc - s;
    if (base + SCAN_ITEMS <= n) {
        uint4 *p = reinterpret_cast<uint4 *>(out + base);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            p[j] = make_uint4(v[4 * j] + off, v[4 * j + 1] + off, v[4 * j + 2] + off, v[4 * j + 3] + off);
    } else {
#pragma unroll
        for (int j = 0; j < SCAN_ITEMS; ++j)
            if (base + j < n) out[base + j] = v[j] + off;
    }
}

// Short inputs (a few 1e4 flags): ONE CTA walks the array in strips of 16 384 elements,
// next strip's loads in flight while this one is scanned. Three launches of a few microseconds each become one.
constexpr int64_t SCAN_ONE_MAX = (int64_t)1 << 15;   // beyond two strips one SM is slower than three launches (measured: 48 us at 250 000)
template <typename T>
__global__ void __launch_bounds__(1024) scan_one_kernel(const T *in, uint32_t *out, int64_t n, uint32_t *total) {   // in may be out
    __shared__ uint32_t warp_tot[32];
    __shared__ uint32_t strip_tot;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    constexpr int64_t STRIP = 1024 * SCAN_ITEMS;
    uint32_t carry = 0;
    uint32_t v[SCAN_ITEMS], nxt[SCAN_ITEMS];
    load_items(in, (int64_t)threadIdx.x * SCAN_ITEMS, n, v);
    for (int64_t strip = 0; strip < n; strip += STRIP) {
        const int64_t base = strip + (int64_t)threadIdx.x * SCAN_ITEMS;
        if (strip + STRIP < n) load_items(in, base + STRIP, n, nxt);
        uint32_t s = 0;
#pragma unroll
        for (int j = 0; j < SCAN_ITEMS; ++j) {
            const uint32_t t = v[j];
            v[j] = s;
            s += t;
        }
        uint32_t inc = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        if (lane == 31) warp_tot[wid] = inc;
        __syncthreads();
        if (wid == 0) {
            const uint32_t t = warp_tot[lane];
            uint32_t ti = t;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, ti, o);
                if (lane >= o) ti += y;
            }
            warp_tot[lane] = ti - t;   // exclusive warp offsets
            if (lane == 31) strip_tot = ti;
        }
        __syncthreads();
        const uint32_t off = carry + warp_tot[wid] + inc - s;
        carry += strip_tot;
        if (base + SCAN_ITEMS <= n) {
            uint4 *p = reinterpret_cast<uint4 *>(out + base);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                p[j] = make_uint4(v[4 * j] + off, v[4 * j + 1] + off, v[4 * j + 2] + off, v[4 * j + 3] + off);
        } else {
#pragma unroll
            for (int j = 0; j < SCAN_ITEMS; ++j)
                if (base + j < n) out[base + j] = v[j] + off;
        }
        __syncthreads();   // warp_tot / strip_tot are rewritten by the next strip
#pragma unroll
        for (int j = 0; j < SCAN_ITEMS; ++j) v[j] = nxt[j];
    }
    if (threadIdx.x == 0 && total != nullptr) *total = carry;
}

size_t scan_scratch_elems(int64_t n) { return (size_t)((n + SCAN_TILE - 1) / SCAN_TILE) + 64; }

template <typename T>
static int scan_impl(const T *in, uint32_t *out, int64_t n, uint32_t *total, uint32_t *scratch, cudaStream_t st) {
    if (n <= 0) {
        if (total) SYM_CUDA_OK(cudaMemsetAsync(total, 0, sizeof(uint32_t), st));
        return SYM_OK;
    }
    if (n <= SCAN_ONE_MAX) {
        scan_one_kernel<T><<<1, 1024, 0, st>>>(in, out, n, total);
        SYM_LAUNCH_OK();
        return SYM_OK;
    }
    int64_t nb = (n + SCAN_TILE - 1) / SCAN_TILE;
    scan_reduce_kernel<T><<<(unsigned)nb, SCAN_THREADS, 0, st>>>(in, n, scratch);
    SYM_LAUNCH_OK();
    scan_sums_kernel<<<1, 1024, 0, st>>>(scratch, nb, total);
    SYM_LAUNCH_OK();
    scan_apply_kernel<T><<<(unsigned)nb, SCAN_THREADS, 0, st>>>(in, out, n, scratch);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

int scan_exclusive_u8(const uint8_t *in, uint32_t *out, int64_t n, uint32_t *total, uint32_t *scratch, cudaStream_t st) {
    return scan_impl<uint8_t>(in, out, n, total, scratch, st);
}
int scan_exclusive_u32(const uint32_t *in, uint32_t *out, int64_t n, uint32_t *total, uint32_t *scratch, cudaStream_t st) {
    return scan_impl<uint32_t>(in, out, n, total, scratch, st);
}

}  // namespace symb

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
using namespace symb;

extern "C" size_t sym_sort_pairs_ws_bytes(int64_t T) {
    if (T < 1) T = 1;
    return arena_need((size_t)T, 8) + arena_need((size_t)T, 4) + arena_need(record_hist_elems(T), 4) + 1024;
}

extern "C" int sym_sort_pairs(uint64_t *keys, uint32_t *vals, int64_t T, int32_t begin_bit, void *ws, size_t ws_bytes,
                              void *stream) {
    SYM_REQUIRE(T >= 0 && T < (int64_t)4000000000LL, "T out of range");
    if (T == 0) return SYM_OK;
    if (ws_bytes < sym_sort_pairs_ws_bytes(T)) {
        set_error("workspace too small");
        return SYM_E_WORKSPACE;
    }
    Arena ar(ws, ws_bytes);
    uint64_t *ka = ar.take<uint64_t>((size_t)T);
    uint32_t *va = ar.take<uint32_t>((size_t)T);
    uint32_t *hist = ar.take<uint32_t>(record_hist_elems(T));
    cudaStream_t st = (cudaStream_t)stream;
    uint64_t *sorted = keys;
    SYM_TRY(radix_sort(keys, vals, ka, va, T, begin_bit, hist, &sorted, st));
    if (sorted != keys) {   // an odd number of passes ends in the workspace
        SYM_CUDA_OK(cudaMemcpyAsync(keys, ka, sizeof(uint64_t) * (size_t)T, cudaMemcpyDeviceToDevice, st));
        SYM_CUDA_OK(cudaMemcpyAsync(vals, va, sizeof(uint32_t) * (size_t)T, cudaMemcpyDeviceToDevice, st));
    }
    return SYM_OK;
}
