// Stable LSD radix sort of 64-bit keys, each optionally carrying a 32-bit value. It is the only radix sort
// of the library: the dedup hot path sorts its records (hash | t | phase) with it, and the pair sort
// (sym_sort_pairs) and the owner-class partition sort (key, value) pairs with it.
// Per pass: (1) per-tile digit histogram, (2) exclusive scan of the digit-major histogram,
// (3) scatter: rank inside the tile with ballots, stage the tile in shared memory in digit order,
// then store — consecutive threads write consecutive addresses within a digit run.
// HBM-bound: 8 B read (hist) + 8 B read + 8 B write (scatter) per key per pass, plus 4 B + 4 B per value.
#include <algorithm>

#include "sort.cuh"

namespace symb {

constexpr int RS_THREADS = 256;
constexpr int RS_ITEMS = 16;
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;  // 4096 records
constexpr int RS_RADIX = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_MIN_BLOCKS = 4;   // CTAs per SM of the scatter passes: 256 threads x 16 records, 4 CTAs/SM measured best
// shared memory of a scatter tile: staged keys, per-warp digit counts, dbase, delta, wtot, the one-sweep ticket;
// with values, the staged values follow
constexpr size_t RS_SMEM_KEYS = RS_TILE * 8 + RS_WARPS * RS_RADIX * 4 + 2 * RS_RADIX * 4 + 32 * 4 + 64;
constexpr size_t rs_smem_bytes(bool vals) { return RS_SMEM_KEYS + (vals ? RS_TILE * 4 : 0); }
// With values, their staging area costs the 4th CTA per SM. Measured on a B200 (1000 W), 1e8 pairs sort in
// 7.6 ms this way against 8.5 ms at 4 CTAs/SM with the values staged through the key area in a second phase.
constexpr int rs_min_blocks(bool vals) { return vals ? 3 : RS_MIN_BLOCKS; }

__global__ void __launch_bounds__(RS_THREADS) rs_hist_kernel(const uint64_t *__restrict__ in, int64_t T, int shift,
                                                              uint32_t mask, uint32_t *__restrict__ hist, int64_t ntiles) {
    __shared__ uint32_t h[RS_RADIX];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * RS_TILE;
#pragma unroll
    for (int j = 0; j < RS_ITEMS; ++j) {
        int64_t idx = base + j * RS_THREADS + threadIdx.x;
        if (idx < T) atomicAdd(&h[(uint32_t)(in[idx] >> shift) & mask], 1u);
    }
    __syncthreads();
    hist[(int64_t)threadIdx.x * ntiles + blockIdx.x] = h[threadIdx.x];
}

// ---------------------------------------------------------------------------------------------
// Ranking and staging of one tile, shared by the scatter kernel and the one-sweep pass kernel.
// Thread d = threadIdx.x handles digit d in the per-digit steps (RS_THREADS == RS_RADIX).
// ---------------------------------------------------------------------------------------------
// the thread's index and the shared-memory layout of its CTA's tile
struct Tile {
    int tid;
    uint64_t *srec;
    uint32_t (*wh)[RS_RADIX];
    uint32_t *dbase, *delta, *wtot;
    uint32_t *sval;
    // tid is read in the kernel, where the compiler knows that it is below RS_THREADS; read in the helpers it
    // would not be, and the record kernels would compile to more spills
    __device__ Tile(unsigned char *p, int tid)
        : tid(tid),
          srec(reinterpret_cast<uint64_t *>(p)),
          wh(reinterpret_cast<uint32_t(*)[RS_RADIX]>(p + RS_TILE * 8)),
          dbase(reinterpret_cast<uint32_t *>(p + RS_TILE * 8 + RS_WARPS * RS_RADIX * 4)),
          delta(dbase + RS_RADIX),
          wtot(delta + RS_RADIX),
          sval(reinterpret_cast<uint32_t *>(p + RS_SMEM_KEYS)) {}
};

// Loads the tile's keys (and values) and ranks every key stably among the keys of its digit in its warp;
// wh[w][d] must be zero on entry. Then per digit d: wh[w][d] becomes the offset of warp w among the tile's
// keys of digit d, publish(d, tile count of d) runs, and the returned exclusive scan over digits (also left
// in dbase[d]) is where the staged run of digit d starts. Ranks are < 4096 and are kept as 16-bit halves to
// save registers. Ends without a barrier: dbase is read by other threads only after the caller's next one.
template <bool VALS, typename Publish>
__device__ __forceinline__ uint32_t rank_tile(const uint64_t *in, const uint32_t *vin, int64_t T, int64_t tile_base,
                                              int shift, uint32_t mask, const Tile &s, uint64_t (&k)[RS_ITEMS],
                                              uint32_t (&v)[VALS ? RS_ITEMS : 1], uint16_t (&r)[RS_ITEMS],
                                              Publish publish) {
    const int lane = s.tid & 31, wid = s.tid >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    const int64_t wbase = tile_base + (int64_t)wid * (32 * RS_ITEMS);
#pragma unroll
    for (int j = 0; j < RS_ITEMS; ++j) {
        int64_t idx = wbase + j * 32 + lane;
        k[j] = (idx < T) ? in[idx] : 0ull;
        if constexpr (VALS) v[j] = (idx < T) ? vin[idx] : 0u;
    }
#pragma unroll
    for (int j = 0; j < RS_ITEMS; ++j) {
        int64_t idx = wbase + j * 32 + lane;
        bool valid = idx < T;
        uint32_t d = valid ? ((uint32_t)(k[j] >> shift) & mask) : 0xffffffffu;
        // lanes holding the same digit, built from 8 ballots (match.any is far slower on sm_100)
        uint32_t peers = __ballot_sync(0xffffffffu, valid);
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const bool bit = (d >> b) & 1u;
            const uint32_t bal = __ballot_sync(0xffffffffu, bit);
            peers &= bit ? bal : ~bal;
        }
        uint32_t before = valid ? s.wh[wid][d] : 0u;
        r[j] = (uint16_t)(before + __popc(peers & lt));
        __syncwarp();
        if (valid && lane == (__ffs(peers) - 1)) s.wh[wid][d] = before + __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    // per digit: exclusive offsets of the warps, tile total, then a block scan over the 256 totals
    const int d = s.tid;
    uint32_t cnt = 0;
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) {
        uint32_t c = s.wh[w][d];
        s.wh[w][d] = cnt;
        cnt += c;
    }
    publish(d, cnt);
    uint32_t inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) s.wtot[wid] = inc;
    s.dbase[d] = inc - cnt;   // exclusive inside the warp; warp offset added below
    __syncthreads();
    uint32_t woff = 0;
#pragma unroll
    for (int w = 0; w < RS_RADIX / 32; ++w)
        if (w < wid) woff += s.wtot[w];
    const uint32_t excl = s.dbase[d] + woff;
    s.dbase[d] = excl;
    return excl;
}

// Writes the ranked keys (and values) to shared memory in digit order.
template <bool VALS>
__device__ __forceinline__ void stage_tile(int64_t T, int64_t tile_base, int shift, uint32_t mask, const Tile &s,
                                           const uint64_t (&k)[RS_ITEMS], const uint32_t (&v)[VALS ? RS_ITEMS : 1],
                                           const uint16_t (&r)[RS_ITEMS]) {
    const int lane = s.tid & 31, wid = s.tid >> 5;
    const int64_t wbase = tile_base + (int64_t)wid * (32 * RS_ITEMS);
#pragma unroll
    for (int j = 0; j < RS_ITEMS; ++j) {
        int64_t idx = wbase + j * 32 + lane;
        if (idx < T) {
            uint32_t d = (uint32_t)(k[j] >> shift) & mask;
            const uint32_t p = s.dbase[d] + s.wh[wid][d] + r[j];
            s.srec[p] = k[j];
            if constexpr (VALS) s.sval[p] = v[j];
        }
    }
}

// Stores the staged tile: staged position pos of digit d goes to delta[d] + pos.
template <bool VALS>
__device__ __forceinline__ void store_tile(uint64_t *out, uint32_t *vout, int64_t T, int64_t tile_base, int shift,
                                           uint32_t mask, const Tile &s) {
    const int64_t remain = T - tile_base;
    const int count = remain < RS_TILE ? (int)remain : RS_TILE;
#pragma unroll
    for (int j = 0; j < RS_ITEMS; ++j) {
        int pos = j * RS_THREADS + s.tid;
        if (pos < count) {
            uint64_t rec = s.srec[pos];
            uint32_t d = (uint32_t)(rec >> shift) & mask;
            out[(size_t)(s.delta[d] + (uint32_t)pos)] = rec;
            if constexpr (VALS) vout[(size_t)(s.delta[d] + (uint32_t)pos)] = s.sval[pos];
        }
    }
}

template <bool VALS>
__global__ void __launch_bounds__(RS_THREADS, rs_min_blocks(VALS))
    rs_scatter_kernel(const uint64_t *__restrict__ in, const uint32_t *__restrict__ vin, uint64_t *__restrict__ out,
                      uint32_t *__restrict__ vout, int64_t T, int shift, uint32_t mask,
                      const uint32_t *__restrict__ hist, int64_t ntiles) {
    static_assert(RS_THREADS == RS_RADIX, "one thread per digit");
    extern __shared__ __align__(16) unsigned char rs_smem[];
    const Tile s(rs_smem, threadIdx.x);
    for (int i = threadIdx.x; i < RS_WARPS * RS_RADIX; i += RS_THREADS) (&s.wh[0][0])[i] = 0;
    __syncthreads();
    const int64_t tile_base = (int64_t)blockIdx.x * RS_TILE;
    uint64_t k[RS_ITEMS];
    uint32_t vals[VALS ? RS_ITEMS : 1];
    uint16_t r[RS_ITEMS];
    const uint32_t excl = rank_tile<VALS>(in, vin, T, tile_base, shift, mask, s, k, vals, r, [](int, uint32_t) {});
    s.delta[threadIdx.x] = hist[(int64_t)threadIdx.x * ntiles + blockIdx.x] - excl;
    __syncthreads();
    stage_tile<VALS>(T, tile_base, shift, mask, s, k, vals, r);
    __syncthreads();
    store_tile<VALS>(out, vout, T, tile_base, shift, mask, s);
}

__global__ void rs_part_counts_kernel(const uint32_t *__restrict__ scanned, int64_t ntiles, int nb, int64_t T,
                                      int64_t *__restrict__ counts) {
    int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d < nb) {
        int64_t lo = scanned[(int64_t)d * ntiles];
        // buckets >= nb are empty, so scanned[(d+1)*ntiles] == T for d == nb-1 as well
        int64_t hi = (d + 1 < RS_RADIX) ? (int64_t)scanned[(int64_t)(d + 1) * ntiles] : T;
        counts[d] = hi - lo;
    }
}

// ---------------------------------------------------------------------------------------------
// One-sweep form (tuning knob 8, default): ONE kernel builds the digit histograms of every pass
// (the keys never change, only their order), then each pass is a single kernel — a tile learns its
// global offsets from the tiles before it by decoupled look-back instead of from a per-pass
// histogram + scan. Per pass 16 B/record of HBM traffic instead of 24 B and two launches fewer.
// Tiles take their index from a ticket counter, so every tile a CTA waits for is already running.
// ---------------------------------------------------------------------------------------------
constexpr int OS_MAX_PASSES = 8;
constexpr int OS_EXTRA_ELEMS = OS_MAX_PASSES * RS_RADIX * 2 + 64;   // global counts + bases + tickets

// histograms of all passes in one read of the keys; grid-stride over tiles
__global__ void __launch_bounds__(RS_THREADS) os_hist_kernel(const uint64_t *in, int64_t T, int begin_bit, int passes,
                                                              int64_t ntiles, uint32_t *__restrict__ counts) {
    __shared__ uint32_t h[OS_MAX_PASSES][RS_RADIX];
    for (int i = threadIdx.x; i < OS_MAX_PASSES * RS_RADIX; i += RS_THREADS) (&h[0][0])[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        uint64_t k[RS_ITEMS];
        const int64_t first = tile * RS_TILE + (int64_t)wid * (32 * RS_ITEMS) + lane;
#pragma unroll
        for (int j = 0; j < RS_ITEMS; ++j) k[j] = first + j * 32 < T ? in[first + j * 32] : 0ull;
#pragma unroll
        for (int j = 0; j < RS_ITEMS; ++j) {
            if (first + j * 32 < T) {
                for (int ps = 0; ps < passes; ++ps) {
                    const int bit = begin_bit + 8 * ps;
                    atomicAdd(&h[ps][(uint32_t)(k[j] >> bit) & 0xffu], 1u);
                }
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < passes * RS_RADIX; i += RS_THREADS) {
        const uint32_t v = (&h[0][0])[i];
        if (v) atomicAdd(counts + i, v);
    }
}

// per pass: exclusive scan of the 256 digit counts -> bases[pass][digit]; one block of 256 threads per pass
__global__ void __launch_bounds__(RS_RADIX) os_bases_kernel(const uint32_t *__restrict__ counts, uint32_t *__restrict__ bases) {
    __shared__ uint32_t wt[RS_RADIX / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t c = counts[blockIdx.x * RS_RADIX + threadIdx.x];
    uint32_t inc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) wt[wid] = inc;
    __syncthreads();
    uint32_t woff = 0;
    for (int w = 0; w < wid; ++w) woff += wt[w];
    bases[blockIdx.x * RS_RADIX + threadIdx.x] = woff + inc - c;
}

__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_volatile_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// One radix pass. state[tile][digit]: bits 31:30 = 0 not published / 1 tile count / 2 inclusive
// prefix over tiles 0..tile; bits 29:0 = value (T < 2^30 on this path).
template <bool VALS>
__global__ void __launch_bounds__(RS_THREADS, rs_min_blocks(VALS))
    os_pass_kernel(const uint64_t *in, const uint32_t *vin, uint64_t *__restrict__ out, uint32_t *__restrict__ vout,
                   int64_t T, int shift, uint32_t mask, const uint32_t *__restrict__ bases,
                   uint32_t *__restrict__ state, uint32_t *__restrict__ ticket) {
    static_assert(RS_THREADS == RS_RADIX, "one look-back thread per digit");
    extern __shared__ __align__(16) unsigned char rs_smem[];
    const Tile s(rs_smem, threadIdx.x);
    uint32_t *s_tile = s.wtot + 32;
    for (int i = threadIdx.x; i < RS_WARPS * RS_RADIX; i += RS_THREADS) (&s.wh[0][0])[i] = 0;
    if (threadIdx.x == 0) *s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = *s_tile;
    const int64_t tile_base = (int64_t)tile * RS_TILE;
    uint64_t k[RS_ITEMS];
    uint32_t vals[VALS ? RS_ITEMS : 1];
    uint16_t r[RS_ITEMS];
    uint32_t cnt = 0;
    // publish the tile count as early as possible: the tiles after this one are waiting for it
    const uint32_t excl_d = rank_tile<VALS>(in, vin, T, tile_base, shift, mask, s, k, vals, r, [&](int d, uint32_t c) {
        cnt = c;
        st_volatile_u32(state + (size_t)tile * RS_RADIX + d, (tile == 0 ? 0x80000000u : 0x40000000u) | c);
    });
    __syncthreads();
    // stage the tile in digit order first: it needs no global offsets, and the tiles this one is about to
    // wait for get that much closer to publishing theirs
    stage_tile<VALS>(T, tile_base, shift, mask, s, k, vals, r);
    {
        const int d = threadIdx.x;
        // decoupled look-back over the tiles before this one, four state words in flight per step
        uint32_t prev = 0;
        if (tile > 0) {
            int64_t t = (int64_t)tile - 1;
            bool done = false;
            while (!done) {
                uint32_t v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) v[u] = (t - u >= 0) ? ld_volatile_u32(state + (size_t)(t - u) * RS_RADIX + d) : 0x80000000u;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (done) break;
                    uint32_t x = v[u], spins = 0;
                    while ((x >> 30) == 0u) {
                        if (++spins > (1u << 22)) __trap();   // a predecessor never published: fail loudly, never hang
                        x = ld_volatile_u32(state + (size_t)(t - u) * RS_RADIX + d);
                    }
                    prev += x & 0x3fffffffu;
                    done = (x >> 30) == 2u;
                }
                t -= 4;
            }
            st_volatile_u32(state + (size_t)tile * RS_RADIX + d, 0x80000000u | (prev + cnt));
        }
        s.delta[d] = bases[d] + prev - excl_d;
    }
    __syncthreads();
    store_tile<VALS>(out, vout, T, tile_base, shift, mask, s);
}

int g_onesweep = 1;   // tuning knob 8

// Short sorts keep one look-back state array PER PASS, so that a single memset clears them all (and the pass
// counters behind them) instead of one memset in front of every pass: on a 250 000-record sort the passes take
// 10 us each and every extra stream operation costs 3-4 us of launch gap.
constexpr int64_t OS_MULTI_STATE_TILES = 1024;
static inline int os_state_copies(int64_t ntiles) { return ntiles <= OS_MULTI_STATE_TILES ? OS_MAX_PASSES : 1; }

size_t record_hist_elems(int64_t T) {
    int64_t ntiles = (T + RS_TILE - 1) / RS_TILE;
    if (ntiles < 1) ntiles = 1;
    size_t h = (size_t)RS_RADIX * (size_t)ntiles;
    return h * (size_t)os_state_copies(ntiles) + scan_scratch_elems((int64_t)h) + 64 + OS_EXTRA_ELEMS;
}

template <bool VALS>
static int os_launch_pass(const uint64_t *in, const uint32_t *vin, uint64_t *out, uint32_t *vout, int64_t T, int shift,
                          uint32_t mask, const uint32_t *bases, uint32_t *state, uint32_t *ticket, int64_t ntiles,
                          cudaStream_t st, bool clear_state) {
    constexpr size_t smem = rs_smem_bytes(VALS);
    static bool attr_done[64] = {};   // per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !attr_done[dev]) {
        SYM_CUDA_OK(cudaFuncSetAttribute(os_pass_kernel<VALS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev] = true;
    }
    if (clear_state) SYM_CUDA_OK(cudaMemsetAsync(state, 0, sizeof(uint32_t) * (size_t)RS_RADIX * (size_t)ntiles, st));
    os_pass_kernel<VALS><<<(unsigned)ntiles, RS_THREADS, smem, st>>>(in, vin, out, vout, T, shift, mask, bases, state, ticket);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

template <bool VALS>
static int rs_pass(const uint64_t *in, const uint32_t *vin, uint64_t *out, uint32_t *vout, int64_t T, int shift,
                   uint32_t mask, uint32_t *hist, cudaStream_t st) {
    int64_t ntiles = (T + RS_TILE - 1) / RS_TILE;
    int64_t hn = (int64_t)RS_RADIX * ntiles;
    uint32_t *scratch = hist + hn;
    rs_hist_kernel<<<(unsigned)ntiles, RS_THREADS, 0, st>>>(in, T, shift, mask, hist, ntiles);
    SYM_LAUNCH_OK();
    SYM_TRY(scan_exclusive_u32(hist, hist, hn, nullptr, scratch, st));
    constexpr size_t smem = rs_smem_bytes(VALS);
    static bool attr_done[64] = {};   // per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !attr_done[dev]) {
        SYM_CUDA_OK(cudaFuncSetAttribute(rs_scatter_kernel<VALS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev] = true;
    }
    rs_scatter_kernel<VALS><<<(unsigned)ntiles, RS_THREADS, smem, st>>>(in, vin, out, vout, T, shift, mask, hist, ntiles);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

// Passes ping-pong (keys, vals) <-> (alt, vals_alt); pass 0 reads keys. One-sweep passes while knob 8 is set
// and the look-back states can hold the counts (T < 2^30), the histogram + scan + scatter form otherwise.
template <bool VALS>
static int sort_passes(uint64_t *a, uint32_t *va, uint64_t *b, uint32_t *vb, int64_t T, int begin_bit, uint32_t *hist,
                       uint64_t **result, cudaStream_t st) {
    const bool onesweep = g_onesweep && T < ((int64_t)1 << 30);
    const int passes = (64 - begin_bit + 7) / 8;
    const int64_t ntiles = (T + RS_TILE - 1) / RS_TILE;
    uint32_t *state = hist;
    const size_t h = (size_t)RS_RADIX * (size_t)ntiles;
    const int copies = os_state_copies(ntiles);
    uint32_t *extra = hist + h * (size_t)copies + scan_scratch_elems((int64_t)h) + 64;
    uint32_t *counts = extra, *bases = extra + OS_MAX_PASSES * RS_RADIX, *tickets = bases + OS_MAX_PASSES * RS_RADIX;
    if (onesweep) {
        if (copies > 1)   // every pass's state, the (unused) scan scratch between, and the counters: one memset
            SYM_CUDA_OK(cudaMemsetAsync(hist, 0, sizeof(uint32_t) * ((size_t)(extra - hist) + OS_EXTRA_ELEMS), st));
        else
            SYM_CUDA_OK(cudaMemsetAsync(extra, 0, sizeof(uint32_t) * OS_EXTRA_ELEMS, st));
        const unsigned hgrid = (unsigned)std::min<int64_t>(ntiles, (int64_t)num_sms() * 8);
        os_hist_kernel<<<hgrid, RS_THREADS, 0, st>>>(a, T, begin_bit, passes, ntiles, counts);
        SYM_LAUNCH_OK();
        os_bases_kernel<<<passes, RS_RADIX, 0, st>>>(counts, bases);
        SYM_LAUNCH_OK();
    }
    int bit = begin_bit;
    for (int ps = 0; ps < passes; ++ps) {
        const int width = (64 - bit) < 8 ? (64 - bit) : 8;
        const uint32_t mask = (1u << width) - 1u;
        if (onesweep) {
            uint32_t *state_ps = copies > 1 ? state + (size_t)ps * h : state;
            SYM_TRY(os_launch_pass<VALS>(a, va, b, vb, T, bit, mask, bases + ps * RS_RADIX, state_ps, tickets + ps, ntiles,
                                         st, copies == 1));
        } else {
            SYM_TRY(rs_pass<VALS>(a, va, b, vb, T, bit, mask, hist, st));
        }
        uint64_t *t = a; a = b; b = t;
        uint32_t *tv = va; va = vb; vb = tv;
        bit += width;
    }
    *result = a;
    return SYM_OK;
}

int radix_sort(uint64_t *keys, uint32_t *vals, uint64_t *alt, uint32_t *vals_alt, int64_t T, int begin_bit,
               uint32_t *hist, uint64_t **result, cudaStream_t st) {
    *result = keys;
    if (T <= 1) return SYM_OK;
    if (begin_bit < 0) begin_bit = 0;
    if (begin_bit > 63) begin_bit = 63;
    return vals ? sort_passes<true>(keys, vals, alt, vals_alt, T, begin_bit, hist, result, st)
                : sort_passes<false>(keys, nullptr, alt, nullptr, T, begin_bit, hist, result, st);
}

int radix_partition(const uint64_t *keys, const uint32_t *vals, uint64_t *out, uint32_t *out_vals, int64_t T, int bits,
                    int64_t *counts, uint32_t *hist, cudaStream_t st) {
    const int nb = 1 << bits;
    if (T <= 0) {
        SYM_CUDA_OK(cudaMemsetAsync(counts, 0, sizeof(int64_t) * nb, st));
        return SYM_OK;
    }
    if (bits == 0) {
        SYM_CUDA_OK(cudaMemcpyAsync(out, keys, sizeof(uint64_t) * (size_t)T, cudaMemcpyDeviceToDevice, st));
        if (vals) SYM_CUDA_OK(cudaMemcpyAsync(out_vals, vals, sizeof(uint32_t) * (size_t)T, cudaMemcpyDeviceToDevice, st));
        int64_t t = T;
        SYM_CUDA_OK(cudaMemcpyAsync(counts, &t, sizeof(int64_t), cudaMemcpyHostToDevice, st));
        SYM_CUDA_OK(cudaStreamSynchronize(st));
        return SYM_OK;
    }
    if (vals)
        SYM_TRY(rs_pass<true>(keys, vals, out, out_vals, T, 64 - bits, (1u << bits) - 1u, hist, st));
    else
        SYM_TRY(rs_pass<false>(keys, nullptr, out, nullptr, T, 64 - bits, (1u << bits) - 1u, hist, st));
    int64_t ntiles = (T + RS_TILE - 1) / RS_TILE;
    rs_part_counts_kernel<<<1, 256, 0, st>>>(hist, ntiles, nb, T, counts);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

}  // namespace symb
