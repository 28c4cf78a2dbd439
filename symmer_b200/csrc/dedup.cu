// Dedup of terms by hashed 64-bit records with exact row verification, segmented coefficient
// reduction in input order, threshold filter and row emission. Replaces qiskit's `unordered_unique`
// + `np.add.at` (symmer/operators/utils.py:271-278) — HBM-bound integer/byte work, no tensor cores.
//
// Pipeline (all on one stream):
//   1. stable LSD radix sort of the records on their top hash bits -> equal rows become neighbours,
//      ordered by t inside a run
//   2. link: every sorted position finds its nearest earlier twin inside its sort bucket (exact row compare)
//   3. sum: each head adds the coefficients of its group in input (t) order and applies |c| > thr
//   4. exclusive scan of keep flags -> output slots ; compact ; emit rows with 16-byte stores
#include <algorithm>
#include <type_traits>

#include "rows.cuh"
#include "sort.cuh"

namespace symb {

constexpr uint8_t FLAG_HEAD = 0, FLAG_PREV = 1, FLAG_LINK = 2;

// A "bucket" is a maximal run of sorted records sharing the sorted hash prefix (bits >= sort_shift).
// The sort leaves each bucket in input (t) order. On average a bucket holds <= 8 records
// (sort_begin_bit), so the scans below are a handful of cached 8-byte reads per record.
//
// link: every sorted position finds the nearest EARLIER record of its bucket with the same row
// (full hash match, then exact word-by-word compare): none -> HEAD, the immediate predecessor ->
// PREV, further back -> LINK (position stored in link[]).
template <class Rows>
__device__ __forceinline__ void link_one(const Rows &rows, const RecFmt &fmt, const uint64_t *__restrict__ sr, int64_t i,
                                         int sort_shift, uint8_t *__restrict__ flag, uint32_t *__restrict__ link,
                                         int64_t lo = 0) {
    uint8_t f = FLAG_HEAD;
    if (i > lo) {
        const uint64_t ri = sr[i];
        const uint32_t ti = fmt.t(ri);
        for (int64_t j = i - 1; j >= lo; --j) {
            const uint64_t rj = sr[j];
            if (((ri ^ rj) >> sort_shift) != 0) break;   // left the bucket
            if (fmt.same_hash(ri, rj) && rows.equal(ti, fmt.t(rj))) {
                if (j == i - 1) {
                    f = FLAG_PREV;
                } else {
                    f = FLAG_LINK;
                    link[i] = (uint32_t)j;
                }
                break;
            }
        }
    }
    flag[i] = f;
}

// Thread per sorted record; the exact row compares are done by the warp, 8 lanes per pair with 16-byte loads.
// A thread comparing two rows alone touches a new 32-byte sector with every load, and a product with many true
// duplicates (A*A: every P_i P_j meets P_j P_i) then sits on the L1 wavefront rate: 40 us for the 250 000 cross
// terms of config C1, against 3 us without duplicates. Eight lanes read 128 contiguous bytes of each row.
template <class Rows>
__global__ void __launch_bounds__(256) link_kernel(Rows rows, RecFmt fmt, const uint64_t *__restrict__ sr, int64_t T,
                                                    int sort_shift, uint8_t *__restrict__ flag, uint32_t *__restrict__ link) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, g = lane & 7, grp = lane >> 3;
    const bool valid = i < T;
    // nearest earlier record of the bucket with the same full hash: the candidate
    int64_t j = -1;
    uint64_t ri = 0;
    uint32_t ti = 0, tj = 0;
    if (valid && i > 0) {
        ri = sr[i];
        ti = fmt.t(ri);
        for (int64_t jj = i - 1; jj >= 0; --jj) {
            const uint64_t rj = sr[jj];
            if (((ri ^ rj) >> sort_shift) != 0) break;   // left the bucket
            if (fmt.same_hash(ri, rj)) {
                j = jj;
                tj = fmt.t(rj);
                break;
            }
        }
    }
    bool eq = false;
    const int chunks = rows.words >> 1;
    for (uint32_t pend = __ballot_sync(0xffffffffu, j >= 0); pend;) {   // uniform: four candidates per step
        int src[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            src[k] = pend ? __ffs(pend) - 1 : -1;
            pend &= pend - 1u;   // 0 stays 0
        }
        const int mine = src[grp];
        const uint32_t t1 = __shfl_sync(0xffffffffu, ti, mine < 0 ? 0 : mine);
        const uint32_t t2 = __shfl_sync(0xffffffffu, tj, mine < 0 ? 0 : mine);
        bool same = true;
        if (mine >= 0) {
            const uint2 h1 = rows.locate(t1), h2 = rows.locate(t2);
            for (int c = g; c < chunks; c += 8) {
                const uint4 a = rows.chunk_at(h1, c), b = rows.chunk_at(h2, c);
                same &= !((a.x != b.x) | (a.y != b.y) | (a.z != b.z) | (a.w != b.w));
            }
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, same);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (lane == src[k]) eq = ((bal >> (8 * k)) & 0xffu) == 0xffu;
    }
    if (!valid) return;
    uint8_t f = FLAG_HEAD;
    if (j >= 0) {
        if (!eq) {   // same hash, different row (2^-40 per pair): go on alone from the record before the candidate
            int64_t jj = j - 1;
            j = -1;
            for (; jj >= 0; --jj) {
                const uint64_t rj = sr[jj];
                if (((ri ^ rj) >> sort_shift) != 0) break;
                if (fmt.same_hash(ri, rj) && rows.equal(ti, fmt.t(rj))) {
                    j = jj;
                    break;
                }
            }
        }
        if (j >= 0) {
            if (j == i - 1) {
                f = FLAG_PREV;
            } else {
                f = FLAG_LINK;
                link[i] = (uint32_t)j;
            }
        }
    }
    flag[i] = f;
}

// Worklist of sorted positions (ordered-tile mode: only the records of non-singleton buckets), kept as
// `nreg` regions of `cap` entries with one counter each: CTA b of the classify pass appends to region
// b % nreg, so no counter is hot (one global counter serialises ~2e6 same-address atomics: 1.5 ms)
// and a region can never overflow (it receives from at most cap records).
// Identity form (class mode, work == nullptr): every position of [begin, end) is on the list; begin and end live
// in device memory (the host never learns them before the launch); region r covers positions
// begin + [r * cap, (r + 1) * cap). begin_ptr / end_ptr also bound the record array for a stored list.
struct WorkList {
    uint32_t *work;
    uint32_t *counts;
    uint32_t nreg, cap;
    const uint32_t *begin_ptr = nullptr;
    const uint32_t *end_ptr = nullptr;
    __device__ __forceinline__ uint32_t begin() const { return begin_ptr ? *begin_ptr : 0u; }
    __device__ __forceinline__ uint32_t region_count(uint32_t r) const {
        if (work) return counts[r];
        const uint32_t b = begin(), e = *end_ptr;
        const uint32_t n = e > b ? e - b : 0u;
        const uint64_t lo = (uint64_t)r * cap;
        return n > lo ? (uint32_t)(n - lo < cap ? n - lo : cap) : 0u;
    }
    __device__ __forceinline__ uint32_t entry(uint32_t r, uint32_t k) const {
        return work ? work[(size_t)r * cap + k] : begin() + r * cap + k;
    }
    // bounds of the record array the listed positions refer to
    __device__ __forceinline__ int64_t lo() const { return (int64_t)begin(); }
    __device__ __forceinline__ int64_t hi(int64_t T) const { return end_ptr ? (int64_t)*end_ptr : T; }
};
// consumers: WORK_SPLIT CTAs per region (grid = nreg * WORK_SPLIT), each striding over the region's entries
constexpr uint32_t WORK_SPLIT = 8;
#define FOR_EACH_WORK(wl, i)                                                                                     \
    for (uint32_t _r = blockIdx.x / WORK_SPLIT, _k = (blockIdx.x % WORK_SPLIT) * blockDim.x + threadIdx.x,       \
                  _n = (wl).region_count(_r);                                                                    \
         _k < _n; _k += WORK_SPLIT * blockDim.x)                                                                 \
        if (const uint32_t i = (wl).entry(_r, _k); true)

template <class Rows>
__global__ void __launch_bounds__(256) link_work_kernel(Rows rows, RecFmt fmt, const uint64_t *__restrict__ sr, int sort_shift,
                                                         WorkList wl, uint8_t *__restrict__ flag, uint32_t *__restrict__ link) {
    const int64_t lo = wl.lo();
    FOR_EACH_WORK(wl, i) link_one(rows, fmt, sr, (int64_t)i, sort_shift, flag, link, lo);
}

__device__ __forceinline__ int64_t chain_root(const uint8_t *flag, const uint32_t *link, int64_t i) {
    while (flag[i] != FLAG_HEAD) i = (flag[i] == FLAG_PREV) ? i - 1 : (int64_t)link[i];
    return i;
}

// sum: each HEAD walks forward through its bucket and adds the coefficients of the records whose
// chain leads back to it, in input (t) order like np.add.at — deterministic, no atomics.
// TILE (ordered-tile mode, see rows.cuh): nothing is written for a record that survives as a
// singleton; a record that does not survive sets its drop bit, and a surviving group head leaves
// its sum in acc[i] with multi[i] = 1 for the fix-up pass after the row emission.
// ---- the reduction of one head's group, in three parts: walk (sequential, may defer a long group to its warp),
// ---- the warp-cooperative walk, and the epilogue that stores the result

// Epilogue: what a finished head (or a non-head) writes.
template <class Rows, bool BY_T, bool DIRECT, bool TILE>
__device__ __forceinline__ void sum_finish(const Rows &rows, const RecFmt &fmt, uint64_t r0, int64_t d, double re, double im,
                                           bool have, bool is_multi, double thr, double2 *__restrict__ acc,
                                           uint8_t *__restrict__ keep, uint8_t *__restrict__ multi, const TileMap &tm) {
    if (TILE) {
        if (is_multi) {
            if (keep_test(re, im, thr)) {
                acc[d] = make_double2(re, im);
                multi[d] = 1;
            } else {
                tm.mark_dropped(fmt.t(r0));
            }
        } else if (!(thr < 0.0 || rows.all_pass())) {
            rows.coeff_unphased(fmt.t(r0), re, im);
            if (!keep_test(re, im, thr)) tm.mark_dropped(fmt.t(r0));
        }
        return;
    }
    if (is_multi || !DIRECT) {
        if (!have) rows.coeff(fmt.t(r0), fmt.e(r0), re, im);
        acc[d] = make_double2(re, im);
        multi[d] = 1;
        keep[d] = keep_test(re, im, thr);
    } else if (thr < 0.0 || rows.all_pass()) {
        keep[d] = 1;         // singleton that cannot fail the threshold: the coefficient is computed once, at emission
    } else {
        rows.coeff(fmt.t(r0), fmt.e(r0), re, im);
        keep[d] = keep_test(re, im, thr);
    }
}

template <class Rows, bool TILE>
__device__ __forceinline__ void head_coeff(const Rows &rows, const RecFmt &fmt, uint64_t r0, double &re, double &im) {
    int e0 = fmt.e(r0);
    if constexpr (TILE) e0 = rows.phase(fmt.t(r0));   // members were stamped by phase_work_kernel, heads were not
    rows.coeff(fmt.t(r0), e0, re, im);
}

// Sequential walk of the head at sorted position i (np.add.at order). Records, flags and coefficients are fetched
// SUM_BATCH at a time. Returns true when the group is still open after SUM_DEFER_BATCHES batches: the caller's warp
// then redoes this head cooperatively (sum_walk_warp) — a long group (the M identity terms of a square, the ~50-term
// groups of a molecular H*H) would otherwise be one thread's chain of dependent loads.
constexpr int SUM_BATCH = 8;
constexpr int SUM_DEFER_BATCHES = 2;
template <class Rows, bool BY_T, bool DIRECT, bool TILE>
__device__ __forceinline__ bool sum_one(const Rows &rows, const RecFmt &fmt, const uint64_t *__restrict__ sr, int64_t T,
                                        int64_t i, int sort_shift, const uint8_t *__restrict__ flag,
                                        const uint32_t *__restrict__ link, double thr, double2 *__restrict__ acc,
                                        uint8_t *__restrict__ keep, uint8_t *__restrict__ multi, const TileMap &tm) {
    const uint64_t r0 = sr[i];
    const int64_t d = BY_T ? (int64_t)fmt.t(r0) : i;
    if (TILE) multi[d] = 0;
    if (flag[i] != FLAG_HEAD) {
        if (TILE) tm.mark_dropped(fmt.t(r0));
        else keep[d] = 0;
        return false;
    }
    double re = 0.0, im = 0.0;
    bool have = false, is_multi = false;
    bool prev_mine = true;   // is record j-1 a member of this head's group?
    bool open = true;
    int batches = 0;
    for (int64_t j0 = i + 1; open && j0 < T; j0 += SUM_BATCH) {
        if (batches++ == SUM_DEFER_BATCHES) return true;   // long group: nothing has been written yet
        uint64_t rj[SUM_BATCH];
        uint8_t fj[SUM_BATCH];
        int n_in = 0;
#pragma unroll
        for (int u = 0; u < SUM_BATCH; ++u) rj[u] = (j0 + u < T) ? sr[j0 + u] : 0ull;
#pragma unroll
        for (int u = 0; u < SUM_BATCH; ++u) {
            const bool in = open && (j0 + u < T) && ((r0 ^ rj[u]) >> sort_shift) == 0;   // still inside the bucket
            open = in;
            n_in += in ? 1 : 0;
        }
        if (n_in == 0) break;
#pragma unroll
        for (int u = 0; u < SUM_BATCH; ++u) fj[u] = (u < n_in) ? flag[j0 + u] : FLAG_HEAD;
        bool mine[SUM_BATCH];
        bool any = false;
#pragma unroll
        for (int u = 0; u < SUM_BATCH; ++u) {
            bool mn = false;
            if (u < n_in) {
                // only records with this head's hash can be members; in ordered-tile mode the others may not even
                // have a flag (they never went on the worklist)
                if (!fmt.same_hash(r0, rj[u])) mn = false;
                else if (fj[u] == FLAG_PREV) mn = prev_mine;
                else if (fj[u] == FLAG_LINK) mn = chain_root(flag, link, (int64_t)link[j0 + u]) == i;
                prev_mine = mn;
            }
            mine[u] = mn;
            any |= mn;
        }
        if (!any) continue;
        double cr[SUM_BATCH], ci[SUM_BATCH];
#pragma unroll
        for (int u = 0; u < SUM_BATCH; ++u) {
            cr[u] = 0.0;
            ci[u] = 0.0;
            if (mine[u]) rows.coeff(fmt.t(rj[u]), fmt.e(rj[u]), cr[u], ci[u]);
        }
        if (!have) {
            head_coeff<Rows, TILE>(rows, fmt, r0, re, im);
            have = true;
        }
#pragma unroll
        for (int u = 0; u < SUM_BATCH; ++u) {
            if (mine[u]) {
                re += cr[u];
                im += ci[u];
            }
        }
        is_multi = true;
    }
    sum_finish<Rows, BY_T, DIRECT, TILE>(rows, fmt, r0, d, re, im, have, is_multi, thr, acc, keep, multi, tm);
    return false;
}

// The same walk by a whole (converged) warp for the head at position i: lane l looks at records base + 32u + l of
// SUM_WIN windows at a time, membership of the FLAG_PREV chains is resolved with ballots (a PREV record follows
// the nearest earlier record that is not PREV), coefficients are gathered in parallel and added by every lane in
// record order — the same additions in the same order as the sequential walk, so the result is bit-identical to
// it. Every lane returns the sums. The loads of the SUM_WIN windows (records and flags, then coefficients) are
// issued together and the broadcasts of a window do not depend on the running sum, so a long group costs two
// memory round trips per 128 records plus its chain of FP64 adds (the 500 identity terms of config C1: 35 -> 6 us).
constexpr int SUM_WIN = 4;
template <class Rows, bool TILE>
__device__ __forceinline__ void sum_walk_warp(const Rows &rows, const RecFmt &fmt, const uint64_t *__restrict__ sr, int64_t T,
                                              int64_t i, int sort_shift, const uint8_t *__restrict__ flag,
                                              const uint32_t *__restrict__ link, int lane, double &re, double &im,
                                              bool &is_multi) {
    const uint64_t r0 = sr[i];
    head_coeff<Rows, TILE>(rows, fmt, r0, re, im);
    is_multi = false;
    bool carry = true;   // membership of the record just before this window (the head itself at first)
    bool open = true;
    for (int64_t base = i + 1; open && base < T; base += 32 * SUM_WIN) {
        uint64_t rj[SUM_WIN];
        uint8_t fj[SUM_WIN];
#pragma unroll
        for (int u = 0; u < SUM_WIN; ++u) {
            const int64_t j = base + 32 * u + lane;
            rj[u] = j < T ? sr[j] : 0ull;
            fj[u] = j < T ? flag[j] : FLAG_HEAD;   // read before the bucket test: one round trip for both
        }
        uint32_t mine_mask[SUM_WIN];
        bool mine[SUM_WIN];
#pragma unroll
        for (int u = 0; u < SUM_WIN; ++u) {
            mine_mask[u] = 0u;
            mine[u] = false;
            if (!open) continue;   // uniform
            const int64_t j = base + 32 * u + lane;
            const bool in = j < T && ((r0 ^ rj[u]) >> sort_shift) == 0;
            const uint32_t out_mask = __ballot_sync(0xffffffffu, !in);
            const int n_in = out_mask ? __ffs(out_mask) - 1 : 32;        // the bucket is contiguous
            if (n_in < 32) open = false;
            if (n_in == 0) continue;
            const bool valid = lane < n_in;
            // only records with this head's hash can be members; in ordered-tile mode the others may not even
            // have a flag (they never went on the worklist)
            const bool sh = valid && fmt.same_hash(r0, rj[u]);
            const bool is_prev = sh && fj[u] == FLAG_PREV;
            const bool m0 = sh && fj[u] == FLAG_LINK && chain_root(flag, link, (int64_t)link[j]) == i;
            const uint32_t decided = __ballot_sync(0xffffffffu, !is_prev);
            const uint32_t m0_mask = __ballot_sync(0xffffffffu, m0);
            const uint32_t lower = decided & ((1u << lane) - 1u);
            mine[u] = is_prev ? (lower ? ((m0_mask >> (31 - __clz(lower))) & 1u) != 0u : carry) : m0;
            mine_mask[u] = __ballot_sync(0xffffffffu, mine[u]);
            carry = (mine_mask[u] >> 31) & 1u;
        }
        double cr[SUM_WIN], ci[SUM_WIN];
#pragma unroll
        for (int u = 0; u < SUM_WIN; ++u) {
            cr[u] = 0.0;
            ci[u] = 0.0;
            if (mine[u]) rows.coeff(fmt.t(rj[u]), fmt.e(rj[u]), cr[u], ci[u]);
        }
#pragma unroll
        for (int u = 0; u < SUM_WIN; ++u) {
            if (mine_mask[u] == 0u) continue;   // uniform
            is_multi = true;
#pragma unroll
            for (int l = 0; l < 32; ++l) {      // record order; the broadcasts run ahead of the adds
                const double vr = __shfl_sync(0xffffffffu, cr[u], l), vi = __shfl_sync(0xffffffffu, ci[u], l);
                if ((mine_mask[u] >> l) & 1u) {
                    re += vr;
                    im += vi;
                }
            }
        }
    }
}

// One record per lane (valid lanes only), then the warp finishes its deferred heads one after the other.
template <class Rows, bool BY_T, bool DIRECT, bool TILE>
__device__ __forceinline__ void sum_warp_step(const Rows &rows, const RecFmt &fmt, const uint64_t *__restrict__ sr, int64_t T,
                                              bool valid, int64_t i, int sort_shift, const uint8_t *__restrict__ flag,
                                              const uint32_t *__restrict__ link, double thr, double2 *__restrict__ acc,
                                              uint8_t *__restrict__ keep, uint8_t *__restrict__ multi, const TileMap &tm) {
    const int lane = threadIdx.x & 31;
    const bool deferred =
        valid && sum_one<Rows, BY_T, DIRECT, TILE>(rows, fmt, sr, T, i, sort_shift, flag, link, thr, acc, keep, multi, tm);
    for (uint32_t pend = __ballot_sync(0xffffffffu, deferred); pend; pend &= pend - 1u) {
        const int l = __ffs(pend) - 1;
        const int64_t il = __shfl_sync(0xffffffffu, (long long)i, l);
        double re, im;
        bool is_multi;
        sum_walk_warp<Rows, TILE>(rows, fmt, sr, T, il, sort_shift, flag, link, lane, re, im, is_multi);
        if (lane == l) {
            const uint64_t r0 = sr[il];
            const int64_t d = BY_T ? (int64_t)fmt.t(r0) : il;
            sum_finish<Rows, BY_T, DIRECT, TILE>(rows, fmt, r0, d, re, im, true, is_multi, thr, acc, keep, multi, tm);
        }
    }
}

template <class Rows, bool BY_T, bool DIRECT>
__global__ void __launch_bounds__(256) sum_kernel(Rows rows, RecFmt fmt, const uint64_t *__restrict__ sr, int64_t T,
                                                   int sort_shift, const uint8_t *__restrict__ flag,
                                                   const uint32_t *__restrict__ link, double thr, double2 *__restrict__ acc,
                                                   uint8_t *__restrict__ keep, uint8_t *__restrict__ multi) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    sum_warp_step<Rows, BY_T, DIRECT, false>(rows, fmt, sr, T, i < T, i, sort_shift, flag, link, thr, acc, keep, multi,
                                             TileMap());
}

// ordered-tile mode: records are generated without a phase exponent (the tiled emission computes it for the
// survivors); the records that join a group (everything link_work_kernel did not leave as a head) get
// theirs here, in parallel, between link and sum
template <class Rows>
__global__ void __launch_bounds__(256) phase_work_kernel(Rows rows, RecFmt fmt, uint64_t *__restrict__ sr, WorkList wl,
                                                          const uint8_t *__restrict__ flag) {
    FOR_EACH_WORK(wl, i) {
        if (flag[i] == FLAG_HEAD) continue;   // a head computes its own, and only if its group has members
        const uint64_t rec = sr[i];
        sr[i] = (rec & ~3ull) | (uint64_t)rows.phase(fmt.t(rec));
    }
}

// ordered-tile mode: the reduction over the worklist (records of non-singleton buckets)
template <class Rows>
__global__ void __launch_bounds__(256) sum_work_kernel(Rows rows, RecFmt fmt, const uint64_t *__restrict__ sr, int64_t T,
                                                        int sort_shift, WorkList wl, const uint8_t *__restrict__ flag,
                                                        const uint32_t *__restrict__ link, double thr, double2 *__restrict__ acc,
                                                        uint8_t *__restrict__ multi, TileMap tm) {
    // whole warps walk the region together (a lane without an entry idles) so that they can finish long groups jointly
    const uint32_t r = blockIdx.x / WORK_SPLIT, n = wl.region_count(r);
    const int64_t hi = wl.hi(T);
    for (uint32_t k0 = (blockIdx.x % WORK_SPLIT) * blockDim.x + (threadIdx.x & ~31u); k0 < n; k0 += WORK_SPLIT * blockDim.x) {
        const uint32_t k = k0 + (threadIdx.x & 31u);
        const bool valid = k < n;
        const int64_t i = valid ? (int64_t)wl.entry(r, k) : 0;
        sum_warp_step<Rows, false, true, true>(rows, fmt, sr, hi, valid, i, sort_shift, flag, link, thr, acc, nullptr, multi, tm);
    }
}

// Ordered-tile mode, first pass over the sorted records: a record whose sort bucket holds no other
// record with its full hash is a singleton survivor (or fails the threshold on its own) — no link,
// no sum, nothing written. Only records with a same-hash bucket mate go on the worklist for
// link / phase / sum / fix-up (0.4 % of the records of a collision-free 1.25e8-term product).
constexpr int CLS_ITEMS = 8;                    // records per thread: eight independent loads in flight, and
constexpr int CLS_TILE = 256 * CLS_ITEMS;       // one counter update (an L2 round trip) per 2048 records
template <class Rows>
__global__ void __launch_bounds__(256) tile_classify_kernel(Rows rows, RecFmt fmt, const uint64_t *__restrict__ sr, int64_t T,
                                                             int sort_shift, double thr, TileMap tm, WorkList wl) {
    __shared__ uint32_t s_warp[8];
    __shared__ uint32_t s_base;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    const int64_t base = (int64_t)blockIdx.x * CLS_TILE + threadIdx.x;
    uint64_t r[CLS_ITEMS];
#pragma unroll
    for (int j = 0; j < CLS_ITEMS; ++j) {
        const int64_t i = base + j * 256;
        r[j] = i < T ? sr[i] : 0ull;
    }
    // pass 1 (unrolled, branch-light): same-hash mate among the two immediate neighbours?
    uint32_t mine = 0, unsure = 0;   // bit j: record j has a same-hash bucket mate / shares its bucket but not with a same-hash neighbour
#pragma unroll
    for (int j = 0; j < CLS_ITEMS; ++j) {
        const int64_t i = base + j * 256;
        // the neighbours come from the adjacent lanes; the warp's edge lanes load theirs
        uint64_t rp = __shfl_up_sync(0xffffffffu, r[j], 1), rn = __shfl_down_sync(0xffffffffu, r[j], 1);
        if (lane == 0 && i > 0 && i < T) rp = sr[i - 1];
        if (lane == 31 && i + 1 < T) rn = sr[i + 1];
        if (i < T) {
            const bool same_prev = i > 0 && ((r[j] ^ rp) >> sort_shift) == 0;
            const bool same_next = i + 1 < T && ((r[j] ^ rn) >> sort_shift) == 0;
            const bool mate = (same_prev && fmt.same_hash(r[j], rp)) || (same_next && fmt.same_hash(r[j], rn));
            if (mate) mine |= 1u << j;
            else if (same_prev || same_next) unsure |= 1u << j;
        }
    }
    // pass 2 (rare: ~3 % of the records share a bucket, almost all of those buckets hold just two): look past
    // the immediate neighbours for a same-hash mate
    while (unsure) {
        const int j = __ffs(unsure) - 1;
        unsure &= unsure - 1u;
        const int64_t i = base + j * 256;
        const uint64_t ri = sr[i];   // (r[] stays in registers: no dynamic indexing)
        bool mate = false;
        for (int64_t k = i - 2; k >= 0 && !mate; --k) {
            const uint64_t rk = sr[k];
            if (((ri ^ rk) >> sort_shift) != 0) break;
            mate = fmt.same_hash(ri, rk);
        }
        for (int64_t k = i + 2; k < T && !mate; ++k) {
            const uint64_t rk = sr[k];
            if (((ri ^ rk) >> sort_shift) != 0) break;
            mate = fmt.same_hash(ri, rk);
        }
        if (mate) mine |= 1u << j;
    }
    // singletons: nothing to do unless a single cross term can fail the threshold
    if (!(thr < 0.0 || rows.all_pass())) {
#pragma unroll
        for (int j = 0; j < CLS_ITEMS; ++j) {
            const int64_t i = base + j * 256;
            if (i < T && !((mine >> j) & 1u)) {
                double re, im;
                rows.coeff_unphased(fmt.t(r[j]), re, im);
                if (!keep_test(re, im, thr)) tm.mark_dropped(fmt.t(r[j]));
            }
        }
    }
    uint32_t m[CLS_ITEMS];
    uint32_t warp_total = 0;
#pragma unroll
    for (int j = 0; j < CLS_ITEMS; ++j) {
        m[j] = __ballot_sync(0xffffffffu, (mine >> j) & 1u);
        warp_total += (uint32_t)__popc(m[j]);
    }
    if (lane == 0) s_warp[wid] = warp_total;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const uint32_t c = s_warp[w];
            s_warp[w] = tot;
            tot += c;
        }
        s_base = tot ? atomicAdd(wl.counts + blockIdx.x % wl.nreg, tot) : 0u;
    }
    __syncthreads();
    if (warp_total == 0u) return;
    uint32_t pos = s_base + s_warp[wid];
    uint32_t *dst = wl.work + (size_t)(blockIdx.x % wl.nreg) * wl.cap;
#pragma unroll
    for (int j = 0; j < CLS_ITEMS; ++j) {
        if ((mine >> j) & 1u) dst[pos + __popc(m[j] & lt)] = (uint32_t)(base + j * 256);
        pos += (uint32_t)__popc(m[j]);
    }
}

// pass_all flag of a product: min|a| * min|b| clears the threshold with a 4x margin (the rounded
// product of any single pair is within a few ulp of |a||b|), so no singleton cross term can fail
// |c| > thr and the reduction need not gather coefficients for them. Grid-stride minimum per operand
// (bit patterns of non-negative doubles order like unsigned integers: atomicMin), then one thread.
__global__ void __launch_bounds__(256) min_abs_kernel(const double2 *__restrict__ a, int64_t M, unsigned long long *__restrict__ out) {
    __shared__ double sm[8];
    double m = INFINITY;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (int64_t)gridDim.x * blockDim.x) {
        double h = hypot(a[i].x, a[i].y);
        if (!(h >= 0.0)) h = 0.0;   // NaN
        m = fmin(m, h);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmin(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) m = fmin(m, sm[w]);
        atomicMin(out, (unsigned long long)__double_as_longlong(m));
    }
}

__global__ void min_abs_flag_finish_kernel(const unsigned long long *__restrict__ mins, double thr, uint32_t *__restrict__ flag) {
    const double prod = __longlong_as_double((long long)mins[0]) * __longlong_as_double((long long)mins[1]);
    *flag = (isfinite(prod) && prod > 4.0 * thr) ? 1u : 0u;
}

// mins: two uint64 of scratch (free until the scans run); flag: device uint32
static int launch_min_abs_flag(const double2 *a, int64_t M, const double2 *b, int64_t N, double thr, unsigned long long *mins,
                               uint32_t *flag, cudaStream_t st) {
    SYM_CUDA_OK(cudaMemsetAsync(mins, 0xff, 2 * sizeof(unsigned long long), st));
    const unsigned ga = (unsigned)std::max<int64_t>(1, std::min<int64_t>((M + 255) / 256, (int64_t)num_sms() * 8));
    const unsigned gb = (unsigned)std::max<int64_t>(1, std::min<int64_t>((N + 255) / 256, (int64_t)num_sms() * 8));
    min_abs_kernel<<<ga, 256, 0, st>>>(a, M, mins);
    SYM_LAUNCH_OK();
    min_abs_kernel<<<gb, 256, 0, st>>>(b, N, mins + 1);
    SYM_LAUNCH_OK();
    min_abs_flag_finish_kernel<<<1, 1, 0, st>>>(mins, thr, flag);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

// Compaction (emit phase): kept_t[slot] = term index of the survivor, out_c[slot] = its coefficient,
// so that the row-emission kernel has a two-step dependency chain (kept_t -> rows) only.
template <class Rows, bool BY_T>
__global__ void __launch_bounds__(256) compact_kernel(Rows rows, RecFmt fmt, const uint64_t *__restrict__ sr,
                                                       const uint8_t *__restrict__ keep, const uint8_t *__restrict__ multi,
                                                       const uint32_t *__restrict__ slot, const double2 *__restrict__ acc,
                                                       int64_t T, uint32_t *__restrict__ kept_t, double2 *__restrict__ out_c) {
    int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= T) return;
    if (keep[d]) {
        const uint32_t s = slot[d];
        uint32_t t;
        int e = 0;
        if (BY_T) {
            t = (uint32_t)d;
        } else {
            const uint64_t rec = sr[d];
            t = fmt.t(rec);
            e = fmt.e(rec);
        }
        kept_t[s] = t;
        if (multi[d]) {
            out_c[s] = acc[d];
        } else {   // singleton survivor: its coefficient was never materialised
            double re, im;
            rows.coeff(t, e, re, im);
            out_c[s] = make_double2(re, im);
        }
    }
}

__global__ void total_to_i64_kernel(const uint32_t *__restrict__ total, int64_t *__restrict__ n_out) { *n_out = (int64_t)*total; }

// Row emission. One thread per (kept record, 16-byte chunk), EMIT_UN records per thread so that
// 2*EMIT_UN independent 16-byte loads are in flight per thread (the kernel is latency-bound
// otherwise). Stores are streaming (st.global.cs): the output is never re-read, and A/B must stay
// L2-resident. LW: chunks per row = 1 << LW.
// Compaction and emission are two kernels: measured on B200, 7.1 ms for 1.25e8 rows of 272 B against 8.8 ms
// for a CTA-fused form, whose barrier between the two phases stalls the block.

// optional CUDA events recorded around the row-emission kernel (sym_set_emit_events)
static cudaEvent_t g_emit_ev0 = nullptr, g_emit_ev1 = nullptr;
void set_emit_events(cudaEvent_t a, cudaEvent_t b) {
    g_emit_ev0 = a;
    g_emit_ev1 = b;
}

__device__ __forceinline__ void store_streaming(uint4 *p, const uint4 &v) {
    asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

template <class Rows, int LW, int EMIT_UN, bool CS>
__global__ void __launch_bounds__(256) emit_kernel(Rows rows, const uint32_t *__restrict__ kept_t, uint32_t U,
                                                    uint4 *__restrict__ out_xz) {
    constexpr uint32_t ROWS_PP = 256u >> LW;
    const uint32_t r_in = threadIdx.x >> LW;
    const uint32_t c = threadIdx.x & ((1u << LW) - 1u);
    uint32_t rec[EMIT_UN], t[EMIT_UN];
    uint4 v[EMIT_UN];
#pragma unroll
    for (int u = 0; u < EMIT_UN; ++u) {
        rec[u] = (blockIdx.x * EMIT_UN + u) * ROWS_PP + r_in;
        t[u] = rec[u] < U ? kept_t[rec[u]] : 0u;
    }
#pragma unroll
    for (int u = 0; u < EMIT_UN; ++u) v[u] = rows.chunk(t[u], (int)c);
#pragma unroll
    for (int u = 0; u < EMIT_UN; ++u) {
        if (rec[u] < U) {
            if (CS) store_streaming(out_xz + (((size_t)rec[u]) << LW) + c, v[u]);
            else out_xz[(((size_t)rec[u]) << LW) + c] = v[u];
        }
    }
}

// generic chunk count (W not a power of two, or W > 16)
template <class Rows>
__global__ void __launch_bounds__(256) emit_generic_kernel(Rows rows, const uint32_t *__restrict__ kept_t, uint32_t U,
                                                            uint32_t chunks, uint4 *__restrict__ out_xz) {
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t rec = (uint32_t)(g / chunks);
    const uint32_t c = (uint32_t)(g - (size_t)rec * chunks);
    if (rec >= U) return;
    out_xz[g] = rows.chunk(kept_t[rec], (int)c);
}

size_t dedup_ws_bytes(int64_t T) {
    if (T < 1) T = 1;
    size_t n = (size_t)T;
    return arena_need(n, 8)                          // alt record buffer
           + arena_need(record_hist_elems(T), 4)     // radix histograms + scan scratch
           + arena_need(n, 1)                        // flag
           + arena_need(n, 4)                        // link
           + arena_need(n, 16)                       // acc
           + arena_need(n, 1)                        // keep
           + arena_need(n, 1)                        // multi
           + arena_need(n, 4)                        // slot
           + arena_need(n, 4)                        // kept
           + arena_need(scan_scratch_elems(T), 4)    // scan scratch
           + arena_need(16, 4) + 4096;
}

// Sort on log2(T) + SORT_EXTRA_BITS hash bits, rounded up to whole 8-bit passes. A sort bucket then
// holds T / 2^bits records on average, which link/sum resolve exactly with in-bucket scans: fewer
// bits save radix passes (24 B of HBM traffic per record each) but lengthen those scans.
constexpr int SORT_EXTRA_BITS = 5;
static int sort_begin_bit(int64_t T, RecFmt fmt) {
    int lg = t_bits_for(T);
    int want = ((lg + SORT_EXTRA_BITS + 7) / 8) * 8;
    if (want < 8) want = 8;
    int begin = 64 - want;
    if (begin < fmt.tb + 2) begin = fmt.tb + 2;
    return begin;
}

static bool sorted_in_alt(int begin_bit) {
    int passes = (64 - begin_bit + 7) / 8;
    return (passes & 1) != 0;
}

struct DedupLayout {
    uint64_t *alt;
    uint32_t *hist;
    uint8_t *flag;
    uint32_t *link;
    double2 *acc;
    uint8_t *keep;
    uint8_t *multi;
    uint32_t *slot;
    uint32_t *kept;
    uint32_t *scratch;
    uint32_t *total;
    bool ok;
};

static DedupLayout dedup_layout(void *ws, size_t ws_bytes, int64_t T) {
    Arena ar(ws, ws_bytes);
    DedupLayout L;
    L.alt = ar.take<uint64_t>((size_t)T);
    L.hist = ar.take<uint32_t>(record_hist_elems(T));
    L.flag = ar.take<uint8_t>((size_t)T);
    L.link = ar.take<uint32_t>((size_t)T);
    L.acc = ar.take<double2>((size_t)T);
    L.keep = ar.take<uint8_t>((size_t)T);
    L.multi = ar.take<uint8_t>((size_t)T);
    L.slot = ar.take<uint32_t>((size_t)T);
    L.kept = ar.take<uint32_t>((size_t)T);
    L.scratch = ar.take<uint32_t>(scan_scratch_elems(T));
    L.total = ar.take<uint32_t>(16);   // [0] scan total, [2] pass_all flag, [8..11] class-mode counters
    L.ok = L.total != nullptr;
    return L;
}

// Phase 1: everything up to the survivor count (synchronises the stream once to read it).
template <class Rows, bool BY_T>
static int dedup_plan(uint64_t *recs, int64_t T, RecFmt fmt, const Rows &rows, double thr, int64_t *n_out,
                      int64_t *n_out_host, void *ws, size_t ws_bytes, cudaStream_t st) {
    if (T == 0) {
        if (n_out) SYM_CUDA_OK(cudaMemsetAsync(n_out, 0, sizeof(int64_t), st));
        if (n_out_host) *n_out_host = 0;
        return SYM_OK;
    }
    if (ws_bytes < dedup_ws_bytes(T)) {
        set_error("workspace too small: need %zu bytes, got %zu", dedup_ws_bytes(T), ws_bytes);
        return SYM_E_WORKSPACE;
    }
    DedupLayout L = dedup_layout(ws, ws_bytes, T);
    if (!L.ok) {
        set_error("workspace arena exhausted");
        return SYM_E_WORKSPACE;
    }
    const int begin = sort_begin_bit(T, fmt);
    uint64_t *sr = nullptr;
    SYM_TRY(radix_sort(recs, nullptr, L.alt, nullptr, T, begin, L.hist, &sr, st));

    const unsigned nb = (unsigned)((T + 255) / 256);
    link_kernel<Rows><<<nb, 256, 0, st>>>(rows, fmt, sr, T, begin, L.flag, L.link);
    SYM_LAUNCH_OK();
    // singleton survivors skip the acc[] round trip when their coefficient can be recomputed at
    // compaction: always in sorted order (the record carries t and the phase), and for stored rows
    constexpr bool DIRECT = !BY_T || std::is_same<Rows, PlainRows>::value;
    SYM_CUDA_OK(cudaMemsetAsync(L.multi, 0, (size_t)T, st));
    Rows rows_sum = rows;
    if constexpr (std::is_same<Rows, ProductRows>::value && !BY_T) {
        if (thr >= 0.0 && rows.N > 0) {
            SYM_TRY(launch_min_abs_flag(reinterpret_cast<const double2 *>(rows.Ac), (int64_t)rows.M,
                                        reinterpret_cast<const double2 *>(rows.Bc), (int64_t)rows.N, thr,
                                        reinterpret_cast<unsigned long long *>(L.scratch), L.total + 2, st));
            rows_sum.pass_all = L.total + 2;
        }
    }
    sum_kernel<Rows, BY_T, DIRECT><<<nb, 256, 0, st>>>(rows_sum, fmt, sr, T, begin, L.flag, L.link, thr, L.acc, L.keep,
                                                      L.multi);
    SYM_LAUNCH_OK();
    SYM_TRY(scan_exclusive_u8(L.keep, L.slot, T, L.total, L.scratch, st));
    if (n_out) {
        total_to_i64_kernel<<<1, 1, 0, st>>>(L.total, n_out);
        SYM_LAUNCH_OK();
    }
    uint32_t U32 = 0;
    SYM_CUDA_OK(cudaMemcpyAsync(&U32, L.total, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    SYM_CUDA_OK(cudaStreamSynchronize(st));
    if (n_out_host) *n_out_host = (int64_t)U32;
    return SYM_OK;
}

// Phase 2: write the U surviving rows + coefficients (asynchronous). `recs` is the same buffer
// that was given to the plan phase.
template <class Rows, bool BY_T>
static int dedup_emit(const uint64_t *recs, int64_t T, RecFmt fmt, const Rows &rows, int64_t U, uint64_t *out_xz,
                      double *out_c, void *ws, size_t ws_bytes, cudaStream_t st) {
    if (T == 0 || U == 0) return SYM_OK;
    DedupLayout L = dedup_layout(ws, ws_bytes, T);
    if (!L.ok) {
        set_error("workspace arena exhausted");
        return SYM_E_WORKSPACE;
    }
    const uint64_t *sr = (T > 1 && sorted_in_alt(sort_begin_bit(T, fmt))) ? L.alt : recs;
    const uint32_t chunks = (uint32_t)(rows.words / 2);
    uint4 *o = reinterpret_cast<uint4 *>(out_xz);
    double2 *oc = reinterpret_cast<double2 *>(out_c);
    // compaction, then row emission
    compact_kernel<Rows, BY_T><<<(unsigned)((T + 255) / 256), 256, 0, st>>>(rows, fmt, sr, L.keep, L.multi, L.slot, L.acc, T,
                                                                           L.kept, oc);
    SYM_LAUNCH_OK();
    if (g_emit_ev0) SYM_CUDA_OK(cudaEventRecord(g_emit_ev0, st));   // bench.py times the row-emission kernel alone
#define EMIT_LAUNCH(LW, UN, CS)                                                                   \
    {                                                                                             \
        const uint32_t rows_per_block = (256u >> LW) * UN;                                        \
        const unsigned nbe = (unsigned)((U + rows_per_block - 1) / rows_per_block);               \
        emit_kernel<Rows, LW, UN, CS><<<nbe, 256, 0, st>>>(rows, L.kept, (uint32_t)U, o);         \
    }
    switch (chunks) {
        case 1: EMIT_LAUNCH(0, 8, false); break;
        case 2: EMIT_LAUNCH(1, 8, false); break;
        case 4: EMIT_LAUNCH(2, 8, false); break;
        case 8: EMIT_LAUNCH(3, 8, false); break;
        case 16: EMIT_LAUNCH(4, 8, false); break;
        default: {
            const size_t threads = (size_t)U * chunks;
            emit_generic_kernel<Rows><<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(rows, L.kept, (uint32_t)U, chunks, o);
        } break;
    }
#undef EMIT_LAUNCH
    SYM_LAUNCH_OK();
    if (g_emit_ev1) SYM_CUDA_OK(cudaEventRecord(g_emit_ev1, st));
    return SYM_OK;
}

// ---------------------------------------------------------------------------------------------
// Ordered-tile mode (rows.cuh): survivors in cross-term order, tiled streaming row emission
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ TileBlock tile_block_of_segment(const TileMap &tm, uint32_t s) {
    TileBlock blk = tm.first;
    for (int b = 1; b < tm.nblk; ++b) {
        const TileBlock nb = tm.blocks[b];
        if (s < nb.seg_base) break;
        blk = nb;
    }
    return blk;
}

// survivors per segment = valid rows whose drop bit is clear
__global__ void __launch_bounds__(256) seg_count_kernel(TileMap tm) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= tm.n_seg) return;
    const TileBlock blk = tile_block_of_segment(tm, s);
    const uint32_t ptile = (s - blk.seg_base) % blk.ptiles;
    const uint4 d = reinterpret_cast<const uint4 *>(tm.drop)[s];
    tm.segoff[s] = __popc(tile_valid_word(blk.m_blk, ptile, 0) & ~d.x) + __popc(tile_valid_word(blk.m_blk, ptile, 1) & ~d.y) +
                   __popc(tile_valid_word(blk.m_blk, ptile, 2) & ~d.z) + __popc(tile_valid_word(blk.m_blk, ptile, 3) & ~d.w);
}

// Row + coefficient emission of one block, CTA = (tile of TILE_ROWS rows of A) x (QG rows of B).
// Thread = (row, word c): it holds X word c and Z word c of its UN rows of A in registers for the
// whole q loop; the B row is two broadcast 8-byte loads per q, so the only traffic that scales
// with the output is the output itself: consecutive survivors of a segment go to consecutive
// slots (streaming stores, a warp writes whole 128-byte lines).
// Holding the X and Z words of the same qubits lets the thread also compute its share of the
// phase exponent (base.py:785-788): popc((xa^xb)&(za^zb)) + 2*popc(xa&zb) mod 4, packed as one
// 4-bit field per row and XOR-shuffle-reduced over the W lanes of the row (all UN rows in one
// word), then 3*(Ya+Yb) is added. Lane u of a row group writes the coefficient a[p]*b[q]*i^e of row
// u; group sums overwrite theirs in the fix-up pass. The kernel stays HBM-write bound.
template <int LW>
__global__ void __launch_bounds__((TILE_ROWS << LW) < 256 ? (TILE_ROWS << LW) : 256)
    tile_emit_kernel(const uint64_t *__restrict__ A, const double2 *__restrict__ Ac, const int32_t *__restrict__ Ay,
                     const uint64_t *__restrict__ B, const double2 *__restrict__ Bc, const int32_t *__restrict__ By,
                     TileBlock first, const TileBlock *__restrict__ blocks, uint32_t qg, const uint32_t *__restrict__ drop,
                     const uint32_t *__restrict__ segoff, uint64_t *__restrict__ out_xz, double2 *__restrict__ out_c) {
    // one launch covers every block of the list (blockIdx.z): no launch tails between the blocks of a sharded product
    const TileBlock blk = blockIdx.z == 0 ? first : blocks[blockIdx.z];
    if (blockIdx.x >= blk.ptiles || blockIdx.y * qg >= blk.nq) return;
    constexpr int TH = (TILE_ROWS << LW) < 256 ? (TILE_ROWS << LW) : 256;
    constexpr int W = 1 << LW;            // words per X (and per Z) block = lanes per row
    constexpr int RP = TH >> LW;          // rows per pass
    constexpr int UN = TILE_ROWS / RP;    // passes per segment (UN <= W)
    static_assert(UN <= W && UN <= 8, "one coefficient lane per row, one 4-bit phase field per row");
    const uint32_t ptile = blockIdx.x;
    const uint32_t r_in = threadIdx.x >> LW, c = threadIdx.x & (W - 1);
    const uint32_t pl0 = ptile * TILE_ROWS;

    uint64_t xa[UN], za[UN];
    uint32_t ya3 = 0;                     // 3*Ya mod 4 of the UN rows, 4 bits apart
    double2 ac = make_double2(0.0, 0.0);  // coefficient of row u == c
#pragma unroll
    for (int u = 0; u < UN; ++u) {
        const uint32_t pl = pl0 + u * RP + r_in;
        const bool ok = pl < blk.m_blk;
        const size_t row = (size_t)(blk.p0 + (ok ? pl : 0u));
        xa[u] = ok ? A[row * (2 * W) + c] : 0ull;
        za[u] = ok ? A[row * (2 * W) + W + c] : 0ull;
        ya3 |= ((3u * (uint32_t)(ok ? Ay[row] : 0)) & 3u) << (4 * u);
        if ((int)c == u && ok) ac = Ac[row];
    }
    uint32_t vm[4];
#pragma unroll
    for (int w = 0; w < 4; ++w) vm[w] = tile_valid_word(blk.m_blk, ptile, w);

    const uint32_t q_lo = blockIdx.y * qg;
    const uint32_t q_hi = min(blk.nq, q_lo + qg);
    for (uint32_t ql = q_lo; ql < q_hi; ++ql) {
        const uint32_t s = blk.seg_base + ql * blk.ptiles + ptile;
        const size_t qrow = (size_t)(blk.q0 + ql);
        const uint4 d = reinterpret_cast<const uint4 *>(drop)[s];
        const uint32_t base = segoff[s];
        const uint64_t xb = B[qrow * (2 * W) + c], zb = B[qrow * (2 * W) + W + c];
        const uint32_t yb3 = (3u * (uint32_t)By[qrow]) & 3u;
        const uint32_t k[4] = {vm[0] & ~d.x, vm[1] & ~d.y, vm[2] & ~d.z, vm[3] & ~d.w};
        uint32_t pre[4];
        pre[0] = base;
        pre[1] = pre[0] + __popc(k[0]);
        pre[2] = pre[1] + __popc(k[1]);
        pre[3] = pre[2] + __popc(k[2]);
        uint32_t ph = 0, my_slot = 0;
        bool my_keep = false;
#pragma unroll
        for (int u = 0; u < UN; ++u) {
            const uint32_t j = u * RP + r_in;
            const uint32_t kw = k[j >> 5], bit = j & 31;
            const bool kept = (kw >> bit) & 1u;
            const uint32_t slot = pre[j >> 5] + __popc(kw & ((1u << bit) - 1u));
            const uint64_t ox = xa[u] ^ xb, oz = za[u] ^ zb;
            ph |= ((uint32_t)(__popcll(ox & oz) + 2 * __popcll(xa[u] & zb)) & 3u) << (4 * u);
            if (kept) {
                uint64_t *o = out_xz + (size_t)slot * (2 * W) + c;
                __stcs(o, ox);
                __stcs(o + W, oz);
            }
            if ((int)c == u) {
                my_slot = slot;
                my_keep = kept;
            }
        }
#pragma unroll
        for (int o = W >> 1; o > 0; o >>= 1) ph = (ph + __shfl_xor_sync(0xffffffffu, ph, o)) & 0x33333333u;
        if ((int)c < UN && my_keep) {
            const int e = (int)(((ph + ya3) >> (4 * c)) + yb3) & 3;
            const double2 bc = Bc[qrow];
            double re, im;
            cmul(ac.x, ac.y, bc.x, bc.y, re, im);
            mul_i_pow(re, im, e);
            out_c[my_slot] = make_double2(re, im);
        }
    }
}

// group sums of the surviving heads -> their output slots (after tile_emit_kernel wrote a[p]*b[q]*i^e there)
__global__ void __launch_bounds__(256) tile_fixup_kernel(TileMap tm, RecFmt fmt, const uint64_t *__restrict__ sr, WorkList wl,
                                                          const uint8_t *__restrict__ multi, const double2 *__restrict__ acc,
                                                          double2 *__restrict__ out_c) {
    FOR_EACH_WORK(wl, i) {
        if (!multi[i]) continue;
        const uint32_t slot = tm.slot_of(fmt.t(sr[i]));
        if (slot != 0xffffffffu) out_c[slot] = acc[i];
    }
}

// worklist storage: L.slot and L.kept (adjacent, both unused in this mode) hold the regions, the
// radix histogram buffer (free once the sort is done) holds the counters
static WorkList tile_worklist(const DedupLayout &L, int64_t T) {
    const int64_t nb = (T + CLS_TILE - 1) / CLS_TILE;   // CTAs of tile_classify_kernel
    WorkList wl;
    wl.nreg = (uint32_t)std::max<int64_t>(1, std::min<int64_t>(2048, nb));
    wl.cap = (uint32_t)std::min<int64_t>(((nb + wl.nreg - 1) / wl.nreg) * CLS_TILE, T);
    wl.work = L.slot;
    wl.counts = L.hist;
    return wl;
}

int g_tile_qgroup = 16;   // tuning knob 7: B rows per CTA of tile_emit_kernel

int dedup_product_plan_tiles(uint64_t *recs, int64_t T, RecFmt fmt, const ProductRows &rows, const TileMap &tm, double thr,
                             int64_t *n_out, int64_t *n_out_host, void *ws, size_t ws_bytes, cudaStream_t st) {
    if (ws_bytes < dedup_ws_bytes(T)) {
        set_error("workspace too small: need %zu bytes, got %zu", dedup_ws_bytes(T), ws_bytes);
        return SYM_E_WORKSPACE;
    }
    DedupLayout L = dedup_layout(ws, ws_bytes, T);
    if (!L.ok) {
        set_error("workspace arena exhausted");
        return SYM_E_WORKSPACE;
    }
    const int begin = sort_begin_bit(T, fmt);
    uint64_t *sr = nullptr;
    SYM_TRY(radix_sort(recs, nullptr, L.alt, nullptr, T, begin, L.hist, &sr, st));
    const unsigned nb = (unsigned)((T + 255) / 256);
    ProductRows rows_sum = rows;
    if (thr >= 0.0 && rows.N > 0) {
        SYM_TRY(launch_min_abs_flag(reinterpret_cast<const double2 *>(rows.Ac), (int64_t)rows.M,
                                    reinterpret_cast<const double2 *>(rows.Bc), (int64_t)rows.N, thr,
                                    reinterpret_cast<unsigned long long *>(L.scratch), L.total + 2, st));
        rows_sum.pass_all = L.total + 2;
    }
    // worklist of the records that share a sort bucket
    const WorkList wl = tile_worklist(L, T);
    if ((size_t)wl.nreg * wl.cap > 2 * (arena_need((size_t)T, 4) / 4)) {
        set_error("worklist does not fit its arena slice");
        return SYM_E_WORKSPACE;
    }
    SYM_CUDA_OK(cudaMemsetAsync(wl.counts, 0, sizeof(uint32_t) * wl.nreg, st));
    tile_classify_kernel<ProductRows><<<(unsigned)((T + CLS_TILE - 1) / CLS_TILE), 256, 0, st>>>(rows_sum, fmt, sr, T, begin, thr,
                                                                                                tm, wl);
    SYM_LAUNCH_OK();
    link_work_kernel<ProductRows><<<wl.nreg * WORK_SPLIT, 256, 0, st>>>(rows, fmt, sr, begin, wl, L.flag, L.link);
    SYM_LAUNCH_OK();
    phase_work_kernel<ProductRows><<<wl.nreg * WORK_SPLIT, 256, 0, st>>>(rows, fmt, sr, wl, L.flag);
    SYM_LAUNCH_OK();
    sum_work_kernel<ProductRows><<<wl.nreg * WORK_SPLIT, 256, 0, st>>>(rows_sum, fmt, sr, T, begin, wl, L.flag, L.link, thr, L.acc, L.multi, tm);
    SYM_LAUNCH_OK();
    seg_count_kernel<<<(tm.n_seg + 255) / 256, 256, 0, st>>>(tm);
    SYM_LAUNCH_OK();
    SYM_TRY(scan_exclusive_u32(tm.segoff, tm.segoff, (int64_t)tm.n_seg, L.total, L.scratch, st));
    if (n_out) {
        total_to_i64_kernel<<<1, 1, 0, st>>>(L.total, n_out);
        SYM_LAUNCH_OK();
    }
    uint32_t U32 = 0;
    SYM_CUDA_OK(cudaMemcpyAsync(&U32, L.total, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    SYM_CUDA_OK(cudaStreamSynchronize(st));
    if (n_out_host) *n_out_host = (int64_t)U32;
    return SYM_OK;
}

// identity worklist over positions [*begin, *end) of the candidate array of the class mode (capacity T positions)
static WorkList class_worklist(const DedupLayout &L, int64_t T, const uint32_t *begin, const uint32_t *end) {
    const WorkList ref = tile_worklist(L, T);
    WorkList wl;
    wl.nreg = ref.nreg;
    wl.cap = ref.cap;
    wl.work = nullptr;
    wl.counts = nullptr;
    wl.begin_ptr = begin;
    wl.end_ptr = end;
    return wl;
}

// ---------------------------------------------------------------------------------------------
// Group pass of the class mode: exact duplicate resolution of the candidate array, one kernel.
// The array is a concatenation of runs sorted by (hash, enumeration order); a BUCKET is a maximal run of
// records with equal top hash bits. Eight lanes own a bucket: lane j holds 16-byte chunk j of the X block
// and of the Z block of a row, so one pass over the members compares rows word by word (the exact
// test: hash equality is only a filter), computes the phase exponent of every member (base.py:785-788)
// and adds the coefficients in array order — the reference's np.add.at order (utils.py:271-278) — with the
// commutative complex product, so anticommuting twins cancel to exact zero. Non-heads and heads whose sum
// fails |c| > thr set their drop bit; a surviving head leaves its sum in acc[] / multi[] for the fix-up after
// the emission. Buckets of more than 32 records (squares, molecular H*H) go to the generic worklist path
// (link / phase / sum kernels above). HBM/L2-bound: 512 B of operand rows per member, from L2.
// ---------------------------------------------------------------------------------------------
constexpr int GRP_MAX = 32;

// WIDE: W >= 2, lane j < W/2 holds words 2j, 2j+1 of the X block and of the Z block; else W == 1 and lane 0 holds the word
template <bool WIDE>
__device__ __forceinline__ void grp_load(const ProductRows &rows, uint32_t t, int j, bool active, uint64_t &ox0, uint64_t &ox1,
                                         uint64_t &oz0, uint64_t &oz1, uint32_t &ph) {
    ox0 = ox1 = oz0 = oz1 = 0ull;
    ph = 0;
    if (!active) return;
    uint32_t p, q;
    rows.split(t, p, q);
    const int W = rows.words >> 1;
    const uint64_t *ra = rows.A + (size_t)p * rows.words, *rb = rows.B + (size_t)q * rows.words;
    if (WIDE) {
        const uint4 xa = *reinterpret_cast<const uint4 *>(ra + 2 * j), za = *reinterpret_cast<const uint4 *>(ra + W + 2 * j);
        const uint4 xb = *reinterpret_cast<const uint4 *>(rb + 2 * j), zb = *reinterpret_cast<const uint4 *>(rb + W + 2 * j);
        const uint64_t xa0 = ((uint64_t)xa.y << 32) | xa.x, xa1 = ((uint64_t)xa.w << 32) | xa.z;
        const uint64_t za0 = ((uint64_t)za.y << 32) | za.x, za1 = ((uint64_t)za.w << 32) | za.z;
        const uint64_t xb0 = ((uint64_t)xb.y << 32) | xb.x, xb1 = ((uint64_t)xb.w << 32) | xb.z;
        const uint64_t zb0 = ((uint64_t)zb.y << 32) | zb.x, zb1 = ((uint64_t)zb.w << 32) | zb.z;
        ox0 = xa0 ^ xb0;
        ox1 = xa1 ^ xb1;
        oz0 = za0 ^ zb0;
        oz1 = za1 ^ zb1;
        ph = (uint32_t)(__popcll(ox0 & oz0) + __popcll(ox1 & oz1) + 2 * (__popcll(xa0 & zb0) + __popcll(xa1 & zb1)));
    } else {
        const uint64_t xa0 = ra[0], za0 = ra[1], xb0 = rb[0], zb0 = rb[1];
        ox0 = xa0 ^ xb0;
        oz0 = za0 ^ zb0;
        ph = (uint32_t)(__popcll(ox0 & oz0) + 2 * __popcll(xa0 & zb0));
    }
}

template <bool WIDE>
__global__ void __launch_bounds__(256) group_kernel(ProductRows rows, const int32_t *__restrict__ a_y, const int32_t *__restrict__ b_y,
                                                     RecFmt fmt, const uint64_t *__restrict__ sr, int sort_shift, WorkList wl,
                                                     double thr, double2 *__restrict__ acc, uint8_t *__restrict__ multi, TileMap tm,
                                                     WorkList big) {
    // The four lane groups of a warp work on four buckets in LOCKSTEP (uniform loops, per-group predicates):
    // divergent per-group loops would serialise the groups and quadruple the instruction count.
    const uint32_t FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, grp = lane >> 3, j = lane & 7;
    const int64_t lo = wl.lo(), hi = wl.hi(0);
    const int W = rows.words >> 1;
    const bool active = WIDE ? (2 * j < W) : (j == 0);
    const bool check_thr = !(thr < 0.0 || rows.all_pass());
    const int64_t nwin = (hi - lo + 31) / 32;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t win = warp0; win < nwin; win += nwarps) {
        const int64_t pos = lo + win * 32 + lane;
        const uint64_t rec = pos < hi ? sr[pos] : 0ull;
        uint64_t prev = __shfl_up_sync(FULL, rec, 1);
        if (lane == 0 && pos > lo) prev = sr[pos - 1];
        const bool start = pos < hi && (pos == lo || ((rec ^ prev) >> sort_shift) != 0ull);
        uint32_t starts = __ballot_sync(FULL, start);
        while (starts) {
            // the four lane groups take the next four bucket starts of the window
            uint32_t m = starts;
            int mine = -1;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                if (m) {
                    const int b = __ffs(m) - 1;
                    if (g == grp) mine = b;
                    m &= m - 1u;
                }
            }
            starts = m;
            const int64_t s = lo + win * 32 + (mine < 0 ? 0 : mine);
            const uint64_t r0 = mine < 0 ? 0ull : sr[s];
            // bucket length: the lanes of a group look at 8 positions at a time
            uint32_t g_len = mine < 0 ? 0u : 1u;
            bool open = mine >= 0;
            for (int64_t b0 = s + 1; __any_sync(FULL, open); b0 += 8) {
                const int64_t x = b0 + j;
                const bool in = open && x < hi && ((sr[x] ^ r0) >> sort_shift) == 0ull;
                const uint32_t out = (~(__ballot_sync(FULL, in) >> (8 * grp))) & 0xffu;
                const uint32_t run = out ? (uint32_t)(__ffs(out) - 1) : 8u;
                if (open) g_len += run;
                open = open && run == 8u;
            }
            if (g_len > (uint32_t)GRP_MAX) {   // long bucket (rare): its positions go on the generic list
                for (uint32_t x = j; x < g_len; x += 8) {
                    const uint32_t px = (uint32_t)(s + x);
                    const uint32_t r = (px / CLS_TILE) % big.nreg;
                    const uint32_t slot = atomicAdd(big.counts + r, 1u);
                    big.work[(size_t)r * big.cap + slot] = px;
                }
                g_len = 0;
            }
            // bit i of `todo`: member i of the bucket is neither a head yet nor merged into one
            uint32_t todo = g_len == 0u ? 0u : (g_len == 32u ? FULL : ((1u << g_len) - 1u));
            while (__any_sync(FULL, todo != 0u)) {
                const int h = todo ? __ffs(todo) - 1 : -1;
                if (h >= 0) todo &= todo - 1u;
                const uint64_t rh = h >= 0 ? sr[s + h] : 0ull;
                const uint32_t th = fmt.t(rh);
                uint64_t hx0, hx1, hz0, hz1;
                uint32_t ph_h;
                grp_load<WIDE>(rows, th, j, active && h >= 0, hx0, hx1, hz0, hz1, ph_h);
                ph_h += __shfl_xor_sync(FULL, ph_h, 1);
                ph_h += __shfl_xor_sync(FULL, ph_h, 2);
                ph_h += __shfl_xor_sync(FULL, ph_h, 4);
                double sre = 0.0, sim = 0.0;
                bool have = false;
                uint32_t pend = h >= 0 ? todo : 0u;   // later members that may be twins of this head
                while (__any_sync(FULL, pend != 0u)) {
                    const int mm = pend ? __ffs(pend) - 1 : -1;
                    if (mm >= 0) pend &= pend - 1u;
                    const uint64_t rm = mm >= 0 ? sr[s + mm] : 0ull;
                    const bool cmp = mm >= 0 && fmt.same_hash(rh, rm);
                    const uint32_t tmm = fmt.t(rm);
                    uint64_t ox0, ox1, oz0, oz1;
                    uint32_t ph_m;
                    grp_load<WIDE>(rows, tmm, j, active && cmp, ox0, ox1, oz0, oz1, ph_m);
                    const bool eq = (ox0 == hx0) & (ox1 == hx1) & (oz0 == hz0) & (oz1 == hz1);
                    const uint32_t eq_all = __ballot_sync(FULL, eq);   // every lane votes: never inside a short-circuit
                    const bool twin = cmp && ((eq_all >> (8 * grp)) & 0xffu) == 0xffu;
                    ph_m += __shfl_xor_sync(FULL, ph_m, 1);
                    ph_m += __shfl_xor_sync(FULL, ph_m, 2);
                    ph_m += __shfl_xor_sync(FULL, ph_m, 4);
                    if (twin) {
                        todo &= ~(1u << mm);
                        if (j == 0) {
                            uint32_t p, q;
                            if (!have) {   // the head's own term first (np.add.at order)
                                rows.split(th, p, q);
                                rows.coeff(th, (int)((ph_h + 3u * (uint32_t)(a_y[p] + b_y[q])) & 3u), sre, sim);
                            }
                            rows.split(tmm, p, q);
                            double cr, ci;
                            rows.coeff(tmm, (int)((ph_m + 3u * (uint32_t)(a_y[p] + b_y[q])) & 3u), cr, ci);
                            sre += cr;
                            sim += ci;
                            tm.mark_dropped(tmm);
                            multi[s + mm] = 0;
                        }
                        have = true;
                    }
                }
                if (j == 0 && h >= 0) {
                    multi[s + h] = 0;
                    if (have) {
                        if (keep_test(sre, sim, thr)) {
                            acc[s + h] = make_double2(sre, sim);
                            multi[s + h] = 1;
                        } else {
                            tm.mark_dropped(th);
                        }
                    } else if (check_thr) {
                        double re, im;
                        rows.coeff_unphased(th, re, im);
                        if (!keep_test(re, im, thr)) tm.mark_dropped(th);
                    }
                }
            }
        }
    }
}

// exact group pass over positions [*begin, *end) of the candidate array
static int class_group_pass(const ProductRows &rows, const ProductRows &rows_sum, const int32_t *a_y, const int32_t *b_y, RecFmt fmt,
                            uint64_t *sr, int64_t T, int sort_shift, const uint32_t *begin, const uint32_t *end,
                            const DedupLayout &L, double thr, const TileMap &tm, cudaStream_t st) {
    const WorkList wl = class_worklist(L, T, begin, end);
    // generic list for the long buckets: few regions (it is almost always empty, and its three kernels launch
    // WORK_SPLIT CTAs per region whether or not there is anything on it)
    WorkList big = tile_worklist(L, T);
    {
        const int64_t nb = (T + CLS_TILE - 1) / CLS_TILE;
        big.nreg = (uint32_t)std::max<int64_t>(1, std::min<int64_t>(64, nb));
        big.cap = (uint32_t)std::min<int64_t>(((nb + big.nreg - 1) / big.nreg) * CLS_TILE, T);
    }
    big.begin_ptr = begin;
    big.end_ptr = end;
    SYM_CUDA_OK(cudaMemsetAsync(big.counts, 0, sizeof(uint32_t) * big.nreg, st));
    const unsigned grid = (unsigned)std::min<int64_t>((T + 255) / 256, (int64_t)num_sms() * 16);
    if (rows.words >= 4)
        group_kernel<true><<<grid, 256, 0, st>>>(rows_sum, a_y, b_y, fmt, sr, sort_shift, wl, thr, L.acc, L.multi, tm, big);
    else
        group_kernel<false><<<grid, 256, 0, st>>>(rows_sum, a_y, b_y, fmt, sr, sort_shift, wl, thr, L.acc, L.multi, tm, big);
    SYM_LAUNCH_OK();
    // long buckets (rare): nearest earlier twin, phase stamps, sums in array order
    link_work_kernel<ProductRows><<<big.nreg * WORK_SPLIT, 256, 0, st>>>(rows, fmt, sr, sort_shift, big, L.flag, L.link);
    SYM_LAUNCH_OK();
    phase_work_kernel<ProductRows><<<big.nreg * WORK_SPLIT, 256, 0, st>>>(rows, fmt, sr, big, L.flag);
    SYM_LAUNCH_OK();
    sum_work_kernel<ProductRows><<<big.nreg * WORK_SPLIT, 256, 0, st>>>(rows_sum, fmt, sr, T, sort_shift, big, L.flag, L.link, thr,
                                                                        L.acc, L.multi, tm);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

// Class mode of the ordered-tile product (class_dedup.cu): no record array, no global sort. The candidate
// array (L.alt) holds, class by class, the records that have a same-hash mate, sorted by (hash, t); the
// group pass runs over all of them with device-side counts, so the common case (no class overflow) costs
// one stream synchronisation like the sort path. Overflowed classes take the global sort afterwards and
// are appended to the candidate array.
int dedup_product_plan_classes(uint64_t *recs, int64_t T, RecFmt fmt, const ProductRows &rows, const TileMap &tm, ClassJob &job,
                               const uint64_t *a_sk, const uint64_t *b_sk, const int32_t *a_y, const int32_t *b_y, void *class_ws,
                               size_t class_ws_bytes, double thr, int64_t *n_out, int64_t *n_out_host, void *ws, size_t ws_bytes,
                               cudaStream_t st) {
    if (ws_bytes < dedup_ws_bytes(T)) {
        set_error("workspace too small: need %zu bytes, got %zu", dedup_ws_bytes(T), ws_bytes);
        return SYM_E_WORKSPACE;
    }
    DedupLayout L = dedup_layout(ws, ws_bytes, T);
    if (!L.ok) {
        set_error("workspace arena exhausted");
        return SYM_E_WORKSPACE;
    }
    ProductRows rows_sum = rows;
    if (thr >= 0.0 && rows.N > 0) {
        SYM_TRY(launch_min_abs_flag(reinterpret_cast<const double2 *>(rows.Ac), (int64_t)rows.M,
                                    reinterpret_cast<const double2 *>(rows.Bc), (int64_t)rows.N, thr,
                                    reinterpret_cast<unsigned long long *>(L.scratch), L.total + 2, st));
        rows_sum.pass_all = L.total + 2;
    }
    uint32_t *counters = L.total + 8;
    uint64_t *cand = L.alt, *over = recs;
    SYM_TRY(class_dedup_run(job, a_sk, b_sk, rows_sum, tm, thr, cand, over, counters, class_ws, class_ws_bytes, st));
    const int sort_shift = 64 - job.hbits;
    SYM_TRY(class_group_pass(rows, rows_sum, a_y, b_y, fmt, cand, T, sort_shift, nullptr, counters, L, thr, tm, st));
    uint32_t host[12] = {0};
    for (int attempt = 0; attempt < 2; ++attempt) {
        seg_count_kernel<<<(tm.n_seg + 255) / 256, 256, 0, st>>>(tm);
        SYM_LAUNCH_OK();
        SYM_TRY(scan_exclusive_u32(tm.segoff, tm.segoff, (int64_t)tm.n_seg, L.total, L.scratch, st));
        SYM_CUDA_OK(cudaMemcpyAsync(host, L.total, sizeof(host), cudaMemcpyDeviceToHost, st));
        SYM_CUDA_OK(cudaStreamSynchronize(st));
        const uint32_t n_cand = host[8], n_over = host[9];
        if (attempt == 1 || n_over == 0u) break;
        // overflowed classes: global sort of their records on (hash, t), appended behind the candidates
        if ((int64_t)n_cand + (int64_t)n_over > T) {
            set_error("class dedup wrote more records than cross terms");
            return SYM_E_CUDA;
        }
        uint64_t *sorted = nullptr;
        SYM_TRY(radix_sort(over, nullptr, reinterpret_cast<uint64_t *>(L.slot), nullptr, (int64_t)n_over, 2, L.hist,
                           &sorted, st));
        SYM_CUDA_OK(cudaMemcpyAsync(cand + n_cand, sorted, sizeof(uint64_t) * (size_t)n_over, cudaMemcpyDeviceToDevice, st));
        SYM_TRY(class_ord_to_t(job, cand + n_cand, n_over, st));
        SYM_TRY(class_group_pass(rows, rows_sum, a_y, b_y, fmt, cand, T, sort_shift, counters, counters + 3, L, thr, tm, st));
    }
    if (n_out) {
        total_to_i64_kernel<<<1, 1, 0, st>>>(L.total, n_out);
        SYM_LAUNCH_OK();
    }
    if (n_out_host) *n_out_host = (int64_t)host[0];
    return SYM_OK;
}

int dedup_product_emit_tiles(const uint64_t *recs, int64_t T, RecFmt fmt, const ProductRows &rows, const TileMap &tm,
                             const TileBlock *blocks_host, const int32_t *a_y, const int32_t *b_y, int64_t U,
                             uint64_t *out_xz, double *out_c, void *ws, size_t ws_bytes, bool class_mode, cudaStream_t st) {
    if (T == 0 || U == 0) return SYM_OK;
    DedupLayout L = dedup_layout(ws, ws_bytes, T);
    if (!L.ok) {
        set_error("workspace arena exhausted");
        return SYM_E_WORKSPACE;
    }
    const uint64_t *sr = class_mode ? L.alt : ((T > 1 && sorted_in_alt(sort_begin_bit(T, fmt))) ? L.alt : recs);
    const int chunks = rows.words / 2;
    const double2 *Ac = reinterpret_cast<const double2 *>(rows.Ac), *Bc = reinterpret_cast<const double2 *>(rows.Bc);
    double2 *oc = reinterpret_cast<double2 *>(out_c);
    const uint32_t qg = (uint32_t)(g_tile_qgroup < 1 ? 1 : g_tile_qgroup);
    if (g_emit_ev0) SYM_CUDA_OK(cudaEventRecord(g_emit_ev0, st));
    uint32_t gx = 0, gy = 0;
    for (int b = 0; b < tm.nblk; ++b) {
        const TileBlock blk = blocks_host[b];
        if (blk.m_blk == 0 || blk.nq == 0) continue;
        gx = std::max(gx, blk.ptiles);
        gy = std::max(gy, (blk.nq + qg - 1) / qg);
    }
    if (gy > 65535 || tm.nblk > 65535) {
        set_error("too many B rows for one tile launch");
        return SYM_E_UNSUPPORTED;
    }
    if (gx > 0 && gy > 0) {
        dim3 grid(gx, gy, (unsigned)tm.nblk);
#define TILE_EMIT(LW) \
    tile_emit_kernel<LW><<<grid, (TILE_ROWS << LW) < 256 ? (TILE_ROWS << LW) : 256, 0, st>>>(                 \
        rows.A, Ac, a_y, rows.B, Bc, b_y, tm.first, tm.blocks, qg, tm.drop, tm.segoff, out_xz, oc)
        switch (chunks) {
            case 1: TILE_EMIT(0); break;
            case 2: TILE_EMIT(1); break;
            case 4: TILE_EMIT(2); break;
            case 8: TILE_EMIT(3); break;
            case 16: TILE_EMIT(4); break;
            default: set_error("ordered-tile mode needs 1, 2, 4, 8 or 16 words per block"); return SYM_E_UNSUPPORTED;
        }
#undef TILE_EMIT
        SYM_LAUNCH_OK();
    }
    if (g_emit_ev1) SYM_CUDA_OK(cudaEventRecord(g_emit_ev1, st));
    const WorkList wl = class_mode ? class_worklist(L, T, nullptr, L.total + 11) : tile_worklist(L, T);
    tile_fixup_kernel<<<wl.nreg * WORK_SPLIT, 256, 0, st>>>(tm, fmt, sr, wl, L.multi, L.acc, oc);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

int dedup_product_plan(uint64_t *recs, int64_t T, RecFmt fmt, const ProductRows &rows, bool by_t, double thr,
                       int64_t *n_out, int64_t *n_out_host, void *ws, size_t ws_bytes, cudaStream_t st) {
    if (by_t) return dedup_plan<ProductRows, true>(recs, T, fmt, rows, thr, n_out, n_out_host, ws, ws_bytes, st);
    return dedup_plan<ProductRows, false>(recs, T, fmt, rows, thr, n_out, n_out_host, ws, ws_bytes, st);
}

int dedup_product_emit(const uint64_t *recs, int64_t T, RecFmt fmt, const ProductRows &rows, bool by_t, int64_t U,
                       uint64_t *out_xz, double *out_c, void *ws, size_t ws_bytes, cudaStream_t st) {
    if (by_t) return dedup_emit<ProductRows, true>(recs, T, fmt, rows, U, out_xz, out_c, ws, ws_bytes, st);
    return dedup_emit<ProductRows, false>(recs, T, fmt, rows, U, out_xz, out_c, ws, ws_bytes, st);
}

int dedup_plain_plan(uint64_t *recs, int64_t T, RecFmt fmt, const PlainRows &rows, double thr, int64_t *n_out,
                     int64_t *n_out_host, void *ws, size_t ws_bytes, cudaStream_t st) {
    return dedup_plan<PlainRows, true>(recs, T, fmt, rows, thr, n_out, n_out_host, ws, ws_bytes, st);
}

int dedup_plain_emit(const uint64_t *recs, int64_t T, RecFmt fmt, const PlainRows &rows, int64_t U, uint64_t *out_xz,
                     double *out_c, void *ws, size_t ws_bytes, cudaStream_t st) {
    return dedup_emit<PlainRows, true>(recs, T, fmt, rows, U, out_xz, out_c, ws, ws_bytes, st);
}

// records of stored rows: hash of the row sketch, t = row index, e = 0
__global__ void __launch_bounds__(256) plain_records_kernel(const uint64_t *__restrict__ xz, int64_t T, int words, uint64_t mask,
                                                             RecFmt fmt, uint64_t *__restrict__ recs) {
    const int lane = threadIdx.x & 31;
    int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= T) return;
    uint64_t h = warp_sketch_row(xz + row * words, words, lane);
    if (lane == 0) recs[row] = fmt.make(mix64(h) & mask, (uint64_t)row, 0);
}

__global__ void __launch_bounds__(256) plain_records8_kernel(const uint64_t *__restrict__ xz, int64_t T, int words, uint64_t mask,
                                                              RecFmt fmt, uint64_t *__restrict__ recs) {
    const int lane = threadIdx.x & 31;
    int64_t row = ((((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) << 2) + (lane >> 3);
    const bool ok = row < T;
    uint64_t h = group8_sketch_row(xz + (ok ? row : 0) * words, words, lane & 7);
    if (ok && (lane & 7) == 0) recs[row] = fmt.make(mix64(h) & mask, (uint64_t)row, 0);
}

}  // namespace symb

using namespace symb;

extern "C" size_t sym_cleanup_ws_bytes(int64_t T, int32_t W) {
    (void)W;
    if (T < 1) T = 1;
    return dedup_ws_bytes(T) + arena_need((size_t)T, 8) + 1024;
}

static int cleanup_check(int64_t T, int32_t W, size_t ws_bytes) {
    SYM_REQUIRE(T >= 0 && T < (int64_t)4000000000LL, "T out of range");
    SYM_REQUIRE(W >= 1, "W must be >= 1");
    if (T > 0 && ws_bytes < sym_cleanup_ws_bytes(T, W)) {
        set_error("workspace too small");
        return SYM_E_WORKSPACE;
    }
    return SYM_OK;
}

extern "C" int sym_cleanup_count(const uint64_t *xz, const double *c, int64_t T, int32_t W, double zero_threshold,
                                 int64_t *n_out, int64_t *n_out_host, void *ws, size_t ws_bytes, void *stream) {
    SYM_TRY(cleanup_check(T, W, ws_bytes));
    cudaStream_t st = (cudaStream_t)stream;
    if (T == 0) {
        if (n_out) SYM_CUDA_OK(cudaMemsetAsync(n_out, 0, sizeof(int64_t), st));
        if (n_out_host) *n_out_host = 0;
        return SYM_OK;
    }
    Arena ar(ws, ws_bytes);
    uint64_t *recs = ar.take<uint64_t>((size_t)T);
    RecFmt fmt{t_bits_for(T)};
    if (group8_ok(W))
        plain_records8_kernel<<<(unsigned)((((T + 3) / 4) * 32 + 255) / 256), 256, 0, st>>>(xz, T, 2 * W, g_key_mask, fmt, recs);
    else
        plain_records_kernel<<<(unsigned)((T * 32 + 255) / 256), 256, 0, st>>>(xz, T, 2 * W, g_key_mask, fmt, recs);
    SYM_LAUNCH_OK();
    PlainRows rows{xz, c, 2 * W};
    return dedup_plain_plan(recs, T, fmt, rows, zero_threshold, n_out, n_out_host, ar.base + ar.off, ws_bytes - ar.off, st);
}

extern "C" int sym_cleanup_emit(const uint64_t *xz, const double *c, int64_t T, int32_t W, int64_t U, uint64_t *out_xz,
                                double *out_c, void *ws, size_t ws_bytes, void *stream) {
    SYM_TRY(cleanup_check(T, W, ws_bytes));
    if (T == 0 || U == 0) return SYM_OK;
    Arena ar(ws, ws_bytes);
    uint64_t *recs = ar.take<uint64_t>((size_t)T);
    RecFmt fmt{t_bits_for(T)};
    PlainRows rows{xz, c, 2 * W};
    return dedup_plain_emit(recs, T, fmt, rows, U, out_xz, out_c, ar.base + ar.off, ws_bytes - ar.off,
                            (cudaStream_t)stream);
}

extern "C" int sym_cleanup(const uint64_t *xz, const double *c, int64_t T, int32_t W, double zero_threshold,
                           uint64_t *out_xz, double *out_c, int64_t out_capacity, int64_t *n_out, int64_t *n_out_host,
                           void *ws, size_t ws_bytes, void *stream) {
    int64_t U = 0;
    SYM_TRY(sym_cleanup_count(xz, c, T, W, zero_threshold, n_out, &U, ws, ws_bytes, stream));
    if (n_out_host) *n_out_host = U;
    if (U > out_capacity) {
        set_error("output capacity %lld < %lld surviving terms", (long long)out_capacity, (long long)U);
        return SYM_E_CAPACITY;
    }
    return sym_cleanup_emit(xz, c, T, W, U, out_xz, out_c, ws, ws_bytes, stream);
}
