// Class-local duplicate detection for large products (ordered-tile mode) — replaces the global radix
// sort of one 8-byte record per cross term (symmer/operators/utils.py:271, qiskit `unordered_unique`).
//
// The row sketch is GF(2)-linear, so any fixed set of its bits is a linear CLASS function:
//   class(A[p] ^ B[q]) = class(A[p]) ^ class(B[q]).
// With the rows of A grouped by class, the cross terms of class c are exactly the pairs
// (p in A_a, q) with a = class(B[q]) ^ c — they can be ENUMERATED from two small L2-resident tables, and
// equal rows (equal sketches) always fall into the same class. One CTA therefore owns one class
// (~4000 cross terms): it lists the class's pairs in shared memory, hashes them into a shared-memory
// table with plain stores (multi-round "last writer wins", no atomics) and learns which records have a
// same-hash mate. Records without one are unique rows: nothing is written for them, no record of theirs
// ever reaches HBM. Records with a mate (true duplicates, or the rare hash collision) are sorted by
// (hash, t) inside the CTA and appended to the candidate array, which the exact group pass (link / phase /
// sum in dedup.cu: word-by-word row compare, np.add.at order) consumes. A class that does not fit
// the CTA (heavily duplicated or low-dimensional operands) spills its records to the overflow array,
// which takes the ordinary global sort. No tensor cores: integer/bit work on L2-resident tables,
// shared-memory bound.
#include <algorithm>
#include <type_traits>

#include "rows.cuh"
#include "sort.cuh"

namespace symb {

// GF(2)-linear in the sketch (XOR of shifted copies); independent of the parity functionals of owner.cu
__host__ __device__ __forceinline__ uint32_t cd_class_of(uint64_t sk, int k) {
    const uint64_t y = sk ^ (sk >> 21) ^ (sk >> 43);
    return (uint32_t)(y >> 5) & ((1u << k) - 1u);
}

// ------------------------------------------------------------------------------------------------
// class tables. Table index of (block b, class a) = (b << (k + 1)) | a: XOR with a class only touches the low k bits.
// Both operands are grouped by (block, class):
//   look8 / lookp  rows of A: sketch and row index p; off[i] = first row of (block, class) i, off[tab] = rows of A
//   bits           bit i set <=> (block, class) i of A is not empty — about half of the visits end at this bit
//   vkey / vq / vsk  rows of B in (block, class) order ("visits"): table index, row index q, sketch
// Visiting B in class order keeps the lookups of neighbouring visits in neighbouring table entries.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int cd_block_of(const uint32_t *base, int nblk, uint32_t e) {
    int b = 0;
    while (b + 1 < nblk && e >= base[b + 1]) ++b;
    return b;
}

// cnt[0, tab): rows of A per table index; cnt[tab, 2 tab): rows of B per table index
__global__ void __launch_bounds__(256) cd_hist_kernel(ClassJob J, const uint64_t *__restrict__ a_sk, uint32_t *__restrict__ cnt,
                                                       uint32_t tab, uint32_t n_rows_a) {   // n_rows_a: J.n_entries, or 0 (done elsewhere)
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n_rows_a) {
        const int b = cd_block_of(J.entry_base, J.nblk, e);
        const uint32_t p = J.p0[b] + (e - J.entry_base[b]);
        atomicAdd(cnt + (((uint32_t)b << (J.k + 1)) | cd_class_of(a_sk[p], J.k)), 1u);
    }
    if (e < J.n_visits) {
        const int b = cd_block_of(J.visit_base, J.nblk, e);
        const uint32_t q = J.q0[b] + (e - J.visit_base[b]);
        atomicAdd(cnt + tab + (((uint32_t)b << (J.k + 1)) | cd_class_of(J.b_sk[q], J.k)), 1u);
    }
}

// off = exclusive scan of cnt over both halves, so off[tab + i] - n_entries = first visit of table index i
__global__ void __launch_bounds__(256) cd_place_kernel(ClassJob J, const uint64_t *__restrict__ a_sk, const uint32_t *__restrict__ off,
                                                        uint32_t *__restrict__ cursor, uint32_t tab, uint64_t *__restrict__ look8,
                                                        uint32_t *__restrict__ lookp, uint32_t *__restrict__ vkey,
                                                        uint32_t *__restrict__ vq, uint64_t *__restrict__ vsk,
                                                        uint32_t *__restrict__ bits, uint32_t n_visits_padded, uint32_t n_rows_a) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= J.n_visits && e < n_visits_padded) vkey[e] = 1u << J.k;   // never matches: classes stop at 2^k - 1
    if (e < n_rows_a) {
        const int b = cd_block_of(J.entry_base, J.nblk, e);
        const uint32_t p = J.p0[b] + (e - J.entry_base[b]);
        const uint64_t sk = a_sk[p];
        const uint32_t key = ((uint32_t)b << (J.k + 1)) | cd_class_of(sk, J.k);
        const uint32_t pos = off[key] + atomicAdd(cursor + key, 1u);
        look8[pos] = sk;
        lookp[pos] = p;
    }
    if (e < J.n_visits) {
        const int b = cd_block_of(J.visit_base, J.nblk, e);
        const uint32_t q = J.q0[b] + (e - J.visit_base[b]);
        const uint64_t sk = J.b_sk[q];
        const uint32_t key = ((uint32_t)b << (J.k + 1)) | cd_class_of(sk, J.k);
        const uint32_t pos = off[tab + key] - J.n_entries + atomicAdd(cursor + tab + key, 1u);
        vkey[pos] = key;
        vq[pos] = q;
        vsk[pos] = sk;
    }
    if (e < (tab + 31) / 32) {
        uint32_t w = 0;
        for (uint32_t i = 0; i < 32; ++i) {
            const uint32_t t = e * 32 + i;
            if (t < tab && off[t + 1] > off[t]) w |= 1u << i;
        }
        bits[e] = w;
    }
}

// Many rows per table entry (a rotation as a block-list product: 1e7 rows of A over a few thousand classes): the global
// atomics of the two kernels above would pile up on the same counters. These forms privatise the counters per CTA in
// shared memory: a CTA owns CD_CHUNK consecutive rows of A, counts them in shared memory and touches every global
// counter at most once.
constexpr uint32_t CD_CHUNK = 65536;

__global__ void __launch_bounds__(1024) cd_hist_priv_kernel(ClassJob J, const uint64_t *__restrict__ a_sk, uint32_t *__restrict__ cnt,
                                                             uint32_t tab) {
    extern __shared__ uint32_t cd_priv[];
    for (uint32_t i = threadIdx.x; i < tab; i += blockDim.x) cd_priv[i] = 0u;
    __syncthreads();
    const uint32_t e0 = blockIdx.x * CD_CHUNK, e1 = min(J.n_entries, e0 + CD_CHUNK);
    for (uint32_t e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
        const int b = cd_block_of(J.entry_base, J.nblk, e);
        const uint32_t p = J.p0[b] + (e - J.entry_base[b]);
        atomicAdd(cd_priv + (((uint32_t)b << (J.k + 1)) | cd_class_of(a_sk[p], J.k)), 1u);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < tab; i += blockDim.x)
        if (cd_priv[i]) atomicAdd(cnt + i, cd_priv[i]);
}

__global__ void __launch_bounds__(1024) cd_place_priv_kernel(ClassJob J, const uint64_t *__restrict__ a_sk,
                                                              const uint32_t *__restrict__ off, uint32_t *__restrict__ cursor,
                                                              uint32_t tab, uint64_t *__restrict__ look8, uint32_t *__restrict__ lookp) {
    extern __shared__ uint32_t cd_priv[];
    uint32_t *count = cd_priv, *base = cd_priv + tab;
    for (uint32_t i = threadIdx.x; i < tab; i += blockDim.x) count[i] = 0u;
    __syncthreads();
    const uint32_t e0 = blockIdx.x * CD_CHUNK, e1 = min(J.n_entries, e0 + CD_CHUNK);
    for (uint32_t e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
        const int b = cd_block_of(J.entry_base, J.nblk, e);
        const uint32_t p = J.p0[b] + (e - J.entry_base[b]);
        atomicAdd(count + (((uint32_t)b << (J.k + 1)) | cd_class_of(a_sk[p], J.k)), 1u);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < tab; i += blockDim.x) {
        base[i] = count[i] ? off[i] + atomicAdd(cursor + i, count[i]) : 0u;   // this CTA's range of the entry
        count[i] = 0u;
    }
    __syncthreads();
    for (uint32_t e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
        const int b = cd_block_of(J.entry_base, J.nblk, e);
        const uint32_t p = J.p0[b] + (e - J.entry_base[b]);
        const uint64_t sk = a_sk[p];
        const uint32_t key = ((uint32_t)b << (J.k + 1)) | cd_class_of(sk, J.k);
        const uint32_t pos = base[key] + atomicAdd(count + key, 1u);
        look8[pos] = sk;
        lookp[pos] = p;
    }
}

// ------------------------------------------------------------------------------------------------
// the class kernel
// ------------------------------------------------------------------------------------------------
// Records are ordered by their position in the block-major enumeration of the cross terms (block, then q, then p)
// — for a single block that IS t = q*M + p, the reference's order (base.py:783-792); for a block list it is the
// order in which the tiled emission writes the survivors. ord <-> t:
__device__ __forceinline__ uint32_t cd_ord_of(const ClassJob &J, int b, uint32_t p, uint32_t q) {
    return J.rec_off[b] + (q - J.q0[b]) * J.m_blk[b] + (p - J.p0[b]);
}
__device__ __forceinline__ uint32_t cd_t_of_ord(const ClassJob &J, uint32_t ord) {
    const int b = J.nblk == 1 ? 0 : cd_block_of(J.rec_off, J.nblk, ord);
    const uint32_t local = ord - J.rec_off[b];
    const uint32_t ql = local / J.m_blk[b];
    return (J.q0[b] + ql) * J.M_total + J.p0[b] + (local - ql * J.m_blk[b]);
}

constexpr int CD_VPT = 12;          // consecutive visits per thread and chunk (a multiple of 4: 16-byte key loads)
constexpr int CD_MAX_THREADS = 1024;
// vkey is padded to whole chunks of the largest CTA with keys that never match: entry K of block 0 is the (empty) end marker
static inline size_t cd_padded_visits(uint32_t n_visits) {
    const size_t chunk = (size_t)CD_MAX_THREADS * CD_VPT;
    return ((size_t)n_visits + chunk - 1) / chunk * chunk + chunk;
}

// Block-wide exclusive prefix of one value per thread (three barriers); *carry accumulates the block total.
template <int THREADS>
__device__ __forceinline__ uint32_t cd_block_prefix(uint32_t x, uint32_t *s_warp, uint32_t *carry, uint32_t &running_total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        const uint32_t t = lane < THREADS / 32 ? s_warp[lane] : 0u;
        uint32_t ti = t;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, ti, o);
            if (lane >= o) ti += y;
        }
        s_warp[lane] = ti - t;
        if (lane == 31) s_warp[32] = *carry + ti;   // the new carry, stored once everyone has read the old one
    }
    __syncthreads();
    const uint32_t base = *carry + s_warp[wid] + inc - x;
    running_total = s_warp[32];
    __syncthreads();
    if (threadIdx.x == 0) *carry = running_total;
    return base;
}

// Enumerates the pairs of class c: every row q of B (all blocks) looks up the rows of A whose class is
// class(B[q]) ^ c. A thread owns VPT consecutive visits; per chunk of THREADS * VPT visits: count the pairs of the
// own visits (one bit test per visit, the two table words of the non-empty ones), one block-wide prefix sum hands
// every thread a private range of the list, then it writes its pairs — no atomics, no warp votes, and the list
// ends up in visit order. OVER = false: pairs (entry of A, visit) go to the shared-memory list (beyond CAP they are
// only counted); OVER = true: the records themselves go to the overflow array at over_base.
__device__ __forceinline__ void cd_store_pair(uint2 *pairs, uint32_t pos, uint32_t lo, uint32_t v, int) { pairs[pos] = make_uint2(lo, v); }
__device__ __forceinline__ void cd_store_pair(uint32_t *pairs, uint32_t pos, uint32_t lo, uint32_t v, int vbits) {
    pairs[pos] = (lo << vbits) | v;
}

template <int THREADS, int CAP, bool OVER, typename PairT = uint2>
__device__ __forceinline__ void cd_enumerate(const ClassJob &J, uint32_t c, const uint32_t *bm, bool bm_shared, uint32_t *s_count,
                                             uint32_t *s_warp, PairT *pairs, uint64_t *__restrict__ over, uint32_t over_base,
                                             int vbits = 0) {
    constexpr int VPT = CD_VPT;
    const int tid = threadIdx.x;
    for (uint32_t v0 = 0; v0 < J.n_visits; v0 += THREADS * VPT) {   // vkey is padded with never-matching keys to whole chunks
        const uint32_t vb = v0 + tid * VPT;
        uint32_t key[VPT];
        const uint4 *src = reinterpret_cast<const uint4 *>(J.vkey + vb);
#pragma unroll
        for (int g = 0; g < VPT / 4; ++g) {
            const uint4 w = __ldg(src + g);
            key[4 * g] = w.x;
            key[4 * g + 1] = w.y;
            key[4 * g + 2] = w.z;
            key[4 * g + 3] = w.w;
        }
        uint32_t lo[VPT], n[VPT];
        uint32_t sum = 0;
#pragma unroll
        for (int u = 0; u < VPT; ++u) {
            const uint32_t idx = key[u] ^ c;
            const uint32_t w = bm_shared ? bm[idx >> 5] : __ldg(J.bits + (idx >> 5));
            lo[u] = 0;
            n[u] = 0;
            if ((w >> (idx & 31u)) & 1u) {
                lo[u] = __ldg(J.off + idx);
                n[u] = __ldg(J.off + idx + 1) - lo[u];
            }
            sum += n[u];
        }
        uint32_t running;
        uint32_t pos = cd_block_prefix<THREADS>(sum, s_warp, s_count, running);
        if (sum == 0u) continue;
        if (!OVER) {
            if (running <= (uint32_t)CAP) {   // block-uniform: the whole chunk fits, no bound checks
#pragma unroll
                for (int u = 0; u < VPT; ++u) {   // predicated stores for the common counts (no divergent branches), a loop beyond
                    const uint32_t v = vb + u, nn = n[u];
                    if (nn > 0u) cd_store_pair(pairs, pos, lo[u], v, vbits);
                    if (nn > 1u) cd_store_pair(pairs, pos + 1, lo[u] + 1, v, vbits);
                    if (nn > 2u) cd_store_pair(pairs, pos + 2, lo[u] + 2, v, vbits);
                    if (nn > 3u) cd_store_pair(pairs, pos + 3, lo[u] + 3, v, vbits);
                    for (uint32_t j = 4; j < nn; ++j) cd_store_pair(pairs, pos + j, lo[u] + j, v, vbits);
                    pos += nn;
                }
            } else {
#pragma unroll
                for (int u = 0; u < VPT; ++u) {
                    const uint32_t v = vb + u;
                    for (uint32_t j = 0; j < n[u]; ++j, ++pos)
                        if (pos < (uint32_t)CAP) cd_store_pair(pairs, pos, lo[u] + j, v, vbits);
                }
            }
        } else {
#pragma unroll
            for (int u = 0; u < VPT; ++u) {
                if (n[u] == 0u) continue;
                const uint32_t v = vb + u;
                const uint64_t skq = J.vsk[v];
                const uint32_t q = J.vq[v];
                for (uint32_t j = 0; j < n[u]; ++j, ++pos) {
                    const uint64_t hm = mix64(J.look8[lo[u] + j] ^ skq) & J.key_mask;
                    const uint64_t ord = cd_ord_of(J, (int)(key[u] >> (J.k + 1)), J.lookp[lo[u] + j], q);
                    over[(size_t)over_base + pos] = (((hm & ~0xffffull) >> (J.tb + 2)) << (J.tb + 2)) | (ord << 2);
                }
            }
        }
    }
}

// slot of a record in round r: a function of its 48 hash bits only (records with equal hash bits share their whole
// slot sequence, which is what makes the mate detection complete). xk = the hash bits folded to 32.
__device__ __forceinline__ uint32_t cd_fold(uint64_t ent) {
    return (uint32_t)(ent >> 32) ^ ((uint32_t)(ent >> 16) & 0xffffu) * 0x9E3779B1u;
}

constexpr int CD_BM_WORDS = 2048;
constexpr int CD32_BM_WORDS = 5120; // the same for the compact kernel (20 KB: 8 blocks of 2^14 table entries)
constexpr int CD_SMALL_GROUP = 16;  // hash groups up to this size are ordered by insertion inside the class kernel   // shared-memory copy of the non-empty bitmap when the table has <= 65536 entries

// counters: [0] candidates written, [1] overflow records written, [2] overflowed classes, [3] = [0] + [1] (set afterwards)
template <int THREADS, int CAP, int LOG_SLOTS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB) class_dedup_kernel(ClassJob J, ProductRows rows, TileMap tm, double thr,
                                                                     uint64_t *__restrict__ cand, uint64_t *__restrict__ over,
                                                                     uint32_t *__restrict__ counters, uint32_t c0, uint32_t c1) {
    constexpr int SLOTS = 1 << LOG_SLOTS;
    constexpr int RPT = CAP / THREADS;
    static_assert(CAP % THREADS == 0 && CAP <= 65536 && CAP <= SLOTS, "record ids are 16 bits; candidates are sorted inside the table");
    static_assert(RPT <= 16, "one state bit per record in a register");
    extern __shared__ __align__(16) unsigned char cd_smem[];
    uint64_t *table = reinterpret_cast<uint64_t *>(cd_smem);
    uint2 *pairs = reinterpret_cast<uint2 *>(cd_smem + (size_t)SLOTS * 8);
    uint8_t *mate = cd_smem + (size_t)SLOTS * 8 + (size_t)CAP * 8;
    uint32_t *s_bits = reinterpret_cast<uint32_t *>(cd_smem + (size_t)SLOTS * 8 + (size_t)CAP * 8 + CAP);
    __shared__ uint32_t s_count, s_ncand, s_base;
    __shared__ uint32_t s_warp[33];
    const int tid = threadIdx.x, lane = tid & 31;
    const uint32_t lt = (1u << lane) - 1u;
    const bool check_thr = !(thr < 0.0 || rows.all_pass());
    const uint32_t bm_words = (((uint32_t)J.nblk << (J.k + 1)) + 31u) / 32u;
    const bool bm_shared = bm_words <= (uint32_t)CD_BM_WORDS;
    if (bm_shared)
        for (uint32_t i = tid; i < bm_words; i += THREADS) s_bits[i] = J.bits[i];

    for (uint32_t c = c0 + blockIdx.x; c < c1; c += gridDim.x) {
        if (tid == 0) {
            s_count = 0;
            s_ncand = 0;
        }
        for (int i = tid; i < CAP / 4; i += THREADS) reinterpret_cast<uint32_t *>(mate)[i] = 0u;
        __syncthreads();
        cd_enumerate<THREADS, CAP, false, uint2>(J, c, s_bits, bm_shared, &s_count, s_warp, pairs, nullptr, 0u);
        __syncthreads();
        const uint32_t total = s_count;
        if (total > (uint32_t)CAP) {   // the class does not fit: its records take the global sort
            __syncthreads();           // everyone has read s_count
            if (tid == 0) {
                s_base = atomicAdd(counters + 1, total);
                atomicAdd(counters + 2, 1u);
                s_count = 0;
            }
            __syncthreads();
            cd_enumerate<THREADS, CAP, true, uint2>(J, c, s_bits, bm_shared, &s_count, s_warp, (uint2 *)nullptr, over, s_base);
            __syncthreads();
            continue;
        }
        // ---- records of this thread: [hash : 48 | local id : 16]; neighbouring lanes hold neighbouring list entries,
        // i.e. neighbouring visits and table entries
        uint64_t ent[RPT];
        uint32_t xk[RPT];
        uint32_t rr[RPT];                          // local id of the record that represents this record's hash group
        uint32_t unres = 0, candm = 0, winm = 0;   // one bit per record: no slot yet / saw a same-hash record / holds a slot
#pragma unroll
        for (int j = 0; j < RPT; ++j) {
            const uint32_t i = tid + j * THREADS;
            ent[j] = 0;
            xk[j] = 0;
            rr[j] = i;
            if (i < total) {
                const uint2 pr = pairs[i];
                const uint64_t hm = mix64(__ldg(J.look8 + pr.x) ^ __ldg(J.vsk + pr.y)) & J.key_mask;
                ent[j] = (hm & ~0xffffull) | i;
                xk[j] = cd_fold(ent[j]);
                unres |= 1u << j;
            }
        }
        for (int round = 0; round < CD_MAX_ROUNDS; ++round) {
            const uint32_t mult = 0x9E3779B1u + 2u * (uint32_t)round * 0x632BE5ABu;   // odd for every round
            const uint32_t add = (uint32_t)round * 0x7F4A7C15u;
            if (unres) {
#pragma unroll
                for (int j = 0; j < RPT; ++j)
                    if ((unres >> j) & 1u) table[(xk[j] * mult + add) >> (32 - LOG_SLOTS)] = ent[j];
            }
            if (!__syncthreads_or(unres != 0u)) break;
            if (unres) {
#pragma unroll
                for (int j = 0; j < RPT; ++j) {
                    if ((unres >> j) & 1u) {
                        const uint64_t v = table[(xk[j] * mult + add) >> (32 - LOG_SLOTS)];
                        if (v == ent[j]) {
                            winm |= 1u << j;
                            unres &= ~(1u << j);
                        } else if (((v ^ ent[j]) >> 16) == 0ull) {
                            rr[j] = (uint32_t)(v & 0xffffull);
                            mate[rr[j]] = 1;
                            candm |= 1u << j;
                            unres &= ~(1u << j);
                        }
                    }
                }
            }
            __syncthreads();
        }
        // ---- candidates: saw a mate, was seen by one, or never found a free slot (then its mates did not either)
        candm |= unres;
#pragma unroll
        for (int j = 0; j < RPT; ++j)
            if (((winm >> j) & 1u) && mate[tid + j * THREADS] != 0) candm |= 1u << j;
        if (check_thr) {   // unique rows survive unless their own coefficient fails the threshold
#pragma unroll
            for (int j = 0; j < RPT; ++j) {
                const uint32_t i = tid + j * THREADS;
                if (i < total && !((candm >> j) & 1u)) {
                    const uint2 pr = pairs[i];
                    const uint32_t t = J.vq[pr.y] * J.M_total + J.lookp[pr.x];
                    double re, im;
                    rows.coeff_unphased(t, re, im);
                    if (!keep_test(re, im, thr)) tm.mark_dropped(t);
                }
            }
        }
        if (__syncthreads_or(candm != 0u)) {
            // Candidates leave grouped by hash, each group in enumeration order. Fast path: counting sort by the
            // group representative (one shared-memory atomic per candidate hands out its rank in the group), then
            // the thread that owns the representative orders the (2-3 member) group by insertion. A class with a
            // group of more than CD_SMALL_GROUP records, or with records that never found a slot, takes a bitonic
            // sort of all its candidates instead.
            uint32_t *cnt = reinterpret_cast<uint32_t *>(table);   // CAP words, then CAP keys
            uint64_t *outk = table + CAP / 2;
            for (int i = tid; i < CAP; i += THREADS) cnt[i] = 0u;
            __syncthreads();
            bool slow = (candm & unres) != 0u;
#pragma unroll
            for (int j = 0; j < RPT; ++j)
                if (((candm & ~unres) >> j) & 1u) rr[j] |= atomicAdd(cnt + rr[j], 1u) << 16;
            __syncthreads();
            uint32_t co[RPT];   // groups represented by this thread's records: [count : 16 | offset : 16]
            uint32_t sum = 0;
#pragma unroll
            for (int j = 0; j < RPT; ++j) {
                co[j] = cnt[tid + j * THREADS];
                slow |= co[j] > (uint32_t)CD_SMALL_GROUP;
                sum += co[j];
            }
            if (!__syncthreads_or(slow)) {
                uint32_t running;
                uint32_t base = cd_block_prefix<THREADS>(sum, s_warp, &s_ncand, running);
#pragma unroll
                for (int j = 0; j < RPT; ++j) {
                    cnt[tid + j * THREADS] = base;
                    const uint32_t c = co[j];
                    co[j] = (c << 16) | base;
                    base += c;
                }
                __syncthreads();
#pragma unroll
                for (int j = 0; j < RPT; ++j) {
                    if ((candm >> j) & 1u) {
                        const uint2 pr = pairs[tid + j * THREADS];
                        const int b = J.nblk == 1 ? 0 : (int)(J.vkey[pr.y] >> (J.k + 1));
                        outk[cnt[rr[j] & 0xffffu] + (rr[j] >> 16)] =
                            ((ent[j] >> (64 - J.hbits)) << 32) | cd_ord_of(J, b, J.lookp[pr.x], J.vq[pr.y]);
                    }
                }
                __syncthreads();
#pragma unroll
                for (int j = 0; j < RPT; ++j) {
                    const uint32_t c = co[j] >> 16;
                    if (c >= 2u) {
                        uint64_t *seg = outk + (co[j] & 0xffffu);
                        for (uint32_t a = 1; a < c; ++a) {
                            const uint64_t key = seg[a];
                            uint32_t bpos = a;
                            while (bpos > 0 && seg[bpos - 1] > key) {
                                seg[bpos] = seg[bpos - 1];
                                --bpos;
                            }
                            seg[bpos] = key;
                        }
                    }
                }
                __syncthreads();
            } else {
                outk = table;
#pragma unroll
                for (int j = 0; j < RPT; ++j) {
                    const bool cnd = (candm >> j) & 1u;
                    const uint32_t bal = __ballot_sync(0xffffffffu, cnd);
                    uint32_t base = 0;
                    if (bal != 0u) {
                        if (lane == 0) base = atomicAdd(&s_ncand, (uint32_t)__popc(bal));
                        base = __shfl_sync(0xffffffffu, base, 0);
                    }
                    if (cnd) {
                        const uint2 pr = pairs[tid + j * THREADS];
                        const int b = J.nblk == 1 ? 0 : (int)(J.vkey[pr.y] >> (J.k + 1));
                        table[base + __popc(bal & lt)] = ((ent[j] >> (64 - J.hbits)) << 32) | cd_ord_of(J, b, J.lookp[pr.x], J.vq[pr.y]);
                    }
                }
                __syncthreads();
                const uint32_t n_all = s_ncand;
                uint32_t np = 2;
                while (np < n_all) np <<= 1;
                for (uint32_t i = n_all + tid; i < np; i += THREADS) table[i] = ~0ull;
                // bitonic sort of [hash | ord]: equal-hash records become neighbours, in enumeration order
                for (uint32_t size = 2; size <= np; size <<= 1) {
                    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
                        __syncthreads();
                        for (uint32_t i = tid; i < (np >> 1); i += THREADS) {
                            const uint32_t pos = 2 * i - (i & (stride - 1));
                            const uint64_t a = table[pos], b = table[pos + stride];
                            const bool up = (pos & size) == 0u;
                            if ((a > b) == up) {
                                table[pos] = b;
                                table[pos + stride] = a;
                            }
                        }
                    }
                }
                __syncthreads();
            }
            const uint32_t nc = s_ncand;
            if (tid == 0) s_base = atomicAdd(counters, nc);
            __syncthreads();
            const uint32_t gb = s_base;
            for (uint32_t i = tid; i < nc; i += THREADS) {
                const uint64_t key = outk[i];
                cand[(size_t)gb + i] = ((key >> 32) << (64 - J.hbits)) | ((uint64_t)cd_t_of_ord(J, (uint32_t)key) << 2);
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// Compact form of the class kernel (tuning knob 11 = 2, the default when the table indices fit 32 bits): 4-byte pair
// entries ((entry of A << vbits) | visit) and 4-byte table entries [hash : 16 | local id : 16] (with the slot, 30-31 hash
// bits decide "same hash": ~0.03 false candidate pairs per class), so one CTA holds 18 432 records instead of 9 216 and
// the product needs HALF the classes: half the visits, half the per-class barriers. Candidates are placed straight
// into the global candidate array by the counting sort (small groups ordered by their owner thread afterwards); a
// class with a large hash group, or with records that never found a slot, sends its candidates to the overflow array.
// ------------------------------------------------------------------------------------------------
// PRE_LOG > 0: a presence filter in front of the table rounds. Two bitmaps of 2^PRE_LOG bits, indexed by a cheap function
// of the masked sketch key (cd_filter_index): every record sets its bit in the first map and, if it was already set, in the
// second. After a barrier a record whose bit is clear in the SECOND map shares its key with nobody in the class: it is a
// unique row (equal rows have equal keys) and is done without ever being hashed. On a product without duplicates ~95 % of
// the records stop here. The others ("survivors") are compacted into a dense list of record ids; the hash (mix64), the
// table rounds, the mate bits and the counting sort of the candidates walk that list, so a thread handles one entry per
// round instead of RPT predicated slots. PRE_LOG = 0 (tuning knob 11 = 3): no filter, every record is a survivor and the
// list is the identity (not stored).
//
// Dynamic shared memory, in 4-byte words, with AREA = SLOTS + 2 * PRE_WORDS:
//   [0, AREA)           enumeration + filter:  table [0, SLOTS) | map1 | map2
//                       table rounds:          table [0, SLOTS) | ... | survivor list (CAP 16-bit ids) [AREA - CAP/2, AREA)
//                       candidates:            group counters [0, CAP) | ... | survivor list
//   [AREA, +CAP)        pairs
//   [.., +CAP/32)       mate bits, by list index
//   [.., +CD32_BM_WORDS) copy of the non-empty bitmap
// The list is written after every thread has read map2 (the barriers of its block prefix) and read until the candidates
// have left, so neither the table nor the group counters may reach it.

// presence-filter bit of a record: a function of the masked key alone, so equal rows share it and a debug key mask that
// zeroes the key forces every record through the table; the 64 -> 32 fold keeps the bits that vary inside a class (the
// class and owner-class functionals fix only a few linear combinations of the key)
template <int PRE_LOG>
__device__ __forceinline__ uint32_t cd_filter_index(uint64_t key) {
    return (((uint32_t)key ^ (uint32_t)(key >> 32)) * 0x85EBCA6Bu) >> (32 - PRE_LOG);
}

template <int THREADS, int CAP, int LOG_SLOTS, int PRE_LOG>
__global__ void __launch_bounds__(THREADS, 1) class_dedup32_kernel(ClassJob J, ProductRows rows, TileMap tm, double thr,
                                                                    uint64_t *__restrict__ cand, uint64_t *__restrict__ over,
                                                                    uint32_t *__restrict__ counters, int vbits, uint32_t c0, uint32_t c1) {
    constexpr int SLOTS = 1 << LOG_SLOTS;
    constexpr int RPT = CAP / THREADS;
    constexpr int PRE_WORDS = PRE_LOG > 0 ? (1 << PRE_LOG) / 32 : 0;
    constexpr int AREA = SLOTS + 2 * PRE_WORDS;
    constexpr int LIST_AT = PRE_LOG > 0 ? AREA - CAP / 2 : AREA;
    static_assert(CAP % THREADS == 0 && CAP <= 65536 && RPT <= 32, "record ids and list indices are 16 bits, one state bit per record");
    static_assert(SLOTS <= LIST_AT && CAP <= LIST_AT, "the table and the group counters stay below the survivor list");
    extern __shared__ __align__(16) unsigned char cd_smem[];
    uint32_t *table = reinterpret_cast<uint32_t *>(cd_smem);
    uint32_t *map1 = table + SLOTS;
    uint32_t *map2 = map1 + PRE_WORDS;
    uint16_t *list = reinterpret_cast<uint16_t *>(table + LIST_AT);
    uint32_t *pairs = table + AREA;
    uint32_t *mate = pairs + CAP;                       // one bit per list entry: a same-hash record saw it holding a slot
    uint32_t *s_bits = mate + CAP / 32;
    __shared__ uint32_t s_count, s_nsurv, s_ncand, s_base;
    __shared__ uint32_t s_warp[33];
    const int tid = threadIdx.x;
    const uint32_t vmask = (1u << vbits) - 1u;
    const bool check_thr = !(thr < 0.0 || rows.all_pass());
    const uint32_t bm_words = (((uint32_t)J.nblk << (J.k + 1)) + 31u) / 32u;
    const bool bm_shared = bm_words <= (uint32_t)CD32_BM_WORDS;
    if (bm_shared)
        for (uint32_t i = tid; i < bm_words; i += THREADS) s_bits[i] = J.bits[i];
    auto record_of = [&](uint32_t e) -> uint32_t {   // pair-list position of survivor e
        if constexpr (PRE_LOG > 0) return list[e];
        else return e;
    };
    auto drop_if_small = [&](uint32_t pr) {          // a unique row survives unless its own coefficient fails the threshold
        const uint32_t t = J.vq[pr & vmask] * J.M_total + J.lookp[pr >> vbits];
        double re, im;
        rows.coeff_unphased(t, re, im);
        if (!keep_test(re, im, thr)) tm.mark_dropped(t);
    };

    for (uint32_t c = c0 + blockIdx.x; c < c1; c += gridDim.x) {
        if (tid == 0) {
            s_count = 0;
            s_nsurv = 0;
            s_ncand = 0;
        }
        for (int i = tid; i < CAP / 32; i += THREADS) mate[i] = 0u;
        for (int i = tid; i < 2 * PRE_WORDS; i += THREADS) map1[i] = 0u;
        __syncthreads();
        cd_enumerate<THREADS, CAP, false, uint32_t>(J, c, s_bits, bm_shared, &s_count, s_warp, pairs, nullptr, 0u, vbits);
        __syncthreads();
        const uint32_t total = s_count;
        if (total > (uint32_t)CAP) {   // the class does not fit: its records take the global sort
            __syncthreads();
            if (tid == 0) {
                s_base = atomicAdd(counters + 1, total);
                atomicAdd(counters + 2, 1u);
                s_count = 0;
            }
            __syncthreads();
            cd_enumerate<THREADS, CAP, true, uint32_t>(J, c, s_bits, bm_shared, &s_count, s_warp, (uint32_t *)nullptr, over, s_base, vbits);
            __syncthreads();
            continue;
        }
        // ---- presence filter over the records of this thread (pair-list positions tid + j * THREADS)
        uint32_t n_surv = total;
        if constexpr (PRE_LOG > 0) {
            uint32_t fi[RPT];
            uint32_t live = 0, surv = 0;
#pragma unroll
            for (int j = 0; j < RPT; ++j) {
                const uint32_t i = tid + j * THREADS;
                fi[j] = 0;
                if (i < total) {
                    const uint32_t pr = pairs[i];
                    fi[j] = cd_filter_index<PRE_LOG>((__ldg(J.look8 + (pr >> vbits)) ^ __ldg(J.vsk + (pr & vmask))) & J.key_mask);
                    const uint32_t bit = 1u << (fi[j] & 31u);
                    if (atomicOr(map1 + (fi[j] >> 5), bit) & bit) atomicOr(map2 + (fi[j] >> 5), bit);
                    live |= 1u << j;
                }
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < RPT; ++j)
                if (((live >> j) & 1u) && ((map2[fi[j] >> 5] >> (fi[j] & 31u)) & 1u)) surv |= 1u << j;
            if (check_thr) {
#pragma unroll
                for (int j = 0; j < RPT; ++j)
                    if (((live & ~surv) >> j) & 1u) drop_if_small(pairs[tid + j * THREADS]);
            }
            uint32_t pos = cd_block_prefix<THREADS>((uint32_t)__popc(surv), s_warp, &s_nsurv, n_surv);
#pragma unroll
            for (int j = 0; j < RPT; ++j)
                if ((surv >> j) & 1u) list[pos++] = (uint16_t)(tid + j * THREADS);
            __syncthreads();
        }
        // ---- the survivors, NS list entries per thread (e = tid + s * THREADS; entries past n_surv are empty). NS is the
        // smallest instance that holds the class's list, so a thread only issues the slots a list of this length can fill.
        auto survivors = [&](auto ns_tag) {
            constexpr int NS = decltype(ns_tag)::value;
            // the top 32 bits of the mixed sketch are THE hash of this kernel; table entries are [hash : 16 | list index : 16]
            uint32_t h32[NS];
            uint32_t rr[NS];      // list index of the representative of the entry's hash group; later | rank << 16
            uint32_t unres = 0, candm = 0, winm = 0;   // one bit per list entry: no slot yet / saw a same-hash entry / holds a slot
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const uint32_t e = tid + s * THREADS;
                h32[s] = 0;
                rr[s] = e;
                if (e < n_surv) {
                    const uint32_t pr = pairs[record_of(e)];
                    h32[s] = (uint32_t)((mix64(__ldg(J.look8 + (pr >> vbits)) ^ __ldg(J.vsk + (pr & vmask))) & J.key_mask) >> 32);
                    unres |= 1u << s;
                }
            }
            for (int round = 0; round < CD_MAX_ROUNDS; ++round) {
                const uint32_t mult = 0x9E3779B1u + 2u * (uint32_t)round * 0x632BE5ABu;   // odd for every round
                const uint32_t add = (uint32_t)round * 0x7F4A7C15u;
                if (unres) {
#pragma unroll
                    for (int s = 0; s < NS; ++s) {
                        if ((unres >> s) & 1u) table[(h32[s] * mult + add) >> (32 - LOG_SLOTS)] = (h32[s] & 0xffff0000u) | (tid + s * THREADS);
                    }
                }
                if (!__syncthreads_or(unres != 0u)) break;
                if (unres) {
#pragma unroll
                    for (int s = 0; s < NS; ++s) {
                        if ((unres >> s) & 1u) {
                            const uint32_t mine = (h32[s] & 0xffff0000u) | (tid + s * THREADS);
                            const uint32_t v = table[(h32[s] * mult + add) >> (32 - LOG_SLOTS)];
                            if (v == mine) {
                                winm |= 1u << s;
                                unres &= ~(1u << s);
                            } else if (((v ^ mine) >> 16) == 0u) {
                                rr[s] = v & 0xffffu;
                                atomicOr(mate + (rr[s] >> 5), 1u << (rr[s] & 31u));
                                candm |= 1u << s;
                                unres &= ~(1u << s);
                            }
                        }
                    }
                }
                __syncthreads();
            }
            // ---- candidates: saw a mate, was seen by one, or never found a free slot (then its mates did not either)
            candm |= unres;
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                if (((winm >> s) & 1u) && ((mate[(tid + s * THREADS) >> 5] >> (tid & 31)) & 1u)) candm |= 1u << s;
            }
            if (check_thr) {
#pragma unroll
                for (int s = 0; s < NS; ++s) {
                    const uint32_t e = tid + s * THREADS;
                    if (e < n_surv && !((candm >> s) & 1u)) drop_if_small(pairs[record_of(e)]);
                }
            }
            if (__syncthreads_or(candm != 0u)) {
                uint32_t *cnt = table;   // group counters by list index, then their offsets
#pragma unroll
                for (int s = 0; s < NS; ++s) {
                    cnt[tid + s * THREADS] = 0u;
                }
                __syncthreads();
                bool slow = (candm & unres) != 0u;
#pragma unroll
                for (int s = 0; s < NS; ++s) {
                    if (((candm & ~unres) >> s) & 1u) rr[s] |= atomicAdd(cnt + rr[s], 1u) << 16;
                }
                __syncthreads();
                uint32_t sum = 0;
#pragma unroll
                for (int s = 0; s < NS; ++s) {
                    const uint32_t cj = cnt[tid + s * THREADS];
                    slow |= cj > (uint32_t)CD_SMALL_GROUP;
                    sum += cj;
                }
                if (!__syncthreads_or(slow)) {
                    uint32_t nc;
                    const uint32_t first = cd_block_prefix<THREADS>(sum, s_warp, &s_ncand, nc);
                    if (tid == 0) s_base = atomicAdd(counters, nc);
                    uint32_t base = first;
#pragma unroll
                    for (int s = 0; s < NS; ++s) {
                        const uint32_t cj = cnt[tid + s * THREADS];
                        cnt[tid + s * THREADS] = base;
                        base += cj;
                    }
                    __syncthreads();
                    uint64_t *dst = cand + s_base;
#pragma unroll
                    for (int s = 0; s < NS; ++s) {
                        if ((candm >> s) & 1u) {
                            const uint32_t pr = pairs[record_of(tid + s * THREADS)];
                            const uint32_t v = pr & vmask, lo = pr >> vbits;
                            const int b = J.nblk == 1 ? 0 : (int)(J.vkey[v] >> (J.k + 1));
                            dst[cnt[rr[s] & 0xffffu] + (rr[s] >> 16)] =
                                ((uint64_t)(h32[s] >> (32 - J.hbits)) << 32) | cd_ord_of(J, b, J.lookp[lo], J.vq[v]);
                        }
                    }
                    __syncthreads();
                    // the thread that owns a representative orders its group (2-3 records) by enumeration position
#pragma unroll
                    for (int s = 0; s < NS; ++s) {
                        const uint32_t off_s = cnt[tid + s * THREADS];
                        const uint32_t end_s = s + 1 < NS ? cnt[tid + (s + 1) * THREADS] : first + sum;
                        const uint32_t cj = end_s - off_s;
                        if (cj >= 2u) {
                            uint64_t *seg = dst + off_s;
                            for (uint32_t a = 1; a < cj; ++a) {
                                const uint64_t key = seg[a];
                                uint32_t bpos = a;
                                while (bpos > 0 && seg[bpos - 1] > key) {
                                    seg[bpos] = seg[bpos - 1];
                                    --bpos;
                                }
                                seg[bpos] = key;
                            }
                        }
                    }
                    __syncthreads();
                    for (uint32_t i = tid; i < nc; i += THREADS) {   // [hash | ord] -> candidate record [hash | t | 0]
                        const uint64_t key = dst[i];
                        dst[i] = ((key >> 32) << (64 - J.hbits)) | ((uint64_t)cd_t_of_ord(J, (uint32_t)key) << 2);
                    }
                } else {
                    // a large hash group (a square's identity terms, a molecular H*H) or records without a slot: this class's
                    // candidates take the global sort with the overflowed classes
                    uint32_t nc;
                    uint32_t pos = cd_block_prefix<THREADS>((uint32_t)__popc(candm), s_warp, &s_ncand, nc);
                    if (tid == 0) s_base = atomicAdd(counters + 1, nc);
                    __syncthreads();
                    const uint32_t ob = s_base;
#pragma unroll
                    for (int s = 0; s < NS; ++s) {
                        if ((candm >> s) & 1u) {
                            const uint32_t pr = pairs[record_of(tid + s * THREADS)];
                            const uint32_t v = pr & vmask, lo = pr >> vbits;
                            const int b = J.nblk == 1 ? 0 : (int)(J.vkey[v] >> (J.k + 1));
                            const uint64_t ord = cd_ord_of(J, b, J.lookp[lo], J.vq[v]);
                            over[(size_t)ob + pos++] = ((((uint64_t)h32[s] << 32) >> (J.tb + 2)) << (J.tb + 2)) | (ord << 2);
                        }
                    }
                }
            }
        };
        // block-uniform. The 2 / 4 / 8 instances pay on duplicate-heavy products: the span-28 product of bench.py fills
        // ~6 entries per thread, and its class kernel takes 2.53 ms with them, 2.77 ms with the 18-entry one (B200)
        const uint32_t ns = (n_surv + THREADS - 1) / THREADS;
        if (ns <= 1) survivors(std::integral_constant<int, 1>());
        else if (ns <= 2) survivors(std::integral_constant<int, 2>());
        else if (ns <= 4) survivors(std::integral_constant<int, 4>());
        else if (ns <= 8) survivors(std::integral_constant<int, 8>());
        else survivors(std::integral_constant<int, RPT>());
        __syncthreads();
    }
}

__global__ void cd_total_kernel(uint32_t *counters) { counters[3] = counters[0] + counters[1]; }

// overflow records were sorted on (hash, ord): put t back into their term field
__global__ void __launch_bounds__(256) cd_ord_to_t_kernel(ClassJob J, uint64_t *__restrict__ recs, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t rec = recs[i];
    const uint64_t field = ((1ull << J.tb) - 1ull) << 2;
    recs[i] = (rec & ~field) | ((uint64_t)cd_t_of_ord(J, (uint32_t)((rec & field) >> 2)) << 2);
}

int class_ord_to_t(const ClassJob &J, uint64_t *recs, uint32_t n, cudaStream_t st) {
    if (n == 0 || (J.nblk == 1 && J.p0[0] == 0 && J.q0[0] == 0 && J.m_blk[0] == J.M_total)) return SYM_OK;   // ord == t
    cd_ord_to_t_kernel<<<(n + 255) / 256, 256, 0, st>>>(J, recs, n);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int cd_bits_for(uint32_t n) {   // bits that hold every index below n
    int b = 1;
    while (b < 32 && (1ull << b) < n) ++b;
    return b;
}
static int class_cap(int variant) { return (variant == 2 || variant == 3) ? 18432 : (variant == 1 ? 9216 : 4096); }

bool class_job_plan(int64_t M_total, const TileBlock *blocks, int nblk, int64_t T, int tb, uint64_t key_mask, int variant,
                    ClassJob &J) {
    if (nblk < 1 || nblk > CD_MAX_BLOCKS || T < 1 || T >= ((int64_t)1 << 32)) return false;
    int64_t entries = 0, visits = 0, recs = 0;
    for (int b = 0; b < nblk; ++b) {
        J.entry_base[b] = (uint32_t)entries;
        J.visit_base[b] = (uint32_t)visits;
        J.rec_off[b] = (uint32_t)recs;
        J.p0[b] = blocks[b].p0;
        J.q0[b] = blocks[b].q0;
        J.m_blk[b] = blocks[b].m_blk > 0 ? blocks[b].m_blk : 1u;
        entries += blocks[b].m_blk;
        visits += blocks[b].nq;
        recs += (int64_t)blocks[b].m_blk * blocks[b].nq;
    }
    for (int b = nblk; b <= CD_MAX_BLOCKS; ++b) {
        J.entry_base[b] = (uint32_t)entries;
        J.visit_base[b] = (uint32_t)visits;
        J.rec_off[b] = (uint32_t)recs;
        if (b < CD_MAX_BLOCKS) {
            J.p0[b] = J.q0[b] = 0;
            J.m_blk[b] = 1;
        }
    }
    if (entries >= ((int64_t)1 << 31) || visits >= ((int64_t)1 << 31)) return false;
    // classes: the average class fills at most 85 % of a CTA's pair list; small products still get enough classes
    // to occupy the GPU
    J.variant = variant;
    if ((J.variant == 2 || J.variant == 3) && cd_bits_for((uint32_t)entries) + cd_bits_for((uint32_t)cd_padded_visits((uint32_t)visits)) > 32) J.variant = 1;
    int64_t target = (int64_t)(0.85 * class_cap(J.variant));
    if (T / 1024 < target) target = T / 1024 > 256 ? T / 1024 : 256;
    int k = 0;
    while (k < 22 && (T >> k) > target) ++k;
    // every class visits every row of B: give up when that costs far more than the records themselves
    if ((visits << k) > 64 * T + ((int64_t)1 << 22)) return false;
    J.k = k;
    J.nblk = nblk;
    J.n_entries = (uint32_t)entries;
    J.n_visits = (uint32_t)visits;
    J.M_total = (uint32_t)M_total;
    J.key_mask = key_mask;
    J.tb = tb;
    J.hbits = 62 - tb < 32 ? 62 - tb : 32;
    J.b_sk = nullptr;
    J.off = J.bits = J.lookp = J.vkey = J.vq = nullptr;
    J.look8 = J.vsk = nullptr;
    return true;
}

static size_t cd_table_elems(const ClassJob &J) { return (size_t)J.nblk << (J.k + 1); }

size_t class_job_ws_bytes(const ClassJob &J) {
    const size_t tab = cd_table_elems(J);
    const size_t ne = J.n_entries ? J.n_entries : 1, nv = J.n_visits ? J.n_visits : 1;
    return 2 * arena_need(2 * tab + 64, 4) + arena_need(tab / 32 + 64, 4) + arena_need(scan_scratch_elems((int64_t)(2 * tab)), 4) +
           arena_need(ne, 8) + arena_need(ne, 4) + arena_need(cd_padded_visits(J.n_visits), 4) + arena_need(nv, 4) + arena_need(nv, 8) + 1024;
}

template <int THREADS, int CAP, int LOG_SLOTS, int MINB>
static int cd_launch(const ClassJob &J, const ProductRows &rows, const TileMap &tm, double thr, uint64_t *cand, uint64_t *over,
                     uint32_t *counters, uint32_t c0, uint32_t c1, uint32_t sms, cudaStream_t st) {
    constexpr size_t smem = ((size_t)1 << LOG_SLOTS) * 8 + (size_t)CAP * 8 + CAP + (size_t)CD_BM_WORDS * 4;
    auto kern = class_dedup_kernel<THREADS, CAP, LOG_SLOTS, MINB>;
    static bool attr_done[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !attr_done[dev]) {
        SYM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev] = true;
    }
    const unsigned grid = (unsigned)std::min<uint32_t>(c1 - c0, sms * (uint32_t)MINB);
    kern<<<grid, THREADS, smem, st>>>(J, rows, tm, thr, cand, over, counters, c0, c1);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

// The class tables in `ws` (and the scratch of their build): carves the arena and points J at the tables.
struct CdTables {
    uint32_t *off, *cursor, *bits, *scratch, *lookp, *vkey, *vq;
    uint64_t *look8, *vsk;
};
static int cd_carve(ClassJob &J, const uint64_t *b_sk, void *ws, size_t ws_bytes, CdTables &t) {
    Arena ar(ws, ws_bytes);
    const size_t tab = cd_table_elems(J);
    const size_t ne = J.n_entries ? J.n_entries : 1, nv = J.n_visits ? J.n_visits : 1;
    t.off = ar.take<uint32_t>(2 * tab + 64);
    t.cursor = ar.take<uint32_t>(2 * tab + 64);
    t.bits = ar.take<uint32_t>(tab / 32 + 64);
    t.scratch = ar.take<uint32_t>(scan_scratch_elems((int64_t)(2 * tab)));
    t.look8 = ar.take<uint64_t>(ne);
    t.lookp = ar.take<uint32_t>(ne);
    t.vkey = ar.take<uint32_t>(cd_padded_visits(J.n_visits));
    t.vq = ar.take<uint32_t>(nv);
    t.vsk = ar.take<uint64_t>(nv);
    if (!t.vsk) {
        set_error("workspace arena exhausted (class tables)");
        return SYM_E_WORKSPACE;
    }
    J.b_sk = b_sk;
    J.off = t.off;
    J.bits = t.bits;
    J.look8 = t.look8;
    J.lookp = t.lookp;
    J.vkey = t.vkey;
    J.vq = t.vq;
    J.vsk = t.vsk;
    return SYM_OK;
}

int class_dedup_bind(ClassJob &J, const uint64_t *b_sk, void *ws, size_t ws_bytes) {
    CdTables t;
    return cd_carve(J, b_sk, ws, ws_bytes, t);
}

int class_dedup_tables(ClassJob &J, const uint64_t *a_sk, const uint64_t *b_sk, uint32_t *counters, void *ws, size_t ws_bytes,
                       cudaStream_t st) {
    CdTables t;
    SYM_TRY(cd_carve(J, b_sk, ws, ws_bytes, t));
    const size_t tab = cd_table_elems(J);
    const size_t nvp = cd_padded_visits(J.n_visits);
    SYM_CUDA_OK(cudaMemsetAsync(t.off, 0, sizeof(uint32_t) * (2 * tab + 64), st));
    SYM_CUDA_OK(cudaMemsetAsync(t.cursor, 0, sizeof(uint32_t) * (2 * tab + 64), st));
    SYM_CUDA_OK(cudaMemsetAsync(counters, 0, sizeof(uint32_t) * 4, st));
    // many rows of A per table entry: privatised counters (the visits still take the plain kernels, with no rows of A)
    const bool priv = tab <= 12288 && (size_t)J.n_entries >= 16 * tab && J.n_entries >= (1u << 18);
    const uint32_t n_rows_a = priv ? 0u : J.n_entries;
    if (priv) {
        static bool attr_done[64] = {};
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev >= 0 && dev < 64 && !attr_done[dev]) {
            SYM_CUDA_OK(cudaFuncSetAttribute(cd_place_priv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 12288 * 4));
            attr_done[dev] = true;
        }
        cd_hist_priv_kernel<<<(J.n_entries + CD_CHUNK - 1) / CD_CHUNK, 1024, tab * 4, st>>>(J, a_sk, t.off, (uint32_t)tab);
        SYM_LAUNCH_OK();
    }
    const uint32_t n1 = n_rows_a > J.n_visits ? n_rows_a : J.n_visits;
    if (n1) {
        cd_hist_kernel<<<(n1 + 255) / 256, 256, 0, st>>>(J, a_sk, t.off, (uint32_t)tab, n_rows_a);
        SYM_LAUNCH_OK();
    }
    SYM_TRY(scan_exclusive_u32(t.off, t.off, (int64_t)(2 * tab), nullptr, t.scratch, st));
    if (priv) {
        cd_place_priv_kernel<<<(J.n_entries + CD_CHUNK - 1) / CD_CHUNK, 1024, 2 * tab * 4, st>>>(J, a_sk, t.off, t.cursor,
                                                                                                 (uint32_t)tab, t.look8, t.lookp);
        SYM_LAUNCH_OK();
    }
    uint32_t n2 = n1 > (uint32_t)((tab + 31) / 32) ? n1 : (uint32_t)((tab + 31) / 32);
    if (n2 < (uint32_t)nvp) n2 = (uint32_t)nvp;
    cd_place_kernel<<<(n2 + 255) / 256, 256, 0, st>>>(J, a_sk, t.off, t.cursor, (uint32_t)tab, t.look8, t.lookp, t.vkey, t.vq,
                                                     t.vsk, t.bits, (uint32_t)nvp, n_rows_a);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

int class_dedup_classes(const ClassJob &J, const ProductRows &rows, const TileMap &tm, double thr, uint64_t *cand, uint64_t *over,
                        uint32_t *counters, uint32_t c0, uint32_t c1, uint32_t sms, cudaStream_t st) {
    if (c0 < c1) {
        if (J.variant == 2 || J.variant == 3) {
            constexpr int CAP = 18432;
            constexpr size_t smem = ((size_t)1 << 15) * 4 + (size_t)CAP * 4 + CAP / 8 + (size_t)CD32_BM_WORDS * 4;   // both shapes
            auto kern_pre = class_dedup32_kernel<1024, CAP, 14, 18>;   // 64 KB table + 2 x 32 KB presence maps
            auto kern_old = class_dedup32_kernel<1024, CAP, 15, 0>;    // 128 KB table (tuning knob 11 = 3)
            static bool attr_done[64] = {};
            int dev = 0;
            cudaGetDevice(&dev);
            if (dev >= 0 && dev < 64 && !attr_done[dev]) {
                SYM_CUDA_OK(cudaFuncSetAttribute(kern_pre, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                SYM_CUDA_OK(cudaFuncSetAttribute(kern_old, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                attr_done[dev] = true;
            }
            const unsigned grid = (unsigned)std::min<uint32_t>(c1 - c0, sms);
            const int vbits = cd_bits_for((uint32_t)cd_padded_visits(J.n_visits));
            if (J.variant == 2) kern_pre<<<grid, 1024, smem, st>>>(J, rows, tm, thr, cand, over, counters, vbits, c0, c1);
            else kern_old<<<grid, 1024, smem, st>>>(J, rows, tm, thr, cand, over, counters, vbits, c0, c1);
            SYM_LAUNCH_OK();
        } else if (class_cap(J.variant) == 9216) {
            SYM_TRY((cd_launch<1024, 9216, 14, 1>(J, rows, tm, thr, cand, over, counters, c0, c1, sms, st)));
        } else {
            SYM_TRY((cd_launch<512, 4096, 13, 2>(J, rows, tm, thr, cand, over, counters, c0, c1, sms, st)));
        }
    }
    cd_total_kernel<<<1, 1, 0, st>>>(counters);
    SYM_LAUNCH_OK();
    return SYM_OK;
}

}  // namespace symb
