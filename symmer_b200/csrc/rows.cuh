// Row accessors and the record format shared by the dedup pipeline.
#pragma once
#include "common.cuh"

namespace symb {

// A dedup record is one 64-bit word:   [ hash : 62 - tb bits | t : tb bits | e : 2 bits ]
// hash = top bits of mix64(sketch(row)); t = term index (cross-term index q*M + p for products);
// e = phase exponent of the cross term (0 for stored rows). Equal rows have equal hash fields.
struct RecFmt {
    int tb;
    __host__ __device__ __forceinline__ uint32_t t(uint64_t rec) const { return (uint32_t)((rec >> 2) & ((1ull << tb) - 1ull)); }
    __host__ __device__ __forceinline__ int e(uint64_t rec) const { return (int)(rec & 3ull); }
    __host__ __device__ __forceinline__ bool same_hash(uint64_t a, uint64_t b) const { return ((a ^ b) >> (tb + 2)) == 0; }
    __host__ __device__ __forceinline__ uint64_t make(uint64_t key, uint64_t t, int e) const {
        return ((key >> (tb + 2)) << (tb + 2)) | (t << 2) | (uint64_t)e;
    }
};

static inline int t_bits_for(int64_t T) {
    int tb = 1;
    while ((int64_t(1) << tb) < T) ++tb;
    return tb;
}

// Exact t / d for 32-bit t by one 64-bit multiply-high: magic = floor(2^64 / d) + 1 (the exact reciprocal when d is a
// power of two). The integer division the hot kernels would otherwise run per lane costs ~20 instructions.
static inline uint64_t fastdiv_magic(uint32_t d) { return d <= 1 ? 0ull : (~0ull / d) + 1ull; }
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t fastdiv(uint32_t t, uint32_t d, uint64_t magic) {
    return magic ? (uint32_t)__umul64hi((uint64_t)t, magic) : t / d;
}
#endif

// Term t is the cross term (p, q) of a product A*B in the reference's flattened order t = q*M + p
// (base.py:783-792); its row is A[p] ^ B[q] and is never stored.
struct ProductRows {
    const uint64_t *__restrict__ A;
    const uint64_t *__restrict__ B;
    const double *__restrict__ Ac;
    const double *__restrict__ Bc;
    uint32_t M;  // rows of A (divisor of t)
    int words;   // 2*W
    uint32_t N = 0;                                // rows of B (0 = unknown)
    const uint32_t *__restrict__ pass_all = nullptr;  // device flag: every single cross term passes |c| > thr
    uint64_t Minv = 0;                             // fastdiv_magic(M), or 0: divide

    __device__ __forceinline__ bool all_pass() const { return pass_all != nullptr && *pass_all != 0u; }

    __device__ __forceinline__ void split(uint32_t t, uint32_t &p, uint32_t &q) const {
        q = fastdiv(t, M, Minv);
        p = t - q * M;
    }
    __device__ __forceinline__ uint4 chunk(uint32_t t, int c) const {  // 16-byte chunk c of the row
        uint32_t p, q;
        split(t, p, q);
        const uint4 a = reinterpret_cast<const uint4 *>(A + (size_t)p * words)[c];
        const uint4 b = reinterpret_cast<const uint4 *>(B + (size_t)q * words)[c];
        return make_uint4(a.x ^ b.x, a.y ^ b.y, a.z ^ b.z, a.w ^ b.w);
    }
    // (p, q) handle of a term, so that the 16 chunk-threads of a row do not each redo the division
    __device__ __forceinline__ uint2 locate(uint32_t t) const {
        uint2 h;
        split(t, h.x, h.y);
        return h;
    }
    __device__ __forceinline__ uint4 chunk_at(uint2 h, int c) const {
        const uint4 a = reinterpret_cast<const uint4 *>(A + (size_t)h.x * words)[c];
        const uint4 b = reinterpret_cast<const uint4 *>(B + (size_t)h.y * words)[c];
        return make_uint4(a.x ^ b.x, a.y ^ b.y, a.z ^ b.z, a.w ^ b.w);
    }
    __device__ __forceinline__ bool equal(uint32_t t1, uint32_t t2) const {
        uint32_t p1, q1, p2, q2;
        split(t1, p1, q1);
        split(t2, p2, q2);
        const uint64_t *a1 = A + (size_t)p1 * words, *b1 = B + (size_t)q1 * words;
        const uint64_t *a2 = A + (size_t)p2 * words, *b2 = B + (size_t)q2 * words;
        // rows are 16-byte aligned (words = 2W is even): compare 16 bytes per step, four loads in flight
        const uint4 *u1 = reinterpret_cast<const uint4 *>(a1), *v1 = reinterpret_cast<const uint4 *>(b1);
        const uint4 *u2 = reinterpret_cast<const uint4 *>(a2), *v2 = reinterpret_cast<const uint4 *>(b2);
        const int chunks = words >> 1;
        for (int k = 0; k < chunks; ++k) {
            const uint4 x1 = u1[k], y1 = v1[k], x2 = u2[k], y2 = v2[k];
            if (((x1.x ^ y1.x) != (x2.x ^ y2.x)) | ((x1.y ^ y1.y) != (x2.y ^ y2.y)) | ((x1.z ^ y1.z) != (x2.z ^ y2.z)) |
                ((x1.w ^ y1.w) != (x2.w ^ y2.w)))
                return false;
        }
        return true;
    }
    // phase exponent of the cross term from its rows (base.py:785-788): ordered-tile mode stamps it on the few
    // records that may take part in a sum (phase_work_kernel); the other modes compute it for every pair up front
    __device__ __noinline__ int phase(uint32_t t) const {
        uint32_t p, q;
        split(t, p, q);
        const uint64_t *ra = A + (size_t)p * words, *rb = B + (size_t)q * words;
        const int W = words >> 1;
        uint64_t s = 0, c0 = 0, c1 = 0;
        int y_in = 0;
#pragma unroll 4
        for (int w = 0; w < W; ++w) {
            const uint64_t xa = ra[w], za = ra[W + w], xb = rb[w], zb = rb[W + w];
            y_in += __popcll(xa & za) + __popcll(xb & zb);
            s ^= xa & zb;
            const uint64_t v = (xa ^ xb) & (za ^ zb);
            c1 ^= c0 & v;
            c0 ^= v;
        }
        return (3 * y_in + __popcll(c0) + 2 * __popcll(c1) + 2 * (__popcll(s) & 1)) & 3;
    }
    __device__ __forceinline__ void coeff(uint32_t t, int e, double &re, double &im) const {
        uint32_t p, q;
        split(t, p, q);
        cmul(Ac[2 * (size_t)p], Ac[2 * (size_t)p + 1], Bc[2 * (size_t)q], Bc[2 * (size_t)q + 1], re, im);
        mul_i_pow(re, im, e);
    }
    // |coefficient| only matters (threshold tests): no phase
    __device__ __forceinline__ void coeff_unphased(uint32_t t, double &re, double &im) const {
        uint32_t p, q;
        split(t, p, q);
        cmul(Ac[2 * (size_t)p], Ac[2 * (size_t)p + 1], Bc[2 * (size_t)q], Bc[2 * (size_t)q + 1], re, im);
    }
};

// Term t is row t of a stored operator.
struct PlainRows {
    const uint64_t *__restrict__ X;
    const double *__restrict__ C;
    int words;

    __device__ __forceinline__ bool all_pass() const { return false; }
    __device__ __forceinline__ uint4 chunk(uint32_t t, int c) const {
        return reinterpret_cast<const uint4 *>(X + (size_t)t * words)[c];
    }
    __device__ __forceinline__ uint2 locate(uint32_t t) const { return make_uint2(t, 0u); }
    __device__ __forceinline__ uint4 chunk_at(uint2 h, int c) const { return chunk(h.x, c); }
    __device__ __forceinline__ bool equal(uint32_t t1, uint32_t t2) const {
        const uint4 *r1 = reinterpret_cast<const uint4 *>(X + (size_t)t1 * words);
        const uint4 *r2 = reinterpret_cast<const uint4 *>(X + (size_t)t2 * words);
        const int chunks = words >> 1;   // words = 2W is even: rows are 16-byte aligned
        for (int k = 0; k < chunks; ++k) {
            const uint4 a = r1[k], b = r2[k];
            if ((a.x != b.x) | (a.y != b.y) | (a.z != b.z) | (a.w != b.w)) return false;
        }
        return true;
    }
    __device__ __forceinline__ void coeff(uint32_t t, int, double &re, double &im) const {
        re = C[2 * (size_t)t];
        im = C[2 * (size_t)t + 1];
    }
    __device__ __forceinline__ void coeff_unphased(uint32_t t, double &re, double &im) const { coeff(t, 0, re, im); }
};

// ---------------------------------------------------------------------------------------------
// Ordered-tile mode of a product (large T): the survivors leave in the order of the cross-term
// index t = q*M + p (the reference's first-occurrence order) and the row emission streams
// rectangular tiles of A x B instead of gathering rows in sorted-hash order.
// The cross terms of block b (rows [p0, p0+m_blk) of A against rows [q0, q0+nq) of B) are cut
// into SEGMENTS of TILE_ROWS consecutive p for one q; segment id
//   s = seg_base + (q - q0) * ptiles + (p - p0) / TILE_ROWS,  bit = (p - p0) % TILE_ROWS.
// Per segment: 4 words of drop bits (set by the reduction for every cross term that does not
// survive) and one output offset (exclusive scan of the survivor counts). Records carry no phase
// exponent in this mode: the emission kernel has both rows in registers and computes it there.
constexpr int TILE_ROWS = 128;

struct TileBlock {
    uint32_t p0, m_blk, q0, nq, ptiles, seg_base;
    uint32_t t_base;   // cross terms of the blocks before this one: the block's first output row when nothing is dropped
};

__host__ __device__ __forceinline__ uint32_t tile_valid_word(uint32_t m_blk, uint32_t ptile, int w) {
    const int64_t left = (int64_t)m_blk - (int64_t)ptile * TILE_ROWS - 32 * w;
    return left >= 32 ? 0xffffffffu : (left <= 0 ? 0u : ((1u << (int)left) - 1u));
}

struct TileMap {
    TileBlock first;           // block 0 inline: the single-rectangle product never reads `blocks`
    const TileBlock *blocks;   // device, nblk entries
    int nblk;
    uint32_t M;                // rows of A: t = q*M + p
    uint64_t Minv = 0;         // fastdiv_magic(M), or 0: divide
    uint32_t n_seg;
    uint32_t *drop;            // uint32[4 * n_seg]
    uint32_t *segoff;          // uint32[n_seg + 1]: counts, then their exclusive scan in place

#ifdef __CUDACC__
    __device__ __forceinline__ bool locate(uint32_t t, TileBlock &blk, uint32_t &s, uint32_t &bit) const {
        const uint32_t q = fastdiv(t, M, Minv), p = t - q * M;
        blk = first;
        for (int b = 0;;) {
            const uint32_t pl = p - blk.p0, ql = q - blk.q0;
            if (pl < blk.m_blk && ql < blk.nq) {
                s = blk.seg_base + ql * blk.ptiles + pl / TILE_ROWS;
                bit = pl % TILE_ROWS;
                return true;
            }
            if (++b >= nblk) return false;
            blk = blocks[b];
        }
    }
    __device__ __forceinline__ void mark_dropped(uint32_t t) const {
        TileBlock blk;
        uint32_t s, bit;
        if (locate(t, blk, s, bit)) atomicOr(drop + 4 * (size_t)s + (bit >> 5), 1u << (bit & 31));
    }
    // output slot of a surviving cross term (valid once segoff holds the scan)
    __device__ __forceinline__ uint32_t slot_of(uint32_t t) const {
        TileBlock blk;
        uint32_t s, bit;
        if (!locate(t, blk, s, bit)) return 0xffffffffu;
        const uint32_t ptile = (s - blk.seg_base) % blk.ptiles;
        uint32_t r = segoff[s];
        const int wb = (int)(bit >> 5);
        for (int w = 0; w <= wb; ++w) {
            uint32_t k = tile_valid_word(blk.m_blk, ptile, w) & ~drop[4 * (size_t)s + w];
            if (w == wb) k &= (1u << (bit & 31)) - 1u;
            r += __popc(k);
        }
        return r;
    }
#endif
};

#ifdef __CUDACC__
__device__ __forceinline__ uint8_t keep_test(double re, double im, double thr) {
    // |c| > thr like the reference (utils.py:275-278); hypot only when the cheap bounds max(|re|,|im|) <= |c| <= |re|+|im|
    // do not decide it
    if (thr < 0.0) return 1;
    const double ar = fabs(re), ai = fabs(im);
    if (ar > thr || ai > thr) return 1;
    if (ar + ai <= thr) return 0;
    return hypot(re, im) > thr ? 1 : 0;
}
#endif

// ---------------------------------------------------------------------------------------------
// Class-local duplicate detection of an ordered-tile product (class_dedup.cu): the cross terms are
// enumerated class by class (a GF(2)-linear function of the row sketch) from the class-grouped rows
// of A and the sketches of B; only records that have a same-hash mate are ever written to memory.
constexpr int CD_MAX_BLOCKS = 16;
constexpr int CD_MAX_ROUNDS = 8;
struct ClassJob {
    int k;                                     // 2^k classes
    int nblk;
    uint32_t n_entries;                        // rows of A over all blocks
    uint32_t n_visits;                         // rows of B over all blocks
    uint32_t entry_base[CD_MAX_BLOCKS + 1];    // first entry / visit of every block
    uint32_t visit_base[CD_MAX_BLOCKS + 1];
    uint32_t p0[CD_MAX_BLOCKS], q0[CD_MAX_BLOCKS], m_blk[CD_MAX_BLOCKS];
    uint32_t rec_off[CD_MAX_BLOCKS + 1];       // first cross term of every block in block-major order
    uint32_t M_total;                          // t = q * M_total + p
    uint64_t key_mask;
    int tb;                                    // RecFmt::tb of the product
    int hbits;                                 // hash bits of a candidate record = min(32, 62 - tb): its sort bucket
    int variant;                               // CTA shape of the class kernel (tuning knob 11)
    const uint64_t *b_sk;                      // sketches of B (global row index)
    // class tables (class_dedup.cu); table index = (block << (k+1)) | class
    const uint32_t *off;                       // first row of the table entry in look8 / lookp
    const uint32_t *bits;                      // bit per table entry: A has rows there
    const uint64_t *look8;                     // rows of A grouped by table entry: sketch
    const uint32_t *lookp;                     //                                    row index p
    const uint32_t *vkey, *vq;                 // rows of B ("visits") in table-entry order: table index, row index q
    const uint64_t *vsk;                       //                                           sketch
};
// false: this product takes the global record sort instead (too many blocks, B much larger than A).
// variant: CTA shape of the class kernel (tuning knob 11)
bool class_job_plan(int64_t M_total, const TileBlock *blocks, int nblk, int64_t T, int tb, uint64_t key_mask, int variant,
                    ClassJob &J);
size_t class_job_ws_bytes(const ClassJob &J);
// overflow records carry their enumeration position in the term field while they are sorted; this puts t back
int class_ord_to_t(const ClassJob &J, uint64_t *recs, uint32_t n, cudaStream_t st);
// Builds the class tables in `ws`, points J at them and zeroes counters: device uint32[4] = {candidates, overflow
// records, overflowed classes, sum}
int class_dedup_tables(ClassJob &J, const uint64_t *a_sk, const uint64_t *b_sk, uint32_t *counters, void *ws, size_t ws_bytes,
                       cudaStream_t st);
// points J at the tables an earlier class_dedup_tables built in the same `ws`
int class_dedup_bind(ClassJob &J, const uint64_t *b_sk, void *ws, size_t ws_bytes);
// Runs the class kernel over classes [c0, c1) on at most `sms` SMs, then sets counters[3]. Every class appends its
// candidates / overflow records at atomically claimed offsets, so launches over disjoint ranges fill cand / over
// (T records each) exactly as one launch over their union does.
int class_dedup_classes(const ClassJob &J, const ProductRows &rows, const TileMap &tm, double thr, uint64_t *cand, uint64_t *over,
                        uint32_t *counters, uint32_t c0, uint32_t c1, uint32_t sms, cudaStream_t st);

// The path of a product through the dedup, decided once per call by mul_blocks_plan (multiply.cu):
//   BY_T         the t fields are a permutation of 0..T-1 and the survivors are written in increasing-t
//                (first occurrence) order;
//   SORTED       survivors in sorted-hash order;
//   TILES_SORT   ordered-tile mode, duplicates found by the global record sort;
//   TILES_CLASS  ordered-tile mode, duplicates found class by class (class_dedup.cu): no record array.
enum class Path { BY_T, SORTED, TILES_SORT, TILES_CLASS };

// Dedup driver (dedup.cu), split where the survivor count is known so the caller can allocate
// exact-size outputs. `recs` holds T records (clobbered). path: BY_T or SORTED.
size_t dedup_ws_bytes(int64_t T);
void set_emit_events(cudaEvent_t before, cudaEvent_t after);
int dedup_product_plan(Path path, uint64_t *recs, int64_t T, RecFmt fmt, const ProductRows &rows, double thr,
                       int64_t *n_out, int64_t *n_out_host, void *ws, size_t ws_bytes, cudaStream_t st);
int dedup_product_emit(Path path, const uint64_t *recs, int64_t T, RecFmt fmt, const ProductRows &rows, int64_t U,
                       uint64_t *out_xz, double *out_c, void *ws, size_t ws_bytes, cudaStream_t st);
int dedup_plain_plan(uint64_t *recs, int64_t T, RecFmt fmt, const PlainRows &rows, double thr, int64_t *n_out,
                     int64_t *n_out_host, void *ws, size_t ws_bytes, cudaStream_t st);
int dedup_plain_emit(const uint64_t *recs, int64_t T, RecFmt fmt, const PlainRows &rows, int64_t U, uint64_t *out_xz,
                     double *out_c, void *ws, size_t ws_bytes, cudaStream_t st);

// ordered-tile mode (products only); blocks_host mirrors tm.blocks
int dedup_product_plan_tiles(uint64_t *recs, int64_t T, RecFmt fmt, const ProductRows &rows, const TileMap &tm, double thr,
                             int64_t *n_out, int64_t *n_out_host, void *ws, size_t ws_bytes, cudaStream_t st);
// class mode: `recs` is only scratch (the overflow array); a_sk / b_sk are the operand sketch tables and
// class_ws holds the class tables (class_job_ws_bytes). speculate != nullptr: the product may stop after a sampled
// first wave of classes with *speculate = true and *n_out_host = T; dedup_product_spec_classes then finishes it.
int dedup_product_plan_classes(uint64_t *recs, int64_t T, RecFmt fmt, const ProductRows &rows, const TileMap &tm, ClassJob &job,
                               const uint64_t *a_sk, const uint64_t *b_sk, const int32_t *a_y, const int32_t *b_y, void *class_ws,
                               size_t class_ws_bytes, double thr, int64_t *n_out, int64_t *n_out_host, bool *speculate, void *ws,
                               size_t ws_bytes, cudaStream_t st);
// the rest of a speculating class-mode product and its output (T rows of capacity); *n_out_host = U
int dedup_product_spec_classes(uint64_t *recs, int64_t T, RecFmt fmt, const ProductRows &rows, const TileMap &tm,
                               const TileBlock *blocks_host, ClassJob &job, const uint64_t *b_sk, const int32_t *a_y,
                               const int32_t *b_y, void *class_ws, size_t class_ws_bytes, double thr, uint64_t *out_xz,
                               double *out_c, int64_t *n_out_host, void *ws, size_t ws_bytes, cudaStream_t st);
// path: TILES_SORT or TILES_CLASS
int dedup_product_emit_tiles(Path path, const uint64_t *recs, int64_t T, RecFmt fmt, const ProductRows &rows, const TileMap &tm,
                             const TileBlock *blocks_host, const int32_t *a_y, const int32_t *b_y, int64_t U,
                             uint64_t *out_xz, double *out_c, void *ws, size_t ws_bytes, cudaStream_t st);

}  // namespace symb
