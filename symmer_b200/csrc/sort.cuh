// Device-wide primitives used by the dedup pipeline: exclusive scan and a stable LSD radix sort of
// 64-bit keys with optional 32-bit values. Hand-written for sm_100a; no CUB/Thrust on the path.
#pragma once
#include "common.cuh"

namespace symb {

// Exclusive prefix sum of n values (uint8 or uint32 input) into uint32 out; the grand total is
// written to *total (device uint32). `in` may alias `out` when the element types match.
// scratch: uint32[scan_scratch_elems(n)].
size_t scan_scratch_elems(int64_t n);
int scan_exclusive_u8(const uint8_t *in, uint32_t *out, int64_t n, uint32_t *total, uint32_t *scratch,
                      cudaStream_t st);
int scan_exclusive_u32(const uint32_t *in, uint32_t *out, int64_t n, uint32_t *total, uint32_t *scratch,
                       cudaStream_t st);

// Stable LSD radix sort (record_sort.cu) of 64-bit keys on bits [begin_bit, 64), 8 bits per pass; each key
// optionally carries a 32-bit value (vals, vals_alt: null for keys alone). Tiles are staged in shared memory so
// that every digit run of a tile leaves as one contiguous (coalesced) store. Passes ping-pong between keys/vals
// and the same-sized alt/vals_alt; `*result` receives whichever of keys/alt holds the sorted keys (no copy-back),
// and the sorted values are in the matching value buffer. hist: uint32 scratch of record_hist_elems(T).
size_t record_hist_elems(int64_t T);
int radix_sort(uint64_t *keys, uint32_t *vals, uint64_t *alt, uint32_t *vals_alt, int64_t T, int begin_bit,
               uint32_t *hist, uint64_t **result, cudaStream_t st);

// One stable partition pass on the top `bits` (<= 8) bits of the key, values (if not null) moving with their
// keys; counts: device int64[1 << bits] receives the bucket sizes. hist as for radix_sort.
int radix_partition(const uint64_t *keys, const uint32_t *vals, uint64_t *out, uint32_t *out_vals, int64_t T, int bits,
                    int64_t *counts, uint32_t *hist, cudaStream_t st);

}  // namespace symb
