// Device-wide primitives used by the dedup pipeline: exclusive scan and a stable LSD radix sort
// of (uint64 key, uint32 value) pairs. Hand-written for sm_100a; no CUB/Thrust on the path.
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

// Stable radix sort on key bits [begin_bit, 64), 8 bits per pass. Buffers: keys/vals hold the
// input and receive the output; keys_alt/vals_alt are same-sized scratch. hist: uint32 scratch of
// sort_hist_elems(T). If vals_iota is true the input values are taken to be 0..T-1 (vals need not
// be initialised).
size_t sort_hist_elems(int64_t T);
int radix_sort_pairs(uint64_t *keys, uint32_t *vals, uint64_t *keys_alt, uint32_t *vals_alt, int64_t T,
                     int begin_bit, bool vals_iota, uint32_t *hist, cudaStream_t st);

// One stable partition pass on the top `bits` bits of the key (bits <= 8); counts[d] (device
// int64[1<<bits]) receives the bucket sizes.
int radix_partition_top(const uint64_t *keys, const uint32_t *vals, uint64_t *out_keys, uint32_t *out_vals,
                        int64_t T, int bits, int64_t *counts, uint32_t *hist, cudaStream_t st);

}  // namespace symb

namespace symb {
// Hot-path sort: stable LSD radix sort of single 64-bit records on bits [begin_bit, 64), shared-
// memory staged so that every digit run of a tile leaves as one contiguous (coalesced) store.
// `*result` receives whichever of keys/alt holds the sorted records (no copy-back).
size_t record_hist_elems(int64_t T);
int radix_sort_records(uint64_t *keys, uint64_t *alt, int64_t T, int begin_bit, uint32_t *hist, uint64_t **result,
                       cudaStream_t st);

// One stable partition pass on the top `bits` (<= 8) bits; counts: device int64[1 << bits].
int radix_partition_records(const uint64_t *keys, uint64_t *out, int64_t T, int bits, int64_t *counts, uint32_t *hist,
                            cudaStream_t st);
}  // namespace symb
