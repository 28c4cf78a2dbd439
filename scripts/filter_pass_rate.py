"""Pass rate of the class kernel's presence filter (csrc/class_dedup.cu, class_dedup32_kernel) on the bench operands,
computed on the CPU: the share of cross terms whose filter bit is shared with another cross term of their class, i.e. the
records that go on to be hashed and enter the table rounds. Restates the row sketch (common.cuh: lane_linear over the
packed words), the class function (cd_class_of) and the filter index (cd_filter_index) in NumPy; beside it the same
count for a filter indexed by the top 32 bits of mix64 (the table's hash). A pass is a cost, never an error: equal rows
always share their bit.

    python scripts/filter_pass_rate.py            # bench operands (12 500 x 10 000 terms, 1000 q) and the span-28 pair
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
from oracle import pauli_oracle as po  # noqa: E402

U64 = np.uint64
PRE_LOG = 18
CAP = 18432


def lane_linear(w, lane):
    a = 5 + lane
    b = 3 + ((lane * 5) % 29)
    c = 11 + ((lane * 11) % 37)
    for sh, left in ((a, True), (b, False), (c, True), (a + 7, False), (b + 2, True), (c - 4, False)):
        w = w ^ ((w << U64(sh)) if left else (w >> U64(sh)))
    return w


def sketch(symp):
    words = po.pack_bits(symp)
    h = np.zeros(words.shape[0], dtype=U64)
    for i in range(words.shape[1]):
        h ^= lane_linear(words[:, i].copy(), i)
    return h


def mix64(x):
    with np.errstate(over="ignore"):
        x = x ^ (x >> U64(33))
        x = x * U64(0xff51afd7ed558ccd)
        x = x ^ (x >> U64(33))
        x = x * U64(0xc4ceb9fe1a85ec53)
        return x ^ (x >> U64(33))


def class_of(sk, k):
    y = sk ^ (sk >> U64(21)) ^ (sk >> U64(43))
    return ((y >> U64(5)) & U64((1 << k) - 1)).astype(np.uint32)


def filter_index(key32):
    with np.errstate(over="ignore"):
        return (key32.astype(np.uint32) * np.uint32(0x85EBCA6B)) >> np.uint32(32 - PRE_LOG)


def class_bits(T):
    """k of class_job_plan for one block: the average class fills at most 85 % of CAP."""
    target, k = int(0.85 * CAP), 0
    while k < 22 and (T >> k) > target:
        k += 1
    return k


def shared_fraction(codes):
    c = np.sort(codes)
    dup = c[1:] == c[:-1]
    m = np.zeros(len(c), dtype=bool)
    m[1:] |= dup
    m[:-1] |= dup
    return float(m.mean())


def pass_rates(a_s, b_s):
    ska, skb = sketch(a_s), sketch(b_s)
    T = len(ska) * len(skb)
    k = class_bits(T)
    fold, full = np.empty(T, dtype=np.uint32), np.empty(T, dtype=np.uint32)
    for q0 in range(0, len(skb), 500):
        key = (skb[q0:q0 + 500, None] ^ ska[None, :]).ravel()
        cls = class_of(key, k) << np.uint32(PRE_LOG)
        sl = slice(q0 * len(ska), q0 * len(ska) + len(key))
        fold[sl] = cls | filter_index((key ^ (key >> U64(32))) & U64(0xffffffff))
        full[sl] = cls | filter_index(mix64(key) >> U64(32))
    return {"cross_terms": T, "classes": 1 << k, "filter_pass": shared_fraction(fold), "mix64_filter_pass": shared_fraction(full)}


def main():
    a_s, _ = po.random_operator(1000, 12500, seed=100)
    b_s, _ = po.random_operator(1000, 10000, seed=7)
    print("bench operands:", pass_rates(a_s, b_s), flush=True)
    rng = np.random.default_rng(11)                       # bench.py secondary_dedup: span of 28 generators
    gens = rng.random((28, 2000)) < 0.3
    spans = []
    for rows in (12500, 10000):
        pick = rng.random((rows, 28)) < 0.5
        spans.append(((pick.astype(np.uint8) @ gens.astype(np.uint8)) % 2).astype(bool))
        rng.standard_normal(rows), rng.standard_normal(rows)   # the coefficient draws, to keep the stream aligned
    print("span-28 operands:", pass_rates(*spans), flush=True)


if __name__ == "__main__":
    main()
