"""TEST INFRASTRUCTURE -- numpy restatement of the seeded permutation generator (pgx_random_perms,
include/pgx.h) and of the curve moments (pgx_curve_moments).

The recipe, restated from include/pgx.h:

* Philox4x32-10 (Salmon et al., SC'11), key = (seed & 0xffffffff, seed >> 32).
* B(N) = the largest power of two <= ceil(N / 2), b = log2 B.  For N <= 65,503, B <= 16,384.
* Permutation i (a 64-bit global index; lo = i & 0xffffffff, hi = i >> 32):
  1. genome c draws bucket  w >> (32 - b)  (0 when b == 0), w = word c % 4 of
     Philox((c // 4, lo, hi, 0), key);
  2. each bucket's genomes are put in ascending genome order;
  3. bucket k of m genomes is Fisher-Yates shuffled from the top: for j = m-1 .. 1, draw v = w & mask(j)
     (mask = smallest 2^t - 1 >= j) until v <= j, swap entries j and v; the t-th word the bucket consumes is
     word t % 4 of Philox((k, lo, hi, 0x80000000 | t // 4), key);
  4. the row is bucket 0, bucket 1, ..., bucket B-1.
"""
from __future__ import annotations

import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_MASK32 = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of counters (c0, c1, c2, c3) and key (k0, k1), elementwise; returns four uint32 arrays."""
    c = [np.asarray(v, dtype=np.uint64) & _MASK32 for v in (c0, c1, c2, c3)]
    k0 = np.asarray(k0, dtype=np.uint64) & _MASK32
    k1 = np.asarray(k1, dtype=np.uint64) & _MASK32
    for r in range(10):
        if r:
            k0 = (k0 + _W0) & _MASK32
            k1 = (k1 + _W1) & _MASK32
        p0 = _M0 * c[0]
        p1 = _M1 * c[2]
        c = [(p1 >> _S32) ^ c[1] ^ k0, p1 & _MASK32, (p0 >> _S32) ^ c[3] ^ k1, p0 & _MASK32]
    return tuple(v.astype(np.uint32) for v in c)


def n_buckets(n):
    """B(N): the largest power of two <= ceil(N / 2) (1 for N <= 2)."""
    half = (int(n) + 1) // 2
    return 1 << (max(half, 1).bit_length() - 1)


def _key(seed):
    seed = int(seed)
    if not 0 <= seed < 2 ** 64:
        raise ValueError("seed must be in [0, 2^64)")
    return seed & 0xFFFFFFFF, seed >> 32


def random_perms(seed, first, n_perm, n):
    """Rows first .. first + n_perm - 1 of the permutation stream of ``seed`` over N = ``n`` genomes (uint16)."""
    n, n_perm, first = int(n), int(n_perm), int(first)
    k0, k1 = _key(seed)
    idx = np.arange(first, first + n_perm, dtype=np.uint64)
    lo, hi = idx & _MASK32, idx >> _S32
    B = n_buckets(n)
    bits = B.bit_length() - 1
    # 1. buckets
    c = np.arange(n, dtype=np.uint64)
    words = philox4x32_10((c >> np.uint64(2))[None, :], lo[:, None], hi[:, None], 0, k0, k1)
    sel = (c & np.uint64(3)).astype(np.int64)
    w = np.choose(sel[None, :].repeat(n_perm, 0), words) if n_perm else np.zeros((0, n), np.uint32)
    bucket = (w.astype(np.int64) >> (32 - bits)) if bits else np.zeros((n_perm, n), dtype=np.int64)
    # 2. ascending genome order inside each bucket, buckets in order
    rows = np.argsort(bucket * n + np.arange(n)[None, :], axis=1, kind="stable")
    counts = np.zeros((n_perm, B), dtype=np.int64)
    np.add.at(counts, (np.repeat(np.arange(n_perm), n), bucket.ravel()), 1)
    starts = np.cumsum(counts, axis=1) - counts
    # 3. Fisher-Yates inside every bucket of two or more genomes, all buckets in lockstep
    pi, pk = np.nonzero(counts >= 2)
    base = starts[pi, pk]
    j = counts[pi, pk] - 1
    t = np.zeros(pi.shape[0], dtype=np.int64)
    while pi.size:
        m = j.copy()
        for s in (1, 2, 4, 8, 16):
            m |= m >> s
        f = philox4x32_10(pk, lo[pi], hi[pi], np.uint64(0x80000000) | (t >> 2).astype(np.uint64), k0, k1)
        wv = np.choose(t & 3, f).astype(np.int64)
        v = wv & m
        ok = v <= j
        a, b = pi[ok], base[ok]
        x, y = b + j[ok], b + v[ok]
        tmp = rows[a, x].copy()
        rows[a, x] = rows[a, y]
        rows[a, y] = tmp
        t += 1
        j = np.where(ok, j - 1, j)
        live = j >= 1
        pi, pk, base, j, t = pi[live], pk[live], base[live], j[live], t[live]
    return rows.astype(np.uint16)


def curve_moments(curves):
    """Exact column moments of an integer [n_rows, width] block: (sum int64, sum of squares uint64, min, max int32)."""
    x = np.asarray(curves, dtype=np.int64)
    return (x.sum(axis=0), (x.astype(np.uint64) ** 2).sum(axis=0, dtype=np.uint64),
            x.min(axis=0).astype(np.int32), x.max(axis=0).astype(np.int32))
