"""TEST INFRASTRUCTURE ONLY -- numpy / scipy restatements of the shared-gene matrix and genomic fluidity.

* ``shared_direct``      S = X^T X of the binary gene x genome table through scipy.
* ``shared_from_plan``   the same S from the classes of a plan (HostPlan of oracle/plan_np.py or of the library's
                         planner), term by term as include/pgx.h states it for pgx_shared_genes.
* ``fluidity_rows`` / ``fluidity_by_definition`` / ``jackknife_by_definition``
                         genomic fluidity (Kislyuk, Haegeman, Bergman & Weitz, BMC Genomics 12:32, 2011) and its
                         leave-one-genome-out jackknife, computed by their definitions from S.
"""
from __future__ import annotations

import math

import numpy as np

from .plan_np import SLICE_ROWS, gene_major_csr


def shared_direct(data):
    """int32 [N, N] S = X^T X, X the binary gene x genome table (``data`` as gene_major_csr takes it)."""
    x = gene_major_csr(data).astype(np.int64)
    return np.asarray((x.T @ x).toarray(), dtype=np.int32)


def _pair_counts(sorted_idx, sorted_ptr, rows, n):
    """[N, N] int64: +1 on (a, b), a < b, for every pair of the sorted lists of ``rows``."""
    out = np.zeros((n, n), dtype=np.int64)
    for r in rows:
        lst = np.asarray(sorted_idx[sorted_ptr[r]:sorted_ptr[r + 1]], dtype=np.int64)
        if lst.size > 1:
            a, b = np.triu_indices(lst.size, 1)
            np.add.at(out, (lst[a], lst[b]), 1)
    return out


def bitmap_dense(hp):
    """[N, n_long] uint8: bitmap row j of the plan in genome c (the E matrix of pgx_shared_genes, unpadded)."""
    n, w = hp.n_genomes, hp.slice_words
    if hp.n_long == 0:
        return np.zeros((n, 0), dtype=np.uint8)
    words = np.asarray(hp.bits, dtype=np.uint32).reshape(hp.n_superblocks, n, 32 * w)
    bits = np.unpackbits(words.view(np.uint8), axis=2, bitorder="little")        # [sb, N, 1024 W]
    dense = bits.transpose(1, 0, 2).reshape(n, hp.n_superblocks * SLICE_ROWS * w)
    return dense[:, :hp.n_long]


def shared_from_plan(hp):
    """S from the plan's classes: closed forms, absent / present list rows and the bitmap rows' product."""
    n = hp.n_genomes
    rows = np.arange(hp.n_rows)
    absent = np.asarray(hp.row_absent, dtype=bool)
    ptr = np.asarray(hp.sorted_ptr, dtype=np.int64)
    idx = np.asarray(hp.sorted_idx, dtype=np.int64)
    w_absent = np.asarray(hp.w_absent, dtype=np.int64)
    u = np.zeros(n, dtype=np.int64)
    for r in rows[absent]:
        u[idx[ptr[r]:ptr[r + 1]]] += 1
    e = bitmap_dense(hp).astype(np.int64)
    s = (hp.n_full + w_absent.sum() - w_absent[:, None] - w_absent[None, :]
         + int(absent.sum()) - u[:, None] - u[None, :]
         + _pair_counts(idx, ptr, rows, n) + e @ e.T)
    s = np.triu(s, 1)
    s = s + s.T
    s[np.diag_indices(n)] = hp.colsum
    return s.astype(np.int32)


def fluidity_distances(shared):
    """[N, N] float64 d_kl = (M_k + M_l - 2 S_kl) / (M_k + M_l), M = diag(S); NaN where M_k + M_l = 0."""
    s = np.asarray(shared, dtype=np.int64)
    m = np.diag(s)
    den = (m[:, None] + m[None, :]).astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        return (m[:, None] + m[None, :] - 2 * s) / den


def fluidity_rows(shared):
    """R[k] = sum over l != k of d_kl (what pgx_fluidity_rows computes)."""
    d = fluidity_distances(shared)
    np.fill_diagonal(d, 0.0)
    return np.array([math.fsum(row) for row in d])


def fluidity_by_definition(shared):
    """Mean of d_kl over the N (N - 1) / 2 pairs k < l."""
    d = fluidity_distances(shared)
    a, b = np.triu_indices(d.shape[0], 1)
    return math.fsum(d[a, b]) / a.size


def jackknife_by_definition(shared):
    """Leave-one-genome-out jackknife standard error: the fluidity of every table without genome i, recomputed."""
    s = np.asarray(shared)
    n = s.shape[0]
    if n < 3:
        return float("nan")
    loo = np.array([fluidity_by_definition(np.delete(np.delete(s, i, 0), i, 1)) for i in range(n)])
    return math.sqrt((n - 1) / n * float(np.sum((loo - loo.mean()) ** 2)))


def fluidity_brute(genome_sets):
    """Fluidity from gene sets: mean over pairs of |A ^ B| / (|A| + |B|)."""
    n = len(genome_sets)
    vals = [len(genome_sets[k] ^ genome_sets[l]) / (len(genome_sets[k]) + len(genome_sets[l]))
            for k in range(n) for l in range(k + 1, n)]
    return math.fsum(vals) / len(vals)


def shared_sample_rows(data, cols):
    """S[cols, :] = X[:, cols]^T X through scipy, for checking rows of a table too large for the whole product."""
    x = gene_major_csr(data).astype(np.int64).tocsc()
    return np.asarray((x[:, cols].T @ x).toarray(), dtype=np.int32)


__all__ = ["shared_direct", "shared_from_plan", "bitmap_dense", "fluidity_distances", "fluidity_rows",
           "fluidity_by_definition", "jackknife_by_definition", "fluidity_brute", "shared_sample_rows"]
