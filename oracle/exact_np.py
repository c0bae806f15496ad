"""TEST INFRASTRUCTURE ONLY -- numpy / python restatements of the exact pan/core rarefaction moments.

* ``spectrum_direct``           genes present in exactly v genomes, v = 0 .. N.
* ``pair_histograms_direct``    H_s[v] = #{g < h : s_gh = v} and H_a[v] = #{g < h : a_gh = v} from a blocked X X^T.
* ``pair_histograms_from_plan`` the same from the classes of a plan, term by term as include/pgx.h states it for
                                pgx_pair_overlap_histograms.
* ``moments_exact``             E / Var of the pan and core sizes of k-subsets in exact rationals.
* ``moments_longdouble``        the same in x87 long double, rho(v, k) as a running product over k (tables too
                                large for rationals).
* ``moments_enumerate``         the same by enumerating every k-subset of a tiny table.

Moments are [4][N] (rows E[pan_k], Var[pan_k], E[core_k], Var[core_k], k = 1 .. N), as pgx_rarefaction_moments
writes them.
"""
from __future__ import annotations

import itertools
import math
from fractions import Fraction

import numpy as np

from .plan_np import gene_major_csr
from .shared_np import bitmap_dense


def dense_table(data):
    """bool [G, N] gene x genome table."""
    return gene_major_csr(data).toarray().astype(bool)


def spectrum_direct(data):
    x = gene_major_csr(data)
    return np.bincount(np.diff(x.indptr), minlength=x.shape[1] + 1).astype(np.int64)


def _histograms_of_rows(rows, n, block=4096):
    """H_s / H_a over the pairs g < h of the rows of a [R, N] 0/1 matrix (float32 products: exact below 2^24)."""
    rows = np.asarray(rows, dtype=np.float32)
    m = rows.sum(axis=1).astype(np.int64)
    hs = np.zeros(n + 1, dtype=np.int64)
    ha = np.zeros(n + 1, dtype=np.int64)
    r = rows.shape[0]
    for i0 in range(0, r, block):
        for j0 in range(i0, r, block):
            s = (rows[i0:i0 + block] @ rows[j0:j0 + block].T).astype(np.int64)
            a = n - m[i0:i0 + block, None] - m[None, j0:j0 + block] + s
            if i0 == j0:
                keep = np.triu(np.ones(s.shape, dtype=bool), 1)
                s, a = s[keep], a[keep]
            hs += np.bincount(s.ravel(), minlength=n + 1)
            ha += np.bincount(a.ravel(), minlength=n + 1)
    return hs, ha


def pair_histograms_direct(data, block=4096):
    x = gene_major_csr(data)
    return _histograms_of_rows(x.toarray(), x.shape[1], block)


def _plan_rows(hp):
    """[R, N] uint8: the list rows (their genomes flipped from the default) then the bitmap rows of a plan."""
    n = hp.n_genomes
    ptr = np.asarray(hp.sorted_ptr, dtype=np.int64)
    idx = np.asarray(hp.sorted_idx, dtype=np.int64)
    absent = np.asarray(hp.row_absent, dtype=bool)
    lists = np.zeros((hp.n_rows, n), dtype=np.uint8)
    for r in range(hp.n_rows):
        lists[r] = 1 if absent[r] else 0
        lists[r, idx[ptr[r]:ptr[r + 1]]] = 0 if absent[r] else 1
    return np.vstack([lists, bitmap_dense(hp).T])


def pair_histograms_from_plan(hp):
    """H_s / H_a from the plan's classes: closed x row and closed x closed terms by the table of include/pgx.h, the
    stored rows' pairs by their product."""
    n = hp.n_genomes
    hs = np.zeros(n + 3, dtype=object)          # two spare bins absorb the zero-count terms of N = 1
    ha = np.zeros(n + 3, dtype=object)

    def add(s, a, count):
        if count:
            hs[s] += int(count)
            ha[a] += int(count)

    wp = np.asarray(hp.w_present, dtype=np.int64)
    wa = np.asarray(hp.w_absent, dtype=np.int64)
    e, u, p1, a1 = int(hp.n_empty), int(hp.n_full), int(wp.sum()), int(wa.sum())
    rows = _plan_rows(hp)
    for row in rows:
        m = int(row.sum())
        w_p, w_a = int(wp[row == 1].sum()), int(wa[row == 1].sum())
        add(0, n - m, e)
        add(m, 0, u)
        add(1, n - m, w_p)
        add(0, n - 1 - m, p1 - w_p)
        add(m - 1, 0, w_a)
        add(m, 1, a1 - w_a)
    same_p, same_a = int((wp * (wp - 1) // 2).sum()), int((wa * (wa - 1) // 2).sum())
    same_pa = int((wp * wa).sum())
    add(0, n, e * (e - 1) // 2)
    add(0, 0, e * u)
    add(0, n - 1, e * p1)
    add(0, 1, e * a1)
    add(n, 0, u * (u - 1) // 2)
    add(1, 0, u * p1)
    add(n - 1, 0, u * a1)
    add(1, n - 1, same_p)
    add(0, n - 2, p1 * (p1 - 1) // 2 - same_p)
    add(n - 1, 1, same_a)
    add(n - 2, 0, a1 * (a1 - 1) // 2 - same_a)
    add(0, 0, same_pa)
    add(1, 1, p1 * a1 - same_pa)
    rs, ra = _histograms_of_rows(rows, n)
    assert not any(hs[n + 1:]) and not any(ha[n + 1:])
    return (hs[:n + 1] + rs).astype(np.int64), (ha[:n + 1] + ra).astype(np.int64)


def moments_exact(spectrum, hs, ha, n_genes, n):
    """[4][N] Fractions.  rho(v, k) = C(v, k) / C(N, k); Z_k = sum_v spectrum[N - v] rho(v, k) genes absent from T."""
    spectrum = [int(v) for v in spectrum]
    hs = None if hs is None else [int(v) for v in hs]
    ha = None if ha is None else [int(v) for v in ha]
    out = [[None] * n for _ in range(4)]
    for k in range(1, n + 1):
        den = math.comb(n, k)
        combs = [math.comb(v, k) for v in range(n + 1)]
        core = Fraction(sum(spectrum[v] * combs[v] for v in range(n + 1)), den)
        none = Fraction(sum(spectrum[n - v] * combs[v] for v in range(n + 1)), den)
        out[0][k - 1] = n_genes - none
        out[2][k - 1] = core
        if hs is not None:
            out[1][k - 1] = none + 2 * Fraction(sum(ha[v] * combs[v] for v in range(n + 1)), den) - none * none
            out[3][k - 1] = core + 2 * Fraction(sum(hs[v] * combs[v] for v in range(n + 1)), den) - core * core
    return out


def moments_longdouble(spectrum, hs, ha, n_genes, n):
    """[4, N] np.longdouble, rho(v, k) = rho(v, k - 1) (v - k + 1) / (N - k + 1) for all v at once."""
    ld = np.longdouble
    v = np.arange(n + 1, dtype=ld)
    spec = np.asarray(spectrum, dtype=ld)
    rev = spec[::-1].copy()
    hs = None if hs is None else np.asarray(hs, dtype=ld)
    ha = None if ha is None else np.asarray(ha, dtype=ld)
    rho = np.ones(n + 1, dtype=ld)
    out = np.full((4, n), np.nan, dtype=ld)
    for k in range(1, n + 1):
        rho = rho * np.maximum(v - (k - 1), 0) / ld(n - k + 1)
        core, none = np.sum(spec * rho), np.sum(rev * rho)
        out[0, k - 1] = ld(n_genes) - none
        out[2, k - 1] = core
        if hs is not None:
            out[1, k - 1] = none + 2 * np.sum(ha * rho) - none * none
            out[3, k - 1] = core + 2 * np.sum(hs * rho) - core * core
    return out


def moments_enumerate(data):
    """[4][N] Fractions over every k-subset T of the genomes: pan = genes in some genome of T, core = in all."""
    x = dense_table(data)
    n = x.shape[1]
    out = [[None] * n for _ in range(4)]
    for k in range(1, n + 1):
        pans, cores = [], []
        for t in itertools.combinations(range(n), k):
            sub = x[:, list(t)]
            pans.append(int(sub.any(axis=1).sum()))
            cores.append(int(sub.all(axis=1).sum()))
        for row, vals in ((0, pans), (2, cores)):
            mean = Fraction(sum(vals), len(vals))
            out[row][k - 1] = mean
            out[row + 1][k - 1] = Fraction(sum(v * v for v in vals), len(vals)) - mean * mean
    return out


__all__ = ["dense_table", "spectrum_direct", "pair_histograms_direct", "pair_histograms_from_plan", "moments_exact",
           "moments_longdouble", "moments_enumerate"]
