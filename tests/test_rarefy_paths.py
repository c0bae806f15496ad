"""Rarefaction paths that random tables reach only by chance, or not at all.

  A  pgx_pan_core_curves_f64, the device float64 entry point: its packed-bin scan instances are reachable through it
     alone.  Every genome count that changes the launch shape, aligned and unaligned scratch and output, guard words.
  B  Profiled calls (pgx_profile_enable): the row kernels run back to back on the caller's stream, without the second
     stream and its gate.  Only the device-pointer calls are profiled; host-buffer calls never are (include/pgx.h).
  C  Concurrent device calls: two host threads on their own streams (each thread has its own second stream, fork/join
     events and list-CTA counter of the probe gate), and one thread alternating between two streams.
  D  Built tables for two branches of the row kernels:
       * the list kernel's min == 0 events (the statistic is then the mex of the list's ranks), queued per warp,
         resolved 32 at a time and flushed at the end;
       * the probe kernel's straggler hand-over: from rank 64, once at most 16 genes of a superblock are pending, the
         warp finishes them one gene at a time.
     The genome orders share a fixed prefix (and, for the probe tables, a fixed suffix), so every statistic is exact
     and the same in every slot of a batch.  CPU tests pin what the builders build.

Every curve is compared bit for bit with oracle.pan_core_curves_minrank, an exact integer reference.
"""
import ctypes
import os
import subprocess
import sys
import threading

import numpy as np
import pytest
import scipy.sparse

from conftest import REPO, draw_perms
from test_int32_bins import (INT32_HEAVY, _device_perms, _engine, _mixed_matrix, chosen_orders, edge_orders,
                             heavy_table, oracle_curves)

PREFIX = 160                    # genomes every order of section D starts with
SUFFIX = 3                      # genomes every order of the probe tables ends with
STRAGGLER_MIN_RANK = 64         # csrc/pgx_rarefy.cu: the hand-over is considered from this rank on ...
STRAGGLER_MAX = 16              # ... once at most this many genes of a superblock are pending (PGX_PROBE_STRAGGLERS)
MEX_THRESHOLD = 96              # long_threshold of the mex tables: lists of up to 95 genomes stay list rows
PGX_OK, PGX_ERR_INVALID = 0, 1
BINS = ["packed", "int32"]


# ---------------------------------------------------------------------------------------------------------------
# Builders
# ---------------------------------------------------------------------------------------------------------------
def prefix_orders(n, count, seed, prefix, suffix=(), rotations=None):
    """``count`` genome orders: ``prefix`` (rotated left by rotations[i] in order i), a random middle, ``suffix``."""
    rng = np.random.RandomState(seed)
    prefix, suffix = np.asarray(prefix, dtype=np.int64), np.asarray(suffix, dtype=np.int64)
    middle = np.setdiff1d(np.arange(n), np.r_[prefix, suffix])
    rows = [np.r_[np.roll(prefix, -(0 if rotations is None else int(rotations[i]))), rng.permutation(middle), suffix]
            for i in range(count)]
    return np.stack(rows).astype(np.int64)


def gene_statistics(coo, order):
    """(first presence, first absence) rank of every gene under one genome order (n where there is none)."""
    x = coo.toarray() != 0
    n = x.shape[1]
    rank = np.empty(n, dtype=np.int64)
    rank[order] = np.arange(n)
    return np.where(x, rank, n).min(axis=1), np.where(~x, rank, n).min(axis=1)


def mex_table(n, threshold=MEX_THRESHOLD, seed=0):
    """List rows whose list holds prefix[0 .. k-1] plus up to four genomes outside the prefix, and not prefix[k], for
    k = 1 .. threshold - 1: five present-list rows and four absent-list rows per k, 9 (threshold - 1) rows in all (odd
    for an even threshold).  Under an order that starts with the prefix every row's list holds the rank-0 genome, so
    its minimum rank is 0 and the statistic is the mex, exactly k: the first absence of a present-list row, the first
    presence of an absent-list row.  Returns (table, prefix, k of every row, absent-list flag of every row, list
    lengths)."""
    rng = np.random.RandomState(seed)
    prefix = rng.permutation(n)[:PREFIX]
    outside = np.setdiff1d(np.arange(n), prefix)
    rows, ks, absent, lengths = [], [], [], []
    for is_absent, reps in ((False, 5), (True, 4)):
        for k in range(1, threshold):
            for _ in range(reps):
                extra = rng.randint(1 if k == 1 else 0, min(4, threshold - 1 - k) + 1)
                row = np.zeros(n, dtype=bool)
                row[prefix[:k]] = True
                row[rng.choice(outside, extra, replace=False)] = True
                lengths.append(k + extra)
                rows.append(~row if is_absent else row)
                ks.append(k)
                absent.append(is_absent)
    coo = scipy.sparse.coo_matrix(np.array(rows, dtype=np.int64))
    return coo, prefix, np.array(ks), np.array(absent), np.array(lengths)


def mex_orders(n, prefix, count, variant, seed=1):
    """"shared": every order starts with the prefix.  "rotated": order i starts with the prefix rotated left by i % 8,
    so the slots of a list batch see different mex values (k - r, or no event where r >= k)."""
    return prefix_orders(n, count, seed, prefix, rotations=None if variant == "shared" else np.arange(count) % 8)


def mex_expected(ks, absent, rotation):
    """(first presence, first absence) of every mex_table row under an order whose prefix is rotated by ``rotation``."""
    event = rotation < ks
    stat = np.where(event, ks - rotation, PREFIX - rotation)          # the mex, or the rank of prefix[0]
    # a present list holding the rank-0 genome: first presence 0, first absence the mex; otherwise first absence 0
    # and first presence the rank of prefix[0].  Absent lists mirror it.
    on_pan = event == absent
    return np.where(on_pan, stat, 0), np.where(on_pan, 0, stat)


def straggler_genes(n, variant):
    """(statistic, rank-0 bit) of the genes whose walks pass rank 64.  Bit 0: the statistic is a first presence (pan
    side), bit 1: a first absence (core side).  "16": exactly 16 genes at or past rank 64, the hand-over happens at
    64.  "17": 17 at 64 (no hand-over), 12 at 96.  "17/16": 17 at 64, exactly 16 at 96."""
    sixteen = [(64, 0), (64, 1), (95, 0), (95, 1), (96, 0), (96, 1), (97, 1), (120, 0), (127, 1), (128, 0),
               (159, 0), (159, 1), (n - 3, 0), (n - 3, 1), (n - 2, 0), (n - 2, 1)]
    if variant == "16":
        return sixteen
    if variant == "17":
        return sixteen + [(80, 1)]
    assert variant == "17/16"
    return [(64, 0), (96, 0), (96, 1), (100, 0), (110, 1), (127, 0), (128, 1), (130, 0), (131, 1), (140, 0), (150, 1),
            (159, 0), (159, 1), (n - 3, 0), (n - 3, 1), (n - 2, 0), (n - 2, 1)]


def straggler_table(n, variant, low_extra=200, seed=0):
    """Genes for the probe kernel (plan them with long_threshold=2: every folded gene is a bitmap row).  Every flip
    rank 1 .. 63 on both sides, ``low_extra`` more below 64, and straggler_genes(n, variant).  A gene of statistic
    s < PREFIX holds bit v on prefix[0 .. s-1] and 1 - v on prefix[s], random bits elsewhere.  A gene of statistic
    n - 3 or n - 2 holds v everywhere but on two suffix genomes (n - 2 is the largest statistic of a folded gene:
    constant over n - 2 ranks).  The planner orders bitmap rows by folded length; the random bits' densities differ
    (0.05 .. 0.5 for the extra genes, 0.15 or 0.5 for the stragglers) so that stragglers land in several lanes and, with
    two superblocks, in both.  Returns (table, prefix, suffix, statistics, rank-0 bits)."""
    rng = np.random.RandomState(seed)
    perm = rng.permutation(n)
    prefix, suffix = perm[:PREFIX], perm[PREFIX:PREFIX + SUFFIX]
    genes = [(s, v) for s in range(1, STRAGGLER_MIN_RANK) for v in (0, 1)]
    genes += list(zip(rng.randint(1, STRAGGLER_MIN_RANK, low_extra), rng.randint(0, 2, low_extra)))
    high = straggler_genes(n, variant)
    genes += high
    density = np.r_[np.full(2 * (STRAGGLER_MIN_RANK - 1), 0.5), rng.uniform(0.05, 0.5, low_extra),
                    np.resize([0.15, 0.5], len(high))]
    x = np.empty((len(genes), n), dtype=bool)
    for i, (s, v) in enumerate(genes):
        if s < PREFIX:
            row = rng.random_sample(n) < density[i]
            row[prefix[:s]] = v
            row[prefix[s]] = not v
        else:
            row = np.full(n, bool(v))
            row[suffix[s - (n - SUFFIX)]] = not v                    # rank s: suffix[0] (n - 3) or suffix[1] (n - 2)
            row[suffix[2]] = not v                                   # and the last genome: the gene is not a closed form
        x[i] = row
    stats = np.array([g[0] for g in genes], dtype=np.int64)
    bits = np.array([g[1] for g in genes], dtype=np.int64)
    return scipy.sparse.coo_matrix(x.astype(np.int64)), prefix, suffix, stats, bits


def superblock_layout(hp):
    """(superblock, lane, word, bit) of every gene in the bitmap, indexed by gene."""
    w = hp.slice_words
    pos = np.full(hp.n_genes, -1, dtype=np.int64)
    pos[hp.long_gene] = np.arange(hp.n_long)
    within = pos % (1024 * w)
    return pos // (1024 * w), within // (32 * w), (within % (32 * w)) // 32, within % 32, pos


def pending_at(stats, superblock, rank):
    """Genes of every superblock still pending when the walk reaches ``rank``."""
    return np.bincount(superblock[stats >= rank], minlength=int(superblock.max()) + 1)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the builders build what the GPU tests rely on
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [333, 700])
def test_mex_table_plans_to_list_rows_with_the_intended_statistics(n):
    from pangenomix_b200.plan import build_host_plan
    coo, prefix, ks, absent, lengths = mex_table(n, seed=n)
    hp = build_host_plan(coo, long_threshold=MEX_THRESHOLD)
    rows = 9 * (MEX_THRESHOLD - 1)
    assert hp.n_rows == rows == ks.size and rows % 2 == 1 and hp.n_long == 0
    assert hp.n_empty == hp.n_full == 0 and not hp.w_present.any() and not hp.w_absent.any()
    assert np.array_equal(np.sort(hp.row_len), np.sort(lengths)) and lengths.max() == MEX_THRESHOLD - 1
    assert int(hp.row_absent.sum()) == int(absent.sum()) == 4 * (MEX_THRESHOLD - 1)
    # sub-block classes (chunk count, list kind): full sub-blocks of 32 rows, and most classes end in a ragged one
    _, counts = np.unique(np.c_[(hp.row_len + 7) // 8, hp.row_absent], axis=0, return_counts=True)
    assert counts.size == 24 and counts.max() > 32 and (counts % 32 != 0).sum() >= 18
    for variant in ("shared", "rotated"):
        orders = mex_orders(n, prefix, 13, variant, seed=n)
        assert all(np.array_equal(np.sort(o), np.arange(n)) for o in orders)
        for i, order in enumerate(orders):
            rotation = 0 if variant == "shared" else i % 8
            fp, fa = gene_statistics(coo, order)
            want_fp, want_fa = mex_expected(ks, absent, rotation)
            assert np.array_equal(fp, want_fp) and np.array_equal(fa, want_fa), (variant, i)
    # min == 0 events of a batch of B orders that share the prefix: every row in every slot.  The row count is odd, so
    # a warp that serves all rows of a batch (one warp per CTA, one row split) ends with 1 to 31 events to flush.
    for b in (1, 2, 4, 8):
        for p0 in range(0, 13, b):
            events = rows * min(b, 13 - p0)
            assert 1 <= events % 32 <= 31 and events >= 32, (b, p0)


@pytest.mark.parametrize("n", [1000, 1023, 1025])
@pytest.mark.parametrize("variant", ["16", "17", "17/16"])
@pytest.mark.parametrize("slice_words", [1, 2, 4])
def test_straggler_table_plans_to_one_superblock_with_the_intended_flips(n, variant, slice_words):
    from pangenomix_b200.plan import build_host_plan
    coo, prefix, suffix, stats, bits = straggler_table(n, variant)
    hp = build_host_plan(coo, long_threshold=2, slice_words=slice_words)
    assert hp.n_rows == 0 and hp.n_long == stats.size < 1024 * slice_words and hp.n_superblocks == 1
    orders = prefix_orders(n, 11, n, prefix, suffix)
    for order in orders[[0, 5, 10]]:
        fp, fa = gene_statistics(coo, order)
        assert np.array_equal(fp, np.where(bits == 0, stats, 0)) and np.array_equal(fa, np.where(bits == 1, stats, 0))
    pairs = set(zip(stats.tolist(), bits.tolist()))
    flips = (63, 96, n - 2) if variant == "17/16" else (63, 64, 95, 96, n - 2)
    assert all((s, v) in pairs for s in flips for v in (0, 1))
    superblock, lane, word, bit, _ = superblock_layout(hp)
    at64, at96 = pending_at(stats, superblock, 64)[0], pending_at(stats, superblock, 96)[0]
    assert (at64, at96) == {"16": (16, 12), "17": (17, 12), "17/16": (17, 16)}[variant]
    assert at96 <= STRAGGLER_MAX
    # n - 2 lies in the ragged last group of 32 ranks at N = 1,000 and 1,023; at 1,025 that group holds rank n - 1
    # alone, where no folded gene can flip
    assert (n - 2 >= (n - 1) // 32 * 32) == (n != 1025)
    # the hand-over must take a gene's rank-0 bits from the lane that owns the gene: some straggler sits in another
    # lane than 0 and its rank-0 bit differs from the bit of lane 0's gene in the same word and bit position
    late = np.flatnonzero(stats >= 64)
    lane0 = {(int(word[g]), int(bit[g])): int(bits[g]) for g in range(stats.size) if lane[g] == 0}
    assert any(lane[g] != 0 and lane0.get((int(word[g]), int(bit[g])), 0) != bits[g] for g in late)


@pytest.mark.parametrize("n", [1000, 1025])
def test_two_superblock_straggler_table(n):
    """The second superblock of the ragged variant is partial, and both superblocks hold genes that reach the
    hand-over."""
    from pangenomix_b200.plan import build_host_plan
    coo, prefix, suffix, stats, bits = straggler_table(n, "17", low_extra=1200, seed=3)
    hp = build_host_plan(coo, long_threshold=2, slice_words=1)
    assert hp.n_superblocks == 2 and 1024 < hp.n_long < 2048
    superblock = superblock_layout(hp)[0]
    assert (pending_at(stats, superblock, 64) >= 1).all() and (pending_at(stats, superblock, 96) <= STRAGGLER_MAX).all()
    fp, fa = gene_statistics(coo, prefix_orders(n, 1, n, prefix, suffix)[0])
    assert np.array_equal(np.maximum(fp, fa), stats)


# ---------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def engine_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")
    from pangenomix_b200 import _native, engine
    _native.load()
    yield engine
    _native.set_tuning(0, 0, 0)
    _native.profile_enable(False)


def _f64_status(eng, d_perms, n_perm, hist, curves):
    """pgx_pan_core_curves_f64 on the current torch stream; returns the status."""
    import torch
    from pangenomix_b200 import _native
    ptr = lambda t: t if t is None else t.data_ptr()                                 # noqa: E731
    with torch.cuda.device(eng.device):
        return _native.load().pgx_pan_core_curves_f64(ctypes.byref(eng.c_plan), ptr(d_perms), int(n_perm), ptr(hist),
                                                      ptr(curves), torch.cuda.current_stream(eng.device).cuda_stream)


def curves_f64(eng, d_perms, hist_offset=0, out_offset=0):
    """Float64 curves from pgx_pan_core_curves_f64, with the int32 scratch and the output as views at element offsets
    of larger buffers; the words around both must stay untouched."""
    import torch
    from pangenomix_b200 import _native
    n_perm, n = int(d_perms.shape[0]), eng.n_genomes
    size = n_perm * 2 * n
    hist_buf = torch.full((size + hist_offset + 4,), -5, dtype=torch.int32, device=eng.device)
    out_buf = torch.full((size + out_offset + 4,), -3.5, dtype=torch.float64, device=eng.device)
    hist = hist_buf[hist_offset:hist_offset + size]
    out = out_buf[out_offset:out_offset + size].view(n_perm, 2 * n)
    _native.check(_f64_status(eng, d_perms, n_perm, hist, out))
    assert np.all(torch.cat([hist_buf[:hist_offset], hist_buf[hist_offset + size:]]).cpu().numpy() == -5)
    assert np.all(torch.cat([out_buf[:out_offset], out_buf[out_offset + size:]]).cpu().numpy() == -3.5)
    return out.cpu().numpy()


def _tuned(tuning, calls):
    from pangenomix_b200 import _native
    _native.set_tuning(*tuning)
    try:
        return calls()
    finally:
        _native.set_tuning(0, 0, 0)


# ---------------------------------------------------------------------------------------------------------------
# A: device float64 curves
# ---------------------------------------------------------------------------------------------------------------
# N: the scatter prep (up to 18,773 genomes packed, 11,264 int32) and the gathering prep; list batches of 8 (up to
# ~14k genomes), 4 (20,000), 2 (40,000) and 1 (65,503); vector and scalar prep and scan (N % 8).
F64_GENOMES = [1, 3, 8, 33, 700, 2304, 20000, 40000, 65503]
# (d_hist, d_curves) element offsets: 16-byte aligned, and 4 / 8 bytes off a 16-byte boundary (the scalar paths)
F64_LAYOUTS = [(0, 0), (1, 0), (0, 1), (1, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
@pytest.mark.parametrize("rows", ["both", "lists"])
@pytest.mark.parametrize("n", F64_GENOMES)
def test_f64_entry_point_at_every_launch_shape(engine_mod, n, rows, bins):
    coo = _mixed_matrix(n, seed=n, per_class=24 if n <= 2304 else 4)
    eng = _engine(engine_mod, coo, bins, long_threshold=None if rows == "both" else 0)
    hp = eng.host_plan
    if rows == "both" and n >= 700:
        assert hp.n_rows > 0 and hp.n_long > 0
    if rows == "lists":
        assert hp.n_long == 0
    perms = edge_orders(hp, 13 if n <= 2304 else 5, seed=n).astype(np.uint16)
    want = oracle_curves(coo, perms)
    d_perms = _device_perms(perms)
    for hist_offset, out_offset in F64_LAYOUTS:
        got = curves_f64(eng, d_perms, hist_offset, out_offset)
        assert got.dtype == np.float64 and np.array_equal(got, want.astype(np.float64)), (hist_offset, out_offset)
    assert np.array_equal(eng.curves_device(d_perms).cpu().numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [12000, 12001])
def test_f64_entry_point_on_native_int32_bins(engine_mod, n):
    """The heavy-genome table (66,000 genes in one genome): int32 bins by themselves, the gathering prep (vector at
    12,000, scalar at 12,001) and a step of exactly 66,000 in one bin."""
    coo = heavy_table(n, INT32_HEAVY, seed=n)
    eng = engine_mod.PanCoreEngine(coo)
    assert eng.c_plan.max_colsum == INT32_HEAVY
    perms = np.r_[chosen_orders(n, 4), draw_perms(4, n, 3)].astype(np.uint16)
    want = oracle_curves(coo, perms)
    d_perms = _device_perms(perms)
    for hist_offset, out_offset in F64_LAYOUTS:
        assert np.array_equal(curves_f64(eng, d_perms, hist_offset, out_offset), want.astype(np.float64))
    assert np.array_equal(eng.curves_device(d_perms).cpu().numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
def test_f64_entry_point_arguments(engine_mod, bins):
    import torch
    coo = _mixed_matrix(33, seed=1)
    eng = _engine(engine_mod, coo, bins, long_threshold=8)
    d_perms = _device_perms(draw_perms(1, 33, 3).astype(np.uint16))
    hist = torch.full((3 * 66,), -5, dtype=torch.int32, device=eng.device)
    out = torch.full((3, 66), -3.5, dtype=torch.float64, device=eng.device)
    # no permutations: nothing is written, null pointers included
    assert _f64_status(eng, d_perms, 0, hist, out) == PGX_OK
    assert _f64_status(eng, None, 0, None, None) == PGX_OK
    torch.cuda.synchronize()
    assert (hist == -5).all() and (out == -3.5).all()
    assert _f64_status(eng, d_perms, 3, None, out) == PGX_ERR_INVALID
    assert _f64_status(eng, d_perms, 3, hist, None) == PGX_ERR_INVALID
    assert _f64_status(eng, d_perms, -1, hist, out) == PGX_ERR_INVALID
    torch.cuda.synchronize()
    assert (out == -3.5).all()
    assert _f64_status(eng, d_perms, 3, hist, out) == PGX_OK
    assert np.array_equal(out.cpu().numpy(), oracle_curves(coo, draw_perms(1, 33, 3)).astype(np.float64))


# ---------------------------------------------------------------------------------------------------------------
# B: profiled launches
# ---------------------------------------------------------------------------------------------------------------
PROFILE_TABLES = {"both": 40, "lists": 0, "bitmap": 2}        # long_threshold of _mixed_matrix(700)


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
@pytest.mark.parametrize("rows", list(PROFILE_TABLES))
def test_profiled_calls_give_the_same_curves(engine_mod, rows, bins):
    """With per-kernel timing on, the row kernels run one after the other on the caller's stream.  Two device calls are
    profiled; the host-buffer calls in between are not (include/pgx.h), in either bin format."""
    from pangenomix_b200 import _native
    coo = _mixed_matrix(700, seed=9)
    eng = _engine(engine_mod, coo, bins, long_threshold=PROFILE_TABLES[rows])
    hp = eng.host_plan
    assert (hp.n_tasks > 0) == (rows != "bitmap") and (hp.n_long > 0) == (rows != "lists")
    perms = edge_orders(hp, 21, seed=9).astype(np.uint16)
    want = oracle_curves(coo, perms)
    d_perms = _device_perms(perms)
    _native.profile_read()
    _native.profile_enable(True)
    try:
        got = eng.curves_device(d_perms).cpu().numpy()
        got_f64 = curves_f64(eng, d_perms, 1, 1)
        host = eng.curves_host(perms, perms_per_block=8)
        host_f64 = eng.curves_host(perms, out_f64=True)
        list_ms, probe_ms, other_ms, calls = _native.profile_read()
    finally:
        _native.profile_enable(False)
        _native.profile_read()
    assert np.array_equal(got, want) and np.array_equal(got_f64, want.astype(np.float64))
    assert np.array_equal(host, want) and np.array_equal(host_f64, want.astype(np.float64))
    assert calls == 2
    assert (list_ms > 0) == (hp.n_tasks > 0) and (probe_ms > 0) == (hp.n_long > 0) and other_ms > 0


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
def test_host_buffer_calls_are_never_profiled(engine_mod, bins):
    """int32-bin host-buffer calls run the same curve kernels as the device calls; profiling still leaves them alone
    (and their two-stream schedule with them)."""
    from pangenomix_b200 import _native
    coo = _mixed_matrix(333, seed=4)
    eng = _engine(engine_mod, coo, bins, long_threshold=20)
    perms = edge_orders(eng.host_plan, 17, seed=4).astype(np.uint16)
    want = oracle_curves(coo, perms)
    _native.profile_read()
    _native.profile_enable(True)
    try:
        assert np.array_equal(eng.curves_host(perms, perms_per_block=5), want)
        assert np.array_equal(eng.curves_host(perms, out_f64=True), want.astype(np.float64))
        np.random.seed(4)
        assert np.array_equal(eng.estimate(17), oracle_curves(coo, draw_perms(4, 333, 17)).astype(np.float64))
        assert _native.profile_read() == (0.0, 0.0, 0.0, 0)
        assert np.array_equal(eng.curves_device(_device_perms(perms)).cpu().numpy(), want)
        assert _native.profile_read()[3] == 1
    finally:
        _native.profile_enable(False)
        _native.profile_read()


# ---------------------------------------------------------------------------------------------------------------
# C: concurrent device calls
# ---------------------------------------------------------------------------------------------------------------
def _two_threads(jobs, rounds):
    """Runs ``jobs`` (engine, list of CUDA permutation tensors) in one thread each, every thread on a torch stream of its
    own, ``rounds`` calls each without synchronising in between; returns the curves of every call."""
    import torch
    barrier = threading.Barrier(len(jobs))
    results, errors = [None] * len(jobs), []

    def work(j, eng, perms):
        try:
            stream = torch.cuda.Stream(device=eng.device)
            with torch.cuda.stream(stream):
                barrier.wait()
                outs = [eng.curves_device(perms[r % len(perms)]) for r in range(rounds)]
            stream.synchronize()
            results[j] = [o.cpu().numpy() for o in outs]
        except BaseException as e:                              # noqa: BLE001 - reported by the caller
            errors.append(e)
            barrier.abort()

    threads = [threading.Thread(target=work, args=(j, eng, perms)) for j, (eng, perms) in enumerate(jobs)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    return results


def _perm_sets(coo, hp, seed, sets=3, count=64):
    perms = [edge_orders(hp, count, seed=seed + s).astype(np.uint16) for s in range(sets)]
    return [_device_perms(p) for p in perms], [oracle_curves(coo, p) for p in perms]


@pytest.mark.gpu
@pytest.mark.parametrize("engines", ["shared", "two"])
def test_two_threads_call_curves_device_at_once(engine_mod, engines):
    import torch
    coo_a = _mixed_matrix(700, seed=31)
    eng_a = _engine(engine_mod, coo_a, "packed", long_threshold=40)
    d_a, want_a = _perm_sets(coo_a, eng_a.host_plan, 1)
    if engines == "shared":
        jobs = [(eng_a, d_a), (eng_a, d_a[::-1])]
        wants = [want_a, want_a[::-1]]
    else:
        coo_b = _mixed_matrix(333, seed=32)
        eng_b = _engine(engine_mod, coo_b, "int32", long_threshold=20)
        d_b, want_b = _perm_sets(coo_b, eng_b.host_plan, 2)
        jobs, wants = [(eng_a, d_a), (eng_b, d_b)], [want_a, want_b]
    for hp in (eng.host_plan for eng, _ in jobs):
        assert hp.n_tasks > 0 and hp.n_long > 0                           # both row kernels, the second stream, the gate
    torch.cuda.synchronize()
    rounds = 8
    results = _two_threads(jobs, rounds)
    for j, want in enumerate(wants):
        for r in range(rounds):
            assert np.array_equal(results[j][r], want[r % len(want)]), (j, r)


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
def test_one_thread_alternates_between_two_streams(engine_mod, bins):
    import torch
    coo = _mixed_matrix(700, seed=33)
    eng = _engine(engine_mod, coo, bins, long_threshold=40)
    d_perms, wants = _perm_sets(coo, eng.host_plan, 5)
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = []
    for r in range(8):
        with torch.cuda.stream(streams[r % 2]):
            outs.append(eng.curves_device(d_perms[r % 3]))
    torch.cuda.synchronize()
    for r, out in enumerate(outs):
        assert np.array_equal(out.cpu().numpy(), wants[r % 3]), r


# ---------------------------------------------------------------------------------------------------------------
# D: the list kernel's mex events
# ---------------------------------------------------------------------------------------------------------------
# (row splits, threads per CTA): one warp per CTA serving every row of a batch (its final flush holds 1 to 31 events),
# the heuristic, and several warps sharing the rows
MEX_TUNINGS = [(1, 32), (0, 0), (3, 256)]


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
@pytest.mark.parametrize("variant", ["shared", "rotated"])
@pytest.mark.parametrize("n", [333, 700])
def test_mex_events_in_every_batch_slot(engine_mod, n, variant, bins):
    coo, prefix, ks, absent, _ = mex_table(n, seed=n)
    eng = _engine(engine_mod, coo, bins, long_threshold=MEX_THRESHOLD)
    assert eng.host_plan.n_long == 0 and eng.host_plan.n_rows == ks.size
    perms = mex_orders(n, prefix, 13, variant, seed=n).astype(np.uint16)
    want = oracle_curves(coo, perms)
    d_perms = _device_perms(perms)
    for b in (1, 2, 4, 8):
        for splits, threads in MEX_TUNINGS:
            got = _tuned((b, splits, threads), lambda: eng.curves_device(d_perms).cpu().numpy())
            assert np.array_equal(got, want), (b, splits, threads)
    assert np.array_equal(_tuned((1, 1, 32), lambda: eng.curves_host(perms)), want)


# ---------------------------------------------------------------------------------------------------------------
# D: the probe kernel's straggler hand-over
# ---------------------------------------------------------------------------------------------------------------
def _straggler_cases():
    """(N, variant, slice_words, low_extra): one superblock at every width, and a second, ragged superblock."""
    one = [(n, v, w, 200) for n in (1000, 1023, 1025) for v in ("16", "17", "17/16") for w in (1, 2, 4)]
    return one + [(n, "17", 1, 1200) for n in (1000, 1025)]


def check_straggler_case(engine_mod, n, variant, slice_words, low_extra, bins):
    from pangenomix_b200.plan import build_host_plan
    coo, prefix, suffix, stats, _ = straggler_table(n, variant, low_extra=low_extra, seed=0 if low_extra == 200 else 3)
    hp = build_host_plan(coo, long_threshold=2, slice_words=slice_words)
    assert hp.n_rows == 0 and hp.n_long == stats.size
    eng = _engine(engine_mod, coo, bins, host_plan=hp)
    perms = prefix_orders(n, 11, n, prefix, suffix).astype(np.uint16)
    want = oracle_curves(coo, perms)
    assert np.array_equal(eng.curves_device(_device_perms(perms)).cpu().numpy(), want)
    assert np.array_equal(eng.curves_host(perms), want)


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
@pytest.mark.parametrize("n,variant,slice_words,low_extra", _straggler_cases())
def test_straggler_handover(engine_mod, n, variant, slice_words, low_extra, bins):
    check_straggler_case(engine_mod, n, variant, slice_words, low_extra, bins)


def probe_tables_child():
    """Every straggler table and _mixed_matrix bitmap tables under this process's PGX_PROBE_STRAGGLERS."""
    from pangenomix_b200 import engine
    from pangenomix_b200.plan import build_host_plan
    done = 0
    for case in _straggler_cases():
        for bins in BINS if case[2] == 1 else ["packed"]:
            check_straggler_case(engine, *case, bins)
            done += 1
    for n, seed, per_class, threshold, slice_words in [(1500, 2, 10, 2, None), (1500, 8, 300, 8, None),
                                                      (600, 21, 600, 6, 1), (600, 21, 600, 6, 2), (600, 21, 600, 6, 4)]:
        coo = _mixed_matrix(n, seed=seed, per_class=per_class)
        hp = build_host_plan(coo, long_threshold=threshold, slice_words=slice_words)
        assert hp.n_long > 0
        eng = engine.PanCoreEngine(coo, host_plan=hp)
        perms = edge_orders(hp, 40, seed=seed).astype(np.uint16)
        want = oracle_curves(coo, perms)
        assert np.array_equal(eng.curves_device(_device_perms(perms)).cpu().numpy(), want)
        assert np.array_equal(eng.curves_host(perms), want)
        done += 1
    print("probe tables ok: %d" % done)


@pytest.mark.gpu
@pytest.mark.parametrize("stragglers", ["0", "1", "100000"])
def test_straggler_threshold_in_a_child_process(engine_mod, stragglers):
    """PGX_PROBE_STRAGGLERS is read once per process.  0: no hand-over; 1: only the last gene of a walk; 100000: every
    warp hands over at rank 64, so every bitmap gene is finished by the one-gene-at-a-time scan."""
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import test_rarefy_paths\n"
            "test_rarefy_paths.probe_tables_child()\n" % (REPO, os.path.join(REPO, "tests")))
    env = dict(os.environ, PGX_PROBE_STRAGGLERS=stragglers)
    run = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    tables = sum(2 if case[2] == 1 else 1 for case in _straggler_cases()) + 5
    assert run.returncode == 0 and "probe tables ok: %d" % tables in run.stdout, run.stdout + run.stderr
