"""The int32-bin rarefaction path, covered as closely as the packed uint16 one.

The kernels of csrc/pgx_rarefy.cu count histogram bins as packed uint16 pairs when 0 < max_colsum <= 65,535 and as
int32 otherwise: a genome with more than 65,535 genes, a table without entries, or a plan whose max_colsum is 0
("unknown", include/pgx.h).  Every template instance and the host-buffer pipeline exist twice, and the two formats
keep the core side differently (int32 core bin 0 = G - colsum[first], packed core bin 0 = colsum[first]).

Two ways to int32 bins are used here:
  * natively: heavy-genome tables whose genome h holds 66,000 genes (max_colsum > 65,535);
  * for any table, in process: ``max_colsum = 0`` written into an engine's uploaded plan (``_engine(..., "int32")``).

The heavy-genome table also sits exactly on the packed boundary (H = 65,535: still packed) and one past it
(H = 65,536: int32, where a uint16 bin would wrap and carry into its neighbour).  Chosen genome orders put a step of
exactly H into one bin, added by a ROW kernel (list or probe), not only by the closed forms.  Every curve is compared
bit for bit with oracle.pan_core_curves_minrank, an exact integer reference.
"""
import numpy as np
import pandas as pd
import pytest
import scipy.sparse

import oracle
from conftest import draw_perms

X, HEAVY = 0, 1                 # genome x (never a partner) and the heavy genome h of heavy_table()
SPLIT_HEAD = 512                # the host-buffer calls' default uint16 head of the split transfer (PGX_SPLIT_HEAD)
INT32_HEAVY = 66000             # genes of h in the native int32 tables


# ---------------------------------------------------------------------------------------------------------------
# Table builders and chosen genome orders
# ---------------------------------------------------------------------------------------------------------------
def partners(n):
    """The genomes that share a gene with h: the upper half (x = 0 and h = 1 are not among them)."""
    return np.arange(n // 2, n)


def heavy_table(n, heavy, seed=0):
    """Gene x genome COO table in which genome h holds ``heavy`` genes, each also present in exactly one partner genome
    (partners(n)), followed by 21 rows of the other classes: empty, single-genome, single-absence (every genome but h),
    short present lists, short absent lists and long lists.  None of those rows holds h, so colsum[h] == heavy exactly
    and every other genome holds far fewer genes.  (A universal row would hold h too; the mixed tables of the in-process
    int32 tests cover that class.)"""
    rng = np.random.RandomState(seed)
    others = np.delete(np.arange(n), HEAVY)
    lists = [np.zeros(0, dtype=np.int64)] * 3                                              # empty
    lists += [rng.choice(others, 1) for _ in range(3)]                                     # single-genome
    lists += [others] * 3                                                                  # single-absence: h
    lists += [rng.choice(others, k, replace=False) for k in (2, 5, 9)]                     # short present lists
    lists += [np.setdiff1d(others, rng.choice(others, k, replace=False)) for k in (1, 4, 8)]   # short absent lists
    lists += [others[rng.random_sample(others.size) < d] for d in (0.3, 0.5, 0.8)]        # long lists
    heavy_cols = np.empty(2 * heavy, dtype=np.int64)
    heavy_cols[0::2] = HEAVY
    heavy_cols[1::2] = rng.choice(partners(n), heavy)
    rows = np.r_[np.repeat(np.arange(heavy), 2), heavy + np.repeat(np.arange(len(lists)), [len(l) for l in lists])]
    cols = np.r_[heavy_cols, np.concatenate(lists)]
    return scipy.sparse.coo_matrix((np.ones(rows.size, dtype=np.int64), (rows, cols)), shape=(heavy + len(lists), n))


def middle_rank(n):
    """Rank of h in order C: 600 (past the split head of 512) from N = 2,400 on, N / 4 below."""
    return min(600, n // 4)


def chosen_orders(n, seed=0):
    """Orders A-D of heavy_table(n, ...):
      A  [x, h, ...]       pan step of exactly H at k = 1, added by a row kernel (every heavy gene first appears at h)
      B  [h, x, ...]       pan[0] = H from the closed form; core step of exactly H at k = 1 (list kernel: H mex events
                           in one permutation; probe kernel: the first bit that differs from h's)
      C  h at middle_rank  x and genomes that are not partners before h, so every heavy gene first appears at h: a pan
                           step of exactly H in the middle of the row (at N = 2,200 in the uint8 tail of the split)
      D  [x, ..., h]       h last: the last bin of the core side holds the rows missing h alone, the pan side's is 0
    """
    rng = np.random.RandomState(seed)
    rest = rng.permutation(np.arange(2, n))
    mid = middle_rank(n)
    before = rng.permutation(np.arange(2, n // 2))[:mid - 1]                # neither x, h nor a partner
    after = rng.permutation(np.setdiff1d(np.arange(2, n), before))
    return np.stack([np.r_[X, HEAVY, rest], np.r_[HEAVY, X, rest], np.r_[X, before, HEAVY, after], np.r_[X, rest, HEAVY]])


def oracle_curves(coo, perms):
    pan, core = oracle.pan_core_curves_minrank(coo, np.asarray(perms, dtype=np.int64))
    return np.hstack([pan, core]).astype(np.int32)


_ORACLE_CACHE = {}


def oracle_curves_cached(key, coo, perms):
    """oracle_curves of a table and orders that several parametrizations share (``key`` names them)."""
    if key not in _ORACLE_CACHE:
        _ORACLE_CACHE[key] = (np.array(perms), oracle_curves(coo, perms))
    cached_perms, want = _ORACLE_CACHE[key]
    assert np.array_equal(cached_perms, perms)
    return want


def assert_heavy_steps(want, n, heavy):
    """The steps orders A-D (rows 0-3 of ``want``) are built to produce."""
    pan, core = want[:, :n].astype(np.int64), want[:, n:].astype(np.int64)
    mid = middle_rank(n)
    assert pan[0, 1] - pan[0, 0] == heavy                                   # A
    assert pan[1, 0] == heavy and core[1, 0] - core[1, 1] == heavy           # B
    assert pan[2, mid] - pan[2, mid - 1] == heavy                           # C
    assert pan[3, n - 1] == pan[3, n - 2] and core[3, n - 2] - core[3, n - 1] == 3   # D


def edge_orders(hp, count, seed):
    """``count`` random orders; the last genome of every other one is chosen so that the last bin of a side is not 0
    (the genome with the most single-genome genes, then the one with the most single-absence genes)."""
    n = hp.n_genomes
    rng = np.random.RandomState(seed)
    perms = np.stack([rng.permutation(n) for _ in range(count)])
    ends = [int(np.argmax(hp.w_present)), int(np.argmax(hp.w_absent))]
    for i in range(0, count, 2):
        row = perms[i]
        j = int(np.flatnonzero(row == ends[(i // 2) % 2])[0])
        row[j], row[-1] = row[-1], row[j]
    return perms


# ---------------------------------------------------------------------------------------------------------------
# CPU: the builders, the planner and the oracle pin the design of the GPU tests
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [64, 2200, 12001])
@pytest.mark.parametrize("heavy", [65535, 65536, INT32_HEAVY])
def test_heavy_table_plans_to_the_intended_max_colsum(n, heavy):
    from pangenomix_b200.plan import build_host_plan
    coo = heavy_table(n, heavy)
    hp = build_host_plan(coo)
    assert int(hp.colsum.max()) == heavy and int(hp.colsum[HEAVY]) == heavy
    assert int(np.sort(hp.colsum)[-2]) < heavy // 8
    assert hp.n_empty == 3 and hp.n_full == 0 and int(hp.w_absent[HEAVY]) == 3 and int(hp.w_present.sum()) == 3


@pytest.mark.parametrize("n", [64, 2200, 12001])
def test_heavy_rows_go_to_the_row_kernel_each_case_names(n):
    from pangenomix_b200.plan import build_host_plan
    coo = heavy_table(n, 65536)
    heavy_genes = np.arange(65536)
    lists = build_host_plan(coo)                                            # default threshold: list rows
    assert lists.long_threshold > 2
    assert np.isin(heavy_genes, lists.row_gene).all() and not np.isin(heavy_genes, lists.long_gene).any()
    assert lists.n_long > 0                                                 # the long mixed rows: bitmap rows
    probe = build_host_plan(coo, long_threshold=2)                         # every general gene: bitmap rows
    assert np.isin(heavy_genes, probe.long_gene).all() and probe.n_rows == 0
    assert probe.slice_words == 4 and probe.n_superblocks == -(-probe.n_long // 4096)


@pytest.mark.parametrize("n", [64, 2200])
@pytest.mark.parametrize("heavy", [65535, 65536])
def test_chosen_orders_put_steps_of_exactly_h_into_one_bin(n, heavy):
    coo = heavy_table(n, heavy)
    orders = chosen_orders(n)
    assert all(np.array_equal(np.sort(o), np.arange(n)) for o in orders)
    assert orders[2, middle_rank(n)] == HEAVY and not np.isin(orders[2, :middle_rank(n)], partners(n)).any()
    want = oracle_curves(coo, orders)
    assert_heavy_steps(want, n, heavy)
    # steps after the split head stay below 256 except order C's, so only C forces the uint16 re-send at N = 2,200
    steps = np.diff(want[:, :n].astype(np.int64), axis=1)
    tail = steps[:, SPLIT_HEAD - 1:]
    if n >= 4 * SPLIT_HEAD:
        assert tail[[0, 1, 3]].max() <= 255 and tail[2].max() == heavy


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


def _engine(engine_mod, coo, bins, **kwargs):
    """An engine whose calls count in ``bins``: "packed" asserts the table's own plan packs; "int32" writes the ABI's
    "unknown" (max_colsum = 0) into the uploaded plan, which makes every kernel count in int32 bins."""
    eng = engine_mod.PanCoreEngine(coo, **kwargs)
    if bins == "int32":
        eng.c_plan.max_colsum = 0
        assert eng.c_plan.max_colsum == 0
    else:
        assert 0 < eng.c_plan.max_colsum <= 65535
    return eng


def _split_head():
    from pangenomix_b200 import _native
    return int(_native.load().pgx_split_head())


def _fresh_staging(engine_mod):
    """A host-buffer call on a 3-genome table: the next call at another genome count sets its staging up anew, with
    the default split head."""
    tiny = engine_mod.PanCoreEngine(scipy.sparse.coo_matrix(np.array([[1, 0, 1], [0, 1, 1]], dtype=np.int64)))
    tiny.curves_host(np.array([[0, 1, 2]], dtype=np.uint16))


def _device_perms(perms, odd=False):
    """perms as a CUDA int16 tensor; ``odd``: a view that starts one element (2 bytes) into its buffer."""
    import torch
    p = torch.from_numpy(np.ascontiguousarray(perms, dtype=np.uint16).view(np.int16)).cuda()
    if not odd:
        return p
    buf = torch.empty(p.numel() + 1, dtype=torch.int16, device="cuda")
    view = buf[1:].view(p.shape)
    view.copy_(p)
    return view


def _curves_into_offset_view(eng, d_perms, offset):
    """curves_device writing into a view at int32 ``offset`` of a larger buffer; the bytes around it must stay."""
    import torch
    n_perm, n = int(d_perms.shape[0]), eng.n_genomes
    size = n_perm * 2 * n
    buf = torch.full((size + offset + 5,), -7, dtype=torch.int32, device="cuda")
    out = buf[offset:offset + size].view(n_perm, 2 * n)
    eng.curves_device(d_perms, out=out)
    guard = torch.cat([buf[:offset], buf[offset + size:]]).cpu().numpy()
    assert np.all(guard == -7)
    return out.cpu().numpy()


def _check_every_path(eng, perms, want, blocks=(0, 7, 16)):
    """curves_device, curves_host (int32 and float64, several block sizes) against ``want``."""
    assert np.array_equal(eng.curves_device(_device_perms(perms)).cpu().numpy(), want)
    for block in blocks:
        assert np.array_equal(eng.curves_host(perms, perms_per_block=block), want), block
        assert np.array_equal(eng.curves_host(perms, out_f64=True, perms_per_block=block), want.astype(np.float64)), block


# ---------------------------------------------------------------------------------------------------------------
# GPU: native int32 bins at every batch size, the gathering prep and both row kernels
# ---------------------------------------------------------------------------------------------------------------
# (N, long_threshold): None routes the heavy rows to the list kernel, 2 to the probe kernel (its bitmap of the 66,000
# heavy rows costs N x 8.7 kB, hence only up to N = 12,001).  From N = 11,265 on the int32 prep needs more shared memory
# than the scatter version may take and the gathering prep_kernel runs: vector at 12,000, scalar at 12,001.
NATIVE_CASES = [(12000, None), (12000, 2), (12001, None), (12001, 2), (20000, None), (40000, None), (65503, None)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,threshold", NATIVE_CASES)
def test_native_int32_bins_at_every_launch_shape(engine_mod, n, threshold):
    coo = heavy_table(n, INT32_HEAVY, seed=n)
    eng = engine_mod.PanCoreEngine(coo, long_threshold=threshold)
    hp = eng.host_plan
    assert eng.c_plan.max_colsum == INT32_HEAVY > 65535
    assert hp.perms_per_cta == {12000: 8, 12001: 8, 20000: 4, 40000: 2, 65503: 1}[n]
    heavy_genes = np.arange(INT32_HEAVY)
    assert np.isin(heavy_genes, hp.long_gene if threshold == 2 else hp.row_gene).all()
    seed = n % 1000 + 3
    perms = np.r_[chosen_orders(n, seed), draw_perms(seed, n, 6)].astype(np.uint16)
    want = oracle_curves(coo, perms)
    assert_heavy_steps(want, n, INT32_HEAVY)
    _check_every_path(eng, perms, want)
    assert _split_head() == 0                                   # the int32 pipeline ran: no split transfer
    np.random.seed(seed)
    assert np.array_equal(eng.estimate(6), want[4:].astype(np.float64))
    assert _split_head() == 0
    # the scalar prep and scan at N % 8 == 0: an output view off a 16-byte boundary, permutations at an odd offset
    if n == 12000:
        for offset in (1, 2, 3):
            assert np.array_equal(_curves_into_offset_view(eng, _device_perms(perms), offset), want), offset
        assert np.array_equal(eng.curves_device(_device_perms(perms, odd=True)).cpu().numpy(), want)
        assert np.array_equal(_curves_into_offset_view(eng, _device_perms(perms, odd=True), 1), want)


@pytest.mark.gpu
def test_int32_summary_equals_pandas_statistics_at_12001_genomes(engine_mod):
    """estimate_pan_core_summary on a native int32 table that takes the gathering prep, against pandas statistics of
    the oracle's curves of the same 50 device-drawn genome orders."""
    from pangenomix_b200 import pangenome_analysis as pa, plot, sparse_utils as su, synth
    n, num_iter, seed = 12001, 50, 77
    coo = heavy_table(n, INT32_HEAVY, seed=5)
    lsdf = su.LightSparseDataFrame(*synth.labels_for(*coo.shape), coo)
    got = pa.estimate_pan_core_summary(lsdf, num_iter, seed=seed)
    eng = pa._engine_for(lsdf)
    assert eng.c_plan.max_colsum == INT32_HEAVY
    perms = engine_mod.random_permutations_device(n, num_iter, seed, device=eng.device).cpu().numpy().view(np.uint16)
    cols = ["Pan%d" % (i + 1) for i in range(n)] + ["Core%d" % (i + 1) for i in range(n)]
    full = pd.DataFrame(oracle_curves(coo, perms).astype(np.float64), columns=cols)
    want = full.agg(['mean', 'std', 'min', 'max'])
    assert list(got.index) == ['mean', 'std', 'min', 'max'] and list(got.columns) == cols
    for row in ('mean', 'min', 'max'):
        assert np.array_equal(got.loc[row].values, want.loc[row].values), row
    assert np.array_equal(got.loc[['mean']].values, plot.calculate_mean(full).values)
    np.testing.assert_allclose(got.loc['std'].values, want.loc['std'].values, rtol=1e-12, atol=0)


# ---------------------------------------------------------------------------------------------------------------
# GPU: the packed boundary, max_colsum = 65,535 (packed) and 65,536 (int32)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("route", ["list", "probe"])
@pytest.mark.parametrize("n", [64, 2200])
@pytest.mark.parametrize("heavy", [65535, 65536])
def test_packed_boundary(engine_mod, heavy, n, route):
    """One genome of exactly 65,535 genes still counts in uint16 bins (the largest step a row kernel adds fits); with
    65,536 the table takes int32 bins.  At N = 2,200 (a genome count no other test uses) order C's step of H lies in the
    uint8 tail of the split transfer: the packed call must send its block again as uint16 and grow the head."""
    coo = heavy_table(n, heavy, seed=heavy + n)
    eng = engine_mod.PanCoreEngine(coo, long_threshold=None if route == "list" else 2)
    hp = eng.host_plan
    packed = heavy == 65535
    assert eng.c_plan.max_colsum == heavy
    assert np.isin(np.arange(heavy), hp.row_gene if route == "list" else hp.long_gene).all()
    seed = n + heavy % 7
    perms = np.r_[chosen_orders(n, seed), draw_perms(seed, n, 5)].astype(np.uint16)
    want = oracle_curves(coo, perms)
    assert_heavy_steps(want, n, heavy)
    if n >= 4 * SPLIT_HEAD:
        _fresh_staging(engine_mod)
        # orders A, B and D: every tail step fits a byte, the head stays (packed) / there is no split (int32)
        assert np.array_equal(eng.curves_host(perms[[0, 1, 3]]), want[[0, 1, 3]])
        assert _split_head() == (SPLIT_HEAD if packed else 0)
        # with order C the packed block overflows its tail: sent again as uint16, the head doubles past N / 4 -> 0
        assert np.array_equal(eng.curves_host(perms), want)
        assert _split_head() == 0
    _check_every_path(eng, perms, want)
    np.random.seed(seed)
    assert np.array_equal(eng.estimate(5), want[4:].astype(np.float64))
    if not packed and n >= 2048:
        assert _split_head() == 0


# ---------------------------------------------------------------------------------------------------------------
# GPU: the launch matrix of test_gpu_parity.py in both bin formats
# ---------------------------------------------------------------------------------------------------------------
BINS = ["packed", "int32"]


def _mixed_matrix(n, seed=5, per_class=24):
    """The density profile of test_gpu_parity.py's launch-shape tables: every row class, lists of many lengths."""
    from test_gpu_parity import _mixed_matrix as mixed
    return mixed(n, seed=seed, per_class=per_class)


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
@pytest.mark.parametrize("perms_per_cta", [1, 2, 4, 8])
@pytest.mark.parametrize("splits,threads", [(1, 64), (3, 256), (7, 1024)])
@pytest.mark.parametrize("threshold", [0, 40])
def test_every_launch_shape_in_both_bin_formats(engine_mod, bins, perms_per_cta, splits, threads, threshold):
    from pangenomix_b200 import _native
    coo = _mixed_matrix(700)
    eng = _engine(engine_mod, coo, bins, long_threshold=threshold)
    hp = eng.host_plan
    assert (hp.n_long > 0) == (threshold > 0) and hp.n_rows > 0
    perms = edge_orders(hp, 13, seed=3).astype(np.uint16)
    want = oracle_curves_cached("launch shapes", coo, perms)
    _native.set_tuning(perms_per_cta, splits, threads)
    try:
        assert np.array_equal(eng.curves_host(perms), want)
        assert np.array_equal(eng.curves_device(_device_perms(perms)).cpu().numpy(), want)
    finally:
        _native.set_tuning(0, 0, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
@pytest.mark.parametrize("slice_words", [1, 2, 4])
def test_bitmap_slices_in_both_bin_formats(engine_mod, bins, slice_words):
    from pangenomix_b200.plan import build_host_plan
    coo = _mixed_matrix(600, seed=21, per_class=600)
    hp = build_host_plan(coo, long_threshold=6, slice_words=slice_words)
    assert hp.n_long > 4096 and hp.n_superblocks >= 2
    eng = _engine(engine_mod, coo, bins, host_plan=hp)
    perms = edge_orders(hp, 40, seed=23).astype(np.uint16)
    want = oracle_curves_cached("bitmap slices", coo, perms)
    assert np.array_equal(eng.curves_host(perms), want)
    assert np.array_equal(eng.curves_device(_device_perms(perms)).cpu().numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
@pytest.mark.parametrize("n", [1, 3, 33, 333, 700])
@pytest.mark.parametrize("threshold", [0, 8])
def test_genome_counts_in_both_bin_formats(engine_mod, bins, n, threshold):
    """Genome counts that are not multiples of 8 (the scalar prep and scan) and the last bin of each side set."""
    coo = _mixed_matrix(n, seed=n)
    eng = _engine(engine_mod, coo, bins, long_threshold=threshold)
    perms = edge_orders(eng.host_plan, 13, seed=n).astype(np.uint16)
    want = oracle_curves(coo, perms)
    _check_every_path(eng, perms, want, blocks=(0, 5))
    np.random.seed(n)
    assert np.array_equal(eng.estimate(9), oracle_curves(coo, draw_perms(n, n, 9)).astype(np.float64))


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
@pytest.mark.parametrize("n", [333, 704])
@pytest.mark.parametrize("offset", [1, 2, 3])
def test_unaligned_output_and_permutations(engine_mod, bins, n, offset):
    """curves_device into a view at int32 offset 1, 2 or 3 of a larger buffer, and from permutations at an odd int16
    offset: the scalar variants of prep and scan, also at N % 8 == 0."""
    coo = _mixed_matrix(n, seed=n + offset)
    eng = _engine(engine_mod, coo, bins, long_threshold=20)
    perms = edge_orders(eng.host_plan, 11, seed=offset).astype(np.uint16)
    want = oracle_curves(coo, perms)
    assert np.array_equal(_curves_into_offset_view(eng, _device_perms(perms), offset), want)
    assert np.array_equal(eng.curves_device(_device_perms(perms, odd=True)).cpu().numpy(), want)
    assert np.array_equal(_curves_into_offset_view(eng, _device_perms(perms, odd=True), offset), want)


# ---------------------------------------------------------------------------------------------------------------
# GPU: the host-buffer staging, kept between calls, across bin formats and output types
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_staging_alternates_between_bin_formats_and_output_types(engine_mod):
    """Calls alternating between a packed and an int32 engine of the SAME table (same N), and between int32 and float64
    results: whenever the staging is reused or set up again the curves must not change.  The split head tells which
    pipeline ran: 512 for the packed one (its tails fit a byte), 0 for the int32 one."""
    from pangenomix_b200 import synth
    n = 2304
    coo = synth.bernoulli_matrix(20000, n, 3000, seed=3).tocoo()
    packed = _engine(engine_mod, coo, "packed")
    wide = _engine(engine_mod, coo, "int32")
    perms = draw_perms(5, n, 16).astype(np.uint16)
    want = oracle_curves(coo, perms)
    calls = [(packed, False), (wide, False), (wide, True), (wide, False), (packed, True), (wide, True),
             (packed, False), (wide, False), (wide, False)]
    for i, (eng, f64) in enumerate(calls):
        got = eng.curves_host(perms, out_f64=f64, perms_per_block=7)
        assert np.array_equal(got, want.astype(np.float64) if f64 else want), i
        assert _split_head() == (SPLIT_HEAD if eng is packed else 0), i
    for eng in (wide, packed, wide):
        np.random.seed(5)
        assert np.array_equal(eng.estimate(16), want.astype(np.float64))
        assert _split_head() == (SPLIT_HEAD if eng is packed else 0)
