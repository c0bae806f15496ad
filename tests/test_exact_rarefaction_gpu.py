"""pgx_plan_spectrum / pgx_pair_overlap_histograms / pgx_rarefaction_moments on the GPU: the histograms bit for bit
against X X^T at every plan shape, over many panel pairs and on both epilogue paths; C4 (and C5 with PGX_TEST_C5=1)
through exact integer identities against the shared-gene matrix; the moments against the long-double and rational
oracles and against 200,000 sampled orders; and exact_pan_core_summary."""
import ctypes
import io
import contextlib
import os

import numpy as np
import pytest
import scipy.sparse

from conftest import CURVE_CASES, golden_matrix
from oracle import exact_np
from test_shared_genes_cpu import random_table

pytestmark = pytest.mark.gpu

# a tile counts into shared-memory bins when its s and a ranges fit (196,608 - 1,024) / 4 = 48,896 uint32 bins; one
# tile whose rows hold m = 2 and m = N - 2 needs 2 (N - 1) of them: shared memory up to N = 24,449
SMEM_LIMIT_N = 24449


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")
    return torch


def _engine(coo, long_threshold=None, slice_words=None):
    from pangenomix_b200 import engine, plan
    return engine.PanCoreEngine(coo, host_plan=plan.build_host_plan(coo, long_threshold=long_threshold,
                                                                    slice_words=slice_words))


def _lsdf(coo):
    from pangenomix_b200 import sparse_utils as su, synth
    index, columns = synth.labels_for(*coo.shape)
    return su.LightSparseDataFrame(index, columns, coo)


def _check_histograms(eng, coo, work_bytes=None):
    hs, ha = eng.pair_histograms_device(work_bytes)
    want = exact_np.pair_histograms_direct(coo)
    assert np.array_equal(hs.cpu().numpy(), want[0])
    assert np.array_equal(ha.cpu().numpy(), want[1])
    assert np.array_equal(eng.spectrum_device().cpu().numpy(), exact_np.spectrum_direct(coo))


def _table(x):
    return scipy.sparse.coo_matrix(np.asarray(x, dtype=np.int64))


@pytest.mark.parametrize("name", CURVE_CASES + ["c2_40000x400"])
def test_histograms_equal_xxt_on_the_fixtures(torch_cuda, name):
    coo = golden_matrix(name)
    _check_histograms(_engine(coo), coo)


@pytest.mark.parametrize("slice_words", [1, 2, 4])
@pytest.mark.parametrize("threshold", ["zero", "one", "default", "above_half"])
@pytest.mark.parametrize("n", [1, 2, 3, 127, 128, 129, 255, 256, 257])
def test_histograms_equal_xxt_at_every_plan_shape(torch_cuda, n, threshold, slice_words):
    coo = random_table(n, seed=n * 10 + slice_words)
    long_threshold = {"zero": 0, "one": 1, "default": None, "above_half": n // 2 + 1}[threshold]
    _check_histograms(_engine(coo, long_threshold, slice_words), coo)


@pytest.mark.parametrize("n_genes", [129, 255, 383, 640, 1000])
def test_histograms_with_row_counts_off_the_tile_grid(torch_cuda, n_genes):
    coo = random_table(200, seed=n_genes, n_genes=n_genes)
    _check_histograms(_engine(coo, long_threshold=1), coo)


@pytest.mark.parametrize("stored", [0, 1, 2])
def test_histograms_with_few_or_no_stored_rows(torch_cuda, stored):
    n = 50
    x = np.zeros((40 + stored, n), dtype=np.int64)
    x[:10] = 1                                              # universal
    for g in range(10, 20):                                 # single genome
        x[g, g % 7] = 1
    for g in range(20, 30):                                 # single absence
        x[g] = 1
        x[g, g % 5] = 0
    for g in range(40, 40 + stored):                        # stored rows
        x[g, :10 + 7 * g % 30] = 1
    coo = _table(x)
    eng = _engine(coo)
    assert eng.host_plan.n_rows + eng.host_plan.n_long == stored
    _check_histograms(eng, coo)


@pytest.mark.parametrize("n", [100, 300])
def test_histograms_over_many_panel_pairs(torch_cuda, n):
    """The smallest workspace the call takes: panels of 256 rows, every pair of them."""
    coo = random_table(n, seed=9 * n, n_genes=3000)
    eng = _engine(coo, long_threshold=1)
    stored = eng.host_plan.n_rows + eng.host_plan.n_long
    least = int(eng.lib.pgx_pair_overlap_work_bytes(n, stored, 0))
    assert stored > 8 * 256
    _check_histograms(eng, coo, work_bytes=least)
    _check_histograms(eng, coo, work_bytes=least + 3 * 256 * 384 + 100)


def _spread_table(n, n_genes, seed):
    """Genes whose genome counts reach from 2 to N - 2, so that one tile's s and a ranges are as wide as they get."""
    rng = np.random.default_rng(seed)
    m = np.linspace(2, n - 2, n_genes).round().astype(np.int64)
    rows, cols = [], []
    for g, k in enumerate(m):
        c = rng.choice(n, int(k), replace=False)
        rows.append(np.full(k, g))
        cols.append(c)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    return scipy.sparse.coo_matrix((np.ones(rows.size, dtype=np.int64), (rows, cols)), shape=(n_genes, n))


@pytest.mark.parametrize("n", [SMEM_LIMIT_N, SMEM_LIMIT_N + 1, 65503])
def test_histograms_on_both_sides_of_the_shared_memory_bins(torch_cuda, n):
    coo = _spread_table(n, 120 if n < 65503 else 300, seed=n)
    _check_histograms(_engine(coo, long_threshold=0), coo)
    _check_histograms(_engine(coo, long_threshold=1), coo)


def _identities(torch_cuda, eng, coo, hs, ha):
    """Sum, first and second moment of H_s and H_a from the shared-gene matrix, in Python integers."""
    n_genes, n = coo.shape
    s = eng.shared_genes_device()
    sq = sum(int(v) for v in (s.to(torch_cuda.int64) ** 2).sum(dim=1).cpu().numpy())
    colsum = np.bincount(coo.col, minlength=n).astype(object)
    m = np.bincount(coo.row, minlength=n_genes).astype(object)
    nnz = int(coo.nnz)
    # complement Y = 1 - X: Y^T Y = G J - colsum 1^T - 1 colsum^T + S, entry by entry in int64 per row
    c = torch_cuda.from_numpy(np.bincount(coo.col, minlength=n).astype(np.int64)).cuda()
    y = n_genes - c[:, None] - c[None, :] + s.to(torch_cuda.int64)
    ysq = sum(int(v) for v in (y ** 2).sum(dim=1).cpu().numpy())
    del s, y
    v = np.arange(n + 1, dtype=object)
    hs, ha = hs.cpu().numpy().astype(object), ha.cpu().numpy().astype(object)
    pairs = n_genes * (n_genes - 1) // 2
    assert hs.sum() == pairs and ha.sum() == pairs
    assert (v * hs).sum() * 2 == (colsum ** 2).sum() - nnz
    assert (v * v * hs).sum() * 2 == sq - (m ** 2).sum()
    ycol, ym = n_genes - colsum, n - m
    assert (v * ha).sum() * 2 == (ycol ** 2).sum() - (n * n_genes - nnz)
    assert (v * v * ha).sum() * 2 == ysq - (ym ** 2).sum()


def _assert_moments_close(got, want):
    means = want[[0, 2]]
    assert np.all(np.abs(got[[0, 2]] - means) <= 1e-12 * np.maximum(1, np.abs(means)))
    assert np.all(np.abs(got[[1, 3]] - want[[1, 3]]) <= 1e-12 * (means ** 2 + 1))


@pytest.fixture(scope="module")
def c4(torch_cuda):
    coo = golden_matrix("c4_200000x10000")
    eng = _engine(coo)
    hs, ha = eng.pair_histograms_device()
    return coo, eng, hs, ha


def test_c4_histograms_satisfy_the_identities(torch_cuda, c4):
    coo, eng, hs, ha = c4
    _identities(torch_cuda, eng, coo, hs, ha)


def test_c4_moments_match_the_long_double_oracle(torch_cuda, c4):
    coo, eng, hs, ha = c4
    got = eng.exact_moments_device().cpu().numpy()
    spectrum = eng.spectrum_device().cpu().numpy()
    want = exact_np.moments_longdouble(spectrum, hs.cpu().numpy(), ha.cpu().numpy(), *coo.shape).astype(np.float64)
    _assert_moments_close(got, want)
    assert np.all(got[[1, 3], -1] == 0)


@pytest.mark.parametrize("name", ["kat_6x5", "tiny_40x1", "tiny_40x2", "edge_500x37", "synth_800x50_s0",
                                  "c2_40000x400"])
def test_moments_match_the_rational_oracle(torch_cuda, name):
    coo = golden_matrix(name)
    got = _engine(coo).exact_moments_device().cpu().numpy()
    hs, ha = exact_np.pair_histograms_direct(coo)
    want = np.array(exact_np.moments_exact(exact_np.spectrum_direct(coo), hs, ha, *coo.shape), dtype=np.float64)
    _assert_moments_close(got, want)


def test_c4_moments_match_200000_sampled_orders(torch_cuda, c4):
    from pangenomix_b200 import pangenome_analysis as pa
    coo = c4[0]
    df = _lsdf(coo)
    exact = pa.exact_pan_core_summary(df)
    runs = 200_000
    sampled = pa.estimate_pan_core_summary(df, runs, seed=2024)
    var = exact.loc["std"].values ** 2
    live = var > 0
    z = (sampled.loc["mean"].values - exact.loc["mean"].values)[live] / np.sqrt(var[live] / runs)
    assert np.abs(z).max() <= 6
    # a sample std is within 2 % of the true one where the spread is made of many small changes; where the variance
    # is far below 1 (the core near k = N) the value moves only in rare events, and the sample std of r events out of
    # 200,000 orders is off by about 1 / (2 sqrt(r)): 3 % at a variance of 1e-3
    ratio = sampled.loc["std"].values / exact.loc["std"].values
    broad = var >= 1
    assert np.abs(ratio[broad] - 1).max() <= 0.02
    assert np.abs(ratio[live & ~broad] - 1).max() <= 0.1
    dead = ~live
    for row in ("min", "max", "mean"):
        assert np.array_equal(sampled.loc[row].values[dead], exact.loc["mean"].values[dead])


@pytest.mark.parametrize("name", ["kat_6x5", "synth_800x50_s1", "c2slice_4000x400"])
def test_api_matches_the_oracle(torch_cuda, name):
    import pandas as pd
    from pangenomix_b200 import pangenome_analysis as pa
    coo = golden_matrix(name)
    df = _lsdf(coo)
    np.random.seed(5)
    state = np.random.get_state()
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        got = pa.exact_pan_core_summary(df)
        mean_only = pa.exact_pan_core_summary(df, std=False)
        again = pa.exact_pan_core_summary(df)
    assert out.getvalue() == ""
    assert all(np.array_equal(x, y) for x, y in zip(state, np.random.get_state()))
    n = coo.shape[1]
    assert isinstance(got, pd.DataFrame) and list(got.index) == ["mean", "std"]
    assert list(got.columns) == ["Pan%d" % k for k in range(1, n + 1)] + ["Core%d" % k for k in range(1, n + 1)]
    assert got.dtypes.unique().tolist() == [np.dtype(np.float64)]
    assert list(mean_only.index) == ["mean"] and list(mean_only.columns) == list(got.columns)
    assert got.values.tobytes() == again.values.tobytes()
    assert mean_only.loc["mean"].values.tobytes() == got.loc["mean"].values.tobytes()
    hs, ha = exact_np.pair_histograms_direct(coo)
    want = np.array(exact_np.moments_exact(exact_np.spectrum_direct(coo), hs, ha, *coo.shape), dtype=np.float64)
    mean = np.concatenate([want[0], want[2]])
    std = np.sqrt(np.maximum(np.concatenate([want[1], want[3]]), 0))
    np.testing.assert_allclose(got.loc["mean"].values, mean, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(got.loc["std"].values, std, rtol=1e-6, atol=1e-6)
    assert got.loc["std"].values[n - 1] == 0 and got.loc["std"].values[2 * n - 1] == 0


def test_api_reuses_the_plan_and_feeds_the_heaps_fit(torch_cuda, capsys):
    from pangenomix_b200 import engine as engine_mod
    from pangenomix_b200 import pangenome_analysis as pa
    df = _lsdf(golden_matrix("synth_800x50_s0"))
    pa.estimate_pan_core_summary(df, 64, seed=3)
    made = []
    original = engine_mod.PanCoreEngine.__init__

    def counting_init(self, *args, **kwargs):
        made.append(1)
        original(self, *args, **kwargs)

    engine_mod.PanCoreEngine.__init__ = counting_init
    try:
        exact = pa.exact_pan_core_summary(df)
    finally:
        engine_mod.PanCoreEngine.__init__ = original
    assert made == []
    capsys.readouterr()
    fit = pa.fit_heaps_by_iteration(exact.loc[["mean"]])
    assert list(fit.index) == ["mean"] and np.all(np.isfinite(fit.values))


def test_std_false_allocates_no_workspace(torch_cuda):
    from pangenomix_b200 import engine as engine_mod
    eng = _engine(golden_matrix("synth_800x50_s1"))
    calls = []
    original = engine_mod.PanCoreEngine.pair_histograms_device
    engine_mod.PanCoreEngine.pair_histograms_device = lambda self, *a: calls.append(1) or original(self, *a)
    try:
        out = eng.exact_moments_device(std=False).cpu().numpy()
    finally:
        engine_mod.PanCoreEngine.pair_histograms_device = original
    assert calls == [] and np.all(np.isnan(out[[1, 3]])) and np.all(np.isfinite(out[[0, 2]]))


def test_inconsistent_plan_is_refused(torch_cuda):
    from pangenomix_b200 import _native
    eng = _engine(random_table(40, seed=3))
    bad = _native.PgxPlan.from_buffer_copy(eng.c_plan)
    zeros = torch_cuda.zeros(40, dtype=torch_cuda.int32, device="cuda")
    bad.d_colsum = zeros.data_ptr()
    out = torch_cuda.empty(41, dtype=torch_cuda.int64, device="cuda")
    assert eng.lib.pgx_plan_spectrum(ctypes.byref(bad), out.data_ptr(), None) == 1
    assert b"inconsistent" in eng.lib.pgx_last_error()
    work_bytes = eng.pair_workspace_bytes()
    work = torch_cuda.empty(work_bytes, dtype=torch_cuda.uint8, device="cuda")
    rc = eng.lib.pgx_pair_overlap_histograms(ctypes.byref(bad), out.data_ptr(), out.data_ptr(), work.data_ptr(),
                                             work_bytes, None)
    assert rc == 1 and b"inconsistent" in eng.lib.pgx_last_error()


@pytest.mark.skipif(os.environ.get("PGX_TEST_C5") != "1", reason="C5 (2 M x 50,000) only with PGX_TEST_C5=1")
def test_c5_histograms_satisfy_the_identities(torch_cuda):
    from pangenomix_b200 import engine as engine_mod
    coo = golden_matrix("c5_2000000x50000")
    eng = _engine(coo)
    assert eng.pair_workspace_bytes() <= engine_mod.SHARED_WORK_CAP + (1 << 30)
    hs, ha = eng.pair_histograms_device()
    _identities(torch_cuda, eng, coo, hs, ha)
