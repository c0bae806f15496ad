"""Exact pan/core rarefaction without a GPU: the moment formulas (oracle/exact_np.py) against enumeration of every
k-subset in exact rationals, the plan decomposition of the pair histograms against X X^T at every plan shape, the
exact moments against the 1,000-permutation live reference of C2, and argument checks of the C calls."""
import ctypes
import shutil
import subprocess

import numpy as np
import pytest

from conftest import CURVE_CASES, golden_matrix, load_golden
from oracle import exact_np, plan_np
from pangenomix_b200 import _native, plan
from test_shared_genes_cpu import random_table


@pytest.mark.parametrize("n", [1, 2, 3, 4, 6, 9, 10])
def test_moment_formulas_equal_subset_enumeration(n):
    coo = random_table(n, seed=500 + n, n_genes=36)      # universal, empty, single-genome and single-absence genes
    hs, ha = exact_np.pair_histograms_direct(coo)
    got = exact_np.moments_exact(exact_np.spectrum_direct(coo), hs, ha, 36, n)
    assert got == exact_np.moments_enumerate(coo)
    assert got[1][n - 1] == 0 and got[3][n - 1] == 0


@pytest.mark.parametrize("n", [2, 7, 40, 300])
def test_long_double_moments_equal_the_rationals(n):
    coo = random_table(n, seed=700 + n, n_genes=400)
    hs, ha = exact_np.pair_histograms_direct(coo)
    spec = exact_np.spectrum_direct(coo)
    want = np.array(exact_np.moments_exact(spec, hs, ha, 400, n), dtype=np.float64)
    got = exact_np.moments_longdouble(spec, hs, ha, 400, n).astype(np.float64)
    means = want[[0, 2]]
    assert np.all(np.abs(got[[0, 2]] - means) <= 1e-14 * np.maximum(1, np.abs(means)))
    assert np.all(np.abs(got[[1, 3]] - want[[1, 3]]) <= 1e-14 * (means ** 2 + 1))


@pytest.mark.parametrize("name", CURVE_CASES)
def test_plan_decomposition_is_xxt_on_the_fixtures(name):
    coo = golden_matrix(name)
    got = exact_np.pair_histograms_from_plan(plan.build_host_plan(coo))
    want = exact_np.pair_histograms_direct(coo)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


@pytest.mark.parametrize("slice_words", [1, 2, 4])
@pytest.mark.parametrize("threshold", ["zero", "one", "default", "above_half"])
@pytest.mark.parametrize("n", [1, 2, 3, 127, 129, 257])
def test_plan_decomposition_is_xxt_on_random_tables(n, threshold, slice_words):
    coo = random_table(n, seed=n * 10 + slice_words)
    long_threshold = {"zero": 0, "one": 1, "default": None, "above_half": n // 2 + 1}[threshold]
    hs, ha = exact_np.pair_histograms_direct(coo)
    assert hs.sum() == ha.sum() == 400 * 399 // 2
    for build in (plan.build_host_plan, plan_np.build_host_plan):
        got = exact_np.pair_histograms_from_plan(build(coo, long_threshold=long_threshold, slice_words=slice_words))
        assert np.array_equal(got[0], hs) and np.array_equal(got[1], ha)


def test_exact_moments_match_the_c2_live_reference():
    """C2's 1,000 permutations (reference runs) against the exact mean and std over all orders."""
    g = load_golden("c2_40000x400")
    coo = golden_matrix("c2_40000x400", g)
    n_genes, n = coo.shape
    hs, ha = exact_np.pair_histograms_from_plan(plan.build_host_plan(coo))
    exact = exact_np.moments_longdouble(exact_np.spectrum_direct(coo), hs, ha, n_genes, n).astype(np.float64)
    mean_e = np.concatenate([exact[0], exact[2]])
    var_e = np.concatenate([exact[1], exact[3]])
    curves = g["curves"].astype(np.float64)
    runs = curves.shape[0]
    mean_f, std_f = curves.mean(axis=0), curves.std(axis=0, ddof=1)
    live = var_e > 0
    assert np.all(np.abs(mean_f - mean_e)[live] <= 5 * np.sqrt(var_e[live] / runs))
    ratio = std_f[live] / np.sqrt(var_e[live])
    assert ratio.min() >= 0.85 and ratio.max() <= 1.15
    assert np.all(curves[:, ~live] == curves[0, ~live])
    assert np.all(np.abs(curves[0, ~live] - mean_e[~live]) < 1e-9 * np.maximum(1, mean_e[~live]))


def _fake_plan(n):
    """A plan struct whose pointers are never dereferenced: every call below must fail its argument checks first."""
    p = _native.PgxPlan()
    p.d_colsum = p.d_w_present = p.d_w_absent = 0x10000
    p.n_genomes = n
    return p


def test_exact_calls_reject_bad_arguments_without_launching():
    lib = _native.load()
    launches = _native.launch_count()
    good = 0x20000                                          # 256-byte aligned, never dereferenced

    def spectrum(p, out=good):
        assert lib.pgx_plan_spectrum(ctypes.byref(p) if p is not None else None, out, None) == 1
        return lib.pgx_last_error().decode()

    def pairs(p, hs=good, ha=good, work=good, work_bytes=1 << 40):
        rc = lib.pgx_pair_overlap_histograms(ctypes.byref(p) if p is not None else None, hs, ha, work, work_bytes, None)
        assert rc == 1
        return lib.pgx_last_error().decode()

    def moments(spec=good, hs=good, ha=good, g=10, n=4, out=good):
        assert lib.pgx_rarefaction_moments(spec, hs, ha, g, n, out, None) == 1
        return lib.pgx_last_error().decode()

    assert "null" in spectrum(None) and "null" in spectrum(_fake_plan(4), out=None)
    assert "aligned" in spectrum(_fake_plan(4), out=good + 4)
    assert "outside" in spectrum(_fake_plan(0)) and "outside" in spectrum(_fake_plan(65504))
    vectors = _fake_plan(4)
    vectors.d_w_present = 0
    assert "vectors" in spectrum(vectors) and "vectors" in pairs(vectors)
    rows = _fake_plan(4)
    rows.n_rows, rows.n_tasks = 3, 1
    assert "list rows" in spectrum(rows) and "list rows" in pairs(rows)
    bitmap = _fake_plan(4)
    bitmap.n_long, bitmap.n_superblocks, bitmap.slice_words, bitmap.d_bits = 5, 1, 3, good
    assert "bitmap" in pairs(bitmap)
    bitmap.slice_words, bitmap.n_long = 1, 1025
    assert "bitmap" in pairs(bitmap)

    assert "null" in pairs(None)
    for key in ("hs", "ha", "work"):
        assert "null" in pairs(_fake_plan(4), **{key: None})
    assert "aligned" in pairs(_fake_plan(4), hs=good + 4)
    assert "aligned" in pairs(_fake_plan(4), work=good + 16)
    assert "outside" in pairs(_fake_plan(0)) and "outside" in pairs(_fake_plan(65504))
    small = _fake_plan(1000)
    small.n_long, small.n_superblocks, small.slice_words, small.d_bits = 600, 1, 1, good
    least = lib.pgx_pair_overlap_work_bytes(1000, 600, 0)
    assert least > 512 * 1024 and lib.pgx_pair_overlap_work_bytes(1000, 600, 1) > least
    assert "work_bytes" in pairs(small, work_bytes=least - 1)

    assert "null" in moments(spec=None) and "null" in moments(out=None)
    assert "both" in moments(hs=None) and "both" in moments(ha=None)
    assert "outside" in moments(n=0) and "outside" in moments(n=65504)
    assert "negative" in moments(g=-1)
    assert "aligned" in moments(out=good + 4) and "aligned" in moments(hs=good + 2)
    assert _native.launch_count() == launches


def test_pair_workspace_sizes():
    lib = _native.load()
    assert lib.pgx_pair_overlap_work_bytes(0, 10, 0) == 0 and lib.pgx_pair_overlap_work_bytes(65504, 10, 0) == 0
    assert lib.pgx_pair_overlap_work_bytes(10, -1, 0) == 0
    # fewer rows than two panels of 256: the minimum already holds them all
    assert lib.pgx_pair_overlap_work_bytes(300, 100, 0) == lib.pgx_pair_overlap_work_bytes(300, 100, 1)
    whole, least = lib.pgx_pair_overlap_work_bytes(300, 5000, 1), lib.pgx_pair_overlap_work_bytes(300, 5000, 0)
    assert whole - least == (5120 - 512) * 384


def test_histogram_gemm_kernel_runs_on_the_tensor_cores():
    """The pair-histogram GEMM compiles to tcgen05 integer MMAs (UTCIMMA), TMA loads and tensor-memory loads."""
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not shutil.which(tool):
        pytest.skip("cuobjdump not installed")
    sass = subprocess.run([tool, "-sass", _native.LIB_PATH], capture_output=True, text=True, check=True).stdout
    gemm = [f for f in sass.split("Function : ") if "pair_hist_gemm_kernel" in f.split("\n", 1)[0]]
    assert len(gemm) == 1
    for op in ("UTCIMMA", "UTMALDG", "LDTM"):
        assert op in gemm[0], op
