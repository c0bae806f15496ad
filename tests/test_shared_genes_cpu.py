"""Shared-gene matrix and genomic fluidity without a GPU: the plan decomposition of S = X^T X that pgx_shared_genes
computes (oracle/shared_np.py) against scipy's product, the fluidity oracle against gene sets, the host finish of
compute_genomic_fluidity against a hand-computed table and an explicit jackknife, and argument checks of the C calls."""
import ctypes
import math

import numpy as np
import pytest
import scipy.sparse

from conftest import CURVE_CASES, golden_matrix
from oracle import plan_np, shared_np
from pangenomix_b200 import _native, plan
from pangenomix_b200.pangenome_analysis import fluidity_series


def random_table(n, seed, n_genes=400):
    """Random binary table with universal, empty, single-presence and single-absence genes among the others."""
    rng = np.random.default_rng(seed)
    x = rng.random((n_genes, n)) < rng.random(n_genes)[:, None] ** 2
    x[:6] = True
    x[6:12] = False
    for g in range(12, 20):
        x[g] = False
        x[g, rng.integers(n)] = True
    if n > 2:
        for g in range(20, 28):
            x[g] = True
            x[g, rng.integers(n)] = False
    return scipy.sparse.coo_matrix(x.astype(np.int64))


@pytest.mark.parametrize("name", CURVE_CASES + ["c2_40000x400"])
def test_plan_decomposition_is_xtx_on_the_fixtures(name):
    coo = golden_matrix(name)
    assert np.array_equal(shared_np.shared_from_plan(plan.build_host_plan(coo)), shared_np.shared_direct(coo))


@pytest.mark.parametrize("slice_words", [1, 2, 4])
@pytest.mark.parametrize("threshold", ["zero", "one", "default", "above_half"])
@pytest.mark.parametrize("n", [1, 2, 3, 127, 129, 257])
def test_plan_decomposition_is_xtx_on_random_tables(n, threshold, slice_words):
    coo = random_table(n, seed=n * 10 + slice_words)
    long_threshold = {"zero": 0, "one": 1, "default": None, "above_half": n // 2 + 1}[threshold]
    want = shared_np.shared_direct(coo)
    for build in (plan.build_host_plan, plan_np.build_host_plan):
        hp = build(coo, long_threshold=long_threshold, slice_words=slice_words)
        assert np.array_equal(shared_np.shared_from_plan(hp), want)


@pytest.mark.parametrize("n", [2, 3, 17, 60])
def test_oracle_fluidity_equals_gene_set_brute_force(n):
    coo = random_table(n, seed=n)
    x = coo.toarray().astype(bool)
    sets = [set(np.flatnonzero(x[:, c]).tolist()) for c in range(n)]
    s = shared_np.shared_direct(coo)
    assert shared_np.fluidity_by_definition(s) == pytest.approx(shared_np.fluidity_brute(sets), rel=1e-14)
    rows = shared_np.fluidity_rows(s)
    assert math.fsum(rows) / 2 / (n * (n - 1) / 2) == pytest.approx(shared_np.fluidity_brute(sets), rel=1e-13)


def test_fluidity_distance_of_two_empty_genomes_is_nan():
    s = np.array([[0, 0, 0], [0, 0, 0], [0, 0, 2]], dtype=np.int32)
    d = shared_np.fluidity_distances(s)
    assert np.isnan(d[0, 1]) and d[0, 2] == 1.0


def test_host_finish_hand_kat():
    # genomes {g1, g2, g3}, {g1, g2}, {g1, g4}: d = 1/5, 3/5, 1/2, fluidity 13/30, jackknife sqrt(13) / 15
    x = np.array([[1, 1, 1], [1, 1, 0], [1, 0, 0], [0, 0, 1]], dtype=np.int64)
    s = shared_np.shared_direct(scipy.sparse.coo_matrix(x))
    assert s.tolist() == [[3, 2, 1], [2, 2, 1], [1, 1, 2]]
    out = fluidity_series(shared_np.fluidity_rows(s))
    assert list(out.index) == ["fluidity", "jackknife_se", "n_genomes"]
    assert out["fluidity"] == pytest.approx(13 / 30, rel=1e-15)
    assert out["jackknife_se"] == pytest.approx(math.sqrt(13) / 15, rel=1e-14)
    assert abs(out["jackknife_se"] - 0.2403700850) < 1e-10
    assert out["n_genomes"] == 3


@pytest.mark.parametrize("n", [3, 4, 25, 90])
def test_host_finish_matches_explicit_leave_one_out(n):
    s = shared_np.shared_direct(random_table(n, seed=100 + n))
    out = fluidity_series(shared_np.fluidity_rows(s))
    assert out["fluidity"] == pytest.approx(shared_np.fluidity_by_definition(s), rel=1e-13)
    assert out["jackknife_se"] == pytest.approx(shared_np.jackknife_by_definition(s), rel=1e-9)


def test_host_finish_edge_sizes():
    with pytest.raises(ValueError):
        fluidity_series(np.zeros(1))
    with pytest.raises(ValueError):
        fluidity_series(np.zeros(0))
    out = fluidity_series(np.array([0.25, 0.25]))
    assert out["fluidity"] == 0.25 and np.isnan(out["jackknife_se"]) and out["n_genomes"] == 2


def _fake_plan(n):
    """A plan struct whose pointers are never dereferenced: every call below must fail its argument checks first."""
    p = _native.PgxPlan()
    p.d_colsum = p.d_w_present = p.d_w_absent = 0x10000
    p.n_genomes = n
    return p


def test_shared_genes_rejects_bad_arguments_without_launching():
    lib = _native.load()
    launches = _native.launch_count()
    good = 0x20000                                          # 16-byte aligned, never dereferenced

    def call(p, shared=good, work=good, work_bytes=1 << 20):
        rc = lib.pgx_shared_genes(ctypes.byref(p) if p is not None else None, shared, work, work_bytes, None)
        assert rc == 1, lib.pgx_last_error()
        return lib.pgx_last_error().decode()

    assert "null" in call(None)
    assert "null" in call(_fake_plan(4), shared=None)
    assert "null" in call(_fake_plan(4), work=None)
    assert "outside" in call(_fake_plan(0))
    assert "outside" in call(_fake_plan(65504))
    assert "aligned" in call(_fake_plan(4), shared=good + 4)
    assert "aligned" in call(_fake_plan(4), work=good + 8)
    assert "work_bytes" in call(_fake_plan(4), work_bytes=4 * 128 - 1)
    assert "work_bytes" in call(_fake_plan(65503), work_bytes=65503 * 128 - 16)
    vectors = _fake_plan(4)
    vectors.d_w_absent = 0
    assert "vectors" in call(vectors)
    rows = _fake_plan(4)
    rows.n_rows, rows.n_tasks = 3, 1
    assert "list rows" in call(rows)
    bitmap = _fake_plan(4)
    bitmap.n_long, bitmap.n_superblocks, bitmap.slice_words, bitmap.d_bits = 5, 1, 3, good
    assert "bitmap" in call(bitmap)
    assert _native.launch_count() == launches


def test_fluidity_rows_rejects_bad_arguments_without_launching():
    lib = _native.load()
    launches = _native.launch_count()
    good = 0x20000
    for shared, n, rows in ((None, 4, good), (good, 4, None), (good, 0, good), (good, 65504, good),
                            (good + 2, 4, good), (good, 4, good + 4)):
        assert lib.pgx_fluidity_rows(shared, n, rows, None) == 1
    assert _native.launch_count() == launches


def test_gemm_kernel_runs_on_the_tensor_cores():
    """The shared-gene GEMM compiles to tcgen05 integer MMAs (UTCIMMA), TMA loads and tensor-memory loads."""
    import shutil
    import subprocess
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not shutil.which(tool):
        pytest.skip("cuobjdump not installed")
    sass = subprocess.run([tool, "-sass", _native.LIB_PATH], capture_output=True, text=True, check=True).stdout
    functions = sass.split("Function : ")
    gemm = [f for f in functions if f.split("\n", 1)[0].strip().find("shared_gemm_kernel") >= 0]
    assert len(gemm) == 1
    for op in ("UTCIMMA", "UTMALDG", "LDTM"):
        assert op in gemm[0], op
