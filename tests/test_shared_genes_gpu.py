"""pgx_shared_genes / pgx_fluidity_rows on the GPU: S against scipy's X^T X and the plan oracle bit for bit at every
plan shape, many K-slabs, C2 whole and C4 sampled; the fluidity rows' bits and value; the API's Series; and that
nothing touches np.random or the rarefaction of the same table."""
import ctypes

import numpy as np
import pytest

from conftest import CURVE_CASES, golden_matrix
from oracle import shared_np
from test_shared_genes_cpu import random_table

pytestmark = pytest.mark.gpu


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


@pytest.mark.parametrize("name", CURVE_CASES + ["c2_40000x400"])
def test_shared_genes_equal_xtx_on_the_fixtures(torch_cuda, name):
    coo = golden_matrix(name)
    got = _engine(coo).shared_genes_device().cpu().numpy()
    assert got.dtype == np.int32
    assert np.array_equal(got, shared_np.shared_direct(coo))


@pytest.mark.parametrize("slice_words", [1, 2, 4])
@pytest.mark.parametrize("threshold", ["zero", "one", "default", "above_half"])
@pytest.mark.parametrize("n", [1, 2, 3, 127, 128, 129, 255, 256, 257, 4097])
def test_shared_genes_equal_the_oracle_at_every_plan_shape(torch_cuda, n, threshold, slice_words):
    if n == 4097 and slice_words != 2:
        pytest.skip("N = 4,097 once per threshold")
    coo = random_table(n, seed=n * 10 + slice_words, n_genes=400 if n < 4097 else 3000)
    long_threshold = {"zero": 0, "one": 1, "default": None, "above_half": n // 2 + 1}[threshold]
    eng = _engine(coo, long_threshold, slice_words)
    got = eng.shared_genes_device().cpu().numpy()
    want = shared_np.shared_direct(coo)
    assert np.array_equal(got, want)
    if n <= 257:
        assert np.array_equal(got, shared_np.shared_from_plan(eng.host_plan))


@pytest.mark.parametrize("per_genome", [128, 384, 1024 + 256])
@pytest.mark.parametrize("n", [129, 300])
def test_shared_genes_over_many_k_slabs(torch_cuda, n, per_genome):
    """A workspace of ``per_genome`` bytes per genome: K-slabs of that many bitmap rows, the last one partial."""
    from pangenomix_b200 import _native
    coo = random_table(n, seed=7 * n, n_genes=6000)
    eng = _engine(coo, long_threshold=1, slice_words=1)
    k_total = eng.host_plan.n_superblocks * 1024
    assert k_total // per_genome >= 5 or per_genome > 1024
    out = torch_cuda.full((n, n), -7, dtype=torch_cuda.int32, device="cuda")
    work = torch_cuda.empty(n * per_genome, dtype=torch_cuda.uint8, device="cuda")
    _native.check(eng.lib.pgx_shared_genes(ctypes.byref(eng.c_plan), out.data_ptr(), work.data_ptr(), n * per_genome,
                                           torch_cuda.cuda.current_stream().cuda_stream))
    assert np.array_equal(out.cpu().numpy(), shared_np.shared_direct(coo))


def test_shared_genes_of_c4_sampled_rows(torch_cuda):
    coo = golden_matrix("c4_200000x10000")
    eng = _engine(coo)
    s = eng.shared_genes_device()
    assert torch_cuda.equal(s, s.T)
    colsum = np.bincount(coo.col, minlength=coo.shape[1]).astype(np.int32)
    assert np.array_equal(torch_cuda.diagonal(s).cpu().numpy(), colsum)
    cols = np.sort(np.random.default_rng(4).choice(coo.shape[1], 64, replace=False))
    cols[:2] = (0, coo.shape[1] - 1)
    assert np.array_equal(s[torch_cuda.from_numpy(cols).cuda()].cpu().numpy(), shared_np.shared_sample_rows(coo, cols))


def test_inconsistent_plan_is_refused(torch_cuda):
    from pangenomix_b200 import _native
    eng = _engine(random_table(40, seed=3))
    bad = _native.PgxPlan.from_buffer_copy(eng.c_plan)
    zeros = torch_cuda.zeros(40, dtype=torch_cuda.int32, device="cuda")
    bad.d_colsum = zeros.data_ptr()                         # no genes in any genome, yet rows that list genomes
    out = torch_cuda.empty((40, 40), dtype=torch_cuda.int32, device="cuda")
    work = torch_cuda.empty(40 * 128, dtype=torch_cuda.uint8, device="cuda")
    rc = eng.lib.pgx_shared_genes(ctypes.byref(bad), out.data_ptr(), work.data_ptr(), 40 * 128, None)
    assert rc == 1 and b"inconsistent" in eng.lib.pgx_last_error()


@pytest.mark.parametrize("name", ["synth_800x50_s0", "c2slice_4000x400", "edge_500x37", "tiny_40x3"])
def test_fluidity_rows_are_reproducible_and_match_the_oracle(torch_cuda, name):
    coo = golden_matrix(name)
    eng = _engine(coo)
    s = eng.shared_genes_device()
    a = eng.fluidity_rows_device(s).cpu().numpy()
    b = eng.fluidity_rows_device(s).cpu().numpy()
    assert a.dtype == np.float64 and a.view(np.uint64).tolist() == b.view(np.uint64).tolist()
    want = shared_np.fluidity_rows(s.cpu().numpy())
    np.testing.assert_allclose(a, want, rtol=1e-12, atol=0)


def test_fluidity_rows_nan_for_empty_genome_pairs(torch_cuda):
    import scipy.sparse
    x = np.zeros((30, 4), dtype=np.int64)
    x[:10, 2] = 1
    x[5:20, 3] = 1
    eng = _engine(scipy.sparse.coo_matrix(x))
    rows = eng.fluidity_rows_device(eng.shared_genes_device()).cpu().numpy()
    assert np.isnan(rows[0]) and np.isnan(rows[1])
    np.testing.assert_allclose(rows[2:], shared_np.fluidity_rows(shared_np.shared_direct(x))[2:], rtol=1e-12)


@pytest.mark.parametrize("name", ["kat_6x5", "synth_800x50_s1", "c2slice_4000x400"])
def test_api_matches_the_oracle_and_leaves_numpy_alone(torch_cuda, name):
    import pandas as pd
    from pangenomix_b200 import pangenome_analysis as pa
    coo = golden_matrix(name)
    df = _lsdf(coo)
    np.random.seed(5)
    state = np.random.get_state()
    shared = pa.shared_gene_counts(df)
    fl = pa.compute_genomic_fluidity(df)
    after = np.random.get_state()
    assert all(np.array_equal(x, y) for x, y in zip(state, after))
    s = shared_np.shared_direct(coo)
    assert isinstance(shared, pd.DataFrame) and shared.dtypes.unique().tolist() == [np.dtype(np.int32)]
    assert list(shared.index) == list(df.columns) and list(shared.columns) == list(df.columns)
    assert np.array_equal(shared.values, s)
    assert fl["fluidity"] == pytest.approx(shared_np.fluidity_by_definition(s), rel=1e-12)
    assert fl["jackknife_se"] == pytest.approx(shared_np.jackknife_by_definition(s), rel=1e-9)
    assert fl["n_genomes"] == coo.shape[1]


def test_api_shares_the_plan_with_rarefaction(torch_cuda, capsys):
    from pangenomix_b200 import pangenome_analysis as pa
    df = _lsdf(golden_matrix("synth_800x50_s0"))
    np.random.seed(11)
    before = pa.estimate_pan_core_size(df, 8)
    engine = pa._engine_for(df)
    capsys.readouterr()
    pa.compute_genomic_fluidity(df)
    pa.shared_gene_counts(df)
    assert capsys.readouterr().out == ""
    assert pa._engine_for(df) is engine
    np.random.seed(11)
    after = pa.estimate_pan_core_size(df, 8)
    assert before.equals(after)


def test_api_rejects_single_genome_tables(torch_cuda):
    import scipy.sparse
    from pangenomix_b200 import pangenome_analysis as pa
    with pytest.raises(ValueError):
        pa.compute_genomic_fluidity(_lsdf(scipy.sparse.coo_matrix(np.ones((5, 1), dtype=np.int64))))
