"""Parity of the CUDA path (through the C ABI) with the oracle and the reference-generated
golden fixtures.  Bit-exact for the curves; fp64 likelihoods within 1e-9 relative (the
tolerance BASELINE.json's north_star states)."""
import numpy as np
import pandas as pd
import pytest
import scipy.sparse

import oracle
from conftest import BIG_CURVE_CASES, CURVE_CASES, config_matrix_cached, draw_perms, golden_matrix, load_golden

pytestmark = pytest.mark.gpu

LL_RTOL = 1e-9


@pytest.fixture(scope="module")
def engine_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")
    from pangenomix_b200 import _native, engine
    _native.load()
    yield engine
    _native.set_tuning(0, 0, 0)


def _oracle_curves(coo, perms):
    pan, core = oracle.pan_core_curves_minrank(coo, np.asarray(perms, dtype=np.int64))
    return np.hstack([pan, core]).astype(np.int32)


@pytest.mark.parametrize("name", CURVE_CASES)
def test_curves_match_reference_fixtures(engine_mod, name):
    import torch
    g = load_golden(name)
    coo = golden_matrix(name, g)
    eng = engine_mod.PanCoreEngine(coo)
    perms = draw_perms(int(g["seed"]), coo.shape[1], int(g["num_iter"])).astype(np.uint16)
    want = g["curves"]
    got_host = eng.curves_host(perms)
    assert got_host.dtype == np.int32 and np.array_equal(got_host, want)
    got_f64 = eng.curves_host(perms, out_f64=True, perms_per_block=3)
    assert got_f64.dtype == np.float64 and np.array_equal(got_f64, want.astype(np.float64))
    d_perms = torch.from_numpy(perms.view(np.int16)).cuda()
    got_dev = eng.curves_device(d_perms).cpu().numpy()
    assert np.array_equal(got_dev, want)


@pytest.mark.parametrize("name", BIG_CURVE_CASES)
def test_curves_match_live_reference_at_full_size(engine_mod, name):
    """Configs C2 and C4 at BASELINE.json's full size against curves the LIVE reference computed for the same table
    and seed (tests/golden/make_golden.py --big): all 1,000 permutations of C2, 16 of C4; both C-ABI paths."""
    import torch
    g = load_golden(name)
    coo = golden_matrix(name, g)
    eng = engine_mod.PanCoreEngine(coo)
    num_iter = int(g["num_iter"])
    np.random.seed(int(g["seed"]))
    perms = engine_mod.draw_legacy_permutations(coo.shape[1], num_iter)
    want = g["curves"]
    assert np.array_equal(eng.curves_host(perms), want)
    assert np.array_equal(eng.curves_host(perms, out_f64=True), want.astype(np.float64))
    assert np.array_equal(eng.curves_device(torch.from_numpy(perms.view(np.int16)).cuda()).cpu().numpy(), want)
    np.random.seed(int(g["seed"]))
    table = eng.estimate(num_iter)
    assert np.array_equal(table, want.astype(np.float64))
    if name == "c2_40000x400":
        # config C2 as BASELINE.json states it: 1,000 permutations + the Heaps fit on their mean
        from pangenomix_b200 import pangenome_analysis as pa, plot
        n = coo.shape[1]
        assert num_iter == 1000
        df = pd.DataFrame(table, columns=["Pan%d" % (i + 1) for i in range(n)] + ["Core%d" % (i + 1) for i in range(n)])
        mean = plot.calculate_mean(df)
        assert np.array_equal(mean.values[0], g["mean"])
        np.testing.assert_allclose(pa.fit_heaps_by_iteration(mean).values[0], g["heaps_mean"], rtol=1e-9)


@pytest.mark.parametrize("name", ["kat_6x5", "synth_800x50_s0", "c1_8000x50", "c2slice_4000x400"])
def test_drop_in_api_frame_rng_and_heaps(engine_mod, name, capsys):
    from pangenomix_b200 import pangenome_analysis as pa, plot, sparse_utils as su, synth
    g = load_golden(name)
    coo = golden_matrix(name, g)
    index, columns = synth.labels_for(*coo.shape)
    lsdf = su.LightSparseDataFrame(index, columns, coo)
    num_iter, n = int(g["num_iter"]), coo.shape[1]
    np.random.seed(int(g["seed"]))
    df = pa.estimate_pan_core_size(lsdf, num_iter, log_batch=max(1, num_iter // 2))
    follow = np.random.random_sample(2)
    out = capsys.readouterr().out
    assert out.startswith("Converting DataFrame to matrix...\nGenerating pan/core curves from shuffled strains\n")
    assert "\tIteration %d of %d" % (max(1, num_iter // 2), num_iter) in out
    assert isinstance(df, pd.DataFrame) and df.values.dtype == np.float64
    assert df.shape == (num_iter, 2 * n)
    assert list(df.index) == ["Iter%d" % (i + 1) for i in range(num_iter)]
    assert list(df.columns) == ["Pan%d" % (i + 1) for i in range(n)] + ["Core%d" % (i + 1) for i in range(n)]
    assert np.array_equal(df.values, g["curves"].astype(np.float64))
    # exactly num_iter shuffles were consumed from the global stream
    draw_perms(int(g["seed"]), n, num_iter)
    assert np.array_equal(follow, np.random.random_sample(2))
    mean = plot.calculate_mean(df)
    assert np.array_equal(mean.values[0], g["mean"])
    fit = pa.fit_heaps_by_iteration(mean)
    np.testing.assert_allclose(fit.values[0], g["heaps_mean"], rtol=1e-12)
    fit_it = pa.fit_heaps_by_iteration(df.iloc[:min(num_iter, 8)])
    np.testing.assert_allclose(fit_it.values, g["heaps_iter"], rtol=1e-12)
    assert list(fit_it.columns) == ["alpha", "kappa"] and fit_it.index[0] == "Iter1"


def test_npz_written_by_the_reference_to_curves(engine_mod, capsys):
    """The whole user path of README.md:146-176 on the file the REFERENCE's own writer produced
    (tests/golden/lsdf_small.npz): read_lsdf -> estimate_pan_core_size -> calculate_mean -> fit_heaps,
    against the curves and fits the live reference computed from the same table and seed."""
    import os
    from conftest import GOLDEN
    from pangenomix_b200 import pangenome_analysis as pa, plot, sparse_utils as su
    g = load_golden("synth_800x50_s0")
    lsdf = su.read_lsdf(os.path.join(GOLDEN, "lsdf_small.npz"))
    assert lsdf.shape == (800, 50)
    np.random.seed(int(g["seed"]))
    df = pa.estimate_pan_core_size(lsdf, int(g["num_iter"]))
    capsys.readouterr()
    assert np.array_equal(df.values, g["curves"].astype(np.float64))
    mean = plot.calculate_mean(df)
    assert np.array_equal(mean.values[0], g["mean"])
    np.testing.assert_allclose(pa.fit_heaps_by_iteration(mean).values[0], g["heaps_mean"], rtol=1e-12)
    # a second call on the same LSDF object reuses the uploaded table
    np.random.seed(int(g["seed"]))
    assert np.array_equal(pa.estimate_pan_core_size(lsdf, 3).values, g["curves"][:3].astype(np.float64))
    capsys.readouterr()


def _mixed_matrix(n, seed=5, per_class=24):
    rng = np.random.RandomState(seed)
    dens = np.concatenate([np.full(per_class, d) for d in
                           (0.0, 2.0 / n, 0.004, 0.015, 0.03, 0.06, 0.12, 0.3, 0.5, 0.8, 0.97, 1.0 - 2.0 / n, 1.0)])
    x = (rng.random_sample((dens.size, n)) < dens[:, None]).astype(np.int64)
    return scipy.sparse.coo_matrix(x)


@pytest.mark.parametrize("perms_per_cta", [1, 2, 4, 8])
@pytest.mark.parametrize("splits,threads", [(1, 64), (3, 256), (7, 1024)])
@pytest.mark.parametrize("threshold", [0, 40])
def test_every_launch_shape_and_row_kind(engine_mod, perms_per_cta, splits, threads, threshold):
    from pangenomix_b200 import _native
    coo = _mixed_matrix(700)
    eng = engine_mod.PanCoreEngine(coo, long_threshold=threshold)
    hp = eng.host_plan
    assert (hp.n_long > 0) == (threshold > 0) and hp.n_rows > 0
    assert len({int(m) & 0xFFFF for m in hp.tasks[:, 1]}) >= 5          # many chunk-count classes
    perms = draw_perms(3, 700, 13).astype(np.uint16)       # 13: not a multiple of any batch
    want = _oracle_curves(coo, perms)
    _native.set_tuning(perms_per_cta, splits, threads)
    try:
        assert np.array_equal(eng.curves_host(perms), want)
    finally:
        _native.set_tuning(0, 0, 0)


@pytest.mark.parametrize("threshold", [2, 8, 64, 200])
def test_bitmap_probe_rows(engine_mod, threshold):
    """Every general gene at or above the threshold goes through the bit-sliced probe kernel:
    several superblocks (the last one partial), walks of very different lengths."""
    coo = _mixed_matrix(1500, seed=threshold, per_class=300 if threshold == 8 else 10)
    eng = engine_mod.PanCoreEngine(coo, long_threshold=threshold)
    hp = eng.host_plan
    assert hp.n_long > 0 and (threshold > 2 or hp.n_rows == 0)
    assert hp.n_superblocks == (hp.n_long + 1024 * hp.slice_words - 1) // (1024 * hp.slice_words)
    perms = draw_perms(17, 1500, 150).astype(np.uint16)
    assert np.array_equal(eng.curves_host(perms), _oracle_curves(coo, perms))


@pytest.mark.parametrize("slice_words", [1, 2, 4])
def test_bitmap_slices_of_1_2_4_words(engine_mod, slice_words):
    """The probe walk with 1, 2 and 4 words per lane: several superblocks, the last one ragged."""
    from pangenomix_b200.plan import build_host_plan
    coo = _mixed_matrix(600, seed=21, per_class=600)
    hp = build_host_plan(coo, long_threshold=6, slice_words=slice_words)
    assert hp.n_long > 4096 and hp.n_superblocks >= 2
    eng = engine_mod.PanCoreEngine(coo, host_plan=hp)
    perms = draw_perms(23, 600, 70).astype(np.uint16)
    assert np.array_equal(eng.curves_host(perms), _oracle_curves(coo, perms))


@pytest.mark.parametrize("n", [14000, 20000, 40000, 65503])
def test_wide_tables_fall_back_to_smaller_batches(engine_mod, n):
    """N above ~14k no longer fits 8 rank tables in shared memory: 4, 2, then 1 per CTA."""
    coo = _mixed_matrix(n, seed=n, per_class=6)
    eng = engine_mod.PanCoreEngine(coo)
    assert eng.host_plan.perms_per_cta == {14000: 8, 20000: 4, 40000: 2, 65503: 1}[n]
    assert eng.host_plan.n_long > 0
    perms = draw_perms(11, n, 5).astype(np.uint16)
    assert np.array_equal(eng.curves_host(perms), _oracle_curves(coo, perms))
    lists_only = engine_mod.PanCoreEngine(coo, long_threshold=0)
    assert np.array_equal(lists_only.curves_host(perms[:2]), _oracle_curves(coo, perms[:2]))


def test_random_tables_every_layout_choice(engine_mod):
    """40 random tables (shape, density profile, threshold, batch size, slice width all drawn at random)
    through the CUDA path, against the oracle, bit for bit."""
    from pangenomix_b200 import _native
    from pangenomix_b200.plan import build_host_plan
    rng = np.random.RandomState(20260101)
    try:
        for case in range(40):
            n = int(rng.choice([1, 2, 3, 7, 31, 32, 33, 64, 100, 257, 400]))
            g = int(rng.choice([0, 1, 5, 40, 300, 1500]))
            style = rng.choice(["mixed", "sparse", "dense", "half"])
            dens = {"mixed": rng.choice([0.0, 0.03, 0.1, 0.3, 0.5, 0.8, 0.97, 1.0], size=g),
                    "sparse": rng.uniform(0.0, 0.1, size=g), "dense": rng.uniform(0.9, 1.0, size=g),
                    "half": np.full(g, 0.5)}[style]
            x = (rng.random_sample((g, n)) < dens[:, None]).astype(np.int64)
            coo = scipy.sparse.coo_matrix(x)
            hp = build_host_plan(coo, long_threshold=int(rng.choice([0, 2, 4, 9, 30])),
                                 perms_per_cta=int(rng.choice([1, 2, 4, 8])), slice_words=int(rng.choice([1, 2, 4])))
            eng = engine_mod.PanCoreEngine(coo, host_plan=hp)
            _native.set_tuning(0, int(rng.choice([0, 1, 5])), int(rng.choice([0, 64, 256, 1024])))
            n_perm = int(rng.choice([1, 7, 8, 9, 129]))
            perms = np.stack([rng.permutation(n) for _ in range(n_perm)]).astype(np.uint16)
            got = eng.curves_host(perms)
            assert np.array_equal(got, _oracle_curves(coo, perms)), (case, n, g, style)
    finally:
        _native.set_tuning(0, 0, 0)


def test_many_permutations_in_one_call(engine_mod):
    """70,001 permutations in ONE call (more than 65,535 batches of the old grid limit would allow, an odd
    count, several host-path blocks): oracle parity on a sample, invariants on all."""
    coo = _mixed_matrix(60, seed=4, per_class=30)
    eng = engine_mod.PanCoreEngine(coo, long_threshold=6)
    assert eng.host_plan.n_long > 0 and eng.host_plan.n_rows > 0
    rng = np.random.RandomState(8)
    perms = np.argsort(rng.random_sample((70001, 60)), axis=1).astype(np.uint16)
    curves = eng.curves_host(perms)
    sample = [0, 1, 7, 8, 65535, 65536, 69999, 70000]
    assert np.array_equal(curves[sample], _oracle_curves(coo, perms[sample]))
    pan, core = curves[:, :60], curves[:, 60:]
    assert np.all(np.diff(pan, axis=1) >= 0) and np.all(np.diff(core, axis=1) <= 0)
    assert np.array_equal(pan[:, 0], core[:, 0])
    col_sums = np.asarray(coo.sum(axis=0)).ravel()
    assert np.array_equal(pan[:, 0], col_sums[perms[:, 0]])


def test_degenerate_shapes(engine_mod):
    import torch
    # no folded rows at all: everything is a closed form
    x = np.zeros((6, 3), dtype=np.int64)
    x[0] = 1
    x[1, 2] = 1
    x[2, :2] = 1
    eng = engine_mod.PanCoreEngine(scipy.sparse.coo_matrix(x))
    assert eng.host_plan.n_tasks == 0
    perms = draw_perms(1, 3, 9).astype(np.uint16)
    assert np.array_equal(eng.curves_host(perms), _oracle_curves(scipy.sparse.coo_matrix(x), perms))
    # zero permutations, one permutation
    assert eng.curves_host(perms[:0]).shape == (0, 6)
    assert np.array_equal(eng.curves_host(perms[:1]), _oracle_curves(scipy.sparse.coo_matrix(x), perms[:1]))
    # a single genome
    one = scipy.sparse.coo_matrix(np.array([[1], [0], [1]], dtype=np.int64))
    e1 = engine_mod.PanCoreEngine(one)
    assert np.array_equal(e1.curves_host(np.zeros((4, 1), dtype=np.uint16)),
                          np.tile(np.array([[2, 2]], dtype=np.int32), (4, 1)))
    with pytest.raises(ValueError):
        eng.curves_device(torch.zeros((2, 5), dtype=torch.int16, device="cuda"))


def test_c2_full_size_properties_and_spot_parity(engine_mod):
    """Config C2 (40,000 x 400, 1,000 permutations): size-independent invariants on every
    curve, oracle parity on a sample of them."""
    import os
    from oracle import cport
    coo = config_matrix_cached("c2")
    eng = engine_mod.PanCoreEngine(coo)
    n, g = 400, 40000
    np.random.seed(12345)
    perms = engine_mod.draw_legacy_permutations(n, 1000)
    curves = eng.curves_host(perms)
    pan, core = curves[:, :n], curves[:, n:]
    counts = np.diff(coo.tocsr().indptr)
    assert np.all(np.diff(pan, axis=1) >= 0) and np.all(np.diff(core, axis=1) <= 0)
    assert np.array_equal(pan[:, 0], core[:, 0])
    assert np.all(pan[:, -1] == np.count_nonzero(counts)) and np.all(core[:, -1] == np.count_nonzero(counts == n))
    col_sums = np.asarray(coo.sum(axis=0)).ravel()
    assert np.array_equal(pan[:, 0], col_sums[perms[:, 0]])
    sample = np.r_[0:8, 496:504, 952:1000]                                  # 64 curves against the oracle's C port
    ref_pan, ref_core = cport.curves_direct(coo, perms[sample].astype(np.int32), n_threads=os.cpu_count() or 1)
    assert np.array_equal(curves[sample], np.hstack([ref_pan, ref_core]).astype(np.int32))
    assert np.array_equal(curves[[0, 999]], _oracle_curves(coo, perms[[0, 999]]))
    # determinism and independence from the batch a permutation lands in
    again = eng.curves_host(perms[::-1].copy())[::-1]
    assert np.array_equal(again, curves)


def test_c4_shape_sample(engine_mod):
    """A 10,000-genome table (the C4 genome count, 1/10 of its genes so that the oracle
    stays in seconds): 8 rank tables of 20 KB per CTA, long rows, every closed form."""
    from pangenomix_b200 import synth
    coo = synth.bernoulli_matrix(20000, 10000, 4500, seed=20244)
    eng = engine_mod.PanCoreEngine(coo)
    np.random.seed(12345)
    perms = engine_mod.draw_legacy_permutations(10000, 24)
    curves = eng.curves_host(perms)
    assert np.array_equal(curves[[0, 7, 8, 23]], _oracle_curves(coo, perms[[0, 7, 8, 23]]))
    pan, core = curves[:, :10000], curves[:, 10000:]
    assert np.all(np.diff(pan, axis=1) >= 0) and np.all(np.diff(core, axis=1) <= 0)
    assert np.array_equal(pan[:, 0], core[:, 0])


def test_c4_full_size_properties_and_spot_parity(engine_mod):
    """Config C4 at BASELINE.json's full size (200,000 genes x 10,000 genomes): size-independent
    invariants on 1,000 curves, oracle parity on two of them, and the two-stream and
    back-to-back kernel schedules must agree bit for bit."""
    import os
    from oracle import build as oracle_build, cport
    from pangenomix_b200 import _native
    coo = config_matrix_cached("c4")
    eng = engine_mod.PanCoreEngine(coo)
    hp = eng.host_plan
    assert hp.n_long > 0 and hp.n_rows > 0 and hp.perms_per_cta == 8
    n, g = 10000, 200000
    np.random.seed(12345)
    perms = engine_mod.draw_legacy_permutations(n, 1000)
    curves = eng.curves_host(perms)
    pan, core = curves[:, :n], curves[:, n:]
    counts = np.diff(coo.tocsr().indptr)
    assert np.all(np.diff(pan, axis=1) >= 0) and np.all(np.diff(core, axis=1) <= 0)
    assert np.array_equal(pan[:, 0], core[:, 0])
    assert np.all(pan[:, -1] == np.count_nonzero(counts)) and np.all(core[:, -1] == np.count_nonzero(counts == n))
    col_sums = np.asarray(coo.sum(axis=0)).ravel()
    assert np.array_equal(pan[:, 0], col_sums[perms[:, 0]])
    # sum over k of pan[k] = sum over genes of (N - first presence): a checksum of checksums against numpy
    oracle_build.build()
    sample = np.r_[0:24, 488:512, 984:1000]                                 # 64 curves against the oracle's C port
    ref_pan, ref_core = cport.curves_direct(coo, perms[sample].astype(np.int32), n_threads=os.cpu_count() or 1)
    assert np.array_equal(curves[sample], np.hstack([ref_pan, ref_core]).astype(np.int32))
    # per-kernel timing mode runs the row kernels back to back instead of side by side (device calls only: host-buffer
    # calls are never profiled)
    import torch
    _native.profile_read()
    _native.profile_enable(True)
    try:
        again = eng.curves_device(torch.from_numpy(perms[:200].view(np.int16)).cuda()).cpu().numpy()
        assert _native.profile_read()[3] == 1
    finally:
        _native.profile_enable(False)
        _native.profile_read()
    assert np.array_equal(again, curves[:200])
    assert np.array_equal(eng.curves_host(perms[:200]), curves[:200])


def test_c5_full_size_spot_parity(engine_mod):
    """Config C5 at BASELINE.json's full size (2,000,000 alleles x 50,000 genomes, nnz 2.0e8): 2 permutations per
    list CTA, 32-lane wavefront groups, ~150,000 bitmap rows.  16 curves bit for bit against the oracle's C port of
    pangenome_analysis.py:81-90 (run in full: 16 x 1e11 cell visits on all host threads), invariants on 64."""
    import os
    from oracle import build as oracle_build, cport
    coo = config_matrix_cached("c5")
    n, g = 50000, 2000000
    assert coo.shape == (g, n) and coo.nnz > 150_000_000
    eng = engine_mod.PanCoreEngine(coo)
    hp = eng.host_plan
    assert hp.perms_per_cta == 2 and hp.n_long > 100000 and hp.n_rows > 500000
    np.random.seed(12345)
    perms = engine_mod.draw_legacy_permutations(n, 64)
    curves = eng.curves_host(perms)
    pan, core = curves[:, :n], curves[:, n:]
    counts = np.bincount(coo.row, minlength=g)
    assert np.all(np.diff(pan, axis=1) >= 0) and np.all(np.diff(core, axis=1) <= 0)
    assert np.array_equal(pan[:, 0], core[:, 0])
    assert np.all(pan[:, -1] == np.count_nonzero(counts)) and np.all(core[:, -1] == np.count_nonzero(counts == n))
    col_sums = np.bincount(coo.col, minlength=n)
    assert np.array_equal(pan[:, 0], col_sums[perms[:, 0]])
    # the table's marginals and gene-frequency spectrum at this size (2.0e8 entries through the pinned lanes)
    row_sum, col_sum, spectrum, first = engine_mod.table_marginals(coo)
    assert np.array_equal(row_sum, counts) and np.array_equal(col_sum, col_sums)
    assert np.array_equal(spectrum, np.bincount(counts, minlength=n + 1))
    seen = np.flatnonzero(spectrum)
    assert np.array_equal(counts[first[seen]], seen) and np.all(first[seen[1:]] >= 0)
    oracle_build.build()
    threads = os.cpu_count() or 1
    sample = np.r_[0:8, 56:64]
    gm = cport.GenomeMajor(coo)
    del coo
    ref_pan, ref_core = cport.curves_direct(gm, perms[sample].astype(np.int32), n_threads=min(threads, 16))
    assert np.array_equal(curves[sample], np.hstack([ref_pan, ref_core]).astype(np.int32))
    # ... and the first curve against the live reference's own (tests/golden/make_golden.py --c5; the same seed)
    fixture = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "c5_2000000x50000.npz")
    if os.path.exists(fixture):
        g5 = np.load(fixture)
        assert int(g5["seed"]) == 12345 and tuple(int(v) for v in g5["shape"]) == (g, n)
        assert np.array_equal(curves[0], g5["curves"][0])
    # the reference-facing call on the same table: float64, the same rows
    np.random.seed(12345)
    assert np.array_equal(eng.estimate(8), curves[:8].astype(np.float64))


def test_genomes_above_65535_genes_use_int32_bins(engine_mod):
    """A table whose genomes hold more than 65,535 genes cannot count in uint16 bins: the int32 path of every
    kernel, natively (not through PGX_WIDE_BINS)."""
    import torch
    rng = np.random.RandomState(7)
    dens = np.concatenate([np.full(68000, 0.985), rng.uniform(0.0, 1.0, size=4000)])
    x = (rng.random_sample((dens.size, 48)) < dens[:, None]).astype(np.int64)
    coo = scipy.sparse.coo_matrix(x)
    eng = engine_mod.PanCoreEngine(coo, long_threshold=12)
    assert eng.c_plan.max_colsum > 65535 and eng.host_plan.n_long > 0 and eng.host_plan.n_rows > 0
    perms = draw_perms(3, 48, 21).astype(np.uint16)
    want = _oracle_curves(coo, perms)
    assert want.max() > 65535
    assert np.array_equal(eng.curves_host(perms), want)
    assert np.array_equal(eng.curves_host(perms, out_f64=True, perms_per_block=8), want.astype(np.float64))
    assert np.array_equal(eng.curves_device(torch.from_numpy(perms.view(np.int16)).cuda()).cpu().numpy(), want)
    np.random.seed(3)
    assert np.array_equal(eng.estimate(21), want.astype(np.float64))


def _many_genomes_table(n, seed):
    from pangenomix_b200 import synth
    return synth.bernoulli_matrix(20000, n, 3000, seed=seed).tocoo()


def test_split_transfer_of_tables_with_many_genomes(engine_mod):
    """Tables of 2,048 genomes or more: the host-buffer calls ship uint16 heads + uint8 tails of the curves' steps
    (split_steps_kernel, pgx_expand_split).  Same curves as the oracle's for int32 and float64 results, ragged blocks
    and the RNG-fed call."""
    from pangenomix_b200 import _native
    n = 2304
    coo = _many_genomes_table(n, seed=3)
    eng = engine_mod.PanCoreEngine(coo)
    perms = draw_perms(5, n, 45).astype(np.uint16)
    want = _oracle_curves(coo, perms)
    for block in (0, 7, 16):
        assert np.array_equal(eng.curves_host(perms, perms_per_block=block), want)
    assert int(_native.load().pgx_split_head()) == 512
    assert np.array_equal(eng.curves_host(perms, out_f64=True, perms_per_block=11), want.astype(np.float64))
    np.random.seed(5)
    assert np.array_equal(eng.estimate(45), want.astype(np.float64))


def test_split_transfer_recovers_from_a_head_that_is_too_short(engine_mod):
    """PGX_SPLIT_HEAD=4 (read when the staging is set up for a new table size): the first genomes add thousands of
    genes each, the 4-entry heads overflow, the blocks in flight travel again as uint16 and the head doubles until the
    tails fit -- with the same curves throughout."""
    import os
    from pangenomix_b200 import _native
    n = 2112                                             # a size no other test uses: the staging is set up anew
    coo = _many_genomes_table(n, seed=4)
    eng = engine_mod.PanCoreEngine(coo)
    perms = draw_perms(6, n, 90).astype(np.uint16)
    want = _oracle_curves(coo, perms)
    old = os.environ.get("PGX_SPLIT_HEAD")
    os.environ["PGX_SPLIT_HEAD"] = "4"
    try:
        got = eng.curves_host(perms, perms_per_block=6)
        grown = int(_native.load().pgx_split_head())
        assert np.array_equal(got, want)
        assert grown > 4 and grown % 4 == 0
        assert np.array_equal(eng.curves_host(perms, out_f64=True, perms_per_block=6), want.astype(np.float64))
        assert int(_native.load().pgx_split_head()) >= grown
    finally:
        if old is None:
            del os.environ["PGX_SPLIT_HEAD"]
        else:
            os.environ["PGX_SPLIT_HEAD"] = old


def test_c_host_program_end_to_end(engine_mod, tmp_path):
    """tests/c/abi_host.c --gpu: plan, upload, rarefy and check 21 genome orders from plain C through the C ABI alone
    (pgx_host_plan_create, pgx_plan_upload, pgx_pan_core_curves_host, pgx_plan_create, pgx_plan_destroy)."""
    import subprocess
    from test_abi_cpu import _build_c_host
    exe = _build_c_host(tmp_path)
    run = subprocess.run([exe, "--gpu"], capture_output=True, text=True)
    assert run.returncode == 0, run.stdout + run.stderr
    assert "gpu ok: 21 curves, the marginals and 13 KS statistics bit-exact" in run.stdout


def test_probe_gate_off_gives_the_same_curves(engine_mod):
    """PGX_PROBE_GATE=0 (read once per process, hence a child process): without the stream-level wait before the
    probe launch the two row kernels may start in either order; the curves must not depend on it."""
    import os
    import subprocess
    import sys
    from conftest import REPO
    code = (
        "import sys, numpy as np; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import oracle\n"
        "from conftest import draw_perms\n"
        "from pangenomix_b200 import engine, synth\n"
        "coo = synth.bernoulli_matrix(6000, 900, 450, seed=5)\n"
        "eng = engine.PanCoreEngine(coo)\n"
        "assert eng.host_plan.n_long > 0 and eng.host_plan.n_rows > 0\n"
        "perms = draw_perms(4, 900, 37)\n"
        "pan, core = oracle.pan_core_curves_minrank(coo, perms)\n"
        "for _ in range(3):\n"
        "    assert np.array_equal(eng.curves_host(perms.astype(np.uint16)), np.hstack([pan, core]).astype(np.int32))\n"
        "print('gate off ok')\n" % (REPO, os.path.join(REPO, "tests")))
    env = dict(os.environ, PGX_PROBE_GATE="0")
    run = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=600)
    assert run.returncode == 0 and "gate off ok" in run.stdout, run.stdout + run.stderr


def test_rows_that_are_not_permutations_are_reported(engine_mod):
    from pangenomix_b200 import _native
    coo = _mixed_matrix(300)
    eng = engine_mod.PanCoreEngine(coo, long_threshold=20)
    perms = draw_perms(3, 300, 12).astype(np.uint16)
    bad = perms.copy()
    bad[5, 17] = bad[5, 18]                                  # one genome twice, another never
    with pytest.raises(_native.PgxError, match="not permutations"):
        eng.curves_host(bad)
    bad[5, 17] = 40000                                       # out of range
    with pytest.raises(_native.PgxError, match="not permutations"):
        eng.curves_host(bad)
    assert np.array_equal(eng.curves_host(perms), _oracle_curves(coo, perms))     # the engine is still usable


def test_estimate_blocks_progress_and_rng_state(engine_mod, capsys):
    """engine.estimate: several staging blocks, a ragged last block, progress lines, RNG consumption."""
    from pangenomix_b200 import synth
    coo = synth.bernoulli_matrix(3000, 300, 450, seed=1)
    eng = engine_mod.PanCoreEngine(coo)
    np.random.seed(5)
    got = eng.estimate(70, log_batch=25, block=16)
    tail = np.random.random_sample(3)
    out = capsys.readouterr().out
    assert [l for l in out.splitlines() if l.startswith("\tIteration")] == [
        "\tIteration 25 of 70", "\tIteration 50 of 70"]
    perms = draw_perms(5, 300, 70)
    assert np.array_equal(tail, np.random.random_sample(3))
    assert got.dtype == np.float64 and np.array_equal(got, _oracle_curves(coo, perms).astype(np.float64))
    # a second call reuses the staging buffers and may use a different block size
    np.random.seed(5)
    assert np.array_equal(eng.estimate(70), got)
    assert eng.estimate(0).shape == (0, 600)


# ---------------------------------------------------------------------------------------
# Batched Heaps-law fits (SURVEY.md 8f rank 2)
# ---------------------------------------------------------------------------------------
# scipy's curve_fit stops at ftol = xtol = 1.49e-8 and lands within ~1e-6 relative of the least-squares
# optimum (1.3e-6 on the 5-point KAT); the GPU fit runs to fp64 convergence.
HEAPS_RTOL = 5e-6


@pytest.mark.parametrize("name", ["kat_6x5", "synth_800x50_s0", "c1_8000x50", "c2slice_4000x400"])
def test_heaps_fits_match_reference_fixtures(engine_mod, name):
    """pgx_heaps_fit against the alpha/kappa the live reference (scipy curve_fit) produced."""
    import torch
    from pangenomix_b200 import pangenome_analysis as pa
    g = load_golden(name)
    n = int(g["shape"][1])
    curves = torch.from_numpy(np.ascontiguousarray(g["curves"].astype(np.int32))).cuda()
    fit, info = engine_mod.fit_heaps_device(curves)
    fit, info = fit.cpu().numpy(), info.cpu().numpy()
    assert np.all(info > 0)
    k = g["heaps_iter"].shape[0]
    np.testing.assert_allclose(fit[:k], g["heaps_iter"], rtol=HEAPS_RTOL)
    # float64 input, the mean row, DataFrame wrapper with the reference's labels
    df = pd.DataFrame(g["curves"].astype(np.float64), index=["Iter%d" % (i + 1) for i in range(g["curves"].shape[0])],
                      columns=["Pan%d" % (i + 1) for i in range(n)] + ["Core%d" % (i + 1) for i in range(n)])
    got = pa.fit_heaps_by_iteration_gpu(df)
    assert list(got.columns) == ["alpha", "kappa"] and list(got.index) == list(df.index)
    np.testing.assert_allclose(got.values[:k], g["heaps_iter"], rtol=HEAPS_RTOL)
    mean = pd.DataFrame([df.mean()], columns=df.columns)
    np.testing.assert_allclose(pa.fit_heaps_by_iteration_gpu(mean).values[0], g["heaps_mean"], rtol=HEAPS_RTOL)
    # bit-reproducible
    fit2, _ = engine_mod.fit_heaps_device(curves)
    assert np.array_equal(fit2.cpu().numpy(), fit)


def test_heaps_fits_of_a_whole_table_against_scipy(engine_mod):
    """Every iteration of a 400-genome table (200 curves): the drop-in scipy path on the host is the checker."""
    import torch
    from pangenomix_b200 import pangenome_analysis as pa, synth
    coo = synth.bernoulli_matrix(4000, 400, 450, seed=20242)
    eng = engine_mod.PanCoreEngine(coo)
    np.random.seed(3)
    perms = engine_mod.draw_legacy_permutations(400, 200)
    d_curves = eng.curves_device(torch.from_numpy(perms.view(np.int16)).cuda())
    fit, info = engine_mod.fit_heaps_device(d_curves)
    assert int(info.min()) > 0
    curves = d_curves.cpu().numpy().astype(np.float64)
    df = pd.DataFrame(curves, index=["Iter%d" % (i + 1) for i in range(200)],
                      columns=["Pan%d" % (i + 1) for i in range(400)] + ["Core%d" % (i + 1) for i in range(400)])
    want = pa.fit_heaps_by_iteration(df.iloc[::10])
    np.testing.assert_allclose(fit.cpu().numpy()[::10], want.values, rtol=HEAPS_RTOL)


# ---------------------------------------------------------------------------------------
# Bernoulli grid
# ---------------------------------------------------------------------------------------
def test_bernoulli_ll_grad_fixtures(engine_mod):
    g = load_golden("bernoulli_300x40")
    grid = engine_mod.BernoulliGrid(g["x"].astype(np.float64))
    for tag in ("0", "1"):
        ll, grad = grid.ll_grad(np.concatenate((g["p" + tag], g["q" + tag])))
        np.testing.assert_allclose(ll, g["ll" + tag], rtol=LL_RTOL)
        np.testing.assert_allclose(grad, g["grad" + tag], rtol=LL_RTOL, atol=1e-9 * np.abs(g["grad" + tag]).max())
    kat = engine_mod.BernoulliGrid(g["kat_x"])
    ll, grad = kat.ll_grad(np.concatenate((g["kat_p"], g["kat_q"])))
    np.testing.assert_allclose(ll, -2.502512292672613, rtol=LL_RTOL)
    np.testing.assert_allclose(grad, g["kat_grad"], rtol=LL_RTOL)
    with pytest.raises(ValueError):
        engine_mod.BernoulliGrid(np.array([[0.0, 2.0]]))


@pytest.mark.parametrize("shape", [(1, 1), (3, 33), (257, 513), (1000, 1300), (4000, 400)])
def test_bernoulli_ll_grad_vs_oracle(engine_mod, shape):
    from pangenomix_b200 import synth
    x, _, _ = synth.bernoulli_grid_matrix(shape[0], shape[1], seed=shape[0] + shape[1])
    rng = np.random.RandomState(1)
    p = rng.uniform(0.8, 0.99999999, size=shape[0])
    q = rng.uniform(0.8, 0.99999999, size=shape[1])
    grid = engine_mod.BernoulliGrid(x)
    ll, grad = grid.ll_grad(np.concatenate((p, q)))
    want_ll, want_grad = oracle.bernoulli_ll(x, p, q), oracle.bernoulli_grad(x, p, q)
    np.testing.assert_allclose(ll, want_ll, rtol=LL_RTOL)
    np.testing.assert_allclose(grad, want_grad, rtol=LL_RTOL, atol=1e-9 * np.abs(want_grad).max())
    ll2, grad2 = engine_mod.BernoulliGrid(x).ll_grad(np.concatenate((p, q)))
    assert ll2 == ll and np.array_equal(grad2, grad)         # bit-reproducible


def test_bernoulli_full_fit_matches_reference(engine_mod, capsys):
    from pangenomix_b200 import pangenome_analysis as pa, synth
    g = load_golden("bernoulli_300x40")
    x = g["x"].astype(np.float64)
    index, columns = synth.labels_for(*x.shape)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        df_opt, res = pa.compute_bernoulli_grid_core_genome(pd.DataFrame(x, index=index, columns=columns))
    out = capsys.readouterr().out
    assert "Initial loglikelihood:" in out and "Final loglikelihood:" in out
    assert list(df_opt.columns) == ["initial", "optimum"]
    assert list(df_opt.index) == ["Loglikelihood"] + ["p_" + s for s in index] + ["q_" + s for s in columns]
    np.testing.assert_allclose(df_opt["initial"].values, g["fit_initial"], rtol=LL_RTOL)
    # the optimiser path is sensitive to the last bits of LL/grad (SURVEY.md section 7):
    # compare the optimum itself and the core-gene call set it implies
    np.testing.assert_allclose(-res.fun, -float(g["fit_fun"]), rtol=1e-7)
    np.testing.assert_allclose(res.x, g["fit_x"], atol=2e-4)
    ref_p, got_p = g["fit_x"][:300], res.x[:300]
    margin = np.abs(ref_p - 0.99) > 1e-3
    assert np.array_equal((got_p >= 0.99)[margin], (ref_p >= 0.99)[margin])


def test_bernoulli_whole_table_fit_against_live_reference(engine_mod, capsys):
    """Config C3 on the WHOLE table (40,000 genes x 400 genomes, README.md:199-211) against the live reference's fit
    (make_golden.py --c3-whole, 3 minutes of reference time): likelihood and gradient at the reference's start point and
    at its optimum to 1e-9.  The optimum is flat at this size -- 147 of the reference's p_i lie within 1e-4 of the call
    threshold 0.99, and the two L-BFGS-B runs take slightly different paths (ulp-level differences of LL and gradient) --
    so of the fit itself the optimum LL is asserted (1e-6 relative) and the agreement of the call sets is REPORTED with
    its margin, and asserted only loosely."""
    import hashlib
    import warnings
    from pangenomix_b200 import pangenome_analysis as pa, synth
    g = load_golden("bernoulli_c3_40000x400")
    x, _, _ = synth.bernoulli_grid_matrix(40000, 400, seed=3)
    assert hashlib.sha256(x.astype(np.uint8).tobytes()).hexdigest() == str(g["x_digest"])
    n_genes, n_genomes = x.shape
    grid = engine_mod.BernoulliGrid(x)
    init = np.clip(np.concatenate((x.sum(axis=1) / float(n_genomes), 0.9999 * np.ones(n_genomes))), 0.8, 0.99999999)
    for tag, pq in (("init", init), ("opt", g["fit_x"])):
        ll, grad = grid.ll_grad(pq)
        np.testing.assert_allclose(ll, g["ll_" + tag], rtol=LL_RTOL)
        np.testing.assert_allclose(grad, g["grad_" + tag], rtol=LL_RTOL, atol=1e-9 * np.abs(g["grad_" + tag]).max())
    np.testing.assert_allclose(grid.ll_grad(init)[0], float(g["fit_ll_initial"]), rtol=LL_RTOL)
    index, columns = synth.labels_for(*x.shape)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        df_opt, res = pa.compute_bernoulli_grid_core_genome(pd.DataFrame(x, index=index, columns=columns))
    capsys.readouterr()
    np.testing.assert_allclose(-res.fun, -float(g["fit_fun"]), rtol=1e-6)
    ref_p, got_p = g["fit_x"][:n_genes], res.x[:n_genes]
    tau = 0.99
    both = int(((got_p >= tau) & (ref_p >= tau)).sum())
    either = int(((got_p >= tau) | (ref_p >= tau)).sum())
    worst = float(np.max(np.abs(res.x - g["fit_x"])))
    with capsys.disabled():
        print("\n[C3 40,000 x 400] L-BFGS-B iterations %d (reference %d), evaluations %d (reference %d), optimum LL %.6f "
              "(reference %.6f), max |x - x_ref| = %.3g; core genes at p >= %.2f: %d (reference %d), in both %d; "
              "reference p_i within 1e-4 of the threshold: %d" % (
                  res.nit, int(g["fit_nit"]), res.nfev, int(g["fit_nfev"]), -res.fun, -float(g["fit_fun"]), worst, tau,
                  int((got_p >= tau).sum()), int((ref_p >= tau).sum()), both, int((np.abs(ref_p - tau) < 1e-4).sum())))
    assert both >= 0.9 * either


def test_bernoulli_full_fit_at_c3_size_matches_live_reference(engine_mod, capsys):
    """Config C3 at its candidate-core size (4,000 genes x 400 genomes, prob_bounds (0.8, 0.99999999)): the whole
    compute_bernoulli_grid_core_genome call against the fixture the LIVE reference produced (make_golden.py --big):
    likelihood and gradient at the reference's start point and optimum to 1e-9, the optimum itself, and the
    core-gene call set {i : p_i >= 0.99} -- identical, with no margin carved out (the distance of the closest p_i to
    the threshold is printed)."""
    import hashlib
    import warnings
    from pangenomix_b200 import pangenome_analysis as pa, synth
    g = load_golden("bernoulli_c3_4000x400")
    x, _, _ = synth.bernoulli_grid_matrix(4000, 400, seed=3)
    assert hashlib.sha256(x.astype(np.uint8).tobytes()).hexdigest() == str(g["x_digest"])
    grid = engine_mod.BernoulliGrid(x)
    for tag, pq in (("init", g["fit_initial"][1:]), ("opt", g["fit_optimum"][1:])):
        ll, grad = grid.ll_grad(pq)
        np.testing.assert_allclose(ll, g["ll_" + tag], rtol=LL_RTOL)
        np.testing.assert_allclose(grad, g["grad_" + tag], rtol=LL_RTOL, atol=1e-9 * np.abs(g["grad_" + tag]).max())
    index, columns = synth.labels_for(*x.shape)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        df_opt, res = pa.compute_bernoulli_grid_core_genome(pd.DataFrame(x, index=index, columns=columns))
    capsys.readouterr()
    assert list(df_opt.index) == ["Loglikelihood"] + ["p_" + s for s in index] + ["q_" + s for s in columns]
    np.testing.assert_allclose(df_opt["initial"].values, g["fit_initial"], rtol=LL_RTOL)
    np.testing.assert_allclose(-res.fun, -float(g["fit_fun"]), rtol=LL_RTOL)
    np.testing.assert_allclose(df_opt["optimum"].values[0], g["fit_optimum"][0], rtol=LL_RTOL)
    ref_p, got_p = g["fit_x"][:4000], res.x[:4000]
    tau = 0.99
    closest = float(np.min(np.abs(ref_p - tau)))
    worst = float(np.max(np.abs(res.x - g["fit_x"])))
    with capsys.disabled():
        print("\n[C3 4,000 x 400] L-BFGS-B iterations %d (reference %d), evaluations %d (reference %d), max |x - x_ref| = %.3g, "
              "core genes at p >= %.2f: %d (reference %d), closest reference p_i to the threshold: %.3g" % (
                  res.nit, int(g["fit_nit"]), res.nfev, int(g["fit_nfev"]), worst, tau, int((got_p >= tau).sum()),
                  int((ref_p >= tau).sum()), closest))
    assert np.array_equal(got_p >= tau, ref_p >= tau)
    assert worst < 1e-6
