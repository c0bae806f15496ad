"""Host planning (pgx_host_plan_create through pangenomix_b200/plan.py) checked on the CPU against the golden
curves by walking the plan exactly as the kernels do (tests/plan_emulator.py), and against the numpy
specification of the planner (oracle/plan_np.py)."""
import numpy as np
import pytest
import scipy.sparse

from conftest import CURVE_CASES, draw_perms, golden_matrix, load_golden
from oracle import plan_np
from pangenomix_b200.plan import build_host_plan
from plan_emulator import check_layout, curves_from_plan


@pytest.mark.parametrize("name", CURVE_CASES)
def test_plan_walk_matches_reference(name):
    g = load_golden(name)
    coo = golden_matrix(name, g)
    hp = build_host_plan(coo)
    iters = min(int(g["num_iter"]), 3 if coo.shape[0] > 2000 else 20)
    perms = draw_perms(int(g["seed"]), coo.shape[1], iters)
    got = curves_from_plan(hp, perms)
    assert np.array_equal(got, g["curves"][:iters].astype(np.int64))


def test_plan_accounts_for_every_gene():
    g = load_golden("edge_500x37")
    coo = golden_matrix("edge_500x37", g)
    hp = build_host_plan(coo)
    assert hp.n_empty >= 10 and hp.n_full >= 10
    assert hp.w_present.sum() >= 20 and hp.w_absent.sum() >= 20
    assert hp.n_rows + hp.n_long + hp.n_empty + hp.n_full + hp.w_present.sum() + hp.w_absent.sum() == 500
    assert hp.n_long > 0 and hp.long_threshold == 8
    assert hp.chunks.shape[0] % (8 * 32) == 0 and hp.chunks.dtype == np.uint16
    assert np.array_equal(hp.colsum, np.asarray(coo.tocsr().sum(axis=0)).ravel())
    check_layout(hp)
    assert hp.algorithmic_bytes_per_perm == 4 * coo.nnz + 4 * 501
    assert np.all(hp.row_len <= 37 // 2)


def test_plan_rejects_non_binary_and_oversize():
    dup = scipy.sparse.coo_matrix((np.ones(3), ([0, 0, 1], [1, 1, 0])), shape=(2, 3))
    with pytest.raises(ValueError):
        build_host_plan(dup)
    with pytest.raises(ValueError):
        build_host_plan(scipy.sparse.coo_matrix((1, 70000)))
    # explicit zeros are tolerated (they are absences)
    z = scipy.sparse.coo_matrix((np.array([1, 0, 1]), ([0, 0, 1], [0, 1, 2])), shape=(2, 3))
    assert build_host_plan(z).nnz == 2


def _mixed_matrix(n, seed=5, per_class=40):
    rng = np.random.RandomState(seed)
    dens = np.concatenate([np.full(per_class, d) for d in (0.004, 0.015, 0.03, 0.06, 0.12, 0.3, 0.5, 0.8, 0.97)])
    return (rng.random_sample((dens.size, n)) < dens[:, None]).astype(np.int64)


@pytest.mark.parametrize("threshold,perms_per_cta", [(0, 8), (24, 8), (64, 4), (2, 2), (100, 1)])
def test_plan_list_and_bitmap_rows(threshold, perms_per_cta):
    n = 700
    x = _mixed_matrix(n)
    hp = build_host_plan(scipy.sparse.coo_matrix(x), long_threshold=threshold, perms_per_cta=perms_per_cta)
    if threshold == 0:
        assert hp.n_long == 0
    else:
        assert hp.n_long > 0 and np.all(hp.row_len < threshold)
        assert hp.bits.shape[0] == hp.n_superblocks * n * 32 * hp.slice_words
    if threshold == 2:
        assert hp.n_rows == 0
    wavefronts = check_layout(hp)
    # random order gives ~2.5 (8 lanes per wavefront) .. ~3.5 (32 lanes per wavefront)
    assert (1.0 <= wavefronts < (1.8 if perms_per_cta >= 4 else 2.6)) or hp.n_rows == 0
    perms = draw_perms(3, n, 4)
    import oracle
    pan, core = oracle.pan_core_curves_minrank(scipy.sparse.coo_matrix(x), perms)
    assert np.array_equal(curves_from_plan(hp, perms), np.hstack([pan, core]).astype(np.int64))


@pytest.mark.parametrize("slice_words", [1, 2, 4])
def test_plan_bitmap_slices_of_1_2_4_words(slice_words):
    """Superblocks of 1,024 / 2,048 / 4,096 rows: several of them, the last one ragged."""
    x = _mixed_matrix(300, seed=11, per_class=700)
    coo = scipy.sparse.coo_matrix(x)
    hp = build_host_plan(coo, long_threshold=4, slice_words=slice_words)
    assert hp.slice_words == slice_words and hp.n_long > 4096
    assert hp.n_superblocks == -(-hp.n_long // (1024 * slice_words))
    assert hp.bits.shape[0] == hp.n_superblocks * 300 * 32 * slice_words
    perms = draw_perms(7, 300, 2)
    import oracle
    pan, core = oracle.pan_core_curves_minrank(coo, perms)
    assert np.array_equal(curves_from_plan(hp, perms), np.hstack([pan, core]).astype(np.int64))
    with pytest.raises(ValueError):
        build_host_plan(coo, slice_words=3)


@pytest.mark.parametrize("perms_per_cta", [8, 4, 2])
def test_plan_native_bank_order_equals_specification(perms_per_cta):
    """The library's bank ordering (C++, threaded) must reproduce plan_np._bank_ordered_chunks bit for bit:
    the colouring for short rows, the positional order for long ones, pads, ragged sub-blocks."""
    x = _mixed_matrix(1300, seed=31, per_class=90)
    coo = scipy.sparse.coo_matrix(x)
    native = build_host_plan(coo, long_threshold=0, perms_per_cta=perms_per_cta)
    spec = plan_np.build_host_plan(coo, long_threshold=0, perms_per_cta=perms_per_cta)
    assert (native.tasks[:, 1] & 0xFFFF).max() > 32 > (native.tasks[:, 1] & 0xFFFF).min()      # both orderings in play
    assert np.array_equal(native.chunks, spec.chunks)
    assert np.array_equal(native.tasks, spec.tasks)
    for w in (1, 2, 4):
        a = build_host_plan(coo, long_threshold=5, slice_words=w)
        b = plan_np.build_host_plan(coo, long_threshold=5, slice_words=w)
        assert a.n_long > 0 and np.array_equal(a.bits, b.bits) and np.array_equal(a.chunks, b.chunks)


def test_plan_bank_order_beats_sorted_order():
    x = _mixed_matrix(4000, seed=9, per_class=64)
    hp = build_host_plan(scipy.sparse.coo_matrix(x), long_threshold=0, perms_per_cta=8)
    assert check_layout(hp) < 1.6


def test_plan_random_tables_property():
    """Property test (hypothesis): for random binary tables, thresholds, batch sizes and slice widths the
    device layout, walked like the kernels walk it, gives the curves of the min-rank oracle; and the
    curves obey the invariants SURVEY.md section 4 lists."""
    import oracle
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=60, deadline=None)
    @given(n=st.integers(1, 70), g=st.integers(0, 160), seed=st.integers(0, 10 ** 6),
           threshold=st.sampled_from([0, 2, 3, 5, 9, 17, 40]), perms_per_cta=st.sampled_from([1, 2, 4, 8]),
           slice_words=st.sampled_from([1, 2, 4]), style=st.sampled_from(["mixed", "sparse", "dense", "half"]))
    def check(n, g, seed, threshold, perms_per_cta, slice_words, style):
        rng = np.random.RandomState(seed)
        dens = {"mixed": rng.choice([0.0, 0.03, 0.1, 0.3, 0.5, 0.8, 0.97, 1.0], size=g),
                "sparse": rng.uniform(0.0, 0.1, size=g), "dense": rng.uniform(0.9, 1.0, size=g),
                "half": np.full(g, 0.5)}[style]
        x = (rng.random_sample((g, n)) < dens[:, None]).astype(np.int64)
        coo = scipy.sparse.coo_matrix(x)
        hp = build_host_plan(coo, long_threshold=threshold, perms_per_cta=perms_per_cta, slice_words=slice_words)
        assert hp.n_rows + hp.n_long + hp.n_empty + hp.n_full + hp.w_present.sum() + hp.w_absent.sum() == g
        check_layout(hp)
        perms = np.stack([rng.permutation(n) for _ in range(3)])
        got = curves_from_plan(hp, perms)
        pan, core = oracle.pan_core_curves_minrank(coo, perms)
        assert np.array_equal(got, np.hstack([pan, core]).astype(np.int64))
        counts = x.sum(axis=1)
        assert np.all(np.diff(got[:, :n], axis=1) >= 0) and np.all(np.diff(got[:, n:], axis=1) <= 0)
        assert np.array_equal(got[:, 0], got[:, n])
        assert np.all(got[:, n - 1] == np.count_nonzero(counts)) and np.all(got[:, 2 * n - 1] == np.count_nonzero(counts == n))

    check()


def _plans_equal(a, b):
    for f in ("colsum", "w_present", "w_absent", "chunks", "tasks", "sorted_idx", "sorted_ptr", "row_gene",
              "row_len", "row_absent", "bits", "long_gene"):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    for f in ("n_genes", "n_genomes", "nnz", "n_empty", "n_full", "nnz_list", "nnz_long", "slice_words"):
        assert getattr(a, f) == getattr(b, f), f


@pytest.mark.parametrize("order", ["column-major", "row-major", "shuffled"])
@pytest.mark.parametrize("shape", [(360, 700), (5000, 90), (70000, 12)])
def test_plan_native_ingest_equals_scipy_specification(order, shape):
    """The library's table ingest, folded lists and missing genomes (threaded C++) against the scipy +
    numpy specification of the same steps: whatever the order of the COO entries, the whole plan is identical.
    70,000 genes make the counting sort use blocks of 256 genes; (5000, 90) holds single-absence rows."""
    g, n = shape
    rng = np.random.RandomState(g + n)
    dens = rng.choice([0.0, 0.01, 0.05, 0.3, 0.6, 0.95, 0.99, 1.0], size=g)
    x = rng.random_sample((g, n)) < dens[:, None]
    row, col = np.nonzero(x.T)[::-1] if order == "column-major" else np.nonzero(x)
    if order == "shuffled":
        p = rng.permutation(row.shape[0])
        row, col = row[p], col[p]
    coo = scipy.sparse.coo_matrix((np.ones(row.shape[0], dtype=np.int64), (row, col)), shape=shape)
    native = build_host_plan(coo, long_threshold=9)
    spec = plan_np.build_host_plan(coo, long_threshold=9)
    _plans_equal(native, spec)
    assert native.w_absent.sum() > 0 or n > 100
    # float ones take the same path, CSR input is made canonical first: same plan
    _plans_equal(build_host_plan(coo.astype(np.float64), long_threshold=9), spec)
    _plans_equal(build_host_plan(coo.tocsr(), long_threshold=9), spec)


def test_plan_native_ingest_errors_and_corner_cases():
    import ctypes
    from pangenomix_b200 import _native
    lib = _native.load()

    def call(row, col, g, n):
        row, col = np.asarray(row, dtype=np.int32), np.asarray(col, dtype=np.int32)
        out = ctypes.POINTER(_native.PgxHostPlan)()
        rc = lib.pgx_host_plan_create(row.ctypes.data, col.ctypes.data, row.size, g, n, -1, 0, 0, ctypes.byref(out))
        if rc == 0:
            lib.pgx_host_plan_destroy(out)
        return rc

    hp = build_host_plan(scipy.sparse.coo_matrix((np.ones(4, dtype=np.int64), ([2, 0, 2, 0], [1, 3, 0, 2])), shape=(4, 5)))
    assert hp.c_owner is not None and hp.colsum.tolist() == [1, 1, 1, 1, 0] and hp.n_empty == 2
    lists = {int(g): hp.sorted_idx[hp.sorted_ptr[r]:hp.sorted_ptr[r + 1]].tolist() for r, g in enumerate(hp.row_gene)}
    assert lists == {0: [2, 3], 2: [0, 1]}
    assert call([0, 0, 1], [1, 1, 0], 2, 3) == 1                  # a duplicate pair: PGX_ERR_INVALID
    assert call([0, 2], [0, 0], 2, 3) != 0 and b"gene index" in lib.pgx_last_error()
    assert call([0, -1], [0, 0], 2, 3) != 0
    assert call([0, 1], [0, 3], 2, 3) != 0 and b"genome index" in lib.pgx_last_error()
    assert call([], [], 3, 2) == 0
    # the Python front end: duplicates are summed to 2 -> rejected, zeros are absences
    with pytest.raises(ValueError):
        build_host_plan(scipy.sparse.coo_matrix((np.ones(3), ([0, 0, 1], [1, 1, 0])), shape=(2, 3)))
    hp = build_host_plan(scipy.sparse.coo_matrix((np.array([1, 0, 1]), ([0, 0, 1], [0, 1, 2])), shape=(2, 3)))
    assert (hp.n_genes, hp.n_genomes, hp.nnz) == (2, 3, 2)
    assert hp.colsum.tolist() == [1, 0, 1] and hp.w_present.tolist() == [1, 0, 1]


def _input_formats(coo):
    x = coo.toarray()
    zeros = scipy.sparse.coo_matrix((np.concatenate([coo.data, np.zeros(5, dtype=coo.data.dtype)]),
                                     (np.concatenate([coo.row, np.arange(5)]), np.concatenate([coo.col, np.full(5, 7)]))),
                                    shape=coo.shape)
    assert zeros.nnz == coo.nnz + 5 and not np.any(x[np.arange(5), 7])
    return {"int64": coo.astype(np.int64), "float64": coo.astype(np.float64), "bool": coo.astype(bool),
            "explicit-zeros": zeros, "csr": coo.tocsr(), "csc": coo.tocsc(), "dense": x,
            "no-entries": scipy.sparse.coo_matrix(coo.shape, dtype=np.int64)}


@pytest.mark.parametrize("fmt", ["int64", "float64", "bool", "explicit-zeros", "csr", "csc", "dense", "no-entries"])
def test_every_input_format_is_planned_by_the_library(fmt):
    """Whatever form the table comes in, the plan is the library's own (c_owner set) and equals the
    specification array by array."""
    coo = scipy.sparse.coo_matrix(_mixed_matrix(300, seed=17, per_class=30))
    data = _input_formats(coo)[fmt]
    hp = build_host_plan(data, long_threshold=12)
    assert hp.c_owner is not None
    spec = plan_np.build_host_plan(data, long_threshold=12)
    _plans_equal(hp, spec)
    if fmt == "no-entries":
        assert hp.n_empty == coo.shape[0]
    else:
        assert hp.nnz == coo.nnz and hp.n_rows > 0 and hp.n_long > 0


def test_plan_row_balance_lowers_bank_conflicts(monkeypatch):
    """Rows are grouped so that the bank residues of a wavefront group are balanced (plan_np._balanced_row_order):
    same rows, same curves, fewer shared-memory wavefronts per gather step than with rows sorted by length;
    the library and the numpy specification agree on the order."""
    import oracle
    from pangenomix_b200 import synth
    coo = synth.bernoulli_matrix(6000, 1500, 450, seed=3)          # thousands of short rows, hundreds per class
    balanced = build_host_plan(coo, long_threshold=100, perms_per_cta=8)
    monkeypatch.setenv("PGX_NO_ROW_BALANCE", "1")
    by_length = build_host_plan(coo, long_threshold=100, perms_per_cta=8)
    monkeypatch.delenv("PGX_NO_ROW_BALANCE")
    assert sorted(balanced.row_gene.tolist()) == sorted(by_length.row_gene.tolist())
    assert np.array_equal(balanced.tasks[:, [0, 1, 3]], by_length.tasks[:, [0, 1, 3]])      # same sub-blocks, other rows in them
    w_bal, w_len = check_layout(balanced), check_layout(by_length)
    assert w_bal < w_len - 0.08 and w_bal < 1.06
    perms = draw_perms(5, 1500, 2)
    pan, core = oracle.pan_core_curves_minrank(coo, perms)
    assert np.array_equal(curves_from_plan(balanced, perms), np.hstack([pan, core]).astype(np.int64))
    spec = plan_np.build_host_plan(coo, long_threshold=100, perms_per_cta=8)
    _plans_equal(balanced, spec)
    # wide wavefront groups (16 and 32 lanes) and a window larger than a class
    for b in (4, 2):
        a = build_host_plan(coo, long_threshold=30, perms_per_cta=b)
        c = plan_np.build_host_plan(coo, long_threshold=30, perms_per_cta=b)
        _plans_equal(a, c)
        check_layout(a)


def test_plan_wide_table_two_permutations_per_cta_with_row_balance():
    """A C5-like width (50,000 genomes: 2 permutations per CTA, 32-lane wavefront groups, bitmap rows and list
    rows side by side) through the library's planner with the residue-balanced row order: the layout
    invariants hold and the emulated kernels reproduce the oracle's curves."""
    from oracle import cport
    from pangenomix_b200 import synth
    coo = synth.bernoulli_matrix(6000, 50000, 160, seed=11)
    hp = build_host_plan(coo)
    assert hp.perms_per_cta == 2 and hp.n_rows > 1000 and hp.n_long > 1000
    assert check_layout(hp) < 1.2                       # wavefronts per gather step (1.38 for rows sorted by length on C5)
    rng = np.random.RandomState(3)
    perms = np.stack([rng.permutation(50000) for _ in range(2)])
    pan, core = cport.curves_direct(coo, perms.astype(np.int32), n_threads=2)
    assert np.array_equal(curves_from_plan(hp, perms), np.hstack([pan, core]).astype(np.int64))


@pytest.mark.parametrize("name", ["c1", "c2"])
def test_library_planner_equals_specification(name):
    """The library's own planner (pgx_host_plan_create, what a C host gets) and the numpy / scipy specification
    (oracle/plan_np.py): the same plan, array by array, on configs C1 and C2."""
    from conftest import config_matrix_cached
    from pangenomix_b200 import synth
    coo = synth.config_matrix("c1") if name == "c1" else config_matrix_cached("c2")
    library = build_host_plan(coo)
    assert library.c_owner is not None and library.n_long > 0 and library.n_rows > 0
    spec = plan_np.build_host_plan(coo)
    assert spec.c_owner is None
    _plans_equal(library, spec)
    for f in ("n_empty", "n_full", "nnz", "nnz_list", "nnz_long", "long_threshold", "perms_per_cta", "slice_words"):
        assert getattr(library, f) == getattr(spec, f), f
    assert np.array_equal(library.row_gene, spec.row_gene) and np.array_equal(library.long_gene, spec.long_gene)
    assert np.array_equal(library.row_len, spec.row_len) and np.array_equal(library.row_absent, spec.row_absent)


def test_library_planner_options_and_errors():
    x = _mixed_matrix(900, seed=2, per_class=60)
    coo = scipy.sparse.coo_matrix(x)
    lists_only = build_host_plan(coo, long_threshold=0)
    assert lists_only.c_owner is not None and lists_only.n_long == 0 and lists_only.bits.size == 0
    assert build_host_plan(coo).long_threshold == 38             # round(1.28 sqrt(900)), as the specification
    with pytest.raises(ValueError):
        build_host_plan(coo, perms_per_cta=3)
    with pytest.raises(ValueError):
        build_host_plan(coo, slice_words=3)
    bad = scipy.sparse.coo_matrix((np.ones(2, dtype=np.int64), ([0, 1], [0, 0])), shape=(3, 2))
    bad.row[1] = 5                                              # gene index outside the table
    with pytest.raises(ValueError):
        build_host_plan(bad)
