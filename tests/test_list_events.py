"""The mex events of the list kernel (csrc/pgx_rarefy.cu, list_kernel, queue_events).

A list row whose minimum under a permutation is 0 holds that permutation's rank-0 genome; its statistic is the mex of
the list's ranks instead, an event queued per warp and resolved 32 at a time.  The end of a sub-block queues all its
events with one exclusive scan over the warp, in rounds when they outnumber the queue: a sub-block of 32 rows that
all hold the rank-0 genome of all 8 permutations of a batch brings 256 events at once.

The table puts genome 0 into every row of its first 1,600 present lists and of its 96 absent lists, and the orders
of the first batch all start with genome 0.  Further orders fill batches of 1 to 7 valid permutations.  Every curve is
compared bit for bit with oracle.pan_core_curves_minrank, an exact integer reference.
"""
import numpy as np
import pytest
import scipy.sparse

from test_int32_bins import _device_perms, oracle_curves
from test_rarefy_paths import _tuned

N = 300
ALL_ZERO_ROWS = 1600            # present lists with genome 0: 50 full sub-blocks of 32 rows
OTHER_ROWS = 700                # present lists without genome 0
ABSENT_ROWS = 96                # absent lists with genome 0
LONG_ROWS = 64                  # bitmap rows, so that the probe kernel adds into the same histograms


@pytest.fixture(scope="module")
def engine_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")
    from pangenomix_b200 import _native, engine
    _native.load()
    yield engine
    _native.set_tuning(0, 0, 0)


def event_table(seed=0):
    rng = np.random.RandomState(seed)
    rows, cols = [], []

    def add(genomes):
        rows.append(np.full(len(genomes), len(rows)))
        cols.append(np.asarray(genomes))

    for _ in range(ALL_ZERO_ROWS):
        add(np.r_[0, 1 + rng.choice(N - 1, rng.randint(1, 9), replace=False)])
    for _ in range(OTHER_ROWS):
        add(1 + rng.choice(N - 1, rng.randint(2, 10), replace=False))
    for _ in range(ABSENT_ROWS):
        add(np.setdiff1d(np.arange(N), np.r_[0, 1 + rng.choice(N - 1, rng.randint(1, 6), replace=False)]))
    for _ in range(LONG_ROWS):
        add(np.flatnonzero(rng.rand(N) < 0.5))
    r, c = np.concatenate(rows), np.concatenate(cols)
    return scipy.sparse.coo_matrix((np.ones(r.size, dtype=np.int64), (r, c)), shape=(len(rows), N))


def orders(n_perm, seed):
    """n_perm genome orders; the first 8 start with genome 0."""
    rng = np.random.RandomState(seed)
    out = np.empty((n_perm, N), dtype=np.uint16)
    for i in range(n_perm):
        out[i] = rng.permutation(N)
        if i < 8:
            out[i] = np.r_[0, rng.permutation(np.arange(1, N))]
    return out


def test_event_table_plans_to_list_rows():
    from pangenomix_b200.plan import build_host_plan
    coo = event_table()
    hp = build_host_plan(coo)
    assert hp.perms_per_cta == 8 and hp.n_long == LONG_ROWS
    assert hp.row_absent.sum() == ABSENT_ROWS and (~hp.row_absent).sum() == ALL_ZERO_ROWS + OTHER_ROWS
    # every list row with genome 0 has min 0 under the first 8 orders: 1,696 x 8 events in the first batch
    csr = coo.tocsr()
    with_zero = np.asarray(csr[:, 0].todense()).ravel() > 0
    assert with_zero[:ALL_ZERO_ROWS].all() and not with_zero[ALL_ZERO_ROWS:ALL_ZERO_ROWS + OTHER_ROWS].any()
    assert not with_zero[ALL_ZERO_ROWS + OTHER_ROWS:ALL_ZERO_ROWS + OTHER_ROWS + ABSENT_ROWS].any()
    assert (orders(13, 1)[:8, 0] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("n_perm", [8, 9, 10, 11, 12, 13, 14, 15, 16])
def test_full_event_sub_blocks_and_partial_batches(engine_mod, n_perm):
    coo = event_table()
    eng = engine_mod.PanCoreEngine(coo)
    assert eng.c_plan.max_colsum <= 65535
    perms = orders(n_perm, n_perm)
    want = oracle_curves(coo, perms)
    d_perms = _device_perms(perms)
    for splits in (1, 3):
        got = _tuned((8, splits, 0), lambda: eng.curves_device(d_perms).cpu().numpy())
        assert np.array_equal(got, want), splits
    assert np.array_equal(eng.curves_host(perms), want)
