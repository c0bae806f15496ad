"""Where the list kernel counts its row minima (csrc/pgx_rarefy.cu, list_kernel).

With packed uint16 bins a present-list sub-block stores its B minima to a scratch of one slot per CTA, and once an
item's gathers are done the CTA counts them in B pan-side histograms in the shared memory of its rank table, then adds
the non-zero words into the global rows.  Absent-list rows, the mex events and int32 bins keep their global REDs, and
so does a launch whose scratch (grid x list rows x B x 2 bytes) would exceed 1 GiB.

  * A bin of exactly 65,535 counted through the shared histograms at every batch size and two row splits: a half of a
    shared or a global word may fill to the brim, never carry into the other.
  * A table with enough list rows that 100 row splits push the scratch past 1 GiB (the launch keeps its global REDs),
    and the same table with 3 splits (a scratch far below it), on the C4-like launch shape: a rank table above 100 KB,
    one list CTA of 896 threads per SM, present- and absent-list rows in one call.

Every curve is compared bit for bit with oracle.pan_core_curves_minrank, an exact integer reference.
"""
import numpy as np
import pytest
import scipy.sparse

from conftest import draw_perms
from test_int32_bins import _device_perms, assert_heavy_steps, chosen_orders, engine_mod, heavy_table, oracle_curves  # noqa: F401
from test_rarefy_paths import _tuned

SCRATCH_MAX = 1 << 30           # csrc/pgx_rarefy.cu: MINIMA_SCRATCH_MAX
BIG_N = 6400                    # rank table of 8 permutations: (N + 32) x 16 bytes > 100 KB -> one CTA per SM
BIG_SPLITS = 100                # 9 permutations = 2 batches of 8: 200 items, a list CTA on every SM
STEPS = np.array([s for s in range(1, 400) if s % 2 and s % 5])     # coprime to BIG_N = 2^8 x 5^2


def big_rows(sm_count):
    """List rows that make the scratch of a launch with BIG_SPLITS splits exceed SCRATCH_MAX by 10 %: its grid holds
    min(2 x BIG_SPLITS, sm_count) CTAs of 8 permutations."""
    grid = min(2 * BIG_SPLITS, sm_count)
    return int(1.1 * SCRATCH_MAX / (grid * 8 * 2)) + 1


def big_table(rows, absent_rows=200, seed=0):
    """``rows`` present lists of 2 .. 8 genomes (s + k t mod N for k < length, t coprime to N: distinct), then
    ``absent_rows`` rows missing 2 .. 8 genomes and a universal row."""
    n = BIG_N
    rng = np.random.RandomState(seed)
    lengths = rng.randint(2, 9, rows)
    start, step = rng.randint(0, n, rows), rng.choice(STEPS, rows)
    k = np.arange(lengths.sum()) - np.repeat(np.cumsum(lengths) - lengths, lengths)
    row_ids = [np.repeat(np.arange(rows), lengths)]
    cols = [(np.repeat(start, lengths) + k * np.repeat(step, lengths)) % n]
    for i in range(absent_rows):
        keep = np.delete(np.arange(n), rng.choice(n, 2 + i % 7, replace=False))
        row_ids.append(np.full(keep.size, rows + i))
        cols.append(keep)
    row_ids.append(np.full(n, rows + absent_rows))
    cols.append(np.arange(n))
    r, c = np.concatenate(row_ids), np.concatenate(cols)
    return scipy.sparse.coo_matrix((np.ones(r.size, dtype=np.int64), (r, c)), shape=(rows + absent_rows + 1, n))


# ---------------------------------------------------------------------------------------------------------------
# CPU: the big table plans to what the GPU test needs
# ---------------------------------------------------------------------------------------------------------------
def test_big_table_plans_past_the_scratch_budget():
    from pangenomix_b200.plan import build_host_plan
    rows = big_rows(148)
    coo = big_table(rows)
    hp = build_host_plan(coo)
    assert hp.n_long == 0 and hp.n_rows == rows + 200 and hp.perms_per_cta == 8
    assert 0 < hp.colsum.max() <= 65535
    absent = hp.row_absent
    assert absent.sum() == 200 and (~absent).sum() == rows
    assert min(2 * BIG_SPLITS, 148) * 8 * 2 * hp.n_rows > SCRATCH_MAX              # 100 splits: global REDs
    assert min(2 * 3, 148) * 8 * 2 * hp.n_rows < SCRATCH_MAX // 10                 # 3 splits: shared-memory counts
    assert (BIG_N + 32) * 16 > 100 * 1024


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [64, 2200])
def test_a_bin_of_65535_at_every_batch_size_and_split(engine_mod, n):
    """heavy_table: genome h holds 65,535 genes, each in one partner genome too, all list rows.  Order A ([x, h, ...])
    puts all of them into pan bin 1 through the list kernel's counts, order B makes them 65,535 mex events."""
    coo = heavy_table(n, 65535, seed=n + 1)
    eng = engine_mod.PanCoreEngine(coo)
    assert eng.c_plan.max_colsum == 65535 and np.isin(np.arange(65535), eng.host_plan.row_gene).all()
    perms = np.r_[chosen_orders(n, n), draw_perms(n + 2, n, 5)].astype(np.uint16)       # 9: a partial batch for B > 1
    want = oracle_curves(coo, perms)
    assert_heavy_steps(want, n, 65535)
    d_perms = _device_perms(perms)
    for b in (1, 2, 4, 8):
        for splits in (1, 3):
            got = _tuned((b, splits, 0), lambda: eng.curves_device(d_perms).cpu().numpy())
            assert np.array_equal(got, want), (b, splits)
    assert np.array_equal(eng.curves_host(perms), want)


@pytest.mark.gpu
def test_scratch_budget_on_both_sides(engine_mod):
    from pangenomix_b200 import _native
    rows = big_rows(int(_native.device_info()["sm_count"]))
    coo = big_table(rows, seed=7)
    eng = engine_mod.PanCoreEngine(coo)
    hp = eng.host_plan
    assert hp.n_long == 0 and hp.perms_per_cta == 8 and 0 < eng.c_plan.max_colsum <= 65535
    perms = draw_perms(11, BIG_N, 9).astype(np.uint16)
    want = oracle_curves(coo, perms)
    d_perms = _device_perms(perms)
    for splits in (BIG_SPLITS, 3):
        got = _tuned((8, splits, 0), lambda: eng.curves_device(d_perms).cpu().numpy())
        assert np.array_equal(got, want), splits
    assert np.array_equal(eng.curves_host(perms), want)
