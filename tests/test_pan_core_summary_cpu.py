"""CPU checks of the seeded on-device rarefaction path: the numpy restatement of the permutation recipe
(oracle/perm_np.py) -- Philox known answers, permutations, index addressing, exact uniformity -- the host
statistics of the integer moments, the gloo sharding of the summary, and argument checks of the new C entry
points (which fail before any CUDA call)."""
import os
import socket
import sys

import numpy as np
import pandas as pd
import pytest
import scipy.stats
import torch.multiprocessing as mp

from conftest import REPO, load_golden
from oracle import pan_core_curves_minrank
from oracle import perm_np
from pangenomix_b200 import _native, engine, pangenome_analysis


@pytest.mark.parametrize("counter,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(counter, key, want):
    got = perm_np.philox4x32_10(*counter, *key)
    assert tuple(int(w) for w in got) == want


def test_bucket_count():
    assert [perm_np.n_buckets(n) for n in (1, 2, 3, 4, 5, 8, 9, 50, 10000, 65503)] == \
        [1, 1, 2, 2, 2, 4, 4, 16, 4096, 16384]


@pytest.mark.parametrize("n", [1, 2, 3, 4, 31, 50, 400, 4097])
def test_oracle_rows_are_permutations(n):
    perms = perm_np.random_perms(12345, 7, 64, n)
    assert perms.dtype == np.uint16 and perms.shape == (64, n)
    assert np.array_equal(np.sort(perms, axis=1), np.broadcast_to(np.arange(n), (64, n)))


@pytest.mark.parametrize("seed", [0, 3, 2 ** 63 + 11])
def test_rows_are_addressed_by_global_index(seed):
    whole = perm_np.random_perms(seed, 0, 40, 57)
    for a, b in ((0, 40), (5, 17), (39, 40), (12, 12)):
        assert np.array_equal(perm_np.random_perms(seed, a, b - a, 57), whole[a:b])
    far = perm_np.random_perms(seed, 2 ** 40 - 3, 6, 57)
    assert np.array_equal(perm_np.random_perms(seed, 2 ** 40, 3, 57), far[3:])
    assert not np.array_equal(perm_np.random_perms(seed + 1, 0, 40, 57), whole)


def test_all_orders_of_four_are_equally_likely():
    perms = perm_np.random_perms(2024, 0, 240000, 4).astype(np.int64)
    code = ((perms[:, 0] * 4 + perms[:, 1]) * 4 + perms[:, 2]) * 4 + perms[:, 3]
    _, counts = np.unique(code, return_counts=True)
    assert counts.size == 24
    assert scipy.stats.chisquare(counts).pvalue > 1e-3


def test_position_marginals_are_uniform():
    n, draws = 50, 20000
    perms = perm_np.random_perms(99, 0, draws, n).astype(np.int64)
    table = np.zeros((n, n), dtype=np.int64)
    np.add.at(table, (np.broadcast_to(np.arange(n), perms.shape).ravel(), perms.ravel()), 1)
    assert np.all(table.sum(axis=0) == draws) and np.all(table.sum(axis=1) == draws)
    expected = draws / n
    stat = ((table - expected) ** 2 / expected).sum()
    assert scipy.stats.chi2.sf(stat, (n - 1) ** 2) > 1e-3


def _oracle_curves(coo, seed, first, count):
    perms = perm_np.random_perms(seed, first, count, coo.shape[1])
    pan, core = pan_core_curves_minrank(coo, perms.astype(np.int64))
    return np.hstack([pan, core]).astype(np.int32)


def _golden_coo(name="synth_800x50_s0"):
    import scipy.sparse
    g = load_golden(name)
    return scipy.sparse.coo_matrix((g["data"], (g["row"], g["col"])), shape=tuple(g["shape"]))


def _labels(n):
    return ["Pan%d" % (i + 1) for i in range(n)] + ["Core%d" % (i + 1) for i in range(n)]


@pytest.mark.parametrize("num_iter", [1, 2, 300])
def test_moments_give_pandas_statistics(num_iter):
    coo = _golden_coo()
    n = coo.shape[1]
    curves = _oracle_curves(coo, 5, 0, num_iter)
    m = engine.CurveMoments(num_iter, *perm_np.curve_moments(curves))
    got = pangenome_analysis.summary_frame(m, n)
    full = pd.DataFrame(curves.astype(np.float64), columns=_labels(n))
    want = full.agg(['mean', 'std', 'min', 'max'])
    assert list(got.index) == ['mean', 'std', 'min', 'max'] and list(got.columns) == _labels(n)
    assert got.values.dtype == np.float64
    for row in ('mean', 'min', 'max'):
        assert np.array_equal(got.loc[row].values, want.loc[row].values), row
    from pangenomix_b200 import plot
    assert np.array_equal(got.loc[['mean']].values, plot.calculate_mean(full).values)
    if num_iter == 1:
        assert np.all(np.isnan(got.loc['std'].values))
        return
    s_got, s_want = got.loc['std'].values, want.loc['std'].values
    constant = curves.min(axis=0) == curves.max(axis=0)
    assert np.all(s_got[constant] == 0.0)
    np.testing.assert_allclose(s_got, s_want, rtol=1e-12, atol=0)


def test_std_of_large_values_is_exact():
    """Large values with a spread of one, as far as the moment bound allows (n * max^2 < 2^63): the host
    statistics of the exact moments are the correctly rounded ddof=1 standard deviation."""
    from fractions import Fraction
    rng = np.random.RandomState(1)
    block = (3 * 10 ** 7 - rng.randint(0, 2, size=(1000, 6))).astype(np.int32)
    engine.check_moment_bound(1000, 3 * 10 ** 7)
    m = engine.CurveMoments(1000, *perm_np.curve_moments(block))
    got = pangenome_analysis.summary_frame(m, 3)
    for c in range(6):
        col = [int(v) for v in block[:, c]]
        mean = Fraction(sum(col), 1000)
        var = sum((v - mean) ** 2 for v in col) / 999
        assert got.loc['std'].values[c] == np.sqrt(float(var))


def test_moment_bound_is_enforced():
    engine.check_moment_bound(2 ** 20, 2 ** 21)
    with pytest.raises(ValueError):
        engine.check_moment_bound(2 ** 21, 2 ** 21)
    with pytest.raises(ValueError):
        pangenome_analysis.estimate_pan_core_summary(None, 0)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, num_iter, seed, dst, result_dir):
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import numpy as np
    import scipy.sparse
    import torch.distributed as dist
    from oracle import pan_core_curves_minrank, perm_np
    from pangenomix_b200 import distributed as pd_, sparse_utils as su
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = dict(np.load(os.path.join(REPO, "tests", "golden", "synth_800x50_s0.npz")))
    coo = scipy.sparse.coo_matrix((g["data"], (g["row"], g["col"])), shape=tuple(g["shape"]))
    lsdf = su.LightSparseDataFrame(["T_C%d" % i for i in range(800)], ["genome%d" % i for i in range(50)], coo)
    calls = []

    def compute(first, count):
        calls.append((first, count))
        perms = perm_np.random_perms(seed, first, count, 50)
        pan, core = pan_core_curves_minrank(coo, perms.astype(np.int64))
        return perm_np.curve_moments(np.hstack([pan, core]).astype(np.int32))

    state = np.random.get_state()
    df = pd_.estimate_pan_core_summary_sharded(lsdf, num_iter, seed=seed, dst=dst, compute=compute)
    after = np.random.get_state()
    assert np.array_equal(state[1], after[1]) and state[2] == after[2]
    lo, hi = pd_.shard_bounds(num_iter, world, rank)
    assert calls == ([(lo, hi - lo)] if hi > lo else [])
    if df is not None:
        np.save(os.path.join(result_dir, "r%d.npy" % rank), df.values)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,num_iter,dst", [(2, 37, None), (3, 40, 1), (3, 2, None)])
def test_sharded_summary_equals_single_process(tmp_path, world, num_iter, dst):
    seed = 2 ** 63 + 5
    coo = _golden_coo()
    m = engine.CurveMoments(num_iter, *perm_np.curve_moments(_oracle_curves(coo, seed, 0, num_iter)))
    want = pangenome_analysis.summary_frame(m, 50).values
    mp.spawn(_worker, args=(world, _free_port(), num_iter, seed, dst, str(tmp_path)), nprocs=world, join=True)
    receivers = range(world) if dst is None else [dst]
    for r in receivers:
        got = np.load(str(tmp_path / ("r%d.npy" % r)))
        assert np.array_equal(got, want, equal_nan=True)
    if dst is not None:
        assert sorted(os.listdir(str(tmp_path))) == ["r%d.npy" % dst]


def test_new_entry_points_reject_bad_arguments():
    lib = _native.load()
    buf = np.zeros(64, dtype=np.int64)
    p = buf.ctypes.data
    for args, text in [((1, 0, 4, 10, None, None), b"null"),
                       ((1, 0, 4, 0, p, None), b"65503"),
                       ((1, 0, 4, 65504, p, None), b"65503"),
                       ((1, 0, -1, 10, p, None), b"n_perm"),
                       ((1, -1, 4, 10, p, None), b"first")]:
        assert lib.pgx_random_perms(*args) == 1
        assert text in lib.pgx_last_error()
    for args, text in [((p, 4, 8, None, p, p, p, 0, None), b"null"),
                       ((None, 4, 8, p, p, p, p, 0, None), b"null"),
                       ((p, -1, 8, p, p, p, p, 0, None), b"negative"),
                       ((p, 4, 7, p, p, p, p, 0, None), b"even")]:
        assert lib.pgx_curve_moments(*args) == 1
        assert text in lib.pgx_last_error()
    with pytest.raises(_native.PgxError):
        _native.check(lib.pgx_random_perms(1, 0, 4, 0, p, None))
