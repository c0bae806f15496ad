"""The seeded on-device rarefaction path on the GPU: pgx_random_perms against its numpy restatement bit for bit,
estimate_pan_core_summary against pandas statistics of the full curve table of the same genome orders, block and
rank splits that must not change the result, and the Heaps fit of the mean row."""
import contextlib
import io
import os
import socket
import sys

import numpy as np
import pandas as pd
import pytest
import scipy.sparse

from conftest import REPO, config_matrix_cached, golden_matrix
from oracle import perm_np

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")
    return torch


def _lsdf(coo):
    from pangenomix_b200 import sparse_utils as su, synth
    index, columns = synth.labels_for(*coo.shape)
    return su.LightSparseDataFrame(index, columns, coo)


@pytest.mark.parametrize("first", [0, 12345, 2 ** 40])
@pytest.mark.parametrize("seed", [0, 77, 2 ** 63 + 12345])
@pytest.mark.parametrize("n", [1, 2, 3, 31, 50, 400, 4097, 10000, 65503])
def test_device_permutations_equal_the_oracle(torch_cuda, n, seed, first):
    from pangenomix_b200 import engine
    count = 48 if n <= 4097 else 6 if n <= 10000 else 2
    got = engine.random_permutations_device(n, count, seed, first=first)
    assert got.dtype == torch_cuda.int16 and tuple(got.shape) == (count, n)
    assert np.array_equal(got.cpu().numpy().view(np.uint16), perm_np.random_perms(seed, first, count, n))


def test_device_permutations_into_unaligned_rows(torch_cuda):
    """Rows written through an output that starts off a 16-byte boundary (the head / tail stores)."""
    from pangenomix_b200 import engine
    buf = torch_cuda.zeros(5 * 333 + 3, dtype=torch_cuda.int16, device="cuda")
    view = buf[3:].view(5, 333)
    engine.random_permutations_device(333, 5, 9, first=4, out=view)
    assert np.array_equal(view.cpu().numpy().view(np.uint16), perm_np.random_perms(9, 4, 5, 333))
    assert int(buf[:3].abs().sum()) == 0


def _pandas_stats(eng, num_iter, seed, torch):
    from pangenomix_b200 import engine
    n = eng.n_genomes
    curves = eng.curves_device(engine.random_permutations_device(n, num_iter, seed, device=eng.device)).cpu().numpy()
    cols = ["Pan%d" % (i + 1) for i in range(n)] + ["Core%d" % (i + 1) for i in range(n)]
    return pd.DataFrame(curves.astype(np.float64), columns=cols)


def _int32_bins_table():
    rng = np.random.RandomState(7)
    dens = np.concatenate([np.full(68000, 0.985), rng.uniform(0.0, 1.0, size=4000)])
    return scipy.sparse.coo_matrix((rng.random_sample((dens.size, 48)) < dens[:, None]).astype(np.int64))


@pytest.mark.parametrize("case,num_iter", [("synth_800x50_s0", 1000), ("c1_8000x50", 100), ("c2", 1000),
                                           ("c4", 2000), ("int32_bins", 300), ("n65503", 40)])
def test_summary_equals_pandas_statistics(torch_cuda, case, num_iter):
    from pangenomix_b200 import pangenome_analysis as pa, plot, synth
    if case in ("c2", "c4"):
        coo = config_matrix_cached(case)
    elif case == "int32_bins":
        coo = _int32_bins_table()
    elif case == "n65503":
        coo = synth.bernoulli_matrix(3000, 65503, 150, seed=5).tocoo()
    else:
        coo = golden_matrix(case)
    lsdf = _lsdf(coo)
    seed = 2024
    got = pa.estimate_pan_core_summary(lsdf, num_iter, seed=seed)
    eng = pa._engine_for(lsdf)
    if case == "int32_bins":
        assert eng.c_plan.max_colsum > 65535
    full = _pandas_stats(eng, num_iter, seed, torch_cuda)
    want = full.agg(['mean', 'std', 'min', 'max'])
    assert list(got.index) == ['mean', 'std', 'min', 'max'] and list(got.columns) == list(full.columns)
    for row in ('mean', 'min', 'max'):
        assert np.array_equal(got.loc[row].values, want.loc[row].values), row
    assert np.array_equal(got.loc[['mean']].values, plot.calculate_mean(full).values)
    s_got = got.loc['std'].values
    constant = want.loc['min'].values == want.loc['max'].values
    assert np.all(s_got[constant] == 0.0)
    np.testing.assert_allclose(s_got, want.loc['std'].values, rtol=1e-12, atol=0)


def test_block_and_offset_splits_do_not_change_the_moments(torch_cuda):
    from pangenomix_b200 import engine
    eng = engine.PanCoreEngine(golden_matrix("synth_800x50_s0"))
    whole = eng.summary(1000, 31, block=1000)
    for block in (1, 37, 999, None):
        part = eng.summary(1000, 31, block=block)
        assert all(np.array_equal(a, b) for a, b in zip(whole[1:], part[1:])), block
    # [0, 1000) = [0, 400) + [400, 1000) combined on the host
    a, b = eng.summary(400, 31), eng.summary(600, 31, first=400)
    assert np.array_equal(a.sum + b.sum, whole.sum) and np.array_equal(a.sumsq + b.sumsq, whole.sumsq)
    assert np.array_equal(np.minimum(a.min, b.min), whole.min) and np.array_equal(np.maximum(a.max, b.max), whole.max)
    empty = eng.summary(0, 31)
    assert not empty.sum.any() and not empty.sumsq.any()
    assert np.all(empty.min == 2 ** 31 - 1) and np.all(empty.max == -2 ** 31)


def test_heaps_fit_of_the_mean_row(torch_cuda):
    import warnings
    from pangenomix_b200 import pangenome_analysis as pa, plot
    coo = golden_matrix("synth_800x50_s0")
    lsdf = _lsdf(coo)
    stats = pa.estimate_pan_core_summary(lsdf, 500, seed=8)
    full = _pandas_stats(pa._engine_for(lsdf), 500, 8, torch_cuda)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        got = pa.fit_heaps_by_iteration(stats.loc[['mean']])
        want = pa.fit_heaps_by_iteration(plot.calculate_mean(full))
    assert np.array_equal(got.values, want.values)
    got_gpu = pa.fit_heaps_by_iteration_gpu(stats.loc[['mean']])
    want_gpu = pa.fit_heaps_by_iteration_gpu(plot.calculate_mean(full))
    assert np.array_equal(got_gpu.values, want_gpu.values)
    np.testing.assert_allclose(got_gpu.values, got.values, rtol=5e-6)


def test_summary_leaves_numpy_rng_alone_and_prints_nothing(torch_cuda):
    from pangenomix_b200 import pangenome_analysis as pa
    lsdf = _lsdf(golden_matrix("synth_800x50_s0"))
    np.random.seed(4)
    np.random.random_sample(5)
    before = np.random.get_state()
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        one = pa.estimate_pan_core_summary(lsdf, 1, seed=3)
        pa.estimate_pan_core_summary(lsdf, 50)
    after = np.random.get_state()
    assert out.getvalue() == ""
    assert before[0] == after[0] and np.array_equal(before[1], after[1]) and before[2:] == after[2:]
    assert np.all(np.isnan(one.loc['std'].values))
    assert np.array_equal(one.loc['mean'].values, one.loc['min'].values)
    with pytest.raises(ValueError):
        pa.estimate_pan_core_summary(lsdf, 0)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, num_iter, dst, result_dir):
    sys.path.insert(0, REPO)
    import numpy as np
    import torch
    import torch.distributed as dist
    from pangenomix_b200 import distributed as pd_, pangenome_analysis as pa, sparse_utils as su, synth
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    coo = synth.bernoulli_matrix(20000, 1000, 2000, seed=11)
    lsdf = su.LightSparseDataFrame(*synth.labels_for(*coo.shape), coo)
    df = pd_.estimate_pan_core_summary_sharded(lsdf, num_iter, seed=2 ** 63 + 1, dst=dst)
    if rank == 0:
        np.save(os.path.join(result_dir, "want.npy"), pa.estimate_pan_core_summary(lsdf, num_iter, seed=2 ** 63 + 1).values)
    if df is not None:
        np.save(os.path.join(result_dir, "r%d.npy" % rank), df.values)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("num_iter,dst", [(3001, None), (640, 0), (1, None)])
def test_sharded_summary_equals_single_gpu(tmp_path, num_iter, dst):
    import torch
    import torch.multiprocessing as mp
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    world = min(torch.cuda.device_count(), 8)
    mp.spawn(_worker, args=(world, _free_port(), num_iter, dst, str(tmp_path)), nprocs=world, join=True)
    want = np.load(str(tmp_path / "want.npy"))
    for r in (range(world) if dst is None else [dst]):
        assert np.array_equal(np.load(str(tmp_path / ("r%d.npy" % r))), want, equal_nan=True)
    if dst is not None:
        assert not os.path.exists(str(tmp_path / "r1.npy"))
