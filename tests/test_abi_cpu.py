"""CPU-side checks of the C-ABI library: it loads, exports everything include/pgx.h
declares, reports errors through pgx_last_error, and its host-only entry point
(pgx_legacy_shuffles) reproduces numpy's legacy stream.  No kernels are launched here."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import REPO, draw_perms
from pangenomix_b200 import _native, engine


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(REPO, "include", "pgx.h")).read()
    declared = set(re.findall(r"\b(pgx_[a-z0-9_]+)\s*\(", header))
    declared -= {"pgx_plan"}
    assert declared == set(_native.EXPORTS)
    lib = _native.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.pgx_version() == 321


def test_plan_struct_layout_matches_header():
    # 9 pointers + int64 + 10 int32 = 120 bytes, no padding surprises
    assert ctypes.sizeof(_native.PgxPlan) == 9 * 8 + 8 + 10 * 4
    assert _native.PgxPlan.max_colsum.offset == 9 * 8 + 8 + 8 * 4


def test_invalid_arguments_set_last_error():
    lib = _native.load()
    rc = lib.pgx_pan_core_curves(None, None, 1, None, None)
    assert rc == 1
    assert b"plan is null" in lib.pgx_last_error()
    plan = _native.PgxPlan(n_genomes=70000)
    rc = lib.pgx_pan_core_curves(ctypes.byref(plan), None, 1, None, None)
    assert rc == 3 and b"65503" in lib.pgx_last_error()
    with pytest.raises(_native.PgxError):
        _native.check(rc)
    assert lib.pgx_bernoulli_scratch_bytes(0, 5) == 0
    assert lib.pgx_bernoulli_scratch_bytes(4000, 400) >= 8 * (4000 + 400)


@pytest.mark.parametrize("n", [1, 2, 3, 5, 50, 255, 256, 257, 400, 4096, 10000, 65503, 65535])
def test_legacy_shuffles_are_numpys(n):
    count = 4 if n < 20000 else 2
    np.random.seed(12345)
    got = engine.draw_legacy_permutations(n, count)
    state_after = np.random.get_state()
    want = draw_perms(12345, n, count)
    assert np.array_equal(got, want)
    ref_state = np.random.get_state()
    assert np.array_equal(state_after[1], ref_state[1]) and state_after[2] == ref_state[2]
    # and the stream continues identically
    np.random.set_state(state_after)
    a = np.random.random_sample(3)
    np.random.set_state(ref_state)
    assert np.array_equal(a, np.random.random_sample(3))


@pytest.mark.parametrize("n,count", [(7, 5000), (64, 3000), (400, 2500), (10000, 120), (65503, 24)])
@pytest.mark.parametrize("mode", ["default", "avx2", "scalar", "one_thread", "seven_threads"])
def test_legacy_shuffles_vector_and_threaded_paths(monkeypatch, n, count, mode):
    """Long streams exercise the AVX2 acceptance spans, every mask boundary, MT19937 block
    boundaries inside a vector and the producer / worker-thread pipeline; all must equal numpy."""
    if mode == "avx2":
        monkeypatch.setenv("PGX_RNG_NO_AVX512", "1")
    elif mode == "scalar":
        monkeypatch.setenv("PGX_RNG_SCALAR", "1")
    elif mode == "one_thread":
        monkeypatch.setenv("PGX_RNG_THREADS", "0")
    elif mode == "seven_threads":
        monkeypatch.setenv("PGX_RNG_THREADS", "7")
    np.random.seed(2024)
    np.random.random_sample(77)
    start = np.random.get_state()
    got = engine.draw_legacy_permutations(n, count)
    after = np.random.get_state()
    np.random.set_state(start)
    want = np.empty((count, n), dtype=np.uint16)
    for i in range(count):
        a = np.arange(n)
        np.random.shuffle(a)
        want[i] = a
    ref_after = np.random.get_state()
    assert np.array_equal(got, want)
    assert np.array_equal(after[1], ref_after[1]) and after[2] == ref_after[2]


@pytest.mark.parametrize("n", [33, 1000, 10000])
def test_legacy_shuffles_calls_interleaved_with_numpy_draws(n):
    """Many short calls, numpy's own draws between them: calls end at every position of an MT19937 block,
    also inside a block tail that the AVX-512 span has carried in front of the next block (the exported
    state is then the previous block's key), and the state handed back must be numpy's every time."""
    sizes = [1 + (7 * k) % 5 for k in range(max(12, 120000 // n))]
    np.random.seed(31)
    got = []
    for c in sizes:
        got.append(engine.draw_legacy_permutations(n, c))
        np.random.random_sample(3)
    state = np.random.get_state()
    np.random.seed(31)
    for c, block in zip(sizes, got):
        for row in block:
            a = np.arange(n)
            np.random.shuffle(a)
            assert np.array_equal(a, row)
        np.random.random_sample(3)
    ref = np.random.get_state()
    assert np.array_equal(state[1], ref[1]) and state[2] == ref[2]


def test_legacy_shuffles_mid_block_state_and_numpy_mode(monkeypatch):
    np.random.seed(99)
    np.random.random_sample(123)           # leave the generator mid-block
    state = np.random.get_state()
    got = engine.draw_legacy_permutations(37, 5)
    np.random.set_state(state)
    monkeypatch.setenv("PGX_NUMPY_SHUFFLE", "1")
    assert np.array_equal(engine.draw_legacy_permutations(37, 5), got)


def test_no_cuda_means_loud_failure(have_cuda):
    if have_cuda:
        pytest.skip("CUDA present")
    import scipy.sparse
    with pytest.raises(_native.PgxError):
        engine.PanCoreEngine(scipy.sparse.coo_matrix(np.eye(4, dtype=np.int64)))
    with pytest.raises(_native.PgxError):
        engine.BernoulliGrid(np.eye(4))


@pytest.mark.parametrize("mode", ["", "PGX_RNG_NO_TAIL", "PGX_RNG_NO_AVX512"])
def test_legacy_shuffles_state_at_every_block_position(monkeypatch, mode):
    """Short calls started from every region of the MT19937 block: the permutations AND the exported state
    (key and position, as np.random.get_state() reports them) equal numpy's.  The vector steps read up to 32
    words ahead and carry block tails in front of the next block, so a call may end inside a carried tail or
    exactly at its end -- numpy is then still on the old block (position 624 - remaining, or 624)."""
    if mode:
        monkeypatch.setenv(mode, "1")
    for n in (33, 40, 47, 64, 65, 97, 100, 129, 400, 1000):
        for skip in range(0, 700, 7):
            np.random.seed(1000 + skip)
            if skip:
                np.random.randint(0, 2 ** 31 - 1, size=skip)          # moves the position inside the block
            start = np.random.get_state()
            count = 1 + skip % 3
            got = engine.draw_legacy_permutations(n, count)
            ours = np.random.get_state()
            np.random.set_state(start)
            for i in range(count):
                a = np.arange(n)
                np.random.shuffle(a)
                assert np.array_equal(a, got[i]), (n, skip, i)
            theirs = np.random.get_state()
            assert ours[2] == theirs[2] and np.array_equal(ours[1], theirs[1]), (n, skip, ours[2], theirs[2])


def test_legacy_shuffles_worker_pool_reuse_sleep_and_fork(monkeypatch):
    """The stage-3 workers are a persistent pool that spins between calls and sleeps after a few idle
    milliseconds: back-to-back calls with changing sizes and thread counts, pauses that put the workers to
    sleep, and a forked child (which has no threads and must start its own pool) all give numpy's stream."""
    import time
    rng = np.random.RandomState(5)
    for rep in range(40):
        n = int(rng.choice([64, 100, 400, 1000, 4097, 10000]))
        count = int(rng.randint(1, 300))
        monkeypatch.setenv("PGX_RNG_THREADS", str(int(rng.choice([0, 1, 2, 4, 7, 16, 40]))))
        seed = int(rng.randint(1 << 30))
        np.random.seed(seed)
        got = engine.draw_legacy_permutations(n, count)
        ours = np.random.get_state()
        assert np.array_equal(got, draw_perms(seed, n, count).astype(np.uint16))
        theirs = np.random.get_state()
        assert ours[2] == theirs[2] and np.array_equal(ours[1], theirs[1])
        if rep % 10 == 0:
            time.sleep(0.05)                     # > the 3 ms the workers spin before they sleep
    monkeypatch.setenv("PGX_RNG_THREADS", "4")
    np.random.seed(3)
    want = engine.draw_legacy_permutations(1000, 300)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", DeprecationWarning)
        pid = os.fork()
    if pid == 0:
        np.random.seed(3)
        os._exit(0 if np.array_equal(engine.draw_legacy_permutations(1000, 300), want) else 1)
    _, status = os.waitpid(pid, 0)
    assert os.WIFEXITED(status) and os.WEXITSTATUS(status) == 0


@pytest.mark.parametrize("n,rows,f64", [(1, 5, 0), (2, 3, 1), (7, 4, 0), (8, 9, 1), (9, 2, 0), (400, 33, 1), (10000, 17, 0), (10000, 5, 1)])
def test_expand_deltas_rebuilds_the_curves(n, rows, f64):
    """pgx_expand_deltas (the host half of the compact transfer) against numpy: steps -> curves."""
    rng = np.random.RandomState(n + rows)
    pan = np.cumsum(rng.randint(0, 4000, size=(rows, n)), axis=1).astype(np.int64)
    core = pan[:, :1] - np.concatenate((np.zeros((rows, 1), dtype=np.int64),
                                        np.cumsum(rng.randint(0, 3, size=(rows, max(n - 1, 0))), axis=1)), axis=1)
    steps = np.empty((rows, 2 * n), dtype=np.uint16)
    steps[:, :n] = np.diff(pan, axis=1, prepend=0)
    steps[:, n] = core[:, 0]
    steps[:, n + 1:] = -np.diff(core, axis=1)
    out = np.full((rows, 2 * n), -1, dtype=np.float64 if f64 else np.int32)
    for threads in (1, 3):
        out[:] = -1
        _native.check(_native.load().pgx_expand_deltas(steps.ctypes.data, rows, n, out.ctypes.data, f64, threads))
        assert np.array_equal(out, np.hstack([pan, core]).astype(out.dtype))
    # the largest step a table can have
    big = np.zeros((1, 2 * n), dtype=np.uint16)
    big[0, 0] = big[0, n] = 65535
    _native.check(_native.load().pgx_expand_deltas(big.ctypes.data, 1, n, out.ctypes.data, f64, 1))
    assert out[0, 0] == 65535 and out[0, n - 1] == 65535 and out[0, 2 * n - 1] == 65535


def _build_c_host(tmp_path):
    import subprocess
    exe = str(tmp_path / "abi_host")
    lib_dir = os.path.join(REPO, "pangenomix_b200")
    subprocess.run(["gcc", "-O2", "-I", os.path.join(REPO, "include"), os.path.join(REPO, "tests", "c", "abi_host.c"),
                    "-L", lib_dir, "-lpgx_b200", "-Wl,-rpath," + lib_dir, "-o", exe], check=True)
    return exe


def test_c_host_links_only_the_library_and_plans_a_table(tmp_path):
    """tests/c/abi_host.c: a plain C program against include/pgx.h and libpgx_b200.so alone (no Python in the loop)
    plans a table with pgx_host_plan_create; its GPU half runs in tests/test_gpu_parity.py."""
    import subprocess
    _native.load()
    exe = _build_c_host(tmp_path)
    out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    assert "host ok" in out and "bitmap rows" in out
    needed = subprocess.run(["ldd", exe], check=True, capture_output=True, text=True).stdout
    assert "libpgx_b200.so" in needed and "python" not in needed.lower() and "torch" not in needed.lower()


@pytest.mark.parametrize("n, head, rows", [(2048, 512, 37), (3001, 7, 11), (5, 5, 3), (9, 1, 4), (40, 39, 5), (10000, 512, 20)])
def test_split_rows_expand_to_the_curves(n, head, rows):
    """pgx_expand_split: uint16 heads + uint8 tails of the curves' steps -> int32 / float64 curves (the host half of
    the host-buffer calls on tables of many genomes), any thread count, aligned or not."""
    lib = _native.load()
    rng = np.random.RandomState(n + head)
    pan = rng.randint(0, 200, size=(rows, n))
    pan[:, :head] = rng.randint(0, 5000, size=(rows, head))
    core = rng.randint(0, 3, size=(rows, n))
    core[:, :head] = rng.randint(0, 300, size=(rows, head))
    core[:, 0] = 60000
    want = np.hstack([np.cumsum(pan, axis=1),
                      core[:, :1] - np.hstack([np.zeros((rows, 1), dtype=np.int64), np.cumsum(core[:, 1:], axis=1)])])
    packed = np.zeros((rows, 2 * n + 2 * head), dtype=np.uint8)
    packed[:, :2 * head].view(np.uint16)[:, :] = pan[:, :head]
    packed[:, 2 * head:4 * head].view(np.uint16)[:, :] = core[:, :head]
    packed[:, 4 * head:4 * head + (n - head)] = pan[:, head:]
    packed[:, 4 * head + (n - head):] = core[:, head:]
    for f64 in (0, 1):
        for threads in (1, 3):
            out = np.full((rows, 2 * n), -7, dtype=np.float64 if f64 else np.int32)
            assert lib.pgx_expand_split(packed.ctypes.data, rows, n, head, out.ctypes.data, f64, threads) == 0
            assert np.array_equal(out.astype(np.int64), want)
    buf = np.zeros(rows * 2 * n + 3, dtype=np.int32)
    unaligned = buf[1:1 + rows * 2 * n]
    assert lib.pgx_expand_split(packed.ctypes.data, rows, n, head, unaligned.ctypes.data, 0, 2) == 0
    assert np.array_equal(unaligned.reshape(rows, 2 * n).astype(np.int64), want)
    assert lib.pgx_expand_split(packed.ctypes.data, rows, n, 0, buf.ctypes.data, 0, 1) == 1          # head out of range
    assert lib.pgx_expand_split(packed.ctypes.data, rows, n, n + 1, buf.ctypes.data, 0, 1) == 1


def _split_rows_from_hist(words, n, head):
    """numpy restatement of split_steps_kernel (csrc/pgx_rarefy.cu): packed histogram rows -- entry e of a row (pan bins,
    then core bins) in half (e & 1) of 32-bit word e >> 1 -- to the split transfer format, plus the overflow flag."""
    rows = words.shape[0]
    entries = words.view(np.uint16).reshape(rows, 2 * n)             # little-endian: the low half is the even entry
    out = np.zeros((rows, 2 * n + 2 * head), dtype=np.uint8)
    heads = out[:, :4 * head].view(np.uint16)
    heads[:, :head] = entries[:, :head]
    heads[:, head:] = entries[:, n:n + head]
    out[:, 4 * head:4 * head + (n - head)] = np.minimum(entries[:, head:n], 255)
    out[:, 4 * head + (n - head):] = np.minimum(entries[:, n + head:], 255)
    overflow = bool((entries[:, head:n] > 255).any() or (entries[:, n + head:] > 255).any())
    return out, overflow


@pytest.mark.parametrize("n, head", [(2048, 512), (2049, 512), (2051, 1), (4097, 1024), (7, 3), (6, 6)])
def test_split_format_agrees_with_the_uint16_rows(n, head):
    """The two transfer formats of the host-buffer calls decode to the same curves: a packed histogram row read as 2N
    uint16 steps (pgx_expand_deltas) and the same row in the split format (pgx_expand_split), odd N included (the
    pan / core boundary then falls inside a word)."""
    lib = _native.load()
    rng = np.random.RandomState(n * 31 + head)
    rows = 9
    steps = rng.randint(0, 256, size=(rows, 2 * n)).astype(np.uint16)
    steps[:, :head] = rng.randint(0, 60000, size=(rows, head))        # large steps inside the heads only
    steps[:, n:n + head] = rng.randint(0, 300, size=(rows, head))
    steps[:, n] = 65535
    words = np.ascontiguousarray(steps).view(np.uint32).reshape(rows, n)
    split, overflow = _split_rows_from_hist(words, n, head)
    assert not overflow
    a = np.empty((rows, 2 * n), dtype=np.int32)
    b = np.empty((rows, 2 * n), dtype=np.int32)
    assert lib.pgx_expand_deltas(steps.ctypes.data, rows, n, a.ctypes.data, 0, 2) == 0
    assert lib.pgx_expand_split(split.ctypes.data, rows, n, head, b.ctypes.data, 0, 2) == 0
    assert np.array_equal(a, b)
    if head < n:
        steps[3, n - 1] = 256                                         # a tail step that does not fit a byte
        words = np.ascontiguousarray(steps).view(np.uint32).reshape(rows, n)
        assert _split_rows_from_hist(words, n, head)[1]
