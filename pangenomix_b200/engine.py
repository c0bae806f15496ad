"""Device-side engines behind the drop-in API: PanCoreEngine (rarefaction) and BernoulliGrid.

PyTorch is used for plumbing only -- device buffers, pinned host buffers, streams.  All
arithmetic happens in libpgx_b200.so (hand-written sm_100a kernels, include/pgx.h).
"""
from __future__ import annotations

import collections
import ctypes
import os

import numpy as np

from . import _native
from .plan import HostPlan, all_ones, build_host_plan


def _torch():
    import torch
    return torch


def _require_cuda(device=None):
    torch = _torch()
    if not torch.cuda.is_available():
        raise _native.PgxError(
            "no CUDA device visible: pangenomix_b200 has no CPU fallback for the pan/core "
            "and Bernoulli-grid kernels")
    if device is None:
        return torch.device("cuda", torch.cuda.current_device())
    device = torch.device(device)
    if device.type != "cuda":
        raise _native.PgxError("device must be a CUDA device, got %s" % device)
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


def pinned_empty(shape, dtype):
    """numpy array backed by page-locked memory (returns (array, owner tensor))."""
    torch = _torch()
    tdtype = {np.dtype(np.uint16): torch.int16, np.dtype(np.int32): torch.int32,
              np.dtype(np.float64): torch.float64, np.dtype(np.int16): torch.int16}[np.dtype(dtype)]
    owner = torch.empty(tuple(int(s) for s in shape), dtype=tdtype, pin_memory=True)
    arr = owner.numpy()
    if np.dtype(dtype) == np.uint16:
        arr = arr.view(np.uint16)
    return arr, owner


def draw_legacy_permutations(n, count, out=None):
    """``count`` x (np.arange(n); np.random.shuffle) from the GLOBAL legacy numpy stream.

    Consumes exactly what /root/reference/pangenomix/pangenome_analysis.py:84-85 consumes,
    so the global RNG state after the call equals the reference's.  The stream is advanced
    by libpgx's bit-exact MT19937 restatement (pgx_legacy_shuffles) through
    np.random.get_state()/set_state(); set PGX_NUMPY_SHUFFLE=1 to call numpy itself.
    """
    n, count = int(n), int(count)
    if out is None:
        out = np.empty((count, n), dtype=np.uint16)
    if out.shape != (count, n) or out.dtype != np.uint16 or not out.flags.c_contiguous:
        raise ValueError("out must be a C-contiguous uint16 array of shape (count, n)")
    if n > 65535:
        raise ValueError("n_genomes = %d exceeds 65535" % n)
    state = np.random.get_state()
    if os.environ.get("PGX_NUMPY_SHUFFLE") == "1" or state[0] != "MT19937":
        for i in range(count):
            a = np.arange(n)
            np.random.shuffle(a)
            out[i] = a
        return out
    key = np.ascontiguousarray(state[1], dtype=np.uint32).copy()
    pos = ctypes.c_int32(int(state[2]))
    _native.check(_native.load().pgx_legacy_shuffles(
        key.ctypes.data, ctypes.byref(pos), n, count, out.ctypes.data))
    np.random.set_state((state[0], key, int(pos.value), state[3], state[4]))
    return out


MAX_SEED = 2 ** 64 - 1
MOMENT_LIMIT = 2 ** 63        # n_perm * max|value|^2 must stay below this for pgx_curve_moments to be exact


class CurveMoments(collections.namedtuple("CurveMoments", "n sum sumsq min max")):
    """Exact column moments of ``n`` pan/core curves: sum (int64), sum of squares (uint64), min and max (int32),
    each of length 2N (Pan1..PanN, Core1..CoreN)."""


def check_moment_bound(n_perm, n_genes):
    """Raises ValueError unless ``n_perm`` curves of a table of ``n_genes`` genes keep the integer moments exact."""
    if int(n_perm) * max(int(n_genes), 1) ** 2 >= MOMENT_LIMIT:
        raise ValueError("%d permutations of a table of %d genes overflow the exact int64 moments "
                         "(n_perm * G^2 must stay below 2^63)" % (int(n_perm), int(n_genes)))


def _check_stream_range(seed, first, n_perm):
    seed, first, n_perm = int(seed), int(first), int(n_perm)
    if not 0 <= seed <= MAX_SEED:
        raise ValueError("seed must be in [0, 2^64)")
    if first < 0 or n_perm < 0 or first + n_perm > 2 ** 63 - 1:
        raise ValueError("permutation indices must lie in [0, 2^63 - 1)")
    return seed, first, n_perm


def random_permutations_device(n_genomes, n_perm, seed, first=0, device=None, out=None):
    """Permutations ``first .. first + n_perm - 1`` of the seeded on-device stream (pgx_random_perms; the recipe is
    in include/pgx.h) as a CUDA int16 tensor [n_perm, n_genomes] holding uint16 genome indices.

    Permutation i depends on (seed, i) only, so any split of an index range over calls or GPUs gives the same rows.
    Asynchronous on the current torch stream.
    """
    torch = _torch()
    dev = _require_cuda(device)
    seed, first, n_perm = _check_stream_range(seed, first, n_perm)
    n_genomes = int(n_genomes)
    if not 1 <= n_genomes <= 65503:
        raise ValueError("n_genomes = %d outside 1 .. 65503" % n_genomes)
    if out is None:
        out = torch.empty((n_perm, n_genomes), dtype=torch.int16, device=dev)
    elif out.shape != (n_perm, n_genomes) or out.element_size() != 2 or not out.is_contiguous() or out.device != dev:
        raise ValueError("out must be a contiguous 16-bit [n_perm, n_genomes] tensor on %s" % dev)
    with torch.cuda.device(dev):
        _native.check(_native.load().pgx_random_perms(
            seed, first, n_perm, n_genomes, out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream))
    return out


class PanCoreEngine:
    """A presence/absence table resident on one GPU, ready to be rarefied.

    ``data`` is ``df_genes.data`` (scipy COO gene x genome, pangenome_analysis.py:74).
    """

    def __init__(self, data, device=None, host_plan: HostPlan | None = None, long_threshold=None):
        torch = _torch()
        self.device = _require_cuda(device)
        self.lib = _native.load()
        if host_plan is None:
            if long_threshold is None and os.environ.get("PGX_LONG_THRESHOLD"):
                long_threshold = int(os.environ["PGX_LONG_THRESHOLD"])
            slice_words = int(os.environ["PGX_SLICE_WORDS"]) if os.environ.get("PGX_SLICE_WORDS") else None
            host_plan = build_host_plan(data, long_threshold=long_threshold, slice_words=slice_words)
        self.host_plan = host_plan
        hp = self.host_plan
        self.n_genes, self.n_genomes = hp.n_genes, hp.n_genomes

        # the device copy is made and owned by the library (pgx_plan_upload / pgx_plan_destroy)
        with torch.cuda.device(self.device):
            self._plan_ptr = self._upload(hp)
        self.c_plan = self._plan_ptr.contents

    def _upload(self, hp):
        if hp.c_owner is None:
            raise ValueError("host_plan must come from pangenomix_b200.plan.build_host_plan (the library's planner)")
        out = ctypes.POINTER(_native.PgxPlan)()
        _native.check(self.lib.pgx_plan_upload(hp.c_owner.pointer, ctypes.byref(out)))
        return out

    def close(self):
        """Frees the device copy of the table (also done when the engine is garbage-collected)."""
        ptr, self._plan_ptr = getattr(self, "_plan_ptr", None), None
        if ptr:
            self.lib.pgx_plan_destroy(ptr)

    def __del__(self):
        try:
            self.close()
        except Exception:                                # noqa: BLE001 - interpreter shutdown
            pass

    # ---- device-resident path -------------------------------------------------------
    def curves_device(self, perms, out=None):
        """perms: CUDA int16/uint16 tensor [n_perm, N] (uint16 bit patterns) -> int32 [n_perm, 2N].

        Asynchronous on the current torch stream.
        """
        torch = _torch()
        if perms.device != self.device or perms.dim() != 2 or perms.shape[1] != self.n_genomes:
            raise ValueError("perms must be a [n_perm, %d] tensor on %s" % (self.n_genomes, self.device))
        if perms.element_size() != 2 or not perms.is_contiguous():
            raise ValueError("perms must be contiguous 16-bit integers")
        n_perm = int(perms.shape[0])
        if out is None:
            out = torch.empty((n_perm, 2 * self.n_genomes), dtype=torch.int32, device=self.device)
        elif out.shape != (n_perm, 2 * self.n_genomes) or out.dtype != torch.int32 or \
                not out.is_contiguous() or out.device != self.device:
            raise ValueError("out must be a contiguous int32 [n_perm, 2N] tensor on the engine's device")
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            _native.check(self.lib.pgx_pan_core_curves(
                ctypes.byref(self.c_plan), perms.data_ptr(), n_perm, out.data_ptr(), stream))
        return out

    # ---- host-buffer path (the C ABI moves the data) ----------------------------------
    def curves_host(self, perms, out=None, out_f64=False, perms_per_block=0):
        """perms: numpy uint16 [n_perm, N] in host memory -> numpy [n_perm, 2N] (int32 or float64)."""
        torch = _torch()
        perms = np.ascontiguousarray(perms)
        if perms.dtype != np.uint16:
            if perms.size and (perms.min() < 0 or perms.max() >= self.n_genomes):
                raise ValueError("permutation entries out of range")
            perms = perms.astype(np.uint16)
        if perms.ndim != 2 or perms.shape[1] != self.n_genomes:
            raise ValueError("perms must have shape [n_perm, %d]" % self.n_genomes)
        n_perm = perms.shape[0]
        want = np.float64 if out_f64 else np.int32
        if out is None:
            out = np.empty((n_perm, 2 * self.n_genomes), dtype=want)
        if out.shape != (n_perm, 2 * self.n_genomes) or out.dtype != want or not out.flags.c_contiguous:
            raise ValueError("out has the wrong shape / dtype")
        with torch.cuda.device(self.device):
            _native.check(self.lib.pgx_pan_core_curves_host(
                ctypes.byref(self.c_plan), perms.ctypes.data, n_perm, out.ctypes.data,
                1 if out_f64 else 0, int(perms_per_block)))
        return out

    # ---- the reference's call: draw from np.random, return float64 (num_iter, 2N) -----
    def estimate(self, num_iter, log_batch=-1, block=None):
        """pangenome_analysis.py:76-90: curves for ``num_iter`` shuffles of the global numpy RNG.

        One C call (pgx_estimate_pan_core) per stretch of iterations: the library draws the shuffles
        from the legacy MT19937 state, and pipelines RNG, H2D, kernels, D2H and the copy into the
        (ordinary, pageable) float64 result over three internal slots.  With ``log_batch`` > 0 the
        stretches end at the reference's progress lines (:82-83).
        """
        torch = _torch()
        num_iter = int(num_iter)
        n = self.n_genomes
        out = np.empty((num_iter, 2 * n), dtype=np.float64)
        if num_iter == 0:
            return out
        state = np.random.get_state()
        if os.environ.get("PGX_NUMPY_SHUFFLE") == "1" or state[0] != "MT19937":
            perms = draw_legacy_permutations(n, num_iter)
            return self.curves_host(perms, out=out, out_f64=True)
        key = np.ascontiguousarray(state[1], dtype=np.uint32).copy()
        pos = ctypes.c_int32(int(state[2]))
        stretch = num_iter if log_batch <= 0 else int(log_batch)
        with torch.cuda.device(self.device):
            p0 = 0
            while p0 < num_iter:
                cnt = min(stretch, num_iter - p0)
                if log_batch > 0 and p0 > 0:
                    print('\tIteration', p0, 'of', num_iter)       # :82-83
                _native.check(self.lib.pgx_estimate_pan_core(
                    ctypes.byref(self.c_plan), key.ctypes.data, ctypes.byref(pos), cnt,
                    out[p0:].ctypes.data, int(block or 0)))
                p0 += cnt
            if log_batch > 0 and num_iter % log_batch == 0:
                print('\tIteration', num_iter, 'of', num_iter)
        np.random.set_state((state[0], key, int(pos.value), state[3], state[4]))
        return out

    # ---- seeded on-device rarefaction, reduced on the device ----------------------------
    def summary_device(self, num_iter, seed, first=0, block=None):
        """Exact column moments of the curves of permutations ``first .. first + num_iter - 1`` of the seeded
        on-device stream, as CUDA tensors (sum int64, sum of squares int64 holding uint64 bits, min int32,
        max int32; each [2N]).  Blocks of ``block`` permutations (default: about 1 GB of permutations and curves)
        go through generate -> curves_device -> pgx_curve_moments, reusing one permutation and one curve buffer;
        nothing crosses PCIe.  ``num_iter == 0`` gives sums 0, min INT32_MAX, max INT32_MIN.  Asynchronous on the
        current torch stream."""
        torch = _torch()
        seed, first, num_iter = _check_stream_range(seed, first, num_iter)
        check_moment_bound(num_iter, self.n_genes)
        n = self.n_genomes
        if block is None:
            block = max(1, 10 ** 9 // (10 * n))              # 2N bytes of permutation + 8N bytes of curves each
        block = max(1, min(int(block), num_iter))
        dev = self.device
        moments = (torch.empty(2 * n, dtype=torch.int64, device=dev), torch.empty(2 * n, dtype=torch.int64, device=dev),
                   torch.empty(2 * n, dtype=torch.int32, device=dev), torch.empty(2 * n, dtype=torch.int32, device=dev))
        ptrs = [m.data_ptr() for m in moments]
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            if num_iter == 0:
                _native.check(self.lib.pgx_curve_moments(None, 0, 2 * n, *ptrs, 0, stream))
                return moments
            perms = torch.empty((block, n), dtype=torch.int16, device=dev)
            curves = torch.empty((block, 2 * n), dtype=torch.int32, device=dev)
            done = 0
            while done < num_iter:
                k = min(block, num_iter - done)
                random_permutations_device(n, k, seed, first + done, device=dev, out=perms[:k])
                self.curves_device(perms[:k], out=curves[:k])
                _native.check(self.lib.pgx_curve_moments(curves.data_ptr(), k, 2 * n, *ptrs, 1 if done else 0, stream))
                done += k
        return moments

    def summary(self, num_iter, seed, first=0, block=None):
        """summary_device() brought to the host as a CurveMoments of numpy arrays (waits for the device)."""
        s, q, lo, hi = self.summary_device(num_iter, seed, first=first, block=block)
        return CurveMoments(int(num_iter), s.cpu().numpy(), q.cpu().numpy().view(np.uint64), lo.cpu().numpy(),
                            hi.cpu().numpy())

    # ---- genome x genome comparisons -------------------------------------------------------
    def shared_workspace_bytes(self):
        """Workspace of pgx_shared_genes: the whole bitmap expanded as one K-slab, at most SHARED_WORK_CAP bytes (a
        larger table takes several slabs), at least the N x 128 bytes the call needs."""
        hp, n = self.host_plan, self.n_genomes
        k_total = hp.n_superblocks * 1024 * hp.slice_words if hp.n_long else 0
        return max(128 * n, min(n * k_total, SHARED_WORK_CAP))

    def shared_genes_device(self, out=None):
        """Shared-gene matrix S = X^T X of the table (pgx_shared_genes): a CUDA int32 tensor [N, N] with S[k, l] =
        genes present in both genome k and genome l.  The workspace is a torch allocation, released on return.
        Asynchronous on the current torch stream after a short wait in which the library checks the plan."""
        torch = _torch()
        n = self.n_genomes
        if out is None:
            out = torch.empty((n, n), dtype=torch.int32, device=self.device)
        elif out.shape != (n, n) or out.dtype != torch.int32 or not out.is_contiguous() or out.device != self.device:
            raise ValueError("out must be a contiguous int32 [N, N] tensor on the engine's device")
        work_bytes = self.shared_workspace_bytes()
        with torch.cuda.device(self.device):
            work = torch.empty(work_bytes, dtype=torch.uint8, device=self.device)
            _native.check(self.lib.pgx_shared_genes(ctypes.byref(self.c_plan), out.data_ptr(), work.data_ptr(),
                                                    work_bytes, torch.cuda.current_stream(self.device).cuda_stream))
        return out

    def fluidity_rows_device(self, shared):
        """R[k] = sum over l != k of the fluidity distances d_kl of a shared-gene matrix (pgx_fluidity_rows) as a
        CUDA float64 tensor [N].  Asynchronous on the current torch stream."""
        torch = _torch()
        n = self.n_genomes
        if shared.shape != (n, n) or shared.dtype != torch.int32 or not shared.is_contiguous() or \
                shared.device != self.device:
            raise ValueError("shared must be a contiguous int32 [N, N] tensor on the engine's device")
        rows = torch.empty(n, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _native.check(self.lib.pgx_fluidity_rows(shared.data_ptr(), n, rows.data_ptr(),
                                                     torch.cuda.current_stream(self.device).cuda_stream))
        return rows

    # ---- exact rarefaction over all genome orders -------------------------------------------------------------
    def spectrum_device(self):
        """Gene-frequency spectrum of the table from its plan (pgx_plan_spectrum): a CUDA int64 tensor [N + 1], entry
        v = genes present in exactly v genomes.  Asynchronous on the current torch stream after a short wait in which
        the library checks the plan."""
        torch = _torch()
        out = torch.empty(self.n_genomes + 1, dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            _native.check(self.lib.pgx_plan_spectrum(ctypes.byref(self.c_plan), out.data_ptr(),
                                                     torch.cuda.current_stream(self.device).cuda_stream))
        return out

    def pair_workspace_bytes(self):
        """Workspace of pgx_pair_overlap_histograms: every stored row's E row in one panel, at most SHARED_WORK_CAP
        bytes of E rows (a larger table takes several panels), at least the minimum the call needs."""
        hp, n = self.host_plan, self.n_genomes
        stored = hp.n_rows + hp.n_long
        least = int(self.lib.pgx_pair_overlap_work_bytes(n, stored, 0))
        whole = int(self.lib.pgx_pair_overlap_work_bytes(n, stored, 1))
        fixed = whole - -(-stored // 128) * 128 * (-(-n // 128) * 128)
        return max(least, min(whole, fixed + SHARED_WORK_CAP))

    def pair_histograms_device(self, work_bytes=None):
        """Pair overlap histograms (pgx_pair_overlap_histograms) as two CUDA int64 tensors [N + 1]: H_s[v] = gene pairs
        g < h present together in exactly v genomes, H_a[v] = pairs absent together from exactly v genomes.  The
        workspace (pair_workspace_bytes() unless given) is a torch allocation, released on return.  Asynchronous on
        the current torch stream after a short wait in which the library checks the plan."""
        torch = _torch()
        n = self.n_genomes
        hs = torch.empty(n + 1, dtype=torch.int64, device=self.device)
        ha = torch.empty(n + 1, dtype=torch.int64, device=self.device)
        work_bytes = int(work_bytes or self.pair_workspace_bytes())
        with torch.cuda.device(self.device):
            work = torch.empty(work_bytes, dtype=torch.uint8, device=self.device)
            _native.check(self.lib.pgx_pair_overlap_histograms(
                ctypes.byref(self.c_plan), hs.data_ptr(), ha.data_ptr(), work.data_ptr(), work_bytes,
                torch.cuda.current_stream(self.device).cuda_stream))
        return hs, ha

    def exact_moments_device(self, std=True):
        """Mean and variance of the pan and core curves over all genome orders (pgx_rarefaction_moments) as a CUDA
        float64 tensor [4, N]: rows E[pan_k], Var[pan_k], E[core_k], Var[core_k], k = 1 .. N.  With std=False no pair
        histograms are computed, no workspace is allocated and the variance rows are NaN."""
        torch = _torch()
        n = self.n_genomes
        spectrum = self.spectrum_device()
        hs, ha = self.pair_histograms_device() if std else (None, None)
        out = torch.full((4, n), float("nan"), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _native.check(self.lib.pgx_rarefaction_moments(
                spectrum.data_ptr(), hs.data_ptr() if std else None, ha.data_ptr() if std else None, self.n_genes, n,
                out.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream))
        return out


SHARED_WORK_CAP = 4 << 30          # bytes of expanded rows per slab / panel of pgx_shared_genes and the pair histograms


def fit_heaps_device(curves, n_points=None):
    """Heaps-law fits of every row of a CUDA tensor of curves (int32 or float64, contiguous rows).

    curves: [n_curves, stride]; the first ``n_points`` entries of each row are fitted (default: the
    first half, i.e. the Pan half of a pan/core table).  Returns (fit float64 [n_curves, 2]
    {alpha, kappa}, info int32 [n_curves]) as CUDA tensors; asynchronous on the current stream.
    """
    torch = _torch()
    if not curves.is_cuda or curves.dim() != 2 or not curves.is_contiguous():
        raise ValueError("curves must be a contiguous 2-D CUDA tensor")
    if curves.dtype not in (torch.int32, torch.float64):
        raise ValueError("curves must be int32 or float64")
    n_curves, stride = int(curves.shape[0]), int(curves.shape[1])
    n_points = stride // 2 if n_points is None else int(n_points)
    if n_points < 1 or n_points > stride:
        raise ValueError("n_points out of range")
    lib = _native.load()
    fit = torch.empty((n_curves, 2), dtype=torch.float64, device=curves.device)
    info = torch.empty((n_curves,), dtype=torch.int32, device=curves.device)
    scratch = torch.empty((int(lib.pgx_heaps_scratch_bytes(n_points)) + 7) // 8, dtype=torch.float64,
                          device=curves.device)
    with torch.cuda.device(curves.device):
        _native.check(lib.pgx_heaps_fit(
            curves.data_ptr(), 1 if curves.dtype == torch.float64 else 0, n_curves, n_points, stride,
            fit.data_ptr(), info.data_ptr(), scratch.data_ptr(),
            torch.cuda.current_stream(curves.device).cuda_stream))
    return fit, info


class BernoulliGrid:
    """Dense 0/1 gene x genome table, bit-packed on the GPU, for LL / gradient evaluations
    (pangenome_analysis.py:244-266)."""

    def __init__(self, x, device=None):
        torch = _torch()
        self.device = _require_cuda(device)
        self.lib = _native.load()
        x = np.asarray(x)
        if x.ndim != 2 or x.shape[0] < 1 or x.shape[1] < 1:
            raise ValueError("expected a non-empty 2-D gene x genome table")
        xb = x != 0
        if not np.array_equal(xb, x):
            raise ValueError("compute_bernoulli_grid_core_genome needs a dense BINARY (0/1) table "
                             "(pangenome_analysis.py:114-115)")
        self.n_genes, self.n_genomes = x.shape
        packed = np.packbits(xb, axis=1, bitorder="little")
        words = (self.n_genomes + 31) // 32
        padded = np.zeros((self.n_genes, words * 4), dtype=np.uint8)
        padded[:, :packed.shape[1]] = packed
        self.words_per_row = words
        self.row_count = xb.sum(axis=1).astype(np.int32)
        self.col_count = xb.sum(axis=0).astype(np.int32)
        dev = self.device
        self._xbits = torch.from_numpy(padded.view(np.int32).reshape(-1)).to(dev)
        self._row_count = torch.from_numpy(self.row_count).to(dev)
        self._col_count = torch.from_numpy(self.col_count).to(dev)
        total = self.n_genes + self.n_genomes
        self._pq = torch.empty(total, dtype=torch.float64, device=dev)
        self._res = torch.empty(total + 1, dtype=torch.float64, device=dev)   # [ll, grad...]
        scratch = int(self.lib.pgx_bernoulli_scratch_bytes(self.n_genes, self.n_genomes))
        if scratch == 0:
            raise _native.PgxError("Bernoulli grid shape %s x %s is not supported" % x.shape)
        self._scratch = torch.empty((scratch + 7) // 8, dtype=torch.float64, device=dev)
        self._h_pq = torch.empty(total, dtype=torch.float64, pin_memory=True)
        self._h_res = torch.empty(total + 1, dtype=torch.float64, pin_memory=True)
        self._last_x = None
        self.evaluations = 0

    def ll_grad(self, pq):
        """(log-likelihood, gradient[G+N]) at PQ = concat(P, Q); one launch pair, cached by value."""
        torch = _torch()
        pq = np.ascontiguousarray(pq, dtype=np.float64)
        if pq.shape != (self.n_genes + self.n_genomes,):
            raise ValueError("PQ must have length n_genes + n_genomes")
        if self._last_x is not None and np.array_equal(pq, self._last_x):
            return self._last
        g = self.n_genes
        with torch.cuda.device(self.device):
            self._h_pq.numpy()[:] = pq
            self._pq.copy_(self._h_pq, non_blocking=True)
            stream = torch.cuda.current_stream(self.device).cuda_stream
            _native.check(self.lib.pgx_bernoulli_ll_grad(
                self._xbits.data_ptr(), self.words_per_row, self.n_genes, self.n_genomes,
                self._row_count.data_ptr(), self._col_count.data_ptr(),
                self._pq.data_ptr(), self._pq.data_ptr() + 8 * g,
                self._res.data_ptr(), self._res.data_ptr() + 8, self._scratch.data_ptr(), stream))
            self._h_res.copy_(self._res, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
        res = self._h_res.numpy()
        self._last_x = pq.copy()
        self._last = (float(res[0]), res[1:].copy())
        self.evaluations += 1
        return self._last

    def loglikelihood(self, p, q):
        return self.ll_grad(np.concatenate((p, q)))[0]

    def gradient(self, p, q):
        return self.ll_grad(np.concatenate((p, q)))[1]


# ---- beta-binomial core estimate (pangenome_analysis.py:295-400): marginals and Monte-Carlo KS ---------------
def table_marginals(data, device=None, spectrum=True):
    """Row sums, column sums and the gene-frequency spectrum of a binary COO table, counted on the GPU
    (pgx_coo_marginals_host): what ``gene_mat.sum(axis=1)`` + collections.Counter give at
    pangenome_analysis.py:354-355 and LightSparseDataFrame.sum at sparse_utils.py:284-292.

    ``data`` is scipy sparse (``df_genes.data``); every stored value must be 1 and (gene, genome) pairs must not
    repeat -- the producers' invariant (pangenome.py:631-650) -- since entries are COUNTED, not summed.  Returns
    (row_sum int64 [G], col_sum int64 [N], spectrum int64 [N + 1], first_gene int32 [N + 1]); the last two are None
    with ``spectrum=False``.
    """
    torch = _torch()
    dev = _require_cuda(device)
    coo = data.tocoo()
    n_genes, n_genomes = (int(v) for v in coo.shape)
    if n_genes > 2 ** 31 - 1 or n_genomes > 2 ** 31 - 1:
        raise ValueError("table too large")
    if coo.nnz and not all_ones(coo.data):
        raise ValueError("table_marginals counts entries: every stored value must be 1 (binary presence/absence table)")
    row = np.ascontiguousarray(coo.row, dtype=np.int32)
    col = np.ascontiguousarray(coo.col, dtype=np.int32)
    row_sum = np.empty(n_genes, dtype=np.int32)
    col_sum = np.empty(n_genomes, dtype=np.int32)
    spec = np.empty(n_genomes + 1, dtype=np.int64) if spectrum else None
    first = np.empty(n_genomes + 1, dtype=np.int32) if spectrum else None
    with torch.cuda.device(dev):
        _native.check(_native.load().pgx_coo_marginals_host(
            row.ctypes.data, col.ctypes.data, int(row.shape[0]), n_genes, n_genomes, row_sum.ctypes.data,
            col_sum.ctypes.data, spec.ctypes.data if spectrum else None, first.ctypes.data if spectrum else None))
    if row_sum.size and int(row_sum.max()) > n_genomes:
        raise ValueError("duplicate (gene, genome) entries in the table")
    return row_sum.astype(np.int64), col_sum.astype(np.int64), spec, first


def legacy_random_raw(count):
    """``count`` raw 32-bit words from the GLOBAL legacy numpy stream (advanced exactly), as uint32."""
    out = np.empty(int(count), dtype=np.uint32)
    state = np.random.get_state()
    if state[0] != "MT19937":
        raise _native.PgxError("the global numpy RNG is not MT19937")
    key = np.ascontiguousarray(state[1], dtype=np.uint32).copy()
    pos = ctypes.c_int32(int(state[2]))
    _native.check(_native.load().pgx_legacy_random_raw(key.ctypes.data, ctypes.byref(pos), out.shape[0], out.ctypes.data))
    np.random.set_state((state[0], key, int(pos.value), state[3], state[4]))
    return out


def ks_montecarlo_statistics(choice_cdf, model_cdf, n_samples, iterations, device=None):
    """ks_sim of pangenome_analysis.py:471-480: ``iterations`` simulated KS statistics of samples of ``n_samples``
    draws from the choice CDF, drawn from the GLOBAL legacy numpy stream exactly as the reference's
    ``np.random.choice(Xs, size=n_samples * iterations, p=probs)`` (:492) draws them (pgx_ks_montecarlo_host)."""
    torch = _torch()
    dev = _require_cuda(device)
    choice_cdf = np.ascontiguousarray(choice_cdf, dtype=np.float64)
    model_cdf = np.ascontiguousarray(model_cdf, dtype=np.float64)
    if choice_cdf.ndim != 1 or choice_cdf.shape != model_cdf.shape or choice_cdf.shape[0] < 1:
        raise ValueError("choice_cdf and model_cdf must be 1-D arrays of the same length")
    iterations, n_samples = int(iterations), int(n_samples)
    out = np.empty(iterations, dtype=np.float64)
    state = np.random.get_state()
    if state[0] != "MT19937":
        raise _native.PgxError("the global numpy RNG is not MT19937")
    key = np.ascontiguousarray(state[1], dtype=np.uint32).copy()
    pos = ctypes.c_int32(int(state[2]))
    lib = _native.load()
    with torch.cuda.device(dev):
        done = 0
        while done < iterations:                      # the C call takes at most 65,535 iterations
            cnt = min(65535, iterations - done)
            _native.check(lib.pgx_ks_montecarlo_host(
                key.ctypes.data, ctypes.byref(pos), cnt, n_samples, choice_cdf.ctypes.data, model_cdf.ctypes.data,
                int(choice_cdf.shape[0]), out[done:].ctypes.data))
            done += cnt
    np.random.set_state((state[0], key, int(pos.value), state[3], state[4]))
    return out
