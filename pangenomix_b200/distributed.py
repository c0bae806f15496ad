"""Permutation sharding across the GPUs of one box (SURVEY.md section 8e).

Genome orders are independent given the matrix, so the matrix is replicated, rank r
rarefies the contiguous block [lo_r, hi_r) of the ``num_iter`` permutations, and one
gather brings the small curve blocks together.  Contiguous blocks keep row ``Iter{i}``
where the single-GPU path puts it.  One process per GPU, ``torch.distributed`` (NCCL over
NVLink on the B200 box; gloo in the CPU tests of this host-side logic).

The only RNG that matters is rank 0's global numpy stream -- rank 0 draws all
``num_iter`` shuffles exactly as the reference does (pangenome_analysis.py:84-85) and
broadcasts the table.

``estimate_pan_core_summary_sharded`` needs neither: its genome orders come from the seeded
on-device stream, which every rank evaluates for its own block of indices, and the ranks
combine exact integer moments with one all-reduce.
"""
from __future__ import annotations

import numpy as np


def shard_bounds(n_items, world_size, rank):
    """Contiguous block of ``rank``: sizes differ by at most one, earlier ranks get the extra."""
    base, extra = divmod(int(n_items), int(world_size))
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def _dist():
    import torch.distributed as dist
    return dist


def _agree(ok, device, group):
    """All ranks learn whether any of them failed before a collective that the failing rank would never join."""
    import torch
    dist = _dist()
    flag = torch.tensor([0 if ok else 1], dtype=torch.int32, device=device)
    dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=group)
    return int(flag.item()) == 0


def sharded_curves(perms, n_genomes, compute=None, device=None, group=None, dst=None, engine=None):
    """Rarefies ``perms`` ([num_iter, N] uint16, significant on rank 0 only) across the group.

    engine  : a PanCoreEngine on this rank's GPU -- the permutation table is broadcast on the device, every rank
              rarefies its contiguous block with ``curves_device`` and the int32 blocks are gathered on the device
              (NCCL over NVLink); nothing but rank 0's permutations and the final table crosses PCIe.
    compute : instead of an engine, callable(numpy uint16 [k, N]) -> numpy int32 [k, 2N] (the CPU tests of this
              host-side logic inject one; tensors then live on ``device``, the CPU by default).
    dst     : None -> every rank returns the full table (all_gather);
              r    -> only rank r returns it (gather), the others return None.
    """
    import torch
    dist = _dist()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    if engine is not None:
        device = engine.device
    device = torch.device("cpu") if device is None else torch.device(device)

    # rank 0 validates before anybody enters a collective the others could hang in
    problem = None
    if rank == 0:
        perms = np.ascontiguousarray(perms, dtype=np.uint16)
        if perms.ndim != 2 or perms.shape[1] != n_genomes:
            problem = "perms must have shape [num_iter, %d]" % n_genomes
    if not _agree(problem is None, device, group):
        raise ValueError(problem or "rank 0 rejected the permutation table")
    shape = torch.zeros(1, dtype=torch.int64, device=device)
    if rank == 0:
        shape[0] = perms.shape[0]
    dist.broadcast(shape, src=0, group=group)
    num_iter = int(shape.item())

    table = torch.empty((num_iter, n_genomes), dtype=torch.int16, device=device)
    if rank == 0:
        table.copy_(torch.from_numpy(perms.view(np.int16)))
    if num_iter:
        # neither gloo nor NCCL moves 16-bit integers: broadcast the bytes
        dist.broadcast(table.view(torch.uint8), src=0, group=group)

    lo, hi = shard_bounds(num_iter, world, rank)
    # equal-sized padded blocks so a single (all_)gather moves everything
    width = shard_bounds(num_iter, world, 0)[1]
    block = torch.zeros((max(width, 1), 2 * n_genomes), dtype=torch.int32, device=device)
    if hi > lo:
        if engine is not None:
            engine.curves_device(table[lo:hi], out=block[:hi - lo])
        else:
            local = np.ascontiguousarray(compute(table[lo:hi].cpu().numpy().view(np.uint16)), dtype=np.int32)
            if local.shape != (hi - lo, 2 * n_genomes):
                raise ValueError("compute returned shape %s, expected %s" % (local.shape, (hi - lo, 2 * n_genomes)))
            block[:hi - lo].copy_(torch.from_numpy(local))
    if dst is None:
        gathered = torch.empty((world * block.shape[0], block.shape[1]), dtype=torch.int32, device=device)
        dist.all_gather_into_tensor(gathered, block, group=group)
        parts = gathered.view(world, block.shape[0], block.shape[1])
    else:
        parts = [torch.empty_like(block) for _ in range(world)] if rank == dst else None
        dist.gather(block, gather_list=parts, dst=dst, group=group)
        if rank != dst:
            return None
    out = np.empty((num_iter, 2 * n_genomes), dtype=np.int32)
    for r in range(world):
        r_lo, r_hi = shard_bounds(num_iter, world, r)
        if r_hi > r_lo:
            out[r_lo:r_hi] = parts[r][:r_hi - r_lo].cpu().numpy()
    return out


def estimate_pan_core_size_sharded(df_genes, num_iter, log_batch=-1, group=None, dst=None, compute=None, engine=None):
    """Multi-GPU ``estimate_pan_core_size``: same DataFrame as the single-GPU call on the
    ranks that receive it (all ranks for ``dst=None``), None elsewhere.

    Every rank must call it with the same table; only rank 0's numpy RNG is consumed (exactly ``num_iter``
    legacy shuffles, as pangenome_analysis.py:84-85).  Each rank plans and uploads the table once per LSDF
    object (the engine cache of the single-GPU call) unless an ``engine`` is passed.  ``compute`` is injectable
    for the CPU tests of the sharding logic.
    """
    import pandas as pd
    from .engine import draw_legacy_permutations
    dist = _dist()
    rank = dist.get_rank(group)
    num_genes, num_strains = df_genes.shape
    if compute is None and engine is None:
        from .pangenome_analysis import _engine_for
        engine = _engine_for(df_genes)
    perms = None
    if rank == 0:
        print('Converting DataFrame to matrix...')
        print('Generating pan/core curves from shuffled strains')
        if log_batch > 0:
            for it in range(log_batch, num_iter + 1, log_batch):
                print('\tIteration', it, 'of', num_iter)
        perms = draw_legacy_permutations(num_strains, num_iter)
    curves = sharded_curves(perms, num_strains, compute, group=group, dst=dst, engine=engine)
    if curves is None:
        return None
    iter_index = ['Iter' + str(x) for x in range(1, num_iter + 1)]
    pan_cols = ['Pan' + str(x) for x in range(1, num_strains + 1)]
    core_cols = ['Core' + str(x) for x in range(1, num_strains + 1)]
    return pd.DataFrame(curves.astype(np.float64), index=iter_index, columns=pan_cols + core_cols, copy=False)


def estimate_pan_core_summary_sharded(df_genes, num_iter, seed=0, group=None, dst=None, compute=None, engine=None):
    """Multi-GPU ``estimate_pan_core_summary``: the same DataFrame, bit for bit, for every world size, on the ranks
    that receive it (all ranks for ``dst=None``), None elsewhere.

    Rank r reduces the permutations ``shard_bounds(num_iter, world, r)`` of the seeded on-device stream to integer
    moments on its own GPU; there is no broadcast of permutations and no gather of curves, only one all-reduce of
    4 x 2N integers (SUM of the sums and of the sums of squares as int64 bit patterns, MIN / MAX of the extremes).
    Every rank must call it with the same table, ``num_iter`` and ``seed``; numpy's RNG is not touched.

    engine  : a PanCoreEngine on this rank's GPU (default: the engine cache of the single-GPU call).
    compute : instead of an engine, callable(first, count) -> (sum int64, sumsq uint64, min int32, max int32) numpy
              arrays of length 2N for permutations first .. first + count - 1 (the CPU tests of this host-side logic
              inject one; tensors then live on the CPU).
    """
    import torch
    from .engine import check_moment_bound, CurveMoments
    from .pangenome_analysis import summary_frame
    dist = _dist()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    num_iter = int(num_iter)
    if num_iter < 1:
        raise ValueError("num_iter must be at least 1")
    n_genes, num_strains = df_genes.shape
    check_moment_bound(num_iter, n_genes)
    if compute is None and engine is None:
        from .pangenome_analysis import _engine_for
        engine = _engine_for(df_genes)
    device = engine.device if engine is not None else torch.device("cpu")
    lo, hi = shard_bounds(num_iter, world, rank)
    width = 2 * num_strains

    problem = None
    try:
        if engine is not None:
            parts = list(engine.summary_device(hi - lo, seed, first=lo))
        else:
            parts = [torch.zeros(width, dtype=torch.int64), torch.zeros(width, dtype=torch.int64),
                     torch.full((width,), 2 ** 31 - 1, dtype=torch.int32), torch.full((width,), -2 ** 31, dtype=torch.int32)]
            if hi > lo:
                local = compute(lo, hi - lo)
                for k, (arr, dtype) in enumerate(zip(local, (np.int64, np.uint64, np.int32, np.int32))):
                    arr = np.ascontiguousarray(arr, dtype=dtype)
                    if arr.shape != (width,):
                        raise ValueError("compute returned shape %s, expected (%d,)" % (arr.shape, width))
                    parts[k] = torch.from_numpy(arr.view(np.int64) if dtype == np.uint64 else arr)
    except Exception as exc:                                    # noqa: BLE001 - reported after the ranks agree
        problem = exc
    if not _agree(problem is None, device, group):
        if problem is not None:
            raise problem
        raise RuntimeError("another rank failed to compute its share of the summary")
    for tensor, op in zip(parts, (dist.ReduceOp.SUM, dist.ReduceOp.SUM, dist.ReduceOp.MIN, dist.ReduceOp.MAX)):
        dist.all_reduce(tensor, op=op, group=group)
    if dst is not None and rank != dst:
        return None
    s, q, mn, mx = (t.cpu().numpy() for t in parts)
    return summary_frame(CurveMoments(num_iter, s, q.view(np.uint64), mn, mx), num_strains)


class CurveGather:
    """Gathers every rank's int32 curve block of a step on rank ``dst`` over NVLink.

    Contract: buffer b may be sent again only after the destination has consumed its previous content; callers
    reuse a buffer after a barrier or a drain on every rank (bench.py alternates two buffers per step and reads the
    gathered blocks only behind a barrier) -- there is no cross-rank flow control inside the class.

    Preferred path: peer memory.  The destination is a symmetric-memory buffer
    (torch.distributed._symmetric_memory: cuMem allocations mapped into every peer over
    NVLink / NVSwitch); each rank PUSHES its block into its slot of rank ``dst``'s buffer with a
    copy-engine peer copy on a side stream, so the transfer costs no SM time on either side and
    overlaps the next step's kernels.  Fallback (no peer access, gloo, one rank): an asynchronous
    ``dist.gather``.  Two buffers per rank: step i may still be travelling while step i+1 runs.
    """

    def __init__(self, rows, width, device, group=None, dst=0, n_buffers=2, prefer_peer=True):
        import torch
        dist = _dist()
        self.torch, self.dist = torch, dist
        self.group, self.dst = group, dst
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.rows, self.width, self.n_buffers = int(rows), int(width), int(n_buffers)
        self.device = torch.device(device)
        self.mode = "nccl-gather"
        self._pending = [None] * self.n_buffers
        self._lists = None
        self._peer = None
        if prefer_peer and self.device.type == "cuda" and self.world > 1:
            try:
                import torch.distributed._symmetric_memory as symm_mem
                numel = self.n_buffers * self.world * self.rows * self.width
                self._symm = symm_mem.empty(numel, dtype=torch.int32, device=self.device)
                handle = symm_mem.rendezvous(self._symm, dist.group.WORLD if group is None else group)
                self._peer = handle.get_buffer(self.dst, (self.n_buffers, self.world, self.rows, self.width),
                                               torch.int32)
                self._stream = torch.cuda.Stream(self.device)
                self._ready = [torch.cuda.Event() for _ in range(self.n_buffers)]
                self._done = [None] * self.n_buffers
                self._own = [None] * self.n_buffers
                self.mode = "peer-push"
            except Exception as exc:                                   # noqa: BLE001 - any failure means "no peer path"
                self._peer = None
                self.fallback_reason = "%s: %s" % (type(exc).__name__, exc)
        if prefer_peer and self.device.type == "cuda" and self.world > 1:
            # the mode is a collective decision: a rank pushing into peer memory while another waits in
            # dist.gather would deadlock the group
            if not _agree(self._peer is not None, self.device, group) and self._peer is not None:
                self._peer = None
                self.mode = "nccl-gather"
                self.fallback_reason = "another rank could not map the symmetric buffer"
        if self._peer is None and self.rank == self.dst:
            self._lists = [[torch.empty((self.rows, self.width), dtype=torch.int32, device=self.device)
                            for _ in range(self.world)] for _ in range(self.n_buffers)]

    def before_overwrite(self, b):
        """Call before the producer writes buffer ``b`` again: its previous transfer must have read it."""
        if self._peer is not None:
            if self._done[b] is not None:
                self.torch.cuda.current_stream(self.device).wait_event(self._done[b])
        elif self._pending[b] is not None:
            self._pending[b].wait()
            self._pending[b] = None

    def send(self, b, block):
        """Ships ``block`` (int32 [rows, width], produced on the current stream) as buffer ``b``."""
        torch = self.torch
        if self._peer is not None:
            if self.rank == self.dst:
                # the destination's own block does not travel: gathered() reads it where it is
                self._own[b] = block
                return
            self._ready[b].record(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(self._stream):
                self._stream.wait_event(self._ready[b])
                self._peer[b, self.rank].copy_(block, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self._stream)
                self._done[b] = ev
        else:
            self._pending[b] = self.dist.gather(block, gather_list=self._lists[b] if self._lists else None,
                                                dst=self.dst, group=self.group, async_op=True)

    def drain(self):
        """Makes the current stream wait until every transfer issued by THIS rank has completed."""
        for b in range(self.n_buffers):
            self.before_overwrite(b)

    def gathered(self, b):
        """On ``dst``: the list of the ``world`` [rows, width] blocks of buffer ``b`` (valid after every
        rank drained and the ranks passed a barrier)."""
        if self.rank != self.dst:
            return None
        if self._peer is not None:
            blocks = [self._peer[b, r] for r in range(self.world)]
            if self._own[b] is not None:
                blocks[self.dst] = self._own[b]
            return blocks
        return list(self._lists[b])
