"""TEST INFRASTRUCTURE -- numpy / scipy specification of the planner (pgx_host_plan_create,
pangenomix_b200/csrc/pgx_plan_build.cpp and the threaded steps of pgx_plan.cpp; see oracle/__init__.py for
who may import this).

``build_host_plan`` makes the same plan as the library's planner, array by array and bit for bit, with one
plain numpy step per C++ step; tests/test_plan.py compares the two.  The device layout is the one
``struct pgx_plan`` documents in include/pgx.h.
"""
from __future__ import annotations

import numpy as np

from pangenomix_b200.plan import CHUNK, MAX_GENOMES, SLICE_ROWS, HostPlan, gene_major_csr, residue_modulus_for

SENTINELS = 32               # rank-table rows N..N+31 hold 0xffff
RUN_LANE_CHUNKS = 32         # most chunk iterations a warp streams per task (sub-blocks of 32 rows x chunks per row)
COLOUR_MAX_CHUNKS = 32       # rows of more chunks than this use the cheap positional bank ordering
RUN_TARGET_TASKS = 1024      # ... but small tables keep enough tasks to spread over the warps of a CTA row
BALANCE_WINDOW = 64          # candidates looked at when a row is chosen for a wavefront group (at least 4 groups' worth)
SMEM_TABLE_BUDGET = 220 * 1024
_COMPLEMENT_BLOCK_CELLS = 1 << 26


def slice_words_for(n_long):
    """Words per lane of the probe walk (1, 2 or 4): wider lines amortise the per-step instructions over
    more genes, as long as (superblocks x permutations) still fills the GPU with warps."""
    return 4 if n_long >= 32768 else (2 if n_long >= 8192 else 1)


def default_long_threshold(n_genomes):
    """Folded length from which a gene is cheaper to serve from the bit-sliced bitmap (a walk of
    ~N/m coalesced lines shared by 1,024 genes) than from its list (m shared-memory gathers):
    the measured break-even on B200 is close to 1.3 sqrt(N) while 8 permutations share every gather
    (N <= 14k; flat between 128 and 160 at N = 10,000) and about 200 at N = 50,000, where only 2 do."""
    batch = perms_per_cta_for(n_genomes)           # fewer permutations share a gather on wide tables
    return max(8, int(round(1.28 * np.sqrt(n_genomes) * (batch / 8.0) ** 0.25)))


def perms_per_cta_for(n_genomes):
    """Permutations whose rank tables fit one CTA's shared memory together (8, 4, 2 or 1)."""
    for b in (8, 4, 2):
        if (n_genomes + SENTINELS) * 2 * b <= SMEM_TABLE_BUDGET:
            return b
    return 1


def _segment_positions(lengths):
    """For concatenated segments of the given lengths: position of every element in its segment."""
    total = int(lengths.sum())
    starts = np.cumsum(lengths) - lengths
    return np.arange(total, dtype=np.int64) - np.repeat(starts, lengths)


def _folded_lists(indptr, indices, m, genes, use_abs, length, n):
    """Concatenated sorted folded lists of ``genes`` (present or absent genomes), int32 (pgx_plan_folded_lists)."""
    ptr = np.concatenate(([0], np.cumsum(length))).astype(np.int64)
    flat = np.empty(int(ptr[-1]), dtype=np.int32)
    keep = np.flatnonzero(~use_abs)
    if keep.size:
        lens = length[keep]
        pos = _segment_positions(lens)
        src = np.repeat(indptr[genes[keep]], lens) + pos
        dst = np.repeat(ptr[:-1][keep], lens) + pos
        flat[dst] = indices[src]
    comp = np.flatnonzero(use_abs)
    if comp.size:
        block = max(1, _COMPLEMENT_BLOCK_CELLS // n)
        for b0 in range(0, comp.size, block):
            rows = comp[b0:b0 + block]
            present_lens = m[genes[rows]]
            pos = _segment_positions(present_lens)
            src = np.repeat(indptr[genes[rows]], present_lens) + pos
            absent = np.ones((rows.size, n), dtype=bool)
            absent[np.repeat(np.arange(rows.size), present_lens), indices[src]] = False
            _, cols = np.nonzero(absent)              # row-major => sorted inside each row
            lens = length[rows]
            assert cols.size == int(lens.sum())
            dst = np.repeat(ptr[:-1][rows], lens) + _segment_positions(lens)
            flat[dst] = cols
    return flat, ptr


def _missing_genome(indptr, indices, genes, n):
    """The genome every gene of ``genes`` (present in exactly n - 1 genomes) is absent from, from prefix sums of
    the indices (pgx_plan_missing_genome)."""
    csum = np.concatenate(([0], np.cumsum(indices, dtype=np.int64)))
    return n * (n - 1) // 2 - (csum[indptr[genes + 1]] - csum[indptr[genes]])


def _balanced_row_order(indptr, indices, genes, use_abs, class_key, n, modulus, window=None):
    """Order of the list rows inside their classes (same chunk count and list kind) that balances the
    shared-memory bank residues of every wavefront group (pgx_plan_balance_rows).

    The ``modulus`` lanes of a group gather in lock step, one entry each; entries whose genome indices agree
    modulo ``modulus`` collide, so a group needs at least max over residues of (its entries of that residue)
    steps, however well ``_bank_ordered_chunks`` arranges them.  Rows sorted by length make the worst groups
    (eight full rows: 64 entries on 8 residues in 8 steps); the kernels do not care which row sits in which
    lane, so groups are formed greedily instead: the class is riffled into ``modulus`` parts (neighbours then
    differ in length), a group starts with the first candidate and then takes, ``modulus`` - 1 times, the one
    among the next ``window`` candidates that keeps the group's largest residue load smallest.  On C4 the
    layout's wavefronts per gather step drop from 1.18 to 1.02 (C2: 1.18 to 1.00; C5, 32-lane groups: 1.38 to 1.09).
    Returns order[i] = current position of the row that takes place i.
    """
    if window is None:
        window = max(BALANCE_WINDOW, 4 * modulus)
    n_rows = genes.shape[0]
    lens = (indptr[genes + 1] - indptr[genes]).astype(np.int64)
    src = np.repeat(indptr[genes], lens) + _segment_positions(lens)
    hist = np.bincount(np.repeat(np.arange(n_rows), lens) * modulus + indices[src] % modulus,
                       minlength=n_rows * modulus).reshape(n_rows, modulus)
    every = (n - np.arange(modulus) + modulus - 1) // modulus                 # genomes c < n with c % modulus == r
    hist = np.where(np.asarray(use_abs, dtype=bool)[:, None], every[None, :] - hist, hist)
    change = np.flatnonzero(np.diff(class_key)) + 1
    starts = np.concatenate(([0], change))
    ends = np.concatenate((change, [n_rows]))
    order = np.empty(n_rows, dtype=np.int64)
    for r0, r1 in zip(starts, ends):
        cnt = int(r1 - r0)
        per = (cnt + modulus - 1) // modulus
        seq = (np.arange(per)[:, None] + per * np.arange(modulus)[None, :]).reshape(-1)
        seq = (r0 + seq[seq < cnt]).tolist()
        cand, pos, out = seq[:window], min(window, cnt), int(r0)
        while cand:
            load = np.zeros(modulus, dtype=np.int64)
            for slot in range(modulus):
                if not cand:
                    break
                pick = 0 if slot == 0 else int(np.argmin((hist[cand] + load).max(axis=1)))
                row = cand.pop(pick)
                order[out] = row
                out += 1
                load += hist[row]
                if pos < cnt:
                    cand.append(seq[pos])
                    pos += 1
    return order


def _colour_groups(cnt, n_steps):
    """Greedy edge colouring, vectorised over wavefront groups.

    ``cnt[g, l, r]`` = entries of residue r in the row of lane l of group g (all rows of a group
    gather in lock step from one shared-memory wavefront).  Chooses for every (group, lane, step) a
    residue, or -1 for a pad, such that every entry gets a step and, wherever possible, the lanes
    of a group use distinct residues at a step (a conflict-free wavefront).  This is edge colouring
    of the bipartite multigraph lanes x residues with ``n_steps`` colours; the greedy rule
    (critical residues first, rows without slack may not pass) gets within a few percent of the
    optimum max(lane degree, residue degree) / n_steps.
    Returns (res_at [G, R, S] int8, pad_res [G, R, S] int8).
    """
    n_groups, r_mod, _ = cnt.shape
    cnt = cnt.astype(np.int32, copy=True)
    res_at = np.full((n_groups, r_mod, n_steps), -1, dtype=np.int8)
    pad_res = np.zeros((n_groups, r_mod, n_steps), dtype=np.int8)
    colload = cnt.sum(axis=1)                      # [G, residue]
    rem = cnt.sum(axis=2)                          # [G, lane]
    ar = np.arange(n_groups)
    for s in range(n_steps):
        taken = np.zeros((n_groups, r_mod), dtype=bool)
        steps_left = n_steps - s
        # rows with the least slack choose first
        order = np.argsort(steps_left - rem, axis=1, kind="stable")           # [G, lane rank] -> lane
        for t in range(r_mod):
            lane = order[:, t]
            c = cnt[ar, lane]                      # [G, residue]
            avail = (c > 0) & ~taken
            score = np.where(avail, colload * 1024 + c, -1)
            choice = score.argmax(axis=1)
            has = avail[ar, choice]
            forced = ~has & (rem[ar, lane] >= steps_left) & (rem[ar, lane] > 0)
            if forced.any():
                choice = np.where(forced, c.argmax(axis=1), choice)
            idx = np.flatnonzero(has | forced)
            if idx.size:
                li, ch = lane[idx], choice[idx]
                res_at[idx, li, s] = ch
                cnt[idx, li, ch] -= 1
                colload[idx, ch] -= 1
                rem[idx, li] -= 1
                taken[idx, ch] = True
        # pads: the k-th idle lane of a group takes the group's k-th unused residue
        idle = res_at[:, :, s] < 0
        if idle.any():
            free_order = np.argsort(taken, axis=1, kind="stable")             # unused residues first
            rank = np.cumsum(idle, axis=1) - 1
            pad_res[:, :, s] = np.where(idle, np.take_along_axis(free_order, np.clip(rank, 0, r_mod - 1), axis=1), 0)
    assert not cnt.any()
    return res_at, pad_res


def _positional_groups(cnt, n_steps):
    """Cheap stand-in for ``_colour_groups`` for very long rows (whose residues are well balanced
    anyway): lane l wants residue (s + l) % R at step s and takes it while it has such entries;
    surplus entries fill the lane's unused steps in order.  Same return convention."""
    n_groups, r_mod, _ = cnt.shape
    steps = np.arange(n_steps)
    lanes = np.arange(r_mod)
    want = (steps[None, :] + lanes[:, None]) % r_mod                         # [lane, step]
    occ = steps[None, :] // r_mod                                            # how many earlier steps wanted the same residue
    have = np.take_along_axis(cnt, np.broadcast_to(want[None], (n_groups, r_mod, n_steps)), axis=2)
    placed = occ[None] < have                                                # [G, lane, step]
    res_at = np.where(placed, want[None], -1).astype(np.int8)
    # surplus entries of a lane, residue by residue, into its unused steps in order
    used = placed.reshape(n_groups, r_mod, n_steps)
    per_res_cap = np.zeros((n_groups, r_mod, r_mod), dtype=np.int64)         # steps that want residue r for lane l
    for r in range(r_mod):
        per_res_cap[:, :, r] = (want == r).sum(axis=1)[None, :]
    surplus = np.maximum(cnt - per_res_cap, 0)                               # [G, lane, residue]
    g_idx, l_idx = np.nonzero(surplus.sum(axis=2))
    for g, l in zip(g_idx, l_idx):
        free = np.flatnonzero(~used[g, l])
        extra = np.repeat(np.arange(r_mod), surplus[g, l])
        res_at[g, l, free[:extra.size]] = extra
    pad_res = np.broadcast_to(want[None], (n_groups, r_mod, n_steps)).astype(np.int8)
    return res_at, pad_res


def _bank_ordered_chunks(flat, ptr, block_first, block_nch, block_first_row, block_rows, n, modulus):
    """Lays the list rows out for the lane-per-row kernel (pgx_plan_bank_order).

    Lane l of a sub-block reads chunk ``first + it * 32 + l`` at iteration ``it`` and gathers the
    rank-table line of the chunk's j-th index at step s = 8 it + j.  The lanes of one shared-memory
    wavefront (``modulus`` consecutive lanes) are conflict-free when their indices differ modulo
    ``modulus``; which entry of a row goes to which step is decided by ``_colour_groups``.  Unused
    steps hold a sentinel index (>= N) of a residue nobody else uses at that step.
    """
    n_blocks = block_nch.shape[0]
    n_slots = int((block_nch * (32 * CHUNK)).sum())
    chunks = np.empty(n_slots, dtype=np.uint16)
    lens = np.diff(ptr)
    n_rows = lens.shape[0]
    row_block = np.repeat(np.arange(n_blocks), block_rows)
    row_lane = np.arange(n_rows) - block_first_row[row_block]
    groups_per_block = 32 // modulus
    row_of_entry = np.repeat(np.arange(n_rows), lens)
    res_of_entry = (flat % modulus).astype(np.int64)
    # entries sorted by (row, residue, index): the k-th entry of a (row, residue) pair takes the
    # k-th step the colouring gave that pair
    e_order = np.lexsort((flat, res_of_entry, row_of_entry))
    for nch in np.unique(block_nch):
        blocks = np.flatnonzero(block_nch == nch)
        n_steps = int(nch) * CHUNK
        local_block = np.full(n_blocks, -1, dtype=np.int64)
        local_block[blocks] = np.arange(blocks.size)
        in_class = local_block[row_block[row_of_entry]] >= 0
        ent = np.flatnonzero(in_class)
        g = local_block[row_block[row_of_entry[ent]]] * groups_per_block + row_lane[row_of_entry[ent]] // modulus
        l = row_lane[row_of_entry[ent]] % modulus
        n_groups = blocks.size * groups_per_block
        cnt = np.bincount((g * modulus + l) * modulus + res_of_entry[ent],
                          minlength=n_groups * modulus * modulus).reshape(n_groups, modulus, modulus)
        if nch <= COLOUR_MAX_CHUNKS:
            res_at, pad_res = _colour_groups(cnt, n_steps)
        else:
            res_at, pad_res = _positional_groups(cnt, n_steps)
        # slot address of (group, lane, step)
        gg, ll, ss = np.meshgrid(np.arange(n_groups), np.arange(modulus), np.arange(n_steps), indexing="ij")
        blk = blocks[gg // groups_per_block]
        lane32 = (gg % groups_per_block) * modulus + ll
        addr = ((block_first[blk] + (ss >> 3) * 32 + lane32) << 3) + (ss & 7)
        is_pad = res_at < 0
        chunks[addr[is_pad]] = (n + ((pad_res[is_pad].astype(np.int64) - n) % modulus)).astype(np.uint16)
        # real slots sorted by (row, residue, step) line up with the class's entries sorted by (row, residue, index)
        real = ~is_pad
        slot_row = (block_first_row[blk] + lane32)[real]
        slot_res = res_at[real].astype(np.int64)
        slot_step = ss[real]
        slot_addr = addr[real]
        s_order = np.lexsort((slot_step, slot_res, slot_row))
        cls_sorted = e_order[in_class[e_order]]                  # entries of this class in (row, residue, index) order
        assert cls_sorted.shape[0] == s_order.shape[0]
        assert np.array_equal(row_of_entry[cls_sorted], slot_row[s_order])
        chunks[slot_addr[s_order]] = flat[cls_sorted].astype(np.uint16)
    return chunks


def _build_bitmap(indptr, indices, m, long_gene, n, slice_words):
    """Genome-major bit-sliced bitmap of the long rows (include/pgx.h, d_bits), a dense block + packbits per
    superblock (pgx_plan_build_bitmap)."""
    sb_rows = SLICE_ROWS * slice_words
    n_super = (long_gene.size + sb_rows - 1) // sb_rows
    bits = np.zeros((n_super, n, sb_rows // 32), dtype=np.uint32)
    for sb in range(n_super):
        rows = long_gene[sb * sb_rows:(sb + 1) * sb_rows]
        lens = m[rows]
        src = np.repeat(indptr[rows], lens) + _segment_positions(lens)
        dense = np.zeros((n, sb_rows), dtype=bool)                       # [genome][row in superblock]
        dense[indices[src], np.repeat(np.arange(rows.size), lens)] = True
        bits[sb] = np.packbits(dense, axis=1, bitorder="little").view(np.uint32)
    return bits.reshape(-1)


def build_host_plan(data, long_threshold=None, perms_per_cta=None, slice_words=None) -> HostPlan:
    """The plan of a table, step by step in numpy (``c_owner`` is None).  ``data`` is anything
    ``gene_major_csr`` takes; the options mean what they mean for pangenomix_b200.plan.build_host_plan."""
    csr = gene_major_csr(data)
    indices = np.asarray(csr.indices)
    colsum = np.bincount(indices, minlength=csr.shape[1]).astype(np.int32)
    indptr = csr.indptr.astype(np.int64)
    n_genes, n = (int(v) for v in csr.shape)
    nnz = int(indices.shape[0])
    if n < 1:
        raise ValueError("table has no genome columns")
    if n > MAX_GENOMES:
        raise ValueError("n_genomes = %d exceeds the supported maximum of %d" % (n, MAX_GENOMES))
    if n_genes >= 2 ** 31 - 1:
        raise ValueError("too many genes")
    if perms_per_cta is None:
        perms_per_cta = perms_per_cta_for(n)
    if perms_per_cta not in (1, 2, 4, 8):
        raise ValueError("perms_per_cta must be 1, 2, 4 or 8")
    modulus = residue_modulus_for(perms_per_cta)
    if long_threshold is None:
        long_threshold = default_long_threshold(n)
    long_threshold = int(long_threshold)
    m = np.diff(indptr)

    empty = m == 0
    full = (m == n) & ~empty
    single_p = (m == 1) & ~full
    single_a = (m == n - 1) & ~single_p & ~full & ~empty
    general = ~(empty | full | single_p | single_a)

    w_present = np.bincount(indices[indptr[:-1][single_p]], minlength=n).astype(np.int32)
    if single_a.any():
        w_absent = np.bincount(_missing_genome(indptr, indices, np.flatnonzero(single_a), n),
                               minlength=n).astype(np.int32)
    else:
        w_absent = np.zeros(n, dtype=np.int32)

    genes = np.flatnonzero(general)
    m_gen = m[genes]
    folded = np.minimum(m_gen, n - m_gen)
    if long_threshold > 0:
        is_long = folded >= long_threshold
    else:
        is_long = np.zeros(genes.shape[0], dtype=bool)

    # ---- bitmap rows: genome-major, bit-sliced, superblocks of 1,024 rows of similar density ----
    long_gene = genes[is_long]
    slice_words = slice_words_for(long_gene.size) if slice_words is None else int(slice_words)
    if slice_words not in (1, 2, 4):
        raise ValueError("slice_words must be 1, 2 or 4")
    if long_gene.size:
        m_long = m[long_gene]
        order = np.argsort(np.minimum(m_long, n - m_long), kind="stable")   # longest walks first
        long_gene = long_gene[order]
        bits = _build_bitmap(indptr, indices, m, long_gene, n, slice_words)
    else:
        bits = np.zeros(0, dtype=np.uint32)

    # ---- list rows -----------------------------------------------------------------------
    genes = genes[~is_long]
    m_gen = m[genes]
    use_abs = m_gen > n - m_gen
    length = np.where(use_abs, n - m_gen, m_gen).astype(np.int64)
    n_chunk = (length + CHUNK - 1) // CHUNK
    order = np.lexsort((-length, use_abs, -n_chunk))         # by chunk count (desc), kind, length
    genes, use_abs, length, n_chunk = (a[order] for a in (genes, use_abs, length, n_chunk))
    if genes.shape[0]:
        # ... and, inside a (chunk count, kind) class, in the order that balances the bank residues of every
        # wavefront group (the kernels do not care which row sits in which lane)
        order = _balanced_row_order(indptr, indices, genes, use_abs, n_chunk * 2 + use_abs, n, modulus)
        genes, use_abs, length, n_chunk = (a[order] for a in (genes, use_abs, length, n_chunk))
    flat, ptr = _folded_lists(indptr, indices, m, genes, use_abs, length, n)
    if ptr[-1] >= 2 ** 31:
        raise ValueError("list rows too large for int32 offsets")

    n_rows = genes.shape[0]
    if n_rows:
        key = n_chunk * 2 + use_abs
        change = np.flatnonzero(np.diff(key)) + 1
        run_starts = np.concatenate(([0], change))
        run_ends = np.concatenate((change, [n_rows]))
        # sub-blocks of 32 rows (one lane per row) ...
        b_first_row, b_rows, b_nch, b_abs, b_run = [], [], [], [], []
        run_id = 0
        total_iters = int(((run_ends - run_starts + 31) // 32 * n_chunk[run_starts]).sum())
        run_budget = int(min(RUN_LANE_CHUNKS, max(2, total_iters // RUN_TARGET_TASKS)))
        for r0, r1 in zip(run_starts, run_ends):
            first_row = np.arange(r0, r1, 32, dtype=np.int64)
            nch = int(n_chunk[r0])
            b_first_row.append(first_row)
            b_rows.append(np.minimum(32, r1 - first_row))
            b_nch.append(np.full(first_row.shape[0], nch, dtype=np.int64))
            b_abs.append(np.full(first_row.shape[0], int(use_abs[r0]), dtype=np.int64))
            # ... streamed by a warp in runs of about RUN_LANE_CHUNKS chunk iterations
            per_run = max(1, run_budget // nch)
            b_run.append(run_id + np.arange(first_row.shape[0]) // per_run)
            run_id = int(b_run[-1][-1]) + 1
        b_first_row, b_rows, b_nch, b_abs, b_run = (np.concatenate(a) for a in (b_first_row, b_rows, b_nch, b_abs, b_run))
        block_first = np.concatenate(([0], np.cumsum(b_nch * 32)))[:-1]
        if (block_first[-1] + b_nch[-1] * 32) * CHUNK >= 2 ** 31:
            raise ValueError("list rows too large for int32 chunk offsets")
        if b_nch.max() >= 1 << 16:
            raise ValueError("list row too long for the task descriptor")
        chunks = _bank_ordered_chunks(flat, ptr, block_first, b_nch, b_first_row, b_rows, n, modulus)
        head = np.flatnonzero(np.concatenate(([True], np.diff(b_run) != 0)))       # first sub-block of every run
        rows_in_run = np.add.reduceat(b_rows, head)
        tasks = np.stack([block_first[head], b_nch[head] | (b_abs[head] << 24), b_first_row[head], rows_in_run],
                         axis=1).astype(np.int32)
        # costly runs first: dynamic fetching then ends on cheap ones
        cost = b_nch[head] * ((rows_in_run + 31) // 32)
        tasks = tasks[np.argsort(-cost, kind="stable")]
    else:
        chunks = np.zeros(0, dtype=np.uint16)
        tasks = np.zeros((0, 4), dtype=np.int32)

    if long_threshold < 0:
        raise ValueError("long_threshold must be >= 0 (0: list rows only)")
    return HostPlan(
        n_genes=int(n_genes), n_genomes=int(n), nnz=nnz,
        perms_per_cta=int(perms_per_cta), long_threshold=long_threshold,
        colsum=colsum, w_present=w_present, w_absent=w_absent,
        n_empty=int(empty.sum()), n_full=int(full.sum()),
        chunks=chunks, tasks=np.ascontiguousarray(tasks),
        sorted_idx=flat.astype(np.uint16), sorted_ptr=ptr.astype(np.int32),
        row_gene=genes, row_len=length.astype(np.int32), row_absent=use_abs.astype(bool),
        bits=bits, slice_words=slice_words, long_gene=long_gene,
        nnz_list=int(m[genes].sum()), nnz_long=int(m[long_gene].sum()))
