"""Host-side planning: COO presence/absence table -> the device layout of ``pgx_plan``.

Input is the object ``estimate_pan_core_size`` reads at
/root/reference/pangenomix/pangenome_analysis.py:74 (``df_genes.data``, a scipy COO
matrix, gene x genome).  The reference transposes it to genome-major CSR (:75) and walks
genomes; the CUDA path needs it gene-major, one row per gene, because a gene's
first-presence / first-absence rank is a reduction over that gene's genomes.

Three populations of genes (include/pgx.h describes the device side):

* closed forms   -- empty / universal / single-genome / single-absence genes are functions of
                    perm[0] and of one rank; they become per-genome weight vectors.
* list rows      -- genes whose shorter list (present or absent genomes) has fewer than
                    ``long_threshold`` entries: uint16 genome indices in 16-byte chunks,
                    one lane per row, sub-blocks of 32 rows of equal chunk count, chunks of a
                    sub-block interleaved so that a warp reads 512 contiguous bytes per step
                    (a warp task streams a run of consecutive sub-blocks), and
                    the entries of every row ordered so that the lanes of a shared-memory
                    bank group hit distinct banks of the rank table.
* bitmap rows    -- the remaining (long) genes as a genome-major bit-sliced bitmap (32 genes per
                    word, 1,024 W per 128 W-byte line, W = 1, 2 or 4); the probe kernel walks genomes in
                    rank order for 1,024 W genes at once instead of scanning long lists.

The planner itself is libpgx's pgx_host_plan_create (csrc/pgx_plan_build.cpp, threaded C++); this module hands it
the table and views the image it returns.  oracle/plan_np.py is its numpy specification.
"""
from __future__ import annotations

import ctypes
import dataclasses

import numpy as np
import scipy.sparse

from . import _native

MAX_GENOMES = 65503          # genome indices, ranks and the 32 sentinel indices N..N+31 are uint16
CHUNK = 8                    # indices per 16-byte chunk
SLICE_ROWS = 1024            # bitmap rows per 128 bytes of a (superblock, genome) line: 32 lanes x 32 bits


def residue_modulus_for(perms_per_cta):
    """Lanes that share one 128-byte shared-memory wavefront when each gathers 2*B bytes."""
    return {8: 8, 4: 16, 2: 32, 1: 32}[int(perms_per_cta)]


@dataclasses.dataclass
class HostPlan:
    n_genes: int
    n_genomes: int
    nnz: int
    perms_per_cta: int
    long_threshold: int
    colsum: np.ndarray        # int32  [N]   genes present in genome c (all genes)
    w_present: np.ndarray     # int32  [N]   genes present ONLY in genome c
    w_absent: np.ndarray      # int32  [N]   genes absent ONLY from genome c
    n_empty: int
    n_full: int
    # list rows
    chunks: np.ndarray        # uint16 [n_chunks * 8]  task-interleaved, bank-ordered
    tasks: np.ndarray         # int32  [n_tasks, 4]  {first_chunk, chunks_per_row | absent<<24, first_row, rows}: a run of
                              #        ceil(rows / 32) consecutive sub-blocks of 32 rows x chunks_per_row chunks
    sorted_idx: np.ndarray    # uint16 [sum(row_len)]  the same lists, plainly sorted (mex probe)
    sorted_ptr: np.ndarray    # int32  [n_rows + 1]
    row_gene: np.ndarray      # int64  [n_rows] gene id of every list row (diagnostics / tests)
    row_len: np.ndarray       # int32  [n_rows] folded list length
    row_absent: np.ndarray    # bool   [n_rows] True when the list holds ABSENT genomes
    # bitmap rows
    bits: np.ndarray          # uint32 [n_superblocks * N * 32 W]  bit b of word (sb, c, w) = row 1024 W sb + 32 w + b in genome c
    slice_words: int          # W: words per lane of a (superblock, genome) line (1, 2 or 4)
    long_gene: np.ndarray     # int64  [n_long]
    nnz_list: int = 0         # present entries of the list-row genes (roofline apportioning)
    nnz_long: int = 0         # present entries of the bitmap-row genes
    c_owner: object = None    # keeps the library's host image alive when the arrays above are views of it

    @property
    def n_rows(self):
        return int(self.row_len.shape[0])

    @property
    def n_long(self):
        return int(self.long_gene.shape[0])

    @property
    def n_superblocks(self):
        rows = SLICE_ROWS * self.slice_words
        return (self.n_long + rows - 1) // rows

    @property
    def n_tasks(self):
        return int(self.tasks.shape[0])

    @property
    def n_chunks(self):
        return int(self.chunks.shape[0] // CHUNK)

    @property
    def folded_nnz(self):
        return int(self.row_len.sum())

    @property
    def algorithmic_bytes_per_perm(self):
        """SURVEY.md section 8d: one pass over the canonical int32 gene-major CSR."""
        return 4 * self.nnz + 4 * (self.n_genes + 1)

    def algorithmic_bytes_of(self, kind):
        """The share of algorithmic_bytes_per_perm that belongs to the genes one row kernel serves."""
        if kind == "list":
            return 4 * self.nnz_list + 4 * self.n_rows
        if kind == "probe":
            return 4 * self.nnz_long + 4 * self.n_long
        raise KeyError(kind)

    @property
    def streamed_bytes_per_pass(self):
        """Bytes the row kernels stream per pass over the rows (list chunks + bitmaps)."""
        return int(self.chunks.nbytes + self.tasks.nbytes + self.bits.nbytes)


def gene_major_csr(data):
    """Canonical binary gene-major CSR of the table; raises on non-binary content.

    ``.tocsr()`` sums duplicate COO entries exactly as the reference's
    ``gene_data.T.tocsr()`` does (pangenome_analysis.py:75).  A summed value other than 1
    changes the reference's core curve but not its pan curve (SURVEY.md a-3'); no producer
    in the reference emits such tables (pangenome.py:631-650), so they are rejected
    rather than silently reinterpreted.
    """
    if isinstance(data, np.ndarray):
        data = scipy.sparse.coo_matrix(data)
    if not scipy.sparse.issparse(data):
        raise TypeError("expected a scipy sparse matrix or a dense ndarray, got %r" % type(data))
    csr = scipy.sparse.csr_matrix(data)
    csr.sum_duplicates()
    csr.sort_indices()
    if csr.nnz:
        values = np.asarray(csr.data)
        if not np.all(values == 1):
            if np.any(values == 0):
                csr.eliminate_zeros()
                values = np.asarray(csr.data)
            if not np.all(values == 1):
                raise ValueError(
                    "presence/absence table is not binary after summing duplicate entries "
                    "(found values other than 0/1); estimate_pan_core_size on the GPU "
                    "requires a binary table")
    return csr


def all_ones(values):
    """True when every stored value of a table is 1 -- what every producer of the reference writes
    (pangenome.py:631-650).  int64 and float64 values are compared word by word on host threads."""
    values = np.asarray(values)
    if values.dtype in (np.dtype(np.int64), np.dtype(np.float64)) and values.flags.c_contiguous:
        one = 1 if values.dtype == np.dtype(np.int64) else int(np.float64(1.0).view(np.uint64))
        return bool(_native.load().pgx_plan_all_equal_u64(values.ctypes.data, values.shape[0], one, 0))
    return values.dtype != object and bool(np.all(values == 1))


class _CHostPlan:
    """Owner of a ``pgx_host_plan`` made by the library's planner (freed with the last HostPlan that views it)."""

    def __init__(self, pointer, destroy):
        self.pointer = pointer
        self._destroy = destroy                  # bound now: module globals may be gone at interpreter shutdown

    def __del__(self):
        if self.pointer is not None:
            self._destroy(self.pointer)
            self.pointer = None


def build_host_plan(data, long_threshold=None, perms_per_cta=None, slice_words=None) -> HostPlan:
    """The plan of a table, made by the library's planner (pgx_host_plan_create).

    A COO matrix whose stored values are all 1 goes to the planner as it is.  Any other table -- CSR, CSC, a dense
    array, explicit zeros, other values, duplicate entries -- is first made canonical by ``gene_major_csr``.
    ``long_threshold`` None: the default (0: list rows only); ``perms_per_cta`` (1, 2, 4, 8) and ``slice_words``
    (1, 2, 4) None or 0: chosen from the table.  The planner's errors (duplicate entries, more than MAX_GENOMES
    genomes, bad options, indices outside the table) raise ValueError.
    """
    if not (scipy.sparse.issparse(data) and data.format == "coo" and data.ndim == 2 and all_ones(data.data)):
        data = gene_major_csr(data).tocoo()
    n_genes, n = (int(v) for v in data.shape)
    options = (-1 if long_threshold is None else int(long_threshold), 0 if perms_per_cta is None else int(perms_per_cta),
               0 if slice_words is None else int(slice_words))
    if not all(-2 ** 31 <= v < 2 ** 31 for v in (n_genes, n) + options):
        raise ValueError("table shape %s or planner options %s outside the int32 range" % ((n_genes, n), options))
    lib = _native.load()
    row = np.ascontiguousarray(data.row, dtype=np.int32)
    col = np.ascontiguousarray(data.col, dtype=np.int32)
    out = ctypes.POINTER(_native.PgxHostPlan)()
    rc = lib.pgx_host_plan_create(row.ctypes.data, col.ctypes.data, int(row.shape[0]), n_genes, n, *options,
                                  ctypes.byref(out))
    if rc != 0:                                  # PGX_ERR_INVALID / PGX_ERR_UNSUPPORTED: a table or option it rejects
        raise ValueError(lib.pgx_last_error().decode("utf-8", "replace"))
    owner = _CHostPlan(out, lib.pgx_host_plan_destroy)
    h = out.contents

    def view(ptr, count, dtype):
        count = int(count)
        if count == 0 or not ptr:
            return np.zeros(0, dtype=dtype)
        buf = (ctypes.c_char * (count * np.dtype(dtype).itemsize)).from_address(ptr)
        arr = np.frombuffer(buf, dtype=dtype, count=count)
        arr.flags.writeable = False
        return arr

    return HostPlan(
        n_genes=int(h.n_genes), n_genomes=int(h.n_genomes), nnz=int(h.nnz), perms_per_cta=int(h.perms_per_cta),
        long_threshold=int(h.long_threshold),
        colsum=view(h.colsum, h.n_genomes, np.int32), w_present=view(h.w_present, h.n_genomes, np.int32),
        w_absent=view(h.w_absent, h.n_genomes, np.int32), n_empty=int(h.n_empty), n_full=int(h.n_full),
        chunks=view(h.chunks, h.n_chunks * CHUNK, np.uint16), tasks=view(h.tasks, h.n_tasks * 4, np.int32).reshape(-1, 4),
        sorted_idx=view(h.sorted_idx, h.n_sorted, np.uint16), sorted_ptr=view(h.sorted_ptr, h.n_rows + 1, np.int32),
        row_gene=view(h.row_gene, h.n_rows, np.int64), row_len=view(h.row_len, h.n_rows, np.int32),
        row_absent=view(h.row_absent, h.n_rows, np.uint8).astype(bool),
        bits=view(h.bits, h.n_bits_words, np.uint32), slice_words=int(h.slice_words),
        long_gene=view(h.long_gene, h.n_long, np.int64), nnz_list=int(h.nnz_list), nnz_long=int(h.nnz_long),
        c_owner=owner)
