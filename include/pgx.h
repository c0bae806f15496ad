/* pgx.h -- C ABI of libpgx_b200.so: the pan/core rarefaction + Bernoulli-grid hot path of
 * pangenomix on NVIDIA B200 (sm_100a).
 *
 * The reference (AnnaLew/pangenomix) is pure Python and has no FFI of its own; the
 * functions declared here are what a ctypes binding inside the reference's
 * pangenome_analysis.py would call instead of its Python loops (see INTEGRATION.md):
 *
 *   pgx_pan_core_curves[_host]   replaces the double loop of estimate_pan_core_size,
 *                                /root/reference/pangenomix/pangenome_analysis.py:81-90
 *   pgx_bernoulli_ll_grad        replaces __bernoulli_grid_loglikelihood__ (:244-249) and
 *                                __bernoulli_grid_loglikelihood_gradient__ (:257-266) as
 *                                called from the L-BFGS-B lambdas at :156-160
 *   pgx_legacy_shuffles          replaces the np.arange + np.random.shuffle pair at :84-85
 *                                (numpy legacy MT19937 stream, bit-exact)
 *   pgx_heaps_fit                batched counterpart of __fit_heaps_single__ (:39-48)
 *   pgx_ks_montecarlo[_host]     replaces the simulation loop of ks_montecarlo_bbn (:471-480) incl. the
 *                                np.random.choice draws of draw_bbn (:484-492), bit-exact
 *   pgx_coo_marginals[_host],    replace ``gene_mat.sum(axis=1)`` + collections.Counter at :352-355
 *   pgx_frequency_spectrum       (LightSparseDataFrame.sum, sparse_utils.py:284-292;
 *                                count_gene_occurence, core_genome.py:127-155)
 *
 * Conventions: every function returns 0 on success and a non-zero code otherwise;
 * pgx_last_error() then returns a thread-local message.  No C++ types, exceptions or
 * torch types cross this boundary.  Pointers prefixed d_ are DEVICE pointers owned by
 * the caller (the library never frees caller memory); h_ are HOST pointers.  Functions
 * taking a ``stream`` (a cudaStream_t passed as void*) are asynchronous on that stream;
 * the *_host variants are synchronous and move the data themselves.
 */
#ifndef PGX_H_
#define PGX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGX_VERSION 321

enum {
    PGX_OK = 0,
    PGX_ERR_INVALID = 1,   /* bad argument (null pointer, size out of range, ...) */
    PGX_ERR_CUDA = 2,      /* a CUDA runtime call or kernel launch failed */
    PGX_ERR_UNSUPPORTED = 3
};

/* Device-resident plan of a BINARY gene x genome presence/absence table, built once per
 * matrix by pgx_plan_create (below; oracle/plan_np.py is its numpy specification) from
 * ``df_genes.data`` -- the same object estimate_pan_core_size reads at pangenome_analysis.py:74.
 * Genes fall into three groups:
 *
 *  closed forms  Empty, universal, single-genome and single-absence genes never reach a row
 *                kernel: they are functions of perm[0] and of one rank and live in the
 *                per-genome vectors d_colsum / d_w_present / d_w_absent.
 *  list rows     Every other gene whose SHORTER list (present genomes or absent genomes) has
 *                fewer than the plan's long threshold entries stores that list as uint16
 *                genome indices in 16-byte chunks.  A sub-block is up to 32 rows with the
 *                same chunk count and list kind, one lane per row; lane l reads chunk
 *                first_chunk + it * 32 + l at iteration it; a warp task streams a run of
 *                consecutive sub-blocks.  Unused slots hold sentinel
 *                indices in [N, N + 32) whose rank-table entry is 0xffff.  Entries are
 *                ordered inside a row so that neighbouring lanes gather from different
 *                shared-memory banks.  d_sorted_* hold the same lists plainly sorted.
 *  bitmap rows   The remaining (long) genes, as a genome-major bit-sliced bitmap: rows are
 *                grouped in superblocks of 1,024 W (W = slice_words = 1, 2 or 4);
 *                d_bits[(sb * N + c) * 32 W + w] holds, in bit b, the presence of row
 *                sb * 1024 W + 32 w + b in genome c (one line of 128 W bytes per (superblock,
 *                genome); lane l of the probing warp owns words l W .. l W + W - 1).  Rows of
 *                similar density share a superblock.
 */
typedef struct pgx_plan {
    const uint16_t *d_chunks;      /* [n_chunks * 8] list rows, 16-byte aligned */
    const int32_t *d_tasks;        /* [n_tasks * 4] {first_chunk, chunks_per_row | absent_list << 24, first_row,
                                      rows}: a run of ceil(rows / 32) consecutive sub-blocks; 16-byte aligned,
                                      costly tasks first */
    const uint16_t *d_sorted_idx;  /* sorted copy of the list rows */
    const int32_t *d_sorted_ptr;   /* [n_rows + 1] offsets into d_sorted_idx */
    const uint32_t *d_bits;        /* [n_superblocks * n_genomes * 32 W] bit-sliced bitmap rows, 16-byte aligned */
    const void *reserved_ptr;
    const int32_t *d_colsum;       /* [n_genomes] #genes present in genome c (all genes of the table) */
    const int32_t *d_w_present;    /* [n_genomes] #genes present ONLY in genome c */
    const int32_t *d_w_absent;     /* [n_genomes] #genes absent ONLY from genome c */
    int64_t n_chunks;
    int32_t n_genomes;             /* N  (1 <= N <= 65503) */
    int32_t n_genes;               /* G  (all genes of the table, incl. closed-form ones) */
    int32_t n_rows;                /* list rows */
    int32_t n_tasks;
    int32_t n_long;                /* bitmap rows */
    int32_t n_superblocks;         /* ceil(n_long / (1024 * slice_words)) */
    int32_t perms_per_cta;         /* 8, 4, 2 or 1: rank tables that share a CTA's shared memory */
    int32_t slice_words;           /* W = 1, 2 or 4: words per lane of a (superblock, genome) line */
    int32_t max_colsum;            /* max over genomes of d_colsum; 1 .. 65535 lets the kernels count in uint16 bins and
                                      the host-buffer calls ship uint16 curve steps (0 = unknown: int32 everywhere) */
    int32_t reserved_i32;
} pgx_plan;

/* Host image of a plan: what pgx_host_plan_create makes of the COO table and pgx_plan_upload copies to the device.
 * All arrays are owned by the image (pgx_host_plan_destroy frees them); sizes as in struct pgx_plan.  The row_* /
 * long_gene arrays say which gene became which list / bitmap row (diagnostics and tests). */
typedef struct pgx_host_plan {
    void *owner;
    const uint16_t *chunks;        /* [n_chunks * 8] */
    const int32_t *tasks;          /* [n_tasks * 4] */
    const uint16_t *sorted_idx;    /* [n_sorted] */
    const int32_t *sorted_ptr;     /* [n_rows + 1] */
    const uint32_t *bits;          /* [n_bits_words] */
    const int32_t *colsum, *w_present, *w_absent;   /* [n_genomes] each */
    const int64_t *row_gene;       /* [n_rows] gene of every list row */
    const int32_t *row_len;        /* [n_rows] folded list length */
    const uint8_t *row_absent;     /* [n_rows] 1 when the list holds the ABSENT genomes */
    const int64_t *long_gene;      /* [n_long] gene of every bitmap row */
    int64_t nnz, nnz_list, nnz_long, n_chunks, n_bits_words, n_sorted;
    int32_t n_genomes, n_genes, n_rows, n_tasks, n_long, n_superblocks, perms_per_cta, slice_words;
    int32_t long_threshold, max_colsum, n_empty, n_full;
} pgx_host_plan;

/* The planner (host only, threaded; no GPU work): COO entries of a BINARY gene x genome table -- row = gene,
 * col = genome, every entry a presence, as every producer of the reference writes ``df_genes.data``
 * (pangenome.py:631-650; read back by read_lsdf, sparse_utils.py:35) -- to the host image of a plan.
 *   long_threshold : folded list length from which a gene is served from the bitmap (< 0: the default,
 *                    about 1.28 sqrt(N); 0: list rows only)
 *   perms_per_cta  : 8, 4, 2, 1 or 0 = as many rank tables as fit one CTA's shared memory
 *   slice_words    : 1, 2, 4 or 0 = choose by the number of bitmap rows
 * Duplicate (gene, genome) entries -- which scipy's tocsr() at pangenome_analysis.py:75 would sum to a non-binary
 * table -- are rejected with PGX_ERR_INVALID. */
int pgx_host_plan_create(const int32_t *row, const int32_t *col, int64_t nnz, int32_t n_genes, int32_t n_genomes,
                         int32_t long_threshold, int32_t perms_per_cta, int32_t slice_words, pgx_host_plan **out);
void pgx_host_plan_destroy(pgx_host_plan *plan);

/* Device plans owned by the library, on the calling thread's current device.  pgx_plan_create = pgx_host_plan_create
 * with the defaults + pgx_plan_upload; the returned plan is what every pgx_pan_core_* call takes and lives until
 * pgx_plan_destroy.  (A caller may instead fill a struct pgx_plan with device pointers of its own, as the Python
 * engine can with torch tensors: the calls never look behind the struct.) */
int pgx_plan_create(const int32_t *row, const int32_t *col, int64_t nnz, int32_t n_genes, int32_t n_genomes,
                    int32_t long_threshold, pgx_plan **out);
int pgx_plan_upload(const pgx_host_plan *host, pgx_plan **out);
int pgx_plan_destroy(pgx_plan *plan);

int pgx_version(void);
const char *pgx_last_error(void);

/* SM count, opt-in shared memory per block and L2 size of the current device. */
int pgx_device_info(int32_t *sm_count, int32_t *smem_optin_bytes, int64_t *l2_bytes);

/* Pan/core curves for n_perm genome orders (pangenome_analysis.py:81-90).
 *   d_perms  : [n_perm][N] uint16, row i = shuffle_indices of iteration i (:84-85).  TRUSTED input: every row
 *              must be a permutation of 0 .. N-1 (entries >= N are ignored, a genome that does not occur counts
 *              as never sampled; the host-buffer calls below report such rows as PGX_ERR_INVALID)
 *   d_curves : [n_perm][2N] int32; columns 0..N-1 = pan_genomes[i,:], N..2N-1 =
 *              core_genomes[i,:] (the np.hstack layout of :97).  Overwritten; also the kernels' workspace
 *              (rank rows and histogram rows live in it until the final scan), 16-byte aligned.
 * Asynchronous on ``stream``. */
int pgx_pan_core_curves(const pgx_plan *plan, const uint16_t *d_perms, int64_t n_perm,
                        int32_t *d_curves, void *stream);

/* Same, float64 output exactly as the reference's DataFrame values (:76-77, :97).
 *   d_hist   : caller scratch of n_perm * 2N int32, 4-byte aligned (the kernels read and write it as uint16 and
 *              32-bit words and use 16-byte accesses only where they find it 16-byte aligned); overwritten
 *   d_curves : [n_perm][2N] float64, 8-byte aligned (16-byte stores where the rows are 16-byte aligned, else 8-byte);
 *              must not overlap d_hist
 * n_perm == 0 writes nothing and returns PGX_OK.  Asynchronous on ``stream``. */
int pgx_pan_core_curves_f64(const pgx_plan *plan, const uint16_t *d_perms, int64_t n_perm,
                            int32_t *d_hist, double *d_curves, void *stream);

/* Host-buffer entry point: h_perms [n_perm][N] uint16 and h_curves [n_perm][2N]
 * (int32 when out_f64 == 0, float64 otherwise) live in host memory (pinned h_perms make
 * the uploads asynchronous).  The plan stays device-resident.  The call pipelines
 * H2D -> kernels -> D2H -> result over three internal slots in blocks of ``perms_per_block``
 * permutations (0 = choose) and returns when h_curves is complete.  When plan->max_colsum <= 65535 the
 * device ships the curves' STEPS as uint16 (half the bytes of int32 curves, a quarter of float64) -- on tables of
 * 2,048 genomes or more as uint16 heads + uint8 tails (pgx_expand_split; PGX_SPLIT_HEAD=0 switches that off) -- into pinned
 * staging owned by the library and host threads rebuild the curves straight into h_curves (PGX_COPY_THREADS).
 * Rows of h_perms that are not permutations of 0 .. N-1 make the call fail with PGX_ERR_INVALID.
 * One host-buffer call (this one or pgx_estimate_pan_core) at a time per process. */
int pgx_pan_core_curves_host(const pgx_plan *plan, const uint16_t *h_perms, int64_t n_perm,
                             void *h_curves, int32_t out_f64, int64_t perms_per_block);

/* estimate_pan_core_size in one call (pangenome_analysis.py:76-90): draws n_iter consecutive
 * ``np.arange(N); np.random.shuffle`` permutations from the numpy-legacy MT19937 state
 * (mt_key[624] / mt_pos as np.random.get_state() reports them; advanced in place exactly as the
 * reference's loop advances the global stream), rarefies them on the current device and writes
 * the float64 [n_iter][2N] table the reference builds with np.hstack (:97) into h_curves
 * (ordinary host memory).  RNG, H2D, kernels, D2H and the final copy are pipelined over three
 * internal slots; staging is cached for the life of the library.  One call at a time per process. */
int pgx_estimate_pan_core(const pgx_plan *plan, uint32_t *mt_key, int32_t *mt_pos, int64_t n_iter,
                          double *h_curves, int64_t perms_per_block);

/* ``head`` of the split row format the host-buffer calls currently use for the table size they last served
 * (pgx_expand_split; 0 = plain uint16 rows): 2N + 2 head bytes per permutation cross PCIe instead of 4N. */
int pgx_split_head(void);

/* Launch-shape overrides for experiments (0 = heuristic): permutations per CTA of the list
 * kernel (1, 2, 4 or 8), row splits per permutation batch and threads per CTA. */
int pgx_set_tuning(int32_t perms_per_cta, int32_t row_splits, int32_t threads_per_cta);

/* Per-kernel timing for roofline reports: while enabled, every pgx_pan_core_curves[_f64]
 * call brackets its kernels with CUDA events on the caller's stream and runs the two row kernels
 * back to back.  The host-buffer calls (pgx_pan_core_curves_host, pgx_estimate_pan_core) are never
 * profiled, whatever the table's bin format, and keep their schedule.  pgx_profile_read waits for the
 * events, returns the summed durations (ms) of the list kernel, the bitmap-probe kernel (a kernel a
 * call did not launch, because the table has no such rows, counts 0) and everything else (prep + scan
 * kernels) and the number of profiled calls since the last read, and releases the events. */
int pgx_profile_enable(int32_t on);
int pgx_profile_read(double *list_ms, double *probe_ms, double *scan_ms, int64_t *calls);

/* Evidence of how the two row kernels share the SMs: while a device buffer of 1 + 3 * capacity_records uint64 is set
 * (zero-initialised by the caller; null switches the trace off), every CTA of the list kernel and every warp of the
 * probe kernel appends {kind (1 list, 2 probe) | smid << 8, start, end} in %globaltimer nanoseconds; word 0 counts
 * the records.  scripts/overlap_trace.py turns it into profiles/r02/overlap_timeline_<name>.json. */
int pgx_set_trace(void *d_trace, int64_t capacity_records);

/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t pgx_launch_count(void);

/* Bernoulli grid: log-likelihood and gradient at (P, Q) (pangenome_analysis.py:244-266).
 *   d_xbits     : [G][words_per_row] uint32, bit (j & 31) of word (j >> 5) = X[i][j]
 *   d_row_count : [G] int32  = X.sum(axis=1);   d_col_count : [N] int32 = X.sum(axis=0)
 *   d_p [G], d_q [N] float64;  d_ll [1], d_grad [G + N] float64 (dL/dp then dL/dq)
 *   d_scratch   : pgx_bernoulli_scratch_bytes(G, N) bytes
 * Deterministic (fixed reduction order).  Asynchronous on ``stream``. */
size_t pgx_bernoulli_scratch_bytes(int64_t n_genes, int64_t n_genomes);
int pgx_bernoulli_ll_grad(const uint32_t *d_xbits, int64_t words_per_row, int64_t n_genes,
                          int64_t n_genomes, const int32_t *d_row_count,
                          const int32_t *d_col_count, const double *d_p, const double *d_q,
                          double *d_ll, double *d_grad, void *d_scratch, void *stream);

/* Batched Heaps-law fits y = kappa * x^alpha, x = 1 .. n_points, one per curve: the GPU counterpart of
 * fit_heaps_by_iteration / __fit_heaps_single__ (pangenome_analysis.py:24-48; scipy curve_fit, start point
 * alpha = 0.5, kappa = min(y)).  Levenberg-Marquardt with the analytic Jacobian, run to fp64 convergence.
 *   d_curves : n_curves rows of ``stride`` elements, int32 (is_f64 == 0) or float64; the first n_points
 *              of every row are fitted (the Pan half of a pgx_pan_core_curves row: stride = 2N)
 *   d_fit    : [n_curves][2] float64 {alpha, kappa}
 *   d_info   : optional [n_curves] int32, LM trials used (negative: stopped without converging)
 *   d_scratch: pgx_heaps_scratch_bytes(n_points) bytes
 * Deterministic.  Asynchronous on ``stream``. */
size_t pgx_heaps_scratch_bytes(int64_t n_points);
int pgx_heaps_fit(const void *d_curves, int32_t is_f64, int64_t n_curves, int64_t n_points, int64_t stride,
                  double *d_fit, int32_t *d_info, void *d_scratch, void *stream);

/* Returns 1 when every 64-bit word of words[0 .. n) equals ``value``, else 0: the planner's "every stored value
 * is 1" test for the int64 (value 1) and float64 (value = bits of 1.0) ``data`` arrays of a table. */
int pgx_plan_all_equal_u64(const uint64_t *words, int64_t n, uint64_t value, int32_t n_threads);

/* LSDF ingest (host): raw DEFLATE (RFC 1951) of one zip member straight into the caller's buffer.
 * Replaces the zlib inflate inside scipy.sparse.load_npz, which read_lsdf calls
 * (/root/reference/pangenomix/sparse_utils.py:35; the archive is written deflated at :314).
 * dst_len must be the exact inflated size (the zip entry's file_size).  Returns PGX_ERR_INVALID for
 * anything that is not a complete, well-formed stream of that size; the caller verifies the
 * entry's CRC-32 and falls back to zlib on any error.  Thread-safe (no shared state). */
int pgx_inflate_raw(const uint8_t *src, int64_t src_len, uint8_t *dst, int64_t dst_len);

/* Host half of the compact transfer (no GPU work): rows of 2N uint16 curve steps
 *   d[0] = pan[0], d[k] = pan[k] - pan[k-1];  d[N] = core[0], d[N+k] = core[k-1] - core[k]
 * -> curves [n_rows][2N], int32 (out_f64 == 0) or float64.  n_threads 0 = choose. */
int pgx_expand_deltas(const uint16_t *h_deltas, int64_t n_rows, int32_t n_genomes, void *h_curves,
                      int32_t out_f64, int32_t n_threads);

/* The same for the SPLIT row format the host-buffer calls use on tables of many genomes: a step above 255 only
 * occurs while the first genomes are added, so the first ``head`` steps of each curve travel as uint16, the rest as
 * uint8 -- per row [pan head: head x u16][core head: head x u16][pan tail: (N - head) x u8][core tail: (N - head) x u8],
 * 2N + 2 head bytes instead of 4N (a block with a larger step in a tail is sent again as uint16 and ``head`` doubled
 * for the blocks after it).  1 <= head <= N. */
int pgx_expand_split(const uint8_t *h_rows, int64_t n_rows, int32_t n_genomes, int32_t head, void *h_curves,
                     int32_t out_f64, int32_t n_threads);

/* numpy legacy RandomState stream (host): ``count`` consecutive
 * ``a = np.arange(n); np.random.shuffle(a)`` results as uint16 rows, continuing from the
 * MT19937 state in ``mt_key`` (624 words) / ``mt_pos`` exactly as
 * np.random.get_state() reports them; the advanced state is written back so the caller
 * can np.random.set_state() it.  Requires n <= 65535. */
int pgx_legacy_shuffles(uint32_t *mt_key, int32_t *mt_pos, int64_t n, int64_t count,
                        uint16_t *h_perms);

/* Raw 32-bit outputs of the same stream (host): ``count`` words continuing the MT19937 state, written back
 * advanced.  numpy's legacy random_sample() consumes two of them per double, (a >> 5, b >> 6) -> (a * 2^26 + b) / 2^53;
 * RandomState.choice(p=...) -- draw_bbn, pangenome_analysis.py:484-492 -- one such double per draw. */
int pgx_legacy_random_raw(uint32_t *mt_key, int32_t *mt_pos, int64_t count, uint32_t *h_out);

/* Marginals of a COO presence/absence table on the device: d_row_sum[g] = entries of gene g (what
 * ``gene_mat.sum(axis=1)`` gives for a binary table without duplicates, pangenome_analysis.py:354-355; also
 * LightSparseDataFrame.sum, sparse_utils.py:284-292, and count_gene_occurence, core_genome.py:127-155),
 * d_col_sum[c] = entries of genome c.  Entries outside the table are skipped and counted in *d_bad.
 *   accumulate == 0 : the three outputs are zeroed first;  != 0 : counts are added (tables sent in chunks)
 * Asynchronous on ``stream``. */
int pgx_coo_marginals(const int32_t *d_row, const int32_t *d_col, int64_t nnz, int32_t n_genes, int32_t n_genomes,
                      int32_t *d_row_sum, int32_t *d_col_sum, int32_t *d_bad, int32_t accumulate, void *stream);

/* Gene-frequency spectrum of the row sums: d_spectrum[m] (int64 [N + 1]) = genes present in exactly m genomes,
 * d_first_gene[m] (int32 [N + 1]) = the lowest gene index among them (INT32_MAX when there is none): the order of
 * first appearance is the order of the collections.Counter the reference slices at pangenome_analysis.py:355, :364.
 * Row sums above N (duplicate entries) are counted at N.  Asynchronous on ``stream``. */
int pgx_frequency_spectrum(const int32_t *d_row_sum, int64_t n_genes, int32_t n_genomes, int64_t *d_spectrum,
                           int32_t *d_first_gene, void *stream);

/* Both of the above for a table in host memory (row / col as read_lsdf returns them in ``.data``); synchronous.
 * h_spectrum / h_first_gene may be null.  Entries outside the table make the call fail with PGX_ERR_INVALID. */
int pgx_coo_marginals_host(const int32_t *h_row, const int32_t *h_col, int64_t nnz, int32_t n_genes, int32_t n_genomes,
                           int32_t *h_row_sum, int32_t *h_col_sum, int64_t *h_spectrum, int32_t *h_first_gene);

/* Monte-Carlo Kolmogorov-Smirnov statistics of ks_montecarlo_bbn (pangenome_analysis.py:457-482): for iteration i,
 * n_samples draws of ``np.random.choice(np.arange(sim_limit), p=probs)`` (draw_bbn, :484-492), their eCDF
 * (ecdf_from_counts, :494-499) and d_ks_sim[i] = max |eCDF - model_cdf| (:479), float64, bit-exact.
 *   d_raw        : [iterations][n_samples][2] uint32, the raw MT19937 words of the draws in stream order
 *                  (pgx_legacy_random_raw), 8-byte aligned
 *   d_choice_cdf : [sim_limit] float64, ``cdf = probs.cumsum(); cdf /= cdf[-1]`` as numpy's choice forms it
 *   d_model_cdf  : [sim_limit] float64, ``np.cumsum(model_pmf)`` of :464-465
 *   d_scratch    : pgx_ks_scratch_bytes(iterations, sim_limit) bytes
 * iterations <= 65,535 per call, n_samples < 2^31.  Deterministic.  Asynchronous on ``stream``. */
size_t pgx_ks_scratch_bytes(int64_t iterations, int32_t sim_limit);
int pgx_ks_montecarlo(const uint32_t *d_raw, int64_t iterations, int64_t n_samples, const double *d_choice_cdf,
                      const double *d_model_cdf, int32_t sim_limit, double *d_ks_sim, void *d_scratch, void *stream);

/* The same with host buffers, drawing from the numpy-legacy MT19937 state (mt_key[624] / mt_pos as
 * np.random.get_state() reports them; advanced in place by the 2 * iterations * n_samples words the reference's
 * np.random.choice call consumes).  The generator (host, serial) fills one block of iterations while the previous one
 * is uploaded and reduced on the current device.  Synchronous; one call at a time per process. */
int pgx_ks_montecarlo_host(uint32_t *mt_key, int32_t *mt_pos, int64_t iterations, int64_t n_samples,
                           const double *h_choice_cdf, const double *h_model_cdf, int32_t sim_limit, double *h_ks_sim);

/* Seeded genome orders generated on the device, for rarefaction curves whose statistics matter rather than numpy's
 * particular shuffles (the drop-in pgx_estimate_pan_core keeps numpy's stream).  Permutation i (a 64-bit global
 * index) is a pure function of (seed, i): results do not depend on block sizes, on how a range is split over calls
 * or over GPUs.  The recipe (oracle/perm_np.py restates it in numpy):
 *
 *   Philox4x32-10 (Salmon et al., SC'11) with key (seed & 0xffffffff, seed >> 32); lo / hi = low / high 32 bits of i.
 *   B(N) = the largest power of two <= ceil(N / 2), b = log2 B (B <= 16,384 for N <= 65,503).
 *   1. Genome c draws bucket  w >> (32 - b)  (0 when b == 0), w = word c % 4 of Philox({c / 4, lo, hi, 0}).
 *   2. Each bucket's genomes are put in ascending genome order.
 *   3. Bucket k of m genomes is Fisher-Yates shuffled from the top: for j = m - 1 down to 1, draw v = w & mask(j)
 *      (mask(j) = smallest 2^t - 1 >= j) until v <= j, then swap entries j and v.  The t-th word (t = 0, 1, ...)
 *      bucket k consumes is word t % 4 of Philox({k, lo, hi, 0x80000000 | t / 4}).
 *   4. The row is bucket 0, bucket 1, ..., bucket B - 1 concatenated.
 * Every bucket is a uniformly random ordering of its members and the bucket draws do not depend on genome labels, so
 * the distribution of the row is invariant under relabelling the genomes: it is exactly uniform for every B (with
 * Philox taken as ideal), unlike sorting by random keys, whose ties make it only approximately so.
 *   d_perms : [n_perm][N] uint16, rows first .. first + n_perm - 1 (the layout pgx_pan_core_curves takes), 2-byte
 *             aligned.  1 <= N <= 65503, 0 <= first, 0 <= n_perm <= 2^31 - 1.
 * One CTA per permutation, the row in shared memory.  Asynchronous on ``stream``. */
int pgx_random_perms(uint64_t seed, int64_t first, int64_t n_perm, int32_t n_genomes, uint16_t *d_perms, void *stream);

/* Exact column moments of a block of curves (int32 [n_rows][width], width even, 8-byte aligned):
 *   d_sum[c] = sum of column c (int64), d_sumsq[c] = sum of squares (uint64), d_min[c] / d_max[c] (int32).
 *   accumulate == 0 : the outputs are first set to 0, 0, INT32_MAX, INT32_MIN;  != 0 : the block is added to them.
 * Integer accumulators make the result independent of the order of the atomics.  Exact while the rows accumulated
 * into one set of outputs, n, satisfy  n * max|value|^2 < 2^63  (sums of squares then also fit an int64, which a
 * caller combining several GPUs relies on); for pan/core curves max|value| <= G, the table's genes: at G = 2 M about
 * 2.3 M permutations.  The caller enforces the bound.  Asynchronous on ``stream``. */
int pgx_curve_moments(const int32_t *d_curves, int64_t n_rows, int64_t width, int64_t *d_sum, uint64_t *d_sumsq,
                      int32_t *d_min, int32_t *d_max, int32_t accumulate, void *stream);

/* Shared-gene matrix S = X^T X of a planned table: S[k][l] = genes present in both genome k and genome l, S[k][k] =
 * d_colsum[k].  With A the absent-list rows, u[k] the absent-list rows listing genome k and n_full the universal genes,
 * for k != l the plan's classes contribute
 *
 *   S[k][l] = n_full + sum(w_absent) - w_absent[k] - w_absent[l]            universal and single-absence genes
 *           + |A| - u[k] - u[l] + #{absent-list rows listing k and l}       absent lists
 *           + #{present-list rows listing k and l}                          present lists
 *           + sum over bitmap rows of bit_k * bit_l                         bitmap rows: an 8-bit integer GEMM
 *
 * (empty and single-presence genes add nothing off the diagonal).  n_full is derived on the device from genome 0's
 * diagonal; a plan whose rows and vectors do not add up to d_colsum[0] fails with PGX_ERR_INVALID.  The bitmap rows are
 * expanded, a K-slab at a time, into a genome-major 0 / 1 byte matrix E [N][K_slab] in the workspace and S += E E^T
 * runs on the tensor cores (tcgen05.mma kind::i8, s32 accumulators), upper-triangle tiles only; the upper triangle is
 * then mirrored into the lower one.  oracle/shared_np.py restates all of it.
 *   d_shared   : [N][N] int32, 16-byte aligned; overwritten
 *   d_work     : caller workspace of work_bytes >= N * 128 bytes, 16-byte aligned; the slab width K_slab is the
 *                largest multiple of 128 with N * K_slab <= work_bytes (capped at the bitmap rows), so a smaller
 *                workspace only means more slabs
 * Asynchronous on ``stream`` except for one wait, after the small kernels that derive n_full, to check the plan. */
int pgx_shared_genes(const pgx_plan *plan, int32_t *d_shared, void *d_work, int64_t work_bytes, void *stream);

/* Row sums of the genomic-fluidity distances (Kislyuk et al., BMC Genomics 12:32, 2011) of a shared-gene matrix:
 *   d_row_sums[k] = sum over l != k of d_kl,   d_kl = (M_k + M_l - 2 S[k][l]) / (M_k + M_l),   M = diag(S)
 * in float64 (a pair with M_k + M_l = 0 gives NaN).  Fixed reduction order: two calls give the same bits.  Fluidity
 * is sum(d_row_sums) / 2 over N (N - 1) / 2 pairs.
 *   d_shared : [N][N] int32 as pgx_shared_genes writes it, 4-byte aligned;  d_row_sums : [N] float64, 8-byte aligned
 * 1 <= N <= 65503.  Asynchronous on ``stream``. */
int pgx_fluidity_rows(const int32_t *d_shared, int32_t n_genomes, double *d_row_sums, void *stream);

/* Exact pan/core rarefaction: the mean and variance of the pan and core sizes of the first k genomes over ALL genome
 * orders, without sampling.  The first k genomes of a uniformly random order are a uniformly random k-subset T; with
 * m_g the genomes holding gene g, s_gh the genomes holding both g and h, a_gh = N - m_g - m_h + s_gh the genomes
 * lacking both, and rho(v, k) = C(v, k) / C(N, k) (the chance that T lies inside a given set of v genomes):
 *
 *   E[core_k] = sum_g rho(m_g, k)                    Var[core_k] = E[core_k] + 2 sum_{g<h} rho(s_gh, k) - E[core_k]^2
 *   E[pan_k]  = G - sum_g rho(N - m_g, k)  (Mao's tau; Colwell, Mao & Chang, Ecology 85:2717, 2004)
 *   Var[pan_k] = Z_k + 2 sum_{g<h} rho(a_gh, k) - Z_k^2,   Z_k = sum_g rho(N - m_g, k)
 *
 * The variance is conditional on the table (the spread over orders of these N genomes, what the permutation std
 * converges to).  The means need the spectrum of m; the variances the pair histograms
 * H_s[v] = #{g < h : s_gh = v} and H_a[v] = #{g < h : a_gh = v}.
 *
 * Gene-frequency spectrum of a planned table: d_spectrum[v] (int64 [N + 1]) = genes present in exactly v genomes,
 * counted from the plan alone (rows by their lists or bit counts, the closed-form classes from the per-genome vectors;
 * the universal and empty counts are derived on the device).  A plan whose rows and vectors do not add up to whole
 * universal and empty counts fails with PGX_ERR_INVALID.  Asynchronous on ``stream`` except for one final wait that
 * checks the plan. */
int pgx_plan_spectrum(const pgx_plan *plan, int64_t *d_spectrum, void *stream);

/* Pair overlap histograms H_s and H_a (int64 [N + 1] each, 8-byte aligned; overwritten) over the unordered pairs of
 * distinct genes of the whole table, closed-form genes included.  With e / u the empty / universal genes,
 * p1 = sum(w_present), a1 = sum(w_absent), and for a stored (list or bitmap) row h: m_h, Wp_h = sum of w_present
 * and Wa_h = sum of w_absent over the genomes holding h, the pairs count as follows ((s, a): count):
 *
 *   empty x row h            (0, N - m_h): e
 *   universal x row h        (m_h, 0): u
 *   single-genome x row h    (1, N - m_h): Wp_h          (0, N - 1 - m_h): p1 - Wp_h
 *   single-absence x row h   (m_h - 1, 0): Wa_h          (m_h, 1): a1 - Wa_h
 *   empty x empty / universal / single-genome / single-absence   (0, N): C(e, 2)  (0, 0): e u  (0, N - 1): e p1
 *                                                                (0, 1): e a1
 *   universal x universal / single-genome / single-absence       (N, 0): C(u, 2)  (1, 0): u p1  (N - 1, 0): u a1
 *   single-genome x single-genome, same / other genome           (1, N - 1): sum_c C(wp_c, 2)  (0, N - 2): the rest
 *   single-absence x single-absence, same / other genome         (N - 1, 1): sum_c C(wa_c, 2)  (N - 2, 0): the rest
 *   single-genome x single-absence, same / other genome          (0, 0): sum_c wp_c wa_c       (1, 1): the rest
 *   row x row                s from an 8-bit integer GEMM, a = N - m_g - m_h + s
 *
 * The stored rows are sorted by m (a tile of sorted rows then knows the range of its s and a), expanded in panels
 * into a gene-major 0 / 1 byte matrix E [P][N_pad] (N_pad = N rounded up to 128) and E E^T runs over panel pairs
 * I <= J on the tensor cores (tcgen05.mma kind::i8, s32 accumulators; the GEMM of pgx_shared_genes with a histogram
 * epilogue): a tile counts into shared-memory bins when its value range fits them, else into the global bins.
 * oracle/exact_np.py restates all of it.
 *   d_work     : caller workspace, 256-byte aligned, of work_bytes >= pgx_pair_overlap_work_bytes(N, R, 0) bytes,
 *                R = n_rows + n_long (the rows' bookkeeping plus two panels of 256 E rows, or all R rows when fewer);
 *                pgx_pair_overlap_work_bytes(N, R, 1) holds every E row in one panel, and any size in between works
 *                with more panels
 * The plan is checked as by pgx_plan_spectrum.  Asynchronous on ``stream`` except for that one wait. */
int pgx_pair_overlap_histograms(const pgx_plan *plan, int64_t *d_hist_shared, int64_t *d_hist_absent, void *d_work,
                                int64_t work_bytes, void *stream);

/* Workspace bytes of pgx_pair_overlap_histograms for N genomes and R = n_rows + n_long stored rows: the minimum
 * (one_panel == 0) or the size that holds every stored row in one panel (one_panel != 0).  0 for N outside
 * 1 .. 65503 or R outside 0 .. 2^31 - 513. */
int64_t pgx_pair_overlap_work_bytes(int32_t n_genomes, int64_t n_stored_rows, int32_t one_panel);

/* The four exact curves from the spectrum and the pair histograms: d_out [4][N] float64 (8-byte aligned), rows
 * E[pan_k], Var[pan_k], E[core_k], Var[core_k] for k = 1 .. N.  One thread per k sums w[v] rho(v, k) over
 * v = N .. k with rho(N, k) = 1 and rho(v - 1, k) = rho(v, k) (v - k) / v (products, never lgamma differences, which
 * lose about 1e-10 relative at N = 50,000; an underflow to 0 ends the sum), in that fixed order: two calls give the
 * same bits, and rho(v, N) = [v = N] makes both variances exactly 0 at k = N.  With both histograms null only the
 * two mean rows are written.  n_genes is G (the table's genes, closed-form ones included).  1 <= N <= 65503.
 * Asynchronous on ``stream``. */
int pgx_rarefaction_moments(const int64_t *d_spectrum, const int64_t *d_hist_shared, const int64_t *d_hist_absent,
                            int64_t n_genes, int32_t n_genomes, double *d_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PGX_H_ */
