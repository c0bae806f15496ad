// pgx_host_plan_create: a gene x genome presence/absence table (COO) -> the host image of ``struct pgx_plan``.
//
// This is the whole planner behind the C ABI, so that a host in any language can feed the library the object
// estimate_pan_core_size reads at /root/reference/pangenomix/pangenome_analysis.py:74 (``df_genes.data``, the COO
// matrix read_lsdf loads, sparse_utils.py:35) without Python: classification of the genes (closed forms, list
// rows, bitmap rows), the order of the list rows, sub-blocks / runs / tasks, and -- through the threaded helpers
// of pgx_plan.cpp -- the canonical CSR, the folded lists, the residue-balanced grouping, the bank ordering and the
// bit-sliced bitmap.  oracle/plan_np.py is the numpy SPECIFICATION of every step; the tests compare
// the two plans array by array, bit for bit.  Nothing here touches the GPU (pgx_plan_create in pgx_api.cu uploads
// the image).
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <new>
#include <numeric>
#include <vector>

#include "pgx.h"

namespace pgx {
int fail(int code, const char *fmt, ...);

// the threaded steps of pgx_plan.cpp (n_threads 0 = choose)
int pgx_plan_coo_to_csr(const int32_t *row, const int32_t *col, int64_t nnz, int32_t n_genes, int32_t n_genomes,
                        int64_t *indptr, int32_t *indices, int32_t *colsum, int64_t *n_duplicates, int32_t n_threads);
int pgx_plan_missing_genome(const int64_t *indptr, const int32_t *indices, const int64_t *genes, int64_t n_rows,
                            int32_t n_genomes, int32_t *missing, int32_t n_threads);
int pgx_plan_build_bitmap(const int64_t *indptr, const int32_t *indices, const int64_t *long_gene, int64_t n_long,
                          int32_t n_genomes, int32_t slice_words, uint32_t *bits, int32_t n_threads);
int pgx_plan_balance_rows(const int64_t *indptr, const int32_t *indices, const int64_t *genes, const uint8_t *use_abs,
                          const int64_t *class_key, int64_t n_rows, int32_t n_genomes, int32_t modulus, int32_t window,
                          int64_t *order, int32_t n_threads);
int pgx_plan_folded_lists(const int64_t *indptr, const int32_t *indices, const int64_t *genes, const uint8_t *use_abs,
                          const int64_t *ptr, int64_t n_rows, int32_t n_genomes, int32_t *flat, int32_t n_threads);
int pgx_plan_bank_order(const int32_t *flat, const int64_t *ptr, int64_t n_rows, const int64_t *block_first,
                        const int64_t *block_nch, const int64_t *block_first_row, const int64_t *block_rows,
                        int64_t n_blocks, int32_t n_genomes, int32_t modulus, int32_t colour_max_chunks,
                        uint16_t *chunks, int32_t n_threads);
}  // namespace pgx

namespace {

constexpr int MAX_GENOMES = 65503;        // plan.py
constexpr int CHUNK = 8;
constexpr int SENTINELS = 32;
constexpr int SLICE_ROWS = 1024;
constexpr int RUN_LANE_CHUNKS = 32;
constexpr int COLOUR_MAX_CHUNKS = 32;
constexpr int RUN_TARGET_TASKS = 1024;
constexpr int BALANCE_WINDOW = 64;
constexpr long long SMEM_TABLE_BUDGET = 220 * 1024;

int perms_per_cta_for(int n)
{
    for (int b : {8, 4, 2})
        if (static_cast<long long>(n + SENTINELS) * 2 * b <= SMEM_TABLE_BUDGET) return b;
    return 1;
}

int residue_modulus_for(int perms_per_cta)
{
    return perms_per_cta == 8 ? 8 : (perms_per_cta == 4 ? 16 : 32);
}

int default_long_threshold(int n)
{
    const int batch = perms_per_cta_for(n);
    const double x = 1.28 * sqrt(static_cast<double>(n)) * pow(batch / 8.0, 0.25);
    return std::max(8, static_cast<int>(nearbyint(x)));          // round half to even, as numpy's round
}

int slice_words_for(long long n_long)
{
    return n_long >= 32768 ? 4 : (n_long >= 8192 ? 2 : 1);
}

// the arrays a pgx_host_plan points into
struct Storage {
    std::vector<uint16_t> chunks, sorted_idx;
    std::vector<int32_t> tasks, sorted_ptr, colsum, w_present, w_absent, row_len;
    std::vector<uint32_t> bits;
    std::vector<int64_t> row_gene, long_gene;
    std::vector<uint8_t> row_absent;
    pgx_host_plan view;
};

}  // namespace

extern "C" void pgx_host_plan_destroy(pgx_host_plan *plan)
{
    if (!plan) return;
    delete reinterpret_cast<Storage *>(plan->owner);
}

extern "C" int pgx_host_plan_create(const int32_t *row, const int32_t *col, int64_t nnz, int32_t n_genes,
                                    int32_t n_genomes, int32_t long_threshold, int32_t perms_per_cta,
                                    int32_t slice_words, pgx_host_plan **out)
{
    if (!out) return pgx::fail(PGX_ERR_INVALID, "out is null");
    *out = nullptr;
    if (n_genes < 0 || nnz < 0 || (nnz > 0 && (!row || !col))) return pgx::fail(PGX_ERR_INVALID, "bad table passed to pgx_host_plan_create");
    if (n_genomes < 1) return pgx::fail(PGX_ERR_INVALID, "table has no genome columns");
    if (n_genomes > MAX_GENOMES)
        return pgx::fail(PGX_ERR_UNSUPPORTED, "n_genomes = %d exceeds the supported maximum of %d", n_genomes, MAX_GENOMES);
    if (n_genes >= INT32_MAX) return pgx::fail(PGX_ERR_UNSUPPORTED, "too many genes");
    if (perms_per_cta <= 0) perms_per_cta = perms_per_cta_for(n_genomes);
    if (perms_per_cta != 1 && perms_per_cta != 2 && perms_per_cta != 4 && perms_per_cta != 8)
        return pgx::fail(PGX_ERR_INVALID, "perms_per_cta must be 1, 2, 4 or 8");
    if (slice_words != 0 && slice_words != 1 && slice_words != 2 && slice_words != 4)
        return pgx::fail(PGX_ERR_INVALID, "slice_words must be 1, 2 or 4");
    const int n = n_genomes;
    const int modulus = residue_modulus_for(perms_per_cta);
    if (long_threshold < 0) long_threshold = default_long_threshold(n);

    Storage *st = new (std::nothrow) Storage();
    if (!st) return pgx::fail(PGX_ERR_INVALID, "out of memory");
    struct Guard {
        Storage *p;
        ~Guard() { delete p; }
    } guard{st};
    // PGX_PLAN_TRACE=1: seconds per phase on stderr (development aid)
    const bool trace = getenv("PGX_PLAN_TRACE") != nullptr;
    auto t_last = std::chrono::steady_clock::now();
    auto phase = [&](const char *name) {
        if (!trace) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[pgx plan] %-28s %.3f s\n", name, std::chrono::duration<double>(now - t_last).count());
        t_last = now;
    };
    try {
        // ---- canonical gene-major CSR (pangenome_analysis.py:74-75 asks scipy for the genome-major one) ----
        std::vector<int64_t> indptr(static_cast<size_t>(n_genes) + 1, 0);
        std::vector<int32_t> indices(static_cast<size_t>(nnz));
        st->colsum.assign(static_cast<size_t>(n), 0);
        int64_t dups = 0;
        if (nnz > 0) {
            if (int rc = pgx::pgx_plan_coo_to_csr(row, col, nnz, n_genes, n, indptr.data(), indices.data(), st->colsum.data(), &dups, 0))
                return rc;
        }
        if (dups)
            return pgx::fail(PGX_ERR_INVALID, "presence/absence table is not binary after summing duplicate entries "
                                              "(%lld duplicate cells); estimate_pan_core_size on the GPU requires a binary table",
                             static_cast<long long>(dups));
        auto m_of = [&](int64_t g) { return indptr[g + 1] - indptr[g]; };

        phase("COO -> CSR");
        // ---- closed forms -------------------------------------------------------------------------------------
        st->w_present.assign(static_cast<size_t>(n), 0);
        st->w_absent.assign(static_cast<size_t>(n), 0);
        std::vector<int64_t> single_a, general;
        long long n_empty = 0, n_full = 0;
        for (int64_t g = 0; g < n_genes; ++g) {
            const int64_t m = m_of(g);
            if (m == 0) ++n_empty;
            else if (m == n) ++n_full;
            else if (m == 1) ++st->w_present[indices[indptr[g]]];
            else if (m == n - 1) single_a.push_back(g);
            else general.push_back(g);
        }
        if (!single_a.empty()) {
            std::vector<int32_t> missing(single_a.size());
            if (int rc = pgx::pgx_plan_missing_genome(indptr.data(), indices.data(), single_a.data(), static_cast<int64_t>(single_a.size()), n, missing.data(), 0))
                return rc;
            for (int32_t c : missing) ++st->w_absent[c];
        }

        phase("closed forms");
        // ---- bitmap rows: genome-major, bit-sliced, superblocks of rows of similar density, longest walks first ----
        std::vector<int64_t> list_gene;
        for (int64_t g : general) {
            const int64_t m = m_of(g), folded = std::min<int64_t>(m, n - m);
            if (long_threshold > 0 && folded >= long_threshold) st->long_gene.push_back(g);
            else list_gene.push_back(g);
        }
        const long long n_long = static_cast<long long>(st->long_gene.size());
        if (slice_words == 0) slice_words = slice_words_for(n_long);
        const long long sb_rows = static_cast<long long>(SLICE_ROWS) * slice_words;
        const long long n_super = (n_long + sb_rows - 1) / sb_rows;
        long long nnz_long = 0;
        if (n_long) {
            std::stable_sort(st->long_gene.begin(), st->long_gene.end(), [&](int64_t a, int64_t b) {
                return std::min<int64_t>(m_of(a), n - m_of(a)) < std::min<int64_t>(m_of(b), n - m_of(b));
            });
            for (int64_t g : st->long_gene) nnz_long += m_of(g);
            st->bits.assign(static_cast<size_t>(n_super) * n * (sb_rows / 32), 0u);
            if (int rc = pgx::pgx_plan_build_bitmap(indptr.data(), indices.data(), st->long_gene.data(), n_long, n, slice_words, st->bits.data(), 0))
                return rc;
        }

        phase("bitmap rows");
        // ---- list rows: by chunk count (descending), list kind, length (descending) ... ----
        const long long n_rows = static_cast<long long>(list_gene.size());
        std::vector<uint8_t> use_abs(static_cast<size_t>(n_rows));
        std::vector<int64_t> length(static_cast<size_t>(n_rows)), n_chunk(static_cast<size_t>(n_rows));
        {
            std::vector<int64_t> order(static_cast<size_t>(n_rows));
            std::iota(order.begin(), order.end(), 0);
            auto len_of = [&](int64_t g) { return std::min<int64_t>(m_of(g), n - m_of(g)); };
            auto abs_of = [&](int64_t g) { return m_of(g) > n - m_of(g); };
            std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) {
                const int64_t ga = list_gene[a], gb = list_gene[b];
                const int64_t ca = (len_of(ga) + CHUNK - 1) / CHUNK, cb = (len_of(gb) + CHUNK - 1) / CHUNK;
                if (ca != cb) return ca > cb;
                if (abs_of(ga) != abs_of(gb)) return !abs_of(ga);
                return len_of(ga) > len_of(gb);
            });
            std::vector<int64_t> sorted(static_cast<size_t>(n_rows));
            for (long long i = 0; i < n_rows; ++i) sorted[i] = list_gene[order[i]];
            list_gene.swap(sorted);
            for (long long i = 0; i < n_rows; ++i) {
                const int64_t g = list_gene[i];
                use_abs[i] = abs_of(g);
                length[i] = len_of(g);
                n_chunk[i] = (length[i] + CHUNK - 1) / CHUNK;
            }
        }
        phase("list rows: sort");
        // ... and, inside a (chunk count, kind) class, in the order that balances the bank residues of every
        // wavefront group (PGX_NO_ROW_BALANCE=1 keeps the rows sorted by length)
        const char *no_balance = getenv("PGX_NO_ROW_BALANCE");
        if (n_rows && !(no_balance && !strcmp(no_balance, "1"))) {
            std::vector<int64_t> class_key(static_cast<size_t>(n_rows)), order(static_cast<size_t>(n_rows));
            for (long long i = 0; i < n_rows; ++i) class_key[i] = n_chunk[i] * 2 + use_abs[i];
            if (int rc = pgx::pgx_plan_balance_rows(indptr.data(), indices.data(), list_gene.data(), use_abs.data(), class_key.data(), n_rows, n,
                                               modulus, std::max(BALANCE_WINDOW, 4 * modulus), order.data(), 0))
                return rc;
            std::vector<int64_t> g2(static_cast<size_t>(n_rows)), l2(static_cast<size_t>(n_rows)), c2(static_cast<size_t>(n_rows));
            std::vector<uint8_t> a2(static_cast<size_t>(n_rows));
            for (long long i = 0; i < n_rows; ++i) {
                g2[i] = list_gene[order[i]];
                l2[i] = length[order[i]];
                c2[i] = n_chunk[order[i]];
                a2[i] = use_abs[order[i]];
            }
            list_gene.swap(g2);
            length.swap(l2);
            n_chunk.swap(c2);
            use_abs.swap(a2);
        }
        phase("list rows: residue balance");
        std::vector<int64_t> ptr(static_cast<size_t>(n_rows) + 1, 0);
        for (long long i = 0; i < n_rows; ++i) ptr[i + 1] = ptr[i] + length[i];
        if (ptr[n_rows] >= (1ll << 31)) return pgx::fail(PGX_ERR_UNSUPPORTED, "list rows too large for int32 offsets");
        std::vector<int32_t> flat(static_cast<size_t>(ptr[n_rows]));
        long long nnz_list = 0;
        if (n_rows) {
            if (int rc = pgx::pgx_plan_folded_lists(indptr.data(), indices.data(), list_gene.data(), use_abs.data(), ptr.data(), n_rows, n, flat.data(), 0))
                return rc;
            for (int64_t g : list_gene) nnz_list += m_of(g);
        }

        phase("list rows: folded lists");
        // ---- sub-blocks of 32 rows (one lane per row), streamed by a warp in runs of about RUN_LANE_CHUNKS iterations ----
        if (n_rows) {
            std::vector<int64_t> cls_start;
            for (long long i = 0; i < n_rows; ++i)
                if (i == 0 || n_chunk[i] != n_chunk[i - 1] || use_abs[i] != use_abs[i - 1]) cls_start.push_back(i);
            cls_start.push_back(n_rows);
            long long total_iters = 0;
            for (size_t c = 0; c + 1 < cls_start.size(); ++c)
                total_iters += (cls_start[c + 1] - cls_start[c] + 31) / 32 * n_chunk[cls_start[c]];
            const long long run_budget = std::min<long long>(RUN_LANE_CHUNKS, std::max<long long>(2, total_iters / RUN_TARGET_TASKS));
            std::vector<int64_t> b_first_row, b_rows, b_nch, b_abs, b_run;
            long long run_id = 0;
            for (size_t c = 0; c + 1 < cls_start.size(); ++c) {
                const int64_t r0 = cls_start[c], r1 = cls_start[c + 1], nch = n_chunk[r0];
                const long long per_run = std::max<long long>(1, run_budget / nch);
                long long i = 0;
                for (int64_t first = r0; first < r1; first += 32, ++i) {
                    b_first_row.push_back(first);
                    b_rows.push_back(std::min<int64_t>(32, r1 - first));
                    b_nch.push_back(nch);
                    b_abs.push_back(use_abs[r0]);
                    b_run.push_back(run_id + i / per_run);
                }
                run_id = b_run.back() + 1;
            }
            const long long n_blocks = static_cast<long long>(b_nch.size());
            std::vector<int64_t> block_first(static_cast<size_t>(n_blocks));
            long long at = 0, max_nch = 0;
            for (long long b = 0; b < n_blocks; ++b) {
                block_first[b] = at;
                at += b_nch[b] * 32;
                max_nch = std::max<long long>(max_nch, b_nch[b]);
            }
            if (at * CHUNK >= (1ll << 31)) return pgx::fail(PGX_ERR_UNSUPPORTED, "list rows too large for int32 chunk offsets");
            if (max_nch >= (1 << 16)) return pgx::fail(PGX_ERR_UNSUPPORTED, "list row too long for the task descriptor");
            st->chunks.resize(static_cast<size_t>(at) * CHUNK);
            if (int rc = pgx::pgx_plan_bank_order(flat.data(), ptr.data(), n_rows, block_first.data(), b_nch.data(), b_first_row.data(), b_rows.data(),
                                             n_blocks, n, modulus, COLOUR_MAX_CHUNKS, st->chunks.data(), 0))
                return rc;
            phase("list rows: bank order");
            // one task per run; costly runs first: dynamic fetching then ends on cheap ones
            struct Task {
                int32_t v[4];
                long long cost;
            };
            std::vector<Task> tasks;
            for (long long b = 0; b < n_blocks;) {
                long long e = b, rows = 0;
                while (e < n_blocks && b_run[e] == b_run[b]) rows += b_rows[e++];
                Task t;
                t.v[0] = static_cast<int32_t>(block_first[b]);
                t.v[1] = static_cast<int32_t>(b_nch[b] | (b_abs[b] << 24));
                t.v[2] = static_cast<int32_t>(b_first_row[b]);
                t.v[3] = static_cast<int32_t>(rows);
                t.cost = b_nch[b] * ((rows + 31) / 32);
                tasks.push_back(t);
                b = e;
            }
            std::stable_sort(tasks.begin(), tasks.end(), [](const Task &a, const Task &b) { return a.cost > b.cost; });
            st->tasks.resize(tasks.size() * 4);
            for (size_t t = 0; t < tasks.size(); ++t) memcpy(&st->tasks[t * 4], tasks[t].v, sizeof(tasks[t].v));
        }
        st->sorted_idx.resize(flat.size());
        for (size_t i = 0; i < flat.size(); ++i) st->sorted_idx[i] = static_cast<uint16_t>(flat[i]);
        st->sorted_ptr.resize(static_cast<size_t>(n_rows) + 1);
        for (long long i = 0; i <= n_rows; ++i) st->sorted_ptr[i] = static_cast<int32_t>(ptr[i]);
        st->row_gene = list_gene;
        st->row_len.resize(static_cast<size_t>(n_rows));
        for (long long i = 0; i < n_rows; ++i) st->row_len[i] = static_cast<int32_t>(length[i]);
        st->row_absent = use_abs;

        phase("tasks, sorted copy");
        pgx_host_plan &v = st->view;
        memset(&v, 0, sizeof(v));
        v.owner = st;
        v.chunks = st->chunks.data();
        v.tasks = st->tasks.data();
        v.sorted_idx = st->sorted_idx.data();
        v.sorted_ptr = st->sorted_ptr.data();
        v.bits = st->bits.data();
        v.colsum = st->colsum.data();
        v.w_present = st->w_present.data();
        v.w_absent = st->w_absent.data();
        v.row_gene = st->row_gene.data();
        v.row_len = st->row_len.data();
        v.row_absent = st->row_absent.data();
        v.long_gene = st->long_gene.data();
        v.nnz = nnz;
        v.nnz_list = nnz_list;
        v.nnz_long = nnz_long;
        v.n_chunks = static_cast<int64_t>(st->chunks.size() / CHUNK);
        v.n_bits_words = static_cast<int64_t>(st->bits.size());
        v.n_sorted = static_cast<int64_t>(st->sorted_idx.size());
        v.n_genomes = n;
        v.n_genes = n_genes;
        v.n_rows = static_cast<int32_t>(n_rows);
        v.n_tasks = static_cast<int32_t>(st->tasks.size() / 4);
        v.n_long = static_cast<int32_t>(n_long);
        v.n_superblocks = static_cast<int32_t>(n_super);
        v.perms_per_cta = perms_per_cta;
        v.slice_words = slice_words;
        v.long_threshold = long_threshold;
        v.max_colsum = st->colsum.empty() ? 0 : *std::max_element(st->colsum.begin(), st->colsum.end());
        v.n_empty = static_cast<int32_t>(n_empty);
        v.n_full = static_cast<int32_t>(n_full);
    } catch (const std::bad_alloc &) {
        return pgx::fail(PGX_ERR_INVALID, "out of memory while planning the table");
    }
    guard.p = nullptr;
    *out = &st->view;
    return PGX_OK;
}
