// Threaded host steps of the planner (pgx_host_plan_create, pgx_plan_build.cpp): the table ingest (COO -> canonical
// gene-major CSR), the folded lists, the missing genome of the single-absence rows, the residue-balanced order of the
// list rows, the bank ordering of their entries and the bit-sliced bitmap of the long rows.  They are internal to the
// library (namespace pgx); oracle/plan_np.py restates every step in numpy and the tests compare the two plans bit for
// bit.  Only pgx_plan_all_equal_u64 is part of the C ABI.  Nothing here touches the GPU.
#include <limits.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#if defined(__linux__)
#include <sys/mman.h>
#endif

#include <algorithm>
#include <atomic>
#include <memory>
#include <new>
#include <thread>
#include <vector>

#include "pgx.h"

namespace pgx {
int fail(int code, const char *fmt, ...);

namespace {

constexpr int MAX_MOD = 32;

struct Group {
    int r_mod, n_steps;
    int cnt[MAX_MOD][MAX_MOD];             // [lane][residue]
    std::vector<int8_t> res_at, pad_res;   // [lane][step]
};

// oracle/plan_np.py, _colour_groups, for one group: greedy edge colouring of lanes x residues with n_steps colours.
// Same choices as the numpy specification (first maximum wins, stable order of the lanes), found with
// less work: the residues a lane still holds are a bit mask, so a lane scans only those; the lane order
// by slack is kept between steps (a lane's slack changes by at most one per step) and repaired by an
// insertion sort on the unique keys slack * 32 + lane.
void colour(Group &g)
{
    const int R = g.r_mod, S = g.n_steps;
    int cnt[MAX_MOD][MAX_MOD], colload[MAX_MOD], rem[MAX_MOD], order[MAX_MOD];
    uint32_t holds[MAX_MOD];                           // bit r: the lane still has entries of residue r
    memcpy(cnt, g.cnt, sizeof(cnt));
    for (int r = 0; r < R; ++r) {
        colload[r] = 0;
        for (int l = 0; l < R; ++l) colload[r] += cnt[l][r];
    }
    for (int l = 0; l < R; ++l) {
        rem[l] = 0;
        holds[l] = 0;
        order[l] = l;
        for (int r = 0; r < R; ++r) {
            rem[l] += cnt[l][r];
            if (cnt[l][r] > 0) holds[l] |= 1u << r;
        }
    }
    for (int s = 0; s < S; ++s) {
        uint32_t taken = 0;
        const int steps_left = S - s;
        // rows with the least slack choose first: ascending (steps_left - rem, lane), i.e. descending rem, then lane
        for (int a = 1; a < R; ++a) {
            const int lane = order[a];
            int at = a;
            while (at > 0 && (rem[order[at - 1]] < rem[lane] || (rem[order[at - 1]] == rem[lane] && order[at - 1] > lane))) {
                order[at] = order[at - 1];
                --at;
            }
            order[at] = lane;
        }
        for (int t = 0; t < R; ++t) {
            const int lane = order[t];
            int choice = -1;
            long best = -1;
            for (uint32_t m = holds[lane] & ~taken; m; m &= m - 1) {   // argmax of colload * 1024 + cnt, first max wins
                const int r = __builtin_ctz(m);
                const long score = static_cast<long>(colload[r]) * 1024 + cnt[lane][r];
                if (score > best) {
                    best = score;
                    choice = r;
                }
            }
            if (choice < 0 && rem[lane] >= steps_left && rem[lane] > 0) {   // forced: no free residue, no slack left
                int top = -1;
                for (uint32_t m = holds[lane]; m; m &= m - 1) {
                    const int r = __builtin_ctz(m);
                    if (cnt[lane][r] > top) {
                        top = cnt[lane][r];
                        choice = r;
                    }
                }
            }
            if (choice >= 0) {
                g.res_at[lane * S + s] = static_cast<int8_t>(choice);
                if (--cnt[lane][choice] == 0) holds[lane] &= ~(1u << choice);
                --colload[choice];
                --rem[lane];
                taken |= 1u << choice;
            }
        }
        // pads: the k-th idle lane of the group takes the group's k-th unused residue
        int free_order[MAX_MOD], n_free = 0;
        for (int r = 0; r < R; ++r)
            if (!(taken >> r & 1)) free_order[n_free++] = r;
        for (int r = 0; r < R; ++r)
            if (taken >> r & 1) free_order[n_free++] = r;
        int rank = 0;
        for (int l = 0; l < R; ++l) {
            if (g.res_at[l * S + s] < 0) {
                g.pad_res[l * S + s] = static_cast<int8_t>(free_order[std::min(rank, R - 1)]);
                ++rank;
            }
        }
    }
}

// oracle/plan_np.py, _positional_groups, for one group.
void positional(Group &g)
{
    const int R = g.r_mod, S = g.n_steps;
    for (int l = 0; l < R; ++l) {
        int cap[MAX_MOD] = {0};
        for (int s = 0; s < S; ++s) {
            const int want = (s + l) % R;
            ++cap[want];
            g.pad_res[l * S + s] = static_cast<int8_t>(want);
            if (s / R < g.cnt[l][want]) g.res_at[l * S + s] = static_cast<int8_t>(want);
        }
        int s_free = 0;
        for (int r = 0; r < R; ++r) {
            for (int extra = std::max(g.cnt[l][r] - cap[r], 0); extra > 0; --extra) {
                while (s_free < S && g.res_at[l * S + s_free] >= 0) ++s_free;
                if (s_free < S) g.res_at[l * S + s_free] = static_cast<int8_t>(r);
            }
        }
    }
}

}  // namespace

// The bank ordering of the list rows (oracle/plan_np.py, _bank_ordered_chunks): which entry of a list row sits at which
// gather step, so that the lanes of a shared-memory wavefront of list_kernel hit distinct banks of the rank table.  The
// same greedy edge colouring, tie breaks and output as the numpy specification, as plain loops over the sub-blocks,
// spread over host threads; the layout is the one struct pgx_plan documents.
//   flat / ptr        : sorted folded lists of the n_rows list rows, concatenated (int32) / offsets (int64)
//   block_*           : per sub-block of 32 rows: first chunk, chunks per row, first row, rows (int64 [n_blocks])
//   modulus           : lanes per 128-byte wavefront: 8, 16 or 32 (= 64 / perms_per_cta, capped)
//   colour_max_chunks : rows of more chunks use the cheap positional order instead of the edge colouring
//   chunks            : out, uint16 [sum(block_nch) * 32 * 8]
//   n_threads         : host threads (0 = choose)
int pgx_plan_bank_order(const int32_t *flat, const int64_t *ptr, int64_t n_rows,
                                   const int64_t *block_first, const int64_t *block_nch,
                                   const int64_t *block_first_row, const int64_t *block_rows, int64_t n_blocks,
                                   int32_t n_genomes, int32_t modulus, int32_t colour_max_chunks,
                                   uint16_t *chunks, int32_t n_threads)
{
    if (!ptr || !block_first || !block_nch || !block_first_row || !block_rows || (!chunks && n_blocks > 0))
        return pgx::fail(PGX_ERR_INVALID, "null pointer passed to pgx_plan_bank_order");
    if (modulus != 8 && modulus != 16 && modulus != 32) return pgx::fail(PGX_ERR_INVALID, "modulus must be 8, 16 or 32");
    if (n_rows < 0 || n_blocks < 0) return pgx::fail(PGX_ERR_INVALID, "negative size");
    const int R = modulus;
    std::atomic<long long> next{0};
    std::atomic<int> bad{0};
    auto work = [&]() {
        Group g;
        g.r_mod = R;
        std::vector<int32_t> byres;                    // entries of one row, grouped by residue, index order kept
        for (;;) {
            const long long b = next.fetch_add(1);
            if (b >= n_blocks) return;
            const int S = static_cast<int>(block_nch[b]) * 8;
            g.n_steps = S;
            g.res_at.assign(static_cast<size_t>(R) * S, -1);
            g.pad_res.assign(static_cast<size_t>(R) * S, 0);
            for (int grp = 0; grp < 32 / R; ++grp) {
                std::fill(g.res_at.begin(), g.res_at.end(), static_cast<int8_t>(-1));
                std::fill(g.pad_res.begin(), g.pad_res.end(), static_cast<int8_t>(0));
                memset(g.cnt, 0, sizeof(g.cnt));
                for (int l = 0; l < R; ++l) {
                    const long long lane32 = grp * R + l;
                    if (lane32 >= block_rows[b]) continue;
                    const long long row = block_first_row[b] + lane32;
                    if (row >= n_rows || ptr[row + 1] - ptr[row] > S) {
                        bad.store(1);
                        continue;
                    }
                    for (long long e = ptr[row]; e < ptr[row + 1]; ++e) ++g.cnt[l][flat[e] % R];
                }
                if (block_nch[b] <= colour_max_chunks) colour(g); else positional(g);
                for (int l = 0; l < R; ++l) {
                    const long long lane32 = grp * R + l;
                    const bool real = lane32 < block_rows[b];
                    int start[MAX_MOD + 1];
                    start[0] = 0;
                    for (int r = 0; r < R; ++r) start[r + 1] = start[r] + g.cnt[l][r];
                    if (real) {
                        const long long row = block_first_row[b] + lane32;
                        byres.resize(static_cast<size_t>(start[R]));
                        int at[MAX_MOD];
                        for (int r = 0; r < R; ++r) at[r] = start[r];
                        for (long long e = ptr[row]; e < ptr[row + 1]; ++e) byres[at[flat[e] % R]++] = flat[e];
                    }
                    int used[MAX_MOD] = {0};
                    for (int s = 0; s < S; ++s) {
                        const long long addr = ((block_first[b] + static_cast<long long>(s >> 3) * 32 + lane32) << 3) + (s & 7);
                        const int r = g.res_at[l * S + s];
                        if (r >= 0 && real && used[r] < g.cnt[l][r]) {
                            chunks[addr] = static_cast<uint16_t>(byres[start[r] + used[r]++]);
                        } else {
                            const int pad = g.pad_res[l * S + s];
                            chunks[addr] = static_cast<uint16_t>(n_genomes + (((pad - n_genomes) % R) + R) % R);
                        }
                    }
                    for (int r = 0; r < R; ++r)
                        if (real && used[r] != g.cnt[l][r]) bad.store(1);
                }
            }
        }
    };
    int threads = n_threads > 0 ? n_threads : static_cast<int>(std::min(16u, std::max(1u, std::thread::hardware_concurrency())));
    threads = static_cast<int>(std::min<long long>(threads, std::max<long long>(1, n_blocks / 64)));
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; ++t) pool.emplace_back(work);
    work();
    for (auto &th : pool) th.join();
    if (bad.load()) return pgx::fail(PGX_ERR_INVALID, "inconsistent list rows passed to pgx_plan_bank_order");
    return PGX_OK;
}

// The bit-sliced bitmap of the long rows (struct pgx_plan, d_bits): bit b of word
// (sb * n_genomes + c) * 32 W + w is the presence of long row sb * 1024 W + 32 w + b in genome c.
// ``bits`` must be zero-initialised; superblocks are independent and spread over host threads.
int pgx_plan_build_bitmap(const int64_t *indptr, const int32_t *indices, const int64_t *long_gene,
                                     int64_t n_long, int32_t n_genomes, int32_t slice_words, uint32_t *bits,
                                     int32_t n_threads)
{
    if (n_long < 0 || n_genomes < 1 || (slice_words != 1 && slice_words != 2 && slice_words != 4))
        return pgx::fail(PGX_ERR_INVALID, "bad shape passed to pgx_plan_build_bitmap");
    if (n_long == 0) return PGX_OK;
    if (!indptr || !indices || !long_gene || !bits) return pgx::fail(PGX_ERR_INVALID, "null pointer passed to pgx_plan_build_bitmap");
    const long long sb_rows = 1024ll * slice_words, line = 32ll * slice_words;
    const long long n_super = (n_long + sb_rows - 1) / sb_rows;
    std::atomic<long long> next{0};
    std::atomic<int> bad{0};
    auto work = [&]() {
        for (;;) {
            const long long sb = next.fetch_add(1);
            if (sb >= n_super) return;
            uint32_t *base = bits + static_cast<size_t>(sb) * n_genomes * line;
            const long long r1 = std::min<long long>(n_long, (sb + 1) * sb_rows);
            for (long long r = sb * sb_rows; r < r1; ++r) {
                const long long local = r - sb * sb_rows, gene = long_gene[r];
                const uint32_t bit = 1u << (local & 31);
                const long long word = local >> 5;
                for (long long e = indptr[gene]; e < indptr[gene + 1]; ++e) {
                    const int32_t c = indices[e];
                    if (c < 0 || c >= n_genomes) {
                        bad.store(1);
                        continue;
                    }
                    base[static_cast<size_t>(c) * line + word] |= bit;
                }
            }
        }
    };
    int threads = n_threads > 0 ? n_threads : static_cast<int>(std::min(16u, std::max(1u, std::thread::hardware_concurrency())));
    threads = static_cast<int>(std::min<long long>(threads, n_super));
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; ++t) pool.emplace_back(work);
    work();
    for (auto &th : pool) th.join();
    if (bad.load()) return pgx::fail(PGX_ERR_INVALID, "genome index out of range in pgx_plan_build_bitmap");
    return PGX_OK;
}

// ---------------------------------------------------------------------------------------------
// Table ingest: ``df_genes.data`` (scipy COO, gene x genome) -> canonical gene-major CSR, the
// folded lists of the list rows and the missing genome of the single-absence rows.  These replace
// scipy's single-threaded coo_tocsr / sum_duplicates / sort_indices and a few O(nnz) numpy
// gathers of the specification (oracle/plan_np.py) with threaded loops.
// ---------------------------------------------------------------------------------------------
namespace {

int host_threads(int32_t wanted, long long units)
{
    int threads = wanted > 0 ? wanted : static_cast<int>(std::min(16u, std::max(1u, std::thread::hardware_concurrency())));
    return static_cast<int>(std::max<long long>(1, std::min<long long>(threads, units)));
}

// Large buffers that are about to be filled for the first time: ask for huge pages (one page fault per
// 2 MB instead of one per 4 KB; a hint, ignored where transparent huge pages are off).
void want_huge_pages(void *ptr, size_t bytes)
{
#if defined(__linux__) && defined(MADV_HUGEPAGE)
    if (getenv("PGX_NO_HUGEPAGES")) return;
    const uintptr_t page = 2u << 20;
    const uintptr_t lo = (reinterpret_cast<uintptr_t>(ptr) + page - 1) & ~(page - 1);
    const uintptr_t hi = (reinterpret_cast<uintptr_t>(ptr) + bytes) & ~(page - 1);
    if (hi > lo) madvise(reinterpret_cast<void *>(lo), hi - lo, MADV_HUGEPAGE);
#else
    (void)ptr;
    (void)bytes;
#endif
}

struct FreeDeleter {
    void operator()(void *p) const { free(p); }
};

template <typename F>
void run_threads(int threads, F &&body)
{
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; ++t) pool.emplace_back([&body, t]() { body(t); });
    body(0);
    for (auto &th : pool) th.join();
}

}  // namespace

// COO of a BINARY table (every stored value is 1; the caller checks) -> CSR with sorted rows, as a
// two-level counting sort that keeps the input order inside a gene (column-sorted input -- what the
// reference's producers and scipy's own conversions emit -- then needs no sorting afterwards):
//   pass 0  every thread histograms its slice of the entries over blocks of 2^shift genes (<= 512 blocks);
//   pass A  every thread appends its entries, packed as (gene - block start) << 16 | genome, to its own
//           part of each block of a temporary array: a few hundred sequential write streams per thread;
//   pass B  inside the blocks, again a counting sort, over pieces of at most 2^21 entries so that a block
//           holding half of the table (the core genes of a pangenome sit next to each other) still spreads
//           over all threads: count per (piece, gene), prefix per block, scatter per piece -- the write set
//           of a piece is one cache line per gene of its block, cache-resident;
//   pass C  per gene (chunks balanced by entries): already ascending?  Otherwise sort -- long rows through a
//           genome bitmap, short ones with std::sort -- and count duplicates; column sums.
// Duplicate (gene, genome) pairs are kept and counted in *n_duplicates: scipy would sum them to 2, i.e.
// a non-binary table.
int pgx_plan_coo_to_csr(const int32_t *row, const int32_t *col, int64_t nnz, int32_t n_genes,
                                   int32_t n_genomes, int64_t *indptr, int32_t *indices, int32_t *colsum,
                                   int64_t *n_duplicates, int32_t n_threads)
{
    if (nnz < 0 || n_genes < 0 || n_genomes < 0) return pgx::fail(PGX_ERR_INVALID, "negative size passed to pgx_plan_coo_to_csr");
    if (n_genomes > 65536) return pgx::fail(PGX_ERR_UNSUPPORTED, "pgx_plan_coo_to_csr packs genome indices in 16 bits");
    if (!indptr || !colsum || !n_duplicates || (nnz > 0 && (!row || !col || !indices)))
        return pgx::fail(PGX_ERR_INVALID, "null pointer passed to pgx_plan_coo_to_csr");
    *n_duplicates = 0;
    std::fill(colsum, colsum + n_genomes, 0);
    std::fill(indptr, indptr + n_genes + 1, 0);
    if (nnz == 0) return PGX_OK;
    if (n_genes == 0) return pgx::fail(PGX_ERR_INVALID, "entries in a table without genes");
    int shift = 6;
    while (shift < 16 && ((static_cast<int64_t>(n_genes) + (1ll << shift) - 1) >> shift) > 512) ++shift;
    const int64_t block_genes = 1ll << shift;
    const int64_t n_blocks = (static_cast<int64_t>(n_genes) + block_genes - 1) >> shift;
    const int threads = host_threads(n_threads, std::max<long long>(1, nnz / (1 << 16)));
    std::vector<int64_t> hist(static_cast<size_t>(threads) * n_blocks, 0);      // [thread][block], then write offsets
    std::vector<int64_t> block_start(n_blocks + 1, 0);
    std::atomic<int> bad{0};
    auto slice = [&](int t, int64_t *lo, int64_t *hi) {
        *lo = nnz * t / threads;
        *hi = nnz * (t + 1) / threads;
    };
    run_threads(threads, [&](int t) {
        int64_t lo, hi;
        slice(t, &lo, &hi);
        int64_t *h = hist.data() + static_cast<size_t>(t) * n_blocks;
        bool oob = false;
        for (int64_t i = lo; i < hi; ++i) {
            const uint32_t r = static_cast<uint32_t>(row[i]);
            if (r >= static_cast<uint32_t>(n_genes)) {
                oob = true;
                continue;
            }
            ++h[r >> shift];
        }
        if (oob) bad.store(1);
    });
    if (bad.load()) return pgx::fail(PGX_ERR_INVALID, "gene index out of range in the COO table");
    for (int64_t b = 0; b < n_blocks; ++b) {
        int64_t at = block_start[b];
        for (int t = 0; t < threads; ++t) {
            const int64_t c = hist[static_cast<size_t>(t) * n_blocks + b];
            hist[static_cast<size_t>(t) * n_blocks + b] = at;
            at += c;
        }
        block_start[b + 1] = at;
    }
    void *packed_mem = nullptr;
    if (posix_memalign(&packed_mem, 2u << 20, sizeof(uint32_t) * static_cast<size_t>(nnz)) != 0 || !packed_mem)
        return pgx::fail(PGX_ERR_INVALID, "out of host memory in pgx_plan_coo_to_csr");
    std::unique_ptr<uint32_t, FreeDeleter> packed_owner(static_cast<uint32_t *>(packed_mem));
    uint32_t *packed = packed_owner.get();
    want_huge_pages(packed, sizeof(uint32_t) * static_cast<size_t>(nnz));
    want_huge_pages(indices, sizeof(int32_t) * static_cast<size_t>(nnz));
    run_threads(threads, [&](int t) {
        int64_t lo, hi;
        slice(t, &lo, &hi);
        int64_t *at = hist.data() + static_cast<size_t>(t) * n_blocks;
        const uint32_t low = static_cast<uint32_t>(block_genes - 1);
        bool oob = false;
        for (int64_t i = lo; i < hi; ++i) {
            const uint32_t r = static_cast<uint32_t>(row[i]), c = static_cast<uint32_t>(col[i]);
            if (c >= static_cast<uint32_t>(n_genomes)) {
                oob = true;
                continue;
            }
            packed[at[r >> shift]++] = (r & low) << 16 | c;
        }
        if (oob) bad.store(1);
    });
    if (bad.load()) return pgx::fail(PGX_ERR_INVALID, "genome index out of range in the COO table");

    // pass B: pieces of the blocks
    struct Piece { int64_t block, lo, hi; };
    const int64_t piece_entries = 1ll << 21;
    std::vector<Piece> pieces;
    std::vector<int64_t> first_piece(n_blocks + 1, 0);
    for (int64_t b = 0; b < n_blocks; ++b) {
        first_piece[b] = static_cast<int64_t>(pieces.size());
        for (int64_t lo = block_start[b]; lo < block_start[b + 1]; lo += piece_entries)
            pieces.push_back({b, lo, std::min(block_start[b + 1], lo + piece_entries)});
    }
    first_piece[n_blocks] = static_cast<int64_t>(pieces.size());
    const int64_t n_pieces = static_cast<int64_t>(pieces.size());
    std::vector<int64_t> piece_pos(static_cast<size_t>(n_pieces) * block_genes);    // [piece][gene of block]: count, then offset
    std::atomic<long long> next{0};
    run_threads(threads, [&](int) {
        for (;;) {
            const long long k = next.fetch_add(1);
            if (k >= n_pieces) return;
            int64_t *cnt = piece_pos.data() + static_cast<size_t>(k) * block_genes;
            std::fill(cnt, cnt + block_genes, 0);
            for (const uint32_t *p = packed + pieces[k].lo, *e = packed + pieces[k].hi; p < e; ++p) ++cnt[*p >> 16];
        }
    });
    next.store(0);
    run_threads(threads, [&](int) {
        for (;;) {
            const long long b = next.fetch_add(1);
            if (b >= n_blocks) return;
            const int64_t g0 = b << shift, g1 = std::min<int64_t>(n_genes, g0 + block_genes);
            int64_t at = block_start[b];
            for (int64_t g = g0; g < g1; ++g) {
                for (int64_t k = first_piece[b]; k < first_piece[b + 1]; ++k) {
                    int64_t &slot = piece_pos[static_cast<size_t>(k) * block_genes + (g - g0)];
                    const int64_t c = slot;
                    slot = at;
                    at += c;
                }
                indptr[g + 1] = at;            // indptr[g0] belongs to the previous block (indptr[0] = 0)
            }
        }
    });
    next.store(0);
    std::vector<std::vector<int32_t>> part_colsum(threads);
    run_threads(threads, [&](int t) {
        std::vector<int32_t> &cs = part_colsum[t];
        cs.assign(n_genomes, 0);
        for (;;) {
            const long long k = next.fetch_add(1);
            if (k >= n_pieces) return;
            int64_t *pos = piece_pos.data() + static_cast<size_t>(k) * block_genes;
            for (const uint32_t *p = packed + pieces[k].lo, *e = packed + pieces[k].hi; p < e; ++p) {
                const uint32_t c = *p & 0xffffu;
                indices[pos[*p >> 16]++] = static_cast<int32_t>(c);
                ++cs[c];
            }
        }
    });
    for (int t = 0; t < threads; ++t)
        for (size_t c = 0; c < part_colsum[t].size(); ++c) colsum[c] += part_colsum[t][c];

    // pass C: canonical rows, gene chunks of about 2^18 entries
    std::vector<int64_t> chunk_first;
    for (int64_t g = 0; g < n_genes;) {
        chunk_first.push_back(g);
        const int64_t limit = indptr[g] + (1ll << 18);
        ++g;
        while (g < n_genes && indptr[g + 1] <= limit) ++g;
    }
    chunk_first.push_back(n_genes);
    const int64_t n_chunks = static_cast<int64_t>(chunk_first.size()) - 1;
    std::atomic<long long> dups{0};
    next.store(0);
    run_threads(threads, [&](int) {
        std::vector<uint64_t> seen((static_cast<size_t>(n_genomes) + 63) / 64, 0);
        long long d = 0;
        for (;;) {
            const long long k = next.fetch_add(1);
            if (k >= n_chunks) break;
            for (int64_t g = chunk_first[k]; g < chunk_first[k + 1]; ++g) {
                int32_t *a = indices + indptr[g], *e = indices + indptr[g + 1];
                bool sorted = true;
                for (int32_t *p = a + 1; p < e; ++p) {
                    if (p[0] <= p[-1]) {
                        sorted = false;
                        break;
                    }
                }
                if (sorted) continue;
                if (static_cast<size_t>(e - a) * 16 < seen.size()) {
                    std::sort(a, e);
                    for (int32_t *p = a + 1; p < e; ++p) d += p[0] == p[-1];
                    continue;
                }
                // long row: mark the genomes in a bitmap, re-emit them ascending; duplicates follow the
                // distinct genomes (still counted, the caller rejects the table anyway)
                int32_t *dup_tail = e;
                for (int32_t *p = a; p < e; ++p) {
                    const uint32_t c = static_cast<uint32_t>(*p);
                    if (seen[c >> 6] >> (c & 63) & 1) {
                        ++d;
                        --dup_tail;               // remember how many slots the duplicates need
                    }
                    seen[c >> 6] |= 1ull << (c & 63);
                }
                const long long n_dup = e - dup_tail;
                int32_t last = 0;
                int32_t *w = a;
                for (size_t word = 0; word < seen.size(); ++word) {
                    uint64_t bits = seen[word];
                    seen[word] = 0;
                    while (bits) {
                        last = static_cast<int32_t>(word * 64 + __builtin_ctzll(bits));
                        *w++ = last;
                        bits &= bits - 1;
                    }
                }
                for (long long x = 0; x < n_dup; ++x) *w++ = last;      // keeps nnz; content is void once d > 0
            }
        }
        dups.fetch_add(d);
    });
    *n_duplicates = dups.load();
    return PGX_OK;
}

// oracle/plan_np.py, _folded_lists: row r of the list rows is gene genes[r]; its folded list -- the present genomes
// (use_abs[r] == 0) or the absent ones -- goes to flat[ptr[r] .. ptr[r + 1]), ascending.
int pgx_plan_folded_lists(const int64_t *indptr, const int32_t *indices, const int64_t *genes,
                                     const uint8_t *use_abs, const int64_t *ptr, int64_t n_rows,
                                     int32_t n_genomes, int32_t *flat, int32_t n_threads)
{
    if (n_rows < 0 || n_genomes < 1) return pgx::fail(PGX_ERR_INVALID, "bad shape passed to pgx_plan_folded_lists");
    if (n_rows == 0) return PGX_OK;
    if (!indptr || !genes || !use_abs || !ptr || (ptr[n_rows] > 0 && (!indices || !flat)))
        return pgx::fail(PGX_ERR_INVALID, "null pointer passed to pgx_plan_folded_lists");
    const long long grain = 512;
    std::atomic<long long> next{0};
    std::atomic<int> bad{0};
    const int threads = host_threads(n_threads, (n_rows + grain - 1) / grain);
    run_threads(threads, [&](int) {
        for (;;) {
            const long long r0 = next.fetch_add(grain);
            if (r0 >= n_rows) return;
            const long long r1 = std::min<long long>(n_rows, r0 + grain);
            for (long long r = r0; r < r1; ++r) {
                const int32_t *a = indices + indptr[genes[r]], *e = indices + indptr[genes[r] + 1];
                int32_t *out = flat + ptr[r];
                const long long want = ptr[r + 1] - ptr[r];
                if (!use_abs[r]) {
                    if (e - a != want) {
                        bad.store(1);
                        continue;
                    }
                    memcpy(out, a, sizeof(int32_t) * static_cast<size_t>(want));
                } else {
                    if (n_genomes - (e - a) != want) {
                        bad.store(1);
                        continue;
                    }
                    int32_t c = 0;
                    for (const int32_t *p = a; p < e; ++p) {
                        for (; c < *p; ++c) *out++ = c;
                        c = *p + 1;
                    }
                    for (; c < n_genomes; ++c) *out++ = c;
                    if (out != flat + ptr[r + 1]) bad.store(1);       // unsorted or duplicated input
                }
            }
        }
    });
    if (bad.load()) return pgx::fail(PGX_ERR_INVALID, "inconsistent rows passed to pgx_plan_folded_lists");
    return PGX_OK;
}

// The one genome every gene of ``genes`` (present in exactly N - 1 genomes) is absent from.
int pgx_plan_missing_genome(const int64_t *indptr, const int32_t *indices, const int64_t *genes,
                                       int64_t n_rows, int32_t n_genomes, int32_t *missing, int32_t n_threads)
{
    if (n_rows < 0 || n_genomes < 1) return pgx::fail(PGX_ERR_INVALID, "bad shape passed to pgx_plan_missing_genome");
    if (n_rows == 0) return PGX_OK;
    if (!indptr || !indices || !genes || !missing) return pgx::fail(PGX_ERR_INVALID, "null pointer passed to pgx_plan_missing_genome");
    const long long grain = std::max<long long>(1, (1 << 20) / n_genomes);
    std::atomic<long long> next{0};
    std::atomic<int> bad{0};
    const long long all = static_cast<long long>(n_genomes) * (n_genomes - 1) / 2;
    const int threads = host_threads(n_threads, (n_rows + grain - 1) / grain);
    run_threads(threads, [&](int) {
        for (;;) {
            const long long r0 = next.fetch_add(grain);
            if (r0 >= n_rows) return;
            const long long r1 = std::min<long long>(n_rows, r0 + grain);
            for (long long r = r0; r < r1; ++r) {
                const int64_t a = indptr[genes[r]], e = indptr[genes[r] + 1];
                long long sum = 0;
                for (int64_t i = a; i < e; ++i) sum += indices[i];
                const long long miss = all - sum;
                if (e - a != n_genomes - 1 || miss < 0 || miss >= n_genomes) {
                    bad.store(1);
                    continue;
                }
                missing[r] = static_cast<int32_t>(miss);
            }
        }
    });
    if (bad.load()) return pgx::fail(PGX_ERR_INVALID, "rows passed to pgx_plan_missing_genome are not single-absence rows");
    return PGX_OK;
}

// oracle/plan_np.py, _balanced_row_order: which list rows share a shared-memory wavefront group.  The lanes of a group
// (``modulus`` consecutive rows of a sub-block) gather in lock step, one entry each, and two entries collide
// when their genome indices agree modulo ``modulus``: a group needs at least max over residues of (entries of
// that residue in the group) steps, however well pgx_plan_bank_order arranges them.  Rows may be put in any
// order inside a class (same chunk count and list kind), so the groups are formed greedily: the candidates
// are the class riffled into ``modulus`` parts (neighbours then differ in length), a group starts with the
// first candidate and then takes, ``modulus`` - 1 times, the candidate among the next ``window`` that keeps
// the largest residue load of the group smallest (first such candidate wins).
//   genes / use_abs / class_key : the list rows in their current order; rows of one class are consecutive
//   order                       : out, int64 [n_rows]: position (in the current order) of the row that goes
//                                 to each place of the new order
int pgx_plan_balance_rows(const int64_t *indptr, const int32_t *indices, const int64_t *genes,
                                     const uint8_t *use_abs, const int64_t *class_key, int64_t n_rows,
                                     int32_t n_genomes, int32_t modulus, int32_t window, int64_t *order,
                                     int32_t n_threads)
{
    if (n_rows < 0 || n_genomes < 1 || window < 1) return pgx::fail(PGX_ERR_INVALID, "bad shape passed to pgx_plan_balance_rows");
    if (modulus != 8 && modulus != 16 && modulus != 32) return pgx::fail(PGX_ERR_INVALID, "modulus must be 8, 16 or 32");
    if (n_rows == 0) return PGX_OK;
    if (!indptr || !indices || !genes || !use_abs || !class_key || !order)
        return pgx::fail(PGX_ERR_INVALID, "null pointer passed to pgx_plan_balance_rows");
    const int R = modulus;
    // residue histogram of every row's folded list
    std::vector<int32_t> hist(static_cast<size_t>(n_rows) * R);
    int32_t all[MAX_MOD];
    for (int r = 0; r < R; ++r) all[r] = (n_genomes - r + R - 1) / R;          // genomes c < N with c % R == r
    {
        const long long grain = 1024;
        std::atomic<long long> next{0};
        const int threads = host_threads(n_threads, (n_rows + grain - 1) / grain);
        run_threads(threads, [&](int) {
            for (;;) {
                const long long r0 = next.fetch_add(grain);
                if (r0 >= n_rows) return;
                const long long r1 = std::min<long long>(n_rows, r0 + grain);
                for (long long row = r0; row < r1; ++row) {
                    int32_t *h = hist.data() + static_cast<size_t>(row) * R;
                    for (int r = 0; r < R; ++r) h[r] = 0;
                    for (int64_t e = indptr[genes[row]]; e < indptr[genes[row] + 1]; ++e) ++h[indices[e] % R];
                    if (use_abs[row])
                        for (int r = 0; r < R; ++r) h[r] = all[r] - h[r];
                }
            }
        });
    }
    // classes
    std::vector<int64_t> class_start;
    for (int64_t row = 0; row < n_rows; ++row)
        if (row == 0 || class_key[row] != class_key[row - 1]) class_start.push_back(row);
    class_start.push_back(n_rows);
    const long long n_classes = static_cast<long long>(class_start.size()) - 1;
    std::atomic<long long> next{0};
    const int threads = host_threads(n_threads, n_classes);
    run_threads(threads, [&](int) {
        std::vector<int64_t> seq, cand;
        for (;;) {
            const long long k = next.fetch_add(1);
            if (k >= n_classes) return;
            const int64_t r0 = class_start[k], cnt = class_start[k + 1] - r0;
            const int64_t per = (cnt + R - 1) / R;
            seq.clear();
            for (int64_t j = 0; j < per; ++j)
                for (int p = 0; p < R; ++p)
                    if (j + per * p < cnt) seq.push_back(r0 + j + per * p);
            int64_t pos = 0, out = r0;
            cand.clear();
            while (static_cast<int64_t>(cand.size()) < window && pos < cnt) cand.push_back(seq[pos++]);
            while (!cand.empty()) {
                int32_t load[MAX_MOD] = {0};
                for (int slot = 0; slot < R && !cand.empty(); ++slot) {
                    size_t pick = 0;
                    if (slot > 0) {
                        int32_t best = INT32_MAX;
                        for (size_t c = 0; c < cand.size(); ++c) {
                            const int32_t *h = hist.data() + static_cast<size_t>(cand[c]) * R;
                            int32_t top = 0;
                            for (int r = 0; r < R; ++r) top = std::max(top, load[r] + h[r]);
                            if (top < best) {
                                best = top;
                                pick = c;
                            }
                        }
                    }
                    const int64_t row = cand[pick];
                    cand.erase(cand.begin() + static_cast<long>(pick));
                    order[out++] = row;
                    const int32_t *h = hist.data() + static_cast<size_t>(row) * R;
                    for (int r = 0; r < R; ++r) load[r] += h[r];
                    if (pos < cnt) cand.push_back(seq[pos++]);
                }
            }
        }
    });
    return PGX_OK;
}

}  // namespace pgx

// 1 when every 64-bit word of ``words`` equals ``value`` (the planner's "all stored values are 1" test for
// int64 and float64 tables), else 0.
extern "C" int pgx_plan_all_equal_u64(const uint64_t *words, int64_t n, uint64_t value, int32_t n_threads)
{
    if (n <= 0 || !words) return n <= 0 ? 1 : 0;
    const int threads = pgx::host_threads(n_threads, std::max<long long>(1, n / (1 << 18)));
    std::atomic<int> differs{0};
    pgx::run_threads(threads, [&](int t) {
        const int64_t lo = n * t / threads, hi = n * (t + 1) / threads;
        uint64_t acc = 0;
        for (int64_t i = lo; i < hi; ++i) acc |= words[i] ^ value;
        if (acc) differs.store(1);
    });
    return differs.load() ? 0 : 1;
}
