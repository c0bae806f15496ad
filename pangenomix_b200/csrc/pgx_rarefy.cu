// Pan/core rarefaction on sm_100a.
//
// Replaces the double loop of estimate_pan_core_size
// (/root/reference/pangenomix/pangenome_analysis.py:81-90).  For one genome order pi with
// rank = pi^-1, a gene g enters the pan-genome at step fp_g = min rank of its present
// genomes and leaves the core genome at step fa_g = min rank of its absent genomes, so
//   pan[k]  = #{g : fp_g <= k} = cumsum(hist(fp))[k]
//   core[k] = #{g : fa_g >  k} = G - cumsum(hist(fa))[k]
// (bit-exact with :89-:90; the identity itself is under test in tests/test_oracle_golden.py).
// Exactly one of fp_g, fa_g is 0 -- the rank-0 genome either has the gene or not -- so bin 0
// of both histograms is a column sum of the table (closed form); the row kernels only ever
// produce the ONE non-zero statistic of every (gene, permutation).
//
// Kernel 0 (prep_kernel): one CTA per permutation.  Inverts the genome order into a rank row
//   (uint16, scattered through shared memory, written out coalesced) and writes the closed-form
//   gene classes (empty, universal, single-genome, single-absence genes; bin 0) into the histogram
//   row, which therefore needs no memset and the scan no table look-ups.
// Kernel 1 (list_kernel<B>): genes with a short list.  Persistent CTAs; per item a CTA stages the
//   rank rows of B permutations in shared memory as T[genome][B] uint16 -- one 16-byte line
//   per genome for B = 8, one conflict-free 16-byte store per genome -- and its warps stream runs
//   of sub-blocks of 32 rows, one lane per row, three chunk loads in flight.  Every index costs
//   ONE shared-memory gather that serves all B permutations, folded into packed uint16x2 running
//   minima (VIMNMX.U16x2).  The host ordered the indices of a row so that the lanes of a
//   wavefront hit distinct banks.  If the min is 0 the wanted statistic is the mex of the list's
//   ranks instead: such (row, permutation) events are queued per warp and resolved 32 at a time
//   against the sorted copy of the lists.  With packed bins the other minima of present lists are
//   counted in shared memory once the item's gathers are done (see list_kernel).
// Kernel 2 (probe_kernel<W>): genes with long lists, stored as a genome-major, bit-sliced
//   bitmap (32 genes per word).  A warp walks one genome order for 1,024 W genes at once, one
//   coalesced line of 128 W bytes per step; the first genome whose bit differs from the rank-0
//   genome's bit is the gene's statistic.  O(N / m) steps instead of O(m) gathers.  It runs
//   beside kernel 1 on a second stream (shared-memory-pipe bound vs issue bound).
// Kernel 3 (scan_kernel): turns each histogram row into its two curves with block-wide prefix scans.
//
// Histogram bins are uint16 pairs packed in 32-bit words ("P16") whenever every genome of the table
// holds at most 65,535 genes (plan.max_colsum): a bin counts genes that first appear in, or first go
// missing at, ONE genome, so it cannot exceed that genome's gene count (pan side) or the first genome's
// (core side), and a 32-bit atomic add of 1 or 1 << 16 never carries.  The packed row is half the size
// of the int32 output row: it lives in the upper half of the caller's output row, the rank row in the
// lower half, and the scan expands in place.  The host-buffer calls skip the scan altogether and ship
// the packed rows -- the curves' STEPS -- to the host, which rebuilds the curves while it fills the
// caller's result (pgx_expand.cpp).  Tables with a larger genome fall back to int32 bins.
// Host entry points at the end of the file: the device-pointer calls, the host-buffer pipeline
// (pgx_pan_core_curves_host) and the reference's whole loop in one call (pgx_estimate_pan_core).
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <unistd.h>

#include <atomic>
#include <chrono>
#include <mutex>
#include <thread>
#include <vector>

#include <type_traits>

#include "pgx_common.cuh"

namespace pgx {

void expand_delta_rows(const uint16_t *deltas, long long r0, long long r1, long long n, void *out, bool out_f64);
void expand_split_rows(const uint8_t *rows, long long r0, long long r1, long long n, long long head, void *out, bool out_f64);

namespace {

constexpr int SENTINELS = 32;          // rank-table rows N .. N+31 hold 0xffff (include/pgx.h)
// Optional CUDA-event brackets around the kernels of every device-pointer call (bench.py's roofline).  A row kernel the
// call did not launch counts 0 ms, not the gap between two events recorded back to back.
struct ProfileEvents {
    cudaEvent_t begin, prep_done, list_done, probe_done, end;
    bool list_ran, probe_ran;
};
bool g_profile_on = false;
std::mutex g_profile_mu;
std::vector<ProfileEvents> g_profile_events;

struct Tuning {
    int perms_per_cta = 0;
    int row_splits = 0;
    int threads = 0;
};
Tuning g_tuning;
const bool g_no_overlap = getenv("PGX_NO_OVERLAP") != nullptr;
const bool g_wide_bins = getenv("PGX_WIDE_BINS") != nullptr;      // force int32 histogram bins (tests, A/B)

// Where the kernels of one call keep their per-permutation rows.
//   hist  : histogram row of permutation p at hist + p * hist_stride (32-bit words); 2N int32 bins
//           (pan | core) or, packed, N words of uint16 pairs (bin i of the 2N in half (i & 1) of word i >> 1)
//   ranks : rank row (uint16 [N]) of permutation p at ranks + p * rank_stride (uint16 units)
struct Work {
    uint32_t *hist;
    long long hist_stride;
    uint16_t *ranks;
    long long rank_stride;
    unsigned long long *trace = nullptr;      // optional CTA timeline (pgx_set_trace), null in normal operation
    long long trace_capacity = 0;
    unsigned int *started = nullptr;          // optional: every list CTA counts itself here when it starts (probe gate)
};

// CTA timeline for the evidence of how the two row kernels share the SMs (scripts/overlap_trace.py): every CTA of the
// list kernel (kind 1) and of the probe kernel (kind 2) appends {kind | smid << 8, start, end} in %globaltimer
// nanoseconds.  trace[0] counts the records.
unsigned long long *g_trace = nullptr;
long long g_trace_capacity = 0;

__device__ __forceinline__ unsigned long long global_timer()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ void trace_cta(const Work &work, unsigned kind, unsigned long long t_start)
{
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    const unsigned long long slot = atomicAdd(work.trace, 1ull);
    if (static_cast<long long>(slot) < work.trace_capacity) {
        unsigned long long *rec = work.trace + 1 + 3 * slot;
        rec[0] = kind | (static_cast<unsigned long long>(smid) << 8);
        rec[1] = t_start;
        rec[2] = global_timer();
    }
}

// bin ``idx`` (0 .. 2N-1: pan bins then core bins) of a histogram row += v
template <bool P16>
__device__ __forceinline__ void hist_add(uint32_t *row, int idx, uint32_t v)
{
    if constexpr (P16) atomicAdd(row + (idx >> 1), v << ((idx & 1) * 16));
    else atomicAdd(row + idx, v);
}

// ---------------------------------------------------------------------------------------------
// Kernel 0: rank rows + closed forms
// ---------------------------------------------------------------------------------------------
// Closed forms (every gene that never reaches a row kernel).  Bin 0 of both sides is the number of genes the
// first genome holds (pan[0] = core[0]).  A gene living in a single genome c has first presence rank[c] and
// first absence 1 if c comes first, 0 otherwise; a gene missing from a single genome c the mirror image.
// int32 bins hold the core side as "genes lost so far" (bin 0 = G - colsum[first]); packed bins hold the
// curve's steps (bin 0 = core[0] = colsum[first]), because G - colsum may not fit 16 bits.
template <bool P16, bool VEC>
__global__ void __launch_bounds__(256)
prep_kernel(const pgx_plan plan, const uint16_t *__restrict__ perms, const Work work, int *__restrict__ bad_rows)
{
    extern __shared__ __align__(16) uint16_t s_rank[];   // [N] (VEC: N % 8 == 0 and every row 16-byte aligned)
    const int n = plan.n_genomes;
    const long long p = blockIdx.x;
    const uint16_t *__restrict__ perm = perms + p * n;
    const int tid = threadIdx.x;
    const uint32_t last = static_cast<uint32_t>(n - 1);
    uint16_t *__restrict__ ranks = work.ranks + p * work.rank_stride;
    bool missing = false;

    // ---- rank row: scatter through shared memory, write out coalesced ----
    if constexpr (VEC) {
        for (int g = tid * 8; g < n; g += blockDim.x * 8) *reinterpret_cast<uint4 *>(s_rank + g) = make_uint4(~0u, ~0u, ~0u, ~0u);
        __syncthreads();
        for (int k = tid * 8; k < n; k += blockDim.x * 8) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(perm + k));
            const uint32_t g[8] = {v.x & 0xffffu, v.x >> 16, v.y & 0xffffu, v.y >> 16, v.z & 0xffffu, v.z >> 16, v.w & 0xffffu, v.w >> 16};
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (g[j] <= last) s_rank[g[j]] = static_cast<uint16_t>(k + j);
        }
        __syncthreads();
        for (int g = tid * 8; g < n; g += blockDim.x * 8) {
            const uint4 v = *reinterpret_cast<const uint4 *>(s_rank + g);
            // a 0xffff left in the row: a genome without a rank
            missing |= ((v.x & 0xffffu) == 0xffffu) | ((v.x >> 16) == 0xffffu) | ((v.y & 0xffffu) == 0xffffu) | ((v.y >> 16) == 0xffffu) |
                       ((v.z & 0xffffu) == 0xffffu) | ((v.z >> 16) == 0xffffu) | ((v.w & 0xffffu) == 0xffffu) | ((v.w >> 16) == 0xffffu);
            *reinterpret_cast<uint4 *>(ranks + g) = v;
        }
    } else {
        for (int g = tid; g < n; g += blockDim.x) s_rank[g] = 0xffffu;
        __syncthreads();
        for (int k = tid; k < n; k += blockDim.x) {
            const uint32_t g = __ldg(perm + k);
            if (g <= last) s_rank[g] = static_cast<uint16_t>(k);
        }
        __syncthreads();
        for (int g = tid; g < n; g += blockDim.x) {
            const uint16_t r = s_rank[g];
            missing |= r == 0xffffu;
            ranks[g] = r;
        }
    }
    // a row that is not a permutation of 0 .. N-1 leaves a genome without a rank
    if (missing && bad_rows) atomicAdd(bad_rows, 1);

    // ---- closed forms: every bin costs a load of perm[k] and a dependent gather from a weight vector.  The loads go
    // through the read-only path (they cannot alias the stores) and eight bins are in flight per thread. ----
    const uint32_t first = min(static_cast<uint32_t>(__ldg(perm)), last);
    const int col_first = __ldg(plan.d_colsum + first);
    const uint32_t head_pan = __ldg(plan.d_w_absent + first), head_core = __ldg(plan.d_w_present + first);
    uint32_t *__restrict__ hist = work.hist + p * work.hist_stride;
    constexpr int BINS = 8;
#pragma unroll 2
    for (int i0 = tid * BINS; i0 < 2 * n; i0 += blockDim.x * BINS) {
        uint32_t g[BINS], v[BINS];
        if constexpr (VEC) {
            // N % 8 == 0: the eight bins lie on one side, ranks k0 .. k0 + 7
            const int k0 = i0 >= n ? i0 - n : i0;
            const uint4 q = __ldg(reinterpret_cast<const uint4 *>(perm + k0));
            g[0] = q.x & 0xffffu; g[1] = q.x >> 16; g[2] = q.y & 0xffffu; g[3] = q.y >> 16;
            g[4] = q.z & 0xffffu; g[5] = q.z >> 16; g[6] = q.w & 0xffffu; g[7] = q.w >> 16;
#pragma unroll
            for (int j = 0; j < BINS; ++j) g[j] = min(g[j], last);
        } else {
#pragma unroll
            for (int j = 0; j < BINS; ++j) {
                const int idx = min(i0 + j, 2 * n - 1);
                g[j] = min(static_cast<uint32_t>(__ldg(perm + (idx >= n ? idx - n : idx))), last);
            }
        }
#pragma unroll
        for (int j = 0; j < BINS; ++j) {
            const int idx = min(i0 + j, 2 * n - 1);
            v[j] = static_cast<uint32_t>(__ldg((idx >= n ? plan.d_w_absent : plan.d_w_present) + g[j]));
        }
#pragma unroll
        for (int j = 0; j < BINS; ++j) {
            const int idx = i0 + j;
            const int side = idx >= n;
            const int k = idx - side * n;
            if (k == 0) v[j] = static_cast<uint32_t>(P16 || side == 0 ? col_first : plan.n_genes - col_first);
            else if (k == 1) v[j] += side == 0 ? head_pan : head_core;
        }
        if constexpr (P16) {
            if constexpr (VEC) {
                *reinterpret_cast<uint4 *>(hist + (i0 >> 1)) =
                    make_uint4(v[0] | (v[1] << 16), v[2] | (v[3] << 16), v[4] | (v[5] << 16), v[6] | (v[7] << 16));
            } else {
#pragma unroll
                for (int j = 0; j < BINS; j += 2)
                    if (i0 + j < 2 * n) hist[(i0 + j) >> 1] = v[j] | (i0 + j + 1 < 2 * n ? v[j + 1] << 16 : 0u);
            }
        } else {
            if constexpr (VEC) {
                *reinterpret_cast<uint4 *>(hist + i0) = make_uint4(v[0], v[1], v[2], v[3]);
                *reinterpret_cast<uint4 *>(hist + i0 + 4) = make_uint4(v[4], v[5], v[6], v[7]);
            } else {
#pragma unroll
                for (int j = 0; j < BINS; ++j)
                    if (i0 + j < 2 * n) hist[i0 + j] = v[j];
            }
        }
    }
}

// The same work for tables whose rank row and histogram row fit shared memory together (6N bytes with packed bins:
// N <= 18,000).  The gathers w[perm[k]] of prep_kernel miss L1 once eight CTAs of rank rows share an SM and then cost
// an L2 sector each (2e8 per 10,000 permutations of C4: the kernel ran at L2 bandwidth, 0.84 ms); here they are turned
// around: the weight vectors are read in genome order, coalesced, and SCATTERED by rank into a shared-memory image of
// the histogram row, which then leaves with 16-byte stores.
template <bool P16>
__global__ void __launch_bounds__(512)
prep_scatter_kernel(const pgx_plan plan, const uint16_t *__restrict__ perms, const Work work, int *__restrict__ bad_rows)
{
    using BinT = typename std::conditional<P16, uint16_t, uint32_t>::type;
    extern __shared__ __align__(16) unsigned char s_raw[];
    const int n = plan.n_genomes;
    BinT *s_bins = reinterpret_cast<BinT *>(s_raw);                                   // [2N]: pan bins | core bins
    uint16_t *s_rank = reinterpret_cast<uint16_t *>(s_raw + ((sizeof(BinT) * 2 * n + 15) & ~size_t(15)));   // [N]
    const long long p = blockIdx.x;
    const uint16_t *__restrict__ perm = perms + p * n;
    const int tid = threadIdx.x;
    const uint32_t last = static_cast<uint32_t>(n - 1);

    // (every loop below handles eight genomes / ranks per thread with 16-byte accesses when N % 8 == 0)
    const bool vec = (n & 7) == 0 && (reinterpret_cast<uintptr_t>(perm) & 15) == 0 && (work.rank_stride & 7) == 0 &&
                     (reinterpret_cast<uintptr_t>(work.ranks) & 15) == 0 &&
                     ((reinterpret_cast<uintptr_t>(plan.d_w_present) | reinterpret_cast<uintptr_t>(plan.d_w_absent)) & 15) == 0;
    {
        uint4 *z = reinterpret_cast<uint4 *>(s_raw);
        const int bins16 = static_cast<int>((sizeof(BinT) * 2 * n + 15) >> 4), rank16 = (2 * n + 15) >> 4;   // smem is padded to 16 bytes
        for (int i = tid; i < bins16; i += blockDim.x) z[i] = make_uint4(0u, 0u, 0u, 0u);
        uint4 *f = reinterpret_cast<uint4 *>(s_rank);
        for (int i = tid; i < rank16; i += blockDim.x) f[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
    }
    __syncthreads();
    if (vec) {
        for (int k = tid * 8; k < n; k += blockDim.x * 8) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(perm + k));
            const uint32_t g[8] = {v.x & 0xffffu, v.x >> 16, v.y & 0xffffu, v.y >> 16, v.z & 0xffffu, v.z >> 16, v.w & 0xffffu, v.w >> 16};
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (g[j] <= last) s_rank[g[j]] = static_cast<uint16_t>(k + j);
        }
    } else {
        for (int k = tid; k < n; k += blockDim.x) {
            const uint32_t g = __ldg(perm + k);
            if (g <= last) s_rank[g] = static_cast<uint16_t>(k);
        }
    }
    __syncthreads();
    uint16_t *__restrict__ ranks = work.ranks + p * work.rank_stride;
    bool missing = false;
    if (vec) {
        for (int g0 = tid * 8; g0 < n; g0 += blockDim.x * 8) {
            const uint4 rv = *reinterpret_cast<const uint4 *>(s_rank + g0);
            *reinterpret_cast<uint4 *>(ranks + g0) = rv;
            const int4 pa = __ldg(reinterpret_cast<const int4 *>(plan.d_w_present + g0));
            const int4 pb = __ldg(reinterpret_cast<const int4 *>(plan.d_w_present + g0 + 4));
            const int4 aa = __ldg(reinterpret_cast<const int4 *>(plan.d_w_absent + g0));
            const int4 ab = __ldg(reinterpret_cast<const int4 *>(plan.d_w_absent + g0 + 4));
            const uint32_t r[8] = {rv.x & 0xffffu, rv.x >> 16, rv.y & 0xffffu, rv.y >> 16, rv.z & 0xffffu, rv.z >> 16, rv.w & 0xffffu, rv.w >> 16};
            const int wp[8] = {pa.x, pa.y, pa.z, pa.w, pb.x, pb.y, pb.z, pb.w};
            const int wa[8] = {aa.x, aa.y, aa.z, aa.w, ab.x, ab.y, ab.z, ab.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if (r[j] <= last) {
                    s_bins[r[j]] = static_cast<BinT>(wp[j]);
                    s_bins[n + r[j]] = static_cast<BinT>(wa[j]);
                } else {
                    missing = true;
                }
            }
        }
    } else {
        for (int g = tid; g < n; g += blockDim.x) {
            const uint32_t r = s_rank[g];
            ranks[g] = static_cast<uint16_t>(r);
            if (r <= last) {
                // genes living in / missing from genome g alone: first presence / first absence at rank r
                s_bins[r] = static_cast<BinT>(__ldg(plan.d_w_present + g));
                s_bins[n + r] = static_cast<BinT>(__ldg(plan.d_w_absent + g));
            } else {
                missing = true;                       // a genome without a rank: the row is not a permutation
            }
        }
    }
    if (missing && bad_rows) atomicAdd(bad_rows, 1);
    __syncthreads();
    if (tid == 0) {
        const uint32_t first = min(static_cast<uint32_t>(__ldg(perm)), last);
        const int col_first = __ldg(plan.d_colsum + first);
        // bin 0: genes of the first genome; rank 1 also sees the first genome's single-absence / single-genome genes
        s_bins[0] = static_cast<BinT>(col_first);
        s_bins[n] = static_cast<BinT>(P16 ? col_first : plan.n_genes - col_first);
        if (n > 1) {
            s_bins[1] += static_cast<BinT>(__ldg(plan.d_w_absent + first));
            s_bins[n + 1] += static_cast<BinT>(__ldg(plan.d_w_present + first));
        }
    }
    __syncthreads();
    uint32_t *__restrict__ hist = work.hist + p * work.hist_stride;
    const int words = P16 ? n : 2 * n;                                                // 32-bit words of the row
    const uint32_t *src = reinterpret_cast<const uint32_t *>(s_bins);
    if ((words & 3) == 0 && (reinterpret_cast<uintptr_t>(hist) & 15) == 0) {
        for (int w = tid * 4; w < words; w += blockDim.x * 4)
            *reinterpret_cast<uint4 *>(hist + w) = *reinterpret_cast<const uint4 *>(src + w);
    } else {
        for (int w = tid; w < words; w += blockDim.x) hist[w] = src[w];
    }
}

// ---------------------------------------------------------------------------------------------
// Kernel 1: list rows
// ---------------------------------------------------------------------------------------------
template <int B>
struct Packed {
    static constexpr int REGS = (B + 1) / 2;
};

// One gather of the B ranks of genome c, folded into the running minima.
template <int B>
__device__ __forceinline__ void gather_min(const uint16_t *table, uint32_t c,
                                           uint32_t (&acc)[Packed<B>::REGS])
{
    if constexpr (B == 8) {
        const uint4 v = *reinterpret_cast<const uint4 *>(table + c * 8u);
        acc[0] = __vminu2(acc[0], v.x);
        acc[1] = __vminu2(acc[1], v.y);
        acc[2] = __vminu2(acc[2], v.z);
        acc[3] = __vminu2(acc[3], v.w);
    } else if constexpr (B == 4) {
        const uint2 v = *reinterpret_cast<const uint2 *>(table + c * 4u);
        acc[0] = __vminu2(acc[0], v.x);
        acc[1] = __vminu2(acc[1], v.y);
    } else if constexpr (B == 2) {
        const uint32_t v = *reinterpret_cast<const uint32_t *>(table + c * 2u);
        acc[0] = __vminu2(acc[0], v);
    } else {
        acc[0] = min(acc[0], static_cast<uint32_t>(table[c]));
    }
}

template <int B>
__device__ __forceinline__ void gather_chunk(const uint16_t *table, const uint4 v,
                                             uint32_t (&acc)[Packed<B>::REGS])
{
    gather_min<B>(table, v.x & 0xffffu, acc);
    gather_min<B>(table, v.x >> 16, acc);
    gather_min<B>(table, v.y & 0xffffu, acc);
    gather_min<B>(table, v.y >> 16, acc);
    gather_min<B>(table, v.z & 0xffffu, acc);
    gather_min<B>(table, v.z >> 16, acc);
    gather_min<B>(table, v.w & 0xffffu, acc);
    gather_min<B>(table, v.w >> 16, acc);
}

// The B minima of one list row, as the packed registers hold them, to and from the list kernel's scratch
// (minima[slot][row][q]).  Evict-first both ways: the scratch streams through L2 while the probe kernel's bitmap is
// meant to stay there.
template <int B>
__device__ __forceinline__ void store_minima(uint16_t *p, const uint32_t (&acc)[Packed<B>::REGS])
{
    if constexpr (B == 8) __stcs(reinterpret_cast<uint4 *>(p), make_uint4(acc[0], acc[1], acc[2], acc[3]));
    else if constexpr (B == 4) __stcs(reinterpret_cast<uint2 *>(p), make_uint2(acc[0], acc[1]));
    else if constexpr (B == 2) __stcs(reinterpret_cast<unsigned int *>(p), acc[0]);
    else __stcs(reinterpret_cast<unsigned short *>(p), static_cast<unsigned short>(acc[0]));
}

template <int B>
__device__ __forceinline__ void load_minima(const uint16_t *p, uint32_t (&m)[Packed<B>::REGS])
{
    if constexpr (B == 8) {
        const uint4 v = __ldcs(reinterpret_cast<const uint4 *>(p));
        m[0] = v.x; m[1] = v.y; m[2] = v.z; m[3] = v.w;
    } else if constexpr (B == 4) {
        const uint2 v = __ldcs(reinterpret_cast<const uint2 *>(p));
        m[0] = v.x; m[1] = v.y;
    } else if constexpr (B == 2) {
        m[0] = __ldcs(reinterpret_cast<const unsigned int *>(p));
    } else {
        m[0] = __ldcs(reinterpret_cast<const unsigned short *>(p));
    }
}

// mex of the ranks of a sorted genome list, given that rank 0 is in it: walk the genome
// order from rank 1 and stop at the first genome that is not in the list.
__device__ __noinline__ int mex_probe(const uint16_t *__restrict__ perm,
                                      const uint16_t *__restrict__ list, int len, int n)
{
    int k = 1;
    while (k < n) {
        const uint32_t c = perm[k];
        int lo = 0, hi = len;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (list[mid] < c) lo = mid + 1; else hi = mid;
        }
        if (lo < len && list[lo] == c) ++k; else break;
    }
    return k;
}

// Deferred mex events of a warp: (list row << 4 | absent_list << 3 | permutation slot).
constexpr int EVENT_QUEUE = 64;

// The chunk stream of a task is prefetched through THREE separately named buffers, each refilled by its own
// load instruction: a rotating buffer refilled by ONE static LDG gets one scoreboard from the compiler, and waiting
// for its oldest chunk then waits for every chunk load in flight (decoded from the SASS control bits of round 1's
// kernel).  The rare "min == 0" events are collected in a per-lane mask and queued under one vote.  REGCAP x threads
// is sized so that CTAs of the probe kernel, which runs beside this one on a second stream, find registers on every
// SM (48 x 1,024 or 64 x 768).
//
// Where the minima go.  Without ``minima`` (int32 bins, or a scratch too large) the end of a sub-block adds its B
// minima straight into the global histogram rows: B REDs whose 32 lanes hit 32 unrelated lines, about 11 LSU
// wavefronts each (29 % of the kernel's wavefronts on C4).  With ``minima`` (packed bins) a present-list sub-block
// stores its minima to the CTA's slot of the scratch, minima[blockIdx.x][row][q] -- one coalesced store of 32 x 2B
// bytes -- and once the item's gathers are done and the rank table is dead, its shared memory holds B packed pan-side
// histograms: the item's minima are read back and counted with shared atomics, and the non-zero words are added
// into the global rows with coalesced atomics (the probe kernel adds into the same rows).  A partial bin cannot
// exceed the full one, so neither the shared nor the global words carry (the argument for packed bins).
// Absent-list rows (about 1 % of C4's) and the mex events keep their global REDs.
template <int B, int REGCAP, bool P16>
__global__ void __maxnreg__(REGCAP)
list_kernel(const pgx_plan plan, const uint16_t *__restrict__ perms, const long long n_perm,
            const Work work, const int splits, const long long n_items, uint16_t *__restrict__ minima)
{
    extern __shared__ __align__(16) uint16_t table[];   // [(N + 32)][B], then the warps' event queues
    __shared__ int s_next_task;

    constexpr int REGS = Packed<B>::REGS;
    const int n = plan.n_genomes;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    uint32_t *queue = reinterpret_cast<uint32_t *>(table + ((static_cast<size_t>(n + SENTINELS) * B + 7) & ~size_t(7))) +
                      (tid >> 5) * EVENT_QUEUE;
    const uint4 *__restrict__ chunks = reinterpret_cast<const uint4 *>(plan.d_chunks);
    const int4 *__restrict__ tasks = reinterpret_cast<const int4 *>(plan.d_tasks);
    const unsigned long long t_start = work.trace ? global_timer() : 0ull;
    if (work.started && tid == 0) atomicAdd(work.started, 1u);

    // Persistent CTAs: item = (batch of B permutations, share ``split`` of the tasks).  The whole
    // grid is resident at once, so CTAs of the probe kernel can fill the rest of every SM.
    for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
    // split-major: CTAs that run at the same time stream the SAME share of the chunks for different
    // batches, so a table whose chunks exceed L2 (C5: 128 MB) is read from HBM once per launch, not per batch
    const long long batches = n_items / splits;
    const long long p0 = (item % batches) * B;
    const int split = static_cast<int>(item / batches);
    const int n_valid = static_cast<int>(min(static_cast<long long>(B), n_perm - p0));

    // ---- stage the rank rows: T[g][q] = rank of genome g under permutation p0 + q (B coalesced loads, one store) ----
    {
        const uint16_t *__restrict__ ranks = work.ranks + p0 * work.rank_stride;
        for (int g = tid; g < n + SENTINELS; g += blockDim.x) {
            uint32_t r[B];
#pragma unroll
            for (int q = 0; q < B; ++q)
                r[q] = (q < n_valid && g < n) ? static_cast<uint32_t>(ranks[q * work.rank_stride + g]) : 0xffffu;   // sentinels never win a min
            if constexpr (B == 8) {
                *reinterpret_cast<uint4 *>(table + g * 8) =
                    make_uint4(r[0] | (r[1] << 16), r[2] | (r[3] << 16), r[4] | (r[5] << 16), r[6] | (r[7] << 16));
            } else if constexpr (B == 4) {
                *reinterpret_cast<uint2 *>(table + g * 4) = make_uint2(r[0] | (r[1] << 16), r[2] | (r[3] << 16));
            } else if constexpr (B == 2) {
                *reinterpret_cast<uint32_t *>(table + g * 2) = r[0] | (r[1] << 16);
            } else {
                table[g] = static_cast<uint16_t>(r[0]);
            }
        }
    }
    if (tid == 0) s_next_task = 0;
    __syncthreads();

    int queued = 0;                                       // warp-uniform

    auto next_task = [&]() -> int4 {
        int t = 0;
        if (lane == 0) t = atomicAdd(&s_next_task, 1);
        t = __shfl_sync(FULL_MASK, t, 0);
        const long long task = static_cast<long long>(t) * splits + split;
        return task < plan.n_tasks ? __ldg(tasks + task) : make_int4(0, 0, 0, 0);
    };
    // mex of one queued (row, permutation): all lanes of the warp work on different events
    auto resolve = [&](uint32_t ev) {
        const int q = ev & 7, row = ev >> 4;
        PGX_DEVICE_CHECK(row < plan.n_rows && q < n_valid);
        const int s0 = plan.d_sorted_ptr[row];
        const int k = mex_probe(perms + (p0 + q) * n, plan.d_sorted_idx + s0, plan.d_sorted_ptr[row + 1] - s0, n);
        // present list: min -> pan histogram, mex -> core histogram; absent list: swapped.
        if (k < n) hist_add<P16>(work.hist + (p0 + q) * work.hist_stride, ((ev & 8) ? 0 : n) + k, 1u);
    };
    // Queue the events of one sub-block close (bit i: permutation 2i, bit 16 + i: permutation 2i + 1): lane l's events take the queue positions queued + (events of lanes < l)
    // onwards, found with one exclusive scan over the warp (ballots of the bits of the per-lane count, at most 8).
    // A close can bring 256 events: the queue is filled in rounds, and whenever it holds 32 or more, 32 are resolved,
    // so that queued < 32 between closes and no position reaches EVENT_QUEUE.
    auto queue_events = [&](uint32_t zero, const uint32_t tag) {
        const uint32_t cnt = __popc(zero), below = (1u << lane) - 1u;
        int at = queued, end = queued;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const uint32_t m = __ballot_sync(FULL_MASK, (cnt >> b) & 1u);
            at += __popc(m & below) << b;
            end += __popc(m) << b;
        }
        for (;;) {
            while (zero && at < EVENT_QUEUE) {
                const int bit = __ffs(zero) - 1;
                zero &= zero - 1u;
                queue[at++] = tag | static_cast<uint32_t>(((bit & 15) << 1) | (bit >> 4));
            }
            __syncwarp();
            if (end < 32) break;
            const uint32_t e = queue[min(end, EVENT_QUEUE) - 32 + lane];
            __syncwarp();
            resolve(e);
            at -= 32;                                     // the queue keeps its min(end, EVENT_QUEUE) - 32 oldest entries
            end -= 32;
        }
        queued = end;
    };

    // A task is a run of consecutive sub-blocks (32 rows x nch chunks each) laid out back to
    // back, so the warp streams chunk iterations 0 .. n_sub * nch - 1 and closes a sub-block every
    // nch iterations.  The next task's descriptor is fetched while the current one streams.
    int4 td = next_task();
    while (td.y & 0xffff) {
        const int4 td_next = next_task();
        const int nch = td.y & 0xffff;
        const uint32_t absent_list = (td.y >> 24) & 1;
        const int n_rows = td.w;
        const int total = ((n_rows + 31) >> 5) * nch;
        const uint4 *cp = chunks + td.x + lane;
        PGX_DEVICE_CHECK(td.x >= 0 && static_cast<long long>(td.x) + static_cast<long long>(total) * 32 <= plan.n_chunks);
        PGX_DEVICE_CHECK(td.z >= 0 && td.z + n_rows <= plan.n_rows);
        uint32_t *list_hist = work.hist + p0 * work.hist_stride;
        const int side = absent_list ? n : 0;
        // warp-uniform: this task's minima go to the scratch and are counted after the gathers
        uint16_t *const slot = P16 && minima && !absent_list ? minima + static_cast<size_t>(blockIdx.x) * plan.n_rows * B : nullptr;

        uint32_t acc[REGS];
#pragma unroll
        for (int i = 0; i < REGS; ++i) acc[i] = 0xffffffffu;
        int left = nch, row = td.z + lane, rows_left = n_rows - lane;

        // one chunk iteration: 8 gathers; every nch-th iteration closes a sub-block of 32 rows
        auto consume = [&](const uint4 cur) {
            PGX_DEVICE_CHECK((cur.x & 0xffffu) < static_cast<uint32_t>(n + SENTINELS) && (cur.x >> 16) < static_cast<uint32_t>(n + SENTINELS) &&
                             (cur.y & 0xffffu) < static_cast<uint32_t>(n + SENTINELS) && (cur.y >> 16) < static_cast<uint32_t>(n + SENTINELS) &&
                             (cur.z & 0xffffu) < static_cast<uint32_t>(n + SENTINELS) && (cur.z >> 16) < static_cast<uint32_t>(n + SENTINELS) &&
                             (cur.w & 0xffffu) < static_cast<uint32_t>(n + SENTINELS) && (cur.w >> 16) < static_cast<uint32_t>(n + SENTINELS));
            gather_chunk<B>(table, cur, acc);
            if (--left) return;
            const bool valid = rows_left > 0;
            if (slot) {
                // Packed close.  Permutations past n_valid and pad lanes gathered only 0xffff entries, so their minima
                // are never 0.  zero: bit i for permutation 2i, bit 16 + i for permutation 2i + 1 (min 0).
                if (valid) store_minima<B>(slot + static_cast<size_t>(row) * B, acc);
                uint32_t zero = 0;
#pragma unroll
                for (int i = 0; i < REGS; ++i) zero |= __vseteq2(acc[i], 0u) << i;
                if constexpr (B == 1) zero &= 1u;                // the high half of a B = 1 minimum is 0
                if (!valid) zero = 0;
                if (__any_sync(FULL_MASK, zero != 0)) queue_events(zero, static_cast<uint32_t>(row) << 4);
            } else {
                uint32_t zero = 0;                        // the packed close's bit for permutation q: min 0
#pragma unroll
                for (int q = 0; q < B; ++q) {
                    if (q < n_valid) {
                        uint32_t mn;
                        if constexpr (B == 1) mn = acc[0] & 0xffffu;
                        else mn = (acc[q >> 1] >> ((q & 1) * 16)) & 0xffffu;
                        if (valid) {
                            // (mn >= n: a rank row with a hole, i.e. not a permutation -- counted nowhere, reported by the host calls)
                            if (mn == 0) zero |= 1u << ((q >> 1) + (q & 1) * 16);
                            else if (mn < static_cast<uint32_t>(n)) hist_add<P16>(list_hist + q * work.hist_stride, side + static_cast<int>(mn), 1u);
                        }
                    }
                }
                // min == 0: the wanted statistic is the mex; queue (row, permutation), resolve 32 at a time
                if (__any_sync(FULL_MASK, zero != 0)) queue_events(zero, (static_cast<uint32_t>(row) << 4) | (absent_list << 3));
            }
#pragma unroll
            for (int i = 0; i < REGS; ++i) acc[i] = 0xffffffffu;
            left = nch;
            row += 32;
            rows_left -= 32;
        };

        uint4 b0 = total > 0 ? ldg_stream(cp) : make_uint4(0, 0, 0, 0);
        uint4 b1 = total > 1 ? ldg_stream(cp + 32) : make_uint4(0, 0, 0, 0);
        uint4 b2 = total > 2 ? ldg_stream(cp + 64) : make_uint4(0, 0, 0, 0);
        for (int s = 0; s < total; s += 3) {
            const uint4 c0 = b0;
            if (s + 3 < total) b0 = ldg_stream(cp + (s + 3) * 32);
            consume(c0);
            if (s + 1 < total) {
                const uint4 c1 = b1;
                if (s + 4 < total) b1 = ldg_stream(cp + (s + 4) * 32);
                consume(c1);
            }
            if (s + 2 < total) {
                const uint4 c2 = b2;
                if (s + 5 < total) b2 = ldg_stream(cp + (s + 5) * 32);
                consume(c2);
            }
        }
        td = td_next;
    }
    if (lane < queued) resolve(queue[lane]);
    __syncthreads();                                      // every warp is done with this table

    if constexpr (P16) {
        if (minima) {
            // ---- count the item's scratch minima in packed pan-side histograms where the table was ----
            // B >= 2: plane i counts permutation 2i in the low and 2i + 1 in the high half of word i * plane + k (pan bin
            // k), so both halves of a packed minimum register are counted with a constant increment.  B == 1: bin k in
            // half k & 1 of word k >> 1.  A minimum is clamped to n first: bin 0 (min 0, the mex events) and bin n (no
            // permutation of the batch, or a rank row with a hole) are counted but never flushed.  Bin 0 counts rows
            // holding the rank-0 genome and cannot exceed its gene count; carries out of bin n only reach bin n of the
            // other half or leave the word.
            uint32_t *s_hist = reinterpret_cast<uint32_t *>(table);
            const int plane = (n + 2) & ~1;
            const int s_words = B == 1 ? (n + 2) >> 1 : REGS * plane;
            for (int i = tid; i < (s_words + 3) >> 2; i += blockDim.x)
                reinterpret_cast<uint4 *>(s_hist)[i] = make_uint4(0u, 0u, 0u, 0u);
            __syncthreads();
            const uint16_t *__restrict__ slot = minima + static_cast<size_t>(blockIdx.x) * plan.n_rows * B;
            const uint32_t clamp = static_cast<uint32_t>(n) * 0x10001u;
            constexpr int AHEAD = 4;                      // rows per lane in flight: the scratch comes back from HBM
            for (long long t = tid >> 5;; t += blockDim.x >> 5) {
                const long long task = t * splits + split;
                if (task >= plan.n_tasks) break;
                const int4 d = __ldg(tasks + task);
                if (!(d.y & 0xffff) || ((d.y >> 24) & 1)) continue;            // absent lists were counted by REDs
                const uint16_t *m = slot + static_cast<size_t>(d.z) * B;
                for (int r0 = lane; r0 < d.w; r0 += 32 * AHEAD) {
                    uint32_t v[AHEAD][REGS];
#pragma unroll
                    for (int j = 0; j < AHEAD; ++j) {
                        if (r0 + 32 * j < d.w) {
                            load_minima<B>(m + static_cast<size_t>(r0 + 32 * j) * B, v[j]);
                        } else {
#pragma unroll
                            for (int i = 0; i < REGS; ++i) v[j][i] = 0xffffffffu;
                        }
                    }
#pragma unroll
                    for (int j = 0; j < AHEAD; ++j) {
                        if (r0 + 32 * j >= d.w) continue;
#pragma unroll
                        for (int i = 0; i < REGS; ++i) {
                            const uint32_t c = __vminu2(v[j][i], clamp);
                            if constexpr (B == 1) {
                                atomicAdd(s_hist + (c >> 1), 1u << ((c & 1u) * 16));
                            } else {
                                atomicAdd(s_hist + i * plane + (c & 0xffffu), 1u);
                                atomicAdd(s_hist + i * plane + (c >> 16), 0x10000u);
                            }
                        }
                    }
                }
            }
            __syncthreads();
            // global word w holds pan bins 2w and 2w + 1; bin n (odd n: the high half of the last word) is core bin 0
            const int words = (n + 1) >> 1;
            for (int i = 0; i < REGS && 2 * i < n_valid; ++i) {
                uint32_t *dst0 = work.hist + (p0 + 2 * i) * work.hist_stride;
                for (int w = tid; w < words; w += blockDim.x) {
                    uint32_t lo, hi;                      // global word w (pan bins 2w, 2w + 1) of permutations 2i and 2i + 1
                    if constexpr (B == 1) {
                        lo = s_hist[w];
                    } else {
                        const uint2 c = *reinterpret_cast<const uint2 *>(s_hist + i * plane + 2 * w);
                        lo = __byte_perm(c.x, c.y, 0x5410);
                        hi = __byte_perm(c.x, c.y, 0x7632);
                    }
                    const uint32_t keep = (w == 0 ? 0xffff0000u : 0xffffffffu) & (2 * w + 1 == n ? 0x0000ffffu : 0xffffffffu);
                    lo &= keep;
                    if (lo) atomicAdd(dst0 + w, lo);
                    if constexpr (B > 1) {
                        hi &= keep;
                        if (2 * i + 1 < n_valid && hi) atomicAdd(dst0 + work.hist_stride + w, hi);
                    }
                }
            }
            __syncthreads();                              // the next item's table overwrites the histograms
        }
    }
    }
    if (work.trace && tid == 0) trace_cta(work, 1u, t_start);
}

// ---------------------------------------------------------------------------------------------
// Kernel 2: bitmap rows
// ---------------------------------------------------------------------------------------------
// Bit-sliced: 32 genes per word, genome-major.  A warp owns one superblock of
// 1,024 W bitmap rows (W = 1, 2 or 4 words per lane) and one permutation; lane l holds rows
// 32 W l .. 32 W l + 32 W - 1 of the superblock as W words.  Walking the genome order, step k
// loads ONE coalesced line of 128 W bytes -- the presence bits of all 1,024 W genes in genome
// perm[k] -- and
//     flipped = (line ^ line_of_rank_0) & pending
// marks the genes whose bit differs from the rank-0 genome's for the first time: k is their
// statistic (first presence if the rank-0 bit was 0, first absence if it was 1).  The walk
// stops when no gene of the superblock is pending: O(N / m) steps of O(1) work per 32 genes,
// the reference's own genome-by-genome accumulation (:87-:90) restricted to unresolved genes.
constexpr int SLICE_WARPS = 4;

template <int W>
struct SliceVec;
template <>
struct SliceVec<1> { using type = uint32_t; };
template <>
struct SliceVec<2> { using type = uint2; };
template <>
struct SliceVec<4> { using type = uint4; };

template <int W>
__device__ __forceinline__ void load_line(const uint32_t *p, uint32_t (&w)[W])
{
    const typename SliceVec<W>::type v = __ldg(reinterpret_cast<const typename SliceVec<W>::type *>(p));
    if constexpr (W == 1) {
        w[0] = v;
    } else if constexpr (W == 2) {
        w[0] = v.x;
        w[1] = v.y;
    } else {
        w[0] = v.x;
        w[1] = v.y;
        w[2] = v.z;
        w[3] = v.w;
    }
}

// Late in a walk a handful of genes keep the whole warp loading 128 W-byte lines.  From STRAGGLER_MIN_RANK on,
// once at most ``straggler_max`` genes are pending, the warp finishes them one by one instead: 32 lanes test 32
// consecutive ranks of ONE gene (a 4-byte load each), the first differing lane is the gene's statistic.  Each
// such scan is a chain of dependent loads, so the hand-over pays only for the last few genes (measured on C4:
// probe kernel 2.39 ms without, 2.13 ms from 16 genes, 2.33 ms from 64, 4.4 ms from 128).
constexpr int STRAGGLER_MIN_RANK = 64;

template <int W, bool P16>
__global__ void __launch_bounds__(SLICE_WARPS * 32, 8)
probe_kernel(const pgx_plan plan, const uint16_t *__restrict__ perms, const long long n_perm,
             const Work work, const int straggler_max)
{
    constexpr int DEPTH = W == 4 ? 4 : 8;          // lines in flight per warp
    const int n = plan.n_genomes;
    const int lane = threadIdx.x & 31;
    const long long unit = static_cast<long long>(blockIdx.x) * SLICE_WARPS + (threadIdx.x >> 5);
    if (unit >= n_perm * plan.n_superblocks) return;           // whole warps leave together
    const unsigned long long t_start = work.trace ? global_timer() : 0ull;
    struct TraceOnExit {                                       // one record per warp (unit), whichever way the walk ends
        const Work &work;
        unsigned long long t_start;
        int lane;
        __device__ ~TraceOnExit() { if (work.trace && lane == 0) trace_cta(work, 2u, t_start); }
    } trace_on_exit{work, t_start, static_cast<int>(threadIdx.x & 31)};
    const long long sb = unit / n_perm, q = unit - sb * n_perm;   // costly superblocks first

    const uint32_t *__restrict__ lines = plan.d_bits + (static_cast<size_t>(sb) * n) * (32 * W) + lane * W;
    const uint16_t *__restrict__ perm = perms + q * n;
    uint32_t *hist_q = work.hist + q * work.hist_stride;
    const int my_side = lane == 1 ? n : 0;                        // lane 0 adds pan counts, lane 1 core counts

    uint32_t pending[W], b0[W];
#pragma unroll
    for (int j = 0; j < W; ++j) {
        const long long left = static_cast<long long>(plan.n_long) - (sb * (1024 * W) + (lane * W + j) * 32);
        pending[j] = left >= 32 ? 0xffffffffu : (left <= 0 ? 0u : ((1u << left) - 1u));
    }
    // (genome indices are clamped: a row that is not a permutation must not read outside the bitmap)
    const uint32_t last = static_cast<uint32_t>(n - 1);
    const uint32_t genome0 = min(static_cast<uint32_t>(perm[0]), last);
    load_line<W>(lines + static_cast<size_t>(genome0) * (32 * W), b0);

    for (int k0 = 0; k0 < n; k0 += 32) {
        // genomes of ranks k0 .. k0 + 31; ranks past the end repeat the rank-0 genome (never a flip)
        const uint32_t chunk = k0 + lane < n ? min(static_cast<uint32_t>(perm[k0 + lane]), last) : genome0;
        if (k0 >= STRAGGLER_MIN_RANK && straggler_max > 0) {
            uint32_t cnt = 0;
#pragma unroll
            for (int x = 0; x < W; ++x) cnt += __popc(pending[x]);
            if (__reduce_add_sync(FULL_MASK, cnt) <= static_cast<uint32_t>(straggler_max)) {
                // all ranks below k0 have been walked; every pending gene flips at some rank >= k0
                const uint32_t *__restrict__ column = plan.d_bits + (static_cast<size_t>(sb) * n) * (32 * W);
#pragma unroll
                for (int x = 0; x < W; ++x) {
                    uint32_t owners = __ballot_sync(FULL_MASK, pending[x] != 0);
                    while (owners) {
                        const int src = __ffs(owners) - 1;
                        owners &= owners - 1;
                        uint32_t word = __shfl_sync(FULL_MASK, pending[x], src);
                        const uint32_t first = __shfl_sync(FULL_MASK, b0[x], src);
                        const uint32_t *__restrict__ cell = column + src * W + x;
                        while (word) {
                            const int bit = __ffs(word) - 1;
                            word &= word - 1;
                            const uint32_t want = (first >> bit) & 1u;
                            uint32_t c = chunk;                       // ranks k0 .. k0 + 31 first
                            int k = k0;
                            while (k < n) {                           // (a bitmap row always flips: the bound only guards a corrupt plan)
                                const uint32_t v = __ldg(cell + static_cast<size_t>(c) * (32 * W));
                                const uint32_t differs = __ballot_sync(FULL_MASK, ((v >> bit) & 1u) != want);
                                if (differs) {
                                    // rank-0 bit 0: first presence (pan side); rank-0 bit 1: first absence (core side)
                                    if (lane == 0) hist_add<P16>(hist_q, (want ? n : 0) + k + __ffs(differs) - 1, 1u);
                                    break;
                                }
                                k += 32;
                                c = k + lane < n ? min(static_cast<uint32_t>(perm[k + lane]), last) : genome0;
                            }
                        }
                    }
                }
                return;
            }
        }
#pragma unroll 1
        for (int j0 = 0; j0 < 32; j0 += DEPTH) {
            uint32_t d[DEPTH][W];
            uint32_t any = 0;
#pragma unroll
            for (int j = 0; j < DEPTH; ++j) {
                const uint32_t c = __shfl_sync(FULL_MASK, chunk, j0 + j);
                PGX_DEVICE_CHECK(c < static_cast<uint32_t>(n));
                load_line<W>(lines + static_cast<size_t>(c) * (32 * W), d[j]);
#pragma unroll
                for (int x = 0; x < W; ++x) {
                    d[j][x] ^= b0[x];
                    any |= d[j][x] & pending[x];
                }
            }
            // late in the walk few genes are pending and most groups of genomes flip none
            if (!__any_sync(FULL_MASK, any)) continue;
#pragma unroll
            for (int j = 0; j < DEPTH; ++j) {
                uint32_t flipped[W], some = 0;
#pragma unroll
                for (int x = 0; x < W; ++x) {
                    flipped[x] = d[j][x] & pending[x];
                    some |= flipped[x];
                }
                if (!__any_sync(FULL_MASK, some)) continue;        // mid / late walk: most single steps flip nothing
                // low half: genes first seen at k (pan side); high half: genes first missed at k (core side)
                uint32_t packed = 0;
#pragma unroll
                for (int x = 0; x < W; ++x) {
                    pending[x] &= ~flipped[x];
                    packed += __popc(flipped[x] & ~b0[x]) | (__popc(flipped[x] & b0[x]) << 16);
                }
                const uint32_t total = __reduce_add_sync(FULL_MASK, packed);     // <= 4,096 per half
                const uint32_t mine = lane == 1 ? total >> 16 : total & 0xffffu;
                PGX_DEVICE_CHECK(k0 + j0 + j > 0 && k0 + j0 + j < n);
                if (lane < 2 && mine) hist_add<P16>(hist_q, my_side + k0 + j0 + j, mine);
            }
            uint32_t left = 0;
#pragma unroll
            for (int x = 0; x < W; ++x) left |= pending[x];
            if (!__any_sync(FULL_MASK, left)) return;
        }
    }
    PGX_DEVICE_CHECK(false && "a bitmap row never flipped: it is empty or universal and must not be in the bitmap");
}

// ---------------------------------------------------------------------------------------------
// Kernel 3: histogram rows -> curves
// ---------------------------------------------------------------------------------------------
// One CTA per permutation: the pan half, then the core half, 4,096 bins per step with 16-byte accesses when the
// genome count allows (VEC: N % 8 == 0).  The output row may BE the buffer the histogram row lives in:
//   int32 bins:  out == hist, every bin is replaced by its curve value;
//   packed bins: the histogram sits in the upper half of the int32 output row (bytes [4N, 8N) of 8N).  The pan half
//                writes bytes [0, 4N) only; the core half reads bin k at byte 6N + 2k and writes curve value k at
//                byte 4N + 4k, which stays behind every bin still to be read while k < N; all loads of a step
//                precede its stores (the block-wide barrier of the scan), and the pan bins are dead by then.
constexpr int SCAN_THREADS = 512;

template <typename OutT, bool P16, bool VEC>
__global__ void __launch_bounds__(SCAN_THREADS)
scan_kernel(const pgx_plan plan, const Work work, OutT *out)
{
    constexpr int ITEMS = 8;
    constexpr int THREADS = SCAN_THREADS;
    __shared__ int warp_tot[THREADS / 32];

    const int n = plan.n_genomes;
    const long long p = blockIdx.x;
    const uint32_t *hist = work.hist + p * work.hist_stride;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // bins k0 .. k0 + 7 of one side as signed steps of the curve (0 past the end)
    auto load_bins = [&](int side, int k0, int (&v)[ITEMS]) {
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) v[i] = 0;
        if (k0 >= n) return;
        if constexpr (P16) {
            const uint16_t *h = reinterpret_cast<const uint16_t *>(hist) + static_cast<long long>(side) * n;
            if constexpr (VEC) {
                const uint4 a = *reinterpret_cast<const uint4 *>(h + k0);
                v[0] = a.x & 0xffffu; v[1] = a.x >> 16; v[2] = a.y & 0xffffu; v[3] = a.y >> 16;
                v[4] = a.z & 0xffffu; v[5] = a.z >> 16; v[6] = a.w & 0xffffu; v[7] = a.w >> 16;
            } else {
#pragma unroll
                for (int i = 0; i < ITEMS; ++i) if (k0 + i < n) v[i] = h[k0 + i];
            }
            // packed bins hold the steps of the curve: core[k] = core[0] - (losses up to k)
            if (side == 1) {
#pragma unroll
                for (int i = 0; i < ITEMS; ++i) if (k0 + i > 0) v[i] = -v[i];
            }
        } else {
            const int32_t *h = reinterpret_cast<const int32_t *>(hist) + static_cast<long long>(side) * n;
            if constexpr (VEC) {
                const int4 a = *reinterpret_cast<const int4 *>(h + k0);
                const int4 b = *reinterpret_cast<const int4 *>(h + k0 + 4);
                v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
                v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
            } else {
#pragma unroll
                for (int i = 0; i < ITEMS; ++i) if (k0 + i < n) v[i] = h[k0 + i];
            }
        }
    };

    // steps (side, base) in order: the whole pan half, then the whole core half; the bins of the next step are
    // loaded before the current one is scanned and stored (reads only ever move ahead of the writes)
    const int chunks = (n + THREADS * ITEMS - 1) / (THREADS * ITEMS);
    int v[ITEMS], nx[ITEMS];
    load_bins(0, tid * ITEMS, v);
    int carry = 0;
    for (int step = 0; step < 2 * chunks; ++step) {
        const int side = step >= chunks;
        const int base = (step - side * chunks) * THREADS * ITEMS;
        const int k0 = base + tid * ITEMS;
        if (step + 1 < 2 * chunks) {
            const int ns = step + 1 >= chunks;
            load_bins(ns, (step + 1 - ns * chunks) * THREADS * ITEMS + tid * ITEMS, nx);
        }
        if (step == chunks) carry = 0;
        OutT *o = out + p * 2ll * n + static_cast<long long>(side) * n;
        int run = 0;
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
            run += v[i];
            v[i] = run;
        }
        int incl = run;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int y = __shfl_up_sync(FULL_MASK, incl, off);
            if (lane >= off) incl += y;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();                          // every load of this step (and of the next) has been issued and consumed
        int before = 0, total = 0;
#pragma unroll
        for (int i = 0; i < THREADS / 32; ++i) {
            const int wt = warp_tot[i];
            if (i < warp) before += wt;
            total += wt;
        }
        const int excl = carry + before + incl - run;
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
            const int c = excl + v[i];
            // int32 bins count the genes LOST so far on the core side; packed bins are already signed steps
            v[i] = (!P16 && side == 1) ? plan.n_genes - c : c;
        }
        if constexpr (VEC) {
            if (k0 < n) {
                if constexpr (sizeof(OutT) == 4) {
                    *reinterpret_cast<int4 *>(o + k0) = make_int4(v[0], v[1], v[2], v[3]);
                    *reinterpret_cast<int4 *>(o + k0 + 4) = make_int4(v[4], v[5], v[6], v[7]);
                } else {
#pragma unroll
                    for (int i = 0; i < ITEMS; i += 2)
                        *reinterpret_cast<double2 *>(o + k0 + i) = make_double2(static_cast<double>(v[i]), static_cast<double>(v[i + 1]));
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < ITEMS; ++i) if (k0 + i < n) o[k0 + i] = static_cast<OutT>(v[i]);
        }
        carry += total;
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) v[i] = nx[i];
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// Launch logic
// ---------------------------------------------------------------------------------------------
int check_plan(const pgx_plan *plan)
{
    if (!plan) return fail(PGX_ERR_INVALID, "plan is null");
    if (plan->n_genomes < 1 || plan->n_genomes > 65503)
        return fail(PGX_ERR_UNSUPPORTED, "n_genomes = %d outside 1..65503 (uint16 genome indices)",
                    plan->n_genomes);
    if (plan->n_genes < 0 || plan->n_rows < 0 || plan->n_tasks < 0 || plan->n_chunks < 0 || plan->n_long < 0)
        return fail(PGX_ERR_INVALID, "negative size in plan");
    if (!plan->d_w_present || !plan->d_w_absent || !plan->d_colsum)
        return fail(PGX_ERR_INVALID, "plan closed-form vectors are null");
    if (plan->n_tasks > 0 && (!plan->d_chunks || !plan->d_tasks || !plan->d_sorted_idx || !plan->d_sorted_ptr))
        return fail(PGX_ERR_INVALID, "plan has list tasks but null list arrays");
    if (plan->n_long > 0 && !plan->d_bits)
        return fail(PGX_ERR_INVALID, "plan has bitmap rows but a null bitmap");
    if (plan->n_long > 0 && plan->slice_words != 1 && plan->slice_words != 2 && plan->slice_words != 4)
        return fail(PGX_ERR_INVALID, "slice_words must be 1, 2 or 4");
    if (plan->n_long > 0 && plan->n_superblocks != (plan->n_long + 1024 * plan->slice_words - 1) / (1024 * plan->slice_words))
        return fail(PGX_ERR_INVALID, "n_superblocks must be ceil(n_long / (1024 * slice_words))");
    if ((reinterpret_cast<uintptr_t>(plan->d_chunks) | reinterpret_cast<uintptr_t>(plan->d_tasks) |
         reinterpret_cast<uintptr_t>(plan->d_bits)) & 15)
        return fail(PGX_ERR_INVALID, "d_chunks, d_tasks and d_bits must be 16-byte aligned");
    if (plan->max_colsum < 0) return fail(PGX_ERR_INVALID, "max_colsum < 0");
    return PGX_OK;
}

// uint16 histogram bins are exact whenever no genome holds more than 65,535 genes (0 = unknown: int32 bins)
bool packed_bins(const pgx_plan *plan)
{
    return !g_wide_bins && plan->max_colsum > 0 && plan->max_colsum <= 65535;
}

struct DeviceLimits {
    int device = -1;
    int sm_count = 0;
    int smem_optin = 0;
};

int device_limits(DeviceLimits *out)
{
    static thread_local DeviceLimits cached;
    int dev = 0;
    PGX_CUDA(cudaGetDevice(&dev));
    if (cached.device != dev) {
        PGX_CUDA(cudaDeviceGetAttribute(&cached.sm_count, cudaDevAttrMultiProcessorCount, dev));
        PGX_CUDA(cudaDeviceGetAttribute(&cached.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        cached.device = dev;
    }
    *out = cached;
    return PGX_OK;
}

// Register cap x threads of the list kernel: 1 = 48 x 1,024 (default), 2 = 64 x 768 (the same share of the register
// file).  Alone, variant 2 is 2 % faster on C4 (5.98 vs 6.09 ms per 10,000 permutations); with the probe kernel running
// beside it -- the way every call runs -- variant 1 wins (8.33 vs 8.67 ms per step).  PGX_LIST_VARIANT overrides.
int list_variant()
{
    static const int v = [] {
        const char *env = getenv("PGX_LIST_VARIANT");
        const int x = env ? atoi(env) : 1;
        return x == 2 ? 2 : 1;
    }();
    return v;
}

// Largest scratch of row minima one list launch takes (grid x n_rows x B x 2 bytes; C4: 244 MB, C5: 774 MB).
constexpr size_t MINIMA_SCRATCH_MAX = size_t(1) << 30;

// The scratch comes from a pool of the library's own per device that keeps its memory between launches: the device's
// default pool hands freed memory back to the driver at every synchronisation, and the host-buffer calls synchronise
// once per block.
int scratch_pool(cudaMemPool_t *out)
{
    static std::mutex mu;
    static cudaMemPool_t pools[64] = {};
    int dev = 0;
    PGX_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return fail(PGX_ERR_UNSUPPORTED, "device ordinal %d out of range", dev);
    std::lock_guard<std::mutex> lock(mu);
    if (!pools[dev]) {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dev;
        cudaMemPool_t pool = nullptr;
        PGX_CUDA(cudaMemPoolCreate(&pool, &props));
        uint64_t keep = ~uint64_t(0);
        PGX_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
        pools[dev] = pool;
    }
    *out = pools[dev];
    return PGX_OK;
}

template <int B, bool P16>
int launch_list(const pgx_plan &plan, const uint16_t *d_perms, long long n_perm, const Work &work,
                const DeviceLimits &lim, cudaStream_t stream, unsigned *grid_out)
{
    const int variant = list_variant();
    int threads = g_tuning.threads;
    if (threads <= 0 && getenv("PGX_LIST_THREADS")) threads = atoi(getenv("PGX_LIST_THREADS"));
    const size_t table_bytes = ((static_cast<size_t>(plan.n_genomes + SENTINELS) * B + 7) & ~size_t(7)) * sizeof(uint16_t);
    // 896 rather than 1,024 threads beside a table that fills the SM: the probe kernel's CTAs, which run beside this
    // kernel, then find registers for three CTAs per SM instead of two (C4: 7.88 vs 8.15 ms per step)
    if (threads <= 0) threads = table_bytes > 100 * 1024 ? (variant == 2 ? 768 : 896) : (table_bytes > 40 * 1024 ? 512 : 256);
    threads = max(32, min(1024, (threads / 32) * 32));
    const size_t smem = table_bytes + static_cast<size_t>(threads / 32) * EVENT_QUEUE * sizeof(uint32_t);
    auto kernel = variant == 2 ? list_kernel<B, 64, P16> : list_kernel<B, 48, P16>;
    PGX_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    const long long batches = (n_perm + B - 1) / B;
    // Row splits: enough CTAs for ~8 waves so the tail is small, but every CTA keeps at
    // least a few tasks per warp (the table build is amortised over them).
    int splits = g_tuning.row_splits;
    if (splits <= 0) {
        const long long resident = static_cast<long long>(lim.sm_count) *
                                   max(1, min(8, static_cast<int>((200 * 1024) / (smem + 1024))));
        const long long want = (8 * resident + batches - 1) / batches;
        const long long most = max(1ll, static_cast<long long>(plan.n_tasks) / ((threads / 32) * 2));
        splits = static_cast<int>(max(1ll, min(want, most)));
    }
    splits = max(1, min(splits, 65535));
    const long long n_items = batches * splits;
    int per_sm = 1;
    PGX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    if (per_sm < 1) return fail(PGX_ERR_UNSUPPORTED, "list kernel does not fit an SM with %d threads", threads);
    const long long grid = max(1ll, min(n_items, static_cast<long long>(lim.sm_count) * max(1, per_sm)));
    // Packed bins: the row minima are counted in shared memory (list_kernel) through a scratch of one slot per CTA,
    // taken stream-ordered for this launch.  Above MINIMA_SCRATCH_MAX, or when the pool has no room, the minima go
    // to the global histogram rows directly.
    uint16_t *minima = nullptr;
    if (P16 && plan.n_rows > 0) {
        const size_t bytes = static_cast<size_t>(grid) * static_cast<size_t>(plan.n_rows) * B * sizeof(uint16_t);
        cudaMemPool_t pool = nullptr;
        if (bytes <= MINIMA_SCRATCH_MAX &&
            (scratch_pool(&pool) != PGX_OK || cudaMallocFromPoolAsync(reinterpret_cast<void **>(&minima), bytes, pool, stream) != cudaSuccess)) {
            cudaGetLastError();
            minima = nullptr;
        }
    }
    kernel<<<static_cast<unsigned>(grid), threads, smem, stream>>>(plan, d_perms, n_perm, work, splits, n_items, minima);
    if (minima) cudaFreeAsync(minima, stream);    // (an error of the launch stays the last error)
    PGX_LAUNCH_CHECK("list_kernel");
    if (grid_out) *grid_out = static_cast<unsigned>(grid);
    return PGX_OK;
}

template <bool P16>
int launch_list_b(const pgx_plan &plan, const uint16_t *d_perms, long long n_perm, const Work &work,
                  const DeviceLimits &lim, cudaStream_t stream, unsigned *grid_out = nullptr)
{
    const size_t per_perm = static_cast<size_t>(plan.n_genomes + SENTINELS) * sizeof(uint16_t);
    const size_t budget = static_cast<size_t>(lim.smem_optin) - 64 - 32 * EVENT_QUEUE * sizeof(uint32_t);
    int b = g_tuning.perms_per_cta;
    if (b != 1 && b != 2 && b != 4 && b != 8) b = plan.perms_per_cta;
    if (b != 1 && b != 2 && b != 4 && b != 8) b = 8;
    while (b > 1 && per_perm * b > budget) b >>= 1;
    if (per_perm * b > budget) return fail(PGX_ERR_UNSUPPORTED, "rank table does not fit shared memory");
    switch (b) {
        case 8: return launch_list<8, P16>(plan, d_perms, n_perm, work, lim, stream, grid_out);
        case 4: return launch_list<4, P16>(plan, d_perms, n_perm, work, lim, stream, grid_out);
        case 2: return launch_list<2, P16>(plan, d_perms, n_perm, work, lim, stream, grid_out);
        default: return launch_list<1, P16>(plan, d_perms, n_perm, work, lim, stream, grid_out);
    }
}

template <bool P16>
int launch_probe(const pgx_plan &plan, const uint16_t *d_perms, long long n_perm, const Work &work,
                 cudaStream_t stream)
{
    // one warp per (superblock, permutation); 2^31 blocks of 4 warps cover any realistic call
    const long long units = n_perm * plan.n_superblocks;
    const long long blocks = (units + SLICE_WARPS - 1) / SLICE_WARPS;
    if (blocks > 2147483647ll) return fail(PGX_ERR_UNSUPPORTED, "too many (superblock, permutation) units in one call");
    // PGX_PROBE_STRAGGLERS: pending genes from which a warp finishes its walk gene by gene (0 = never)
    static const int straggler_max = [] {
        const char *env = getenv("PGX_PROBE_STRAGGLERS");
        return env ? max(0, atoi(env)) : 16;
    }();
    const unsigned grid = static_cast<unsigned>(blocks);
    switch (plan.slice_words) {
        case 4: probe_kernel<4, P16><<<grid, SLICE_WARPS * 32, 0, stream>>>(plan, d_perms, n_perm, work, straggler_max); break;
        case 2: probe_kernel<2, P16><<<grid, SLICE_WARPS * 32, 0, stream>>>(plan, d_perms, n_perm, work, straggler_max); break;
        default: probe_kernel<1, P16><<<grid, SLICE_WARPS * 32, 0, stream>>>(plan, d_perms, n_perm, work, straggler_max); break;
    }
    PGX_LAUNCH_CHECK("probe_kernel");
    return PGX_OK;
}

// Second stream + fork/join events of the calling thread's current device.
struct Aux {
    int device = -1;
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
    unsigned int *d_started = nullptr;        // list CTAs that have started, over all calls through this Aux
    unsigned int expected = 0;                // ... and how many the host has launched
};

// The gate of the second stream.  The list kernel's CTAs need an SM whose shared-memory carve-out is at its maximum,
// and an SM changes its carve-out only when it is empty: if the probe kernel's small CTAs get to the SMs first -- as
// in a call that finds the device idle -- every list CTA waits until its SM has drained and the two kernels run one
// after the other (9.0 instead of 7.6 ms per 10,000 permutations of C4).  So the probe launch waits, IN THE STREAM
// (cuStreamWaitValue32: no CTA is resident while it waits -- a spinning gate kernel blocks the carve-out change of
// its own SM, measured), until every list CTA of the call has counted itself in Aux::d_started.
// PGX_PROBE_GATE=0 switches the gate off.
typedef int (*StreamWaitValue32)(cudaStream_t, unsigned long long, unsigned int, unsigned int);
std::atomic<bool> g_gate_refused{false};

StreamWaitValue32 stream_wait_value32()
{
    static const StreamWaitValue32 fn = [] {
        const char *env = getenv("PGX_PROBE_GATE");
        if (env && atoi(env) == 0) return static_cast<StreamWaitValue32>(nullptr);
        void *entry = nullptr;
        cudaDriverEntryPointQueryResult status;
        if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &entry, cudaEnableDefault, &status) != cudaSuccess ||
            status != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            return static_cast<StreamWaitValue32>(nullptr);
        }
        return reinterpret_cast<StreamWaitValue32>(entry);
    }();
    return fn;
}

int aux_init(Aux &a, int dev)
{
    PGX_CUDA(cudaStreamCreateWithFlags(&a.stream, cudaStreamNonBlocking));
    PGX_CUDA(cudaEventCreateWithFlags(&a.fork, cudaEventDisableTiming));
    PGX_CUDA(cudaEventCreateWithFlags(&a.join, cudaEventDisableTiming));
    PGX_CUDA(cudaMalloc(reinterpret_cast<void **>(&a.d_started), sizeof(unsigned int)));
    PGX_CUDA(cudaMemset(a.d_started, 0, sizeof(unsigned int)));
    a.expected = 0;
    a.device = dev;
    return PGX_OK;
}

int aux_for_device(Aux **out)
{
    static thread_local Aux aux[64];
    int dev = 0;
    PGX_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return fail(PGX_ERR_UNSUPPORTED, "device ordinal %d out of range", dev);
    Aux &a = aux[dev];
    if (a.device != dev) {
        if (int rc = aux_init(a, dev)) return rc;
    }
    *out = &a;
    return PGX_OK;
}

// prep + the two row kernels of n_perm permutations into ``work`` (histogram rows complete when the stream is)
template <bool P16>
int run_rows(const pgx_plan *plan, const uint16_t *d_perms, long long n_perm, const Work &work_in, int *d_bad_rows,
             cudaStream_t stream, Aux *own_aux, ProfileEvents *ev)
{
    Work work = work_in;
    work.trace = g_trace;
    work.trace_capacity = g_trace_capacity;
    DeviceLimits lim;
    if (int rc = device_limits(&lim)) return rc;
    const int n = plan->n_genomes;
    // prep: the shared-memory image of the histogram row when it fits twice per SM, else the gathering version
    const size_t bins_bytes = ((P16 ? 4 : 8) * static_cast<size_t>(n) + 15) & ~size_t(15);
    const size_t scatter_smem = bins_bytes + ((static_cast<size_t>(n) * sizeof(uint16_t) + 15) & ~size_t(15));
    static const bool no_scatter = getenv("PGX_PREP_GATHER") != nullptr;
    if (scatter_smem <= 110 * 1024 && !no_scatter) {
        if (scatter_smem > 48 * 1024)
            PGX_CUDA(cudaFuncSetAttribute(prep_scatter_kernel<P16>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(scatter_smem)));
        for (long long p0 = 0; p0 < n_perm; p0 += 2147483647ll) {
            const long long np = min(2147483647ll, n_perm - p0);
            Work w = work;
            w.hist += p0 * work.hist_stride;
            w.ranks += p0 * work.rank_stride;
            prep_scatter_kernel<P16><<<static_cast<unsigned>(np), 512, scatter_smem, stream>>>(*plan, d_perms + p0 * n, w, d_bad_rows);
            PGX_LAUNCH_CHECK("prep_scatter_kernel");
        }
    } else {
        const size_t prep_smem = static_cast<size_t>(n) * sizeof(uint16_t);
        // 16-byte accesses: N % 8 == 0 makes every permutation row aligned; the rank and histogram rows must be too
        const bool vec = n % 8 == 0 && work.hist_stride % 4 == 0 && work.rank_stride % 8 == 0 &&
                         ((reinterpret_cast<uintptr_t>(d_perms) | reinterpret_cast<uintptr_t>(work.hist) | reinterpret_cast<uintptr_t>(work.ranks)) & 15) == 0;
        auto prep = vec ? prep_kernel<P16, true> : prep_kernel<P16, false>;
        if (prep_smem > 48 * 1024)
            PGX_CUDA(cudaFuncSetAttribute(prep, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(prep_smem)));
        for (long long p0 = 0; p0 < n_perm; p0 += 2147483647ll) {
            const long long np = min(2147483647ll, n_perm - p0);
            Work w = work;
            w.hist += p0 * work.hist_stride;
            w.ranks += p0 * work.rank_stride;
            prep<<<static_cast<unsigned>(np), 256, prep_smem, stream>>>(*plan, d_perms + p0 * n, w, d_bad_rows);
            PGX_LAUNCH_CHECK("prep_kernel");
        }
    }
    if (ev) PGX_CUDA(cudaEventRecord(ev->prep_done, stream));
    // The two row kernels only add into the histogram, in any order: unless per-kernel timing is
    // on (or PGX_NO_OVERLAP is set), the probe kernel runs beside the list kernel on a second stream.
    Aux *aux = own_aux;
    const bool overlap = !ev && !g_no_overlap && plan->n_tasks > 0 && plan->n_long > 0;
    if (overlap) {
        if (!aux) {
            if (int rc = aux_for_device(&aux)) return rc;
        }
        PGX_CUDA(cudaEventRecord(aux->fork, stream));
        PGX_CUDA(cudaStreamWaitEvent(aux->stream, aux->fork, 0));
    }
    const StreamWaitValue32 gate = overlap && aux->d_started ? stream_wait_value32() : nullptr;
    unsigned list_grid = 0;
    if (plan->n_tasks > 0) {
        if (gate) work.started = aux->d_started;
        if (int rc = launch_list_b<P16>(*plan, d_perms, n_perm, work, lim, stream, &list_grid)) return rc;
    }
    if (ev) {
        ev->list_ran = plan->n_tasks > 0;
        ev->probe_ran = plan->n_long > 0;
        PGX_CUDA(cudaEventRecord(ev->list_done, stream));
    }
    if (overlap) {
        // launched AFTER the list kernel: one list CTA per SM first, probe CTAs fill what is left
        if (gate) {
            aux->expected += list_grid;
            // CU_STREAM_WAIT_VALUE_GEQ (0): until (int32_t)(*addr - value) >= 0, i.e. cyclic like the counter
            // (a driver that refuses stream memory operations just leaves the launch order to the block scheduler)
            if (!g_gate_refused.load(std::memory_order_relaxed) &&
                gate(aux->stream, reinterpret_cast<unsigned long long>(aux->d_started), aux->expected, 0u) != 0)
                g_gate_refused.store(true, std::memory_order_relaxed);
        }
        if (int rc = launch_probe<P16>(*plan, d_perms, n_perm, work, aux->stream)) return rc;
        PGX_CUDA(cudaEventRecord(aux->join, aux->stream));
        PGX_CUDA(cudaStreamWaitEvent(stream, aux->join, 0));
    } else if (plan->n_long > 0) {
        if (int rc = launch_probe<P16>(*plan, d_perms, n_perm, work, stream)) return rc;
    }
    if (ev) PGX_CUDA(cudaEventRecord(ev->probe_done, stream));
    return PGX_OK;
}

template <typename OutT, bool P16>
int launch_scan(const pgx_plan *plan, long long n_perm, const Work &work, OutT *d_out, cudaStream_t stream)
{
    const int n = plan->n_genomes;
    for (long long p0 = 0; p0 < n_perm; p0 += 2147483647ll) {
        const long long np = min(2147483647ll, n_perm - p0);
        Work w = work;
        w.hist += p0 * work.hist_stride;
        const unsigned grid = static_cast<unsigned>(np);
        // 16-byte accesses need 16-byte aligned rows: N % 8 == 0 and an aligned base
        const bool vec = n % 8 == 0 && ((reinterpret_cast<uintptr_t>(w.hist) | reinterpret_cast<uintptr_t>(d_out)) & 15) == 0 &&
                         (work.hist_stride % 4) == 0;
        if (vec) scan_kernel<OutT, P16, true><<<grid, SCAN_THREADS, 0, stream>>>(*plan, w, d_out + p0 * 2ll * n);
        else scan_kernel<OutT, P16, false><<<grid, SCAN_THREADS, 0, stream>>>(*plan, w, d_out + p0 * 2ll * n);
        PGX_LAUNCH_CHECK("scan_kernel");
    }
    return PGX_OK;
}

// Curves of n_perm permutations: d_work is an int32 [n_perm][2N] buffer (the output itself for OutT = int32).
// ``profiled``: bracket the kernels with the events of pgx_profile_enable (the device-pointer calls only).
template <typename OutT>
int run_curves(const pgx_plan *plan, const uint16_t *d_perms, long long n_perm, int32_t *d_work,
               OutT *d_out, cudaStream_t stream, bool profiled, Aux *own_aux = nullptr, int *d_bad_rows = nullptr)
{
    if (int rc = check_plan(plan)) return rc;
    if (n_perm < 0) return fail(PGX_ERR_INVALID, "n_perm < 0");
    if (n_perm == 0) return PGX_OK;
    if (!d_perms || !d_work || !d_out) return fail(PGX_ERR_INVALID, "null permutation / output pointer");
    const long long n = plan->n_genomes;
    const bool p16 = packed_bins(plan);
    ProfileEvents ev{};
    const bool profile = profiled && g_profile_on;
    if (profile) {
        PGX_CUDA(cudaEventCreate(&ev.begin));
        PGX_CUDA(cudaEventCreate(&ev.prep_done));
        PGX_CUDA(cudaEventCreate(&ev.list_done));
        PGX_CUDA(cudaEventCreate(&ev.probe_done));
        PGX_CUDA(cudaEventCreate(&ev.end));
        PGX_CUDA(cudaEventRecord(ev.begin, stream));
    }
    Work work;
    uint16_t *scratch = nullptr;
    if (p16) {
        // row of 8N bytes: [rank row 2N | free 2N | packed histogram 4N]
        work.hist = reinterpret_cast<uint32_t *>(d_work) + n;
        work.hist_stride = 2 * n;
        work.ranks = reinterpret_cast<uint16_t *>(d_work);
        work.rank_stride = 4 * n;
    } else {
        // int32 bins fill the row: the rank rows go to stream-ordered scratch from the device's pool
        PGX_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&scratch), sizeof(uint16_t) * n * n_perm, stream));
        work.hist = reinterpret_cast<uint32_t *>(d_work);
        work.hist_stride = 2 * n;
        work.ranks = scratch;
        work.rank_stride = n;
    }
    int rc = p16 ? run_rows<true>(plan, d_perms, n_perm, work, d_bad_rows, stream, own_aux, profile ? &ev : nullptr)
                 : run_rows<false>(plan, d_perms, n_perm, work, d_bad_rows, stream, own_aux, profile ? &ev : nullptr);
    if (scratch) cudaFreeAsync(scratch, stream);
    if (rc) return rc;
    rc = p16 ? launch_scan<OutT, true>(plan, n_perm, work, d_out, stream)
             : launch_scan<OutT, false>(plan, n_perm, work, d_out, stream);
    if (rc) return rc;
    if (profile) {
        PGX_CUDA(cudaEventRecord(ev.end, stream));
        std::lock_guard<std::mutex> lock(g_profile_mu);
        g_profile_events.push_back(ev);
    }
    return PGX_OK;
}

// ---------------------------------------------------------------------------------------------
// Host-buffer pipeline: permutations from host memory (or drawn from the numpy-legacy stream), curves into host
// memory.  Blocks of permutations travel through three slots: while one block's rows go down to the host, the next
// block's kernels run and the one after that uploads (or draws) its permutations.  With packed bins the device
// ships the histogram rows themselves -- the curves' steps, uint16 -- into pinned staging and a few host threads
// rebuild the curves straight into the caller's result; otherwise int32 / float64 curves are copied as they are.
// ---------------------------------------------------------------------------------------------
constexpr int SLOTS = 3;

// Packed histogram rows -> the SPLIT transfer format (pgx_expand.cpp): per row [pan head: head x u16][core head: head x
// u16][pan tail: (N - head) x u8][core tail: (N - head) x u8].  A step above 255 only occurs while the first genomes are
// added (C4: none after position 123), so the tails fit a byte; a row that breaks the rule raises ``overflow`` and its
// block travels again as uint16.  One CTA per row; entry e of the row (pan bins, then core bins) is half (e & 1) of
// word e >> 1.
__global__ void __launch_bounds__(256)
split_steps_kernel(const uint32_t *__restrict__ hist, const long long hist_stride, const int n, const int head,
                   uint8_t *__restrict__ out, const long long out_stride, int *__restrict__ overflow)
{
    const uint32_t *row = hist + static_cast<long long>(blockIdx.x) * hist_stride;
    uint8_t *dst = out + static_cast<long long>(blockIdx.x) * out_stride;
    uint16_t *head16 = reinterpret_cast<uint16_t *>(dst);                   // [2][head]
    uint8_t *tail8 = dst + 4ll * head;                                      // [2][n - head]
    int over = 0;
    for (int w = threadIdx.x; w < n; w += blockDim.x) {
        const uint32_t v = row[w];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int e = 2 * w + h;
            const uint32_t x = h ? v >> 16 : v & 0xffffu;
            const int half = e >= n ? 1 : 0, pos = e - half * n;
            if (pos < head) {
                head16[half * head + pos] = static_cast<uint16_t>(x);
            } else {
                tail8[static_cast<long long>(half) * (n - head) + (pos - head)] = static_cast<uint8_t>(min(x, 255u));
                over |= x > 255u;
            }
        }
    }
    if (__syncthreads_or(over) && threadIdx.x == 0) *overflow = 1;         // host-mapped flag: any writer writes 1
}

// First guess of ``head`` (PGX_SPLIT_HEAD; 0 = never split) -- doubled whenever a block overflows; the split format
// is used while 4 head <= N.
int split_head_initial()
{
    const char *env = getenv("PGX_SPLIT_HEAD");
    return env ? std::max(0, atoi(env)) : 512;
}

struct Slot {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    Aux aux;
    uint16_t *h_perm = nullptr;       // pinned; RNG mode only
    uint16_t *d_perm = nullptr;
    uint16_t *d_rank = nullptr;       // packed mode
    uint32_t *d_hist = nullptr;       // packed mode: [block][N] words; wide mode: int32 [block][2N]
    double *d_f64 = nullptr;          // wide mode, float64 output
    uint16_t *h_rows = nullptr;       // pinned staging: packed rows (uint16 [block][2N]); wide mode: curves as they are
    uint8_t *d_split = nullptr;       // packed mode: the block's rows in the split format
    int *h_overflow = nullptr;        // host-mapped: a tail step of the block did not fit a byte
    int head = 0;                     // split format of the block in flight (0: plain uint16 rows)
};

struct Pipe {
    int device = -1;
    long long block = 0, n = 0;
    bool packed = false, f64 = false, rng = false;
    int *bad_rows = nullptr;          // host-mapped counter of rows that are not permutations
    std::atomic<int> split_head{0};   // current ``head`` of the split format for this table size (0: plain uint16 rows)
    Slot slot[SLOTS];
};

void release(Pipe &b)
{
    for (auto &s : b.slot) {
        if (s.h_perm) cudaFreeHost(s.h_perm);
        if (s.h_rows) cudaFreeHost(s.h_rows);
        if (s.d_perm) cudaFree(s.d_perm);
        if (s.d_rank) cudaFree(s.d_rank);
        if (s.d_hist) cudaFree(s.d_hist);
        if (s.d_f64) cudaFree(s.d_f64);
        if (s.d_split) cudaFree(s.d_split);
        if (s.h_overflow) cudaFreeHost(s.h_overflow);
        if (s.done) cudaEventDestroy(s.done);
        if (s.stream) cudaStreamDestroy(s.stream);
        if (s.aux.stream) cudaStreamDestroy(s.aux.stream);
        if (s.aux.fork) cudaEventDestroy(s.aux.fork);
        if (s.aux.join) cudaEventDestroy(s.aux.join);
        if (s.aux.d_started) cudaFree(s.aux.d_started);
        s = Slot{};
    }
    if (b.bad_rows) cudaFreeHost(b.bad_rows);
    b.bad_rows = nullptr;
    b.device = -1;
    b.block = b.n = 0;
}

int acquire(Pipe &b, int device, long long block, long long n, bool packed, bool f64, bool rng)
{
    if (b.device == device && b.n == n && b.block >= block && b.packed == packed && (b.f64 || !f64 || packed) &&
        (b.rng || !rng))
        return PGX_OK;
    release(b);
    PGX_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&b.bad_rows), sizeof(int), cudaHostAllocMapped));
    *b.bad_rows = 0;
    for (auto &s : b.slot) {
        PGX_CUDA(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        PGX_CUDA(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
        if (int rc = aux_init(s.aux, device)) return rc;
        if (rng) PGX_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&s.h_perm), sizeof(uint16_t) * block * n, cudaHostAllocDefault));
        PGX_CUDA(cudaMalloc(reinterpret_cast<void **>(&s.d_perm), sizeof(uint16_t) * block * n));
        if (packed) {
            PGX_CUDA(cudaMalloc(reinterpret_cast<void **>(&s.d_rank), sizeof(uint16_t) * block * n));
            PGX_CUDA(cudaMalloc(reinterpret_cast<void **>(&s.d_hist), sizeof(uint32_t) * block * n));
            PGX_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&s.h_rows), sizeof(uint16_t) * block * 2 * n, cudaHostAllocDefault));
            PGX_CUDA(cudaMalloc(reinterpret_cast<void **>(&s.d_split), sizeof(uint16_t) * block * 2 * n));      // never more than the plain rows
            PGX_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&s.h_overflow), sizeof(int), cudaHostAllocMapped));
            *s.h_overflow = 0;
        } else {
            PGX_CUDA(cudaMalloc(reinterpret_cast<void **>(&s.d_hist), sizeof(int32_t) * block * 2 * n));
            if (f64) PGX_CUDA(cudaMalloc(reinterpret_cast<void **>(&s.d_f64), sizeof(double) * block * 2 * n));
            PGX_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&s.h_rows), (f64 ? sizeof(double) : sizeof(int32_t)) * block * 2 * n,
                                   cudaHostAllocDefault));
        }
    }
    b.device = device;
    b.block = block;
    b.n = n;
    b.packed = packed;
    b.f64 = f64;
    b.rng = rng;
    const int head = split_head_initial();
    b.split_head.store(packed && head > 0 && 4ll * head <= n ? head : 0);
    return PGX_OK;
}

std::mutex g_pipe_mu;              // one host-buffer call at a time per process (it owns the staging)
Pipe g_pipe;

// h_perms != nullptr: the caller's permutations; otherwise they are drawn from the numpy-legacy MT19937 state.
int host_pipeline(const pgx_plan *plan, const uint16_t *h_perms, uint32_t *mt_key, int32_t *mt_pos, long long n_perm,
                  void *h_curves, bool out_f64, long long perms_per_block)
{
    const long long n = plan->n_genomes;
    const bool rng = h_perms == nullptr;
    const bool packed = packed_bins(plan);
    // Block schedule.  About 32 MB of packed rows per block: large enough for the persistent list CTAs to amortise
    // their rank tables, small enough that the first upload and the last download + rebuild, which nothing overlaps,
    // stay short (a schedule with larger middle blocks measured slower: 15.5 vs 14.5 ms per 10,000 permutations of
    // C4).  The RNG-fed call is bound by the serial shuffle stream: short blocks, halving at the end so that little is
    // left to do when the last shuffle is drawn.
    std::vector<long long> first_perm;          // block k covers [first_perm[k], first_perm[k + 1])
    long long max_block = 0;
    {
        long long base = perms_per_block;
        const bool uniform = base > 0;
        if (!uniform) {
            base = rng ? std::max(32ll, std::min(4096ll, (8ll << 20) / (4 * n))) : std::max(64ll, std::min(1ll << 16, (32ll << 20) / (4 * n)));
            base = (base + 7) / 8 * 8;
        }
        long long at = 0;
        first_perm.push_back(0);
        while (at < n_perm) {
            const long long left = n_perm - at;
            long long take = base;
            if (!uniform && rng) {
                if (left < 2 * base) take = std::max(32ll, (left / 2 + 7) / 8 * 8);
            }
            take = std::min(take, left);
            at += take;
            first_perm.push_back(at);
            max_block = std::max(max_block, take);
        }
        // the staging is sized for the largest block of the default schedule even when this call is shorter, so that
        // the next call need not reallocate
        if (!uniform) max_block = std::max(max_block, base);
    }
    std::lock_guard<std::mutex> lock(g_pipe_mu);
    int dev = 0;
    PGX_CUDA(cudaGetDevice(&dev));
    Pipe &buf = g_pipe;
    if (int rc = acquire(buf, dev, max_block, n, packed, out_f64, rng)) return rc;
    const long long n_blocks = static_cast<long long>(first_perm.size()) - 1;
    *buf.bad_rows = 0;
    int *d_bad_rows = nullptr;
    PGX_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void **>(&d_bad_rows), buf.bad_rows, 0));
    {
        // The result is usually fresh memory: ask for huge pages so that filling it costs one page
        // fault per 2 MB instead of one per 4 KB (a hint; ignored where THP is off).
        const size_t elem = out_f64 ? sizeof(double) : sizeof(int32_t);
        const uintptr_t page = 2u << 20;
        const uintptr_t lo = (reinterpret_cast<uintptr_t>(h_curves) + page - 1) & ~(page - 1);
        const uintptr_t hi = (reinterpret_cast<uintptr_t>(h_curves) + elem * 2ull * n * n_perm) & ~(page - 1);
        if (hi > lo) madvise(reinterpret_cast<void *>(lo), hi - lo, MADV_HUGEPAGE);
    }
    // PGX_ESTIMATE_TRACE=1: per-block timeline of the pipeline on stderr (development aid)
    const bool trace = getenv("PGX_ESTIMATE_TRACE") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    auto since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };

    // issuing thread (the caller): draws / uploads block k, enqueues its kernels and its download; the movers
    // (copy threads) wait for block k's download and rebuild / copy its rows into the result.  Both sides poll atomic
    // counters: on the virtualised hosts this runs on, waking a sleeping thread costs 0.2-0.5 ms.
    std::atomic<long long> issued{0}, retired{0};
    std::atomic<int> failed{0};
    std::vector<std::atomic<int>> parts_done(static_cast<size_t>(n_blocks)), refetch(static_cast<size_t>(n_blocks));
    for (auto &c : parts_done) c.store(0, std::memory_order_relaxed);
    for (auto &c : refetch) c.store(0, std::memory_order_relaxed);
    int movers = std::max(1, std::min(rng ? 6 : 12, static_cast<int>(std::thread::hardware_concurrency()) - (rng ? 3 : 2)));
    if (const char *env = getenv("PGX_COPY_THREADS")) movers = std::max(1, std::min(32, atoi(env)));
    movers = static_cast<int>(std::max<long long>(1, std::min<long long>(movers, max_block * n / 32768)));
    const size_t out_elem = out_f64 ? sizeof(double) : sizeof(int32_t);
    auto mover = [&](int t) {
        cudaSetDevice(dev);
        for (long long k = 0; k < n_blocks; ++k) {
            while (issued.load(std::memory_order_acquire) <= k) {
                if (failed.load(std::memory_order_relaxed)) return;
                std::this_thread::yield();
            }
            Slot &s = buf.slot[k % SLOTS];
            if (cudaEventSynchronize(s.done) != cudaSuccess) {
                failed.store(1);
                return;
            }
            const long long p0 = first_perm[k], cnt = first_perm[k + 1] - p0;
            const long long r0 = cnt * t / movers, r1 = cnt * (t + 1) / movers;
            char *dst = static_cast<char *>(h_curves) + out_elem * 2 * n * p0;
            if (packed && s.head > 0 && *s.h_overflow) {
                // a tail step above 255: the block's plain uint16 rows are still in the slot; the first mover to get
                // here fetches them, the others wait, and later blocks get a longer head
                int expect = 0;
                std::atomic<int> &state = refetch[static_cast<size_t>(k)];
                if (state.compare_exchange_strong(expect, 1, std::memory_order_acq_rel)) {
                    int next = 2 * s.head;
                    if (4ll * next > n) next = 0;
                    int seen = buf.split_head.load();
                    while (seen == s.head && !buf.split_head.compare_exchange_weak(seen, next)) {}
                    const bool ok = cudaMemcpyAsync(s.h_rows, s.d_hist, sizeof(uint16_t) * cnt * 2 * n, cudaMemcpyDeviceToHost, s.stream) == cudaSuccess &&
                                    cudaStreamSynchronize(s.stream) == cudaSuccess;
                    if (trace) fprintf(stderr, "[pgx trace] block %lld: head %d overflowed, fetched as uint16 (%.2f ms)\n", k, s.head, since());
                    state.store(ok ? 2 : 3, std::memory_order_release);
                }
                int st;
                while ((st = state.load(std::memory_order_acquire)) < 2) std::this_thread::yield();
                if (st == 3) {
                    failed.store(1);
                    return;
                }
                expand_delta_rows(s.h_rows, r0, r1, n, dst, out_f64);
            } else if (packed && s.head > 0) {
                expand_split_rows(reinterpret_cast<const uint8_t *>(s.h_rows), r0, r1, n, s.head, dst, out_f64);
            } else if (packed) {
                expand_delta_rows(s.h_rows, r0, r1, n, dst, out_f64);
            } else {
                const size_t row = out_elem * 2 * n;
                memcpy(dst + row * r0, reinterpret_cast<const char *>(s.h_rows) + row * r0, row * (r1 - r0));
            }
            if (parts_done[static_cast<size_t>(k)].fetch_add(1, std::memory_order_acq_rel) + 1 == movers) {
                retired.store(k + 1, std::memory_order_release);     // blocks retire in order: every mover walks them in order
                if (trace) fprintf(stderr, "[pgx trace] block %lld: in the result %.2f ms\n", k, since());
            }
        }
    };
    std::vector<std::thread> pool;
    for (int t = 0; t < movers; ++t) pool.emplace_back(mover, t);

    int rc = PGX_OK;
    for (long long k = 0; k < n_blocks && !rc; ++k) {
        while (retired.load(std::memory_order_acquire) + SLOTS <= k) {
            if (failed.load(std::memory_order_relaxed)) break;
            std::this_thread::yield();
        }
        if (failed.load(std::memory_order_relaxed)) break;
        Slot &s = buf.slot[k % SLOTS];
        const long long p0 = first_perm[k], cnt = first_perm[k + 1] - p0;
        const double t_wait = since();
        const uint16_t *src = h_perms ? h_perms + p0 * n : s.h_perm;
        if (rng) rc = pgx_legacy_shuffles(mt_key, mt_pos, n, cnt, s.h_perm);
        const double t_rng = since();
        if (!rc && cudaMemcpyAsync(s.d_perm, src, sizeof(uint16_t) * cnt * n, cudaMemcpyHostToDevice, s.stream) != cudaSuccess)
            rc = fail(PGX_ERR_CUDA, "H2D copy of the permutations failed: %s", cudaGetErrorString(cudaGetLastError()));
        if (!rc && packed) {
            Work work{s.d_hist, n, s.d_rank, n};
            rc = run_rows<true>(plan, s.d_perm, cnt, work, d_bad_rows, s.stream, &s.aux, nullptr);
            s.head = buf.split_head.load();
            if (!rc && s.head > 0) {
                // uint16 heads + uint8 tails: 2N + 2 head bytes per row over PCIe and through the host's memory
                int *d_overflow = nullptr;
                *s.h_overflow = 0;
                if (cudaHostGetDevicePointer(reinterpret_cast<void **>(&d_overflow), s.h_overflow, 0) != cudaSuccess)
                    rc = fail(PGX_ERR_CUDA, "cudaHostGetDevicePointer failed: %s", cudaGetErrorString(cudaGetLastError()));
                const long long row_bytes = 2 * n + 2ll * s.head;
                if (!rc) {
                    split_steps_kernel<<<static_cast<unsigned>(cnt), 256, 0, s.stream>>>(s.d_hist, n, static_cast<int>(n), s.head, s.d_split,
                                                                                         row_bytes, d_overflow);
                    if (cudaGetLastError() != cudaSuccess) rc = fail(PGX_ERR_CUDA, "launch of split_steps_kernel failed");
                    else g_launches.fetch_add(1, std::memory_order_relaxed);
                }
                if (!rc && cudaMemcpyAsync(s.h_rows, s.d_split, static_cast<size_t>(row_bytes) * cnt, cudaMemcpyDeviceToHost, s.stream) != cudaSuccess)
                    rc = fail(PGX_ERR_CUDA, "D2H copy of the curve steps failed: %s", cudaGetErrorString(cudaGetLastError()));
            } else if (!rc && cudaMemcpyAsync(s.h_rows, s.d_hist, sizeof(uint16_t) * cnt * 2 * n, cudaMemcpyDeviceToHost, s.stream) != cudaSuccess)
                rc = fail(PGX_ERR_CUDA, "D2H copy of the curve steps failed: %s", cudaGetErrorString(cudaGetLastError()));
        } else if (!rc) {
            s.head = 0;
            // (host-buffer calls are never profiled, in either bin format: include/pgx.h)
            rc = out_f64 ? run_curves<double>(plan, s.d_perm, cnt, reinterpret_cast<int32_t *>(s.d_hist), s.d_f64, s.stream, false,
                                              &s.aux, d_bad_rows)
                         : run_curves<int32_t>(plan, s.d_perm, cnt, reinterpret_cast<int32_t *>(s.d_hist),
                                               reinterpret_cast<int32_t *>(s.d_hist), s.stream, false, &s.aux, d_bad_rows);
            const void *from = out_f64 ? static_cast<const void *>(s.d_f64) : static_cast<const void *>(s.d_hist);
            if (!rc && cudaMemcpyAsync(s.h_rows, from, out_elem * cnt * 2 * n, cudaMemcpyDeviceToHost, s.stream) != cudaSuccess)
                rc = fail(PGX_ERR_CUDA, "D2H copy of the curves failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
        if (!rc && cudaEventRecord(s.done, s.stream) != cudaSuccess) rc = fail(PGX_ERR_CUDA, "event record failed");
        if (trace) fprintf(stderr, "[pgx trace] block %lld: waited until %.2f, rng until %.2f, enqueued %.2f ms\n", k, t_wait, t_rng, since());
        if (rc) {
            failed.store(1);
            break;
        }
        issued.store(k + 1, std::memory_order_release);
    }
    if (rc) failed.store(1);
    for (auto &th : pool) th.join();
    if (!rc && failed.load()) rc = fail(PGX_ERR_CUDA, "a block of curves failed on the device: %s", cudaGetErrorString(cudaGetLastError()));
    if (rc) {
        char text[512];
        snprintf(text, sizeof(text), "%s", pgx_last_error());
        for (auto &s : buf.slot) cudaStreamSynchronize(s.stream);
        return fail(rc, "%s", text);
    }
    if (*buf.bad_rows)
        return fail(PGX_ERR_INVALID, "%d of the %lld genome orders are not permutations of 0 .. %lld", *buf.bad_rows, n_perm, n - 1);
    return PGX_OK;
}

}  // namespace

}  // namespace pgx

extern "C" {

int pgx_pan_core_curves(const pgx_plan *plan, const uint16_t *d_perms, int64_t n_perm,
                        int32_t *d_curves, void *stream)
{
    return pgx::run_curves<int32_t>(plan, d_perms, n_perm, d_curves, d_curves,
                                    static_cast<cudaStream_t>(stream), true);
}

int pgx_pan_core_curves_f64(const pgx_plan *plan, const uint16_t *d_perms, int64_t n_perm,
                            int32_t *d_hist, double *d_curves, void *stream)
{
    return pgx::run_curves<double>(plan, d_perms, n_perm, d_hist, d_curves,
                                   static_cast<cudaStream_t>(stream), true);
}

int pgx_pan_core_curves_host(const pgx_plan *plan, const uint16_t *h_perms, int64_t n_perm,
                             void *h_curves, int32_t out_f64, int64_t perms_per_block)
{
    if (int rc = pgx::check_plan(plan)) return rc;
    if (n_perm < 0) return pgx::fail(PGX_ERR_INVALID, "n_perm < 0");
    if (n_perm == 0) return PGX_OK;
    if (!h_perms || !h_curves) return pgx::fail(PGX_ERR_INVALID, "null host pointer");
    return pgx::host_pipeline(plan, h_perms, nullptr, nullptr, n_perm, h_curves, out_f64 != 0, perms_per_block);
}

int pgx_estimate_pan_core(const pgx_plan *plan, uint32_t *mt_key, int32_t *mt_pos, int64_t n_iter,
                          double *h_curves, int64_t perms_per_block)
{
    if (int rc = pgx::check_plan(plan)) return rc;
    if (n_iter < 0) return pgx::fail(PGX_ERR_INVALID, "n_iter < 0");
    if (!mt_key || !mt_pos || (!h_curves && n_iter > 0)) return pgx::fail(PGX_ERR_INVALID, "null pointer");
    if (n_iter == 0) return PGX_OK;
    return pgx::host_pipeline(plan, nullptr, mt_key, mt_pos, n_iter, h_curves, true, perms_per_block);
}

int pgx_split_head(void)
{
    return pgx::g_pipe.split_head.load();
}

int pgx_profile_enable(int32_t on)
{
    pgx::g_profile_on = on != 0;
    return PGX_OK;
}

int pgx_profile_read(double *list_ms, double *probe_ms, double *scan_ms, int64_t *calls)
{
    std::lock_guard<std::mutex> lock(pgx::g_profile_mu);
    double a = 0.0, b = 0.0, c = 0.0;
    for (auto &ev : pgx::g_profile_events) {
        float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
        PGX_CUDA(cudaEventSynchronize(ev.end));
        PGX_CUDA(cudaEventElapsedTime(&t0, ev.begin, ev.prep_done));
        PGX_CUDA(cudaEventElapsedTime(&t1, ev.prep_done, ev.list_done));
        PGX_CUDA(cudaEventElapsedTime(&t2, ev.list_done, ev.probe_done));
        PGX_CUDA(cudaEventElapsedTime(&t3, ev.probe_done, ev.end));
        if (ev.list_ran) a += t1;
        if (ev.probe_ran) b += t2;
        c += t0 + t3;                    // prep + scan: everything that is not a row kernel
        cudaEventDestroy(ev.begin);
        cudaEventDestroy(ev.prep_done);
        cudaEventDestroy(ev.list_done);
        cudaEventDestroy(ev.probe_done);
        cudaEventDestroy(ev.end);
    }
    if (list_ms) *list_ms = a;
    if (probe_ms) *probe_ms = b;
    if (scan_ms) *scan_ms = c;
    if (calls) *calls = static_cast<int64_t>(pgx::g_profile_events.size());
    pgx::g_profile_events.clear();
    return PGX_OK;
}

int pgx_set_trace(void *d_trace, int64_t capacity_records)
{
    pgx::g_trace = static_cast<unsigned long long *>(d_trace);
    pgx::g_trace_capacity = d_trace ? capacity_records : 0;
    return PGX_OK;
}

int pgx_set_tuning(int32_t perms_per_cta, int32_t row_splits, int32_t threads_per_cta)
{
    pgx::g_tuning.perms_per_cta = perms_per_cta;
    pgx::g_tuning.row_splits = row_splits;
    pgx::g_tuning.threads = threads_per_cta;
    return PGX_OK;
}

}  // extern "C"
