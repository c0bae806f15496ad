// Genome x genome shared-gene matrix S = X^T X of a planned table (pgx_shared_genes), the per-genome sums of
// genomic-fluidity distances (pgx_fluidity_rows), and the gene-pair overlap histograms and exact rarefaction moments
// further down (pgx_plan_spectrum, pgx_pair_overlap_histograms, pgx_rarefaction_moments), whose GEMM shares the
// mainloop of S.  The decomposition of S over the plan's gene classes is stated in
// include/pgx.h; oracle/shared_np.py restates it in numpy.
//
//   count   u[k] / p[k] = absent / present list rows listing genome k, |A|, sum(w_absent) and the bitmap popcount
//           of genome 0, then n_full (universal genes) from genome 0's diagonal
//   init    closed-form and vector terms into the upper triangle, colsum on the diagonal
//   pairs   +1 per genome pair of every sorted list row (present and absent lists alike)
//   expand  a K-slab of the bitmap rows into E [N][K_slab] uint8 (0 / 1), genome-major
//   gemm    S += E E^T on the tensor cores (tcgen05.mma kind::i8, TMA loads with 128-byte swizzle, s32 accumulators in
//           tensor memory), upper-triangle tiles only; the epilogue adds the tile into S above the diagonal
//   mirror  upper triangle -> lower triangle
#include "pgx_common.cuh"

#include <cuda.h>
#include <cudaTypedefs.h>
#include <limits.h>

namespace {

constexpr int32_t MAX_GENOMES = 65503;

// ---- count ------------------------------------------------------------------------------------------------------
// header of the workspace during count / init (E overwrites it afterwards)
struct CountHeader {
    int32_t n_full, n_absent_rows, sum_w_absent, bitmap_pop0;
};

// one warp per task: every row of a task has the task's list kind (bit 24 of word 1)
__global__ void shared_count_kernel(const int32_t *__restrict__ tasks, int32_t n_tasks,
                                    const uint16_t *__restrict__ sorted_idx, const int32_t *__restrict__ sorted_ptr,
                                    int32_t *__restrict__ u, int32_t *__restrict__ p, CountHeader *hdr)
{
    const int lane = threadIdx.x & 31;
    const int32_t warp = static_cast<int32_t>((blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5);
    const int32_t n_warps = static_cast<int32_t>((gridDim.x * static_cast<int64_t>(blockDim.x)) >> 5);
    for (int32_t t = warp; t < n_tasks; t += n_warps) {
        const int4 task = reinterpret_cast<const int4 *>(tasks)[t];
        const bool absent = (task.y >> 24) & 1;
        int32_t *hist = absent ? u : p;
        if (absent && lane == 0) atomicAdd(&hdr->n_absent_rows, task.w);
        const int32_t e0 = sorted_ptr[task.z], e1 = sorted_ptr[task.z + task.w];
        for (int32_t e = e0 + lane; e < e1; e += 32) atomicAdd(&hist[sorted_idx[e]], 1);
    }
}

// one block: sum(w_absent) and the popcount of genome 0's bitmap lines
__global__ void shared_count_vectors_kernel(const int32_t *__restrict__ w_absent, int32_t n,
                                            const uint32_t *__restrict__ bits, int32_t n_superblocks,
                                            int32_t slice_words, CountHeader *hdr)
{
    int32_t s = 0, pop = 0;
    for (int32_t c = threadIdx.x; c < n; c += blockDim.x) s += w_absent[c];
    const int32_t line = 32 * slice_words;
    for (int32_t i = threadIdx.x; i < n_superblocks * line; i += blockDim.x) {
        const int32_t sb = i / line, w = i % line;
        pop += __popc(bits[(static_cast<int64_t>(sb) * n) * line + w]);
    }
    atomicAdd(&hdr->sum_w_absent, s);
    atomicAdd(&hdr->bitmap_pop0, pop);
}

// n_full = S[0,0] minus every other class's contribution to it
__global__ void shared_full_kernel(const int32_t *__restrict__ colsum, const int32_t *__restrict__ w_present,
                                   const int32_t *__restrict__ w_absent, const int32_t *__restrict__ u,
                                   const int32_t *__restrict__ p, CountHeader *hdr)
{
    hdr->n_full = colsum[0] - (hdr->sum_w_absent - w_absent[0]) - w_present[0] - (hdr->n_absent_rows - u[0]) - p[0] -
                  hdr->bitmap_pop0;
}

// ---- init -------------------------------------------------------------------------------------------------------
// one block per genome k: S[k, k] = colsum[k], S[k, l > k] = the closed-form and vector terms
__global__ void shared_init_kernel(int32_t n, const int32_t *__restrict__ colsum, const int32_t *__restrict__ w_absent,
                                   const int32_t *__restrict__ u, const CountHeader *__restrict__ hdr,
                                   int32_t *__restrict__ shared)
{
    const int32_t k = blockIdx.x;
    const int32_t base = hdr->n_full + hdr->sum_w_absent + hdr->n_absent_rows - w_absent[k] - u[k];
    int32_t *row = shared + static_cast<int64_t>(k) * n;
    if (threadIdx.x == 0) row[k] = colsum[k];
    for (int32_t l = k + 1 + threadIdx.x; l < n; l += blockDim.x) row[l] = base - w_absent[l] - u[l];
}

// ---- pairs ------------------------------------------------------------------------------------------------------
// one warp per list row: +1 on S[a, b] for every pair a < b of its sorted list
__global__ void shared_pairs_kernel(int32_t n_rows, const uint16_t *__restrict__ sorted_idx,
                                    const int32_t *__restrict__ sorted_ptr, int32_t n, int32_t *__restrict__ shared)
{
    const int lane = threadIdx.x & 31;
    const int32_t warp = static_cast<int32_t>((blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5);
    const int32_t n_warps = static_cast<int32_t>((gridDim.x * static_cast<int64_t>(blockDim.x)) >> 5);
    for (int32_t r = warp; r < n_rows; r += n_warps) {
        const int32_t e0 = sorted_ptr[r], e1 = sorted_ptr[r + 1];
        for (int32_t i = e0; i + 1 < e1; ++i) {
            int32_t *row = shared + static_cast<int64_t>(sorted_idx[i]) * n;
            for (int32_t j = i + 1 + lane; j < e1; j += 32) atomicAdd(&row[sorted_idx[j]], 1);
        }
    }
}

// ---- expand -----------------------------------------------------------------------------------------------------
// one thread per (genome, 32 rows): bitmap rows k0 .. k0 + k_cur - 1 of genome c -> E[c][0 .. k_cur) as 0 / 1 bytes
__global__ void shared_expand_kernel(const uint32_t *__restrict__ bits, int32_t n, int32_t slice_words, int64_t k0,
                                     int64_t k_cur, int64_t k_slab, uint8_t *__restrict__ e)
{
    const int64_t words = k_cur >> 5;
    const int64_t total = words * n;
    const int32_t line = 32 * slice_words, sb_rows = 1024 * slice_words;
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int32_t c = static_cast<int32_t>(i / words);
        const int64_t w = i % words;
        const int64_t k = k0 + 32 * w;
        const int64_t sb = k / sb_rows;
        const uint32_t v = __ldg(&bits[(sb * n + c) * line + (k % sb_rows) / 32]);
        uint32_t out[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const uint32_t nib = (v >> (4 * q)) & 0xfu;       // 4 rows -> 4 bytes
            out[q] = (nib & 1u) | ((nib >> 1) & 1u) << 8 | ((nib >> 2) & 1u) << 16 | (nib >> 3) << 24;
        }
        uint4 *dst = reinterpret_cast<uint4 *>(e + static_cast<int64_t>(c) * k_slab + 32 * w);
        dst[0] = make_uint4(out[0], out[1], out[2], out[3]);
        dst[1] = make_uint4(out[4], out[5], out[6], out[7]);
    }
}

// ---- gemm: S += E E^T on tcgen05 ---------------------------------------------------------------------------------
constexpr int BM = 128, BN = 256, BK = 128;               // BK bytes = one 128-byte swizzle atom of uint8
constexpr int UMMA_K = 32;                                 // K of one kind::i8 MMA
constexpr int STAGES = 4;
constexpr int A_BYTES = BM * BK, B_BYTES = BN * BK, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int GEMM_SMEM = STAGES * STAGE_BYTES + 1024;   // + alignment of the stages to 1,024 bytes
constexpr int GEMM_THREADS = 128;                          // warp 0 TMA, warp 1 MMA, warp 2 TMEM owner; all 4 epilogue
constexpr uint32_t TMEM_COLS = BN;                         // one 128 x 256 s32 accumulator

// instruction descriptor: D s32 (bits 4-5 = 2), A and B u8 (bits 7-9, 10-12 = 0), both K-major, N >> 3 at bit 17,
// M >> 4 at bit 24
constexpr uint32_t IDESC = (2u << 4) | (uint32_t(BN >> 3) << 17) | (uint32_t(BM >> 4) << 24);

__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(bar), "r"(parity)
                     : "memory");
    } while (!done);
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int32_t c0, int32_t c1, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar)
                 : "memory");
}

// shared-memory matrix descriptor of a K-major operand in 128-byte-swizzled 8-row groups of 1,024 bytes
__device__ __forceinline__ uint64_t sw128_desc(uint32_t addr)
{
    return static_cast<uint64_t>((addr & 0x3ffffu) >> 4)   // start address
           | static_cast<uint64_t>(1) << 16                // leading byte offset (unused with this swizzle)
           | static_cast<uint64_t>(1024 >> 4) << 32        // stride byte offset: 8 rows x 128 bytes
           | static_cast<uint64_t>(1) << 46                // descriptor version of sm_100
           | static_cast<uint64_t>(2) << 61;               // 128-byte swizzle
}

__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t a, uint64_t b, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "setp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(a), "l"(b), "r"(IDESC), "r"(accumulate)
                 : "memory");
}

__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void tmem_ld_32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]),
                   "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]),
                   "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]),
                   "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Tile order: groups of GROUP_ROWS row tiles; inside a group, column tile by column tile (from the first one that
// reaches the group's diagonal), the group's row tiles in turn.  A wave of CTAs then covers a block of about
// GROUP_ROWS x 9 tiles, whose A and B panels it shares through L2, instead of a strip of one row tile whose B panels
// every CTA would fetch alone from HBM.
constexpr int32_t GROUP_ROWS = 16;

__host__ __device__ inline int64_t group_tiles(int32_t g, int32_t col_tiles)
{
    return int64_t(col_tiles - g * (GROUP_ROWS / 2)) * GROUP_ROWS;
}

// One CTA per tile of the order above over the rows 0 .. n - 1 of the operand ``map`` describes, E E^T on tcgen05.
// A tile without an entry above the diagonal (cb < rb / 2), or one the epilogue skips, returns at once.  The epilogue
// reads the tile's accumulator from tensor memory: Epi::skip(rb, cb) and Epi::run(tmem, warp, lane, m0, n0, n, stages),
// where ``stages`` (the shared-memory stage buffers, free once the MMAs are done) is its scratch.
template <class Epi>
__device__ __forceinline__ void gemm_tiles(const CUtensorMap &map, int32_t n, int32_t k_blocks, const Epi &epi)
{
    const int32_t row_tiles = (n + BM - 1) / BM, col_tiles = (n + BN - 1) / BN;
    int64_t id = blockIdx.x;
    int32_t g = 0;
    while (id >= group_tiles(g, col_tiles)) id -= group_tiles(g++, col_tiles);
    const int32_t cb = g * (GROUP_ROWS / 2) + static_cast<int32_t>(id / GROUP_ROWS);
    const int32_t rb = g * GROUP_ROWS + static_cast<int32_t>(id % GROUP_ROWS);
    if (rb >= row_tiles || cb < rb / 2 || epi.skip(rb, cb)) return;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[STAGES], empty_bar[STAGES], done_bar;
    __shared__ uint32_t tmem_base;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t stages = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int32_t m0 = rb * BM, n0 = cb * BN;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(smem_u32(&full_bar[s]), 1);
            mbar_init(smem_u32(&empty_bar[s]), 1);
        }
        mbar_init(smem_u32(&done_bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map)) : "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(&tmem_base)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base;

    if (warp == 0 && lane == 0) {                          // TMA producer
        for (int32_t kb = 0; kb < k_blocks; ++kb) {
            const int s = kb % STAGES;
            if (kb >= STAGES) mbar_wait(smem_u32(&empty_bar[s]), ((kb / STAGES) & 1) ^ 1);
            const uint32_t a = stages + s * STAGE_BYTES, bar = smem_u32(&full_bar[s]);
            mbar_expect_tx(bar, STAGE_BYTES);
            tma_load_2d(a, &map, kb * BK, m0, bar);
            tma_load_2d(a + A_BYTES, &map, kb * BK, n0, bar);
            tma_load_2d(a + A_BYTES + BM * BK, &map, kb * BK, n0 + BM, bar);
        }
    } else if (warp == 1 && lane == 0) {                   // MMA issuer
        for (int32_t kb = 0; kb < k_blocks; ++kb) {
            const int s = kb % STAGES;
            mbar_wait(smem_u32(&full_bar[s]), (kb / STAGES) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t a = stages + s * STAGE_BYTES;
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k)
                umma_i8(tmem, sw128_desc(a + k * UMMA_K), sw128_desc(a + A_BYTES + k * UMMA_K), (kb | k) != 0);
            umma_commit(smem_u32(&empty_bar[s]));          // frees the stage once these MMAs have read it
        }
        umma_commit(smem_u32(&done_bar));
    }
    __syncwarp();

    // epilogue: warp w owns TMEM lanes 32 w .. 32 w + 31 = tile rows; thread = one row
    mbar_wait(smem_u32(&done_bar), 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    epi.run(tmem, warp, lane, m0, n0, n, stages);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
    }
}

// S epilogue: the tile, 32 columns per load, added into S above the diagonal
struct SharedEpilogue {
    int32_t *shared;

    __device__ __forceinline__ bool skip(int32_t, int32_t) const { return false; }

    __device__ __forceinline__ void run(uint32_t tmem, int warp, int lane, int32_t m0, int32_t n0, int32_t n,
                                        uint32_t) const
    {
        const int32_t row = m0 + 32 * warp + lane;
        int32_t *dst = shared + static_cast<int64_t>(row) * n;
        const bool vec = (n & 3) == 0;
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
            uint32_t acc[32];
            tmem_ld_32(tmem + (static_cast<uint32_t>(32 * warp) << 16) + c, acc);
            const int32_t col0 = n0 + c;
            if (row >= n || col0 + 31 <= row || col0 >= n) continue;
            if (vec && col0 > row && col0 + 32 <= n) {
                int4 *p = reinterpret_cast<int4 *>(dst + col0);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    int4 v = p[q];
                    v.x += static_cast<int32_t>(acc[4 * q]);
                    v.y += static_cast<int32_t>(acc[4 * q + 1]);
                    v.z += static_cast<int32_t>(acc[4 * q + 2]);
                    v.w += static_cast<int32_t>(acc[4 * q + 3]);
                    p[q] = v;
                }
            } else {
#pragma unroll
                for (int q = 0; q < 32; ++q) {
                    const int32_t col = col0 + q;
                    if (col > row && col < n) dst[col] += static_cast<int32_t>(acc[q]);
                }
            }
        }
    }
};

__global__ void __launch_bounds__(GEMM_THREADS, 1) shared_gemm_kernel(const __grid_constant__ CUtensorMap map,
                                                                       int32_t n, int32_t k_blocks,
                                                                       int32_t *__restrict__ shared)
{
    gemm_tiles(map, n, k_blocks, SharedEpilogue{shared});
}

// ---- mirror -----------------------------------------------------------------------------------------------------
// 32 x 32 tiles on or above the diagonal, transposed through shared memory: S[c, r] = S[r, c] for r < c
__global__ void shared_mirror_kernel(int32_t n, int32_t *__restrict__ shared)
{
    const int32_t ti = blockIdx.y, tj = blockIdx.x;
    if (ti > tj) return;
    __shared__ int32_t tile[32][33];
    const int32_t r0 = ti * 32, c0 = tj * 32;
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        const int32_t r = r0 + y, c = c0 + threadIdx.x;
        if (r < n && c < n) tile[y][threadIdx.x] = shared[static_cast<int64_t>(r) * n + c];
    }
    __syncthreads();
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        const int32_t dst_row = c0 + y, dst_col = r0 + threadIdx.x;      // = source (row dst_col, col dst_row)
        if (dst_row < n && dst_col < dst_row) shared[static_cast<int64_t>(dst_row) * n + dst_col] = tile[threadIdx.x][y];
    }
}

// ---- fluidity rows ----------------------------------------------------------------------------------------------
// block = ROWS genomes k; thread t sums l = t, t + 256, ... in order, then a fixed shared-memory tree: bit-reproducible
constexpr int ROW_THREADS = 256, ROWS = 8;

__global__ void __launch_bounds__(ROW_THREADS) fluidity_rows_kernel(const int32_t *__restrict__ shared, int32_t n,
                                                                    double *__restrict__ row_sums)
{
    __shared__ double part[ROWS][ROW_THREADS];
    const int32_t k0 = blockIdx.x * ROWS;
    int64_t mk[ROWS];
    double acc[ROWS];
#pragma unroll
    for (int i = 0; i < ROWS; ++i) {
        mk[i] = k0 + i < n ? shared[static_cast<int64_t>(k0 + i) * (n + 1)] : 0;
        acc[i] = 0.0;
    }
    for (int32_t l = threadIdx.x; l < n; l += ROW_THREADS) {
        const int64_t ml = shared[static_cast<int64_t>(l) * (n + 1)];
#pragma unroll
        for (int i = 0; i < ROWS; ++i) {
            const int32_t k = k0 + i;
            if (k >= n || k == l) continue;
            const int64_t s = shared[static_cast<int64_t>(k) * n + l];
            acc[i] += static_cast<double>(mk[i] + ml - 2 * s) / static_cast<double>(mk[i] + ml);
        }
    }
#pragma unroll
    for (int i = 0; i < ROWS; ++i) part[i][threadIdx.x] = acc[i];
    __syncthreads();
    for (int h = ROW_THREADS / 2; h > 0; h >>= 1) {
        if (threadIdx.x < h)
#pragma unroll
            for (int i = 0; i < ROWS; ++i) part[i][threadIdx.x] += part[i][threadIdx.x + h];
        __syncthreads();
    }
    if (threadIdx.x < ROWS && k0 + threadIdx.x < n) row_sums[k0 + threadIdx.x] = part[threadIdx.x][0];
}

// ---- pair overlap histograms and exact rarefaction moments ------------------------------------------------------
// (pgx_plan_spectrum, pgx_pair_overlap_histograms, pgx_rarefaction_moments; the decomposition is stated in
// include/pgx.h and restated in oracle/exact_np.py)
//
//   vectors  p1 = sum(w_present), a1 = sum(w_absent), nnz = sum(colsum) and the same-genome pair sums
//   rows     m, Wp = sum of w_present over the row's genomes, Wa likewise, for every list and bitmap row; counted
//            by m into rows_m / wp_m / wa_m
//   classes  the universal count u = (nnz - sum of row m - p1 - a1 (N - 1)) / N and the empty count; a plan for
//            which these are not whole and non-negative is refused
//   closed   every pair with a closed-form gene, from the counts above, into H_s / H_a
//   sort     the rows by m (counting sort), so that a GEMM tile knows the range its s and a can take
//   expand   a panel of sorted rows into E [P][N_pad] (0 / 1 bytes, gene-major, genomes padded to 128)
//   gemm     E E^T over panel pairs on the tensor cores with a histogram epilogue (gemm_tiles above)
//   moments  T_w[k] = sum_v w[v] rho(v, k) for the four weight vectors, rho a running product
struct ClassCounts {
    int64_t p1, a1, nnz, sum_m, n_full, n_empty, same_p, same_a, same_pa;
    int32_t valid, pad;
};

__device__ __forceinline__ void hist_add(unsigned long long *h, int64_t v, int64_t n, int64_t count)
{
    if (count != 0 && v >= 0 && v <= n) atomicAdd(h + v, static_cast<unsigned long long>(count));
}

// one warp per task (its rows share the list kind): m, Wp, Wa of every list row
__global__ void pair_list_rows_kernel(const int32_t *__restrict__ tasks, int32_t n_tasks,
                                      const uint16_t *__restrict__ sorted_idx, const int32_t *__restrict__ sorted_ptr,
                                      const int32_t *__restrict__ w_present, const int32_t *__restrict__ w_absent,
                                      int32_t n, const ClassCounts *__restrict__ cc, uint32_t *__restrict__ m_row,
                                      unsigned long long *__restrict__ rows_m, unsigned long long *__restrict__ wp_m,
                                      unsigned long long *__restrict__ wa_m)
{
    const int lane = threadIdx.x & 31;
    const int32_t warp = static_cast<int32_t>((blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5);
    const int32_t n_warps = static_cast<int32_t>((gridDim.x * static_cast<int64_t>(blockDim.x)) >> 5);
    for (int32_t t = warp; t < n_tasks; t += n_warps) {
        const int4 task = reinterpret_cast<const int4 *>(tasks)[t];
        const bool absent = (task.y >> 24) & 1;
        for (int32_t r = task.z; r < task.z + task.w; ++r) {
            const int32_t e0 = sorted_ptr[r], e1 = sorted_ptr[r + 1];
            int32_t sp = 0, sa = 0;
            for (int32_t e = e0 + lane; e < e1; e += 32) {
                const int32_t c = sorted_idx[e];
                sp += w_present[c];
                sa += w_absent[c];
            }
            sp = __reduce_add_sync(0xffffffffu, sp);
            sa = __reduce_add_sync(0xffffffffu, sa);
            if (lane == 0) {
                const int32_t m = absent ? n - (e1 - e0) : e1 - e0;
                const int64_t wp = absent && wp_m ? cc->p1 - sp : sp, wa = absent && wp_m ? cc->a1 - sa : sa;
                atomicAdd(rows_m + m, 1ull);
                if (m_row) m_row[r] = static_cast<uint32_t>(m) | (absent ? 0x80000000u : 0u);
                if (wp_m) {
                    atomicAdd(wp_m + m, static_cast<unsigned long long>(wp));
                    atomicAdd(wa_m + m, static_cast<unsigned long long>(wa));
                }
            }
        }
    }
}

// one block per 32 bitmap rows (one word of a superblock line): m, Wp, Wa by a masked sum over the genomes
__global__ void __launch_bounds__(256) pair_bitmap_rows_kernel(const uint32_t *__restrict__ bits, int32_t n,
                                                               int32_t slice_words, int32_t n_long, int32_t n_rows,
                                                               const int32_t *__restrict__ w_present,
                                                               const int32_t *__restrict__ w_absent,
                                                               uint32_t *__restrict__ m_row,
                                                               unsigned long long *__restrict__ rows_m,
                                                               unsigned long long *__restrict__ wp_m,
                                                               unsigned long long *__restrict__ wa_m)
{
    __shared__ int32_t part[3][32];
    const int32_t line = 32 * slice_words;
    const int32_t sb = blockIdx.x / line, w = blockIdx.x % line;
    if (threadIdx.x < 32) part[0][threadIdx.x] = part[1][threadIdx.x] = part[2][threadIdx.x] = 0;
    __syncthreads();
    int32_t cnt[32], sp[32], sa[32];
#pragma unroll
    for (int b = 0; b < 32; ++b) cnt[b] = sp[b] = sa[b] = 0;
    const bool sums = wp_m != nullptr;
    for (int32_t c = threadIdx.x; c < n; c += blockDim.x) {
        const uint32_t v = __ldg(&bits[(static_cast<int64_t>(sb) * n + c) * line + w]);
        const int32_t p = sums ? w_present[c] : 0, a = sums ? w_absent[c] : 0;
#pragma unroll
        for (int b = 0; b < 32; ++b) {
            const int32_t bit = (v >> b) & 1;
            cnt[b] += bit;
            sp[b] += bit * p;
            sa[b] += bit * a;
        }
    }
#pragma unroll
    for (int b = 0; b < 32; ++b) {
        const int32_t c = __reduce_add_sync(0xffffffffu, cnt[b]);
        const int32_t p = __reduce_add_sync(0xffffffffu, sp[b]);
        const int32_t a = __reduce_add_sync(0xffffffffu, sa[b]);
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&part[0][b], c);
            atomicAdd(&part[1][b], p);
            atomicAdd(&part[2][b], a);
        }
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        const int64_t k = static_cast<int64_t>(sb) * 1024 * slice_words + 32 * w + threadIdx.x;
        if (k < n_long) {
            const int32_t m = part[0][threadIdx.x];
            atomicAdd(rows_m + m, 1ull);
            if (m_row) m_row[n_rows + k] = static_cast<uint32_t>(m);
            if (sums) {
                atomicAdd(wp_m + m, static_cast<unsigned long long>(part[1][threadIdx.x]));
                atomicAdd(wa_m + m, static_cast<unsigned long long>(part[2][threadIdx.x]));
            }
        }
    }
}

// block-wide sums of Q int64 values per thread in a fixed order (blockDim.x = 1,024); the result in thread 0
template <int Q>
__device__ void block_sums(int64_t (&acc)[Q])
{
    __shared__ int64_t red[Q][32];
    for (int q = 0; q < Q; ++q) {
        for (int h = 16; h > 0; h >>= 1) acc[q] += __shfl_down_sync(0xffffffffu, acc[q], h);
        if ((threadIdx.x & 31) == 0) red[q][threadIdx.x >> 5] = acc[q];
    }
    __syncthreads();
    for (int q = 0; q < Q; ++q) {
        acc[q] = 0;
        for (int w = 0; w < 32; ++w) acc[q] += red[q][w];
    }
    __syncthreads();
}

// p1, a1, nnz and the same-genome pair sums of the per-genome vectors (one block of 1,024 threads)
__device__ void vector_sums(int32_t n, const int32_t *__restrict__ colsum, const int32_t *__restrict__ w_present,
                            const int32_t *__restrict__ w_absent, ClassCounts *cc)
{
    int64_t acc[6] = {0, 0, 0, 0, 0, 0};
    for (int32_t c = threadIdx.x; c < n; c += blockDim.x) {
        const int64_t p = w_present[c], a = w_absent[c];
        acc[0] += p;
        acc[1] += a;
        acc[2] += colsum[c];
        acc[3] += p * (p - 1) / 2;
        acc[4] += a * (a - 1) / 2;
        acc[5] += p * a;
    }
    block_sums(acc);
    if (threadIdx.x == 0) {
        cc->p1 = acc[0], cc->a1 = acc[1], cc->nnz = acc[2];
        cc->same_p = acc[3], cc->same_a = acc[4], cc->same_pa = acc[5];
    }
    __syncthreads();
}

// universal and empty counts from the rows' spectrum: nnz = sum of row m + N u + p1 + (N - 1) a1
__device__ void class_counts(int32_t n, int64_t n_genes, int64_t n_stored, const unsigned long long *__restrict__ rows_m,
                             ClassCounts *cc)
{
    int64_t acc[1] = {0};
    for (int32_t v = threadIdx.x; v <= n; v += blockDim.x) acc[0] += static_cast<int64_t>(rows_m[v]) * v;
    block_sums(acc);
    if (threadIdx.x == 0) {
        cc->sum_m = acc[0];
        const int64_t rest = cc->nnz - cc->sum_m - cc->p1 - cc->a1 * (n - 1);
        cc->n_full = rest / n;
        cc->n_empty = n_genes - cc->n_full - cc->p1 - cc->a1 - n_stored;
        cc->valid = rest >= 0 && rest % n == 0 && cc->n_empty >= 0;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(1024) pair_vectors_kernel(int32_t n, const int32_t *__restrict__ colsum,
                                                            const int32_t *__restrict__ w_present,
                                                            const int32_t *__restrict__ w_absent, ClassCounts *cc)
{
    vector_sums(n, colsum, w_present, w_absent, cc);
}

__global__ void __launch_bounds__(1024) pair_classes_kernel(int32_t n, int64_t n_genes, int64_t n_stored,
                                                            const unsigned long long *__restrict__ rows_m,
                                                            ClassCounts *cc)
{
    class_counts(n, n_genes, n_stored, rows_m, cc);
}

// the rows' spectrum (already in d_spectrum) + the closed-form classes; an inconsistent plan leaves -1 in bin 0
__global__ void __launch_bounds__(1024) spectrum_finish_kernel(int32_t n, int64_t n_genes, int64_t n_stored,
                                                               const int32_t *__restrict__ colsum,
                                                               const int32_t *__restrict__ w_present,
                                                               const int32_t *__restrict__ w_absent,
                                                               int64_t *spectrum)
{
    __shared__ ClassCounts cc;
    vector_sums(n, colsum, w_present, w_absent, &cc);
    class_counts(n, n_genes, n_stored, reinterpret_cast<const unsigned long long *>(spectrum), &cc);
    if (threadIdx.x == 0) {
        if (!cc.valid) {
            spectrum[0] = -1;
            return;
        }
        spectrum[0] += cc.n_empty;
        spectrum[n] += cc.n_full;
        if (n > 1) {
            spectrum[1] += cc.p1;
            spectrum[n - 1] += cc.a1;
        }
    }
}

// every pair with a closed-form gene (the table in include/pgx.h): thread v = the rows with m = v; thread 0 also the
// closed x closed pairs
__global__ void pair_closed_kernel(int32_t n, const ClassCounts *__restrict__ ccp,
                                   const unsigned long long *__restrict__ rows_m,
                                   const unsigned long long *__restrict__ wp_m,
                                   const unsigned long long *__restrict__ wa_m, unsigned long long *__restrict__ hs,
                                   unsigned long long *__restrict__ ha)
{
    const ClassCounts cc = *ccp;
    const int64_t e = cc.n_empty, u = cc.n_full, p1 = cc.p1, a1 = cc.a1;
    const int32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v == 0) {
        hist_add(hs, 0, n, e * (e - 1) / 2), hist_add(ha, n, n, e * (e - 1) / 2);
        hist_add(hs, 0, n, e * u), hist_add(ha, 0, n, e * u);
        hist_add(hs, 0, n, e * p1), hist_add(ha, n - 1, n, e * p1);
        hist_add(hs, 0, n, e * a1), hist_add(ha, 1, n, e * a1);
        hist_add(hs, n, n, u * (u - 1) / 2), hist_add(ha, 0, n, u * (u - 1) / 2);
        hist_add(hs, 1, n, u * p1), hist_add(ha, 0, n, u * p1);
        hist_add(hs, n - 1, n, u * a1), hist_add(ha, 0, n, u * a1);
        hist_add(hs, 1, n, cc.same_p), hist_add(ha, n - 1, n, cc.same_p);
        hist_add(hs, 0, n, p1 * (p1 - 1) / 2 - cc.same_p), hist_add(ha, n - 2, n, p1 * (p1 - 1) / 2 - cc.same_p);
        hist_add(hs, n - 1, n, cc.same_a), hist_add(ha, 1, n, cc.same_a);
        hist_add(hs, n - 2, n, a1 * (a1 - 1) / 2 - cc.same_a), hist_add(ha, 0, n, a1 * (a1 - 1) / 2 - cc.same_a);
        hist_add(hs, 0, n, cc.same_pa), hist_add(ha, 0, n, cc.same_pa);
        hist_add(hs, 1, n, p1 * a1 - cc.same_pa), hist_add(ha, 1, n, p1 * a1 - cc.same_pa);
    }
    if (v > n) return;
    const int64_t rows = static_cast<int64_t>(rows_m[v]);
    if (rows == 0) return;
    const int64_t wp = static_cast<int64_t>(wp_m[v]), wa = static_cast<int64_t>(wa_m[v]);
    hist_add(hs, 0, n, e * rows), hist_add(ha, n - v, n, e * rows);
    hist_add(hs, v, n, u * rows), hist_add(ha, 0, n, u * rows);
    hist_add(hs, 1, n, wp), hist_add(ha, n - v, n, wp);
    hist_add(hs, 0, n, p1 * rows - wp), hist_add(ha, n - 1 - v, n, p1 * rows - wp);
    hist_add(hs, v - 1, n, wa), hist_add(ha, 0, n, wa);
    hist_add(hs, v, n, a1 * rows - wa), hist_add(ha, 1, n, a1 * rows - wa);
}

// one block: cursor[v] = rows with m < v (exclusive scan of rows_m), in chunks of 1,024
__global__ void __launch_bounds__(1024) pair_scan_kernel(int32_t n, const unsigned long long *__restrict__ rows_m,
                                                         int32_t *__restrict__ cursor)
{
    __shared__ int32_t buf[1024];
    __shared__ int32_t carry;
    if (threadIdx.x == 0) carry = 0;
    for (int32_t base = 0; base <= n; base += 1024) {
        const int32_t v = base + threadIdx.x;
        const int32_t x = v <= n ? static_cast<int32_t>(rows_m[v]) : 0;
        buf[threadIdx.x] = x;
        __syncthreads();
        for (int h = 1; h < 1024; h <<= 1) {
            const int32_t y = threadIdx.x >= h ? buf[threadIdx.x - h] : 0;
            __syncthreads();
            buf[threadIdx.x] += y;
            __syncthreads();
        }
        if (v <= n) cursor[v] = carry + buf[threadIdx.x] - x;
        __syncthreads();
        if (threadIdx.x == 1023) carry += buf[1023];
        __syncthreads();
    }
}

// thread per row: its place in the m order (rows of equal m in any order: the histograms do not depend on it)
__global__ void pair_sort_kernel(int32_t n_stored, const uint32_t *__restrict__ m_row, int32_t *__restrict__ cursor,
                                 uint32_t *__restrict__ row_at, int32_t *__restrict__ m_sorted,
                                 int32_t *__restrict__ pos_of)
{
    const int32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_stored) return;
    const uint32_t v = m_row[r];
    const int32_t m = static_cast<int32_t>(v & 0x7fffffffu);
    const int32_t p = atomicAdd(cursor + m, 1);
    row_at[p] = static_cast<uint32_t>(r) | (v & 0x80000000u);
    m_sorted[p] = m;
    pos_of[r] = p;
}

// one warp per list row of the panel (sorted positions p0 .. p1 - 1): E row = the default byte, then the list's
// genomes flipped
__global__ void pair_expand_list_kernel(const uint32_t *__restrict__ row_at, int32_t p0, int32_t p1, int32_t n_rows,
                                        const uint16_t *__restrict__ sorted_idx,
                                        const int32_t *__restrict__ sorted_ptr, int32_t n, int32_t n_pad,
                                        uint8_t *__restrict__ e)
{
    const int lane = threadIdx.x & 31;
    const int32_t warp = static_cast<int32_t>((blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5);
    const int32_t n_warps = static_cast<int32_t>((gridDim.x * static_cast<int64_t>(blockDim.x)) >> 5);
    for (int32_t i = p0 + warp; i < p1; i += n_warps) {
        const uint32_t v = row_at[i];
        const int32_t r = static_cast<int32_t>(v & 0x7fffffffu);
        if (r >= n_rows) continue;
        const bool absent = v >> 31;
        uint8_t *row = e + static_cast<int64_t>(i - p0) * n_pad;
        for (int32_t q = lane; q < n_pad / 16; q += 32) {
            uint32_t fill[4] = {0u, 0u, 0u, 0u};                 // padding genomes (c >= N) stay 0
            if (absent)
                for (int b = 0; b < 16; ++b) fill[b >> 2] |= (16 * q + b < n ? 1u : 0u) << (8 * (b & 3));
            reinterpret_cast<uint4 *>(row)[q] = make_uint4(fill[0], fill[1], fill[2], fill[3]);
        }
        __syncwarp();
        for (int32_t x = sorted_ptr[r] + lane; x < sorted_ptr[r + 1]; x += 32) row[sorted_idx[x]] = absent ? 0 : 1;
    }
}

// one block per 32 bitmap rows: those in the panel -> E rows, 4 genomes (one uint32 of bytes) per thread and row
__global__ void __launch_bounds__(256) pair_expand_bitmap_kernel(const uint32_t *__restrict__ bits, int32_t n,
                                                                 int32_t slice_words, int32_t n_long, int32_t n_rows,
                                                                 const int32_t *__restrict__ pos_of, int32_t p0,
                                                                 int32_t p1, int32_t n_pad, uint8_t *__restrict__ e)
{
    __shared__ int32_t dst[32];
    const int32_t line = 32 * slice_words;
    const int32_t sb = blockIdx.x / line, w = blockIdx.x % line;
    bool mine = false;
    if (threadIdx.x < 32) {
        const int64_t k = static_cast<int64_t>(sb) * 1024 * slice_words + 32 * w + threadIdx.x;
        const int32_t p = k < n_long ? pos_of[n_rows + k] : -1;
        mine = p >= p0 && p < p1;
        dst[threadIdx.x] = mine ? p - p0 : -1;
    }
    if (!__syncthreads_or(mine)) return;
    for (int32_t q = threadIdx.x; q < n_pad / 4; q += blockDim.x) {
        uint32_t v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int32_t c = 4 * q + j;
            v[j] = c < n ? __ldg(&bits[(static_cast<int64_t>(sb) * n + c) * line + w]) : 0u;
        }
#pragma unroll 4
        for (int b = 0; b < 32; ++b) {
            const int32_t d = dst[b];
            if (d < 0) continue;
            const uint32_t out = ((v[0] >> b) & 1u) | ((v[1] >> b) & 1u) << 8 | ((v[2] >> b) & 1u) << 16 |
                                 ((v[3] >> b) & 1u) << 24;
            reinterpret_cast<uint32_t *>(e + static_cast<int64_t>(d) * n_pad)[q] = out;
        }
    }
}

// Histogram epilogue.  Buffer row i is sorted row base_lo + i below ``split`` and base_hi + i - split from it on.
// A diagonal panel (split = buffer rows) counts the pairs i < j, a panel pair (split = P) the pairs i < split <= j.
// Each tile's s and a lie in ranges known from the m of its first and last rows (rows sorted by m); when both fit
// the stage buffers as uint32 bins they are counted there (at most BM x BN pairs: no bin can overflow) and added
// into the global bins once, otherwise every pair goes straight to the global bins.
constexpr int32_t PAIR_BINS = (STAGES * STAGE_BYTES - BN * 4) / 4;

struct PairHistEpilogue {
    const int32_t *m_sorted;
    unsigned long long *hs, *ha;
    int32_t n_stored, n, base_lo, base_hi, split;
    bool cross;

    __device__ __forceinline__ int32_t sorted_row(int32_t i) const
    {
        return i < split ? base_lo + i : base_hi + (i - split);
    }

    __device__ __forceinline__ bool skip(int32_t rb, int32_t cb) const
    {
        if (cross && (rb * BM >= split || (cb + 1) * BN <= split)) return true;
        return sorted_row(rb * BM) >= n_stored || sorted_row(cb * BN) >= n_stored;
    }

    template <bool LOCAL>
    __device__ __forceinline__ void count(uint32_t tmem, int warp, int lane, int32_t m0, int32_t n0,
                                          const int32_t *col_m, uint32_t *bins, int32_t s_lo, int32_t sw,
                                          int32_t a_lo) const
    {
        const int32_t row = m0 + 32 * warp + lane;
        const int32_t gr = sorted_row(row);
        const bool row_ok = gr < n_stored;
        const int32_t base = n - (row_ok ? m_sorted[gr] : 0);
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
            uint32_t acc[32];
            tmem_ld_32(tmem + (static_cast<uint32_t>(32 * warp) << 16) + c, acc);
            if (!row_ok || (!cross && n0 + c + 31 <= row)) continue;
#pragma unroll
            for (int q = 0; q < 32; ++q) {
                const int32_t mc = col_m[c + q];
                if (mc < 0 || (!cross && n0 + c + q <= row)) continue;
                const int32_t s = static_cast<int32_t>(acc[q]), a = base - mc + s;
                if (LOCAL) {
                    atomicAdd(bins + (s - s_lo), 1u);
                    atomicAdd(bins + sw + (a - a_lo), 1u);
                } else {
                    atomicAdd(hs + s, 1ull);
                    atomicAdd(ha + a, 1ull);
                }
            }
        }
    }

    __device__ __forceinline__ void run(uint32_t tmem, int warp, int lane, int32_t m0, int32_t n0, int32_t,
                                        uint32_t stages) const
    {
        extern __shared__ uint8_t smem_raw[];
        int32_t *col_m = reinterpret_cast<int32_t *>(smem_raw + (stages - smem_u32(smem_raw)));
        uint32_t *bins = reinterpret_cast<uint32_t *>(col_m + BN);
        for (int j = threadIdx.x; j < BN; j += GEMM_THREADS) {
            const int32_t g = sorted_row(n0 + j);
            col_m[j] = g < n_stored ? m_sorted[g] : -1;
        }
        const int32_t r_lo = m_sorted[sorted_row(m0)], r_hi = m_sorted[min(sorted_row(m0 + BM - 1), n_stored - 1)];
        const int32_t c_lo = m_sorted[sorted_row(n0)], c_hi = m_sorted[min(sorted_row(n0 + BN - 1), n_stored - 1)];
        const int32_t s_lo = max(0, r_lo + c_lo - n), s_hi = min(r_hi, c_hi);
        const int32_t a_lo = max(0, n - r_hi - c_hi), a_hi = n - max(r_lo, c_lo);
        const int32_t sw = s_hi - s_lo + 1, width = sw + a_hi - a_lo + 1;
        const bool local = width <= PAIR_BINS;
        if (local)
            for (int32_t v = threadIdx.x; v < width; v += GEMM_THREADS) bins[v] = 0;
        __syncthreads();
        if (local) {
            count<true>(tmem, warp, lane, m0, n0, col_m, bins, s_lo, sw, a_lo);
            __syncthreads();
            for (int32_t v = threadIdx.x; v < width; v += GEMM_THREADS) {
                const uint32_t x = bins[v];
                if (x) atomicAdd(v < sw ? hs + s_lo + v : ha + a_lo + (v - sw), static_cast<unsigned long long>(x));
            }
        } else {
            count<false>(tmem, warp, lane, m0, n0, col_m, bins, s_lo, sw, a_lo);
        }
    }
};

__global__ void __launch_bounds__(GEMM_THREADS, 1) pair_hist_gemm_kernel(const __grid_constant__ CUtensorMap map,
                                                                          int32_t rows, int32_t k_blocks,
                                                                          PairHistEpilogue epi)
{
    gemm_tiles(map, rows, k_blocks, epi);
}

// Double-double arithmetic (a value is hi + lo, |lo| <= ulp(hi) / 2): the pan variance Z + 2 T_a - Z^2 cancels two
// terms of about Z^2 (4e10 at C4 for k = 1), so rho and the sums carry about 32 significant digits.
struct dd {
    double hi, lo;
};

__device__ __forceinline__ dd dd_norm(double s, double e)
{
    const double hi = s + e;
    return {hi, e - (hi - s)};
}

__device__ __forceinline__ dd dd_add(dd x, dd y)
{
    const double s = x.hi + y.hi, b = s - x.hi;
    const double e = (x.hi - (s - b)) + (y.hi - b) + x.lo + y.lo;
    return dd_norm(s, e);
}

__device__ __forceinline__ dd dd_mul(dd x, dd y)
{
    const double p = x.hi * y.hi;
    return dd_norm(p, fma(x.hi, y.hi, -p) + (x.hi * y.lo + x.lo * y.hi));
}

// (v - k) / v to double-double: the quotient and the exact remainder's quotient
__device__ __forceinline__ dd dd_ratio(int32_t v, int32_t k)
{
    const double num = v - k, den = v, q = num / den;
    return {q, fma(-q, den, num) / den};
}

__device__ __forceinline__ dd dd_shfl_up(dd x, int d)
{
    return {__shfl_up_sync(0xffffffffu, x.hi, d), __shfl_up_sync(0xffffffffu, x.lo, d)};
}

__device__ __forceinline__ dd dd_shfl_down(dd x, int d)
{
    return {__shfl_down_sync(0xffffffffu, x.hi, d), __shfl_down_sync(0xffffffffu, x.lo, d)};
}

// One warp per k: T_w[k] = sum over v = N .. k of w[v] rho(v, k), rho(N, k) = 1, rho(v - 1, k) = rho(v, k) (v - k) / v.
// Lane j takes the j-th run of ``c`` values of v from the top; a multiplicative scan of the runs' products gives each
// lane its starting rho; the lanes' sums are then added in a fixed tree, so two calls give the same bits.
constexpr int MOMENT_WARPS = 4;

__global__ void __launch_bounds__(32 * MOMENT_WARPS) rarefaction_moments_kernel(
    const int64_t *__restrict__ spectrum, const int64_t *__restrict__ hs, const int64_t *__restrict__ ha,
    int64_t n_genes, int32_t n, double *__restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const int32_t k = blockIdx.x * MOMENT_WARPS + (threadIdx.x >> 5) + 1;
    if (k > n) return;
    const int32_t len = n - k + 1, c = (len + 31) / 32;
    const int32_t top = n - lane * c, bottom = max(k, top - c + 1);        // this lane: v = top .. bottom
    dd run = {1.0, 0.0};
    for (int32_t v = top; v >= bottom && v > k; --v) run = dd_mul(run, dd_ratio(v, k));
    if (top < k) run = {1.0, 0.0};
    // exclusive product scan over the lanes: rho(top, k) = product of the runs above this lane
    dd rho = dd_shfl_up(run, 1);
    if (lane == 0) rho = {1.0, 0.0};
    for (int d = 1; d < 32; d <<= 1) {
        const dd other = dd_shfl_up(rho, d);
        if (lane >= d) rho = dd_mul(rho, other);
    }
    dd core = {0.0, 0.0}, none = {0.0, 0.0}, ts = {0.0, 0.0}, ta = {0.0, 0.0};
    for (int32_t v = top; v >= bottom && rho.hi != 0.0; --v) {
        core = dd_add(core, dd_mul(rho, dd{static_cast<double>(spectrum[v]), 0.0}));
        none = dd_add(none, dd_mul(rho, dd{static_cast<double>(spectrum[n - v]), 0.0}));
        if (hs) {
            ts = dd_add(ts, dd_mul(rho, dd{static_cast<double>(hs[v]), 0.0}));
            ta = dd_add(ta, dd_mul(rho, dd{static_cast<double>(ha[v]), 0.0}));
        }
        rho = dd_mul(rho, dd_ratio(v, k));
    }
    for (int d = 16; d > 0; d >>= 1) {
        core = dd_add(core, dd_shfl_down(core, d));
        none = dd_add(none, dd_shfl_down(none, d));
        ts = dd_add(ts, dd_shfl_down(ts, d));
        ta = dd_add(ta, dd_shfl_down(ta, d));
    }
    if (lane != 0) return;
    const int64_t nn = n;
    const dd g = {static_cast<double>(n_genes), 0.0};
    const dd pan = dd_add(g, dd{-none.hi, -none.lo});
    out[k - 1] = pan.hi + pan.lo;
    out[2 * nn + k - 1] = core.hi + core.lo;
    if (hs) {
        const dd two = {2.0, 0.0};
        const dd vp = dd_add(dd_add(none, dd_mul(two, ta)), dd_mul(dd{-none.hi, -none.lo}, none));
        const dd vc = dd_add(dd_add(core, dd_mul(two, ts)), dd_mul(dd{-core.hi, -core.lo}, core));
        out[nn + k - 1] = vp.hi + vp.lo;
        out[3 * nn + k - 1] = vc.hi + vc.lo;
    }
}

// ---- host -------------------------------------------------------------------------------------------------------
PFN_cuTensorMapEncodeTiled_v12000 tensor_map_encoder()
{
    static PFN_cuTensorMapEncodeTiled_v12000 fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &p, 12000, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
    }();
    return fn;
}

int launch_blocks(int64_t work, int threads)
{
    return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((work + threads - 1) / threads, 148 * 16)));
}

// ---- host: pair histograms ----------------------------------------------------------------------------------------
int64_t align256(int64_t x)
{
    return (x + 255) / 256 * 256;
}

int32_t padded_genomes(int32_t n)
{
    return (n + BK - 1) / BK * BK;
}

// workspace of pgx_pair_overlap_histograms: the fixed part, then the E panels
struct PairLayout {
    int64_t cc, m_row, rows_m, wp_m, wa_m, cursor, row_at, m_sorted, pos_of, e;

    PairLayout(int32_t n, int64_t rows)
    {
        cc = 0;
        m_row = align256(sizeof(ClassCounts));
        rows_m = m_row + align256(4 * rows);
        wp_m = rows_m + align256(8 * (int64_t(n) + 1));
        wa_m = wp_m + align256(8 * (int64_t(n) + 1));
        cursor = wa_m + align256(8 * (int64_t(n) + 1));
        row_at = cursor + align256(4 * (int64_t(n) + 1));
        m_sorted = row_at + align256(4 * rows);
        pos_of = m_sorted + align256(4 * rows);
        e = pos_of + align256(4 * rows);
    }
};

// E rows the workspace must hold: all stored rows (one panel), or at least two panels of 256 rows
int64_t pair_min_e_rows(int64_t rows)
{
    return std::min<int64_t>((rows + BM - 1) / BM * BM, 2 * BN);
}

int check_pair_plan(const char *who, const pgx_plan *plan)
{
    const int32_t n = plan->n_genomes;
    if (n < 1 || n > MAX_GENOMES) return pgx::fail(PGX_ERR_INVALID, "%s: n_genomes = %d outside 1 .. %d", who, n, MAX_GENOMES);
    if (plan->n_genes < 0) return pgx::fail(PGX_ERR_INVALID, "%s: negative n_genes", who);
    if (!plan->d_colsum || !plan->d_w_present || !plan->d_w_absent)
        return pgx::fail(PGX_ERR_INVALID, "%s: plan without its per-genome vectors", who);
    if (plan->n_rows < 0 || plan->n_tasks < 0 || plan->n_long < 0 || plan->n_superblocks < 0)
        return pgx::fail(PGX_ERR_INVALID, "%s: negative plan sizes", who);
    if (plan->n_rows > 0 && (!plan->d_tasks || !plan->d_sorted_idx || !plan->d_sorted_ptr))
        return pgx::fail(PGX_ERR_INVALID, "%s: plan without its list rows", who);
    if (plan->n_long > 0 && (!plan->d_bits || (plan->slice_words != 1 && plan->slice_words != 2 && plan->slice_words != 4) ||
                             int64_t(plan->n_superblocks) * 1024 * plan->slice_words < plan->n_long))
        return pgx::fail(PGX_ERR_INVALID, "%s: plan without a valid bitmap", who);
    return PGX_OK;
}

// m (and with wp_m, Wp and Wa) of every list and bitmap row, counted by m
int count_rows(const pgx_plan *plan, const ClassCounts *cc, uint32_t *m_row, unsigned long long *rows_m,
               unsigned long long *wp_m, unsigned long long *wa_m, cudaStream_t s)
{
    const int32_t n = plan->n_genomes;
    if (plan->n_tasks > 0) {
        pair_list_rows_kernel<<<launch_blocks(int64_t(plan->n_tasks) * 32, 256), 256, 0, s>>>(
            plan->d_tasks, plan->n_tasks, plan->d_sorted_idx, plan->d_sorted_ptr, plan->d_w_present, plan->d_w_absent,
            n, cc, m_row, rows_m, wp_m, wa_m);
        PGX_LAUNCH_CHECK("pair_list_rows_kernel");
    }
    if (plan->n_long > 0) {
        pair_bitmap_rows_kernel<<<plan->n_superblocks * 32 * plan->slice_words, 256, 0, s>>>(
            plan->d_bits, n, plan->slice_words, plan->n_long, plan->n_rows, plan->d_w_present, plan->d_w_absent, m_row,
            rows_m, wp_m, wa_m);
        PGX_LAUNCH_CHECK("pair_bitmap_rows_kernel");
    }
    return PGX_OK;
}

// sorted rows lo .. lo + rows - 1 -> E rows 0 .. rows - 1 at ``e``
int expand_panel(const pgx_plan *plan, const uint32_t *row_at, const int32_t *pos_of, int32_t lo, int32_t rows,
                 int32_t n_pad, uint8_t *e, cudaStream_t s)
{
    if (plan->n_rows > 0) {
        pair_expand_list_kernel<<<launch_blocks(int64_t(rows) * 32, 256), 256, 0, s>>>(
            row_at, lo, lo + rows, plan->n_rows, plan->d_sorted_idx, plan->d_sorted_ptr, plan->n_genomes, n_pad, e);
        PGX_LAUNCH_CHECK("pair_expand_list_kernel");
    }
    if (plan->n_long > 0) {
        pair_expand_bitmap_kernel<<<plan->n_superblocks * 32 * plan->slice_words, 256, 0, s>>>(
            plan->d_bits, plan->n_genomes, plan->slice_words, plan->n_long, plan->n_rows, pos_of, lo, lo + rows, n_pad, e);
        PGX_LAUNCH_CHECK("pair_expand_bitmap_kernel");
    }
    return PGX_OK;
}

// histogram GEMM over the first ``rows`` rows of E (tensor map over exactly those rows)
int pair_gemm(uint8_t *e, int32_t rows, int32_t n_pad, const PairHistEpilogue &epi, cudaStream_t s)
{
    CUtensorMap map;
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(n_pad), static_cast<cuuint64_t>(rows)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(n_pad)};
    const cuuint32_t box[2] = {BK, BM}, elem[2] = {1, 1};
    const CUresult rc = tensor_map_encoder()(&map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, e, dims, strides, box, elem,
                                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS)
        return pgx::fail(PGX_ERR_CUDA, "pgx_pair_overlap_histograms: cuTensorMapEncodeTiled failed (%d)", int(rc));
    const int32_t row_tiles = (rows + BM - 1) / BM, col_tiles = (rows + BN - 1) / BN;
    int64_t tiles = 0;
    for (int32_t g = 0; g * GROUP_ROWS < row_tiles; ++g) tiles += group_tiles(g, col_tiles);
    pair_hist_gemm_kernel<<<static_cast<unsigned>(tiles), GEMM_THREADS, GEMM_SMEM, s>>>(map, rows, n_pad / BK, epi);
    PGX_LAUNCH_CHECK("pair_hist_gemm_kernel");
    return PGX_OK;
}

}  // namespace

extern "C" {

int pgx_shared_genes(const pgx_plan *plan, int32_t *d_shared, void *d_work, int64_t work_bytes, void *stream)
{
    if (!plan || !d_shared || !d_work) return pgx::fail(PGX_ERR_INVALID, "pgx_shared_genes: null pointer");
    const int32_t n = plan->n_genomes;
    if (n < 1 || n > MAX_GENOMES)
        return pgx::fail(PGX_ERR_INVALID, "pgx_shared_genes: n_genomes = %d outside 1 .. %d", n, MAX_GENOMES);
    if ((reinterpret_cast<uintptr_t>(d_shared) & 15) != 0)
        return pgx::fail(PGX_ERR_INVALID, "pgx_shared_genes: d_shared must be 16-byte aligned");
    if ((reinterpret_cast<uintptr_t>(d_work) & 15) != 0)
        return pgx::fail(PGX_ERR_INVALID, "pgx_shared_genes: d_work must be 16-byte aligned");
    if (work_bytes < static_cast<int64_t>(n) * 128)
        return pgx::fail(PGX_ERR_INVALID, "pgx_shared_genes: work_bytes = %lld below N x 128 = %lld",
                         static_cast<long long>(work_bytes), static_cast<long long>(n) * 128);
    if (!plan->d_colsum || !plan->d_w_present || !plan->d_w_absent)
        return pgx::fail(PGX_ERR_INVALID, "pgx_shared_genes: plan without its per-genome vectors");
    if (plan->n_rows < 0 || plan->n_tasks < 0 || plan->n_long < 0 || plan->n_superblocks < 0)
        return pgx::fail(PGX_ERR_INVALID, "pgx_shared_genes: negative plan sizes");
    if (plan->n_rows > 0 && (!plan->d_tasks || !plan->d_sorted_idx || !plan->d_sorted_ptr))
        return pgx::fail(PGX_ERR_INVALID, "pgx_shared_genes: plan without its list rows");
    if (plan->n_long > 0 && (!plan->d_bits || (plan->slice_words != 1 && plan->slice_words != 2 && plan->slice_words != 4)))
        return pgx::fail(PGX_ERR_INVALID, "pgx_shared_genes: plan without a valid bitmap");
    const int64_t k_total = plan->n_long > 0 ? int64_t(plan->n_superblocks) * 1024 * plan->slice_words : 0;
    if (k_total > 0 && !tensor_map_encoder())
        return pgx::fail(PGX_ERR_CUDA, "pgx_shared_genes: the driver does not provide cuTensorMapEncodeTiled");
    cudaStream_t s = static_cast<cudaStream_t>(stream);

    // count: u, p and the scalars live at the front of the workspace until the init kernel has used them
    CountHeader *hdr = static_cast<CountHeader *>(d_work);
    int32_t *u = reinterpret_cast<int32_t *>(hdr + 1), *p = u + n;
    PGX_CUDA(cudaMemsetAsync(d_work, 0, sizeof(CountHeader) + sizeof(int32_t) * 2 * size_t(n), s));
    if (plan->n_tasks > 0) {
        shared_count_kernel<<<launch_blocks(int64_t(plan->n_tasks) * 32, 256), 256, 0, s>>>(
            plan->d_tasks, plan->n_tasks, plan->d_sorted_idx, plan->d_sorted_ptr, u, p, hdr);
        PGX_LAUNCH_CHECK("shared_count_kernel");
    }
    shared_count_vectors_kernel<<<1, 1024, 0, s>>>(plan->d_w_absent, n, plan->d_bits, plan->n_long > 0 ? plan->n_superblocks : 0,
                                                   plan->slice_words, hdr);
    PGX_LAUNCH_CHECK("shared_count_vectors_kernel");
    shared_full_kernel<<<1, 1, 0, s>>>(plan->d_colsum, plan->d_w_present, plan->d_w_absent, u, p, hdr);
    PGX_LAUNCH_CHECK("shared_full_kernel");
    // a plan whose vectors and rows do not add up to its column sums would give a wrong S: refuse it before the
    // heavy phases (the only point at which the call waits for the device)
    int32_t n_full = 0;
    PGX_CUDA(cudaMemcpyAsync(&n_full, &hdr->n_full, sizeof(n_full), cudaMemcpyDeviceToHost, s));
    PGX_CUDA(cudaStreamSynchronize(s));
    if (n_full < 0)
        return pgx::fail(PGX_ERR_INVALID, "pgx_shared_genes: inconsistent plan (universal-gene count %d < 0)", n_full);

    shared_init_kernel<<<n, 256, 0, s>>>(n, plan->d_colsum, plan->d_w_absent, u, hdr, d_shared);
    PGX_LAUNCH_CHECK("shared_init_kernel");
    if (plan->n_rows > 0) {
        shared_pairs_kernel<<<launch_blocks(int64_t(plan->n_rows) * 32, 256), 256, 0, s>>>(
            plan->n_rows, plan->d_sorted_idx, plan->d_sorted_ptr, n, d_shared);
        PGX_LAUNCH_CHECK("shared_pairs_kernel");
    }

    if (k_total > 0) {
        // slab width: as many bitmap rows as the workspace holds per genome, a multiple of 128
        const int64_t k_slab = std::min<int64_t>(k_total, work_bytes / n / BK * BK);
        uint8_t *e = static_cast<uint8_t *>(d_work);
        PGX_CUDA(cudaFuncSetAttribute(shared_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM));
        const int32_t row_tiles = (n + BM - 1) / BM, col_tiles = (n + BN - 1) / BN;
        int64_t tiles = 0;
        for (int32_t g = 0; g * GROUP_ROWS < row_tiles; ++g) tiles += group_tiles(g, col_tiles);
        const dim3 grid(static_cast<unsigned>(tiles));
        for (int64_t k0 = 0; k0 < k_total; k0 += k_slab) {
            const int64_t k_cur = std::min<int64_t>(k_slab, k_total - k0);
            shared_expand_kernel<<<launch_blocks((k_cur >> 5) * n, 256), 256, 0, s>>>(
                plan->d_bits, n, plan->slice_words, k0, k_cur, k_slab, e);
            PGX_LAUNCH_CHECK("shared_expand_kernel");
            CUtensorMap map;
            const cuuint64_t dims[2] = {static_cast<cuuint64_t>(k_cur), static_cast<cuuint64_t>(n)};
            const cuuint64_t strides[1] = {static_cast<cuuint64_t>(k_slab)};
            const cuuint32_t box[2] = {BK, BM}, elem[2] = {1, 1};
            const CUresult rc = tensor_map_encoder()(&map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, e, dims, strides, box, elem,
                                                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (rc != CUDA_SUCCESS) return pgx::fail(PGX_ERR_CUDA, "pgx_shared_genes: cuTensorMapEncodeTiled failed (%d)", int(rc));
            shared_gemm_kernel<<<grid, GEMM_THREADS, GEMM_SMEM, s>>>(map, n, static_cast<int32_t>(k_cur / BK), d_shared);
            PGX_LAUNCH_CHECK("shared_gemm_kernel");
        }
    }

    const int32_t tiles = (n + 31) / 32;
    shared_mirror_kernel<<<dim3(tiles, tiles), dim3(32, 8), 0, s>>>(n, d_shared);
    PGX_LAUNCH_CHECK("shared_mirror_kernel");
    return PGX_OK;
}

int pgx_fluidity_rows(const int32_t *d_shared, int32_t n_genomes, double *d_row_sums, void *stream)
{
    if (!d_shared || !d_row_sums) return pgx::fail(PGX_ERR_INVALID, "pgx_fluidity_rows: null pointer");
    if (n_genomes < 1 || n_genomes > MAX_GENOMES)
        return pgx::fail(PGX_ERR_INVALID, "pgx_fluidity_rows: n_genomes = %d outside 1 .. %d", n_genomes, MAX_GENOMES);
    if ((reinterpret_cast<uintptr_t>(d_shared) & 3) != 0 || (reinterpret_cast<uintptr_t>(d_row_sums) & 7) != 0)
        return pgx::fail(PGX_ERR_INVALID, "pgx_fluidity_rows: d_shared must be 4-byte and d_row_sums 8-byte aligned");
    fluidity_rows_kernel<<<(n_genomes + ROWS - 1) / ROWS, ROW_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
        d_shared, n_genomes, d_row_sums);
    PGX_LAUNCH_CHECK("fluidity_rows_kernel");
    return PGX_OK;
}

int64_t pgx_pair_overlap_work_bytes(int32_t n_genomes, int64_t n_stored_rows, int32_t one_panel)
{
    if (n_genomes < 1 || n_genomes > MAX_GENOMES || n_stored_rows < 0 || n_stored_rows > INT32_MAX - 2 * BN) return 0;
    const int64_t e_rows = one_panel ? (n_stored_rows + BM - 1) / BM * BM : pair_min_e_rows(n_stored_rows);
    return PairLayout(n_genomes, n_stored_rows).e + e_rows * padded_genomes(n_genomes);
}

int pgx_plan_spectrum(const pgx_plan *plan, int64_t *d_spectrum, void *stream)
{
    if (!plan || !d_spectrum) return pgx::fail(PGX_ERR_INVALID, "pgx_plan_spectrum: null pointer");
    if ((reinterpret_cast<uintptr_t>(d_spectrum) & 7) != 0)
        return pgx::fail(PGX_ERR_INVALID, "pgx_plan_spectrum: d_spectrum must be 8-byte aligned");
    if (const int rc = check_pair_plan("pgx_plan_spectrum", plan)) return rc;
    const int32_t n = plan->n_genomes;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PGX_CUDA(cudaMemsetAsync(d_spectrum, 0, sizeof(int64_t) * (size_t(n) + 1), s));
    if (const int rc = count_rows(plan, nullptr, nullptr, reinterpret_cast<unsigned long long *>(d_spectrum), nullptr,
                                  nullptr, s))
        return rc;
    spectrum_finish_kernel<<<1, 1024, 0, s>>>(n, plan->n_genes, int64_t(plan->n_rows) + plan->n_long, plan->d_colsum,
                                             plan->d_w_present, plan->d_w_absent, d_spectrum);
    PGX_LAUNCH_CHECK("spectrum_finish_kernel");
    int64_t empty = 0;
    PGX_CUDA(cudaMemcpyAsync(&empty, d_spectrum, sizeof(empty), cudaMemcpyDeviceToHost, s));
    PGX_CUDA(cudaStreamSynchronize(s));
    if (empty < 0)
        return pgx::fail(PGX_ERR_INVALID, "pgx_plan_spectrum: inconsistent plan (rows and vectors do not add up to the "
                                          "column sums in whole universal and empty genes)");
    return PGX_OK;
}

int pgx_pair_overlap_histograms(const pgx_plan *plan, int64_t *d_hist_shared, int64_t *d_hist_absent, void *d_work,
                                int64_t work_bytes, void *stream)
{
    if (!plan || !d_hist_shared || !d_hist_absent || !d_work)
        return pgx::fail(PGX_ERR_INVALID, "pgx_pair_overlap_histograms: null pointer");
    if ((reinterpret_cast<uintptr_t>(d_hist_shared) & 7) != 0 || (reinterpret_cast<uintptr_t>(d_hist_absent) & 7) != 0 ||
        (reinterpret_cast<uintptr_t>(d_work) & 255) != 0)
        return pgx::fail(PGX_ERR_INVALID, "pgx_pair_overlap_histograms: the histograms must be 8-byte and d_work "
                                          "256-byte aligned");
    if (const int rc = check_pair_plan("pgx_pair_overlap_histograms", plan)) return rc;
    const int32_t n = plan->n_genomes, n_pad = padded_genomes(n);
    const int64_t stored = int64_t(plan->n_rows) + plan->n_long;
    const int64_t need = pgx_pair_overlap_work_bytes(n, stored, 0);
    if (need == 0) return pgx::fail(PGX_ERR_INVALID, "pgx_pair_overlap_histograms: %lld stored rows", (long long)stored);
    if (work_bytes < need)
        return pgx::fail(PGX_ERR_INVALID, "pgx_pair_overlap_histograms: work_bytes = %lld below the minimum %lld",
                         static_cast<long long>(work_bytes), static_cast<long long>(need));
    if (stored > 1 && !tensor_map_encoder())
        return pgx::fail(PGX_ERR_CUDA, "pgx_pair_overlap_histograms: the driver does not provide cuTensorMapEncodeTiled");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const PairLayout L(n, stored);
    uint8_t *w = static_cast<uint8_t *>(d_work);
    ClassCounts *cc = reinterpret_cast<ClassCounts *>(w + L.cc);
    uint32_t *m_row = reinterpret_cast<uint32_t *>(w + L.m_row);
    auto *rows_m = reinterpret_cast<unsigned long long *>(w + L.rows_m);
    auto *wp_m = reinterpret_cast<unsigned long long *>(w + L.wp_m);
    auto *wa_m = reinterpret_cast<unsigned long long *>(w + L.wa_m);
    int32_t *cursor = reinterpret_cast<int32_t *>(w + L.cursor);
    uint32_t *row_at = reinterpret_cast<uint32_t *>(w + L.row_at);
    int32_t *m_sorted = reinterpret_cast<int32_t *>(w + L.m_sorted);
    int32_t *pos_of = reinterpret_cast<int32_t *>(w + L.pos_of);
    uint8_t *e = w + L.e;
    auto *hs = reinterpret_cast<unsigned long long *>(d_hist_shared);
    auto *ha = reinterpret_cast<unsigned long long *>(d_hist_absent);

    PGX_CUDA(cudaMemsetAsync(w, 0, L.m_row, s));
    PGX_CUDA(cudaMemsetAsync(w + L.rows_m, 0, L.cursor - L.rows_m, s));
    PGX_CUDA(cudaMemsetAsync(hs, 0, sizeof(int64_t) * (size_t(n) + 1), s));
    PGX_CUDA(cudaMemsetAsync(ha, 0, sizeof(int64_t) * (size_t(n) + 1), s));
    pair_vectors_kernel<<<1, 1024, 0, s>>>(n, plan->d_colsum, plan->d_w_present, plan->d_w_absent, cc);
    PGX_LAUNCH_CHECK("pair_vectors_kernel");
    if (const int rc = count_rows(plan, cc, m_row, rows_m, wp_m, wa_m, s)) return rc;
    pair_classes_kernel<<<1, 1024, 0, s>>>(n, plan->n_genes, stored, rows_m, cc);
    PGX_LAUNCH_CHECK("pair_classes_kernel");
    // a plan whose rows and vectors do not add up to its column sums would give wrong histograms: refuse it before
    // the heavy phases (the only point at which the call waits for the device)
    ClassCounts host{};
    PGX_CUDA(cudaMemcpyAsync(&host, cc, sizeof(host), cudaMemcpyDeviceToHost, s));
    PGX_CUDA(cudaStreamSynchronize(s));
    if (!host.valid)
        return pgx::fail(PGX_ERR_INVALID, "pgx_pair_overlap_histograms: inconsistent plan (rows and vectors do not add "
                                          "up to the column sums in whole universal and empty genes)");
    pair_closed_kernel<<<(n + 1 + 255) / 256, 256, 0, s>>>(n, cc, rows_m, wp_m, wa_m, hs, ha);
    PGX_LAUNCH_CHECK("pair_closed_kernel");
    if (stored < 2) return PGX_OK;

    pair_scan_kernel<<<1, 1024, 0, s>>>(n, rows_m, cursor);
    PGX_LAUNCH_CHECK("pair_scan_kernel");
    pair_sort_kernel<<<static_cast<unsigned>((stored + 255) / 256), 256, 0, s>>>(static_cast<int32_t>(stored), m_row,
                                                                                 cursor, row_at, m_sorted, pos_of);
    PGX_LAUNCH_CHECK("pair_sort_kernel");

    // one panel when every stored row fits, else panels of P rows (a multiple of BN), two at a time
    const int64_t e_rows = (work_bytes - L.e) / n_pad;
    const int32_t panel = e_rows >= (stored + BM - 1) / BM * BM ? static_cast<int32_t>(stored)
                                                                 : static_cast<int32_t>(e_rows / 2 / BN * BN);
    PGX_CUDA(cudaFuncSetAttribute(pair_hist_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM));
    PairHistEpilogue epi{m_sorted, hs, ha, static_cast<int32_t>(stored), n, 0, 0, 0, false};
    for (int32_t lo_i = 0; lo_i < stored; lo_i += panel) {
        const int32_t rows_i = static_cast<int32_t>(std::min<int64_t>(panel, stored - lo_i));
        if (const int rc = expand_panel(plan, row_at, pos_of, lo_i, rows_i, n_pad, e, s)) return rc;
        epi.base_lo = lo_i, epi.base_hi = static_cast<int32_t>(stored), epi.split = rows_i, epi.cross = false;
        if (const int rc = pair_gemm(e, rows_i, n_pad, epi, s)) return rc;
        for (int32_t lo_j = lo_i + panel; lo_j < stored; lo_j += panel) {
            const int32_t rows_j = static_cast<int32_t>(std::min<int64_t>(panel, stored - lo_j));
            if (const int rc = expand_panel(plan, row_at, pos_of, lo_j, rows_j, n_pad, e + int64_t(panel) * n_pad, s))
                return rc;
            epi.base_hi = lo_j, epi.split = panel, epi.cross = true;
            if (const int rc = pair_gemm(e, panel + rows_j, n_pad, epi, s)) return rc;
        }
    }
    return PGX_OK;
}

int pgx_rarefaction_moments(const int64_t *d_spectrum, const int64_t *d_hist_shared, const int64_t *d_hist_absent,
                            int64_t n_genes, int32_t n_genomes, double *d_out, void *stream)
{
    if (!d_spectrum || !d_out) return pgx::fail(PGX_ERR_INVALID, "pgx_rarefaction_moments: null pointer");
    if (!d_hist_shared != !d_hist_absent)
        return pgx::fail(PGX_ERR_INVALID, "pgx_rarefaction_moments: pass both histograms or neither");
    if (n_genomes < 1 || n_genomes > MAX_GENOMES)
        return pgx::fail(PGX_ERR_INVALID, "pgx_rarefaction_moments: n_genomes = %d outside 1 .. %d", n_genomes,
                         MAX_GENOMES);
    if (n_genes < 0) return pgx::fail(PGX_ERR_INVALID, "pgx_rarefaction_moments: negative n_genes");
    if (((reinterpret_cast<uintptr_t>(d_spectrum) | reinterpret_cast<uintptr_t>(d_hist_shared) |
          reinterpret_cast<uintptr_t>(d_hist_absent) | reinterpret_cast<uintptr_t>(d_out)) & 7) != 0)
        return pgx::fail(PGX_ERR_INVALID, "pgx_rarefaction_moments: every pointer must be 8-byte aligned");
    rarefaction_moments_kernel<<<(n_genomes + MOMENT_WARPS - 1) / MOMENT_WARPS, 32 * MOMENT_WARPS, 0,
                                 static_cast<cudaStream_t>(stream)>>>(
        d_spectrum, d_hist_shared, d_hist_absent, n_genes, n_genomes, d_out);
    PGX_LAUNCH_CHECK("rarefaction_moments_kernel");
    return PGX_OK;
}

}  // extern "C"
