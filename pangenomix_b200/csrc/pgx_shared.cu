// Genome x genome shared-gene matrix S = X^T X of a planned table (pgx_shared_genes) and the per-genome sums of
// genomic-fluidity distances (pgx_fluidity_rows).  The decomposition of S over the plan's gene classes is stated in
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

// one CTA per tile of the order above; a tile without an entry above the diagonal (cb < rb / 2) returns at once
__global__ void __launch_bounds__(GEMM_THREADS, 1) shared_gemm_kernel(const __grid_constant__ CUtensorMap map,
                                                                       int32_t n, int32_t k_blocks,
                                                                       int32_t *__restrict__ shared)
{
    const int32_t row_tiles = (n + BM - 1) / BM, col_tiles = (n + BN - 1) / BN;
    int64_t id = blockIdx.x;
    int32_t g = 0;
    while (id >= group_tiles(g, col_tiles)) id -= group_tiles(g++, col_tiles);
    const int32_t cb = g * (GROUP_ROWS / 2) + static_cast<int32_t>(id / GROUP_ROWS);
    const int32_t rb = g * GROUP_ROWS + static_cast<int32_t>(id % GROUP_ROWS);
    if (rb >= row_tiles || cb < rb / 2) return;
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

    // epilogue: warp w owns TMEM lanes 32 w .. 32 w + 31 = tile rows; thread = one row, 32 columns per load
    mbar_wait(smem_u32(&done_bar), 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
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
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
    }
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

}  // extern "C"
