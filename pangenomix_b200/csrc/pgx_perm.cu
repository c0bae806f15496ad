// Seeded on-device genome orders (pgx_random_perms) and exact column moments of curve blocks
// (pgx_curve_moments).  The permutation recipe is specified in include/pgx.h; oracle/perm_np.py restates it.
#include "pgx_common.cuh"

#include <limits.h>

namespace {

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) {
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
        const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    }
    return c;
}

__device__ __forceinline__ uint32_t word_of(const uint4 &w, uint32_t k)
{
    return k == 0 ? w.x : k == 1 ? w.y : k == 2 ? w.z : w.w;
}

constexpr uint32_t FY_DOMAIN = 0x80000000u;

// One CTA per permutation; the row (uint16[N]) and the bucket counters (int32[B]) live in shared memory.
// Thread t owns the contiguous bucket range [t * seg, (t + 1) * seg) for the scan, the sort and the shuffle.
__global__ void __launch_bounds__(1024) random_perms_kernel(uint32_t k0, uint32_t k1, int64_t first, int32_t n,
                                                            int32_t bucket_bits, uint16_t *__restrict__ out)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int32_t n_buckets = 1 << bucket_bits;
    int32_t *cnt = reinterpret_cast<int32_t *>(smem);
    uint16_t *row = reinterpret_cast<uint16_t *>(smem + sizeof(int32_t) * n_buckets);
    __shared__ int32_t warp_total[32];

    const uint64_t perm = static_cast<uint64_t>(first) + blockIdx.x;
    const uint32_t lo = static_cast<uint32_t>(perm), hi = static_cast<uint32_t>(perm >> 32);
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const int32_t n_groups = (n + 3) >> 2;
    const int shift = 32 - bucket_bits;                    // bucket_bits == 0: every genome is in bucket 0

    for (int32_t k = tid; k < n_buckets; k += nthreads) cnt[k] = 0;
    __syncthreads();
    for (int32_t g = tid; g < n_groups; g += nthreads) {
        const uint4 w = philox4x32_10(make_uint4(static_cast<uint32_t>(g), lo, hi, 0u), k0, k1);
        for (int j = 0; j < 4 && 4 * g + j < n; ++j)
            atomicAdd(&cnt[bucket_bits ? word_of(w, j) >> shift : 0u], 1);
    }
    __syncthreads();

    // exclusive scan of the counters: serial over the thread's segment, then across threads
    const int32_t seg = (n_buckets + nthreads - 1) / nthreads;
    const int32_t b0 = min(n_buckets, tid * seg), b1 = min(n_buckets, b0 + seg);
    int32_t local = 0;
    for (int32_t k = b0; k < b1; ++k) local += cnt[k];
    const int lane = tid & 31, warp = tid >> 5;
    int32_t incl = local;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int32_t v = __shfl_up_sync(pgx::FULL_MASK, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) warp_total[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const int n_warps = nthreads >> 5;
        int32_t v = lane < n_warps ? warp_total[lane] : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int32_t u = __shfl_up_sync(pgx::FULL_MASK, v, d);
            if (lane >= d) v += u;
        }
        if (lane < n_warps) warp_total[lane] = v;           // inclusive over warps
    }
    __syncthreads();
    const int32_t seg_base = incl - local + (warp ? warp_total[warp - 1] : 0);
    {
        int32_t run = seg_base;
        for (int32_t k = b0; k < b1; ++k) {
            const int32_t c = cnt[k];
            cnt[k] = run;                                      // cursor = start of bucket k
            run += c;
        }
    }
    __syncthreads();

    // scatter (order inside a bucket depends on the atomics; the sort below removes that)
    for (int32_t g = tid; g < n_groups; g += nthreads) {
        const uint4 w = philox4x32_10(make_uint4(static_cast<uint32_t>(g), lo, hi, 0u), k0, k1);
        for (int j = 0; j < 4 && 4 * g + j < n; ++j) {
            const int32_t pos = atomicAdd(&cnt[bucket_bits ? word_of(w, j) >> shift : 0u], 1);
            row[pos] = static_cast<uint16_t>(4 * g + j);
        }
    }
    __syncthreads();

    // every bucket: ascending genome order, then Fisher-Yates from the top with masked-rejection draws
    int32_t start = seg_base;
    for (int32_t k = b0; k < b1; ++k) {
        const int32_t end = cnt[k];                            // cursors now hold the bucket ends
        uint16_t *a = row + start;
        const int32_t m = end - start;
        for (int32_t x = 1; x < m; ++x) {
            const uint16_t v = a[x];
            int32_t y = x - 1;
            while (y >= 0 && a[y] > v) {
                a[y + 1] = a[y];
                --y;
            }
            a[y + 1] = v;
        }
        uint32_t t = 0;
        uint4 w = make_uint4(0, 0, 0, 0);
        for (int32_t j = m - 1; j >= 1; --j) {
            uint32_t mask = static_cast<uint32_t>(j);
            mask |= mask >> 1;
            mask |= mask >> 2;
            mask |= mask >> 4;
            mask |= mask >> 8;
            mask |= mask >> 16;
            uint32_t v;
            do {
                if ((t & 3) == 0)
                    w = philox4x32_10(make_uint4(static_cast<uint32_t>(k), lo, hi, FY_DOMAIN | (t >> 2)), k0, k1);
                v = word_of(w, t & 3) & mask;
                ++t;
            } while (v > static_cast<uint32_t>(j));
            const uint16_t tmp = a[j];
            a[j] = a[v];
            a[v] = tmp;
        }
        start = end;
    }
    __syncthreads();

    // row out: scalar head up to a 16-byte boundary of the output, 16-byte stores, scalar tail
    uint16_t *dst = out + static_cast<int64_t>(blockIdx.x) * n;
    const int32_t head = min(n, static_cast<int32_t>(((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15) >> 1));
    const int32_t n_vec = (n - head) >> 3;
    if (tid < head) dst[tid] = row[tid];
    for (int32_t v = tid; v < n_vec; v += nthreads) {
        const uint16_t *s = row + head + 8 * v;
        uint4 pack;
        pack.x = s[0] | (static_cast<uint32_t>(s[1]) << 16);
        pack.y = s[2] | (static_cast<uint32_t>(s[3]) << 16);
        pack.z = s[4] | (static_cast<uint32_t>(s[5]) << 16);
        pack.w = s[6] | (static_cast<uint32_t>(s[7]) << 16);
        reinterpret_cast<uint4 *>(dst + head)[v] = pack;
    }
    for (int32_t e = head + 8 * n_vec + tid; e < n; e += nthreads) dst[e] = row[e];
}

__global__ void moments_init_kernel(int64_t width, int64_t *sum, uint64_t *sumsq, int32_t *mn, int32_t *mx)
{
    for (int64_t c = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; c < width;
         c += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        sum[c] = 0;
        sumsq[c] = 0;
        mn[c] = INT_MAX;
        mx[c] = INT_MIN;
    }
}

// blockIdx.x: a run of 2 * blockDim.x columns (two per thread, one 8-byte load per row); blockIdx.y: a slice of rows.
constexpr int MOMENT_THREADS = 256;

__global__ void __launch_bounds__(MOMENT_THREADS) curve_moments_kernel(
    const int32_t *__restrict__ curves, int64_t n_rows, int64_t width, int64_t rows_per_slice,
    int64_t *sum, uint64_t *sumsq, int32_t *mn, int32_t *mx)
{
    const int64_t col = 2 * (blockIdx.x * static_cast<int64_t>(MOMENT_THREADS) + threadIdx.x);
    if (col >= width) return;
    const int64_t r0 = blockIdx.y * rows_per_slice;
    const int64_t r1 = min(n_rows, r0 + rows_per_slice);
    if (r0 >= r1) return;
    int64_t s0 = 0, s1 = 0;
    uint64_t q0 = 0, q1 = 0;
    int32_t lo0 = INT_MAX, lo1 = INT_MAX, hi0 = INT_MIN, hi1 = INT_MIN;
    const int32_t *p = curves + r0 * width + col;
    for (int64_t r = r0; r < r1; ++r, p += width) {
        const int2 v = __ldcs(reinterpret_cast<const int2 *>(p));
        s0 += v.x;
        s1 += v.y;
        q0 += static_cast<uint64_t>(static_cast<int64_t>(v.x) * v.x);
        q1 += static_cast<uint64_t>(static_cast<int64_t>(v.y) * v.y);
        lo0 = min(lo0, v.x);
        lo1 = min(lo1, v.y);
        hi0 = max(hi0, v.x);
        hi1 = max(hi1, v.y);
    }
    atomicAdd(reinterpret_cast<unsigned long long *>(sum + col), static_cast<unsigned long long>(s0));
    atomicAdd(reinterpret_cast<unsigned long long *>(sum + col + 1), static_cast<unsigned long long>(s1));
    atomicAdd(reinterpret_cast<unsigned long long *>(sumsq + col), static_cast<unsigned long long>(q0));
    atomicAdd(reinterpret_cast<unsigned long long *>(sumsq + col + 1), static_cast<unsigned long long>(q1));
    atomicMin(mn + col, lo0);
    atomicMin(mn + col + 1, lo1);
    atomicMax(mx + col, hi0);
    atomicMax(mx + col + 1, hi1);
}

}  // namespace

extern "C" {

int pgx_random_perms(uint64_t seed, int64_t first, int64_t n_perm, int32_t n_genomes, uint16_t *d_perms, void *stream)
{
    if (!d_perms) return pgx::fail(PGX_ERR_INVALID, "pgx_random_perms: d_perms is null");
    if (n_genomes < 1 || n_genomes > 65503)
        return pgx::fail(PGX_ERR_INVALID, "pgx_random_perms: n_genomes = %d outside 1 .. 65503", n_genomes);
    if (n_perm < 0) return pgx::fail(PGX_ERR_INVALID, "pgx_random_perms: n_perm < 0");
    if (first < 0) return pgx::fail(PGX_ERR_INVALID, "pgx_random_perms: first < 0");
    if (n_perm > INT_MAX) return pgx::fail(PGX_ERR_INVALID, "pgx_random_perms: n_perm > 2^31 - 1 per call");
    if (n_perm == 0) return PGX_OK;
    if ((reinterpret_cast<uintptr_t>(d_perms) & 1) != 0)
        return pgx::fail(PGX_ERR_INVALID, "pgx_random_perms: d_perms must be 2-byte aligned");
    const int32_t half = (n_genomes + 1) / 2;
    int32_t bits = 0;
    while ((2 << bits) <= half) ++bits;                      // B = 2^bits = largest power of two <= ceil(N / 2)
    const int threads = n_genomes > 16384 ? 1024 : n_genomes > 2048 ? 512 : 256;
    const size_t smem = sizeof(int32_t) * (size_t(1) << bits) + sizeof(uint16_t) * size_t(n_genomes);
    PGX_CUDA(cudaFuncSetAttribute(random_perms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    random_perms_kernel<<<static_cast<unsigned>(n_perm), threads, smem, static_cast<cudaStream_t>(stream)>>>(
        static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32), first, n_genomes, bits, d_perms);
    PGX_LAUNCH_CHECK("random_perms_kernel");
    return PGX_OK;
}

int pgx_curve_moments(const int32_t *d_curves, int64_t n_rows, int64_t width, int64_t *d_sum, uint64_t *d_sumsq,
                      int32_t *d_min, int32_t *d_max, int32_t accumulate, void *stream)
{
    if (!d_sum || !d_sumsq || !d_min || !d_max || (!d_curves && n_rows > 0))
        return pgx::fail(PGX_ERR_INVALID, "pgx_curve_moments: null pointer");
    if (n_rows < 0 || width < 0) return pgx::fail(PGX_ERR_INVALID, "pgx_curve_moments: negative size");
    if (width & 1) return pgx::fail(PGX_ERR_INVALID, "pgx_curve_moments: width must be even");
    if (n_rows > 0 && (reinterpret_cast<uintptr_t>(d_curves) & 7) != 0)
        return pgx::fail(PGX_ERR_INVALID, "pgx_curve_moments: d_curves must be 8-byte aligned");
    if (width == 0) return PGX_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (!accumulate) {
        const int64_t blocks = std::min<int64_t>((width + 255) / 256, 4096);
        moments_init_kernel<<<static_cast<unsigned>(blocks), 256, 0, s>>>(width, d_sum, d_sumsq, d_min, d_max);
        PGX_LAUNCH_CHECK("moments_init_kernel");
    }
    if (n_rows == 0) return PGX_OK;
    int dev = 0, sms = 148;
    PGX_CUDA(cudaGetDevice(&dev));
    PGX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int64_t col_blocks = (width / 2 + MOMENT_THREADS - 1) / MOMENT_THREADS;
    // about eight CTAs of 256 threads per SM in all, and at least 64 rows per slice to keep the atomics rare
    int64_t slices = std::max<int64_t>(1, (8 * int64_t(sms) + col_blocks - 1) / col_blocks);
    slices = std::min<int64_t>(slices, std::max<int64_t>(1, n_rows / 64));
    slices = std::min<int64_t>(slices, 65535);
    const int64_t rows_per_slice = (n_rows + slices - 1) / slices;
    slices = (n_rows + rows_per_slice - 1) / rows_per_slice;
    if (col_blocks > INT_MAX) return pgx::fail(PGX_ERR_INVALID, "pgx_curve_moments: width too large");
    curve_moments_kernel<<<dim3(static_cast<unsigned>(col_blocks), static_cast<unsigned>(slices)), MOMENT_THREADS, 0, s>>>(
        d_curves, n_rows, width, rows_per_slice, d_sum, d_sumsq, d_min, d_max);
    PGX_LAUNCH_CHECK("curve_moments_kernel");
    return PGX_OK;
}

}  // extern "C"
