// Bayesian logCPM (SURVEY 8f-4; reference src/normalisr/lcpm.py:21-208, default arguments):
//   lcpm[g][k] = digamma(1 + reads[g][k]) - digamma(total + 2) - log(sum_g exp(.)) + log(1e6)
// The digamma values come from a look-up table over the count values (the reference builds the
// same table, lcpm.py:96-109); the per-cell normalisation is a column reduction of exp(LUT[reads])
// (lcpm.py:155-157).  Two HBM-streaming passes over the count matrix: column statistics (sum of
// exp, total reads, non-zero genes: the covariates of lcpm.py:193-199 come from the same pass),
// then the gather + shift.  Rows = genes, columns = cells: a thread owns a cell column, so every
// access is coalesced; gene ranges are split over blockIdx.y and combined in a fixed order.
#include <limits.h>

#include "nsr_common.cuh"

namespace {

constexpr int kLcThreads = 256;
constexpr int kLcGeneSplit = 64;       // genes per CTA in the column pass

// ---- counter-based normal deviates (posterior resampling, lcpm.py:134-150 with varscale != 0) ----
// Philox4x32-10 (Salmon et al. 2011) keyed by the seed, counter = the entry's global index: the same
// entry gets the same deviate in both passes and for any chunking of the matrix.  Box-Muller on the
// first two 32-bit outputs.
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
}
__device__ __forceinline__ double philox_normal(uint64_t index, uint64_t seed) {
    uint32_t c[4] = {(uint32_t)index, (uint32_t)(index >> 32), 0u, 0u};
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c, k0, k1);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    const double u1 = ((double)c[0] + 0.5) * 2.3283064365386963e-10;       // (0, 1)
    const double u2 = ((double)c[1] + 0.5) * 2.3283064365386963e-10;
    return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}

// digamma(x), x >= 1: recurrence up to x >= 10, then the asymptotic series up to B14 (5e-16 absolute against
// scipy on [1, 2e7]; host twin in the tests).  Only counts beyond the look-up table take this path.
__device__ __forceinline__ double lc_digamma(double x) {
    double r = 0.0;
    while (x < 10.0) { r -= 1.0 / x; x += 1.0; }
    const double i = 1.0 / x, i2 = i * i;
    double s = -1.0 / 12.0;
    s = fma(s, i2, 691.0 / 32760.0);
    s = fma(s, i2, -1.0 / 132.0);
    s = fma(s, i2, 1.0 / 240.0);
    s = fma(s, i2, -1.0 / 252.0);
    s = fma(s, i2, 1.0 / 120.0);
    s = fma(s, i2, -1.0 / 12.0);
    return r + (log(x) - 0.5 * i + s * i2);
}

struct LcNoise {
    const double* lut_sd;      // sqrt(varscale * (trigamma(1 + c) - trigamma(total + 2))) per count value, or nullptr
    const double* noise;       // standard normal deviates, one per entry (ld_noise), or nullptr -> Philox
    int64_t ld_noise;
    uint64_t seed;
    int64_t row0, n_total;     // global gene index of row 0 and global row length (Philox counters)
};

// min / max / total of the counts in one pass (the checks and the table size of lcpm.py:88-99)
template <typename T>
__global__ void __launch_bounds__(kLcThreads)
lcpm_scan_kernel(const T* __restrict__ reads, int64_t genes, int64_t n, int64_t ld, long long* __restrict__ out) {
    long long mn = LLONG_MAX, mx = LLONG_MIN, tot = 0;
    const int64_t count = genes * n;
    for (int64_t i = (int64_t)blockIdx.x * kLcThreads + threadIdx.x; i < count; i += (int64_t)gridDim.x * kLcThreads) {
        const long long c = (long long)reads[(i / n) * ld + (i % n)];
        mn = c < mn ? c : mn;
        mx = c > mx ? c : mx;
        tot += c;
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        const long long a = __shfl_xor_sync(0xffffffffu, mn, m), b = __shfl_xor_sync(0xffffffffu, mx, m);
        mn = a < mn ? a : mn;
        mx = b > mx ? b : mx;
        tot += __shfl_xor_sync(0xffffffffu, tot, m);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(out, mn);
        atomicMax(out + 1, mx);
        atomicAdd((unsigned long long*)(out + 2), (unsigned long long)tot);
    }
}

// The per-cell loops of both passes for the CSR kernels: count(g) is the count of gene g in the thread's cell,
// read from the shared-memory tile the kernel expanded its entries into.  Each is the loop of the dense kernel
// below (lcpm_colstats_kernel, lcpm_apply_kernel) statement for statement, so that both paths compute the same
// bits; the dense kernels keep their own copy because calling these through a strided-load accessor changes
// their SASS.  Genes [g0, g1): one range of at most kLcGeneSplit.
// Column pass: the sum of exponentials starts at 0.0 for the range and takes the genes in batches of 8, in gene
// order (table values first, then the exponentials of counts beyond the table); every gene contributes, zeros
// included, so this order is part of the result.
template <typename T, bool NOISY, typename Count>
__device__ __forceinline__ void lc_colstats_cell(Count count, int64_t g0, int64_t g1, int64_t k, const double* __restrict__ lut,
                                                 const double* __restrict__ lut_exp, T len_t, const LcNoise& nz_,
                                                 double& se, unsigned long long& tot, int& nz, T& any_or, T& mx) {
    constexpr int kBatch = 8;                    // counts loaded before any of them is used: the table gather
                                                 // and the rare large-count branch must not serialise the loads
#pragma unroll 1
    for (int64_t g = g0; g < g1; g += kBatch) {
        T cc[kBatch];
#pragma unroll
        for (int i = 0; i < kBatch; ++i) cc[i] = g + i < g1 ? count(g + i) : (T)0;
        bool big = false;
#pragma unroll
        for (int i = 0; i < kBatch; ++i) {
            const T c = cc[i];
            const bool in = g + i < g1;
            const T ci = c < 0 ? (T)0 : (c >= len_t ? (T)(len_t - 1) : c);
            if (NOISY) {
                if (in) {
                    const double z = nz_.noise ? nz_.noise[(g + i) * nz_.ld_noise + k]
                                               : philox_normal((uint64_t)((nz_.row0 + g + i) * nz_.n_total + k), nz_.seed);
                    se += exp(fma(nz_.lut_sd[ci], z, lut[ci]));
                }
            } else {
                // exp(lut[c]) tabulated: the pass is a pure gather; counts beyond the table are added below
                const double v = lut_exp[ci];
                se += (in && c < len_t) ? v : 0.0;
                big = big || c >= len_t;
            }
            tot += (unsigned long long)(long long)c;
            nz += c != 0 ? 1 : 0;
            any_or |= c;
            mx = c > mx ? c : mx;
        }
        if (!NOISY && big) {
#pragma unroll
            for (int i = 0; i < kBatch; ++i)
                if (cc[i] >= len_t) se += exp(lc_digamma(1.0 + (double)cc[i]));
        }
    }
}

// Apply pass: out[g][k] = value - sh for the genes of the range.
template <bool NOISY, typename Count>
__device__ __forceinline__ void lc_apply_cell(Count count, int64_t g0, int64_t g1, int64_t k, const double* __restrict__ lut,
                                              int64_t lut_len, const LcNoise& nz_, double sh, double* __restrict__ out,
                                              int64_t ldo) {
#pragma unroll 8
    for (int64_t g = g0; g < g1; ++g) {
        const long long c = (long long)count(g);
        const long long ci = c < 0 ? 0 : (c >= lut_len ? lut_len - 1 : c);
        double v = (NOISY || c < lut_len) ? lut[ci] : lc_digamma(1.0 + (double)c);
        if (NOISY) {
            const double z = nz_.noise ? nz_.noise[g * nz_.ld_noise + k]
                                       : philox_normal((uint64_t)((nz_.row0 + g) * nz_.n_total + k), nz_.seed);
            v = fma(nz_.lut_sd[ci], z, v);
        }
        out[g * ldo + k] = v - sh;
    }
}

// Negativity check and largest count of the CTA (one atomic per warp)
template <typename T>
__device__ __forceinline__ void lc_minmax(T any_or, T mx, long long* __restrict__ minmax) {
    long long neg = any_or < 0 ? -1 : 0, m = (long long)mx;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        neg |= __shfl_xor_sync(0xffffffffu, neg, d);
        const long long b = __shfl_xor_sync(0xffffffffu, m, d);
        m = b > m ? b : m;
    }
    if ((threadIdx.x & 31) == 0) {
        if (neg < 0) atomicMin(minmax, -1ll);    // "some count is negative" (lcpm.py:88-89); rare
        if (m > *(volatile long long*)(minmax + 1)) atomicMax(minmax + 1, m);
    }
}

template <typename T, bool NOISY>
__global__ void __launch_bounds__(kLcThreads)
lcpm_colstats_kernel(const T* __restrict__ reads, int64_t genes, int64_t n, int64_t ld,
                     const double* __restrict__ lut, const double* __restrict__ lut_exp, int64_t lut_len, LcNoise nz_,
                     double* __restrict__ partial, long long* __restrict__ minmax) {
    const int64_t k = (int64_t)blockIdx.x * kLcThreads + threadIdx.x;
    const int64_t g0 = (int64_t)blockIdx.y * kLcGeneSplit, g1 = min(genes, g0 + kLcGeneSplit);
    // everything but the sum of exponentials stays in the counts' own integer type until the end (a gene
    // range holds 64 counts: the total is kept in 64 bits); negativity = the OR of the sign bits
    double se = 0.0;
    unsigned long long tot = 0;
    int nz = 0;
    T any_or = 0, mx = 0;
    const T len_t = (T)(lut_len > (int64_t)INT_MAX ? (int64_t)INT_MAX : lut_len);
    if (k < n) {
        const T* col = reads + k;
        constexpr int kBatch = 8;                    // counts loaded before any of them is used: the table gather
                                                     // and the rare large-count branch must not serialise the loads
#pragma unroll 1
        for (int64_t g = g0; g < g1; g += kBatch) {
            T cc[kBatch];
#pragma unroll
            for (int i = 0; i < kBatch; ++i) cc[i] = g + i < g1 ? col[(g + i) * ld] : (T)0;
            bool big = false;
#pragma unroll
            for (int i = 0; i < kBatch; ++i) {
                const T c = cc[i];
                const bool in = g + i < g1;
                const T ci = c < 0 ? (T)0 : (c >= len_t ? (T)(len_t - 1) : c);
                if (NOISY) {
                    if (in) {
                        const double z = nz_.noise ? nz_.noise[(g + i) * nz_.ld_noise + k]
                                                   : philox_normal((uint64_t)((nz_.row0 + g + i) * nz_.n_total + k), nz_.seed);
                        se += exp(fma(nz_.lut_sd[ci], z, lut[ci]));
                    }
                } else {
                    // exp(lut[c]) tabulated: the pass is a pure gather; counts beyond the table are added below
                    const double v = lut_exp[ci];
                    se += (in && c < len_t) ? v : 0.0;
                    big = big || c >= len_t;
                }
                tot += (unsigned long long)(long long)c;
                nz += c != 0 ? 1 : 0;
                any_or |= c;
                mx = c > mx ? c : mx;
            }
            if (!NOISY && big) {
#pragma unroll
                for (int i = 0; i < kBatch; ++i)
                    if (cc[i] >= len_t) se += exp(lc_digamma(1.0 + (double)cc[i]));
            }
        }
        double* o = partial + ((int64_t)blockIdx.y * 3) * n + k;
        o[0] = se;
        o[n] = (double)(long long)tot;
        o[2 * n] = (double)nz;
    }
    if (minmax != nullptr) {                         // negativity check and largest count from the same read
        long long neg = any_or < 0 ? -1 : 0, m = (long long)mx;
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            neg |= __shfl_xor_sync(0xffffffffu, neg, d);
            const long long b = __shfl_xor_sync(0xffffffffu, m, d);
            m = b > m ? b : m;
        }
        if ((threadIdx.x & 31) == 0) {
            if (neg < 0) atomicMin(minmax, -1ll);    // "some count is negative" (lcpm.py:88-89); rare
            if (m > *(volatile long long*)(minmax + 1)) atomicMax(minmax + 1, m);
        }
    }
}

__global__ void lcpm_colreduce_kernel(const double* __restrict__ partial, int64_t n, int n_split, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // over 3 * n
    if (i >= 3 * n) return;
    double s = 0.0;
    for (int p = 0; p < n_split; ++p) s += partial[(int64_t)p * 3 * n + i];
    out[i] = s;
}

template <typename T, bool NOISY>
__global__ void __launch_bounds__(kLcThreads)
lcpm_apply_kernel(const T* __restrict__ reads, int64_t genes, int64_t n, int64_t ld, const double* __restrict__ lut,
                  int64_t lut_len, LcNoise nz_, const double* __restrict__ shift, double* __restrict__ out, int64_t ldo) {
    const int64_t k = (int64_t)blockIdx.x * kLcThreads + threadIdx.x;
    if (k >= n) return;
    const double sh = shift ? shift[k] : 0.0;
    const int64_t g0 = (int64_t)blockIdx.y * kLcGeneSplit, g1 = min(genes, g0 + kLcGeneSplit);
#pragma unroll 8
    for (int64_t g = g0; g < g1; ++g) {
        const long long c = (long long)reads[g * ld + k];
        const long long ci = c < 0 ? 0 : (c >= lut_len ? lut_len - 1 : c);
        double v = (NOISY || c < lut_len) ? lut[ci] : lc_digamma(1.0 + (double)c);
        if (NOISY) {
            const double z = nz_.noise ? nz_.noise[g * nz_.ld_noise + k]
                                       : philox_normal((uint64_t)((nz_.row0 + g) * nz_.n_total + k), nz_.seed);
            v = fma(nz_.lut_sd[ci], z, v);
        }
        out[g * ldo + k] = v - sh;
    }
}


// ---- CSR counts (lcpm on sparse read-count matrices, never expanded to genes x cells) ----
// A CTA owns one range of kLcGeneSplit genes (blockIdx.y, as the dense kernels) and a span of consecutive
// 256-cell windows (blockIdx.x).  Per window it expands the range's stored entries into a 64 x 256 shared-memory
// tile of counts (zeros elsewhere) and runs the dense kernels' per-cell loop on it: the same per-cell order of
// operations, hence the same bits.  Column indices are ascending and unique within a row; each row keeps a cursor
// that only moves forward through the span (one binary search per row at the start of the span), so the counts
// are read once per pass: O(nnz) global traffic plus the (genes x cells) output of the apply pass.
constexpr int kLcCsrCtasPerSm = 3;     // 64 KB int32 tile per CTA (a 128 KB int64 tile for counts >= 2^31: one)

template <typename T>
struct LcCsrTile {
    T* tile;                           // [kLcGeneSplit][kLcThreads]
    int64_t* cur;                      // per row: next entry to place
    int64_t* stop;                     // per row: end of the row's entries
    int rows;

    // cursors of the range's rows at the first entry of column >= k_first
    __device__ __forceinline__ void begin(const int64_t* __restrict__ indptr, const int32_t* __restrict__ idx,
                                          int64_t k_first) {
        const int t = threadIdx.x;
        if (t < rows) {
            int64_t lo = indptr[t], hi = indptr[t + 1];
            stop[t] = hi;
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if ((int64_t)idx[mid] < k_first) lo = mid + 1;
                else hi = mid;
            }
            cur[t] = lo;
        }
        __syncthreads();
    }

    // the counts of cells [k0, k0 + kLcThreads) into the tile: a warp owns 8 rows and takes 32 entries of a row at a
    // time; the entries of the window are a prefix of what is left of the row.  The first 32 of all 8 rows are
    // loaded together (independent loads), only rows with more than 32 entries in the window go round again.
    __device__ __forceinline__ void expand(const int32_t* __restrict__ idx, const T* __restrict__ val, int64_t k0) {
        constexpr int kWarps = kLcThreads / 32, kRows = kLcGeneSplit / kWarps;
#pragma unroll 8
        for (int g = 0; g < kLcGeneSplit; ++g) tile[g * kLcThreads + threadIdx.x] = (T)0;
        __syncthreads();
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        int64_t p[kRows], c[kRows];
        T v[kRows];
#pragma unroll
        for (int q = 0; q < kRows; ++q) {
            const int r = warp + q * kWarps;
            p[q] = r < rows ? cur[r] : 0;
            const int64_t j = p[q] + lane;
            const bool live = r < rows && j < stop[r];
            c[q] = live ? (int64_t)idx[j] : LLONG_MAX;
            v[q] = live ? val[j] : (T)0;
        }
#pragma unroll
        for (int q = 0; q < kRows; ++q) {
            const int r = warp + q * kWarps;
            for (;;) {
                const bool in = c[q] < k0 + kLcThreads;
                if (in) tile[r * kLcThreads + (int)(c[q] - k0)] = v[q];
                const int m = __popc(__ballot_sync(0xffffffffu, in));
                p[q] += m;
                if (m < 32) break;
                const int64_t j = p[q] + lane;
                const bool live = j < stop[r];
                c[q] = live ? (int64_t)idx[j] : LLONG_MAX;
                v[q] = live ? val[j] : (T)0;
            }
            if (lane == 0 && r < rows) cur[r] = p[q];
        }
        __syncthreads();
    }
};

template <typename T, bool NOISY>
__global__ void __launch_bounds__(kLcThreads, kLcCsrCtasPerSm)
lcpm_colstats_csr_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ idx, const T* __restrict__ val,
                         int64_t genes, int64_t n, int64_t span, const double* __restrict__ lut,
                         const double* __restrict__ lut_exp, int64_t lut_len, LcNoise nz_, double* __restrict__ partial,
                         long long* __restrict__ minmax) {
    extern __shared__ __align__(16) unsigned char lc_smem[];
    __shared__ int64_t cur[kLcGeneSplit], stop[kLcGeneSplit];
    const int64_t g0 = (int64_t)blockIdx.y * kLcGeneSplit, g1 = min(genes, g0 + kLcGeneSplit);
    LcCsrTile<T> t{reinterpret_cast<T*>(lc_smem), cur, stop, (int)(g1 - g0)};
    const int64_t windows = (n + kLcThreads - 1) / kLcThreads;
    const int64_t w0 = (int64_t)blockIdx.x * span, w1 = min(windows, w0 + span);
    t.begin(indptr + g0, idx, w0 * kLcThreads);
    const T len_t = (T)(lut_len > (int64_t)INT_MAX ? (int64_t)INT_MAX : lut_len);
    T any_or = 0, mx = 0;
    const T* my = t.tile + threadIdx.x - g0 * kLcThreads;
    for (int64_t w = w0; w < w1; ++w) {
        t.expand(idx, val, w * kLcThreads);
        const int64_t k = w * kLcThreads + threadIdx.x;
        if (k < n) {
            double se = 0.0;
            unsigned long long tot = 0;
            int nz = 0;
            lc_colstats_cell<T, NOISY>([&](int64_t g) { return my[g * kLcThreads]; }, g0, g1, k, lut, lut_exp, len_t,
                                       nz_, se, tot, nz, any_or, mx);
            double* o = partial + ((int64_t)blockIdx.y * 3) * n + k;
            o[0] = se;
            o[n] = (double)(long long)tot;
            o[2 * n] = (double)nz;
        }
        __syncthreads();                               // the tile is refilled for the next window
    }
    if (minmax != nullptr) lc_minmax(any_or, mx, minmax);
}

template <typename T, bool NOISY>
__global__ void __launch_bounds__(kLcThreads, kLcCsrCtasPerSm)
lcpm_apply_csr_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ idx, const T* __restrict__ val,
                      int64_t genes, int64_t n, int64_t span, const double* __restrict__ lut, int64_t lut_len, LcNoise nz_,
                      const double* __restrict__ shift, double* __restrict__ out, int64_t ldo) {
    extern __shared__ __align__(16) unsigned char lc_smem[];
    __shared__ int64_t cur[kLcGeneSplit], stop[kLcGeneSplit];
    const int64_t g0 = (int64_t)blockIdx.y * kLcGeneSplit, g1 = min(genes, g0 + kLcGeneSplit);
    LcCsrTile<T> t{reinterpret_cast<T*>(lc_smem), cur, stop, (int)(g1 - g0)};
    const int64_t windows = (n + kLcThreads - 1) / kLcThreads;
    const int64_t w0 = (int64_t)blockIdx.x * span, w1 = min(windows, w0 + span);
    t.begin(indptr + g0, idx, w0 * kLcThreads);
    const T* my = t.tile + threadIdx.x - g0 * kLcThreads;
    for (int64_t w = w0; w < w1; ++w) {
        t.expand(idx, val, w * kLcThreads);
        const int64_t k = w * kLcThreads + threadIdx.x;
        if (k < n) {
            const double sh = shift ? shift[k] : 0.0;
            lc_apply_cell<NOISY>([&](int64_t g) { return my[g * kLcThreads]; }, g0, g1, k, lut, lut_len, nz_, sh, out, ldo);
        }
        __syncthreads();
    }
}

// windows per CTA: enough CTAs for about four waves at kLcCsrCtasPerSm, one window each on small problems
int64_t lc_csr_span(const nsr_ctx* ctx, int64_t n, int n_split) {
    const int64_t windows = (n + kLcThreads - 1) / kLcThreads;
    const int64_t want = (int64_t)ctx->sm_count * kLcCsrCtasPerSm * 4;
    const int64_t per_range = max((int64_t)1, min(windows, (want + n_split - 1) / n_split));
    return (windows + per_range - 1) / per_range;
}

}  // namespace

extern "C" int nsr_lcpm_scan(nsr_ctx* ctx, uintptr_t stream, const void* reads, int itemsize, int64_t genes, int64_t n,
                             int64_t ld, long long* out3) {
    NSR_REQUIRE(ctx && reads && out3, "nsr_lcpm_scan: null argument");
    NSR_REQUIRE((itemsize == 4 || itemsize == 8) && genes >= 1 && n >= 1 && ld >= n, "nsr_lcpm_scan: bad arguments");
    NSR_CHECK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const long long init[3] = {LLONG_MAX, LLONG_MIN, 0};
    NSR_CHECK(cudaMemcpyAsync(out3, init, sizeof(init), cudaMemcpyHostToDevice, st));
    const unsigned grid = (unsigned)(ctx->sm_count * 8);
    if (itemsize == 4) lcpm_scan_kernel<int32_t><<<grid, kLcThreads, 0, st>>>((const int32_t*)reads, genes, n, ld, out3);
    else lcpm_scan_kernel<int64_t><<<grid, kLcThreads, 0, st>>>((const int64_t*)reads, genes, n, ld, out3);
    NSR_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int nsr_lcpm_colstats(nsr_ctx* ctx, uintptr_t stream, const void* reads, int itemsize, int64_t genes,
                                 int64_t n, int64_t ld, const double* lut, const double* lut_exp, int64_t lut_len,
                                 const double* lut_sd, const double* noise, int64_t ld_noise, uint64_t seed, int64_t row0,
                                 double* colstats, long long* minmax) {
    NSR_REQUIRE(ctx && reads && lut && colstats && (lut_sd || lut_exp), "nsr_lcpm_colstats: null argument");
    NSR_REQUIRE((itemsize == 4 || itemsize == 8) && genes >= 1 && n >= 1 && ld >= n && lut_len >= 1 &&
                    (!noise || ld_noise >= n),
                "nsr_lcpm_colstats: bad arguments (itemsize %d)", itemsize);
    NSR_CHECK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int n_split = (int)((genes + kLcGeneSplit - 1) / kLcGeneSplit);
    NSR_REQUIRE(n_split <= 65535, "nsr_lcpm_colstats: too many genes for one call");
    void* scratch = nullptr;
    if (nsr_scratch(ctx, (size_t)n_split * 3 * n * sizeof(double), &scratch)) return 1;
    const dim3 grid((unsigned)((n + kLcThreads - 1) / kLcThreads), (unsigned)n_split);
    const LcNoise nz{lut_sd, noise, ld_noise, seed, row0, n};
#define NSR_LC(T_, N_) lcpm_colstats_kernel<T_, N_><<<grid, kLcThreads, 0, st>>>((const T_*)reads, genes, n, ld, lut, lut_exp, lut_len, nz, (double*)scratch, minmax)
    if (itemsize == 4) { if (lut_sd) NSR_LC(int32_t, true); else NSR_LC(int32_t, false); }
    else { if (lut_sd) NSR_LC(int64_t, true); else NSR_LC(int64_t, false); }
#undef NSR_LC
    lcpm_colreduce_kernel<<<(unsigned)((3 * n + 255) / 256), 256, 0, st>>>((const double*)scratch, n, n_split, colstats);
    NSR_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int nsr_lcpm_apply(nsr_ctx* ctx, uintptr_t stream, const void* reads, int itemsize, int64_t genes, int64_t n,
                              int64_t ld, const double* lut, int64_t lut_len, const double* lut_sd, const double* noise,
                              int64_t ld_noise, uint64_t seed, int64_t row0, const double* shift, double* out,
                              int64_t ldo) {
    NSR_REQUIRE(ctx && reads && lut && out, "nsr_lcpm_apply: null argument");
    NSR_REQUIRE((itemsize == 4 || itemsize == 8) && genes >= 1 && n >= 1 && ld >= n && ldo >= n && lut_len >= 1 &&
                    (!noise || ld_noise >= n),
                "nsr_lcpm_apply: bad arguments (itemsize %d)", itemsize);
    NSR_CHECK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int n_split = (int)((genes + kLcGeneSplit - 1) / kLcGeneSplit);
    NSR_REQUIRE(n_split <= 65535, "nsr_lcpm_apply: too many genes for one call");
    const dim3 grid((unsigned)((n + kLcThreads - 1) / kLcThreads), (unsigned)n_split);
    const LcNoise nz{lut_sd, noise, ld_noise, seed, row0, n};
#define NSR_LA(T_, N_) lcpm_apply_kernel<T_, N_><<<grid, kLcThreads, 0, st>>>((const T_*)reads, genes, n, ld, lut, lut_len, nz, shift, out, ldo)
    if (itemsize == 4) { if (lut_sd) NSR_LA(int32_t, true); else NSR_LA(int32_t, false); }
    else { if (lut_sd) NSR_LA(int64_t, true); else NSR_LA(int64_t, false); }
#undef NSR_LA
    NSR_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int nsr_lcpm_colstats_csr(nsr_ctx* ctx, uintptr_t stream, const int64_t* indptr, const int32_t* indices,
                                     const void* values, int itemsize, int64_t genes, int64_t n, const double* lut,
                                     const double* lut_exp, int64_t lut_len, const double* lut_sd, const double* noise,
                                     int64_t ld_noise, uint64_t seed, int64_t row0, double* colstats, long long* minmax) {
    NSR_REQUIRE(ctx && indptr && indices && values && lut && colstats && (lut_sd || lut_exp),
                "nsr_lcpm_colstats_csr: null argument");
    NSR_REQUIRE((itemsize == 4 || itemsize == 8) && genes >= 1 && n >= 1 && n <= (int64_t)INT_MAX && lut_len >= 1 &&
                    (!noise || ld_noise >= n),
                "nsr_lcpm_colstats_csr: bad arguments (itemsize %d)", itemsize);
    NSR_CHECK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int n_split = (int)((genes + kLcGeneSplit - 1) / kLcGeneSplit);
    NSR_REQUIRE(n_split <= 65535, "nsr_lcpm_colstats_csr: too many genes for one call");
    void* scratch = nullptr;
    if (nsr_scratch(ctx, (size_t)n_split * 3 * n * sizeof(double), &scratch)) return 1;
    const int64_t span = lc_csr_span(ctx, n, n_split);
    const dim3 grid((unsigned)((n + kLcThreads * span - 1) / (kLcThreads * span)), (unsigned)n_split);
    const size_t smem = (size_t)kLcGeneSplit * kLcThreads * itemsize;
    const LcNoise nz{lut_sd, noise, ld_noise, seed, row0, n};
#define NSR_LCS(T_, N_)                                                                                                \
    do {                                                                                                               \
        NSR_CHECK(cudaFuncSetAttribute((const void*)lcpm_colstats_csr_kernel<T_, N_>,                                  \
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                       \
        lcpm_colstats_csr_kernel<T_, N_><<<grid, kLcThreads, smem, st>>>(indptr, indices, (const T_*)values, genes, n, \
                                                                         span, lut, lut_exp, lut_len, nz,              \
                                                                         (double*)scratch, minmax);                    \
    } while (0)
    if (itemsize == 4) { if (lut_sd) NSR_LCS(int32_t, true); else NSR_LCS(int32_t, false); }
    else { if (lut_sd) NSR_LCS(int64_t, true); else NSR_LCS(int64_t, false); }
#undef NSR_LCS
    lcpm_colreduce_kernel<<<(unsigned)((3 * n + 255) / 256), 256, 0, st>>>((const double*)scratch, n, n_split, colstats);
    NSR_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int nsr_lcpm_apply_csr(nsr_ctx* ctx, uintptr_t stream, const int64_t* indptr, const int32_t* indices,
                                  const void* values, int itemsize, int64_t genes, int64_t n, const double* lut,
                                  int64_t lut_len, const double* lut_sd, const double* noise, int64_t ld_noise,
                                  uint64_t seed, int64_t row0, const double* shift, double* out, int64_t ldo) {
    NSR_REQUIRE(ctx && indptr && indices && values && lut && out, "nsr_lcpm_apply_csr: null argument");
    NSR_REQUIRE((itemsize == 4 || itemsize == 8) && genes >= 1 && n >= 1 && n <= (int64_t)INT_MAX && ldo >= n &&
                    lut_len >= 1 && (!noise || ld_noise >= n),
                "nsr_lcpm_apply_csr: bad arguments (itemsize %d)", itemsize);
    NSR_CHECK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int n_split = (int)((genes + kLcGeneSplit - 1) / kLcGeneSplit);
    NSR_REQUIRE(n_split <= 65535, "nsr_lcpm_apply_csr: too many genes for one call");
    const int64_t span = lc_csr_span(ctx, n, n_split);
    const dim3 grid((unsigned)((n + kLcThreads * span - 1) / (kLcThreads * span)), (unsigned)n_split);
    const size_t smem = (size_t)kLcGeneSplit * kLcThreads * itemsize;
    const LcNoise nz{lut_sd, noise, ld_noise, seed, row0, n};
#define NSR_LAS(T_, N_)                                                                                                \
    do {                                                                                                               \
        NSR_CHECK(cudaFuncSetAttribute((const void*)lcpm_apply_csr_kernel<T_, N_>,                                     \
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                       \
        lcpm_apply_csr_kernel<T_, N_><<<grid, kLcThreads, smem, st>>>(indptr, indices, (const T_*)values, genes, n,    \
                                                                      span, lut, lut_len, nz, shift, out, ldo);        \
    } while (0)
    if (itemsize == 4) { if (lut_sd) NSR_LAS(int32_t, true); else NSR_LAS(int32_t, false); }
    else { if (lut_sd) NSR_LAS(int64_t, true); else NSR_LAS(int64_t, false); }
#undef NSR_LAS
    NSR_CHECK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------
// compute_var (norm.py:56-128), column pass: with res = X - coef Qt (the covariate-projection
// residual, never materialised), per cell k
//     out[k] = sum_g ((res[g][k] - mean[g]) * inv_std[g])^2          (norm.py:103)
// A thread owns a cell column and keeps Qt[:, k] in registers; the coefficients, means and inverse
// standard deviations of the CTA's gene range sit in shared memory.  Gene ranges are split over
// blockIdx.y and combined in a fixed order.
namespace {

constexpr int kCvRank = 16;            // covariate rank handled (4 k-steps of the FP64 MMA)
constexpr int kCvGenes = 256;          // genes per CTA (blockIdx.y), combined in a fixed order afterwards
constexpr int kCvWarps = kLcThreads / 32;
constexpr int kCvCells = 16;           // cells per warp: two 8-cell MMA tiles

__device__ __forceinline__ void cv_dmma(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

// The residual tile X - coef Qt comes out of the FP64 tensor cores (A = -coef: 8 genes x 4 covariates per
// MMA, B = Qt: 4 covariates x 8 cells, fixed per warp and kept in registers, accumulator initialised with the
// X tile); lane (g, t) then holds gene g, cells 2 t and 2 t + 1 of each tile, standardises and squares
// them, and sums over its genes; the eight lanes of a cell are combined with shuffles at the end.
// KS = ceil(rank / 4).  FAST: rows are 16-byte aligned (vector loads for warps whose 16 cells all exist).
template <int KS, bool FAST>
__global__ void __launch_bounds__(kLcThreads)
colvar_kernel(const double* __restrict__ X, int64_t genes, int64_t n, int64_t ld, const double* __restrict__ Qt,
              int rank, int64_t ldq, const double* __restrict__ coef, int64_t ldcoef,
              const double* __restrict__ mean, const double* __restrict__ inv_std, double* __restrict__ partial) {
    constexpr int U = kCvCells / 8;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const int64_t c0 = ((int64_t)blockIdx.x * kCvWarps + warp) * kCvCells;
    if (c0 >= n) return;
    const int64_t g0 = (int64_t)blockIdx.y * kCvGenes, g1 = min(genes, g0 + kCvGenes);
    const bool full = FAST && c0 + kCvCells <= n;
    double bq[U][KS > 0 ? KS : 1], acc[U][2];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        acc[u][0] = acc[u][1] = 0.0;
        const int64_t cb = c0 + 8 * u + g;
#pragma unroll
        for (int kk = 0; kk < KS; ++kk) {
            const int j = 4 * kk + t;
            bq[u][kk] = (j < rank && cb < n) ? Qt[(int64_t)j * ldq + cb] : 0.0;
        }
    }
#pragma unroll 2
    for (int64_t gt = g0; gt < g1; gt += 8) {
        const int64_t gene = gt + g;
        const bool live = gene < g1;
        const int64_t gl = live ? gene : g0;
        double a[KS > 0 ? KS : 1];
#pragma unroll
        for (int kk = 0; kk < KS; ++kk) {
            const int j = 4 * kk + t;
            a[kk] = (live && j < rank) ? -coef[gl * ldcoef + j] : 0.0;
        }
        const double m = mean[gl], is = live ? inv_std[gl] : 0.0;
        const double* row = X + gl * ld + c0 + 2 * t;
        double d[U][2];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (full) {
                const double2 v = *reinterpret_cast<const double2*>(row + 8 * u);
                d[u][0] = v.x; d[u][1] = v.y;
            } else {
#pragma unroll
                for (int e = 0; e < 2; ++e) d[u][e] = (c0 + 8 * u + 2 * t + e < n) ? row[8 * u + e] : 0.0;
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
#pragma unroll
            for (int kk = 0; kk < KS; ++kk) cv_dmma(d[u][0], d[u][1], a[kk], bq[u][kk]);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const double z = (d[u][e] - m) * is;          // is = 0 for rows beyond the range
                acc[u][e] = fma(z, z, acc[u][e]);
            }
        }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            double v = acc[u][e];
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            const int64_t k = c0 + 8 * u + 2 * t + e;
            if (g == 0 && k < n) partial[(int64_t)blockIdx.y * n + k] = v;
        }
    }
}

__global__ void colvar_reduce_kernel(const double* __restrict__ partial, int64_t n, int n_split, double* __restrict__ out) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    double s = 0.0;
    for (int p = 0; p < n_split; ++p) s += partial[(int64_t)p * n + k];
    out[k] = s;
}

}  // namespace

extern "C" int nsr_colvar(nsr_ctx* ctx, uintptr_t stream, const double* X, int64_t genes, int64_t n, int64_t ld,
                          const double* Qt, int rank, int64_t ldq, const double* coef, int64_t ldcoef,
                          const double* mean, const double* inv_std, double* out) {
    NSR_REQUIRE(ctx && X && mean && inv_std && out, "nsr_colvar: null argument");
    NSR_REQUIRE(genes >= 1 && n >= 1 && ld >= n && rank >= 0 && rank <= kCvRank && (rank == 0 || (Qt && coef && ldq >= n && ldcoef >= rank)),
                "nsr_colvar: bad arguments (rank %d, at most %d)", rank, kCvRank);
    NSR_CHECK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int n_split = (int)((genes + kCvGenes - 1) / kCvGenes);
    NSR_REQUIRE(n_split <= 65535, "nsr_colvar: too many genes for one call");
    void* scratch = nullptr;
    if (nsr_scratch(ctx, (size_t)n_split * n * sizeof(double), &scratch)) return 1;
    const int64_t cells_per_cta = (int64_t)kCvWarps * kCvCells;
    const dim3 grid((unsigned)((n + cells_per_cta - 1) / cells_per_cta), (unsigned)n_split);
    const bool fast = ((uintptr_t)X % 16 == 0) && (ld % 2 == 0);          // vector loads: rows 16-byte aligned
#define NSR_CV(KS_)                                                                                                    \
    do {                                                                                                               \
        if (fast) colvar_kernel<KS_, true><<<grid, kLcThreads, 0, st>>>(X, genes, n, ld, Qt, rank, ldq, coef, ldcoef, mean, inv_std, (double*)scratch); \
        else colvar_kernel<KS_, false><<<grid, kLcThreads, 0, st>>>(X, genes, n, ld, Qt, rank, ldq, coef, ldcoef, mean, inv_std, (double*)scratch);     \
    } while (0)
    switch ((rank + 3) / 4) {
        case 0: NSR_CV(0); break;
        case 1: NSR_CV(1); break;
        case 2: NSR_CV(2); break;
        case 3: NSR_CV(3); break;
        default: NSR_CV(4); break;
    }
#undef NSR_CV
    colvar_reduce_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const double*)scratch, n, n_split, out);
    NSR_CHECK(cudaGetLastError());
    return 0;
}
