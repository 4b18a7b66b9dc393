// P-value network -> binary network: per-row Benjamini-Hochberg + threshold, without sorting.
// Reference: src/normalisr/binnet.py:134-170 (binnet) calling bh (:77-131) on every row with the
// diagonal removed.  HBM-streaming: 8 B read + 1 B written per matrix entry.
//
// bh() gives entry j of a row (n0 off-diagonal entries, c_j = #{k : p_k <= p_j}) the Q-value
//   q_j = min_{k : p_k >= p_j} min(1, p_k / (c_k / n0)),
// so for qcut < 1:  q_j <= qcut  <=>  p_j <= p_(k*),  k* = max{c_k : p_k / (c_k / n0) <= qcut}.
// With g(c) = #{k : p_k / (c / n0) <= qcut} (non-increasing as c decreases) the sequence
// c <- g(c) started at c = n0 decreases to the largest fixed point, which is k*: every index
// that passes the reference's test at its own rank also passes it at any larger c, so the
// iterate never drops below k*, and a fixed point c = g(c) is itself an index set that passes.
// The kernel evaluates the SAME floating-point expression as the reference, p / (c / n0) <= qcut
// (binnet.py:122-124 computes w = cumsum / n0 and p / w), so the boolean output is bit-identical.
// One CTA per row: the row is read from HBM once into shared memory (rows up to 25,000 entries;
// wider rows re-read themselves from L2).
// The sparse (CSR) network takes two launches: the same row kernels instantiated with kCount write each
// row's threshold and edge count instead of the uint8 row (nsr_binnet_count), then binnet_csr_fill_kernel
// re-reads the rows and compacts the edges (nsr_binnet_csr_fill): 16 B read per entry + 4 B per edge.
#include "nsr_common.cuh"

namespace {

constexpr int kThreads = 1024;
constexpr int kSmemRowMax = 25000;     // doubles of a row kept in shared memory (200 KB; + 21 KB of tables)

__device__ __forceinline__ int block_sum(int v, int* s_red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();                                   // s_red reuse
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    int t = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) t += s_red[w];
    return t;
}

// Largest double t with fl(t / w) <= qcut.  Correctly rounded division is monotone in its
// numerator, so  fl(p / w) <= qcut  <=>  p <= t : the row passes compare against t instead of
// dividing every entry.  fl(qcut * w) is within a few ulp of t; step to it exactly.
__device__ __forceinline__ double bh_threshold(double w, double qcut) {
    double t = qcut * w;
    while (t / w > qcut) t = nextafter(t, 0.0);
    for (;;) {
        const double u = nextafter(t, 2.0);
        if (u / w <= qcut) t = u; else break;
    }
    return t;
}

__device__ __forceinline__ uint32_t bn_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// entries <= thr among s_row[0, cols): two per 16-byte shared-memory load
__device__ __forceinline__ int count_le(const double* s_row, int64_t cols, double thr) {
    int mine = 0;
    const double2* v = reinterpret_cast<const double2*>(s_row);
    const int64_t half = cols >> 1;
#pragma unroll 4
    for (int64_t j = threadIdx.x; j < half; j += kThreads) {
        const double2 p = v[j];
        mine += (p.x <= thr ? 1 : 0) + (p.y <= thr ? 1 : 0);
    }
    if ((cols & 1) && threadIdx.x == 0) mine += s_row[cols - 1] <= thr ? 1 : 0;
    return mine;
}

// ---------------------------------------------------------------------------------------------
// Rows that fit in shared memory: the fixed point is bracketed with a histogram, then finished
// exactly on the handful of entries inside the bracket - 4 passes over the row however slowly the
// plain iteration would converge (dense networks need dozens of iterations).
//   * non-negative doubles order like their bit patterns; key(p) = bits(p) >> (52 - m) is a
//     monotone bin index (relative width 2^-m).  Only thresholds between t(1) and qcut can occur,
//     so bins cover [key(t(1)), key(qcut)]: entries below are always counted, entries above never;
//   * cum[b] = #{p : bin(p) < b}.  With b = bin(t(c)):  cum[b] <= g(c) <= cum[b + 1].  Iterating
//     c <- cum[bin(t(c)) + 1] from the top ends at c_hi >= k*, iterating c <- cum[bin(t(c))] from
//     c_hi ends at c_lo <= k* (every fixed point of a minorant of g lies below k*);
//   * for c in [c_lo, c_hi] only entries in bins bin(t(c_lo)) .. bin(t(c_hi)) are undecided; they
//     are gathered (a few) and the exact iteration c <- base + #{window <= t(c)} runs on them.
constexpr int kBins = 4096;
constexpr int kWindow = 512;

struct RowShared {
    int hist[kBins + 1];
    double window[kWindow];
    int red[kThreads / 32];
    int n_window, c_final, fallback, b_lo, b_hi, base_w, c_hi;
    double thr;
    unsigned long long bar;
};


// kCount: instead of the uint8 row, write the row's threshold (thr_out, -1 without an edge) and its edge count
// (count_out): entry j is an edge iff j is not the diagonal and P[j] <= thr_out (nsr_binnet_csr_fill).
template <bool kCount>
__global__ void __launch_bounds__(kThreads)
binnet_rows_smem_kernel(const double* __restrict__ P, int64_t cols, int64_t ld, int64_t diag0, double qcut,
                        uint8_t* __restrict__ net, int64_t ld_net, unsigned long long* __restrict__ stats,
                        double* __restrict__ thr_out, int64_t* __restrict__ count_out) {
    extern __shared__ __align__(16) double s_row[];
    __shared__ RowShared sh;
    const int64_t row = blockIdx.x;
    const double* p_row = P + row * ld;
    const int64_t diag = row + diag0;
    const bool has_diag = diag >= 0 && diag < cols;
    const int64_t n0 = cols - (has_diag ? 1 : 0);
    const double n0d = (double)n0;
    if (n0 <= 0) {                                       // a 1 x 1 block holding only its diagonal entry
        if constexpr (kCount) {
            if (threadIdx.x == 0) { thr_out[row] = -1.0; count_out[row] = 0; }
        } else {
            for (int64_t j = threadIdx.x; j < cols; j += kThreads) net[row * ld_net + j] = 0;
        }
        return;
    }

    // ---- stage the row
    const bool bulk = (((uintptr_t)p_row & 15) == 0) && ((cols & 1) == 0);
    if (bulk) {
        const uint32_t bar = bn_smem_u32(&sh.bar);
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t bytes = (uint32_t)(cols * sizeof(double));
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(bn_smem_u32(s_row)), "l"(p_row), "r"(bytes), "r"(bar) : "memory");
        }
        for (int b = threadIdx.x; b <= kBins; b += kThreads) sh.hist[b] = 0;     // overlaps the copy
        uint32_t ok = 0;
        const long long t0 = clock64();
        while (!ok) {
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                         "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(0u) : "memory");
            if (!ok && clock64() - t0 > 4000000000ll) __trap();      // never hang the device
        }
    } else {
#pragma unroll 8
        for (int64_t j = threadIdx.x; j < cols; j += kThreads) s_row[j] = p_row[j];
        for (int b = threadIdx.x; b <= kBins; b += kThreads) sh.hist[b] = 0;
    }
    int bad = 0;
    if (threadIdx.x == 0) {
        sh.n_window = 0;
        sh.fallback = 0;
    }
    __syncthreads();
    if (has_diag && threadIdx.x == 0) {                  // the diagonal entry: validated, then made inert
        const double d = s_row[diag];
        if (!(d >= 0.0 && d <= 1.0)) bad = 1;
        s_row[diag] = 2.0;
    }

    // ---- bins: keys between t(1) and qcut; m mantissa bits so that they fit.  The key is taken from
    // the high word of the double (sign, exponent, 20 mantissa bits): 32-bit integer arithmetic only;
    // -0.0 has a negative high word and lands below the first bin, like every entry under t(1).
    // t_dn(c) <= t(c) <= t_up(c): fl(qcut * c / n0) moved a few ulp either way.  The bracketing only
    // needs bounds (a multiply instead of the divisions and nextafter steps of the exact threshold,
    // whose latency - not the passes over the row - dominated the first version of this kernel).
    const double kUp = 1.0 + 0x1p-48, kDn = 1.0 - 0x1p-48;
    const double t1 = (qcut / n0d) * kDn;
    int sh32 = 20 - 8;
    while ((__double2hiint(qcut) >> sh32) - (__double2hiint(t1) >> sh32) + 1 > kBins - 1) ++sh32;
    const int lo_key = __double2hiint(t1) >> sh32;
    const int n_bins = (__double2hiint(qcut) >> sh32) - lo_key + 1;
    __syncthreads();

    // ---- pass 1: validate (binnet.py:152-153), histogram of the candidates (p <= qcut)
    int below = 0;
    const int diag_i = has_diag ? (int)diag : -1;
    auto visit = [&](double p, int idx) {
        if (!(p >= 0.0 && p <= 1.0) && idx != diag_i) bad = 1;       // also catches NaN (the patched diagonal holds 2.0)
        if (p <= qcut) {
            const int key = (__double2hiint(p) >> sh32) - lo_key;
            if (key < 0) ++below;
            else atomicAdd(&sh.hist[key < n_bins ? key : n_bins - 1], 1);
        }
    };
    {
        const double2* v = reinterpret_cast<const double2*>(s_row);
        const int64_t half = cols >> 1;
#pragma unroll 4
        for (int64_t j = threadIdx.x; j < half; j += kThreads) {
            const double2 p = v[j];
            visit(p.x, 2 * (int)j);
            visit(p.y, 2 * (int)j + 1);
        }
        if ((cols & 1) && threadIdx.x == 0) visit(s_row[cols - 1], (int)cols - 1);
    }
    if (bad) atomicAdd(&stats[1], 1ull);
    below = block_sum(below, sh.red);                    // (syncs: histogram complete)

    // ---- exclusive prefix over the bins (4 per thread), cum[b] = below + sum_{b' < b} hist[b']
    {
        const int b0 = 4 * threadIdx.x;
        int h[4], tot = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) { h[i] = (b0 + i < n_bins) ? sh.hist[b0 + i] : 0; tot += h[i]; }
        int incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if ((threadIdx.x & 31) >= o) incl += v;
        }
        __syncthreads();
        if ((threadIdx.x & 31) == 31) sh.red[threadIdx.x >> 5] = incl;
        __syncthreads();
        int warp_off = 0;
        for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) warp_off += sh.red[w];
        int run = below + warp_off + incl - tot;
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (b0 + i <= n_bins) sh.hist[b0 + i] = run;   // entry n_bins = all candidates
            run += h[i];
        }
        __syncthreads();
    }

    // ---- bracket the fixed point (one thread; a multiply and two table reads per step)
    if (threadIdx.x == 0) {
        auto bin_of = [&](double t) {
            const int k = (__double2hiint(t) >> sh32) - lo_key;
            return k < 0 ? 0 : (k >= n_bins ? n_bins - 1 : k);
        };
        const double qn = qcut / n0d;
        int c = sh.hist[n_bins];
        while (c > 0) {                                   // majorant of g: ends at c_hi >= k*
            const int c2 = sh.hist[bin_of(fmin((double)c * qn * kUp, qcut)) + 1];
            if (c2 == c) break;
            c = c2;
        }
        const int c_hi = c;
        while (c > 0) {                                   // minorant of g: ends at c_lo <= k*
            const int c2 = sh.hist[bin_of((double)c * qn * kDn)];
            if (c2 == c) break;
            c = c2;
        }
        sh.c_hi = c_hi;
        if (c_hi > 0) {
            sh.b_lo = bin_of((double)(c > 1 ? c : 1) * qn * kDn);
            sh.b_hi = bin_of(fmin((double)c_hi * qn * kUp, qcut));
            sh.base_w = sh.hist[sh.b_lo];
        }
    }
    __syncthreads();
    int c = sh.c_hi;
    double thr = -1.0;
    if (c > 0) {
        // ---- gather the undecided entries
        const int b_lo = sh.b_lo, b_hi = sh.b_hi;
        auto pick = [&](double p) {
            if (p <= qcut) {
                int key = (__double2hiint(p) >> sh32) - lo_key;
                if (key >= n_bins) key = n_bins - 1;
                if (key >= b_lo && key <= b_hi) {
                    const int slot = atomicAdd(&sh.n_window, 1);
                    if (slot < kWindow) sh.window[slot] = p; else sh.fallback = 1;
                }
            }
        };
        {
            const double2* v = reinterpret_cast<const double2*>(s_row);
            const int64_t half = cols >> 1;
#pragma unroll 4
            for (int64_t j = threadIdx.x; j < half; j += kThreads) {
                const double2 p = v[j];
                pick(p.x);
                pick(p.y);
            }
            if ((cols & 1) && threadIdx.x == 0) pick(s_row[cols - 1]);
        }
        __syncthreads();
        if (!sh.fallback) {
            // ---- exact finish on the window (warp 0): the reference's own test, p / (c / n0) <= qcut
            if (threadIdx.x < 32) {
                const int nw = sh.n_window, base_w = sh.base_w;
                while (c > 0) {
                    const double w = (double)c / n0d;
                    int mine = 0;
                    for (int k = threadIdx.x; k < nw; k += 32) mine += sh.window[k] / w <= qcut ? 1 : 0;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
                    const int c2 = base_w + mine;
                    if (c2 == c) break;
                    c = c2;
                }
                if (threadIdx.x == 0) { sh.c_final = c; sh.thr = c > 0 ? bh_threshold((double)c / n0d, qcut) : -1.0; }
            }
            __syncthreads();
            c = sh.c_final;
            thr = sh.thr;
        } else {
            // window too large (a row packed with near-ties around the BH line): plain exact iteration
            // over the whole row from c_hi
            while (c > 0) {
                const double w = (double)c / n0d;
                int mine = 0;
#pragma unroll 4
                for (int64_t j = threadIdx.x; j < cols; j += kThreads) mine += s_row[j] / w <= qcut ? 1 : 0;
                const int c2 = block_sum(mine, sh.red);
                if (c2 == c) break;
                c = c2;
            }
            thr = c > 0 ? bh_threshold((double)c / n0d, qcut) : -1.0;
        }
    }
    // ---- output (thr = -1 when nothing passes; the patched diagonal holds 2.0)
    if constexpr (kCount) {
        if (threadIdx.x == 0) { thr_out[row] = c > 0 ? thr : -1.0; count_out[row] = c > 0 ? c : 0; }
    } else {
        uint8_t* o_row = net + row * ld_net;
        int64_t done = 0;
        if (((uintptr_t)o_row & 7) == 0) {               // 8 entries -> one 8-byte store
            const double2* v = reinterpret_cast<const double2*>(s_row);
            const int64_t oct = cols >> 3;
            for (int64_t j = threadIdx.x; j < oct; j += kThreads) {
                uint64_t out_bits = 0;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const double2 p = v[4 * j + q];
                    out_bits |= (uint64_t)(p.x <= thr ? 1 : 0) << (16 * q);
                    out_bits |= (uint64_t)(p.y <= thr ? 1 : 0) << (16 * q + 8);
                }
                reinterpret_cast<uint64_t*>(o_row)[j] = out_bits;
            }
            done = oct << 3;
        }
        for (int64_t j = done + threadIdx.x; j < cols; j += kThreads) o_row[j] = s_row[j] <= thr ? 1 : 0;
    }
    if (c > 0 && threadIdx.x == 0) atomicAdd(&stats[0], (unsigned long long)c);
}

// ---------------------------------------------------------------------------------------------
// Same procedure with the row kept as 2-byte KEYS instead of 8-byte values: key = 0 for an entry under the
// first bin (always below the threshold; -0.0 has a negative high word and lands here like 0), 1 + bin for an
// entry in a bin up to qcut's own, n_bins + 1 for everything above (and NaN, and the diagonal).  Entries of
// qcut's bin that exceed qcut are counted with the candidates: the tables only have to bracket g from both
// sides, and every entry near the threshold is compared by value.  A quarter of the shared memory, so
// FOUR rows are resident per SM (4 CTAs of 256 threads) and one row's table work (prefix, bracketing, exact
// finish: a few microseconds in which the SM of the 8-byte kernel loaded nothing) overlaps the other rows'
// streaming.  The row is read from HBM once with plain 16-byte loads; validation and the histogram happen on
// the values in flight.  Keys are monotone in p, so  key < key(thr) => p < thr  and  key > key(thr) => p > thr;
// only entries in the threshold's own bin (the undecided window: a few) are looked at again in global memory
// (L2).  Booleans bit-identical to the reference.
constexpr int kKeyThreads = 256;
constexpr int kKeyBins = 2048;

struct KeyShared {
    int hist[kKeyBins + 1];
    double window[kWindow];
    int window_idx[kWindow];
    int red[kKeyThreads / 32];
    int n_window, c_final, fallback, b_lo, b_hi, base_w, c_hi, below_adj;
    double thr;
};

__device__ __forceinline__ int block_sum_k(int v, int* s_red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();                                   // s_red reuse
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    int t = 0;
#pragma unroll
    for (int w = 0; w < kKeyThreads / 32; ++w) t += s_red[w];
    return t;
}

template <bool kCount>
__global__ void __launch_bounds__(kKeyThreads, 4)
binnet_rows_key_kernel(const double* __restrict__ P, int64_t cols, int64_t ld, int64_t diag0, double qcut,
                       uint8_t* __restrict__ net, int64_t ld_net, unsigned long long* __restrict__ stats,
                       double* __restrict__ thr_out, int64_t* __restrict__ count_out) {
    extern __shared__ __align__(16) uint16_t s_key[];
    __shared__ KeyShared sh;
    const int64_t row = blockIdx.x;
    const double* p_row = P + row * ld;
    const int64_t diag = row + diag0;
    const bool has_diag = diag >= 0 && diag < cols;
    const int diag_i = has_diag ? (int)diag : -1;
    const int64_t n0 = cols - (has_diag ? 1 : 0);
    const double n0d = (double)n0;
    if (n0 <= 0) {                                       // a 1 x 1 block holding only its diagonal entry
        if constexpr (kCount) {
            if (threadIdx.x == 0) { thr_out[row] = -1.0; count_out[row] = 0; }
        } else {
            for (int64_t j = threadIdx.x; j < cols; j += kKeyThreads) net[row * ld_net + j] = 0;
        }
        return;
    }
    for (int b = threadIdx.x; b <= kKeyBins; b += kKeyThreads) sh.hist[b] = 0;
    if (threadIdx.x == 0) {
        sh.n_window = 0;
        sh.fallback = 0;
    }
    // ---- bins (see binnet_rows_smem_kernel)
    const double kUp = 1.0 + 0x1p-48, kDn = 1.0 - 0x1p-48;
    const double t1 = (qcut / n0d) * kDn;
    int sh32 = 20 - 8;
    while ((__double2hiint(qcut) >> sh32) - (__double2hiint(t1) >> sh32) + 1 > kKeyBins - 1) ++sh32;
    const int lo_key = __double2hiint(t1) >> sh32;
    const int n_bins = (__double2hiint(qcut) >> sh32) - lo_key + 1;
    __syncthreads();

    // ---- pass 1 (the only read of the row from HBM): validate (binnet.py:152-153), keep the key, histogram
    // of the keys 1 .. n_bins.  Branch-free per entry; the diagonal entry is treated like any other and
    // taken out again afterwards.  Validation by the high word: anything that is not a plain number in [0, 1)
    // (NaN, negative, -0.0, >= 1) sets `susp`, and only then is the batch compared as doubles.
    int bad = 0, below = 0;
    uint32_t susp = 0;
    const int top = n_bins + 1;                          // key of everything above qcut's bin (NaN, the diagonal)
    const uint32_t hist_addr = bn_smem_u32(sh.hist);
    auto visit = [&](double p) -> uint32_t {
        const int hi = __double2hiint(p);
        susp |= ((uint32_t)hi >= 0x3FF00000u) ? 1u : 0u;
        const int key1 = min(max(((hi >> sh32) - lo_key) + 1, 0), top);   // 0: under the first bin (or negative zero)
        below += key1 == 0 ? 1 : 0;
        const uint32_t inside = (uint32_t)(key1 - 1) < (uint32_t)n_bins ? 1u : 0u;
        asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %1, 0;\n\t@q red.shared.add.u32 [%0], 1;\n\t}"
                     ::"r"(hist_addr + 4u * (uint32_t)(key1 - 1)), "r"(inside) : "memory");
        return (uint32_t)key1;
    };
    const bool vec = (((uintptr_t)p_row & 15) == 0) && ((cols & 1) == 0);
    if (vec) {
        const double2* v = reinterpret_cast<const double2*>(p_row);
        uint32_t* k2 = reinterpret_cast<uint32_t*>(s_key);
        const int half = (int)(cols >> 1);
        int j = threadIdx.x;
        for (; j + 7 * kKeyThreads < half; j += 8 * kKeyThreads) {      // eight 16-byte loads in flight per thread
            double2 p[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) p[u] = __ldcs(&v[j + u * kKeyThreads]);
#pragma unroll
            for (int u = 0; u < 8; ++u) k2[j + u * kKeyThreads] = visit(p[u].x) | (visit(p[u].y) << 16);
            if (susp) {
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    if (!(p[u].x >= 0.0 && p[u].x <= 1.0) || !(p[u].y >= 0.0 && p[u].y <= 1.0)) bad = 1;
                susp = 0;
            }
        }
        for (; j < half; j += kKeyThreads) {
            const double2 p = __ldcs(&v[j]);
            k2[j] = visit(p.x) | (visit(p.y) << 16);
            if (susp) {
                if (!(p.x >= 0.0 && p.x <= 1.0) || !(p.y >= 0.0 && p.y <= 1.0)) bad = 1;
                susp = 0;
            }
        }
    } else {
#pragma unroll 4
        for (int j = threadIdx.x; j < (int)cols; j += kKeyThreads) {
            const double p = p_row[j];
            s_key[j] = (uint16_t)visit(p);
            if (!(p >= 0.0 && p <= 1.0)) bad = 1;
        }
    }
    if (bad) atomicAdd(&stats[1], 1ull);
    below = block_sum_k(below, sh.red);                  // (syncs: keys and histogram complete)
    if (threadIdx.x == 0) {                              // the diagonal entry: out of the counts, key = never
        int adj = 0;
        if (has_diag) {
            const uint32_t k = s_key[diag_i];
            if (k == 0) adj = -1;
            else if (k != (uint32_t)top) sh.hist[k - 1] -= 1;
            s_key[diag_i] = (uint16_t)top;
        }
        sh.below_adj = adj;
    }
    __syncthreads();
    below += sh.below_adj;

    // ---- exclusive prefix over the bins (8 per thread), cum[b] = below + sum_{b' < b} hist[b']
    {
        constexpr int kPer = kKeyBins / kKeyThreads;
        const int b0 = kPer * threadIdx.x;
        int h[kPer], tot = 0;
#pragma unroll
        for (int i = 0; i < kPer; ++i) { h[i] = (b0 + i < n_bins) ? sh.hist[b0 + i] : 0; tot += h[i]; }
        int incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if ((threadIdx.x & 31) >= o) incl += v;
        }
        __syncthreads();
        if ((threadIdx.x & 31) == 31) sh.red[threadIdx.x >> 5] = incl;
        __syncthreads();
        int warp_off = 0;
        for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) warp_off += sh.red[w];
        int run = below + warp_off + incl - tot;
        __syncthreads();
#pragma unroll
        for (int i = 0; i < kPer; ++i) {
            if (b0 + i <= n_bins) sh.hist[b0 + i] = run;   // entry n_bins (<= kKeyBins - 1) = all candidates
            run += h[i];
        }
        __syncthreads();
    }

    // ---- bracket the fixed point (one thread; a multiply and two table reads per step)
    auto bin_of = [&](double t) {
        const int k = (__double2hiint(t) >> sh32) - lo_key;
        return k < 0 ? 0 : (k >= n_bins ? n_bins - 1 : k);
    };
    if (threadIdx.x == 0) {
        const double qn = qcut / n0d;
        int c = sh.hist[n_bins];
        while (c > 0) {                                   // majorant of g: ends at c_hi >= k*
            const int c2 = sh.hist[bin_of(fmin((double)c * qn * kUp, qcut)) + 1];
            if (c2 == c) break;
            c = c2;
        }
        const int c_hi = c;
        while (c > 0) {                                   // minorant of g: ends at c_lo <= k*
            const int c2 = sh.hist[bin_of((double)c * qn * kDn)];
            if (c2 == c) break;
            c = c2;
        }
        sh.c_hi = c_hi;
        if (c_hi > 0) {
            sh.b_lo = bin_of((double)(c > 1 ? c : 1) * qn * kDn);
            sh.b_hi = bin_of(fmin((double)c_hi * qn * kUp, qcut));
            sh.base_w = sh.hist[sh.b_lo];
        }
    }
    __syncthreads();
    int c = sh.c_hi;
    double thr = -1.0;
    if (c > 0) {
        // ---- gather the undecided entries: candidates in bins b_lo .. b_hi.  Two keys per 32-bit word are
        // tested at once: with bit 15 of each half set, subtracting k per half cannot borrow across halves and
        // leaves bit 15 set exactly where key >= k.
        const uint32_t k_lo = (uint32_t)sh.b_lo + 1u, k_hi = (uint32_t)sh.b_hi + 1u;
        {
            const uint4* k8 = reinterpret_cast<const uint4*>(s_key);
            const int octs = (int)(cols >> 3);
            const uint32_t H = 0x80008000u, lo2 = k_lo * 0x10001u, hi2 = (k_hi + 1u) * 0x10001u;
            auto pick = [&](uint32_t key, int idx) {
                if (key >= k_lo && key <= k_hi) {
                    const int slot = atomicAdd(&sh.n_window, 1);
                    if (slot < kWindow) sh.window_idx[slot] = idx; else sh.fallback = 1;
                }
            };
            auto in_range = [&](uint32_t w) { return ((w | H) - lo2) & ~((w | H) - hi2) & H; };
            for (int j = threadIdx.x; j < octs; j += kKeyThreads) {
                const uint4 k = k8[j];
                if (in_range(k.x) | in_range(k.y) | in_range(k.z) | in_range(k.w)) {
                    const uint32_t w[4] = {k.x, k.y, k.z, k.w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) { pick(w[q] & 0xFFFFu, 8 * j + 2 * q); pick(w[q] >> 16, 8 * j + 2 * q + 1); }
                }
            }
            for (int j = (octs << 3) + threadIdx.x; j < (int)cols; j += kKeyThreads) pick(s_key[j], j);
        }
        __syncthreads();
        if (!sh.fallback) {
            // ---- exact finish on the window (warp 0): the reference's own test, p / (c / n0) <= qcut
            if (threadIdx.x < 32) {
                const int nw = sh.n_window, base_w = sh.base_w;
                for (int k = threadIdx.x; k < nw; k += 32) sh.window[k] = p_row[sh.window_idx[k]];
                __syncwarp();
                while (c > 0) {
                    const double w = (double)c / n0d;
                    int mine = 0;
                    for (int k = threadIdx.x; k < nw; k += 32) mine += sh.window[k] / w <= qcut ? 1 : 0;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
                    const int c2 = base_w + mine;
                    if (c2 == c) break;
                    c = c2;
                }
                if (threadIdx.x == 0) { sh.c_final = c; sh.thr = c > 0 ? bh_threshold((double)c / n0d, qcut) : -1.0; }
            }
            __syncthreads();
            c = sh.c_final;
            thr = sh.thr;
        } else {
            // window too large (a row packed with near-ties around the BH line): plain exact iteration
            // over the whole row (from L2) from c_hi
            while (c > 0) {
                const double w = (double)c / n0d;
                int mine = 0;
#pragma unroll 4
                for (int j = threadIdx.x; j < (int)cols; j += kKeyThreads)
                    mine += (j != diag_i && p_row[j] / w <= qcut) ? 1 : 0;
                const int c2 = block_sum_k(mine, sh.red);
                if (c2 == c) break;
                c = c2;
            }
            thr = c > 0 ? bh_threshold((double)c / n0d, qcut) : -1.0;
        }
    }
    if constexpr (kCount) {
        if (threadIdx.x == 0) { thr_out[row] = c > 0 ? thr : -1.0; count_out[row] = c > 0 ? c : 0; }
        if (c > 0 && threadIdx.x == 0) atomicAdd(&stats[0], (unsigned long long)c);
        return;
    }
    // ---- output from the keys (c == 0: nothing passes).  thr = t(c) with 1 <= c, so t1 <= thr <= qcut and
    // its bin needs no clamping.  Entries in the threshold's own bin are the undecided window: the vector path
    // writes them as 0 and they are patched from the window's values afterwards.
    const uint32_t k_thr = c > 0 ? (uint32_t)bin_of(thr) + 1u : 0u;
    const bool windowed = c > 0 && !sh.fallback;
    auto decide = [&](uint32_t key, int idx) -> uint8_t {
        if (c <= 0) return 0;
        if (key != k_thr) return key < k_thr ? 1 : 0;
        return p_row[idx] <= thr ? 1 : 0;                 // (never the diagonal: its key is n_bins + 1)
    };
    uint8_t* o_row = net + row * ld_net;
    int done = 0;
    if (((uintptr_t)o_row & 7) == 0 && (windowed || c <= 0)) {         // 8 entries -> one 8-byte store
        const uint4* k8 = reinterpret_cast<const uint4*>(s_key);
        const int oct = (int)(cols >> 3);
        const uint32_t H = 0x80008000u, thr2 = k_thr * 0x10001u;
        auto below_thr = [&](uint32_t w) { return ~((w | H) - thr2) & H; };   // 0x80 in bytes 1 / 3 where key < k_thr
        for (int j = threadIdx.x; j < oct; j += kKeyThreads) {
            const uint4 k = k8[j];
            uint2 o;
            o.x = __byte_perm(below_thr(k.x), below_thr(k.y), 0x7531) >> 7;
            o.y = __byte_perm(below_thr(k.z), below_thr(k.w), 0x7531) >> 7;
            reinterpret_cast<uint2*>(o_row)[j] = o;
        }
        done = oct << 3;
        if (windowed) {
            __syncthreads();                              // the patch below lands after the vector stores
            const int nw = sh.n_window;
            for (int k = threadIdx.x; k < nw; k += kKeyThreads) {
                const int idx = sh.window_idx[k];
                if (idx < done && s_key[idx] == k_thr && sh.window[k] <= thr) o_row[idx] = 1;
            }
        }
    }
    for (int j = done + threadIdx.x; j < (int)cols; j += kKeyThreads) o_row[j] = decide(s_key[j], j);
    if (c > 0 && threadIdx.x == 0) atomicAdd(&stats[0], (unsigned long long)c);
}

// Rows wider than shared memory: plain iteration, the row re-read from L2 every step.
template <bool kCount>
__global__ void __launch_bounds__(kThreads)
binnet_rows_wide_kernel(const double* __restrict__ P, int64_t cols, int64_t ld, int64_t diag0, double qcut,
                        uint8_t* __restrict__ net, int64_t ld_net, unsigned long long* __restrict__ stats,
                        double* __restrict__ thr_out, int64_t* __restrict__ count_out) {
    __shared__ int s_red[kThreads / 32];
    const int64_t row = blockIdx.x;
    const double* p_row = P + row * ld;
    const int64_t diag = row + diag0;
    const bool has_diag = diag >= 0 && diag < cols;
    const int64_t n0 = cols - (has_diag ? 1 : 0);
    if (n0 <= 0) {
        if constexpr (kCount) {
            if (threadIdx.x == 0) { thr_out[row] = -1.0; count_out[row] = 0; }
        } else {
            for (int64_t j = threadIdx.x; j < cols; j += kThreads) net[row * ld_net + j] = 0;
        }
        return;
    }
    int bad = 0, mine = 0;
#pragma unroll 8
    for (int64_t j = threadIdx.x; j < cols; j += kThreads) {
        const double p = p_row[j];
        if (!(p >= 0.0 && p <= 1.0)) bad = 1;
        mine += (j != diag && p <= qcut) ? 1 : 0;
    }
    if (bad) atomicAdd(&stats[1], 1ull);
    int c = block_sum(mine, s_red);                    // g(n0): w = 1
    const double n0d = (double)n0;
    double thr = qcut;
    while (c > 0) {
        thr = bh_threshold((double)c / n0d, qcut);
        mine = 0;
#pragma unroll 8
        for (int64_t j = threadIdx.x; j < cols; j += kThreads) mine += (j != diag && p_row[j] <= thr) ? 1 : 0;
        const int c_new = block_sum(mine, s_red);
        if (c_new == c) break;
        c = c_new;
    }
    if (c == 0) thr = -1.0;
    if constexpr (kCount) {
        if (threadIdx.x == 0) { thr_out[row] = thr; count_out[row] = c; }
    } else {
        uint8_t* o_row = net + row * ld_net;
#pragma unroll 8
        for (int64_t j = threadIdx.x; j < cols; j += kThreads) o_row[j] = (j != diag && p_row[j] <= thr) ? 1 : 0;
    }
    if (c > 0 && threadIdx.x == 0) atomicAdd(&stats[0], (unsigned long long)c);
}

// ---------------------------------------------------------------------------------------------
// CSR compaction of rows whose threshold nsr_binnet_count found: entry j of row i is kept iff
// j != i + diag0 and P[j] <= thr[i] - the dense kernels' own decision (the key kernel's "key < key(thr)
// => p < thr" and exact finish on the threshold's bin, the 8-byte and wide kernels' p <= thr).  One CTA
// per row walks it in steps of 1024 entries: each warp takes 4 chunks of 32, a ballot per chunk gives the
// kept lanes, and a CTA prefix over the warps' counts (double-buffered, one barrier a step) places them, so
// the column indices come out ascending.  Optionally the same pass gathers P and a second matrix D at the
// kept positions.  A row never writes past its indptr range; a count that disagrees with it raises *err.
constexpr int kFillThreads = 256;
constexpr int kFillChunks = 4;          // 32-entry chunks per warp and step

template <typename Idx>
__global__ void __launch_bounds__(kFillThreads)
binnet_csr_fill_kernel(const double* __restrict__ P, int64_t cols, int64_t ld, int64_t diag0,
                       const double* __restrict__ thr, const int64_t* __restrict__ indptr, Idx* __restrict__ indices,
                       const double* __restrict__ D, int64_t ld_d, double* __restrict__ p_out,
                       double* __restrict__ d_out, unsigned long long* __restrict__ err) {
    __shared__ int s_tot[2][kFillThreads / 32];
    const int64_t row = blockIdx.x;
    const double t = thr[row];
    const int64_t begin = indptr[row], want = indptr[row + 1] - begin;
    if (!(t >= 0.0)) {                                   // a row without edges
        if (want != 0 && threadIdx.x == 0) atomicAdd(err, 1ull);
        return;
    }
    const double* p_row = P + row * ld;
    const double* d_row = D != nullptr ? D + row * ld_d : nullptr;
    const int64_t diag = row + diag0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t lower = (1u << lane) - 1u;
    int64_t written = 0;                                 // entries of the row placed by earlier steps
    int par = 0;
    for (int64_t j0 = 0; j0 < cols; j0 += kFillThreads * kFillChunks) {
        const int64_t jw = j0 + (int64_t)warp * (32 * kFillChunks) + lane;
        uint32_t m[kFillChunks];
        double pv[kFillChunks];
        int mine = 0;
#pragma unroll
        for (int u = 0; u < kFillChunks; ++u) {
            const int64_t j = jw + 32 * u;
            pv[u] = j < cols ? p_row[j] : 2.0;
            m[u] = __ballot_sync(0xffffffffu, j != diag && pv[u] <= t);
            mine += __popc(m[u]);
        }
        if (lane == 0) s_tot[par][warp] = mine;
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < kFillThreads / 32; ++w) {
            const int v = s_tot[par][w];
            before += w < warp ? v : 0;
            total += v;
        }
        int64_t pos = written + before;
#pragma unroll
        for (int u = 0; u < kFillChunks; ++u) {
            const int64_t k = pos + __popc(m[u] & lower);
            if (((m[u] >> lane) & 1u) && k < want) {
                const int64_t j = jw + 32 * u;
                indices[begin + k] = (Idx)j;
                if (p_out != nullptr) {
                    p_out[begin + k] = pv[u];
                    d_out[begin + k] = d_row[j];
                }
            }
            pos += __popc(m[u]);
        }
        written += total;
        par ^= 1;
    }
    if (written != want && threadIdx.x == 0) atomicAdd(err, 1ull);
}

constexpr int kKeyRowMax = 100000;     // keys of a row kept in shared memory (200 KB; four rows per SM up to ~20,000)

}  // namespace

int nsr_binnet_keys = 1;               // test hook (nsr_set_option "binnet_keys"): 0 = the 8-byte-row kernel

namespace {

// the row kernel nsr_binnet_keys and the row width select; kCount as in binnet_rows_smem_kernel
template <bool kCount>
int binnet_launch(nsr_ctx* ctx, uintptr_t stream, const double* P, int64_t rows, int64_t cols, int64_t ld,
                  int64_t diag0, double qcut, uint8_t* net, int64_t ld_net, unsigned long long* stats, double* thr,
                  int64_t* count) {
    NSR_REQUIRE(rows >= 1 && cols >= 1 && ld >= cols && (kCount || ld_net >= cols) && rows < (1ll << 31),
                "nsr_binnet: bad shape rows=%lld cols=%lld", (long long)rows, (long long)cols);
    NSR_REQUIRE(qcut > 0.0 && qcut < 1.0, "nsr_binnet: qcut must be in (0, 1)");
    NSR_CHECK(cudaSetDevice(ctx->device));
    if (nsr_binnet_keys != 0 && cols <= kKeyRowMax) {
        const int smem = (int)(((cols + 7) & ~(int64_t)7) * sizeof(uint16_t));
        NSR_CHECK(cudaFuncSetAttribute(binnet_rows_key_kernel<kCount>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       kKeyRowMax * (int)sizeof(uint16_t)));
        binnet_rows_key_kernel<kCount><<<(unsigned)rows, kKeyThreads, smem, (cudaStream_t)stream>>>(
            P, cols, ld, diag0, qcut, net, ld_net, stats, thr, count);
    } else if (cols <= kSmemRowMax) {
        const int smem = (int)(((cols + 1) & ~(int64_t)1) * sizeof(double));
        NSR_CHECK(cudaFuncSetAttribute(binnet_rows_smem_kernel<kCount>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       kSmemRowMax * (int)sizeof(double)));
        binnet_rows_smem_kernel<kCount><<<(unsigned)rows, kThreads, smem, (cudaStream_t)stream>>>(
            P, cols, ld, diag0, qcut, net, ld_net, stats, thr, count);
    } else {
        binnet_rows_wide_kernel<kCount><<<(unsigned)rows, kThreads, 0, (cudaStream_t)stream>>>(
            P, cols, ld, diag0, qcut, net, ld_net, stats, thr, count);
    }
    NSR_CHECK(cudaGetLastError());
    return 0;
}

}  // namespace

extern "C" int nsr_binnet(nsr_ctx* ctx, uintptr_t stream, const double* P, int64_t rows, int64_t cols, int64_t ld,
                          int64_t diag0, double qcut, uint8_t* net, int64_t ld_net, unsigned long long* stats) {
    NSR_REQUIRE(ctx && P && net && stats, "nsr_binnet: null argument");
    return binnet_launch<false>(ctx, stream, P, rows, cols, ld, diag0, qcut, net, ld_net, stats, nullptr, nullptr);
}

extern "C" int nsr_binnet_count(nsr_ctx* ctx, uintptr_t stream, const double* P, int64_t rows, int64_t cols,
                                int64_t ld, int64_t diag0, double qcut, double* thr, int64_t* count,
                                unsigned long long* stats) {
    NSR_REQUIRE(ctx && P && thr && count && stats, "nsr_binnet_count: null argument");
    return binnet_launch<true>(ctx, stream, P, rows, cols, ld, diag0, qcut, nullptr, 0, stats, thr, count);
}

extern "C" int nsr_binnet_csr_fill(nsr_ctx* ctx, uintptr_t stream, const double* P, int64_t rows, int64_t cols,
                                   int64_t ld, int64_t diag0, const double* thr, const int64_t* indptr, void* indices,
                                   int index_bytes, const double* D, int64_t ld_d, double* p_out, double* d_out,
                                   unsigned long long* err) {
    NSR_REQUIRE(ctx && P && thr && indptr && indices && err, "nsr_binnet_csr_fill: null argument");
    NSR_REQUIRE(index_bytes == 4 || index_bytes == 8, "nsr_binnet_csr_fill: index_bytes must be 4 or 8");
    NSR_REQUIRE((p_out == nullptr) == (d_out == nullptr) && (p_out == nullptr || (D && ld_d >= cols)),
                "nsr_binnet_csr_fill: p_out, d_out and D go together");
    NSR_REQUIRE(rows >= 1 && cols >= 1 && ld >= cols && rows < (1ll << 31),
                "nsr_binnet_csr_fill: bad shape rows=%lld cols=%lld", (long long)rows, (long long)cols);
    NSR_CHECK(cudaSetDevice(ctx->device));
    if (index_bytes == 4)
        binnet_csr_fill_kernel<int32_t><<<(unsigned)rows, kFillThreads, 0, (cudaStream_t)stream>>>(
            P, cols, ld, diag0, thr, indptr, (int32_t*)indices, D, ld_d, p_out, d_out, err);
    else
        binnet_csr_fill_kernel<int64_t><<<(unsigned)rows, kFillThreads, 0, (cudaStream_t)stream>>>(
            P, cols, ld, diag0, thr, indptr, (int64_t*)indices, D, ld_d, p_out, d_out, err);
    NSR_CHECK(cudaGetLastError());
    return 0;
}
