// Every gene's k strongest co-expression partners (coextop), folded over strips of tile rows so that
// the genes x genes matrices never exist.  The host contracts one strip of tile rows [r0, r1) in
// NSR_MODE_COEX_UPPER into strip buffers P, D (rows r0 .. r1 - 1, full width) and then launches
// nsr_topk_strip once; each unordered pair (i < j) lies in exactly one strip, in the strip of row i, and
// reaches both of its rows there:
//   row r >= r0, column side : (i, P[i][r], D[i][r]) for r0 <= i < min(r1, r)   (column r of the strip)
//   row r in [r0, r1), row side: (j, P[r][j], D[r][j]) for j > r                 (row r of the strip)
// Only strictly-upper entries are read (diagonal tiles may hold anything below their diagonal), so a
// column never reaches a row twice.
//
// Ranking key r2 = dot^2 / (var_i var_j) with __dmul_rn / __ddiv_rn (no FMA): the same bits as numpy's
// dot * dot / (var_i * var_j).  Order: key descending, then column ascending - a total order, so the
// result does not depend on the strip height or on the order in which candidates arrive.
//
// Every row has one owner per launch, no atomics.  A row of the strip gets a CTA of its own, which scans
// its column side and its row side with all 8 warps (the row side is up to G entries long; a warp per row
// would leave the GPU idle at small strip heights).  Rows below the strip go 32 to a CTA, a warp owning 4:
// their column side stages 32 x 32 panels of D (32 strip rows x the CTA's 32 columns: one 256-byte segment
// per strip row) through shared memory.  A candidate that does not beat the row's current k-th entry is
// dropped at once; survivors wait in a shared-memory buffer and, once it is half full, one warp sorts them
// (bitonic) and merges them into the row's k slots in global memory: every slot that has to move moves once,
// to its rank in the merged order (ranks by binary search of each list in the other), and slots ranked k or
// later drop out.  P and dot of a survivor are fetched from the strip only when it enters the slots.
#include <limits.h>

#include <algorithm>

#include "nsr_common.cuh"
#include "topk.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kPanel = 32;                       // output rows per CTA below the strip
constexpr int kRowsPerWarp = kPanel / kWarps;
constexpr int kBuf = 64;                         // survivors buffered per row
constexpr int kFlush = kBuf - 32;                // merge when more than this many wait (a ballot adds <= 32)
constexpr int kRowBuf = 512;                     // survivors buffered by a strip row's CTA
constexpr int kRowFlush = kRowBuf - kThreads;    // ... merged when more than this many wait
constexpr int kUnroll = 4;                       // a strip row's candidate loads in flight per thread

struct RowState {                                // per output row of the CTA, shared memory
    double thr_key;                              // the k-th slot once all k are filled, else the empty key
    int thr_col;
    int count;                                   // survivors waiting in the buffer
    int n_valid;                                 // filled slots (a prefix of the k)
    int pad;
};

__device__ __forceinline__ double r2_key(double dot, double vi, double vj) {
    return __ddiv_rn(__dmul_rn(dot, dot), __dmul_rn(vi, vj));
}

// Merge the B (a power of two) survivors buffered for row r into its slots S[0, k) (warp-collective).
template <int B>
__device__ __forceinline__ void merge_row(Slot* __restrict__ S, int k, RowState& rs, double* __restrict__ bkey,
                                       int* __restrict__ bcol, const double* __restrict__ P,
                                       const double* __restrict__ D, int64_t ld, int64_t r0, int64_t r) {
    const int lane = threadIdx.x & 31;
    const int n_u = rs.count;
    const int n_v = rs.n_valid;
    __syncwarp();
    for (int q = n_u + lane; q < B; q += 32) { bkey[q] = -1.0; bcol[q] = kEmptyCol; }
    __syncwarp();
    // bitonic sort of the buffer into (key desc, col asc)
    for (int size = 2; size <= B; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = lane; t < B / 2; t += 32) {
                const int i = ((t & ~(stride - 1)) << 1) | (t & (stride - 1));
                const int j = i + stride;
                const double ki = bkey[i], kj = bkey[j];
                const int ci = bcol[i], cj = bcol[j];
                const bool first_wins = (i & size) == 0;
                if (first_wins ? beats(kj, cj, ki, ci) : beats(ki, ci, kj, cj)) {
                    bkey[i] = kj; bkey[j] = ki;
                    bcol[i] = cj; bcol[j] = ci;
                }
            }
            __syncwarp();
        }
    }
    // rank of each survivor among the filled slots (before any slot moves)
    int pos_u[B / 32];
#pragma unroll
    for (int t = 0; t < B / 32; ++t) {
        const int q = lane + 32 * t;
        pos_u[t] = INT_MAX;
        if (q < n_u) {
            const double ku = bkey[q];
            const int cu = bcol[q];
            int lo = 0, hi = n_v;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (beats(S[mid].key, S[mid].col, ku, cu)) lo = mid + 1; else hi = mid;
            }
            pos_u[t] = q + lo;
        }
    }
    __syncwarp();
    // filled slots move down by the number of survivors that beat them, last slot first
    for (int base = n_v - 1; base >= 0; base -= 32) {
        const int p = base - lane;
        Slot s;
        int b = 0;
        if (p >= 0) {
            s = S[p];
            int lo = 0, hi = n_u;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (beats(bkey[mid], bcol[mid], s.key, s.col)) lo = mid + 1; else hi = mid;
            }
            b = lo;
        }
        const bool moves = p >= 0 && b > 0;
        __syncwarp();                                   // every read of this batch before any write
        if (moves && p + b < k) S[p + b] = s;
        if (!__any_sync(0xffffffffu, moves)) break;     // b does not grow towards the top of the list
        __syncwarp();
    }
    __syncwarp();
    // the survivors into the gaps
#pragma unroll
    for (int t = 0; t < B / 32; ++t) {
        const int q = lane + 32 * t;
        if (q < n_u && pos_u[t] < k) {
            const int c = bcol[q];
            const int64_t at = c < r ? (int64_t)(c - r0) * ld + r : (r - r0) * ld + c;
            Slot s;
            s.key = bkey[q];
            s.p = P[at];
            s.dot = D[at];
            s.col = c;
            s.pad = 0;
            S[pos_u[t]] = s;
        }
    }
    __syncwarp();
    const int n_new = min(k, n_v + n_u);
    if (n_new == k) {
        const Slot last = S[k - 1];
        if (lane == 0) { rs.thr_key = last.key; rs.thr_col = last.col; }
    }
    if (lane == 0) { rs.n_valid = n_new; rs.count = 0; }
    __syncwarp();
}

// One batch of up to 32 candidates (one per lane) for row r: keep the ones that beat the k-th slot.
__device__ __forceinline__ void offer(bool valid, double key, int col, Slot* S, int k, RowState& rs,
                                      double* bkey, int* bcol, const double* P, const double* D, int64_t ld,
                                      int64_t r0, int64_t r) {
    const int lane = threadIdx.x & 31;
    const bool take = valid && beats(key, col, rs.thr_key, rs.thr_col);
    const unsigned m = __ballot_sync(0xffffffffu, take);
    if (m == 0) return;
    const int count = rs.count;
    if (take) {
        const int at = count + __popc(m & ((1u << lane) - 1u));
        bkey[at] = key;
        bcol[at] = col;
    }
    __syncwarp();
    if (lane == 0) rs.count = count + __popc(m);
    __syncwarp();
    if (rs.count > kFlush) merge_row<kBuf>(S, k, rs, bkey, bcol, P, D, ld, r0, r);
}

// Slots of row r at the start of a launch: the filled count, the threshold (warp-collective).
__device__ __forceinline__ void load_row(Slot* S, int k, int64_t r0, RowState& rs) {
    const int lane = threadIdx.x & 31;
    int n_v = 0;
    if (r0 == 0) {                                    // first strip: the slots are uninitialised
        for (int p = lane; p < k; p += 32) { S[p].key = -1.0; S[p].col = kEmptyCol; }
    } else if (S[k - 1].key >= 0.0) {
        n_v = k;
    } else {
        int lo = 0, hi = k - 1;                       // first empty slot
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (S[mid].key >= 0.0) lo = mid + 1; else hi = mid;
        }
        n_v = lo;
    }
    if (lane == 0) {
        rs.count = 0;
        rs.n_valid = n_v;
        rs.thr_key = n_v == k ? S[k - 1].key : -1.0;
        rs.thr_col = n_v == k ? S[k - 1].col : kEmptyCol;
    }
    __syncwarp();
}

// A row of the strip, one CTA: its column side (i in [r0, r), column r of the strip) and its row side
// (j > r, row r of the strip) as one index range, kThreads candidates per step and kUnroll steps' loads in
// flight; survivors are placed by a CTA-wide prefix of the warps' ballots, warp 0 merges.
__device__ __forceinline__ void strip_row(const double* __restrict__ P, const double* __restrict__ D, int64_t ld,
                                          int64_t r0, int64_t r, const double* __restrict__ var, int64_t G, int k,
                                          Slot* __restrict__ state) {
    __shared__ double s_key[kRowBuf];
    __shared__ int s_col[kRowBuf];
    __shared__ RowState s_rs;
    __shared__ int s_wcount[kWarps];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    Slot* S = state + r * k;
    if (warp == 0) load_row(S, k, r0, s_rs);
    __syncthreads();
    const double vr = var[r];
    const int64_t n_col = r - r0;
    const int64_t n_all = n_col + (G - 1 - r);
    for (int64_t t0 = 0; t0 < n_all; t0 += kThreads * kUnroll) {
        double key[kUnroll];
        int col[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const int64_t t = t0 + u * kThreads + threadIdx.x;
            key[u] = -1.0;
            col[u] = kEmptyCol;
            if (t < n_col) {
                key[u] = r2_key(D[t * ld + r], var[r0 + t], vr);
                col[u] = (int)(r0 + t);
            } else if (t < n_all) {
                const int64_t j = r + 1 + (t - n_col);
                key[u] = r2_key(D[n_col * ld + j], vr, var[j]);
                col[u] = (int)j;
            }
        }
        bool any = false;
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) any |= key[u] >= 0.0 && beats(key[u], col[u], s_rs.thr_key, s_rs.thr_col);
        if (!__syncthreads_or(any)) continue;         // the common case once the row's k slots are good
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const bool take = key[u] >= 0.0 && beats(key[u], col[u], s_rs.thr_key, s_rs.thr_col);
            if (!__syncthreads_or(take)) continue;
            const unsigned m = __ballot_sync(0xffffffffu, take);
            if (lane == 0) s_wcount[warp] = __popc(m);
            __syncthreads();
            int at = s_rs.count, total = 0;
            for (int w = 0; w < kWarps; ++w) {
                at += w < warp ? s_wcount[w] : 0;
                total += s_wcount[w];
            }
            if (take) {
                at += __popc(m & ((1u << lane) - 1u));
                s_key[at] = key[u];
                s_col[at] = col[u];
            }
            __syncthreads();
            if (warp == 0) {
                const int count = s_rs.count + total;
                __syncwarp();
                if (lane == 0) s_rs.count = count;
                __syncwarp();
                if (count > kRowFlush) merge_row<kRowBuf>(S, k, s_rs, s_key, s_col, P, D, ld, r0, r);
            }
            __syncthreads();
        }
    }
    if (warp == 0 && s_rs.count > 0) merge_row<kRowBuf>(S, k, s_rs, s_key, s_col, P, D, ld, r0, r);
}

// 32 consecutive rows below the strip (r >= r1), column side only: strip rows i in [r0, r1), 32 at a time
// through shared memory; a warp owns 4 of the rows.
__device__ __forceinline__ void panel_rows(const double* __restrict__ P, const double* __restrict__ D, int64_t ld,
                                           int64_t r0, int64_t r1, int64_t c0, const double* __restrict__ var,
                                           int64_t G, int k, Slot* __restrict__ state) {
    __shared__ double s_d[kPanel][kPanel + 1];     // D panel: 32 strip rows x the CTA's 32 columns
    __shared__ double s_var[kPanel];
    __shared__ double s_bkey[kPanel][kBuf];
    __shared__ int s_bcol[kPanel][kBuf];
    __shared__ RowState s_rs[kPanel];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int64_t c_end = min(G, c0 + kPanel);
    for (int w = 0; w < kRowsPerWarp; ++w) {
        const int lr = warp * kRowsPerWarp + w;
        if (c0 + lr >= G) break;
        load_row(state + (c0 + lr) * k, k, r0, s_rs[lr]);
    }
    for (int64_t i0 = r0; i0 < r1; i0 += kPanel) {
        __syncthreads();                              // previous panel consumed
        for (int e = threadIdx.x; e < kPanel * kPanel; e += kThreads) {
            const int ii = e / kPanel, cc = e % kPanel;
            const int64_t i = i0 + ii, c = c0 + cc;
            s_d[ii][cc] = (i < r1 && c < c_end) ? D[(i - r0) * ld + c] : 0.0;
        }
        if (threadIdx.x < kPanel) s_var[threadIdx.x] = i0 + threadIdx.x < r1 ? var[i0 + threadIdx.x] : 1.0;
        __syncthreads();
        for (int w = 0; w < kRowsPerWarp; ++w) {
            const int lr = warp * kRowsPerWarp + w;
            const int64_t r = c0 + lr;
            if (r >= G) break;
            const int64_t i = i0 + lane;
            const double key = r2_key(s_d[lane][lr], s_var[lane], var[r]);
            offer(i < r1, key, (int)i, state + r * k, k, s_rs[lr], s_bkey[lr], s_bcol[lr], P, D, ld, r0, r);
        }
    }
    for (int w = 0; w < kRowsPerWarp; ++w) {
        const int lr = warp * kRowsPerWarp + w;
        const int64_t r = c0 + lr;
        if (r >= G) break;
        if (s_rs[lr].count > 0)
            merge_row<kBuf>(state + r * k, k, s_rs[lr], s_bkey[lr], s_bcol[lr], P, D, ld, r0, r);
    }
}

// CTAs [0, r1 - r0): the rows of the strip, one each; then one CTA per 32 rows of [r1, G).
__global__ void __launch_bounds__(kThreads, 3)
topk_strip_kernel(const double* __restrict__ P, const double* __restrict__ D, int64_t ld, int64_t r0, int64_t r1,
                  const double* __restrict__ var, int64_t G, int k, Slot* __restrict__ state) {
    const int64_t n_strip = r1 - r0;
    if ((int64_t)blockIdx.x < n_strip)
        strip_row(P, D, ld, r0, r0 + blockIdx.x, var, G, k, state);
    else
        panel_rows(P, D, ld, r0, r1, r1 + ((int64_t)blockIdx.x - n_strip) * kPanel, var, G, k, state);
}

__global__ void topk_finish_kernel(const Slot* __restrict__ state, int64_t n, int64_t* __restrict__ idx,
                                   double* __restrict__ P_k, double* __restrict__ dot_k) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const Slot s = state[e];
        idx[e] = s.col;
        P_k[e] = s.p;
        dot_k[e] = s.dot;
    }
}

}  // namespace

extern "C" int nsr_topk_strip(nsr_ctx* ctx, uintptr_t stream, const double* P, const double* D, int64_t ld,
                              int64_t r0, int64_t r1, const double* var, int64_t G, int k, void* state) {
    NSR_REQUIRE(ctx && P && D && var && state, "nsr_topk_strip: null argument");
    NSR_REQUIRE(G >= 2 && G < INT_MAX && ld >= G, "nsr_topk_strip: bad shape G=%lld ld=%lld", (long long)G,
                (long long)ld);
    NSR_REQUIRE(k >= 1 && k <= NSR_TOPK_MAX && k <= G - 1, "nsr_topk_strip: k=%d outside [1, min(G - 1, %d)]", k,
                NSR_TOPK_MAX);
    NSR_REQUIRE(r0 >= 0 && r0 < r1 && r1 <= G, "nsr_topk_strip: bad strip [%lld, %lld) of %lld rows", (long long)r0,
                (long long)r1, (long long)G);
    NSR_CHECK(cudaSetDevice(ctx->device));
    const int64_t blocks = (r1 - r0) + (G - r1 + kPanel - 1) / kPanel;
    topk_strip_kernel<<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(P, D, ld, r0, r1, var, G, k,
                                                                               (Slot*)state);
    NSR_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int nsr_topk_finish(nsr_ctx* ctx, uintptr_t stream, const void* state, int64_t G, int k, int64_t* idx,
                               double* P_k, double* dot_k) {
    NSR_REQUIRE(ctx && state && idx && P_k && dot_k, "nsr_topk_finish: null argument");
    NSR_REQUIRE(G >= 2 && k >= 1 && k <= NSR_TOPK_MAX && k <= G - 1, "nsr_topk_finish: bad shape G=%lld k=%d",
                (long long)G, k);
    NSR_CHECK(cudaSetDevice(ctx->device));
    const int64_t n = G * k;
    const unsigned blocks = (unsigned)std::min<int64_t>((n + 255) / 256, 4 * 148 * 8);
    topk_finish_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const Slot*)state, n, idx, P_k, dot_k);
    NSR_CHECK(cudaGetLastError());
    return 0;
}
