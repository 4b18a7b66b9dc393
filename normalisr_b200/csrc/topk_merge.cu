// coextop on several GPUs: the strips of tile rows are dealt out to the GPUs, each GPU runs the strip
// kernels of topk.cu on a state it has reset (nsr_topk_reset), and the owner of a block of rows merges the
// partial top-k lists of every GPU into the final one (nsr_topk_merge).
//
// The merge needs no sort and no atomics.  Every part holds a row's slots sorted by the selection order
// (topk.cuh's beats), the filled ones first, and a column reaches a row in one part only (a pair lives in
// exactly one strip).  The output rank of a filled slot is therefore its position in its own part plus, for
// every other part, the number of that part's slots that beat it (a binary search, the parts are sorted):
// the ranks of all filled slots of a row are a permutation, and the slots ranked below k are written once,
// straight to their place in idx / P_k / dot_k.  Parts are read through L1; a row's parts are not staged.
#include <algorithm>

#include "nsr_common.cuh"
#include "topk.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarpRowsMaxK = 128;               // up to this k a warp merges a row, above it a CTA does

struct Parts {
    const Slot* p[NSR_TOPK_MAX_PARTS];
};

__global__ void topk_reset_kernel(Slot* __restrict__ state, int64_t n) {
    Slot empty;
    empty.key = -1.0;
    empty.p = 0.0;
    empty.dot = 0.0;
    empty.col = kEmptyCol;
    empty.pad = 0;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x)
        state[e] = empty;
}

__device__ __forceinline__ double slot_key(const Slot* s) { return __ldg(&s->key); }
__device__ __forceinline__ int slot_col(const Slot* s) { return __ldg(&s->col); }

// kRowThreads threads (a warp or the CTA) per row, kThreads / kRowThreads rows per CTA.
template <int kRowThreads>
__global__ void __launch_bounds__(kThreads)
topk_merge_kernel(Parts parts, int n_parts, int64_t rows, int k, int64_t* __restrict__ idx, double* __restrict__ P_k,
                  double* __restrict__ dot_k, int* __restrict__ status) {
    constexpr int kRowsPerCta = kThreads / kRowThreads;
    __shared__ const Slot* s_parts[NSR_TOPK_MAX_PARTS];     // (indexed at run time: not from the parameters)
    __shared__ int s_n[kRowsPerCta][NSR_TOPK_MAX_PARTS];     // filled slots of each part
    const int lr = threadIdx.x / kRowThreads;
    const int t = threadIdx.x % kRowThreads;
    const int64_t r = (int64_t)blockIdx.x * kRowsPerCta + lr;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int q = 0; q < NSR_TOPK_MAX_PARTS; ++q) s_parts[q] = parts.p[q];
    }
    __syncthreads();
    if (r < rows && t < n_parts) {
        const Slot* S = s_parts[t] + r * k;
        int lo = 0, hi = k;                                    // first empty slot
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (slot_key(S + mid) >= 0.0) lo = mid + 1; else hi = mid;
        }
        s_n[lr][t] = lo;
    }
    __syncthreads();
    if (r >= rows) return;
    int total = 0;
    for (int q = 0; q < n_parts; ++q) total += s_n[lr][q];
    if (total < k) {
        if (t == 0) *status = 1;
        return;
    }
    for (int e = t; e < total; e += kRowThreads) {
        int p = 0, i = e;
        while (i >= s_n[lr][p]) i -= s_n[lr][p++];
        const Slot* S = s_parts[p] + r * k;
        const double key = slot_key(S + i);
        const int col = slot_col(S + i);
        int rank = i;
        for (int q = 0; q < n_parts && rank < k; ++q) {
            if (q == p) continue;
            const Slot* Q = s_parts[q] + r * k;
            int lo = 0, hi = min(s_n[lr][q], k - rank);        // a count of k - rank already drops the slot
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (beats(slot_key(Q + mid), slot_col(Q + mid), key, col)) lo = mid + 1; else hi = mid;
            }
            rank += lo;
        }
        if (rank < k) {
            const int64_t at = r * k + rank;
            idx[at] = col;
            P_k[at] = __ldg(&S[i].p);
            dot_k[at] = __ldg(&S[i].dot);
        }
    }
}

}  // namespace

extern "C" int nsr_topk_reset(nsr_ctx* ctx, uintptr_t stream, void* state, int64_t rows, int k) {
    NSR_REQUIRE(ctx && state, "nsr_topk_reset: null argument");
    NSR_REQUIRE(rows >= 0 && k >= 1 && k <= NSR_TOPK_MAX, "nsr_topk_reset: bad shape rows=%lld k=%d", (long long)rows,
                k);
    if (rows == 0) return 0;
    NSR_CHECK(cudaSetDevice(ctx->device));
    const int64_t n = rows * k;
    const unsigned blocks = (unsigned)std::min<int64_t>((n + 255) / 256, 4 * 148 * 8);
    topk_reset_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((Slot*)state, n);
    NSR_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int nsr_topk_merge(nsr_ctx* ctx, uintptr_t stream, const void* const* parts, int n_parts, int64_t rows,
                              int k, int64_t* idx, double* P_k, double* dot_k, int* status) {
    NSR_REQUIRE(ctx && parts && idx && P_k && dot_k && status, "nsr_topk_merge: null argument");
    NSR_REQUIRE(n_parts >= 1 && n_parts <= NSR_TOPK_MAX_PARTS, "nsr_topk_merge: %d parts outside [1, %d]", n_parts,
                NSR_TOPK_MAX_PARTS);
    NSR_REQUIRE(rows >= 0 && k >= 1 && k <= NSR_TOPK_MAX, "nsr_topk_merge: bad shape rows=%lld k=%d", (long long)rows,
                k);
    Parts ps = {};
    for (int q = 0; q < n_parts; ++q) {
        NSR_REQUIRE(parts[q], "nsr_topk_merge: part %d is null", q);
        ps.p[q] = (const Slot*)parts[q];
    }
    if (rows == 0) return 0;
    NSR_CHECK(cudaSetDevice(ctx->device));
    if (k <= kWarpRowsMaxK) {
        const int64_t blocks = (rows + kThreads / 32 - 1) / (kThreads / 32);
        topk_merge_kernel<32><<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(ps, n_parts, rows, k, idx, P_k,
                                                                                     dot_k, status);
    } else {
        topk_merge_kernel<kThreads><<<(unsigned)rows, kThreads, 0, (cudaStream_t)stream>>>(ps, n_parts, rows, k, idx,
                                                                                           P_k, dot_k, status);
    }
    NSR_CHECK(cudaGetLastError());
    return 0;
}
