// Shared epilogue of the contraction kernels: exact integer cell-sums -> dot, r^2, P.
// Reference: association.py:234-249 (gamma, R2, beta.cdf) and :1036-1057 (dot, symmetry).
#pragma once
#include "nsr_common.cuh"
#include "pvalue.cuh"

struct ContractParams {
    int mode;                    // NSR_MODE_*
    int n_groups;                // weight groups kept (w = 2 .. n_groups + 1)
    int64_t rows_a, rows_b, ld;
    const double* qa; const double* va;
    const double* qb; const double* vb;
    double* P; double* out2;
    double inv_n;
    int acc_in;                  // add the float64 partial already stored at out2[i][j] (cell chunking)
    int raw_out;                 // store the running sum instead of finishing (not the last chunk)
    double refine_r2;            // adaptive schedule, first phase: r^2 above this marks the tile for the
                                 // full-precision second phase (< 0: off)
    int* need;                   // [n_tiles] flags of the first phase (device), or nullptr
    double group_scale[4];       // 256^(2S - w), relative to the least significant kept group
    double scale_all;            // weight of the least significant kept group
    NsrPvalParams pv;
};

// acc = exact sum_k V_ik V_jk restricted to the kept digit products, as a double
__device__ __forceinline__ double nsr_combine(const ContractParams& p, const int32_t* acc_g) {
    double s = 0.0;
#pragma unroll
    for (int g = 0; g < 4; ++g)
        if (g < p.n_groups) s = fma((double)acc_g[g], p.group_scale[g], s);
    return s * p.scale_all;
}

// One column segment of a contraction launch: its B operand's per-row scales and where its columns
// land in the output.  A plain nsr_contract call is a single segment built from ContractParams; the
// multi-GPU path (nsr_contract_segments) contracts the local gene block against itself and against
// every remote block it owns in ONE persistent launch, one segment per block.
struct SegInfo {
    const double* qb; const double* vb;      // quantum / variance of the segment's B rows
    int64_t rows_b;                          // valid B rows
    int64_t col0;                            // output column of B row 0
    int mode;                                // NSR_MODE_* of this segment's tiles
    const uint32_t* ready;                   // device flag: B may be read once *ready - ready_value >= 0 (or nullptr)
    uint32_t ready_value;
    uint32_t* done;                          // incremented once per epilogue warp and finished tile (or nullptr)
    double* mP; double* mO;                  // mirrored copy: element (i, j) also lands at m*[j * ldm + i] (or nullptr);
    int64_t ldm;                             // tiles on the diagonal of a symmetric segment are not mirrored
};

// host-side description of a segment's operand (what the tensor map is built from) + its SegInfo
struct NsrSegOperand {
    const int8_t* slices;
    int64_t rows_alloc;
    SegInfo info;
};

// One tcgen05 contraction launch as the host describes it: the A operand, the B segments, the device tile list
// and the cell range [cell_begin, cell_end) of this launch.
struct UmmaLaunch {
    const int8_t* a;
    int64_t rows_a, rows_alloc_a;
    int n_slices_a;
    const NsrSegOperand* segs;
    int n_segs;
    int n_slices_b;
    int64_t n_pad;
    int wmax;
    const int32_t* tiles;        // (tile_row, tile_col | segment << 24); pair kernel: nsr_pair_tiles entries
    int64_t n_tiles;             // entries of `tiles`
    const int* n_tiles_dev;      // if set, the count is read on the device (adaptive second phase), else nullptr
    int64_t cell_begin, cell_end;
};

// contract_umma.cu: the single-CTA kernel, the cta_group::2 pair kernel (one segment, equal plane counts) and, from
// contract_umma_splitk.cu, the single-CTA kernel split over the cells into n_parts parts whose unscaled sums go to
// slabs of part_stride doubles at part_out; nsr_launch_contract_finish adds those slabs and finishes.
int nsr_launch_contract_umma(nsr_ctx* ctx, cudaStream_t st, const UmmaLaunch& l, const ContractParams& ep);
int nsr_launch_contract_umma2(nsr_ctx* ctx, cudaStream_t st, const UmmaLaunch& l, const ContractParams& ep);
int nsr_launch_contract_umma_splitk(nsr_ctx* ctx, cudaStream_t st, const UmmaLaunch& l, const ContractParams& ep,
                                    int n_parts, double* part_out, int64_t part_stride);
int nsr_launch_contract_finish(cudaStream_t st, const int32_t* tiles_dev, int64_t n_tiles, const ContractParams& ep,
                               const SegInfo& sg, int n_parts, const double* part, int64_t part_stride);

// From sum = sum_k res_i res_j over ALL cells to the stored statistics of one output element (i = row in A,
// j = row in B); with `mP` the transposed element is written too (COEX, i != j tile: the other triangle of the
// same matrix; multi-GPU block pairs: the mirrored block).  Returns true when the element asks for the
// full-precision phase (adaptive schedule).
__device__ __forceinline__ bool nsr_finish_sum(const ContractParams& p, int mode, int64_t col0, int64_t i, int64_t j,
                                               double vi, double vj, double sum, double* mP, double* mO, int64_t ldm) {
    const int64_t at = i * p.ld + col0 + j;
    if (mode == NSR_MODE_RAW) {
        p.out2[at] = sum;
        return false;
    }
    const double dot = sum * p.inv_n;
    double P, o2;
    bool refine = false;
    if ((mode == NSR_MODE_COEX || mode == NSR_MODE_COEX_UPPER) && i == j) {
        P = 0.0; o2 = 0.0;                         // triu(.,1) + transpose leaves a zero diagonal
    } else {
        const double r2 = (dot * dot) / (vi * vj);
        refine = p.refine_r2 >= 0.0 && !(r2 <= p.refine_r2);
        P = nsr_pvalue_r2(r2, p.pv);
        o2 = (mode == NSR_MODE_DE) ? dot / vi : dot;
    }
    p.P[at] = P;
    p.out2[at] = o2;
    if (mP != nullptr) {
        mP[j * ldm + i] = P;
        mO[j * ldm + i] = o2;
    }
    return refine;
}

// One output element from the exact integer sum `acc` of this launch's cells: running sum over sequential
// cell chunks (acc_in / raw_out), then the statistics.  Kept as ONE function with its own copy of the
// statistics (not a call into nsr_finish_sum): the fused epilogue is power-bound at the headline size and the
// refactored form compiled to a 2.5 % slower step (profiles/r02_splitk_ab.md).  Launches split over the cells
// store the UNSCALED integer-valued sums per part instead (epilogue_tile<.., SPLIT>); contract_finish_kernel
// adds the parts in a fixed order, exactly while the total stays below 2^53, scales once and calls
// nsr_finish_sum: the single-pass result.
__device__ __forceinline__ bool nsr_finish(const ContractParams& p, int mode, int64_t col0, int64_t i, int64_t j,
                                           double qi, double vi, double qj, double vj, double acc, double* mP,
                                           double* mO, int64_t ldm) {
    double sum = (qi * qj) * acc;                  // sum_k res_i res_j over this launch's cells
    const int64_t at = i * p.ld + col0 + j;
    if (p.acc_in) sum += p.out2[at];               // earlier cell chunks
    if (mode == NSR_MODE_RAW || p.raw_out) {
        p.out2[at] = sum;
        return false;
    }
    const double dot = sum * p.inv_n;
    double P, o2;
    bool refine = false;
    if ((mode == NSR_MODE_COEX || mode == NSR_MODE_COEX_UPPER) && i == j) {
        P = 0.0; o2 = 0.0;                         // triu(.,1) + transpose leaves a zero diagonal
    } else {
        const double r2 = (dot * dot) / (vi * vj);
        refine = p.refine_r2 >= 0.0 && !(r2 <= p.refine_r2);
        P = nsr_pvalue_r2(r2, p.pv);
        o2 = (mode == NSR_MODE_DE) ? dot / vi : dot;
    }
    p.P[at] = P;
    p.out2[at] = o2;
    if (mP != nullptr) {
        mP[j * ldm + i] = P;
        mO[j * ldm + i] = o2;
    }
    return refine;
}
__device__ __forceinline__ bool nsr_finish(const ContractParams& p, int64_t i, int64_t j, double qi,
                                           double vi, double qj, double vj, double acc, bool mirror) {
    return nsr_finish(p, p.mode, 0, i, j, qi, vi, qj, vj, acc, mirror ? p.P : nullptr, p.out2, p.ld);
}
