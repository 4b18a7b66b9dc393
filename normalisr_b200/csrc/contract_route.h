// Which kernel a contraction call runs.  Host-only C++ without CUDA (tests/test_contract_route.py compiles it
// with g++): contract_impl (api.cu) collects the facts, nsr_contract_route decides, and the kernel-block rule is
// shared with the launchers in contract_umma.cu.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include "../../include/normalisr_b200.h"

enum class ContractRoute {
    SIMT,          // dp4a CUDA-core kernel, once per cell chunk
    ONE_PASS,      // single-CTA tcgen05 kernel, once per cell chunk
    PAIR,          // cta_group::2 pair kernel on pair tiles (nsr_pair_tiles), once per cell chunk
    ADAPTIVE,      // single-CTA kernel, 6 products on every tile, then 8 on the flagged ones
    SPLIT_CELLS,   // single-CTA kernel with work items (tile, part of the cells), then contract_finish_kernel
};

struct ContractRouteFacts {
    int engine;                   // NSR_ENGINE_*
    int mode;                     // NSR_MODE_* of the call
    int n_segs;
    int seg0_mode;                // NSR_MODE_* of segment 0
    int n_slices_a, n_slices_b, wmax;
    int64_t n, n_pad;             // cells, padded cells
    int64_t chunk;                // cells per pass: n_pad, or the caller's k_chunk when that is shorter
    int64_t n_tiles;
    int sm_count;
    int64_t slab;                 // rows_a * ld: doubles in one part's image of out2 (split over the cells)
    // nsr_set_option values
    int umma_pair, adaptive_min_cells, split_k, umma_kblock;
};

struct ContractRouteChoice {
    ContractRoute route;
    int parts;                    // SPLIT_CELLS: parts of the cells (> 1); otherwise 1
};

// Cells per pipeline stage of the single-CTA kernel: two stages of (sa + sb) planes x 128 rows x kb cells must
// fit its operand ring.  The pair kernel always takes 128.
inline int nsr_umma_kb(int n_slices_a, int n_slices_b, int umma_kblock) {
    return n_slices_a + n_slices_b > 6 ? 64 : umma_kblock;
}

// Number of parts the split kernel really uses for a request of n_parts over `cells` cells (no empty part).
inline int nsr_umma_parts(int64_t cells, int kb, int n_parts) {
    const int num_kb = (int)(cells / kb);
    if (n_parts <= 1 || num_kb < 1) return 1;
    const int per = (num_kb + n_parts - 1) / n_parts;
    return (num_kb + per - 1) / per;
}

// The rules in order of precedence: the first that applies wins.
inline ContractRouteChoice nsr_contract_route(const ContractRouteFacts& f) {
    if (f.engine == NSR_ENGINE_SIMT) return {ContractRoute::SIMT, 1};
    const bool adaptive = f.adaptive_min_cells > 0 && f.n >= f.adaptive_min_cells;
    // Pair kernel: one segment, equal plane counts, at least 3 of them.  umma_pair < 0 (default) picks it for
    // single-segment co-expression at 3 planes / 8 products, where its stacked-B schedule beats the single-CTA
    // kernel (profiles/r03_pair_stacked_ab.md), unless the adaptive schedule was asked for.
    const bool pair_ok = f.n_segs == 1 && f.n_slices_a == f.n_slices_b && f.n_slices_a >= 3;
    const bool pair_auto = f.mode == NSR_MODE_COEX && f.seg0_mode == NSR_MODE_COEX && f.n_slices_a == 3 && f.wmax == 5 &&
                           !adaptive;
    if (pair_ok && (f.umma_pair > 0 || (f.umma_pair < 0 && pair_auto))) return {ContractRoute::PAIR, 1};
    if (f.n_segs != 1) return {ContractRoute::ONE_PASS, 1};
    // Adaptive schedule (see nsr_adaptive_min_cells in api.cu): 3 planes / 8 products, one pass over the cells.
    if (adaptive && f.chunk == f.n_pad && f.mode != NSR_MODE_RAW && f.n_slices_a == 3 && f.n_slices_b == 3 &&
        f.wmax == 5)
        return {ContractRoute::ADAPTIVE, 1};
    // Few tiles, many cells (de: a few hundred groupings against every gene; the groupings' own Gram matrix):
    // with one CTA per tile the last wave of tiles leaves most SMs idle.  Split the cells into parts instead -
    // work items (tile, part) over all SMs, partial sums into per-part slabs, one small kernel that adds the
    // slabs in a fixed order and finishes.  The parts also serve as the overflow chunks (each part <= chunk).
    // Only the rectangular modes: their sums (two different variables, or an exact small-integer operand) stay
    // below 2^53, so the parts add up exactly and the result is the single-pass one bit for bit; co-expression
    // keeps its one-pass tiles (self-products of 24-bit values over 1e5 cells exceed 2^53, and its results are
    // promised to be identical across tilings and GPU counts).
    // Worth it when the one-CTA-per-tile launch would leave more than a quarter of the machine idle (its last wave):
    // the second kernel and the slabs cost about as much as a 20 % imbalance on these short launches (measured at
    // 300 x 10k x 50k cells: 237 tiles = 1.6 waves ran 0.52 ms one-pass, 0.6 ms split; 160 tiles over 1M cells ran
    // 10.6 ms one-pass, 7.9 ms split).
    const int64_t waves = (f.n_tiles + f.sm_count - 1) / f.sm_count;
    const bool unbalanced = 4 * f.n_tiles < 3 * waves * (int64_t)f.sm_count;
    if (f.split_k != 0 && f.n_tiles < 2 * (int64_t)f.sm_count && unbalanced &&
        (f.mode == NSR_MODE_DE || f.mode == NSR_MODE_RAW)) {
        const int64_t target = 4 * (int64_t)f.sm_count;                  // ~4 waves of work items
        int64_t want = (target + f.n_tiles - 1) / f.n_tiles;
        const int64_t for_overflow = (f.n_pad + f.chunk - 1) / f.chunk;
        if (want < for_overflow) want = for_overflow;
        const int64_t max_parts = f.n_pad / (8 * NSR_KBLOCK) > 0 ? f.n_pad / (8 * NSR_KBLOCK) : 1;   // >= 1024 cells per part
        if (want > max_parts && max_parts >= for_overflow) want = max_parts;
        const int parts = nsr_umma_parts(f.n_pad, nsr_umma_kb(f.n_slices_a, f.n_slices_b, f.umma_kblock), (int)want);
        if (parts > 1 && parts >= for_overflow && (size_t)parts * (size_t)f.slab * sizeof(double) <= ((size_t)1 << 30))
            return {ContractRoute::SPLIT_CELLS, parts};
    }
    return {ContractRoute::ONE_PASS, 1};
}
