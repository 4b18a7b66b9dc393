// Host build of csrc/contract_route.h for tests/test_contract_route.py (no GPU needed).
#include "contract_route.h"

// returns the route as an int (the order of ContractRoute) and its part count in *parts
extern "C" int route(int engine, int mode, int n_segs, int seg0_mode, int n_slices_a, int n_slices_b, int wmax, int64_t n,
                     int64_t n_pad, int64_t chunk, int64_t n_tiles, int sm_count, int64_t slab, int umma_pair,
                     int adaptive_min_cells, int split_k, int umma_kblock, int* parts) {
    const ContractRouteChoice c = nsr_contract_route({engine, mode, n_segs, seg0_mode, n_slices_a, n_slices_b, wmax, n, n_pad,
                                                      chunk, n_tiles, sm_count, slab, umma_pair, adaptive_min_cells, split_k,
                                                      umma_kblock});
    *parts = c.parts;
    return (int)c.route;
}
