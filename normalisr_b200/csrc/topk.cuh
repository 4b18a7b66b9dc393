// The slot layout and the order of coextop's selection, shared by the strip kernels (topk.cu) and the
// reset / merge kernels of the multi-GPU path (topk_merge.cu).
#pragma once
#include <limits.h>
#include <stdint.h>

namespace {

constexpr int kEmptyCol = INT_MAX;

struct __align__(16) Slot {                      // one of a row's k slots (32 B); empty: key < 0
    double key, p, dot;
    int32_t col, pad;
};
static_assert(sizeof(Slot) == 32, "Slot is 32 bytes (nsr_topk_strip's state layout)");

// The total order of the selection: key descending, then column ascending.
__device__ __forceinline__ bool beats(double ka, int ca, double kb, int cb) {
    return ka > kb || (ka == kb && ca < cb);
}

}  // namespace
