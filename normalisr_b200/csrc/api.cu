// C ABI of normalisr_b200 (see include/normalisr_b200.h for the contract of each entry).
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <array>
#include <unordered_map>
#include <vector>

#include <cuda.h>

#include "contract_route.h"
#include "epilogue.cuh"

int nsr_launch_contract_simt(cudaStream_t st, const int8_t* a, int64_t rows_alloc_a, int n_slices_a, const int8_t* b,
                             int64_t rows_alloc_b, int n_slices_b, int64_t n_pad, int wmax,
                             const int32_t* tiles_dev, int64_t n_tiles, const ContractParams& ep,
                             int64_t cell_begin, int64_t cell_end);
extern int nsr_use_hadamard;
extern int nsr_prefetch;
extern int nsr_umma_kblock;
extern int nsr_umma_pair;
extern int nsr_epi_warps;
extern int nsr_umma_stack;
extern int nsr_binnet_keys;
extern int nsr_umma_dynamic;
int nsr_split_k = 1;          // 1: few-tile launches split the cells over work items (nsr_contract_route)
extern int nsr_epi_sleep_ns;

// Adaptive digit-product schedule, OPT-IN (tcgen05 engine, 3 planes / 8 products, one pass over the
// cells): for n >= nsr_adaptive_min_cells every tile first runs the 6-product schedule (weight-5 products
// (2,3), (3,2) dropped: |dr| ~ 1.0e-6 / sqrt(n) at random sign, harmless unless the pair is extremely
// significant), tiles holding a pair with r^2 n > kRefineZ2 are redone with all 8.  For an
// unrefined pair the relative error of P is n |r| dr <= sqrt(kRefineZ2) * 1.0e-6 = 8e-6 (1 sigma).
// It pays only when extremely significant pairs are confined to few tiles (screens, sparse networks):
// on the 100k x 20k benchmark matrix 86 % of the tiles hold such a pair and the two phases cost twice
// the full schedule (profiles/r01am_adaptive_ab.md), hence off unless asked for.
int nsr_adaptive_min_cells = 0;        // 0 = always the full schedule; >= 8192 sensible when enabled
static constexpr double kRefineZ2 = 64.0;

namespace {
// tiles flagged by the first phase -> compact list (order irrelevant: integer sums) + count
__global__ void refine_compact_kernel(const int* __restrict__ need, const int32_t* __restrict__ tiles, int n_tiles,
                                      int32_t* __restrict__ out_tiles, int* __restrict__ out_count) {
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n_tiles; t += gridDim.x * blockDim.x) {
        if (need[t]) {
            const int slot = atomicAdd(out_count, 1);
            out_tiles[2 * slot] = tiles[2 * t];
            out_tiles[2 * slot + 1] = tiles[2 * t + 1];
        }
    }
}
}  // namespace

static thread_local char g_err[1024] = "";

void nsr_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int nsr_scratch(nsr_ctx* ctx, size_t bytes, void** out) {
    if (bytes > ctx->scratch_bytes) {
        // grow-only; a synchronising free is fine here (size changes are rare)
        if (ctx->scratch) NSR_CHECK(cudaFree(ctx->scratch));
        ctx->scratch = nullptr;
        ctx->scratch_bytes = 0;
        size_t want = bytes + bytes / 4;
        NSR_CHECK(cudaMalloc(&ctx->scratch, want));
        ctx->scratch_bytes = want;
    }
    *out = ctx->scratch;
    return 0;
}

extern "C" int nsr_version(void) { return NSR_VERSION; }
extern "C" const char* nsr_last_error(void) { return g_err; }

extern "C" int nsr_ctx_create(int device, nsr_ctx** out) {
    NSR_REQUIRE(out != nullptr, "nsr_ctx_create: null output pointer");
    int count = 0;
    NSR_CHECK(cudaGetDeviceCount(&count));
    NSR_REQUIRE(device >= 0 && device < count, "nsr_ctx_create: device %d of %d", device, count);
    NSR_CHECK(cudaSetDevice(device));
    cudaDeviceProp prop;
    NSR_CHECK(cudaGetDeviceProperties(&prop, device));
    NSR_REQUIRE(prop.major == 10, "normalisr_b200 is built for sm_100a only; device %d is sm_%d%d (%s)",
                device, prop.major, prop.minor, prop.name);
    nsr_ctx* ctx = new nsr_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    cudaDriverEntryPointQueryResult qres;
    void* fn = nullptr;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess) fn = nullptr;
    ctx->encode_tiled = fn;
    if (cudaMalloc(&ctx->tile_counters, NSR_TILE_COUNTERS * sizeof(int)) != cudaSuccess) {
        delete ctx;
        nsr_set_error("nsr_ctx_create: cudaMalloc failed");
        return 1;
    }
    *out = ctx;
    return 0;
}

extern "C" int nsr_ctx_destroy(nsr_ctx* ctx) {
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    if (ctx->scratch) cudaFree(ctx->scratch);
    if (ctx->tiles_dev) cudaFree(ctx->tiles_dev);
    if (ctx->tiles_pinned) cudaFreeHost(ctx->tiles_pinned);
    if (ctx->tiles_event) cudaEventDestroy(ctx->tiles_event);
    if (ctx->tile_counters) cudaFree(ctx->tile_counters);
    if (ctx->refine_dev) cudaFree(ctx->refine_dev);
    delete ctx;
    return 0;
}

// the options and their values: include/normalisr_b200.h
extern "C" int nsr_set_option(const char* name, int value) {
    if (!strcmp(name, "hadamard")) { nsr_use_hadamard = value ? 1 : 0; return 0; }
    if (!strcmp(name, "prefetch")) { nsr_prefetch = value ? 1 : 0; return 0; }
    if (!strcmp(name, "umma_pair")) { nsr_umma_pair = value < 0 ? -1 : (value ? 1 : 0); return 0; }
    if (!strcmp(name, "umma_dynamic")) { nsr_umma_dynamic = value ? 1 : 0; return 0; }
    if (!strcmp(name, "split_k")) { nsr_split_k = value ? 1 : 0; return 0; }
    if (!strcmp(name, "adaptive_min_cells")) { nsr_adaptive_min_cells = value < 0 ? 0 : value; return 0; }
    if (!strcmp(name, "binnet_keys")) { nsr_binnet_keys = value ? 1 : 0; return 0; }
    if (!strcmp(name, "umma_stack")) { nsr_umma_stack = value ? 1 : 0; return 0; }
    if (!strcmp(name, "epi_warps")) {
        NSR_REQUIRE(value == 8 || value == 16, "epi_warps must be 8 or 16");
        nsr_epi_warps = value;
        return 0;
    }
    if (!strcmp(name, "epi_sleep_ns")) { nsr_epi_sleep_ns = value < 0 ? 0 : value; return 0; }
    if (!strcmp(name, "umma_kblock")) {
        NSR_REQUIRE(value == 64 || value == 128, "umma_kblock must be 64 or 128");
        nsr_umma_kblock = value;
        return 0;
    }
    nsr_set_error("nsr_set_option: unknown option %s", name);
    return 2;
}

// Pair tiles for the cta_group::2 kernel: entries (row block of CTA 0, row block of CTA 1 or -1, column block).
// Tiles of one column are paired in the order they arrive, so an entry's rows usually are adjacent blocks.  A
// column with an odd number of tiles leaves one CTA of a pair idle; with `symmetric` (co-expression of one
// operand with itself: tile (j, i) holds the same sums as (i, j), and the epilogue writes both triangles) the
// next column with an odd count gives up its tile (lo, hi) as the transposed tile (hi, lo) of the column lo,
// which makes both counts even: 20,000 genes (157 block columns, 79 of them odd) leave one half-tile idle
// instead of 79.  Entries keep the order in which the caller's list first reaches them (it carries the
// L2-locality plan).  Returns the number of entries written to out (room for 3 * n_tiles).
extern "C" int64_t nsr_pair_tiles(const int32_t* tiles, int64_t n_tiles, int symmetric, int32_t* out) {
    struct Col { int32_t c; int64_t live; std::vector<int32_t> rows; std::vector<int64_t> pos; };
    std::vector<Col> cols;
    std::unordered_map<int32_t, size_t> col_of;
    std::unordered_map<uint64_t, size_t> slot_of;            // (column, row) -> index in the column's rows
    for (int64_t t = 0; t < n_tiles; ++t) {
        const int32_t r = tiles[2 * t], c = tiles[2 * t + 1];
        auto it = col_of.find(c);
        if (it == col_of.end()) { it = col_of.emplace(c, cols.size()).first; cols.push_back(Col{c, 0, {}, {}}); }
        Col& col = cols[it->second];
        slot_of.emplace(((uint64_t)(uint32_t)c << 32) | (uint32_t)r, col.rows.size());
        col.rows.push_back(r);
        col.pos.push_back(t);
        ++col.live;
    }
    if (symmetric) {
        int64_t pending = -1;                                 // earlier column with an odd count
        for (size_t k = 0; k < cols.size(); ++k) {
            if (cols[k].live % 2 == 0) continue;
            if (pending >= 0) {
                Col& a = cols[(size_t)pending];
                Col& b = cols[k];
                Col& lo = a.c < b.c ? a : b;
                Col& hi = a.c < b.c ? b : a;
                auto it = slot_of.find(((uint64_t)(uint32_t)hi.c << 32) | (uint32_t)lo.c);
                if (it != slot_of.end()) {                    // tile (lo, hi) exists: move it as (hi, lo)
                    lo.rows.push_back(hi.c);
                    lo.pos.push_back(hi.pos[it->second]);
                    ++lo.live;
                    hi.rows[it->second] = -1;
                    --hi.live;
                    slot_of.erase(it);
                    pending = -1;
                    continue;
                }
            }
            pending = (int64_t)k;
        }
    }
    std::vector<std::pair<int64_t, std::array<int32_t, 3>>> ent;
    ent.reserve((size_t)n_tiles);
    for (const Col& col : cols) {
        int64_t first = -1;
        int32_t r0 = -1;
        for (size_t q = 0; q < col.rows.size(); ++q) {
            if (col.rows[q] < 0) continue;
            if (r0 < 0) { r0 = col.rows[q]; first = col.pos[q]; continue; }
            ent.push_back({std::min(first, col.pos[q]), {r0, col.rows[q], col.c}});
            r0 = -1;
        }
        if (r0 >= 0) ent.push_back({first, {r0, -1, col.c}});
    }
    std::stable_sort(ent.begin(), ent.end(), [](const auto& x, const auto& y) { return x.first < y.first; });
    for (size_t e = 0; e < ent.size(); ++e)
        for (int q = 0; q < 3; ++q) out[3 * e + q] = ent[e].second[q];
    return (int64_t)ent.size();
}

// tile list: page-locked host memory (read over PCIe, zero-copy) -> device memory
__global__ void tiles_upload_kernel(int4* __restrict__ dst, const int4* __restrict__ src, int64_t n_vec) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

// One nsr_contract / nsr_contract_ab / nsr_contract_segments call.
// tile_stride = 2: host_tiles holds (tile_row, tile_col), one segment; 3: (segment, tile_row, tile_col).
struct ContractCall {
    int engine, mode;
    const int8_t* a_slices;
    int64_t rows_a, rows_alloc_a;
    int n_slices_a;
    const double* quantum_a;
    const double* var_a;
    const NsrSegOperand* segs;
    int n_segs, n_slices_b;
    int64_t n, n_pad;
    int n_products;
    const int32_t* host_tiles;
    int tile_stride;
    int64_t n_tiles;
    double dof_a;
    double* P;
    double* out2;
    int64_t ld, k_chunk;
};

// Checks a call's arguments but the tile list; *wmax = the largest digit weight kept, *need_p = P is written.
static int check_call(const ContractCall& c, int* wmax, bool* need_p) {
    NSR_REQUIRE(c.engine == NSR_ENGINE_UMMA || c.engine == NSR_ENGINE_SIMT, "nsr_contract: unknown engine %d", c.engine);
    NSR_REQUIRE(c.n_segs >= 1 && c.n_segs <= NSR_MAX_SEGMENTS && c.segs != nullptr, "nsr_contract: %d segments (1..%d)",
                c.n_segs, NSR_MAX_SEGMENTS);
    NSR_REQUIRE(c.n_segs == 1 || c.engine == NSR_ENGINE_UMMA, "nsr_contract: segments need the tcgen05 engine");
    NSR_REQUIRE(c.rows_a > 0 && c.n > 0 && c.n_pad == nsr_padded_cells(c.n),
                "nsr_contract: bad shape rows_a=%lld n=%lld n_pad=%lld", (long long)c.rows_a, (long long)c.n,
                (long long)c.n_pad);
    *wmax = nsr_wmax_ab(c.n_slices_a, c.n_slices_b, c.n_products);
    NSR_REQUIRE(*wmax > 0, "nsr_contract: unsupported (n_slices_a=%d, n_slices_b=%d, n_products=%d)", c.n_slices_a,
                c.n_slices_b, c.n_products);
    NSR_REQUIRE(c.out2 != nullptr && c.quantum_a && c.a_slices, "nsr_contract: null buffer");
    NSR_REQUIRE(((uintptr_t)c.a_slices & 15) == 0, "nsr_contract: slice planes must be 16-byte aligned");
    *need_p = false;
    for (int s = 0; s < c.n_segs; ++s) {
        const SegInfo& si = c.segs[s].info;
        NSR_REQUIRE(si.mode == NSR_MODE_COEX || si.mode == NSR_MODE_DE || si.mode == NSR_MODE_RAW ||
                        si.mode == NSR_MODE_COEX_UPPER || si.mode == NSR_MODE_COEX_RECT,
                    "nsr_contract: unknown mode %d", si.mode);
        const bool sym = si.mode == NSR_MODE_COEX || si.mode == NSR_MODE_COEX_UPPER;
        NSR_REQUIRE(si.rows_b > 0 && si.col0 >= 0 && c.ld >= si.col0 + si.rows_b && (!sym || c.rows_a == si.rows_b),
                    "nsr_contract: bad segment %d (rows_b=%lld col0=%lld ld=%lld)", s, (long long)si.rows_b,
                    (long long)si.col0, (long long)c.ld);
        NSR_REQUIRE(si.mode != NSR_MODE_COEX || c.n_segs == 1, "nsr_contract: NSR_MODE_COEX (mirrored) takes one segment");
        NSR_REQUIRE(c.segs[s].slices && si.qb && ((uintptr_t)c.segs[s].slices & 15) == 0,
                    "nsr_contract: segment %d: bad planes", s);
        NSR_REQUIRE(si.mode == NSR_MODE_RAW || si.vb != nullptr, "nsr_contract: segment %d: var missing", s);
        *need_p = *need_p || si.mode != NSR_MODE_RAW;
    }
    NSR_REQUIRE(!*need_p || (c.P != nullptr && c.var_a != nullptr && c.dof_a > 0.0), "nsr_contract: P / var / dof missing");
    return 0;
}

// Checks the call's tile list and packs it as (tile_row, tile_col | segment << 24).
static int pack_tiles(const ContractCall& c, std::vector<int32_t>& packed) {
    NSR_REQUIRE(c.host_tiles != nullptr && c.n_tiles > 0 && c.n_tiles < (1ll << 30), "nsr_contract: bad tile list");
    const int64_t tr_max = (c.rows_a + NSR_TILE - 1) / NSR_TILE;
    const int ts = c.tile_stride;
    packed.resize((size_t)c.n_tiles * 2);
    for (int64_t t = 0; t < c.n_tiles; ++t) {
        const int32_t sg = ts == 3 ? c.host_tiles[3 * t] : 0;
        const int32_t tr = c.host_tiles[ts * t + ts - 2], tc = c.host_tiles[ts * t + ts - 1];
        NSR_REQUIRE(sg >= 0 && sg < c.n_segs, "nsr_contract: tile %lld: segment %d out of range", (long long)t, sg);
        const int64_t tc_max = (c.segs[sg].info.rows_b + NSR_TILE - 1) / NSR_TILE;
        NSR_REQUIRE(tr >= 0 && tr < tr_max && tc >= 0 && tc < tc_max && tc < (1 << 24),
                    "nsr_contract: tile %lld = (%d,%d) out of range", (long long)t, tr, tc);
        const int m = c.segs[sg].info.mode;
        NSR_REQUIRE(!(m == NSR_MODE_COEX || m == NSR_MODE_COEX_UPPER) || tr <= tc, "nsr_contract: COEX tiles must have row <= col");
        packed[2 * t] = tr;
        packed[2 * t + 1] = tc | (sg << 24);
    }
    return 0;
}

// The epilogue's parameters of a call (segment 0 stands for the B operand).
static ContractParams contract_params(const ContractCall& c, int wmax, bool need_p) {
    const SegInfo& s0 = c.segs[0].info;
    ContractParams ep;
    ep.mode = c.mode;
    ep.n_groups = wmax - 1 < c.n_slices_a + c.n_slices_b - 1 ? wmax - 1 : c.n_slices_a + c.n_slices_b - 1;
    ep.rows_a = c.rows_a; ep.rows_b = s0.rows_b; ep.ld = c.ld;
    ep.qa = c.quantum_a; ep.va = c.var_a; ep.qb = s0.qb; ep.vb = s0.vb;
    ep.P = c.P; ep.out2 = c.out2;
    ep.inv_n = 1.0 / (double)c.n;
    ep.acc_in = 0;
    ep.raw_out = 0;
    ep.refine_r2 = -1.0;
    ep.need = nullptr;
    for (int g = 0; g < 4; ++g) ep.group_scale[g] = (g < ep.n_groups) ? ldexp(1.0, 8 * (ep.n_groups - 1 - g)) : 0.0;
    ep.scale_all = ldexp(1.0, 8 * (c.n_slices_a + c.n_slices_b - 1 - ep.n_groups));
    ep.pv = nsr_pval_params(need_p ? c.dof_a : 1.0);
    return ep;
}

// Puts n int32 of the tile list into ctx->tiles_dev.  The list travels through a pinned staging buffer owned by
// the context (a pageable source would make cudaMemcpyAsync block the host until the stream drains, and would tie
// the lifetime of the caller's vector to that staging behaviour); an event guards its reuse by the next call.
static int stage_tiles(nsr_ctx* ctx, cudaStream_t st, const int32_t* tiles, int64_t n) {
    if ((size_t)n > ctx->tiles_cap) {
        NSR_CHECK(cudaStreamSynchronize(st));
        if (ctx->tiles_dev) NSR_CHECK(cudaFree(ctx->tiles_dev));
        if (ctx->tiles_pinned) NSR_CHECK(cudaFreeHost(ctx->tiles_pinned));
        ctx->tiles_dev = nullptr;
        ctx->tiles_pinned = nullptr;
        ctx->tiles_cap = 0;
        NSR_CHECK(cudaMalloc(&ctx->tiles_dev, (size_t)n * sizeof(int32_t) * 2));
        NSR_CHECK(cudaMallocHost(&ctx->tiles_pinned, (size_t)n * sizeof(int32_t) * 2));
        ctx->tiles_cap = (size_t)n * 2;
    }
    if (ctx->tiles_event == nullptr) NSR_CHECK(cudaEventCreateWithFlags(&ctx->tiles_event, cudaEventDisableTiming));
    else NSR_CHECK(cudaEventSynchronize(ctx->tiles_event));       // previous upload has left the staging buffer
    memcpy(ctx->tiles_pinned, tiles, (size_t)n * sizeof(int32_t));
    // NOT a cudaMemcpyAsync: a host-to-device copy queues on the H2D copy engine, and in the streamed pipelines that
    // engine is busy with the next gigabyte-sized chunk of the expression matrix - the tile list then waits ~22 ms
    // behind it and so does the contraction (measured: every strip's launch started one chunk late, 350 -> 3xx ms
    // end to end at 100k x 20k).  A small kernel reads the page-locked list over PCIe instead.
    const int64_t n_vec = (n + 3) / 4;                     // the buffers are allocated with twice the room asked for
    const int blocks = (int)((n_vec + 255) / 256 < 16 ? (n_vec + 255) / 256 : 16);
    tiles_upload_kernel<<<blocks > 0 ? blocks : 1, 256, 0, st>>>(reinterpret_cast<int4*>(ctx->tiles_dev),
                                                                reinterpret_cast<const int4*>(ctx->tiles_pinned), n_vec);
    NSR_CHECK(cudaGetLastError());
    NSR_CHECK(cudaEventRecord(ctx->tiles_event, st));
    return 0;
}

// Cell chunking: int32 accumulators are exact only while no partial sum can overflow; the caller
// bounds that (Cauchy-Schwarz on the digit-plane energies) and passes the chunk length.  Chunks
// but the last leave the float64 running sum in out2; the last one adds it and finishes.
template <class Launch>
static int over_chunks(ContractParams ep, int64_t n_pad, int64_t chunk, Launch launch) {
    for (int64_t c0 = 0; c0 < n_pad; c0 += chunk) {
        const int64_t c1 = c0 + chunk < n_pad ? c0 + chunk : n_pad;
        ep.acc_in = c0 > 0;
        ep.raw_out = c1 < n_pad;
        if (int rc = launch(ep, c0, c1)) return rc;
    }
    return 0;
}

// Adaptive schedule: 6 products on every tile of l, then all 8 on the tiles the first phase flagged, whose list
// and count stay on the device.
static int contract_adaptive(nsr_ctx* ctx, cudaStream_t st, UmmaLaunch l, const ContractParams& ep, int64_t n) {
    const int64_t n_tiles = l.n_tiles;
    const size_t want = 3 * (size_t)n_tiles + 4;
    if (want > ctx->refine_cap) {
        if (ctx->refine_dev) NSR_CHECK(cudaFree(ctx->refine_dev));
        ctx->refine_dev = nullptr;
        ctx->refine_cap = 0;
        NSR_CHECK(cudaMalloc(&ctx->refine_dev, want * 2 * sizeof(int32_t)));
        ctx->refine_cap = want * 2;
    }
    int* need = ctx->refine_dev;
    int32_t* list = ctx->refine_dev + n_tiles;
    int* count = ctx->refine_dev + 3 * n_tiles;
    NSR_CHECK(cudaMemsetAsync(need, 0, (size_t)n_tiles * sizeof(int32_t), st));
    NSR_CHECK(cudaMemsetAsync(count, 0, sizeof(int32_t), st));
    ContractParams ep1 = ep;
    ep1.n_groups = 3;                                             // wmax = 4
    for (int g = 0; g < 4; ++g) ep1.group_scale[g] = (g < 3) ? ldexp(1.0, 8 * (2 - g)) : 0.0;
    ep1.scale_all = ldexp(1.0, 8 * (2 * 3 - 4));
    ep1.refine_r2 = kRefineZ2 / (double)n;
    ep1.need = need;
    l.wmax = 4;
    if (int rc = nsr_launch_contract_umma(ctx, st, l, ep1)) return rc;
    refine_compact_kernel<<<(unsigned)((n_tiles + 255) / 256 < 64 ? (n_tiles + 255) / 256 : 64), 256, 0, st>>>(
        need, l.tiles, (int)n_tiles, list, count);
    NSR_CHECK(cudaGetLastError());
    l.wmax = 5;
    l.tiles = list;
    l.n_tiles_dev = count;
    return nsr_launch_contract_umma(ctx, st, l, ep);
}

// Split over the cells: each of `parts` parts of the cells stores its partial sums in a slab of its own, then one
// small kernel adds the slabs in a fixed order and finishes.
static int contract_split(nsr_ctx* ctx, cudaStream_t st, const UmmaLaunch& l, const ContractParams& ep, int parts,
                          int64_t slab) {
    void* scratch = nullptr;
    if (nsr_scratch(ctx, (size_t)parts * (size_t)slab * sizeof(double), &scratch)) return 1;
    if (int rc = nsr_launch_contract_umma_splitk(ctx, st, l, ep, parts, (double*)scratch, slab)) return rc;
    return nsr_launch_contract_finish(st, l.tiles, l.n_tiles, ep, l.segs[0].info, parts, (const double*)scratch, slab);
}

// Shared implementation of nsr_contract / nsr_contract_ab / nsr_contract_segments: check the call, pack its tile
// list, route it (nsr_contract_route), stage the list on the device and run the route.
static int contract_impl(nsr_ctx* ctx, uintptr_t stream, const ContractCall& c) {
    NSR_REQUIRE(ctx != nullptr, "nsr_contract: null context");
    int wmax;
    bool need_p;
    if (int rc = check_call(c, &wmax, &need_p)) return rc;
    if (c.n_tiles == 0) return 0;
    NSR_REQUIRE(c.k_chunk >= 0 && c.k_chunk % NSR_KBLOCK == 0, "nsr_contract: k_chunk must be a multiple of %d", NSR_KBLOCK);
    std::vector<int32_t> tiles;
    if (int rc = pack_tiles(c, tiles)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    NSR_CHECK(cudaSetDevice(ctx->device));

    const NsrSegOperand& s0 = c.segs[0];
    const int64_t chunk = (c.k_chunk == 0 || c.k_chunk >= c.n_pad) ? c.n_pad : c.k_chunk;
    const ContractRouteChoice rt = nsr_contract_route({c.engine, c.mode, c.n_segs, s0.info.mode, c.n_slices_a, c.n_slices_b,
                                                       wmax, c.n, c.n_pad, chunk, c.n_tiles, ctx->sm_count, c.rows_a * c.ld,
                                                       nsr_umma_pair, nsr_adaptive_min_cells, nsr_split_k, nsr_umma_kblock});
    int64_t n_entries = c.n_tiles;
    if (rt.route == ContractRoute::PAIR) {
        // a transposed tile (j, i) holds the sums of (i, j) bit for bit when both operands are the same planes
        const int sym = c.mode == NSR_MODE_COEX && s0.info.mode == NSR_MODE_COEX && s0.slices == c.a_slices &&
                        s0.info.qb == c.quantum_a && s0.info.vb == c.var_a;
        std::vector<int32_t> entries((size_t)c.n_tiles * 3);
        n_entries = nsr_pair_tiles(tiles.data(), c.n_tiles, sym, entries.data());
        entries.resize((size_t)n_entries * 3);
        tiles.swap(entries);
    }
    if (int rc = stage_tiles(ctx, st, tiles.data(), (int64_t)tiles.size())) return rc;

    const ContractParams ep = contract_params(c, wmax, need_p);
    UmmaLaunch l = {c.a_slices, c.rows_a, c.rows_alloc_a, c.n_slices_a, c.segs, c.n_segs, c.n_slices_b, c.n_pad, wmax,
                    ctx->tiles_dev, n_entries, nullptr, 0, c.n_pad};
    switch (rt.route) {
    case ContractRoute::SIMT:
        return over_chunks(ep, c.n_pad, chunk, [&](const ContractParams& e, int64_t c0, int64_t c1) {
            if (nsr_launch_contract_simt(st, c.a_slices, c.rows_alloc_a, c.n_slices_a, s0.slices, s0.rows_alloc,
                                         c.n_slices_b, c.n_pad, wmax, l.tiles, l.n_tiles, e, c0, c1) == 0)
                return 0;
            nsr_set_error("nsr_contract: SIMT launch failed: %s", cudaGetErrorString(cudaGetLastError()));
            return 1;
        });
    case ContractRoute::ONE_PASS:
    case ContractRoute::PAIR:
        return over_chunks(ep, c.n_pad, chunk, [&](const ContractParams& e, int64_t c0, int64_t c1) {
            l.cell_begin = c0;
            l.cell_end = c1;
            return rt.route == ContractRoute::PAIR ? nsr_launch_contract_umma2(ctx, st, l, e)
                                                   : nsr_launch_contract_umma(ctx, st, l, e);
        });
    case ContractRoute::ADAPTIVE:
        return contract_adaptive(ctx, st, l, ep, c.n);
    case ContractRoute::SPLIT_CELLS:
        return contract_split(ctx, st, l, ep, rt.parts, c.rows_a * c.ld);
    }
    return 0;
}

extern "C" int nsr_contract_ab(nsr_ctx* ctx, uintptr_t stream, int engine, int mode,
                               const int8_t* a_slices, int64_t rows_a, int64_t rows_alloc_a, int n_slices_a,
                               const double* quantum_a, const double* var_a, const int8_t* b_slices,
                               int64_t rows_b, int64_t rows_alloc_b, int n_slices_b, const double* quantum_b,
                               const double* var_b, int64_t n, int64_t n_pad, int n_products,
                               const int32_t* host_tiles, int64_t n_tiles, double dof_a,
                               double* P, double* out2, int64_t ld, int64_t k_chunk) {
    NsrSegOperand sg;
    sg.slices = b_slices;
    sg.rows_alloc = rows_alloc_b;
    sg.info.qb = quantum_b; sg.info.vb = var_b; sg.info.rows_b = rows_b; sg.info.col0 = 0; sg.info.mode = mode;
    sg.info.ready = nullptr; sg.info.ready_value = 0; sg.info.done = nullptr;
    const bool mir = mode == NSR_MODE_COEX;          // both triangles of the same matrix
    sg.info.mP = mir ? P : nullptr; sg.info.mO = mir ? out2 : nullptr; sg.info.ldm = ld;
    return contract_impl(ctx, stream, {engine, mode, a_slices, rows_a, rows_alloc_a, n_slices_a, quantum_a, var_a, &sg, 1,
                                       n_slices_b, n, n_pad, n_products, host_tiles, 2, n_tiles, dof_a, P, out2, ld, k_chunk});
}

extern "C" int nsr_contract(nsr_ctx* ctx, uintptr_t stream, int engine, int mode,
                            const int8_t* a_slices, int64_t rows_a, int64_t rows_alloc_a,
                            const double* quantum_a, const double* var_a, const int8_t* b_slices,
                            int64_t rows_b, int64_t rows_alloc_b, const double* quantum_b,
                            const double* var_b, int64_t n, int64_t n_pad, int n_slices,
                            int n_products, const int32_t* host_tiles, int64_t n_tiles, double dof_a,
                            double* P, double* out2, int64_t ld, int64_t k_chunk) {
    return nsr_contract_ab(ctx, stream, engine, mode, a_slices, rows_a, rows_alloc_a, n_slices, quantum_a, var_a, b_slices,
                           rows_b, rows_alloc_b, n_slices, quantum_b, var_b, n, n_pad, n_products, host_tiles, n_tiles, dof_a,
                           P, out2, ld, k_chunk);
}

extern "C" int nsr_contract_segments(nsr_ctx* ctx, uintptr_t stream, const int8_t* a_slices, int64_t rows_a,
                                     int64_t rows_alloc_a, const double* quantum_a, const double* var_a,
                                     int64_t n, int64_t n_pad, int n_slices, int n_products,
                                     const nsr_segment* segments, int n_segments, const int32_t* host_tiles,
                                     int64_t n_tiles, double dof_a, double* P, double* out2, int64_t ld,
                                     int64_t k_chunk) {
    NSR_REQUIRE(segments != nullptr && n_segments >= 1 && n_segments <= NSR_MAX_SEGMENTS, "nsr_contract_segments: %d segments (1..%d)",
                n_segments, NSR_MAX_SEGMENTS);
    NsrSegOperand sg[NSR_MAX_SEGMENTS];
    for (int s = 0; s < n_segments; ++s) {
        const nsr_segment& in = segments[s];
        sg[s].slices = in.b_slices;
        sg[s].rows_alloc = in.rows_alloc_b;
        sg[s].info.qb = in.quantum_b; sg[s].info.vb = in.var_b; sg[s].info.rows_b = in.rows_b; sg[s].info.col0 = in.col0;
        sg[s].info.mode = in.diagonal ? NSR_MODE_COEX_UPPER : NSR_MODE_COEX_RECT;
        sg[s].info.ready = in.ready; sg[s].info.ready_value = in.ready_value; sg[s].info.done = in.done;
        NSR_REQUIRE((in.mirror_P == nullptr) == (in.mirror_out2 == nullptr) && (in.mirror_P == nullptr || in.ld_mirror >= rows_a),
                    "nsr_contract_segments: segment %d: bad mirror (ld_mirror=%lld)", s, (long long)in.ld_mirror);
        sg[s].info.mP = in.mirror_P; sg[s].info.mO = in.mirror_out2; sg[s].info.ldm = in.ld_mirror;
    }
    return contract_impl(ctx, stream, {NSR_ENGINE_UMMA, NSR_MODE_COEX_RECT, a_slices, rows_a, rows_alloc_a, n_slices,
                                       quantum_a, var_a, sg, n_segments, n_slices, n, n_pad, n_products, host_tiles, 3,
                                       n_tiles, dof_a, P, out2, ld, k_chunk});
}

// Stream-ordered 32-bit flag operations (cuStreamWriteValue32 / cuStreamWaitValue32): no kernel, no SM.
typedef CUresult (*StreamValueFn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
static int stream_value_op(nsr_ctx* ctx, const char* sym, uintptr_t stream, uint32_t* flag, uint32_t value, unsigned flags) {
    NSR_REQUIRE(ctx != nullptr && flag != nullptr, "%s: null argument", sym);
    NSR_CHECK(cudaSetDevice(ctx->device));
    cudaDriverEntryPointQueryResult qres;
    void* fn = nullptr;
    cudaError_t e = cudaGetDriverEntryPoint(sym, &fn, cudaEnableDefault, &qres);
    NSR_REQUIRE(e == cudaSuccess && qres == cudaDriverEntryPointSuccess && fn != nullptr, "%s unavailable", sym);
    CUresult r = ((StreamValueFn)fn)((CUstream)stream, (CUdeviceptr)(uintptr_t)flag, value, flags);
    NSR_REQUIRE(r == CUDA_SUCCESS, "%s failed with CUresult %d", sym, (int)r);
    return 0;
}
extern "C" int nsr_stream_signal(nsr_ctx* ctx, uintptr_t stream, uint32_t* flag, uint32_t value) {
    return stream_value_op(ctx, "cuStreamWriteValue32", stream, flag, value, 0 /* CU_STREAM_WRITE_VALUE_DEFAULT */);
}
extern "C" int nsr_stream_wait_geq(nsr_ctx* ctx, uintptr_t stream, uint32_t* flag, uint32_t value) {
    return stream_value_op(ctx, "cuStreamWaitValue32", stream, flag, value, 0 /* CU_STREAM_WAIT_VALUE_GEQ */);
}

extern "C" int nsr_last_refined(nsr_ctx* ctx, uintptr_t stream, int64_t n_tiles, int64_t* refined) {
    NSR_REQUIRE(ctx && refined && n_tiles >= 1, "nsr_last_refined: bad arguments");
    NSR_REQUIRE(ctx->refine_dev != nullptr && 3 * (size_t)n_tiles + 1 <= ctx->refine_cap, "nsr_last_refined: no adaptive launch of that size yet");
    NSR_CHECK(cudaSetDevice(ctx->device));
    int32_t c = 0;
    NSR_CHECK(cudaMemcpyAsync(&c, ctx->refine_dev + 3 * n_tiles, sizeof(int32_t), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    NSR_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    *refined = c;
    return 0;
}

namespace {
// lets the current device (ctx->device) reach `other`'s memory directly (NVLink / PCIe peer path); where it
// cannot, the driver stages peer copies through the host
int enable_peer(nsr_ctx* ctx, int other) {
    if (other == ctx->device) return 0;
    int can = 0;
    NSR_CHECK(cudaDeviceCanAccessPeer(&can, ctx->device, other));
    if (can) {
        cudaError_t e = cudaDeviceEnablePeerAccess(other, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) (void)cudaGetLastError();
        else NSR_CHECK(e);
    }
    return 0;
}
}  // namespace

extern "C" int nsr_copy2d(nsr_ctx* ctx, uintptr_t stream, void* dst, int64_t dst_pitch, const void* src,
                          int64_t src_pitch, int64_t width_bytes, int64_t height, int kind) {
    NSR_REQUIRE(ctx != nullptr && dst && src && width_bytes >= 0 && height >= 0 && dst_pitch >= width_bytes &&
                    src_pitch >= width_bytes && kind >= 0 && kind <= 2,
                "nsr_copy2d: bad arguments");
    if (width_bytes == 0 || height == 0) return 0;
    NSR_CHECK(cudaSetDevice(ctx->device));
    cudaMemcpyKind how = kind == 0 ? cudaMemcpyDeviceToHost : cudaMemcpyHostToDevice;
    if (kind == 2) {                               // device to device, either end possibly another GPU
        for (const void* p : {(const void*)dst, src}) {
            cudaPointerAttributes a;
            NSR_CHECK(cudaPointerGetAttributes(&a, p));
            NSR_REQUIRE(a.type == cudaMemoryTypeDevice, "nsr_copy2d: kind 2 takes device memory");
            if (enable_peer(ctx, a.device)) return 1;
        }
        how = cudaMemcpyDefault;                   // unified addressing: the driver routes a copy between two GPUs
    }
    NSR_CHECK(cudaMemcpy2DAsync(dst, (size_t)dst_pitch, src, (size_t)src_pitch, (size_t)width_bytes, (size_t)height,
                                how, (cudaStream_t)stream));
    return 0;
}

extern "C" int nsr_copy_peer(nsr_ctx* ctx, uintptr_t stream, void* dst, const void* src, int src_device, int64_t nbytes) {
    NSR_REQUIRE(ctx != nullptr && dst && src && nbytes >= 0 && src_device >= 0, "nsr_copy_peer: bad arguments");
    if (nbytes == 0) return 0;
    NSR_CHECK(cudaSetDevice(ctx->device));
    if (enable_peer(ctx, src_device)) return 1;
    NSR_CHECK(cudaMemcpyPeerAsync(dst, ctx->device, src, src_device, (size_t)nbytes, (cudaStream_t)stream));
    return 0;
}

namespace {
__global__ void pvalue_kernel(const double* __restrict__ r2, const double* __restrict__ a, int64_t row_len,
                              int64_t count, double* __restrict__ P) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const NsrPvalParams p = nsr_pval_params(a[i / row_len]);
    P[i] = nsr_pvalue_r2(r2[i], p);
}
}  // namespace

extern "C" int nsr_pvalue(nsr_ctx* ctx, uintptr_t stream, const double* r2, const double* a, int64_t row_len,
                          int64_t count, double* P) {
    NSR_REQUIRE(ctx != nullptr && r2 && a && P && row_len > 0 && count >= 0, "nsr_pvalue: bad arguments");
    if (count == 0) return 0;
    NSR_CHECK(cudaSetDevice(ctx->device));
    pvalue_kernel<<<(unsigned)((count + 127) / 128), 128, 0, (cudaStream_t)stream>>>(r2, a, row_len, count, P);
    NSR_CHECK(cudaGetLastError());
    return 0;
}
