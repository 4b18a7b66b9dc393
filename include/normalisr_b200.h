/* normalisr_b200 -- C ABI of the B200-native association-testing hot path.
 *
 * The reference (lingfeiwang/normalisr v1.0.0) is pure Python and has no FFI; these
 * entry points are what a ctypes binding for its hot path binds instead of the numpy /
 * scipy calls cited per function (paths relative to the reference tree).  The Python
 * side that mirrors the reference's functional API (normalisr_b200/association.py)
 * calls exactly these; INTEGRATION.md shows the stub a maintainer would add upstream.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless named host_*; matrices are row-major
 *     with rows = variables (genes / groupings) and columns = cells, like the reference;
 *   - `stream` is a cudaStream_t passed as an integer (0 = legacy default stream); calls
 *     are asynchronous with respect to the host unless stated otherwise;
 *   - every function returns 0 on success, non-zero on error, and nsr_last_error()
 *     then returns a message (thread-local);
 *   - a context is bound to one device and must not be used from two threads at once.
 */
#ifndef NORMALISR_B200_H
#define NORMALISR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nsr_ctx nsr_ctx;

#define NSR_VERSION 100          /* 0.1.0 */
#define NSR_TILE 128             /* output tiles are NSR_TILE x NSR_TILE            */
#define NSR_KBLOCK 128           /* cells are padded to a multiple of this          */
#define NSR_MAX_SLICES 4
#define NSR_MAX_RANK 64          /* covariate rank handled by the projection kernels */
#define NSR_MAX_SPLITS 64        /* cell splits of the projection kernels (depends on n only) */
#define NSR_MAX_SEGMENTS 10      /* column segments of one nsr_contract_segments launch */
#define NSR_TOPK_MAX 2048        /* largest k of nsr_topk_strip / nsr_topk_finish */
#define NSR_TOPK_MAX_PARTS 16    /* partial selections one nsr_topk_merge launch merges */

/* contraction modes */
#define NSR_MODE_COEX 0   /* A == B, symmetric: both triangles written, diagonal = 0,
                             out2 = dot = sum(res_i res_j)/n   (association.py:1036-1057) */
#define NSR_MODE_DE 1     /* rectangular: out2 = gamma = dot / var_x (association.py:234)  */
#define NSR_MODE_RAW 2    /* rectangular: out2 = sum(res_i res_j) (Gram tile, prod1,
                             association.py:393-418); P is not written                    */
#define NSR_MODE_COEX_UPPER 3 /* like COEX but only the listed tiles are written (no mirrored
                             copy): a rank that owns a strip of tile rows produces the upper
                             triangle of its strip; the full matrix is U + U^T            */
#define NSR_MODE_COEX_RECT 4 /* rectangular block of a co-expression matrix between two DISJOINT
                             gene blocks A (rows) and B (columns): out2 = dot like COEX, no diagonal
                             rule, no mirrored copy.  The multi-GPU path computes the off-diagonal
                             block pairs with it while the planes of later blocks are in flight  */
/* contraction engines */
#define NSR_ENGINE_UMMA 0 /* tcgen05 int8 tensor-core kernel (the product path)           */
#define NSR_ENGINE_SIMT 1 /* dp4a CUDA-core kernel, bit-identical integer sums; used by the
                             tests to cross-check the tensor-core kernel on device         */

int nsr_version(void);
const char* nsr_last_error(void);

int nsr_ctx_create(int device, nsr_ctx** ctx);
int nsr_ctx_destroy(nsr_ctx* ctx);

/* Number of int8 bytes one slice plane of a rows x n matrix occupies, and the padded
 * cell count (multiple of NSR_KBLOCK). */
int64_t nsr_padded_cells(int64_t n);
int nsr_cell_splits(int64_t n);

/* The tile list of the cta_group::2 pair kernel, made from a list of n_tiles (tile_row, tile_col) pairs:
 * entries (row block of CTA 0, row block of CTA 1 or -1, column block), at most n_tiles of them in `out`
 * (3 int32 each); returns their count.  Every tile of the input is covered exactly once, as itself or - with
 * `symmetric` (one operand against itself, tile_row <= tile_col) - as its transpose. */
int64_t nsr_pair_tiles(const int32_t* tiles, int64_t n_tiles, int symmetric, int32_t* out);

/* Residualise `rows` variables against an orthonormal covariate basis and quantise.
 *
 * Replaces association.py:226-233 (dx1 = dx - (dci (dc dx^T))^T dc; var = mean(dx1^2),
 * 0 -> 1).  Qt is the (rank x n) orthonormal basis of the row space of dc that the host
 * derives from the same SVD-with-tolerance rule as inv_rank (association.py:66-80), so
 * X - (X Qt^T) Qt is the same projection.
 *
 * Outputs
 *   var[rows]        mean squared residual, 0 replaced by 1 (reference rule)
 *   coef[rows*rank]  X Qt^T, row-major (needed for alpha when lowmem=False)
 *   slices           int8 [n_slices][rows_alloc][n_pad]: balanced base-256 digits of
 *                    round(z' / quantum[row]), z' = residual after a sign-randomised
 *                    128-point Walsh-Hadamard transform along cells (orthonormal, so
 *                    all inner products are unchanged; it only flattens outliers so
 *                    that a fixed-point row scale loses no precision)
 *   quantum[rows]    z' ~= quantum * integer
 *   energy_max       optional [NSR_MAX_SPLITS][NSR_MAX_SLICES] doubles, zeroed by the caller before
 *                    the first call for an operand: entry (k, a) is raised to the largest
 *                    sum of squared digits of plane a that any row has within cell split k
 *                    (split k = 128-cell blocks [nblk k / ks, nblk (k+1) / ks), nblk = n_pad/128,
 *                    ks = nsr_cell_splits(n)).  With it the caller bounds the contraction's
 *                    int32 partial sums (Cauchy-Schwarz) and picks nsr_contract's k_chunk.
 *                    A row whose sum of squares is not finite (NaN / Inf in X or Qt) sets entry
 *                    (0, 0) to NaN: the caller, who reads the report before contracting, must fail
 *                    like the reference's finite-ness asserts (association.py:252-255).
 * rows_alloc >= rows is the plane pitch in rows; bytes beyond `rows` are not touched.
 */
int nsr_residualize(nsr_ctx* ctx, uintptr_t stream,
                    const double* X, int64_t rows, int64_t n, int64_t ldx,
                    const double* Qt, int rank, int64_t ldq,
                    int n_slices, int8_t* slices, int64_t rows_alloc, int64_t n_pad,
                    double* quantum, double* var, double* coef, double* energy_max);

/* nsr_residualize for rows of SMALL INTEGERS (binary gRNA / condition indicators, the dg of de.de,
 * de.py:4-132): one int8 plane holding the Hadamard mix of the RAW row - sums of +-1 over the row's
 * non-zero cells of a 128-cell block, i.e. small integers, stored exactly (quantum = 1/sqrt(128)).
 * Because every y operand is residualised, sum_k res_x res_y = sum_k x res_y: the raw row can stand in
 * for its residual in every cross product (association.py:234 numerator; prod1 tiles of A dy^T,
 * :963-966), and with an exact x the contraction needs n_slices_b digit products instead of 8
 * (nsr_contract_ab, n_slices_a = 1).  var and coef are those of the RESIDUAL, as in nsr_residualize.
 * status (device int, accumulated with OR): 1 = some mixed value is not an integer of magnitude <= 127
 * (rows are not small integers: use nsr_residualize), 2 = some row is explained by the covariates to
 * more than 3/4 of its raw second moment (the partner's quantisation error would be amplified more than
 * 2x: use nsr_residualize).  The plane is unusable unless *status == 0. */
int nsr_residualize_exact(nsr_ctx* ctx, uintptr_t stream,
                          const double* X, int64_t rows, int64_t n, int64_t ldx,
                          const double* Qt, int rank, int64_t ldq,
                          int8_t* plane, int64_t rows_alloc, int64_t n_pad,
                          double* quantum, double* var, double* coef, double* energy_max, int* status);

/* All-pairs contraction over cells + P-value epilogue for a list of output tiles.
 *
 * Replaces association.py:234-249 (gamma = res_y res_x^T / (n var_x); R2; P =
 * beta.cdf(1-R2, dof/2, 1/2)) and, in NSR_MODE_COEX, the assembly at :1036-1057.
 * A (rows_a) indexes output rows, B (rows_b) output columns.  tiles = n_tiles pairs
 * (tile_row, tile_col) of NSR_TILE-sized blocks, host_tiles is a HOST pointer.
 * dof_a = (n - 1 - rank - dimreduce) / 2.  Sums over cells are exact integer sums
 * (int8 digits, int32 accumulation), combined in float64.  k_chunk = 0 contracts all cells in
 * one pass; k_chunk > 0 (a multiple of NSR_KBLOCK) processes the cells in chunks of that length,
 * keeping the float64 running sum in out2 between chunks - required when the int32 partial sums
 * could overflow (see nsr_residualize `energy`).
 */
int nsr_contract(nsr_ctx* ctx, uintptr_t stream, int engine, int mode,
                 const int8_t* a_slices, int64_t rows_a, int64_t rows_alloc_a,
                 const double* quantum_a, const double* var_a,
                 const int8_t* b_slices, int64_t rows_b, int64_t rows_alloc_b,
                 const double* quantum_b, const double* var_b,
                 int64_t n, int64_t n_pad, int n_slices, int n_products,
                 const int32_t* host_tiles, int64_t n_tiles, double dof_a,
                 double* P, double* out2, int64_t ld, int64_t k_chunk);

/* nsr_contract with different plane counts for the two operands: A with n_slices_a planes, B with
 * n_slices_b.  Besides the symmetric presets of nsr_contract it takes n_slices_a = 1 (an operand from
 * nsr_residualize_exact: one plane of exact small integers) against n_slices_b = 3 / 4 / 1 with
 * n_products = n_slices_b - every digit product is kept, so the sums are exact in the A operand.
 * Replaces the same reference lines as nsr_contract (association.py:234-249; prod1 :393-418 in RAW mode). */
int nsr_contract_ab(nsr_ctx* ctx, uintptr_t stream, int engine, int mode,
                    const int8_t* a_slices, int64_t rows_a, int64_t rows_alloc_a, int n_slices_a,
                    const double* quantum_a, const double* var_a,
                    const int8_t* b_slices, int64_t rows_b, int64_t rows_alloc_b, int n_slices_b,
                    const double* quantum_b, const double* var_b,
                    int64_t n, int64_t n_pad, int n_products,
                    const int32_t* host_tiles, int64_t n_tiles, double dof_a,
                    double* P, double* out2, int64_t ld, int64_t k_chunk);

/* Multi-GPU co-expression: everything one GPU owns under the block-pair schedule in ONE persistent
 * launch.  A = the local gene block (output rows).  Segment s = one block of output columns with its
 * own B operand: the local block itself (diagonal = 1: tiles with tile_row <= tile_col, zero diagonal,
 * like NSR_MODE_COEX_UPPER) or a block pulled from a peer (diagonal = 0, like NSR_MODE_COEX_RECT);
 * B row j of segment s lands in output column col0 + j.  Replaces the thread pool over tiles
 * (parallel.autopooler, parallel.py:12-74, used at association.py:997) for the multi-device case.
 *   ready / ready_value  optional device flag (uint32): the kernel does not read the segment's planes
 *                        or scales before  (int32)(*ready - ready_value) >= 0.  The caller sets it
 *                        with nsr_stream_signal on the stream that copies the block in, so tiles of
 *                        blocks that have arrived are contracted while later blocks are in flight;
 *   done                 optional device counter (uint32): += 8 per finished tile of the segment (one
 *                        per epilogue warp, after its stores are visible system-wide); a copy stream
 *                        can nsr_stream_wait_geq on it and send the segment's columns home while the
 *                        launch continues with the next segment;
 *   mirror_P / mirror_out2 / ld_mirror  optional: the lower triangle.  The reference returns the full
 *                        symmetric matrices to one caller (association.py:1036-1057); with these every
 *                        GPU also writes the transposed copy of what it computes - for the diagonal
 *                        segment into its own rows (mirror_P = P + col0, ld_mirror = ld), for a block
 *                        pair into a (rows_b x rows_a) buffer that is sent home as rows of block b - so
 *                        the matrices are assembled without a pass over the lower triangle on the host.
 * host_tiles: n_tiles triples (segment, tile_row, tile_col), processed in list order (claimed from a
 * global counter), so list segments in the order their blocks arrive.  tcgen05 engine only; the
 * waiting launch occupies every SM, so the flags must be set by work that needs none (copy engines). */
typedef struct nsr_segment {
    const int8_t* b_slices;
    int64_t rows_b;
    int64_t rows_alloc_b;
    const double* quantum_b;
    const double* var_b;
    int64_t col0;
    int32_t diagonal;
    uint32_t ready_value;
    const uint32_t* ready;
    uint32_t* done;
    double* mirror_P;          /* optional transposed copy: the element of A row i and B row j also lands at  */
    double* mirror_out2;       /* mirror_*[j * ld_mirror + i] (both or neither; ld_mirror >= rows_a).  The    */
    int64_t ld_mirror;         /* diagonal segment skips tiles with tile_row == tile_col (already symmetric). */
} nsr_segment;
int nsr_contract_segments(nsr_ctx* ctx, uintptr_t stream,
                          const int8_t* a_slices, int64_t rows_a, int64_t rows_alloc_a,
                          const double* quantum_a, const double* var_a,
                          int64_t n, int64_t n_pad, int n_slices, int n_products,
                          const nsr_segment* segments, int n_segments,
                          const int32_t* host_tiles, int64_t n_tiles, double dof_a,
                          double* P, double* out2, int64_t ld, int64_t k_chunk);
/* Stream-ordered flag operations on a device uint32 (cuStreamWriteValue32 / cuStreamWaitValue32, no
 * kernel): *flag = value once the stream reaches this point / the stream waits until
 * (int32)(*flag - value) >= 0. */
int nsr_stream_signal(nsr_ctx* ctx, uintptr_t stream, uint32_t* flag, uint32_t value);
int nsr_stream_wait_geq(nsr_ctx* ctx, uintptr_t stream, uint32_t* flag, uint32_t value);

/* Covariate basis: the two products with the (nc x n) covariate matrix C that turn `dc` into the
 * orthonormal basis Qt of nsr_residualize.  Replaces np.matmul(dc, dc.T) feeding inv_rank at
 * association.py:899-903: the host factorises the nc x nc Gram matrix G = C C^T (SVD with the
 * reference's tolerance rule, association.py:66-80) and the device applies the resulting small
 * matrix, Q = M C (M: rank x nc, row-major, device).  nc, rank <= NSR_MAX_RANK.  Sums over
 * cells are combined in a fixed order: results do not depend on the launch. */
int nsr_cov_gram(nsr_ctx* ctx, uintptr_t stream, const double* C, int nc, int64_t n, int64_t ldc,
                 double* G);
int nsr_cov_apply(nsr_ctx* ctx, uintptr_t stream, const double* M, int rank, int nc,
                  const double* C, int64_t n, int64_t ldc, double* Q, int64_t ldq);

/* de(single=1) building blocks (association_test_2, association.py:263-390: every grouping x is
 * tested on its own subset of cells S_x = U + T_x; U = cells without any gRNA, T_x = cells that
 * carry only x, association.py:913-916).  All statistics of that test are sums over S_x of
 * products of covariates, x and y, and sum_{S_x} = sum_U + sum_{T_x} with disjoint T_x:
 *   nsr_project_coef  coef = X Q^T (rows x rank) and sumsq[row] = sum_k X^2 for any (rank x n) Q:
 *                     with Q = covariates masked to U it yields every U-part in one pass over dy
 *                     (it is pass A of nsr_residualize: FP64 tensor cores, fixed summation order);
 *   nsr_group_stats   Y (genes x m) holds the non-U columns of dy gathered in group order, C
 *                     (nc1 x m) the covariates (+ a row of ones) gathered alike, goff[n_groups+1]
 *                     (device, int64) the group boundaries:
 *                       out[g][y][j] = sum_{k in g} C[j][k] Y[y][k]  (j < nc1),
 *                       out[g][y][nc1] = sum_{k in g} Y[y][k]^2,   out is [n_groups][genes][nc1+1].
 * The per-(x, y) closed form (pseudo-inverse of the nc x nc Gram matrix of S_x with the reference's
 * rank rule, gamma, R2, d.o.f.) is host-side logic in normalisr_b200/single1.py; P-values come from
 * nsr_pvalue with one `a` per grouping. */
int nsr_project_coef(nsr_ctx* ctx, uintptr_t stream, const double* X, int64_t rows, int64_t n,
                     int64_t ldx, const double* Q, int rank, int64_t ldq, double* coef,
                     double* sumsq);
int nsr_group_stats(nsr_ctx* ctx, uintptr_t stream, const double* Y, int64_t genes, int64_t ldy,
                    const double* C, int nc1, int64_t ldc, const int64_t* goff, int n_groups,
                    double* out);
/* Closed form of association_test_2 (association.py:352-377) for `genes` genes x n_groups groupings,
 * fused with the P-value: cu [genes][nc+1] = nsr_project_coef output for the covariates masked to
 * U (+ the mask), yy_u[genes] = sum_U y^2, st = nsr_group_stats output; per grouping x: ci = C+
 * (nc x nc, pseudo-inverse of the covariate Gram matrix of S_x), cx = sum_{T_x} dc, ccx = C+ cx,
 * ns = |S_x|, vx = var_x, dof = ns - 1 - rank - dimreduce.  Writes P, gamma, vy at
 * [x * ld_out + col0 + gene] and alpha (optional, [..][nc]); *flag |= 1 if an R^2 leaves [0, 1].
 * nc <= 16. */
int nsr_single1_finish(nsr_ctx* ctx, uintptr_t stream, const double* cu, const double* yy_u,
                       const double* st, int64_t genes, int n_groups, int nc, const double* ci,
                       const double* cx, const double* ccx, const double* ns, const double* vx,
                       const double* dof, double* P, double* gamma, double* vy, double* alpha,
                       int64_t ld_out, int64_t col0, int* flag);

/* Variance normalisation, the step upstream of coex / de (norm.normvar / normvar1,
 * src/normalisr/norm.py:131-289): gene x is scaled per cell by s_k = w_k ** wt_x and its own
 * weighted covariates dc * s are projected out of it.  Two streaming passes over dt (genes x n):
 *   nsr_normvar_stats  G_x = sum_k s^2 dc dc^T depends on the gene only through s, so with the
 *                      gene-independent matrix M = [ products c_i c_j (i <= j, row-major), zero rows
 *                      up to 8 T | dc, zero rows up to 16 ] ((8 T + 16) x n, built by the host
 *                      layer, T from nsr_normvar_width) the statistics are two skinny GEMMs over
 *                      cells on the FP64 tensor cores:  stats[x] = { [s^2] M_D^T (8 T columns: the
 *                      upper triangle of G), [s^2 dt] M_C^T (16 columns: b = sum_k s^2 dc dt),
 *                      S1 = sum_k s dt, S2 = sum_k (s dt)^2 };  nsr_normvar_width(nc) = 8 T + 18 is
 *                      the length of one stats row.  Replaces the per-gene np.matmul(dc, dc.T) /
 *                      np.matmul(dc, dt.T) of normvar1 (norm.py:159-163);
 *   nsr_normvar_apply  out = scale[x] * s * (dt - coef[x]^T dc), coef (genes x nc) = G+ b from the
 *                      host layer (pseudo-inverse with the rank rule of inv_rank), scale = the
 *                      keepvar factor (norm.py:251-254) or 1.
 *   nsr_normvar_rhs    the part of the statistics that depends on dt, for up to 16 covariates:
 *                      stats[x] = { b (16 columns: sum_k s^2 dt c for the rows of C16, a (16 x n) matrix:
 *                      the covariates, zero rows up to 16), S1, S2 } - 18 doubles per gene.  The Gram
 *                      matrices G_x depend on the gene only through the scalar wt_x and are smooth in it;
 *                      the host layer interpolates them (normalisr_b200/norm.py: Chebyshev nodes in wt,
 *                      barycentric evaluation), which takes 3/4 of the float64 work out of the pass.
 * logw = log(w) per cell, wt per gene; s = w ** wt = exp(wt * logw), 1 when wt == 0.  nsr_normvar_stats:
 * 1 <= nc <= 12; nsr_normvar_apply: 1 <= nc <= 16. */
int nsr_normvar_width(int nc);
int nsr_normvar_rhs(nsr_ctx* ctx, uintptr_t stream, const double* dt, int64_t genes, int64_t n, int64_t ld,
                    const double* C16, int64_t ldc, const double* logw, const double* wt, double* stats);
int nsr_normvar_stats(nsr_ctx* ctx, uintptr_t stream, const double* dt, int64_t genes, int64_t n,
                      int64_t ld, const double* M, int nc, int64_t ldm, const double* logw,
                      const double* wt, double* stats);
int nsr_normvar_apply(nsr_ctx* ctx, uintptr_t stream, const double* dt, int64_t genes, int64_t n,
                      int64_t ld, const double* dc, int nc, int64_t ldc, const double* logw,
                      const double* wt, const double* coef, const double* scale, double* out,
                      int64_t ldo);

/* de(single=4), association_test_4 (association.py:421-576) without a per-grouping pseudo-inverse.
 *   nsr_gram_f64   G = X X^T - Cx Cx^T in float64: the Gram matrix of the covariate-residualised rows of
 *                  X (rows x n) given Cx = X Qt^T (rows x rank, nsr_residualize's coef output).  Replaces
 *                  the prod1 tiles of A A^T (association.py:393-418, 945-957) for the groupings block.
 *   nsr_de4_solve  from Gxx (nx x nx, row-major, contiguous; DESTROYED: holds its Cholesky factor on
 *                  return), Gxy = Rx Ry^T (nx x ny, from nsr_contract in NSR_MODE_RAW) and yy[y] = sum_k
 *                  res_y^2: K = Gxx^-1 by blocked Cholesky, w = K Gxy (written to w: the full-regression
 *                  coefficients, needed for alpha), and per (x, y) the leave-one-out quantities the
 *                  reference gets from one pseudo-inverse per x (:521-544): dxx = 1/(n K_xx) (0 -> 1,
 *                  :545-547), dxy = w/(n K_xx), dyy = (yy - sum_x Gxy w + w^2/K_xx)/n, gamma = dxy/dxx,
 *                  R2 = dxy^2/(dxx dyy), P = I_{1-R2}((n - 1 - (nx - 1 + rank_c) - dimreduce)/2, 1/2) (:563).
 *                  Outputs P, out2 (gamma, or gamma * dxx when return_dot), vary = dyy (nx x ny, ld_out)
 *                  and varx = dxx (nx).  status (device int, OR-ed): 1 = a Cholesky pivot fell below
 *                  tol * max diag (rank-deficient groupings: outputs are not usable, the host layer takes
 *                  the reference's per-grouping branch), 2 = an R2 left [0, 1 + 1e-8] or a result is not
 *                  finite (the reference's asserts, :557, :565-568). */
int nsr_gram_f64(nsr_ctx* ctx, uintptr_t stream, const double* X, int64_t rows, int64_t n, int64_t ldx,
                 const double* coef, int rank, double* G, int64_t ldg);
/* G = (G + G^T)/2 - Cx Cx^T in place: the same correction for a Gram matrix of RAW rows that was formed
 * exactly on the tensor cores (nsr_contract_ab, NSR_MODE_RAW, on nsr_residualize_exact planes). */
int nsr_gram_correct(nsr_ctx* ctx, uintptr_t stream, double* G, int64_t rows, int64_t ldg, const double* coef,
                     int rank);
int nsr_de4_solve(nsr_ctx* ctx, uintptr_t stream, double* Gxx, int nx, const double* Gxy, int64_t ny,
                  int64_t ld_xy, const double* yy, int64_t n_cells, int rank_c, int dimreduce, double tol,
                  int return_dot, double* P, double* out2, double* vary, int64_t ld_out, double* varx,
                  double* w, int64_t ld_w, int* status);

/* Batched inv_rank (association.py:66-80) for `batch` symmetric positive semi-definite n x n
 * matrices (n <= 16), row-major, contiguous: pinv[m] = pseudo-inverse keeping the eigenvalues
 * >= tol * largest (and > 0), rank[m] = how many were kept.  One warp per matrix, cyclic Jacobi.
 * Replaces the per-gene / per-grouping scipy.linalg.svd calls of normvar1 (norm.py:159-160). */
int nsr_sym_pinv(nsr_ctx* ctx, uintptr_t stream, const double* G, int64_t batch, int n, double tol,
                 double* pinv, int32_t* rank);

/* Adaptive digit-product schedule of nsr_contract, opt-in (tcgen05 engine, one segment, n_slices = 3,
 * n_products = 8, k_chunk = 0, any mode but RAW, n >= option "adaptive_min_cells"; default 0 = off,
 * 8192 or more sensible; an explicit "umma_pair" = 1 takes precedence, see nsr_set_option; pays only when
 * extremely significant pairs are confined to few tiles): every
 * tile first runs 6 products; a tile holding a pair with r^2 n > 64 is recomputed with all 8 by a
 * second launch whose tile list and count stay on the device.  Unrefined pairs carry |dr| ~
 * 1e-6 / sqrt(n) (random sign) from the two dropped weight-5 products, i.e. a relative error of P
 * of at most 8e-6 (1 sigma); refined tiles are bit-identical to the full schedule.  Decisions are
 * per 128 x 128 tile of the global pair grid, so results do not depend on tiling or GPU count.
 * nsr_last_refined: number of tiles the most recent adaptive nsr_contract call of `n_tiles` tiles
 * recomputed (synchronises `stream`; bookkeeping for benchmarks). */
int nsr_last_refined(nsr_ctx* ctx, uintptr_t stream, int64_t n_tiles, int64_t* refined);

/* Bayesian logCPM (lcpm.lcpm, src/normalisr/lcpm.py:21-208): reads is a (genes x n) matrix of
 * non-negative counts (int32 or int64, itemsize 4 / 8), lut[c] = digamma(1 + c) for c = 0 .. lut_len - 1
 * (the reference's table, :96-109, without its constant - digamma(total + 2), which the caller folds into
 * `shift`: it is the same for every entry) and lut_exp[c] = exp(lut[c]).  Without resampling, counts
 * >= lut_len are evaluated directly (recurrence + asymptotic series), so the table need not cover the
 * largest count and no pass is needed to find it: the counts are read twice in all.
 *   nsr_lcpm_scan      out3 (device, 3 x int64) = min, max and total of the counts in one pass (only needed
 *                      with resampling, whose standard-deviation table must cover every count);
 *   nsr_lcpm_colstats  colstats = [3][n]: per cell sum_g exp(value), total reads, number of genes with a
 *                      non-zero count (per-cell normaliser :155-157 and the covariates :193-199 from one
 *                      pass over the counts; without resampling the exponentials are a table gather);
 *                      minmax (device, 2 x int64, optional, initialised by the caller to INT64_MAX /
 *                      INT64_MIN, accumulated): [0] turns negative if any count is (the check :88-89), [1] = largest count;
 *   nsr_lcpm_apply     out[g][k] = value[g][k] - shift[k]  (shift may be NULL).
 * value = lut[reads] or, with posterior resampling (varscale != 0, :134-150), lut[reads] + lut_sd[reads] z
 * with lut_sd[c] = sqrt(varscale (trigamma(1 + c) - trigamma(total + 2))) and z a standard normal
 * deviate per entry: read from `noise` (genes x n, ld_noise; e.g. numpy's own stream for a bit-exact
 * drop-in of the reference) or, noise == NULL, generated by Philox4x32-10 keyed by `seed` with the entry's
 * global index (row0 + g) * n + k as counter (the same in both passes and for any row chunking).
 * lut_sd == NULL: no resampling. */
int nsr_lcpm_scan(nsr_ctx* ctx, uintptr_t stream, const void* reads, int itemsize, int64_t genes, int64_t n,
                  int64_t ld, long long* out3);
int nsr_lcpm_colstats(nsr_ctx* ctx, uintptr_t stream, const void* reads, int itemsize, int64_t genes,
                      int64_t n, int64_t ld, const double* lut, const double* lut_exp, int64_t lut_len,
                      const double* lut_sd, const double* noise, int64_t ld_noise, uint64_t seed, int64_t row0,
                      double* colstats, long long* minmax);
int nsr_lcpm_apply(nsr_ctx* ctx, uintptr_t stream, const void* reads, int itemsize, int64_t genes,
                   int64_t n, int64_t ld, const double* lut, int64_t lut_len, const double* lut_sd,
                   const double* noise, int64_t ld_noise, uint64_t seed, int64_t row0, const double* shift,
                   double* out, int64_t ldo);

/* The same two passes on a CSR count matrix (genes x n, never expanded): row g holds the entries
 * indptr[g] .. indptr[g + 1] - 1 of (indices, values), column indices ascending and unique within a row,
 * values int32 or int64 (itemsize 4 / 8; device arrays; indptr holds absolute offsets, so a block of rows
 * is passed as indptr + first row).  Cells without an entry have count 0.  Arguments and results as
 * nsr_lcpm_colstats / nsr_lcpm_apply, and the same bits: a CTA expands the entries of 64 genes x 256 cells
 * into shared memory (64 KB as int32, 128 KB as int64) and runs the dense kernels' per-cell loop on it.
 * The counts are read once per pass (O(nnz)); n <= INT_MAX.  The min / max / total that resampling needs
 * is nsr_lcpm_scan over the values as a 1 x nnz matrix, with 0 added when some entry is not stored. */
int nsr_lcpm_colstats_csr(nsr_ctx* ctx, uintptr_t stream, const int64_t* indptr, const int32_t* indices,
                          const void* values, int itemsize, int64_t genes, int64_t n, const double* lut,
                          const double* lut_exp, int64_t lut_len, const double* lut_sd, const double* noise,
                          int64_t ld_noise, uint64_t seed, int64_t row0, double* colstats, long long* minmax);
int nsr_lcpm_apply_csr(nsr_ctx* ctx, uintptr_t stream, const int64_t* indptr, const int32_t* indices,
                       const void* values, int itemsize, int64_t genes, int64_t n, const double* lut,
                       int64_t lut_len, const double* lut_sd, const double* noise, int64_t ld_noise,
                       uint64_t seed, int64_t row0, const double* shift, double* out, int64_t ldo);

/* compute_var (norm.compute_var, src/normalisr/norm.py:56-128), column pass: with res = X - coef Qt
 * (the covariate-projection residual, not materialised; coef from nsr_project_coef),
 *   out[k] = sum_g ((res[g][k] - mean[g]) * inv_std[g])^2      (norm.py:103).   rank <= 16. */
int nsr_colvar(nsr_ctx* ctx, uintptr_t stream, const double* X, int64_t genes, int64_t n, int64_t ld,
               const double* Qt, int rank, int64_t ldq, const double* coef, int64_t ldcoef,
               const double* mean, const double* inv_std, double* out);

/* P[i] = I_{1 - r2[i]}(a[i / row_len], 1/2)  -- scipy.stats.beta.cdf(1-r2, a, 0.5),
 * association.py:249, 563.  `a` holds one value per row of row_len entries. */
int nsr_pvalue(nsr_ctx* ctx, uintptr_t stream, const double* r2, const double* a,
               int64_t row_len, int64_t count, double* P);

/* P-value network -> binary network (the consumer of NSR_MODE_COEX output).
 *
 * Replaces binnet.binnet (src/normalisr/binnet.py:134-170), i.e. bh() (:77-131) on every row
 * with its diagonal entry removed, followed by Q <= qcut: net[i][j] = 1 iff the Benjamini-
 * Hochberg Q-value of P[i][j] among row i's off-diagonal entries is <= qcut; diagonal = 0.
 * The booleans are bit-identical to the reference's (same floating-point test p / (c / n0) <= qcut
 * at the BH rank, found without sorting).  P is rows x cols (rows of a possibly larger matrix:
 * the diagonal entry of row i is column i + diag0, outside [0, cols) = none).  stats (device,
 * 2 x uint64, accumulated): [0] += number of edges, [1] += rows holding a value outside [0, 1]
 * or NaN (the reference asserts on those, binnet.py:152-153). */
int nsr_binnet(nsr_ctx* ctx, uintptr_t stream, const double* P, int64_t rows, int64_t cols,
               int64_t ld, int64_t diag0, double qcut, uint8_t* net, int64_t ld_net,
               unsigned long long* stats);

/* First half of the sparse (CSR) network: the row procedure of nsr_binnet (same kernels, same
 * "binnet_keys" choice, same arguments and stats), but instead of the uint8 row it writes, per row i,
 * the threshold thr[i] (double; -1 when the row has no edge) and the edge count count[i] (int64).
 * Entry (i, j) is an edge iff j != i + diag0 and P[i][j] <= thr[i]: exactly the entries nsr_binnet sets. */
int nsr_binnet_count(nsr_ctx* ctx, uintptr_t stream, const double* P, int64_t rows, int64_t cols,
                     int64_t ld, int64_t diag0, double qcut, double* thr, int64_t* count,
                     unsigned long long* stats);

/* Second half: CSR compaction.  One CTA per row re-reads the row and writes the column indices of its
 * edges (by the rule above, given thr from nsr_binnet_count) in ascending order into
 * indices[indptr[i] .. indptr[i+1]), as int32 (index_bytes = 4) or int64 (8).  indptr: rows + 1 int64
 * row pointers (the exclusive prefix sum of count; indptr[0] need not be 0).  With p_out / d_out given
 * (both or neither), the same pass stores P[i][j] and D[i][j] (D: rows x cols, leading dimension ld_d)
 * beside every index.  A row whose number of edges differs from its indptr range writes nothing past
 * that range and adds 1 to *err (device uint64), which the caller turns into an error. */
int nsr_binnet_csr_fill(nsr_ctx* ctx, uintptr_t stream, const double* P, int64_t rows, int64_t cols,
                        int64_t ld, int64_t diag0, const double* thr, const int64_t* indptr,
                        void* indices, int index_bytes, const double* D, int64_t ld_d, double* p_out,
                        double* d_out, unsigned long long* err);

/* Every gene's k strongest co-expression partners without a genes x genes matrix (coextop).  The caller
 * contracts one strip of tile rows [r0, r1) at a time in NSR_MODE_COEX_UPPER into P and D (strip row 0 is
 * gene r0, leading dimension ld >= G) and calls nsr_topk_strip after each.  Either the strips go in increasing
 * order from r0 = 0 and cover [0, G), or the state was set empty by nsr_topk_reset first: then the strips may
 * come in any order and start at any r0, and the state ends up holding, for each row, the top k of the pairs
 * in those strips only (one GPU's share of the strips, for nsr_topk_merge).  Row r >= r0 receives (i, P[i][r], D[i][r]) for r0 <= i < min(r1, r) and, when
 * r0 <= r < r1, (j, P[r][j], D[r][j]) for j > r; only strictly-upper entries (j > i) are read.  Ranking key
 * r2 = dot * dot / (var_i * var_j) in float64 without FMA; order: key descending, then column ascending.
 * state: G x k slots of 32 bytes (key, P, dot as doubles, column as int32, 4 bytes of padding), owned by the
 * caller and left alone between calls; the launch with r0 = 0 initialises it unless it was reset.  var: G residual variances
 * (coex's var).  1 <= k <= min(G - 1, NSR_TOPK_MAX).  One launch, no atomics: the result does not depend on
 * the strip heights. */
int nsr_topk_strip(nsr_ctx* ctx, uintptr_t stream, const double* P, const double* D, int64_t ld, int64_t r0,
                   int64_t r1, const double* var, int64_t G, int k, void* state);

/* After the last strip: the slots of `state` in rank order as idx (G x k int64 column indices), P_k and
 * dot_k (G x k float64), row-major. */
int nsr_topk_finish(nsr_ctx* ctx, uintptr_t stream, const void* state, int64_t G, int k, int64_t* idx,
                    double* P_k, double* dot_k);

/* Set the `rows` x k slots of `state` empty (key -1, column INT_MAX): the start of a selection over a subset
 * of the strips of nsr_topk_strip, in any order. */
int nsr_topk_reset(nsr_ctx* ctx, uintptr_t stream, void* state, int64_t rows, int k);

/* Merge n_parts (1 .. NSR_TOPK_MAX_PARTS) partial selections of the same `rows` rows: parts is a host array of
 * device pointers, each to rows x k slots as nsr_topk_strip leaves them (per row sorted, the filled slots
 * first), where a column reaches a row in at most one part (each GPU selected over different strips).  Per
 * row, the k best filled slots of the union in rank order go to idx, P_k and dot_k (rows x k, the layout of
 * nsr_topk_finish).  A row whose parts hold fewer than k filled slots in all writes nothing and sets *status
 * (device int) to 1; the caller zeroes it first and raises.  One launch, no atomics: a slot's output rank is
 * its position in its part plus the number of slots of every other part that beat it. */
int nsr_topk_merge(nsr_ctx* ctx, uintptr_t stream, const void* const* parts, int n_parts, int64_t rows, int k,
                   int64_t* idx, double* P_k, double* dot_k, int* status);

/* Strided copy on `stream` (cudaMemcpy2DAsync): lets the host layer return finished blocks of
 * P / dot while later tiles are still being computed.  kind: 0 = device to host, 1 = host to
 * device, 2 = device to device (also between two GPUs of the process with peer access: the
 * multi-GPU coexnet gathers complete rows of P with it).  Pitches and width in bytes. */
int nsr_copy2d(nsr_ctx* ctx, uintptr_t stream, void* dst, int64_t dst_pitch, const void* src,
               int64_t src_pitch, int64_t width_bytes, int64_t height, int kind);

/* Host-to-host strided copy by a team of threads (threads <= 0: all cores): the staging step between a caller's
 * ordinary (pageable) arrays and the page-locked ring the copy engines work on, so that plain numpy input and
 * freshly allocated numpy results run the same overlapped pipeline as page-locked buffers (a pageable
 * cudaMemcpy stages through one driver thread at ~3 GB/s and takes the result array's page faults one by one).
 * Replaces nothing in the reference: it is what keeps `normalisr.coex(dt, dc)` (coex.py:4) a drop-in for numpy
 * callers.  Pitches and width in bytes; no CUDA call inside. */
int nsr_host_copy2d(void* dst, int64_t dst_pitch, const void* src, int64_t src_pitch, int64_t width_bytes,
                    int64_t height, int threads);

/* Asynchronous copy of nbytes from device `src_device` into this context's device on `stream` (a stream of
 * the context's device): cudaMemcpyPeerAsync, peer access enabled on first use.  No kernel, no SM: the
 * single-process multi-GPU path (normalisr_b200.parallel.coex_all_devices) pulls the digit planes of the
 * other GPUs' gene blocks with it while the persistent contraction launch is already running. */
int nsr_copy_peer(nsr_ctx* ctx, uintptr_t stream, void* dst, const void* src, int src_device, int64_t nbytes);

/* Text I/O of the command-line layer around the hot path (run.py:10-35), host side: files are mapped and
 * parsed by a pool of threads straight into the caller's buffers (page-locked memory in the Python layer,
 * so a matrix reaches the device with one asynchronous copy).  threads <= 0: all cores.
 *   nsr_tsv_shape / nsr_tsv_read   numpy.loadtxt(f, delimiter) (file_read_tsv, run.py:20-27): data lines
 *                                  (blank lines and '#' comments skipped) x delimiter-separated fields ->
 *                                  out[r * ld + c], float64;
 *   nsr_tsv_write                  numpy.savetxt(f, d, delimiter, fmt='%.<precision>G') (file_write_tsv,
 *                                  run.py:30-35; the reference's fmt_float is '%.8G', run.py:6): same bytes;
 *   nsr_mtx_shape / nsr_mtx_read   scipy.io.mmread of a 'matrix coordinate' file (file_read_coo,
 *                                  run.py:10-17): the stored entries as 0-based triplets (pattern files
 *                                  give 1.0); *symmetric = 0 general / 1 symmetric / 2 skew-symmetric (the
 *                                  caller mirrors the entries, as scipy does). */
int nsr_tsv_shape(const char* path, char delimiter, int64_t* rows, int64_t* cols);
int nsr_tsv_read(const char* path, char delimiter, double* out, int64_t rows, int64_t cols, int64_t ld, int threads);
int nsr_tsv_write(const char* path, char delimiter, const double* data, int64_t rows, int64_t cols, int64_t ld,
                  int precision, int threads);
int nsr_mtx_shape(const char* path, int64_t* rows, int64_t* cols, int64_t* nnz, int* is_integer);
int nsr_mtx_read(const char* path, int64_t nnz, int32_t* row, int32_t* col, double* val, int* symmetric, int threads);

/* Process-wide options, mostly test hooks.  Which kernel nsr_contract runs is decided by the first rule that
 * applies (nsr_contract_route in csrc/contract_route.h):
 *   1. the dp4a engine (NSR_ENGINE_SIMT) runs as asked;
 *   2. the cta_group::2 pair kernel, for one segment with equal plane counts of at least 3, when "umma_pair" is 1,
 *      or when it is -1 and the call is single-segment NSR_MODE_COEX at 3 planes / 8 products without the adaptive
 *      schedule (n < "adaptive_min_cells" or that option 0);
 *   3. the adaptive schedule (see nsr_last_refined), for one segment at 3 planes / 8 products, any mode but RAW,
 *      k_chunk = 0 (or >= n_pad) and n >= "adaptive_min_cells" > 0;
 *   4. the split over the cells, when "split_k" is 1, for one segment in NSR_MODE_DE or NSR_MODE_RAW with fewer
 *      than two waves of tiles (one tile per SM) that would leave more than a quarter of their SM slots idle
 *      (4 tiles < 3 waves x SMs): work items (tile, part of the cells) over all SMs, partial sums added in a
 *      fixed order by a second small kernel.  It needs at least two parts, at least as many as the k_chunk
 *      chunks, and at most 1 GiB of partial-sum slabs; otherwise rule 5;
 *   5. the single-CTA tcgen05 kernel, once per k_chunk chunk of the cells.
 * Options:
 *   "umma_pair"           -1 (default), 0 (never the pair kernel) or 1 (wherever it applies), as above;
 *   "adaptive_min_cells"  0 = off (default), 8192 or more sensible: rule 3;
 *   "split_k"             1 (default) / 0: rule 4;
 *   "umma_dynamic"        1 = tcgen05 kernels claim tiles from a global counter (default), 0 = static round-robin;
 *   "umma_kblock"         64 or 128 cells per pipeline stage of the single-CTA kernel (default 128; 64 whenever
 *                         the two operands have more than 6 planes together);
 *   "umma_stack"          1 = N = 256 MMAs over two stacked B planes in the single-CTA kernel at 128-cell stages
 *                         (default), 0 = one N = 128 MMA per digit product;
 *   "epi_warps"           8 (default) or 16 epilogue warps in the single-CTA kernel;
 *   "epi_sleep_ns"        back-off in ns of the tcgen05 epilogue warps while they wait for a tile (default 500,
 *                         0 = spin);
 *   "hadamard"            1 = Walsh-Hadamard mixing in nsr_residualize (default), 0 = off;
 *   "prefetch"            1 = L2 prefetch of the next cell block in the residual pass; measured neutral, default 0;
 *   "binnet_keys"         1 = nsr_binnet and nsr_binnet_count keep rows as 2-byte bin keys, four rows per SM
 *                         (default); 0 = the 8-byte row staged with one bulk copy. */
int nsr_set_option(const char* name, int value);

/* Debug / test helper: reconstruct z' (float64, rows x n_pad) from slices and quantum. */
int nsr_unslice(nsr_ctx* ctx, uintptr_t stream, const int8_t* slices, int64_t rows,
                int64_t rows_alloc, int64_t n_pad, int n_slices, const double* quantum,
                double* out);

#ifdef __cplusplus
}
#endif
#endif
