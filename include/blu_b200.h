/* blu_b200.h -- C ABI of the B200-native BLU hot path (libblu_b200.so).
 *
 * Drop-in boundary for the public surface of the rwl/blu crate (paths relative to
 * /root/reference/src).  Every entry point takes plain host pointers and sizes; the
 * library owns all device memory, does the H2D/D2H copies and launches hand-written
 * sm_100a kernels.  There is no CPU fallback: without a CUDA device every call
 * returns BLU_ERROR_CUDA.
 *
 * Index type: the reference uses usize/LUInt = 64-bit (lib.rs:32); so does this ABI.
 * Return codes: the Rust `Status` enum (lib.rs:39-64) has no discriminants; BASICLU's
 * numbering is used.  Ok(()) == BLU_OK.  WarningSingularMatrix is returned like an
 * error by the crate but the factorization IS valid (factorize.rs:115-119,176-178).
 * `Reallocate` never escapes the object API (blu.rs:95-118 loops on it); it does not
 * escape this ABI either -- the library grows device memory and re-runs.
 */
#ifndef BLU_B200_H
#define BLU_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
    BLU_OK = 0,
    BLU_REALLOCATE = 1,                 /* lib.rs:41  (internal, never returned) */
    BLU_WARNING_SINGULAR_MATRIX = 2,    /* lib.rs:44 */
    BLU_ERROR_INVALID_CALL = -2,        /* lib.rs:48 */
    BLU_ERROR_ARGUMENT_MISSING = -3,    /* lib.rs:51 */
    BLU_ERROR_INVALID_ARGUMENT = -4,    /* lib.rs:54 */
    BLU_ERROR_MAXIMUM_UPDATES = -5,     /* lib.rs:58 */
    BLU_ERROR_SINGULAR_UPDATE = -6,     /* lib.rs:63 */
    BLU_ERROR_INTERNAL = -100,          /* a device-side invariant (a reference assert!) failed */
    BLU_ERROR_CUDA = -101,              /* no device / CUDA runtime error */
    BLU_ERROR_OUT_OF_MEMORY = -102
};

/* parameter / info selectors for blu_set_param, blu_get_param, blu_get_info.
 * Parameters: pub fields of `LU` (lu/lu.rs:10-66) and BLU.realloc_factor (blu.rs:19).
 * Info: the getters of lu/lu.rs:399-683. */
enum {
    BLU_P_DROPTOL = 0, BLU_P_ABSTOL, BLU_P_RELTOL, BLU_P_NZBIAS, BLU_P_MAXSEARCH, BLU_P_PAD,
    BLU_P_STRETCH, BLU_P_COMPRESS_THRES, BLU_P_SPARSE_THRES, BLU_P_SEARCH_ROWS,
    BLU_P_REALLOC_FACTOR, BLU_P_L_MEM, BLU_P_U_MEM, BLU_P_W_MEM,
    BLU_P_THREADS_PER_BASIS,            /* CTA size of the factorization kernel (32..1024) */
    BLU_P_NORMS,                        /* 1 (default): factorize also runs condest x2 + residual_test as factorize.rs:121-147 does; 0: skip them (their getters then read 0) */
    BLU_P_DENSE_K,                      /* order at which the active submatrix switches to the dense-tail representation (multiple of 32, <= 256; 0 = never; default: the largest order whose values fit in shared memory, 160 on B200).  Results do not depend on it. */
    BLU_P_TAIL_THREADS,                 /* CTA size of the dense-tail launch of a split batch factorization (default 512) */
    BLU_P_SPLIT_MIN,                    /* batches of more bases than this run as three launches: sparse head, dense tail with one CTA per SM, build_factors (default 0: always, when the dense tail is shared-memory resident -- a single launch sized for 200+ KB of shared memory would leave the sparse head without L1) */
    BLU_P_TREE_MIN,                     /* bumps with more active columns than this find their Markowitz candidates through a min-tree over the column keys instead of a scan (default 4096; needs maxsearch <= 4) */
    BLU_P_DENSE_K_BIG,                  /* two-stage dense tail: the active submatrix turns dense already at this order (multiple of 32, <= 256, > BLU_P_DENSE_K) with its values in HBM/L2, and moves into shared memory when it has shrunk to BLU_P_DENSE_K (0 = one stage; default 256 for batches when BLU_P_DENSE_K is shared-memory resident).  Results do not depend on it. */
    BLU_I_M = 100, BLU_I_RANK, BLU_I_BUMP_SIZE, BLU_I_BUMP_NZ, BLU_I_MATRIX_NZ, BLU_I_L_NZ,
    BLU_I_U_NZ, BLU_I_R_NZ, BLU_I_NSEARCH_PIVOT, BLU_I_NEXPAND, BLU_I_NGARBAGE,
    BLU_I_FACTOR_FLOPS, BLU_I_MIN_PIVOT, BLU_I_MAX_PIVOT, BLU_I_MAX_ETA, BLU_I_NUPDATE,
    BLU_I_NFORREST, BLU_I_NFACTORIZE, BLU_I_NUPDATE_TOTAL, BLU_I_NFORREST_TOTAL,
    BLU_I_NSYMPERM_TOTAL, BLU_I_L_FLOPS, BLU_I_U_FLOPS, BLU_I_R_FLOPS, BLU_I_CONDEST_L,
    BLU_I_CONDEST_U, BLU_I_NORM_L, BLU_I_NORM_U, BLU_I_NORMEST_L_INV, BLU_I_NORMEST_U_INV,
    BLU_I_ONENORM, BLU_I_INFNORM, BLU_I_RESIDUAL_TEST, BLU_I_PIVOT_ERROR, BLU_I_UPDATE_COST,
    BLU_I_TIME_FACTORIZE, BLU_I_TIME_SOLVE, BLU_I_TIME_UPDATE, BLU_I_ELIM_BYTES, BLU_I_NELIM_DIV,
    BLU_I_PIVOTLEN, BLU_I_RANKDEF, BLU_I_INTERNAL_ERROR, BLU_I_STATUS, BLU_I_NREALLOC,
    BLU_I_ELIM_BYTES_HEAD,              /* part of BLU_I_ELIM_BYTES done by the head launch of a split batch factorization */
    BLU_I_NRUNS,                        /* factorization passes started on this basis since creation (a Reallocate re-run counts) */
    BLU_I_ADDMEM_L, BLU_I_ADDMEM_U, BLU_I_ADDMEM_W, /* lu.rs:308-314: entries missing in L / U / W when the last call answered Reallocate */
    BLU_I_T_PHASE0 = 200, /* +0..15: SM cycles per phase of the factorization kernel (diagnostic) */
    BLU_I_N_KIND0 = 220,  /* +0..4: pivots taken by singleton-row / singleton-col / doubleton / small / any; +5: of those, steps taken in the dense tail; +6: entries into it */
    BLU_I_NORMS_CYC0 = 230 /* +0..3: SM cycles of condest(L), condest(U), residual forward, residual transposed (diagnostic) */
};

/* ------------------------------------------------------------------ */
/* object API: struct BLU, blu.rs:9-334                                 */
/* ------------------------------------------------------------------ */
typedef struct blu_b200 blu_t;

/* BLU::new(m, b_nz), blu.rs:61-70.  device < 0: current device.
 * 1 <= m < 2^23 (BLU_ERROR_INVALID_ARGUMENT otherwise); each of the L, U and W stores holds fewer than 2^30
 * (W: 2^29) entries per basis, beyond which growing them reports BLU_ERROR_OUT_OF_MEMORY. */
int blu_create(blu_t **out, int64_t m, int64_t b_nz, int device);
void blu_destroy(blu_t *o);

int blu_set_param(blu_t *o, int what, double value);
double blu_get_param(const blu_t *o, int what);
double blu_get_info(blu_t *o, int what);

/* BLU::factorize, blu.rs:95-118 -> factorize(), factorize.rs:34.  Column j of B is
 * b_i/b_x[b_begin[j] .. b_end[j]); pass (colptr, colptr+1) for CSC. */
int blu_factorize(blu_t *o, const int64_t *b_begin, const int64_t *b_end,
                  const int64_t *b_i, const double *b_x);

/* factorize() of the crate's FREE-FUNCTION surface (lib.rs:11-19, factorize.rs:34-119), where Reallocate escapes:
 * returns BLU_REALLOCATE with BLU_I_ADDMEM_L/U/W set; the caller grows the stores (blu_set_param with
 * BLU_P_L_MEM / BLU_P_U_MEM / BLU_P_W_MEM -- lu_realloc_obj, blu.rs:345-377) and calls again with c0ntinue != 0.
 * c0ntinue != 0 without a pending Reallocate: BLU_ERROR_INVALID_CALL (factorize.rs:102-105). */
int blu_factorize_c0ntinue(blu_t *o, const int64_t *b_begin, const int64_t *b_end,
                           const int64_t *b_i, const double *b_x, int c0ntinue);

/* BLU::get_factors, blu.rs:139-160 -> get_factors.rs:48.  Every output may be NULL. */
int blu_get_factors(blu_t *o, int64_t *rowperm, int64_t *colperm,
                    int64_t *l_colptr, int64_t *l_rowidx, double *l_value,
                    int64_t *u_colptr, int64_t *u_rowidx, double *u_value);

/* BLU::solve_dense, blu.rs:182-184 -> solve_dense.rs:24.  trans 't'/'T' = transposed. */
int blu_solve_dense(blu_t *o, const double *rhs, double *lhs, char trans);

/* Many right-hand sides against one factorization (SURVEY.md 8f, N4): rhs and lhs hold nrhs vectors of
 * length m back to back; the result is bit-identical to nrhs calls of blu_solve_dense.  This is
 * blu_batch_solve_dense_multi on the object's one basis: the right-hand sides run in chunks of at most
 * BLU_B200_SOLVE_UNITS (read from the environment when the object is created, default 8192), and the device
 * scratch is bounded by that chunk, 24*m bytes per right-hand side, not by nrhs. */
int blu_solve_dense_multi(blu_t *o, int64_t nrhs, const double *rhs, double *lhs, char trans);

/* Many sparse right-hand sides against one factorization: right-hand side r is
 * irhs/xrhs[rhs_begin[r] .. rhs_begin[r+1]).  For every r: nzlhs[r] (or -1 and status[r], which may be NULL),
 * the pattern ilhs[r*m .. r*m+nzlhs[r]) in the order blu_solve_sparse returns it, and the VALUES of those
 * entries compacted in xlhs[r*m + n].  The rest of row r, and the rows of a rejected right-hand side, are
 * unspecified: the rows of m come back whole, which is the faster copy for the dense solutions these calls often
 * have.  Bit-identical to nrhs calls of blu_solve_sparse; returns the first non-OK status.  An offset of rhs_begin
 * outside [0, rhs_begin[nrhs]]: BLU_ERROR_INVALID_ARGUMENT, nothing runs.  This is blu_batch_solve_sparse with every
 * unit on the object's one basis: at most BLU_B200_SOLVE_UNITS right-hand sides per launch, so the device scratch is
 * bounded by that chunk, not by nrhs. */
int blu_solve_sparse_multi(blu_t *o, int64_t nrhs, const int64_t *rhs_begin, const int64_t *irhs, const double *xrhs,
                           int64_t *nzlhs, int64_t *ilhs, double *xlhs, int *status, char trans);

/* BLU::solve_sparse, blu.rs:207-230 -> solve_sparse.rs:35.  The result is returned like
 * BLU.lhs / ilhs / nzlhs: lhs[m] scattered (zero elsewhere), ilhs[0..*nzlhs) its pattern. */
int blu_solve_sparse(blu_t *o, int64_t nzrhs, const int64_t *irhs, const double *xrhs,
                     int64_t *nzlhs, int64_t *ilhs, double *lhs, char trans);

/* BLU::solve_for_update, blu.rs:257-294 -> solve_for_update.rs:72.  xrhs may be NULL for
 * trans; nzlhs/ilhs/lhs may all be NULL when the solution is not wanted. */
int blu_solve_for_update(blu_t *o, int64_t nzrhs, const int64_t *irhs, const double *xrhs,
                         int64_t *nzlhs, int64_t *ilhs, double *lhs, char trans);

/* BLU::update, blu.rs:319-334 -> update.rs:49 */
int blu_update(blu_t *o, double xtbl);

/* BLU: Clone.  *out becomes a new object on src's device that holds what src holds: the factors and the update history,
 * a pending solve_for_update of either direction, every getter (the host-side BLU_I_TIME_* and BLU_I_NREALLOC too),
 * every parameter, the L/U/W capacities exactly, the resident B and a pending blu_factorize_c0ntinue Reallocate.  From
 * then on the clone behaves bit for bit as src would under the same calls, and src does not change (its launch count
 * grows by the three launches that write its image).  A never-factorized src gives a never-factorized clone.  The
 * clone goes through an image of src in device scratch (blu_save_dev's bytes), so it needs that much device memory
 * for the duration of the call.  src from blu_batch_create, or a NULL argument: BLU_ERROR_INVALID_ARGUMENT.  A clone
 * on another device: restore an image there. */
int blu_clone(blu_t **out, blu_t *src);

/* blu_batch_save / blu_batch_restore (below) for an object: the same image format, so an image of an object restores
 * into any batch slot of the same m and an image of a batch slot into any object of the same m.
 * blu_save: the object's image into buf (cap bytes, 16-byte aligned), its size into *bytes; buf == NULL: a size query.
 * Save changes nothing.  A cap smaller than the image: BLU_ERROR_INVALID_ARGUMENT after *bytes is written.
 * blu_restore: the object becomes the basis of the image in buf (cap bytes readable), with the batch call's checks and
 * rejections (BLU_ERROR_INVALID_ARGUMENT, nothing changes).  Then:
 * - its L, U and W stores take the image's capacities exactly (the object's own stores are reallocated; the sorted
 *   row-wise U with the U store); if the image's row-wise B needs more room than the object's, that room grows;
 * - a fresh basis (nupdate 0, status OK or BLU_WARNING_SINGULAR_MATRIX) gets the sorted row-wise U a factorization
 *   builds, so that it solves as after that factorization;
 * - the resident B becomes the image's columns;
 * - parameters, BLU_I_TIME_* and BLU_I_NREALLOC stay the object's own (an image carries none of them), and a pending
 *   blu_factorize_c0ntinue Reallocate is dropped (blu_factorize_c0ntinue with c0ntinue != 0 answers
 *   BLU_ERROR_INVALID_CALL).
 * The _dev variants take a buffer in device memory on the object's device; their host traffic is that of the batch
 * calls with n = 1.  An object from blu_batch_create: BLU_ERROR_INVALID_ARGUMENT. */
int blu_save(blu_t *o, void *buf, int64_t cap, int64_t *bytes);
int blu_restore(blu_t *o, const void *buf, int64_t cap);
int blu_save_dev(blu_t *o, void *d_buf, int64_t cap, int64_t *bytes);
int blu_restore_dev(blu_t *o, const void *d_buf, int64_t cap);

/* ------------------------------------------------------------------ */
/* batch API: many independent bases of one dimension on one GPU       */
/* (what "one BLU instance per core" is on the CPU; SURVEY.md 8e)      */
/* ------------------------------------------------------------------ */
typedef struct blu_b200 blu_batch_t;

/* nmat objects of dimension m whose B has at most bnz_cap entries each. */
int blu_batch_create(blu_batch_t **out, int64_t nmat, int64_t m, int64_t bnz_cap, int device);
void blu_batch_destroy(blu_batch_t *b);

/* Column j of basis k is b_i/b_x[b_begin[k*m+j] .. b_end[k*m+j]); b_i/b_x hold `bnz_total`
 * entries in all.  status[k] (may be NULL) receives the per-basis code; the return value
 * is BLU_OK unless a call-level error occurred. */
int blu_batch_factorize(blu_batch_t *b, const int64_t *b_begin, const int64_t *b_end,
                        const int64_t *b_i, const double *b_x, int64_t bnz_total, int *status);
/* rhs, lhs: nmat*m, basis k at offset k*m */
int blu_batch_solve_dense(blu_batch_t *b, const double *rhs, double *lhs, char trans, int *status);
double blu_batch_get_info(blu_batch_t *b, int64_t k, int what);
int blu_batch_get_factors(blu_batch_t *b, int64_t k, int64_t *rowperm, int64_t *colperm,
                          int64_t *l_colptr, int64_t *l_rowidx, double *l_value,
                          int64_t *u_colptr, int64_t *u_rowidx, double *u_value);

/* One basis change on every basis of the batch at once (many LPs advancing together): solve_for_update
 * (blu.rs:257) and update (blu.rs:319) with one warp per basis.  Right-hand side of basis k:
 * irhs/xrhs[rhs_begin[k] .. rhs_begin[k+1]); for trans 't'/'T' one index (the leaving column), xrhs may be
 * NULL.  With want_solution: nzlhs[k], the pattern ilhs[k*m ..] and the values of those entries compacted
 * in xlhs[k*m + n].  status[k] carries the per-basis code (may be NULL); the return value is the first
 * non-OK one.  Reallocate never escapes (blu.rs:268-291, 319-334): the stores of the whole batch are grown,
 * content kept, and the bases that asked run again. */
int blu_batch_solve_for_update(blu_batch_t *b, const int64_t *rhs_begin, const int64_t *irhs, const double *xrhs,
                               int want_solution, int64_t *nzlhs, int64_t *ilhs, double *xlhs, int *status, char trans);
int blu_batch_update(blu_batch_t *b, const double *xtbl, int *status);

/* solve_sparse (solve_sparse.rs:35-73) for many right-hand sides on every basis of the batch, one warp per
 * (basis, right-hand side).  Basis k owns units unit_begin[k] .. unit_begin[k+1) (unit_begin has nmat+1 entries,
 * unit_begin[0] == 0, non-decreasing; a basis may own none).  Unit u solves with
 * irhs/xrhs[rhs_begin[u] .. rhs_begin[u+1]) and returns, exactly as blu_solve_sparse_multi does:
 * nzlhs[u] (-1 on error), the pattern ilhs[u*m ..] in blu_solve_sparse's order, the values compacted in
 * xlhs[u*m + n], status[u] (may be NULL).  Bit-identical to calling solve_sparse for the units of basis k in
 * order.  The return value is the first non-OK unit status.  A malformed unit_begin or rhs_begin, or a missing
 * array: BLU_ERROR_INVALID_ARGUMENT, nothing runs.  A unit's own argument errors (an index >= m, more than m
 * entries, a basis never factorized) go to its status word; the other units carry on.  A pending
 * solve_for_update / update sequence is not disturbed.  At most BLU_B200_SOLVE_UNITS units (read from the
 * environment at batch creation, default 8192) are in flight per launch; their scratch takes 60*m bytes each. */
int blu_batch_solve_sparse(blu_batch_t *b, const int64_t *unit_begin, const int64_t *rhs_begin,
                           const int64_t *irhs, const double *xrhs,
                           int64_t *nzlhs, int64_t *ilhs, double *xlhs, int *status, char trans);

/* solve_dense (solve_dense.rs:24) for nrhs right-hand sides on every basis: the right-hand side r of basis k is
 * rhs[(k*nrhs + r)*m ..], its solution lhs[(k*nrhs + r)*m ..], status[k*nrhs + r] (may be NULL).  Bit-identical to
 * nrhs blu_solve_dense calls on each basis.  Returns the first non-OK status; nrhs < 0: BLU_ERROR_INVALID_ARGUMENT. */
int blu_batch_solve_dense_multi(blu_batch_t *b, int64_t nrhs, const double *rhs, double *lhs, char trans, int *status);

/* maxvolume (maxvolume.rs:64-224) on every basis of the batch, all bases in lockstep over the pool columns.
 * Basis k has its own pool of ncol columns: column j is a_i/a_x[a_begin[k*ncol+j] .. a_end[k*ncol+j]) (anz_total
 * entries in all, the same convention as blu_batch_factorize).  basis[k*m .. +m) and isbasic[k*ncol .. +ncol) are
 * updated in place; nupdate[k] and status[k] (either may be NULL) receive what maxvolume returns for basis k: a
 * basis stops at its first non-OK status, the others carry on.  The return value is the first non-OK status.
 * volumetol < 1, a basis entry outside [0, ncol) or a pool offset outside [0, anz_total]:
 * BLU_ERROR_INVALID_ARGUMENT, nothing runs.  Reallocate never escapes.  Afterwards every basis is in the state
 * maxvolume leaves it in (getters, solves and updates continue from there), and the resident B of the batch is
 * the basis' columns of the pool. */
int blu_batch_maxvolume(blu_batch_t *b, int64_t ncol, const int64_t *a_begin, const int64_t *a_end,
                        const int64_t *a_i, const double *a_x, int64_t anz_total,
                        int64_t *basis, int64_t *isbasic, double volumetol, int64_t *nupdate, int *status);

/* The batch calls on a subset of the bases, so that each basis keeps its own schedule: the bases sel[0..nsel)
 * (distinct, in [0, nmat), any order) run, every other basis keeps its factors, its update history, a pending
 * solve_for_update, its getters and its status.  Each selected basis ends exactly as its own BLU object would after
 * the calls it was selected in.  status[r] (may be NULL) receives the code of basis sel[r]; the return value is the
 * first non-OK one.  nsel < 0 or > nmat, an index outside [0, nmat), a duplicate index, a missing array when
 * nsel > 0, a malformed rhs_begin, a b_begin/b_end value outside [0, bnz_total], or an object from blu_create:
 * BLU_ERROR_INVALID_ARGUMENT, nothing runs.  nsel == 0: BLU_OK, nothing runs.  A basis' own errors (a column with
 * b_end < b_begin, a row index >= m, an update without both solves, ...) go to its status word, the other selected
 * bases carry on.  Reallocate never escapes.
 *
 * blu_batch_factorize_subset: column j of the r-th selected basis is b_i/b_x[b_begin[r*m+j] .. b_end[r*m+j]).
 * Afterwards the resident B (blu_batch_factorize_resident) holds, for every basis, the B it was last factorized
 * from, in library-owned memory; a graph captured before (blu_batch_graph_capture) is dropped, and
 * blu_batch_graph_launch answers BLU_ERROR_INVALID_CALL until the next capture. */
int blu_batch_factorize_subset(blu_batch_t *b, int64_t nsel, const int64_t *sel,
                               const int64_t *b_begin, const int64_t *b_end,
                               const int64_t *b_i, const double *b_x, int64_t bnz_total, int *status);
/* blu_batch_solve_for_update for the selected bases only; right-hand side r is irhs/xrhs[rhs_begin[r] .. rhs_begin[r+1]),
 * outputs compacted by r: nzlhs[r], ilhs[r*m ..], xlhs[r*m + n], status[r]. */
int blu_batch_solve_for_update_subset(blu_batch_t *b, int64_t nsel, const int64_t *sel, const int64_t *rhs_begin,
                                      const int64_t *irhs, const double *xrhs, int want_solution,
                                      int64_t *nzlhs, int64_t *ilhs, double *xlhs, int *status, char trans);
/* blu_batch_update for the selected bases only, basis sel[r] with xtbl[r] */
int blu_batch_update_subset(blu_batch_t *b, int64_t nsel, const int64_t *sel, const double *xtbl, int *status);

/* Device-resident variants for throughput measurement: upload once, then time kernels only. */
int blu_batch_upload(blu_batch_t *b, const int64_t *b_begin, const int64_t *b_end,
                     const int64_t *b_i, const double *b_x, int64_t bnz_total, const double *rhs);
int blu_batch_factorize_resident(blu_batch_t *b);
int blu_batch_solve_dense_resident(blu_batch_t *b, char trans);
int blu_batch_download(blu_batch_t *b, double *lhs, int *status);
/* SURVEY.md 8(f) N4.  Caller-owned DEVICE buffers (same layout as the host variants): no staging, no copies;
 * B must stay valid and unchanged until the next factorization of the batch.  d_status (nmat ints on the device)
 * may be NULL. */
int blu_batch_factorize_dev(blu_batch_t *b, const int64_t *d_b_begin, const int64_t *d_b_end,
                            const int64_t *d_b_i, const double *d_b_x, int64_t bnz_total);
int blu_batch_solve_dense_dev(blu_batch_t *b, const double *d_rhs, double *d_lhs, char trans, int *d_status);
/* The basis-change step of a batch on caller-owned DEVICE buffers, for a driver that keeps its state on the GPU.
 * Every array argument is device memory on the batch's device, in the layout of the host variant, except that the
 * per-basis arrays of a masked call keep the per-basis layout (index k) and are not compacted by selection.
 * d_run: NULL = every basis runs; otherwise nmat ints on the device, nonzero = this basis runs.
 *
 * - Same results: every basis that runs ends exactly as the host variant leaves it, bit for bit (statuses, nzlhs, the
 *   order of ilhs, the values, every getter including l_flops / u_flops / r_flops / update_cost / nupdate, later solves
 *   and get_factors).  A masked call matches the *_subset call whose sel is the set bits of d_run, in index order; with
 *   d_run == NULL the whole-batch call.
 * - A basis that does not run does not move: its state, a pending solve_for_update pair, its getters, and its entries
 *   of d_status, d_nzlhs, d_ilhs, d_xlhs, d_xtbl are neither read nor written.  An all-zero mask changes nothing and
 *   returns BLU_OK.
 * - The arguments the host cannot see are checked on the device before anything runs: rhs_begin offsets of running
 *   bases (and rhs_begin[nmat] >= 0), B offsets of running bases within [0, bnz_total], unit_begin[0] == 0, unit_begin
 *   non-decreasing, unit_begin[nmat] == nunits, unit rhs_begin offsets within [0, rhs_begin[nunits]], a non-empty
 *   right-hand side set without its index (or value) array.  A violation: BLU_ERROR_INVALID_ARGUMENT, no state change, no
 *   output written.  A missing pointer, nrhs < 0 or nunits < 0 is rejected on the host the same way.  A basis' or unit's
 *   own errors go to its status word, as in the host variants.
 * - The return value is the first non-OK status among the running bases or units in index order, found on the device.
 * - Reallocate never escapes: the stores are grown and the bases that asked run again (at most 40 attempts); only then
 *   does the host read per-basis data (the info block).
 * - Host traffic: solve_for_update_dev, update_dev, solve_sparse_dev and solve_dense_multi_dev copy nothing between host
 *   and device whose size grows with nmat, nunits, m or the right-hand sides: per launch attempt (and once for the
 *   argument check) the host reads a summary of DEV_SUM_N = 5 words from pinned memory.  solve_sparse_dev runs its chunks
 *   of BLU_B200_SOLVE_UNITS units back to back and writes the solutions to d_ilhs[u*m ..] / d_xlhs[u*m ..].
 * - The calls queue on the batch's stream (blu_batch_set_stream applies) and return when their outputs are complete.
 *   last_kernel_ms and launch_count account for them as for the host variants.
 * - d_status and, when want_solution == 0, d_nzlhs / d_ilhs / d_xlhs may be NULL.
 *
 * blu_batch_factorize_subset_dev: column j of basis k is d_b_i/d_b_x[d_b_begin[k*m+j] .. d_b_end[k*m+j]).  As after
 * blu_batch_factorize_subset, the resident B holds, for every basis, the B it was last factorized from in library-owned
 * memory (the caller's buffers need not outlive the call; it is rebuilt on the device and only its new size comes
 * back), a captured graph is dropped and blu_batch_graph_launch answers BLU_ERROR_INVALID_CALL until the next capture.
 * This call reads the mask (nmat ints) and the info block on the host. */
int blu_batch_factorize_subset_dev(blu_batch_t *b, const int *d_run,
                                   const int64_t *d_b_begin, const int64_t *d_b_end, const int64_t *d_b_i, const double *d_b_x,
                                   int64_t bnz_total, int *d_status);
/* right-hand side of basis k: d_irhs/d_xrhs[d_rhs_begin[k] .. d_rhs_begin[k+1]) (nmat+1 offsets); outputs d_nzlhs[k],
 * d_ilhs[k*m ..], d_xlhs[k*m + n], d_status[k] */
int blu_batch_solve_for_update_dev(blu_batch_t *b, const int *d_run, const int64_t *d_rhs_begin,
                                   const int64_t *d_irhs, const double *d_xrhs, int want_solution,
                                   int64_t *d_nzlhs, int64_t *d_ilhs, double *d_xlhs, int *d_status, char trans);
/* basis k with d_xtbl[k], status in d_status[k] */
int blu_batch_update_dev(blu_batch_t *b, const int *d_run, const double *d_xtbl, int *d_status);
/* blu_batch_solve_sparse with nunits given by the caller (checked against d_unit_begin[nmat] on the device) */
int blu_batch_solve_sparse_dev(blu_batch_t *b, int64_t nunits, const int64_t *d_unit_begin,
                               const int64_t *d_rhs_begin, const int64_t *d_irhs, const double *d_xrhs,
                               int64_t *d_nzlhs, int64_t *d_ilhs, double *d_xlhs, int *d_status, char trans);
int blu_batch_solve_dense_multi_dev(blu_batch_t *b, int64_t nrhs, const double *d_rhs, double *d_lhs,
                                    char trans, int *d_status);

/* Copy bases within a batch (Clone of a BLU, for branch-and-bound and strong-branching drivers that start child LPs
 * from a parent's basis).  Basis dst[r] becomes a copy of basis src[r], for r < ncopy: factors, update history (etas,
 * nforrest, nupdate, ...), a pending solve_for_update of either direction, every per-basis getter, the resident B, and
 * the capacities of its L/U/W stores.  From then on dst[r] behaves, bit for bit, as src[r] would under the same calls
 * (and as a BLU object that went through src[r]'s history).  Sources and all bases not named in dst do not move.
 * - Capacities: a destination takes its source's L, U and W capacities exactly -- a private store of the same size
 *   where the source has one (all new private stores of a call in one block), the uniform store otherwise.  So the
 *   copy's later Reallocates and garbage collections happen exactly where the source's would.  A private store a
 *   destination held before is reclaimed at the next whole-batch store change, as the store of a re-grown basis is.
 * - Only the live part of each store is copied: L up to the end of the row-eta file, U up to u_begin[m] (plus a pending
 *   spike), the live half of W up to its fill pointer, the row-wise B up to its last entry; and the O(m) state arrays.
 * - The resident B: the destination's column pointers become the source's (offsets into the one b_i / b_x of the batch,
 *   also when B is caller-owned after blu_batch_factorize_dev or after maxvolume), so blu_batch_factorize_resident
 *   refactorizes the destination from the source's B, and a later blu_batch_factorize_subset keeps it.
 * - A source that was never factorized is copied as it is: the copy is never factorized either (nupdate None).
 * - ncopy < 0 or > nmat, an index outside [0, nmat), a repeated dst, dst[r] == src[r], a dst that is also a src of
 *   the same call (no chains, so the result never depends on order), a missing array when ncopy > 0, or an object from
 *   blu_create: BLU_ERROR_INVALID_ARGUMENT, nothing changes.  One src may appear many times (fan-out).  ncopy == 0:
 *   BLU_OK, nothing changes.
 * - A captured graph is dropped; blu_batch_graph_launch answers BLU_ERROR_INVALID_CALL until the next capture.
 * - The copy queues on the batch's stream (blu_batch_set_stream applies), is complete when the call returns, and is
 *   one launch in blu_batch_launch_count. */
int blu_batch_copy(blu_batch_t *b, int64_t ncopy, const int64_t *dst, const int64_t *src);
/* d_from: nmat ints on the device; d_from[k] = -1 keeps basis k, otherwise basis k becomes a copy of d_from[k].  The
 * map is read on the host (nmat ints) and checked as blu_batch_copy checks its pairs (any other negative value is
 * rejected as well); then the call is blu_batch_copy with the pairs in index order. */
int blu_batch_copy_dev(blu_batch_t *b, const int *d_from);

/* Save bases to images in caller memory and restore them into any slot of any batch of the same m (park more open nodes
 * of a branch-and-bound or strong-branching driver than the batch has slots, move a basis to another batch or GPU,
 * checkpoint a run, recreate a batch with more slots).  An image is a self-contained byte string: the factors, the
 * update history, a pending solve_for_update of either direction, every per-basis getter and the status word, the
 * L/U/W capacities, and the basis' resident B as entries (not as offsets into this batch's B).  It carries no
 * parameters: the destination batch's apply from the restore on.  Images are meant for the same build of the library,
 * in this process or written to disk and read back in another; there is no compatibility across versions.  Layout: a
 * fixed-size header (magic word, format version, m, sizeof(BluInfo), total length, the three capacities, the section
 * extents, the BluInfo, a 64-bit checksum of the whole image computed on the device), then the sections
 * (blu_b200/csrc/blu_save.cuh).  Every buf[r] is 16-byte aligned.
 *
 * blu_batch_save: the image of basis idx[r] into buf[r] (cap[r] bytes), its size into bytes[r], for r < n.  idx may
 * repeat.  buf == NULL: only bytes[] is written (a size query).  Save changes nothing: no state, no store, and a
 * captured graph stays valid.
 * - A cap[r] smaller than the image: BLU_ERROR_INVALID_ARGUMENT after bytes[] is written, and no image is written.
 * - n < 0, an idx outside [0, nmat), a missing idx / bytes (n > 0) or cap (buf given), a buf[r] that is NULL or not
 *   16-byte aligned, or an object from blu_create: BLU_ERROR_INVALID_ARGUMENT.
 *
 * blu_batch_restore: basis dst[r] becomes the basis saved in image buf[r] (cap[r] bytes readable), for r < n.
 * - Same batch: restoring into slot d the image of basis s of the same batch leaves d exactly as blu_batch_copy(d <- s)
 *   would, bit for bit, in every getter, solve, get_factors and later call.  Another batch (same m, same or another
 *   device): the restored basis behaves as the saved one would under the same calls and the same parameters.
 * - Capacities: the destination takes the image's L, U and W capacities exactly -- the uniform store where the
 *   capacity equals the batch's uniform one, otherwise a private store of that size (all new private stores of a call
 *   in one block; a destination's old private block is reclaimed at the next whole-batch store change, as after a
 *   copy).  If the image's row-wise B needs more room than the batch's bnz_cap, that room grows first.
 * - Resident B: the destination's becomes the image's columns (a column with a negative length stays negative; a
 *   never-factorized basis has all-empty columns), with the whole resident B rebuilt in library-owned memory as
 *   blu_batch_factorize_subset rebuilds it (a caller-owned B from blu_batch_factorize_dev moves into library memory).
 *   blu_batch_factorize_resident then refactorizes the destination from the saved basis' B.  A captured graph is
 *   dropped: blu_batch_graph_launch answers BLU_ERROR_INVALID_CALL until the next capture.
 * - BLU_ERROR_INVALID_ARGUMENT, and nothing changes: a wrong magic word, version, m or sizeof(BluInfo); a length
 *   greater than cap[r]; an extent outside its capacity; a checksum mismatch; a buf[r] that is NULL or not 16-byte
 *   aligned; n < 0 or n > nmat; a dst outside [0, nmat) or a repeated dst; a missing array when n > 0; an object from
 *   blu_create.  The same image may be restored into several slots (fan-out).  n == 0: BLU_OK, nothing changes.
 * - The host variants move the images through device scratch in chunks of about 1 GB; a restore of more than one chunk
 *   checks every image before it changes anything.
 *
 * Both calls queue on the batch's stream (blu_batch_set_stream applies), are complete on return, and are counted in
 * blu_batch_launch_count. */
int blu_batch_save(blu_batch_t *b, int64_t n, const int64_t *idx, void *const *buf, const int64_t *cap, int64_t *bytes);
int blu_batch_restore(blu_batch_t *b, int64_t n, const int64_t *dst, const void *const *buf, const int64_t *cap);
/* The same two calls with every buf[r] in device memory on the batch's device (idx, dst, cap, bytes and the pointer
 * arrays stay on the host).  Host traffic: save reads the n image sizes back; restore reads the n fixed-size headers
 * and a checksum verdict; nothing else whose size grows with the images crosses the bus. */
int blu_batch_save_dev(blu_batch_t *b, int64_t n, const int64_t *idx, void *const *d_buf, const int64_t *cap, int64_t *bytes);
int blu_batch_restore_dev(blu_batch_t *b, int64_t n, const int64_t *dst, const void *const *d_buf, const int64_t *cap);
/* The steady-state step of a resident batch (factorization launches + condest/residual_test + solve_dense of the
 * uploaded rhs) captured into a CUDA graph once, then replayed with one launch per step; a basis that answers
 * Reallocate during a replay is grown and re-run by the classic path before the call returns. */
int blu_batch_graph_capture(blu_batch_t *b, char trans);
int blu_batch_graph_launch(blu_batch_t *b);
/* cudaStream_t the library launches on (so callers can bracket it with their own events),
 * and a way to make it use the caller's stream instead */
void *blu_batch_stream(blu_batch_t *b);
int blu_batch_set_stream(blu_batch_t *b, void *cuda_stream);
int blu_batch_synchronize(blu_batch_t *b);
/* device time of the last factorize / solve kernels, measured with CUDA events on the launching stream */
double blu_batch_last_kernel_ms(blu_batch_t *b, int which /*0 factorize (all kernels of the call), 1 solve_dense, 2 the condest/residual_test kernel alone, 3 / 4 / 5 the head / tail / build launch of the last split factorization pass (3 = the single launch when not split)*/);
/* number of kernels this library launched since creation */
int64_t blu_batch_launch_count(blu_batch_t *b);

/* ------------------------------------------------------------------ */
/* one batch over several GPUs of this process (SURVEY.md 8b/8e: "a device list")  */
/* Bases are split into contiguous ranges, one per device (sizes differ by at most   */
/* one); every device has its own blu_batch_t, host thread and stream; there is no   */
/* collective -- the results land in the caller's arrays at the bases' own offsets.  */
/* ------------------------------------------------------------------ */
typedef struct blu_multi blu_multi_t;
int blu_multi_create(blu_multi_t **out, int64_t nmat, int64_t m, int64_t bnz_cap, const int *devices, int ndev);
void blu_multi_destroy(blu_multi_t *mb);
/* factorize every basis and (if rhs and lhs are given) solve with it; layout as blu_batch_factorize /
 * blu_batch_solve_dense.  status[k]: per-basis code of the factorization, or of the solve if that failed. */
int blu_multi_factorize_solve(blu_multi_t *mb, const int64_t *b_begin, const int64_t *b_end, const int64_t *b_i,
                              const double *b_x, int64_t bnz_total, const double *rhs, double *lhs, char trans, int *status);
/* the batch object of device slot d and the range of bases it owns (for the getters / further calls) */
blu_batch_t *blu_multi_part(blu_multi_t *mb, int d, int64_t *first, int64_t *count);

const char *blu_version(void);

#ifdef __cplusplus
}
#endif
#endif
