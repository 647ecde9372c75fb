/* blu_maxvolume.cuh -- device side of blu_batch_maxvolume: maxvolume (maxvolume.rs:64-224) on every basis of a
 * batch, all bases in lockstep over their pool columns.  The sparse solves, the update and the factorization are
 * the batch kernels of blu_sparse.cuh / blu_factor_*.cuh run under the per-slot run mask (BluDev::run); the
 * kernels here do what maxvolume.rs does between those calls: pick the next column, choose the leaving row,
 * keep basis / isbasic / nupdate, decide on a refactorization and point B at the pool columns of the basis.
 * Nothing leaves the device per column except status words and counts. */
#ifndef BLU_MAXVOLUME_CUH
#define BLU_MAXVOLUME_CUH
#include "blu_types.h"

/* per-call state of blu_batch_maxvolume (all device pointers) */
struct MvDev {
    int nmat, m;
    blu_i64 ncol;
    const blu_i64 *a_begin, *a_end;     /* nmat*ncol: column j of basis k's pool is [a_begin[k*ncol+j], a_end[k*ncol+j]) */
    blu_i64 *basis;                     /* nmat*m */
    blu_i64 *isbasic;                   /* nmat*ncol */
    blu_i64 *nupdate;                   /* nmat */
    int *mvst;                          /* nmat: what maxvolume returns for the basis; BLU_OK while it is still running */
    int *run;                           /* nmat: the run mask of the next masked launches (BluDev::run) */
    blu_i64 *rhs_begin, *rhs_end;       /* nmat: right-hand side of the solve for the current column (into the pool) */
    blu_i64 *leave;                     /* nmat: the position leaving the basis (right-hand side of the transposed solve) */
    double *xtbl;                       /* nmat: pivot of the update */
    blu_i64 *b_begin, *b_end;           /* nmat*m: B as a view of the pool, maxvolume.rs:180-224 */
    unsigned long long *cnt;            /* MV_CNT_* */
};
#define MV_CNT_NEXT 0       /* first column >= j0 that is a candidate for some running basis (ncol if none) */
#define MV_CNT_REFACTOR 1   /* bases that refactorize after this column */
#define MV_CNT_REALLOC 2    /* bases whose factorization answered Reallocate */
#define MV_CNT_MAXNZ 3      /* most entries of a B about to be factorized */
#define MV_CNT_N 4

/* the next column any running basis examines (maxvolume.rs:97-99 skips the basic ones).  One warp per basis scans
 * from j0 in chunks of 32 columns.  cnt[MV_CNT_NEXT] is reset to ~0 by the host before the launch. */
__global__ void __launch_bounds__(32) k_mv_next(MvDev V, blu_i64 j0) {
    const int k = blockIdx.x, lane = threadIdx.x & 31;
    if (V.mvst[k] != BLU_OK) return;
    const blu_i64 *isb = V.isbasic + (size_t)k * V.ncol;
    blu_i64 found = V.ncol;
    for (blu_i64 c = j0; c < V.ncol; c += 32) {
        const blu_i64 j = c + lane;
        const unsigned hit = __ballot_sync(FULLMASK, j < V.ncol && isb[j] == 0);
        if (hit) { found = c + __ffs((int)hit) - 1; break; }
    }
    if (lane == 0) atomicMin(&V.cnt[MV_CNT_NEXT], (unsigned long long)found);
}

/* masks and right-hand sides of column j: a basis runs when it is still running and j is not basic for it */
__global__ void k_mv_setup(MvDev V, blu_i64 j) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= V.nmat) return;
    const size_t q = (size_t)k * V.ncol + j;
    V.run[k] = V.mvst[k] == BLU_OK && V.isbasic[q] == 0;
    V.rhs_begin[k] = V.a_begin[q];
    V.rhs_end[k] = V.a_end[q];
}

/* leaving-row selection, maxvolume.rs:111-142, one warp per basis over the compacted solution of the 'N' solve
 * (xout[k*m + n] is the value of entry ilhs[k*m + n]).  The reference keeps the FIRST strict maximum of |x| in
 * ilhs order starting from 0.0: every lane keeps the first strict maximum of its own entries, and the warp
 * reduction prefers the larger value, then the earlier position -- the same entry, and NaN never wins.
 * scal[2k], scal[2k+1]: status and nzlhs of the solve. */
__global__ void __launch_bounds__(32) k_mv_select(MvDev V, blu_i64 j, const int *scal, const blu_i64 *ilhs, const double *xout, double volumetol) {
    const int k = blockIdx.x, lane = threadIdx.x & 31;
    if (!V.run[k]) return;
    const int st = scal[2 * k];
    if (st != BLU_OK) {
        if (lane == 0) { V.mvst[k] = st; V.run[k] = 0; }
        return;
    }
    const int nz = scal[2 * k + 1];
    const double *x = xout + (size_t)k * V.m;
    double best = 0.0; int pos = 0x7fffffff;
    for (int n = lane; n < nz; n += 32) {
        const double a = fabs(x[n]);
        if (a > best) { best = a; pos = n; }
    }
    for (int d = 16; d > 0; d >>= 1) {
        const double ob = __shfl_xor_sync(FULLMASK, best, d);
        const int op = __shfl_xor_sync(FULLMASK, pos, d);
        if (ob > best || (ob == best && op < pos)) { best = ob; pos = op; }
    }
    if (lane != 0) return;
    if (best <= volumetol) { V.run[k] = 0; return; }      /* keep the basis (maxvolume.rs:133-135) */
    const bool none = pos == 0x7fffffff;                 /* no entry above 0.0: imax = 0, xtbl = 0.0 as in the reference */
    const blu_i64 imax = none ? 0 : ilhs[(size_t)k * V.m + pos];
    blu_i64 *bas = V.basis + (size_t)k * V.m, *isb = V.isbasic + (size_t)k * V.ncol;
    isb[bas[imax]] = 0;
    isb[j] = 1;
    bas[imax] = j;
    V.nupdate[k]++;
    V.leave[k] = imax;
    V.xtbl[k] = none ? 0.0 : x[pos];
}

/* a masked solve is over: a basis whose solve failed stops with that status.  Reallocate is left alone (the host
 * grows the stores and runs those bases again), so the kernel can run again after the re-run. */
__global__ void k_mv_absorb(MvDev V, const int *scal, int stride) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= V.nmat || !V.run[k]) return;
    const int st = scal[(size_t)k * stride];
    if (st != BLU_OK && st != BLU_REALLOCATE) { V.mvst[k] = st; V.run[k] = 0; }
}

/* after the update (ust != null): a basis whose update failed stops; the others refactorize when
 * nforrest == m, pivot_error > 1e-8 or update_cost > 1 (maxvolume.rs:161-170; update_cost as lu.rs:324).
 * ust == null: the first factorization, every running basis.  The bases that will be factorized keep run = 1 and
 * get B as a view of their pool (maxvolume.rs:180-224); cnt counts them and the largest nnz(B).  A basis whose
 * update answered Reallocate is left for the re-run; the decision is idempotent, so the kernel runs again then. */
__global__ void __launch_bounds__(32) k_mv_decide(MvDev V, BluDev D, const int *ust) {
    const int k = blockIdx.x, lane = threadIdx.x & 31;
    if (!V.run[k]) return;
    if (ust) {
        const int st = ust[k];
        if (st == BLU_REALLOCATE) return;
        if (st != BLU_OK) { if (lane == 0) { V.mvst[k] = st; V.run[k] = 0; } return; }
        const BluInfo &I = D.info[k];
        const bool refactor = I.nforrest == V.m || I.pivot_error > 1e-8 || I.update_cost_numer / I.update_cost_denom > 1.0;
        if (!refactor) { if (lane == 0) V.run[k] = 0; return; }
    }
    const blu_i64 *bas = V.basis + (size_t)k * V.m, *ab = V.a_begin + (size_t)k * V.ncol, *ae = V.a_end + (size_t)k * V.ncol;
    blu_i64 *bb = V.b_begin + (size_t)k * V.m, *be = V.b_end + (size_t)k * V.m;
    long long nnz = 0;
    for (int i = lane; i < V.m; i += 32) {
        const blu_i64 c = bas[i], b = ab[c], e = ae[c];
        bb[i] = b; be[i] = e;
        nnz += e > b ? e - b : 0;
    }
    for (int d = 16; d > 0; d >>= 1) nnz += __shfl_xor_sync(FULLMASK, nnz, d);
    if (lane == 0) {
        atomicAdd(&V.cnt[MV_CNT_REFACTOR], 1ull);
        atomicMax(&V.cnt[MV_CNT_MAXNZ], (unsigned long long)nnz);
    }
}

/* after a masked factorization: count the bases that asked for more memory (absorb == 0), or, once the
 * factorization is final, stop every basis whose status is not OK (absorb != 0; WarningSingularMatrix stops
 * maxvolume too, maxvolume.rs:93-95, 166-169).  The factorized bases leave with run = 0. */
__global__ void k_mv_factor_status(MvDev V, BluDev D, int absorb) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= V.nmat || !V.run[k]) return;
    const int st = D.info[k].status;
    if (!absorb) { if (st == BLU_REALLOCATE) atomicAdd(&V.cnt[MV_CNT_REALLOC], 1ull); return; }
    if (st != BLU_OK) V.mvst[k] = st;
    V.run[k] = 0;
}

#endif
