/* blu_solve.cuh -- dense solves and factor export on the device.
 * Reference: src/lu/solve_dense.rs:7-120, src/lu/garbage_perm.rs:16-48, src/get_factors.rs:48-180. */
#ifndef BLU_SOLVE_CUH
#define BLU_SOLVE_CUH
#include "blu_dev_common.cuh"

__device__ __forceinline__ bool is_trans(char t) { return t == 't' || t == 'T'; }

/* garbage_perm.rs:16-48; one thread (only after > m updates worth of pivots accumulated) */
__device__ __forceinline__ void dev_garbage_perm(Mat &M) {
    BluInfo *I = M.info;
    const int m = M.m, pivotlen = I->pivotlen;
    if (pivotlen > m) {
        int marker = ++I->marker;
        int put = pivotlen;
        for (int get = pivotlen - 1; get >= 0; get--) {
            int j = M.pivotcol[get];
            if (M.marked[j] != marker) {
                M.marked[j] = marker;
                --put;
                M.pivotcol[put] = j;
                M.pivotrow[put] = M.pivotrow[get];
            }
        }
        for (int k = 0; k < m; k++) { M.pivotcol[k] = M.pivotcol[put + k]; M.pivotrow[k] = M.pivotrow[put + k]; }
        I->pivotlen = m;
    }
}

/* acc += term of lanes 0..n-1 in lane order, one rounding per step: exactly the sum the
 * reference's sequential dot-product loop produces (lu/solve_dense.rs:64-66,83-85). */
__device__ __forceinline__ double ordered_acc(double acc, double term, int n) {
    /* the lanes park their terms in shared memory and every lane runs the same serial sum over them
     * (broadcast reads): ~3x cheaper per term than walking the lanes with shuffles */
    __shared__ double obuf[4][32];
    double *b = obuf[(threadIdx.x >> 5) & 3];
    __syncwarp();
    b[threadIdx.x & 31] = term;
    __syncwarp();
    if (n == 32) {
        #pragma unroll
        for (int t = 0; t < 32; t++) acc = __dadd_rn(acc, b[t]);
    } else {
        for (int t = 0; t < n; t++) acc = __dadd_rn(acc, b[t]);
    }
    return acc;
}

/* Dot-product sweep over the pivot order (ascending or descending) where the batch of 32 pivots in
 * flight is processed as wavefronts: lane l owns the l-th pivot of the batch and computes its WHOLE
 * dot product serially, in storage order and with one rounding per operation -- exactly the
 * reference's arithmetic -- as soon as every pivot it can depend on is finished.  dep[k] is the
 * furthest pivot position line k reaches (blu_factor_build.cuh); "all lanes up to that one are done"
 * is a conservative readiness test.  Lines are terminated by a negative index.
 *   head(k)            -> start of line k
 *   tail(k, acc)       -> epilogue of pivot k, run by the owning lane (stores into vec)
 *   batch_end(cnt)     -> after each batch (e.g. ordered accumulation of per-lane values)
 * Valid only for a fresh factorization (nupdate == 0); after updates the sequential sweeps run. */
__device__ __forceinline__ double dev_line_dot_n(const int *idx, const double *val, int pos, int len, const double *vec, double acc, bool subtract);
__device__ __forceinline__ void dev_line_prefetch(const int *idx, const double *val, int pos, int len);
__device__ __forceinline__ void dev_line_axpy_n(const int *idx, const double *val, int pos, int len, double *vec, double x);
#define SWEEP_SHORT 8   /* lines of up to this many entries are summed by their own lane; longer ones by the whole warp */
template <typename Head, typename Init, typename Tail, typename BatchEnd>
__device__ __forceinline__ void dev_dot_sweep_init(int m, bool asc, const int *dep, const int *idx, const double *val,
                                                   const double *vec, bool subtract, Head head, Init init, Tail tail, BatchEnd batch_end) {
    const int lane = threadIdx.x & 31;
    for (int s = 0; s < m; s += 32) {
        const int cnt = m - s < 32 ? m - s : 32;
        const bool mine = lane < cnt;
        const int k = asc ? s + lane : m - 1 - s - lane;
        int nd = 0, b = 0, len = 0;
        if (mine) {
            const int need = dep[k];
            nd = asc ? need - s + 1 : (m - 1 - s) - need + 1;   /* leading lanes of the batch that must be done */
            head(k, &b, &len);
            if (len > SWEEP_SHORT) { lane_prefetch(idx + b); lane_prefetch(val + b); }
        }
        const unsigned full = cnt == 32 ? FULLMASK : ((1u << cnt) - 1u);
        const unsigned lm = nd <= 0 ? 0u : (nd >= 32 ? FULLMASK : ((1u << nd) - 1u));
        unsigned done = 0;
        bool fin = !mine;
        while (done != full) {
            const bool ready = !fin && (done & lm) == lm;
            const unsigned rshort = __ballot_sync(FULLMASK, ready && len <= SWEEP_SHORT);
            if (rshort) {
                /* every ready short line at once, one lane each; the loads of a line are independent */
                if (ready && len <= SWEEP_SHORT) {
                    int r[SWEEP_SHORT]; double v[SWEEP_SHORT];
                    #pragma unroll
                    for (int q = 0; q < SWEEP_SHORT; q++) { r[q] = q < len ? idx[b + q] : -1; v[q] = q < len ? val[b + q] : 0.0; }
                    double acc = init(k);       /* the value the reference's running vector holds before the terms */
                    #pragma unroll
                    for (int q = 0; q < SWEEP_SHORT; q++) {
                        if (q < len) { const double t = __dmul_rn(vec[r[q]], v[q]); acc = subtract ? __dsub_rn(acc, t) : __dadd_rn(acc, t); }
                    }
                    tail(k, acc);
                    fin = true;
                }
                __syncwarp();
                done |= rshort;
            } else {
                /* the first ready long line, all lanes together (ordered chunked sum) */
                const unsigned rlong = __ballot_sync(FULLMASK, ready);
                const int t = __ffs((int)rlong) - 1;
                const int bb = __shfl_sync(FULLMASK, b, t), ll = __shfl_sync(FULLMASK, len, t);
                if (t + 1 < cnt) dev_line_prefetch(idx, val, __shfl_sync(FULLMASK, b, t + 1), __shfl_sync(FULLMASK, len, t + 1));
                double a0 = 0.0;
                if (lane == t) a0 = init(k);
                a0 = __shfl_sync(FULLMASK, a0, t);
                const double acc = dev_line_dot_n(idx, val, bb, ll, vec, a0, subtract);
                if (lane == t) { tail(k, acc); fin = true; }
                __syncwarp();
                done |= 1u << t;
            }
        }
        batch_end(cnt);
    }
}
struct NoBatchEnd { __device__ __forceinline__ void operator()(int) const {} };
struct ZeroInit { __device__ __forceinline__ double operator()(int) const { return 0.0; } };
template <typename Head, typename Tail, typename BatchEnd>
__device__ __forceinline__ void dev_dot_sweep(int m, bool asc, const int *dep, const int *idx, const double *val,
                                              const double *vec, bool subtract, Head head, Tail tail, BatchEnd batch_end) {
    dev_dot_sweep_init(m, asc, dep, idx, val, vec, subtract, head, ZeroInit(), tail, batch_end);
}

/* One warp per basis.  The sweeps are sequential over the pivot order (as in the
 * reference); the lanes share the dot product / axpy of each step and the pointer
 * loads are batched 32 pivots at a time.  Every multiply, add, subtract and divide is
 * rounded once and sums run in the reference's order, so the result is bit-identical. */
/* Two shapes: (a) multi_work == unit_slot == nullptr: unit u = basis D.slot0 + u of a batch, one right-hand
 * side each; (b) both given: nrhs units, unit u reads the basis in slot unit_slot[u] (many right-hand sides
 * on every basis of a batch, blu_batch_solve_dense_multi).  The factors are only read; every unit has its
 * own work vector multi_work + u*m; the pivot sequences must have been compacted by k_garbage_perm before. */
__global__ void __launch_bounds__(32) k_solve_dense(BluDev D, const double *rhs_all, double *lhs_all, char trans, int *status,
                                                     double *multi_work, int nrhs, const int *unit_slot) {
    __shared__ Mat M;
    const int lane = threadIdx.x & 31;
    const bool multi = multi_work != nullptr;
    const int nunits = multi ? nrhs : D.nslot;
    for (int unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
        const int s = multi ? unit : D.slot0 + unit;       /* index of rhs / lhs / status */
        __syncwarp();
        if (lane == 0) mat_view(M, D, unit_slot ? unit_slot[unit] : s);
        __syncwarp();
        const int m = M.m;
        BluInfo *I = M.info;
        if (I->nupdate < 0) { if (lane == 0 && status) status[s] = BLU_ERROR_INVALID_CALL; __syncwarp(); continue; }
        if (!multi && lane == 0) dev_garbage_perm(M);
        __syncwarp();
        const double *rhs = rhs_all + (size_t)s * m;
        double *lhs = lhs_all + (size_t)s * m;
        double *work = multi ? multi_work + (size_t)unit * m : M.work1;
        const int nforrest = I->nforrest;
        const bool fresh = I->nupdate == 0;   /* the wavefront sweeps need the dependency reach computed by build_factors */
        for (int i = lane; i < m; i += 32) work[i] = rhs[i];
        __syncwarp();
        if (is_trans(trans)) {
            /* U', lu/solve_dense.rs:40-48.  Fresh factorization: column k' of U (ascending pivot order by
             * construction) lists exactly the terms work[jp_k'] receives, in the order the reference's row
             * sweep applies them, so the sweep runs as wavefront dot products. */
            if (fresh) {
                dev_dot_sweep_init(m, true, M.dep_uc, M.u_idx, M.u_val, lhs, true,
                                   [&](int k, int *b, int *len) { *b = M.u_begin[M.pivotrow[k]]; *len = M.len_uc[k]; },
                                   [&](int k) { return work[M.pivotcol[k]]; },
                                   [&](int k, double acc) { lhs[M.pivotrow[k]] = __ddiv_rn(acc, M.colpiv[M.pivotcol[k]]); }, NoBatchEnd());
            } else
            for (int kb = 0; kb < m; kb += 32) {
                int k = kb + lane;
                int jp = k < m ? M.pivotcol[k] : 0, ip = k < m ? M.pivotrow[k] : 0;
                int b = k < m ? M.lbeg[jp] : 0, e = k < m ? M.lend[jp] : 0;
                double piv = k < m ? M.colpiv[jp] : 1.0;
                if (e > b) { lane_prefetch(M.w_idx + b); lane_prefetch(M.w_val + b); }
                int n = m - kb < 32 ? m - kb : 32;
                for (int t = 0; t < n; t++) {
                    int jj = __shfl_sync(FULLMASK, jp, t), ii = __shfl_sync(FULLMASK, ip, t);
                    int bb = __shfl_sync(FULLMASK, b, t), ee = __shfl_sync(FULLMASK, e, t);
                    double pv = __shfl_sync(FULLMASK, piv, t);
                    double x = __ddiv_rn(work[jj], pv);
                    __syncwarp();
                    for (int pos = bb + lane; pos < ee; pos += 32) { const int r = M.w_idx[pos]; work[r] = __dsub_rn(work[r], __dmul_rn(x, M.w_val[pos])); }
                    if (lane == 0) lhs[ii] = x;
                    __syncwarp();
                }
            }
            /* etas backwards, :52-59 */
            for (int t = nforrest - 1; t >= 0; t--) {
                double x = lhs[M.eta_row[t]];
                __syncwarp();
                for (int pos = M.r_begin[t] + lane; pos < M.r_begin[t + 1]; pos += 32) { const int r = M.l_idx[pos]; lhs[r] = __dsub_rn(lhs[r], __dmul_rn(x, M.l_val[pos])); }
                __syncwarp();
            }
            /* L', :63-73 */
            if (fresh) {
                dev_dot_sweep(m, false, M.dep_lc, M.l_idx, M.l_val, lhs, false,
                              [&](int k, int *b, int *len) { *b = M.l_begin_p[k]; *len = M.l_begin_p[k + 1] - *b - 1; },
                              [&](int k, double x) { const int i = M.p[k]; lhs[i] = __dsub_rn(lhs[i], x); }, NoBatchEnd());
            } else
            for (int kb = ((m - 1) / 32) * 32; kb >= 0; kb -= 32) {
                int k = kb + lane;
                int b = k < m ? M.l_begin_p[k] : 0, e = k < m ? M.l_begin_p[k + 1] - 1 : 0;
                int ip = k < m ? M.p[k] : 0;
                if (e > b) { lane_prefetch(M.l_idx + b); lane_prefetch(M.l_val + b); }
                unsigned ne = __ballot_sync(FULLMASK, e > b);
                while (ne) {
                    int t = 31 - __clz((int)ne);
                    ne &= ~(1u << t);
                    int bb = __shfl_sync(FULLMASK, b, t), ee = __shfl_sync(FULLMASK, e, t), ii = __shfl_sync(FULLMASK, ip, t);
                    double x = 0.0;
                    for (int cb = bb; cb < ee; cb += 32) {
                        const int pos = cb + lane;
                        const double term = pos < ee ? __dmul_rn(lhs[M.l_idx[pos]], M.l_val[pos]) : 0.0;
                        x = ordered_acc(x, term, ee - cb < 32 ? ee - cb : 32);
                    }
                    if (lane == 0) lhs[ii] = __dsub_rn(lhs[ii], x);
                    __syncwarp();
                }
            }
        } else {
            /* L, :81-90 (row-wise dot form) */
            if (fresh) {
                dev_dot_sweep(m, true, M.dep_lt, M.l_idx, M.l_val, work, false,
                              [&](int k, int *b, int *len) { *b = M.lt_begin_p[k]; *len = M.lt_begin_p[k + 1] - *b - 1; },
                              [&](int k, double x) { const int i = M.p[k]; work[i] = __dsub_rn(work[i], x); }, NoBatchEnd());
            } else
            for (int kb = 0; kb < m; kb += 32) {
                int k = kb + lane;
                int b = k < m ? M.lt_begin_p[k] : 0, e = k < m ? M.lt_begin_p[k + 1] - 1 : 0;
                int ip = k < m ? M.p[k] : 0;
                if (e > b) { lane_prefetch(M.l_idx + b); lane_prefetch(M.l_val + b); }
                unsigned ne = __ballot_sync(FULLMASK, e > b);
                while (ne) {
                    int t = __ffs((int)ne) - 1;
                    ne &= ne - 1;
                    int bb = __shfl_sync(FULLMASK, b, t), ee = __shfl_sync(FULLMASK, e, t), ii = __shfl_sync(FULLMASK, ip, t);
                    double x = 0.0;
                    for (int cb = bb; cb < ee; cb += 32) {
                        const int pos = cb + lane;
                        const double term = pos < ee ? __dmul_rn(work[M.l_idx[pos]], M.l_val[pos]) : 0.0;
                        x = ordered_acc(x, term, ee - cb < 32 ? ee - cb : 32);
                    }
                    if (lane == 0) work[ii] = __dsub_rn(work[ii], x);
                    __syncwarp();
                }
            }
            /* etas, :93-102 */
            for (int t = 0; t < nforrest; t++) {
                double x = 0.0;
                const int rb = M.r_begin[t], re = M.r_begin[t + 1];
                for (int cb = rb; cb < re; cb += 32) {
                    const int pos = cb + lane;
                    const double term = pos < re ? __dmul_rn(work[M.l_idx[pos]], M.l_val[pos]) : 0.0;
                    x = ordered_acc(x, term, re - cb < 32 ? re - cb : 32);
                }
                if (lane == 0) work[M.eta_row[t]] = __dsub_rn(work[M.eta_row[t]], x);
                __syncwarp();
            }
            /* U, :106-118 (column-wise axpy form, terminator-delimited) */
            if (fresh && M.ur_ptr && I->have_ur) {
                /* the same arithmetic row by row: row k of U, columns in descending pivot order, starting
                 * from the value L left in work[] -- wavefronts of independent pivots */
                dev_dot_sweep_init(m, false, M.dep_ur, M.ur_idx, M.ur_val, work, true,
                                   [&](int k, int *b, int *len) { *b = M.ur_ptr[k]; *len = M.ur_ptr[k + 1] - *b; },
                                   [&](int k) { return work[M.pivotrow[k]]; },
                                   [&](int k, double acc) {
                                       const int ip = M.pivotrow[k];
                                       const double x = __ddiv_rn(acc, M.rowpiv[ip]);
                                       work[ip] = x; lhs[M.pivotcol[k]] = x;
                                   }, NoBatchEnd());
            } else
            for (int kb = ((m - 1) / 32) * 32; kb >= 0; kb -= 32) {
                int k = kb + lane;
                int jp = k < m ? M.pivotcol[k] : 0, ip = k < m ? M.pivotrow[k] : 0;
                int b = k < m ? M.u_begin[ip] : 0;
                double piv = k < m ? M.rowpiv[ip] : 1.0;
                if (k < m) { lane_prefetch(M.u_idx + b); lane_prefetch(M.u_val + b); }
                const int ln = (fresh && k < m) ? M.len_uc[k] : -1;
                int n = m - kb < 32 ? m - kb : 32;
                for (int t = n - 1; t >= 0; t--) {
                    int jj = __shfl_sync(FULLMASK, jp, t), ii = __shfl_sync(FULLMASK, ip, t);
                    int bb = __shfl_sync(FULLMASK, b, t);
                    const int ll = __shfl_sync(FULLMASK, ln, t);
                    double pv = __shfl_sync(FULLMASK, piv, t);
                    if (fresh && t > 0) dev_line_prefetch(M.u_idx, M.u_val, __shfl_sync(FULLMASK, b, t - 1), __shfl_sync(FULLMASK, ln, t - 1));
                    double x = __ddiv_rn(work[ii], pv);
                    __syncwarp();
                    if (ll >= 0) dev_line_axpy_n(M.u_idx, M.u_val, bb, ll, work, x);
                    else
                    for (int pos = bb;; pos += 32) {
                        int idx = M.u_idx[pos + lane];
                        unsigned term = __ballot_sync(FULLMASK, idx < 0);
                        int nvalid = term ? __ffs((int)term) - 1 : 32;
                        if (lane < nvalid) work[idx] = __dsub_rn(work[idx], __dmul_rn(x, M.u_val[pos + lane]));
                        if (term) break;
                    }
                    if (lane == 0) lhs[jj] = x;
                    __syncwarp();
                }
            }
        }
        if (lane == 0 && status) status[s] = BLU_OK;
        __syncwarp();
    }
}

/* garbage_perm on slot D.slot0 + blockIdx.x: before units that share a basis read its pivot sequence */
__global__ void k_garbage_perm(BluDev D) {
    __shared__ Mat M;
    if (threadIdx.x == 0) { mat_view(M, D, D.slot0 + (int)blockIdx.x); if (M.info->nupdate >= 0) dev_garbage_perm(M); }
}

/* get_factors.rs:48-180.  Output in 64-bit indices straight into device staging buffers:
 *   rowperm[m] colperm[m] l_colptr[m+1] l_rowidx/l_value[m+l_nz] u_colptr[m+1] u_rowidx/u_value[m+u_nz]
 * One CTA; the fills run in pivot order on one warp so the rows inside every output column
 * come out ascending, as get_factors.rs:97-113 and :150-167 produce them. */
template <int NT> __global__ void __launch_bounds__(NT) k_get_factors(BluDev D, int s, i64 *rowperm, i64 *colperm,
                                                                       i64 *l_colptr, i64 *l_rowidx, double *l_value,
                                                                       i64 *u_colptr, i64 *u_rowidx, double *u_value, int *status) {
    __shared__ Mat M;
    __shared__ int iscr[40];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) mat_view(M, D, s);
    bsync<NT>();
    const int m = M.m;
    if (M.info->nupdate != 0) { if (tid == 0) *status = BLU_ERROR_INVALID_CALL; return; }
    for (int k = tid; k < m; k += NT) { rowperm[k] = M.pivotrow[k]; colperm[k] = M.pivotcol[k]; }
    int *fill = M.iwork1;   /* m */
    /* L */
    {
        int put = 0;
        for (int base = 0; base < m; base += NT) {
            int k = base + tid;
            int c = k < m ? M.l_begin_p[k + 1] - M.l_begin_p[k] : 0; /* entries + 1 (terminator <-> unit diagonal) */
            int tot, ex = block_excl_scan<NT>(c, &tot, iscr);
            if (k < m) {
                l_colptr[k] = put + ex;
                l_rowidx[put + ex] = k; l_value[put + ex] = 1.0;
                fill[k] = put + ex + 1;
            }
            put += tot;
        }
        if (tid == 0) l_colptr[m] = put;
    }
    bsync<NT>();
    if (wid == 0) {
        for (int k = 0; k < m; k++) {
            const int b = M.lt_begin_p[k], e = M.lt_begin_p[k + 1] - 1;
            for (int pos = b + lane; pos < e; pos += 32) {
                int c = M.prank[M.l_idx[pos]];
                int dst = fill[c]; fill[c] = dst + 1;
                l_rowidx[dst] = k; l_value[dst] = M.l_val[pos];
            }
            __syncwarp();
        }
    }
    bsync<NT>();
    /* U */
    for (int k = tid; k < m; k += NT) fill[k] = 0;
    bsync<NT>();
    for (int j = wid; j < m; j += NT / 32)
        for (int pos = M.lbeg[j] + lane; pos < M.lend[j]; pos += 32) atomicAdd(&fill[M.qrank[M.w_idx[pos]]], 1);
    bsync<NT>();
    {
        int put = 0;
        for (int base = 0; base < m; base += NT) {
            int k = base + tid;
            int c = k < m ? fill[k] + 1 : 0;
            int tot, ex = block_excl_scan<NT>(c, &tot, iscr);
            if (k < m) {
                u_colptr[k] = put + ex;
                u_rowidx[put + ex + c - 1] = k; u_value[put + ex + c - 1] = M.colpiv[M.pivotcol[k]];
                fill[k] = put + ex;
            }
            put += tot;
        }
        if (tid == 0) u_colptr[m] = put;
    }
    bsync<NT>();
    if (wid == 0) {
        for (int k = 0; k < m; k++) {
            const int j = M.pivotcol[k];
            for (int pos = M.lbeg[j] + lane; pos < M.lend[j]; pos += 32) {
                int c = M.qrank[M.w_idx[pos]];
                int dst = fill[c]; fill[c] = dst + 1;
                u_rowidx[dst] = k; u_value[dst] = M.w_val[pos];
            }
            __syncwarp();
        }
        if (lane == 0) *status = BLU_OK;
    }
}

#endif

/* ------------------------------------------------------------------ */
/* condest x2, residual_test, matrix_norm: the tail of factorize()      */
/* (factorize.rs:121-147; lu/condest.rs:15-157, lu/residual_test.rs:    */
/* 16-152, lu/matrix_norm.rs:8-48).  They back the getters condest_l/u, */
/* norm_l/u, normest_l/u_inv, onenorm, infnorm, residual_test.          */
/* One warp per basis; every sweep is sequential over the pivot order   */
/* like the reference, the lanes share each dot product / axpy, and all */
/* sums run in the reference's order (bit-identical results).           */
/* ------------------------------------------------------------------ */
#ifndef BLU_SOLVE_NORMS
#define BLU_SOLVE_NORMS

/* acc -= term of lanes 0..n-1 in lane order */
__device__ __forceinline__ double ordered_sub(double acc, double term, int n) {
    __shared__ double obuf[4][32];
    double *b = obuf[(threadIdx.x >> 5) & 3];
    __syncwarp();
    b[threadIdx.x & 31] = term;
    __syncwarp();
    if (n == 32) {
        #pragma unroll
        for (int t = 0; t < 32; t++) acc = __dsub_rn(acc, b[t]);
    } else {
        for (int t = 0; t < n; t++) acc = __dsub_rn(acc, b[t]);
    }
    return acc;
}

/* sum of |x[i]|, i ascending (residual_test.rs onenorm helper) */
__device__ __forceinline__ double dev_vec_onenorm(int m, const double *x) {
    const int lane = threadIdx.x & 31;
    double d = 0.0;
    for (int b = 0; b < m; b += 32) {
        const double t = b + lane < m ? fabs(x[b + lane]) : 0.0;
        d = ordered_acc(d, t, m - b < 32 ? m - b : 32);
    }
    return d;
}

/* dot of a terminated line with `vec`, accumulated in storage order into acc (subtract or add) */
__device__ __forceinline__ double dev_line_dot(const int *idx, const double *val, int pos, const double *vec, double acc, bool subtract) {
    const int lane = threadIdx.x & 31;
    for (;; pos += 32) {
        const int r = idx[pos + lane];
        const unsigned tm = __ballot_sync(FULLMASK, r < 0);
        const int nvalid = tm ? __ffs((int)tm) - 1 : 32;
        const double term = lane < nvalid ? __dmul_rn(vec[r], val[pos + lane]) : 0.0;
        acc = subtract ? ordered_sub(acc, term, nvalid) : ordered_acc(acc, term, nvalid);
        if (tm) break;
    }
    return acc;
}
/* vec[idx] -= x * val down a terminated line */
__device__ __forceinline__ void dev_line_axpy(const int *idx, const double *val, int pos, double *vec, double x) {
    const int lane = threadIdx.x & 31;
    for (;; pos += 32) {
        const int r = idx[pos + lane];
        const unsigned tm = __ballot_sync(FULLMASK, r < 0);
        const int nvalid = tm ? __ffs((int)tm) - 1 : 32;
        if (lane < nvalid) vec[r] = __dsub_rn(vec[r], __dmul_rn(x, val[pos + lane]));
        if (tm) break;
    }
}

/* The same two line kernels when the length is known: no load feeds the loop condition, and the
 * (idx, val, vec[idx]) of the next chunk are requested before the current chunk is summed. */
__device__ __forceinline__ double dev_line_dot_n(const int *idx, const double *val, int pos, int len, const double *vec,
                                                 double acc, bool subtract) {
    const int lane = threadIdx.x & 31;
    double term = 0.0;
    if (lane < len) term = __dmul_rn(vec[idx[pos + lane]], val[pos + lane]);
    for (int c = 0; c < len; c += 32) {
        double nterm = 0.0;
        const int q = c + 32 + lane;
        if (q < len) nterm = __dmul_rn(vec[idx[pos + q]], val[pos + q]);
        const int n = len - c < 32 ? len - c : 32;
        acc = subtract ? ordered_sub(acc, term, n) : ordered_acc(acc, term, n);
        term = nterm;
    }
    return acc;
}
__device__ __forceinline__ void dev_line_axpy_n(const int *idx, const double *val, int pos, int len, double *vec, double x) {
    const int lane = threadIdx.x & 31;
    #pragma unroll 4
    for (int q = lane; q < len; q += 32) {
        const int r = idx[pos + q];
        vec[r] = __dsub_rn(vec[r], __dmul_rn(x, val[pos + q]));
    }
}
/* start pulling a whole line (indices and values) into L2 */
__device__ __forceinline__ void dev_line_prefetch(const int *idx, const double *val, int pos, int len) {
    if (len > 16) { warp_prefetch_l2(idx + pos, len * 4); warp_prefetch_l2(val + pos, len * 8); }
}

/* lu/condest.rs:15-157 for one triangular factor stored as terminated lines begin[j] */
__device__ double dev_condest(int m, const int *begin, const int *idx, const double *val, const double *pivot,
                              const int *perm, bool upper, const int *dep, const int *lens, const int *lptr, const int *rowdep, const int *rowptr, const int *rowidx, const double *rowval, double *work, double *norm, double *norminv) {
    const int lane = threadIdx.x & 31;
    /* 1-norm: every lane sums whole columns serially (storage order), the maximum is order-free */
    double u_norm = 0.0;
    if (dep) {
        /* lengths are known: short columns one lane each with all loads in flight, long ones by the warp */
        for (int s = 0; s < m; s += 32) {
            const int k = s + lane;
            const bool ok = k < m;
            const int j = ok ? perm[k] : 0;
            const int b = ok ? begin[j] : 0;
            const int len = !ok ? 0 : (lens ? lens[k] : lptr[k + 1] - lptr[k] - 1);
            double colsum = !ok ? 0.0 : (pivot ? fabs(pivot[j]) : 1.0);
            if (len <= SWEEP_SHORT) {
                double v[SWEEP_SHORT];
                #pragma unroll
                for (int q = 0; q < SWEEP_SHORT; q++) v[q] = q < len ? fabs(val[b + q]) : 0.0;
                #pragma unroll
                for (int q = 0; q < SWEEP_SHORT; q++) if (q < len) colsum = __dadd_rn(colsum, v[q]);
            }
            unsigned lg = __ballot_sync(FULLMASK, len > SWEEP_SHORT);
            while (lg) {
                const int t = __ffs((int)lg) - 1;
                lg &= lg - 1;
                const int bb = __shfl_sync(FULLMASK, b, t), ll = __shfl_sync(FULLMASK, len, t);
                double cs = __shfl_sync(FULLMASK, colsum, t);
                for (int c0 = 0; c0 < ll; c0 += 32) {
                    const double a = c0 + lane < ll ? fabs(val[bb + c0 + lane]) : 0.0;
                    cs = ordered_acc(cs, a, ll - c0 < 32 ? ll - c0 : 32);
                }
                if (lane == t) colsum = cs;
            }
            u_norm = fmax(u_norm, colsum);
        }
    } else
    for (int j = lane; j < m; j += 32) {
        double colsum = pivot ? fabs(pivot[j]) : 1.0;
        for (int p = begin[j]; idx[p] >= 0; p++) colsum = __dadd_rn(colsum, fabs(val[p]));
        u_norm = fmax(u_norm, colsum);
    }
    u_norm = warp_maxd(u_norm);
    __syncwarp();
    /* normest */
    double x1norm = 0.0, xinfnorm = 0.0, y1norm = 0.0;
    if (dep) {
        double mytemp = 0.0;
        dev_dot_sweep(m, upper, dep, idx, val, work, true,
                      [&](int k, int *b, int *len) { *b = begin[perm[k]]; *len = lens ? lens[k] : lptr[k + 1] - lptr[k] - 1; },
                      [&](int k, double temp) {
                          const int j = perm[k];
                          temp = __dadd_rn(temp, temp >= 0.0 ? 1.0 : -1.0);
                          if (pivot) temp = __ddiv_rn(temp, pivot[j]);
                          work[j] = temp;
                          mytemp = fabs(temp);
                      },
                      [&](int cnt) {
                          x1norm = ordered_acc(x1norm, mytemp, cnt);       /* sweep order == lane order */
                          double mx = (int)(threadIdx.x & 31) < cnt ? mytemp : 0.0;
                          xinfnorm = fmax(xinfnorm, warp_maxd(mx));
                      });
    } else
    for (int s = 0; s < m; s += 32) {
        const int kk = s + lane;
        const bool ok = kk < m;
        const int k = upper ? kk : m - 1 - kk;
        const int j = ok ? perm[k] : 0;
        const int b = ok ? begin[j] : 0;
        const double pv = (ok && pivot) ? pivot[j] : 1.0;
        if (ok) { lane_prefetch(idx + b); lane_prefetch(val + b); }
        const int cnt = m - s < 32 ? m - s : 32;
        for (int t = 0; t < cnt; t++) {
            const int jj = __shfl_sync(FULLMASK, j, t), bb = __shfl_sync(FULLMASK, b, t);
            const double pp = __shfl_sync(FULLMASK, pv, t);
            double temp = dev_line_dot(idx, val, bb, work, 0.0, true);
            temp = __dadd_rn(temp, temp >= 0.0 ? 1.0 : -1.0);
            if (pivot) temp = __ddiv_rn(temp, pp);
            if (lane == 0) work[jj] = temp;
            x1norm = __dadd_rn(x1norm, fabs(temp));
            xinfnorm = fmax(xinfnorm, fabs(temp));
            __syncwarp();
        }
    }
    if (dep && upper && rowdep) {
        /* U: the backward column-axpy sweep == for every pivot the dot with its ROW of U in descending
         * pivot order of the columns (ur_*), started from the pass-1 value, then the division */
        double mytemp = 0.0;
        dev_dot_sweep_init(m, false, rowdep, rowidx, rowval, work, true,
                           [&](int k, int *b, int *len) { *b = rowptr[k]; *len = rowptr[k + 1] - rowptr[k]; },
                           [&](int k) { return work[perm[k]]; },
                           [&](int k, double acc) { const int j = perm[k]; const double temp = __ddiv_rn(acc, pivot[j]); work[j] = temp; mytemp = fabs(temp); },
                           [&](int cnt) { y1norm = ordered_acc(y1norm, mytemp, cnt); });
    } else
    if (dep && !upper && rowdep) {
        /* L: the column-axpy sweep (ascending) == for every pivot the dot with its ROW of L (entries in
         * ascending pivot order by construction), started from the pass-1 value */
        double mytemp = 0.0;
        dev_dot_sweep_init(m, true, rowdep, idx, val, work, true,
                           [&](int k, int *b, int *len) { *b = rowptr[k]; *len = rowptr[k + 1] - rowptr[k] - 1; },
                           [&](int k) { return work[perm[k]]; },
                           [&](int k, double temp) { work[perm[k]] = temp; mytemp = fabs(temp); },
                           [&](int cnt) { y1norm = ordered_acc(y1norm, mytemp, cnt); });
    } else
    for (int s = 0; s < m; s += 32) {
        const int kk = s + lane;
        const bool ok = kk < m;
        const int k = upper ? m - 1 - kk : kk;
        const int j = ok ? perm[k] : 0;
        const int b = ok ? begin[j] : 0;
        const double pv = (ok && pivot) ? pivot[j] : 1.0;
        const int ln = (!ok || !dep) ? -1 : (lens ? lens[k] : lptr[k + 1] - lptr[k] - 1);
        if (ok) { lane_prefetch(idx + b); lane_prefetch(val + b); }
        const int cnt = m - s < 32 ? m - s : 32;
        for (int t = 0; t < cnt; t++) {
            const int jj = __shfl_sync(FULLMASK, j, t), bb = __shfl_sync(FULLMASK, b, t), ll = __shfl_sync(FULLMASK, ln, t);
            const double pp = __shfl_sync(FULLMASK, pv, t);
            if (dep && t + 1 < cnt) dev_line_prefetch(idx, val, __shfl_sync(FULLMASK, b, t + 1), __shfl_sync(FULLMASK, ln, t + 1));
            double temp = work[jj];
            __syncwarp();
            if (pivot) { temp = __ddiv_rn(temp, pp); if (lane == 0) work[jj] = temp; }
            if (ll >= 0) dev_line_axpy_n(idx, val, bb, ll, work, temp); else dev_line_axpy(idx, val, bb, work, temp);
            y1norm = __dadd_rn(y1norm, fabs(temp));
            __syncwarp();
        }
    }
    const double u_invnorm = fmax(__ddiv_rn(y1norm, x1norm), xinfnorm);
    *norm = u_norm; *norminv = u_invnorm;
    return __dmul_rn(u_norm, u_invnorm);
}

/* Forward residual and matrix norms over B (lu/residual_test.rs:60-74, lu/matrix_norm.rs:8-48).  The
 * reference walks the columns of B in pivot order and scatters into rhs / rowsum; here every ROW is
 * evaluated by its own lane from the row-wise copy of B, whose rows build_factors re-sorted by the
 * pivot position of the column -- the terms of a row arrive in the reference's order, so rhs, rowsum,
 * onenorm and infnorm are bit-identical, and all rows run in parallel. */
__device__ void dev_b_forward_pass(Mat &M, int rank, const double *lhs, double *rhs, double *rowsum,
                                   double *onenorm_out, double *infnorm_out) {
    const int m = M.m, lane = threadIdx.x & 31;
    (void)rowsum;
    double infnorm = 0.0;
    for (int i = lane; i < m; i += 32) {
        const int rb = M.bt_ptr[i], re = M.bt_ptr[i + 1];
        double acc = rhs[i], rs = 0.0;
        #pragma unroll 4
        for (int pos = rb; pos < re; pos++) {
            const int j = M.bt_idx[pos];
            const double x = M.bt_val[pos];
            if (M.qrank[j] < rank) {
                acc = __dsub_rn(acc, __dmul_rn(lhs[M.pinv[j]], x));      /* pinv == pmap after build_factors */
                rs = __dadd_rn(rs, fabs(x));
            }
        }
        if (M.prank[i] >= rank) { rs = __dadd_rn(rs, 1.0); acc = __dsub_rn(acc, lhs[i]); }
        rhs[i] = acc;
        infnorm = fmax(infnorm, rs);
    }
    infnorm = warp_maxd(infnorm);
    double onenorm = 0.0;
    for (int k = lane; k < rank; k += 32) {
        const int jp = M.pivotcol[k];
        double colsum = 0.0;
        for (i64 pos = M.b_begin[jp]; pos < M.b_end[jp]; pos++) colsum = __dadd_rn(colsum, fabs(M.b_x[pos]));
        onenorm = fmax(onenorm, colsum);
    }
    onenorm = warp_maxd(onenorm);
    if (rank < m) onenorm = fmax(onenorm, 1.0);
    __syncwarp();
    *onenorm_out = onenorm; *infnorm_out = infnorm;
}

/* lu/residual_test.rs:26-74: forward system.  Returns the two 1-norms and (fused) the matrix norms. */
__device__ void dev_residual_forward(Mat &M, int rank, double *rhs, double *lhs, double *rowsum, double *out4) {
    const int m = M.m, lane = threadIdx.x & 31;
    i64 tq = clock64();
    dev_dot_sweep(m, true, M.dep_lt, M.l_idx, M.l_val, lhs, false,
                  [&](int k, int *b, int *len) { *b = M.lt_begin_p[k]; *len = M.lt_begin_p[k + 1] - *b - 1; },
                  [&](int k, double d) {
                      const int ii = M.p[k];
                      const double r = d <= 0.0 ? 1.0 : -1.0;
                      rhs[ii] = r; lhs[ii] = __dsub_rn(r, d);
                  }, NoBatchEnd());
    if (lane == 0) { M.info->norms_cycles[4] = clock64() - tq; } tq = clock64();
    if (M.ur_ptr && M.info->have_ur) {
        dev_dot_sweep_init(m, false, M.dep_ur, M.ur_idx, M.ur_val, lhs, true,
                           [&](int k, int *b, int *len) { *b = M.ur_ptr[k]; *len = M.ur_ptr[k + 1] - *b; },
                           [&](int k) { return lhs[M.pivotrow[k]]; },
                           [&](int k, double acc) { const int ip = M.pivotrow[k]; lhs[ip] = __ddiv_rn(acc, M.rowpiv[ip]); }, NoBatchEnd());
    } else
    for (int s = 0; s < m; s += 32) {
        const int k = m - 1 - (s + lane);
        const int ip = k >= 0 ? M.pivotrow[k] : 0;
        const int b = k >= 0 ? M.u_begin[ip] : 0;
        const double pv = k >= 0 ? M.rowpiv[ip] : 1.0;
        const int ln = k >= 0 ? M.len_uc[k] : 0;
        if (k >= 0) { lane_prefetch(M.u_idx + b); lane_prefetch(M.u_val + b); }
        const int cnt = m - s < 32 ? m - s : 32;
        for (int t = 0; t < cnt; t++) {
            const int bb = __shfl_sync(FULLMASK, b, t), ii = __shfl_sync(FULLMASK, ip, t), ll = __shfl_sync(FULLMASK, ln, t);
            const double pp = __shfl_sync(FULLMASK, pv, t);
            if (t + 1 < cnt) dev_line_prefetch(M.u_idx, M.u_val, __shfl_sync(FULLMASK, b, t + 1), __shfl_sync(FULLMASK, ln, t + 1));
            const double d = __ddiv_rn(lhs[ii], pp);
            __syncwarp();
            if (lane == 0) lhs[ii] = d;
            dev_line_axpy_n(M.u_idx, M.u_val, bb, ll, lhs, d);
            __syncwarp();
        }
    }
    if (lane == 0) { M.info->norms_cycles[5] = clock64() - tq; } tq = clock64();
    double onenorm, infnorm;
    dev_b_forward_pass(M, rank, lhs, rhs, rowsum, &onenorm, &infnorm);
    __syncwarp();
    if (lane == 0) { M.info->norms_cycles[6] = clock64() - tq; } tq = clock64();
    const double norm_ftran = dev_vec_onenorm(m, lhs);
    const double norm_ftran_res = dev_vec_onenorm(m, rhs);
    if (lane == 0) { M.info->norms_cycles[7] = clock64() - tq; }
    if (lane == 0) { out4[0] = norm_ftran; out4[1] = norm_ftran_res; out4[2] = onenorm; out4[3] = infnorm; }
}

/* lu/residual_test.rs:76-120: transposed system */
__device__ void dev_residual_transposed(Mat &M, int rank, double *rhs, double *lhs, double *out2) {
    const int m = M.m, lane = threadIdx.x & 31;
    dev_dot_sweep(m, true, M.dep_uc, M.u_idx, M.u_val, lhs, false,
                  [&](int k, int *b, int *len) { *b = M.u_begin[M.pivotrow[k]]; *len = M.len_uc[k]; },
                  [&](int k, double d) {
                      const int ii = M.pivotrow[k];
                      const double r = d <= 0.0 ? 1.0 : -1.0;
                      rhs[ii] = r; lhs[ii] = __ddiv_rn(__dsub_rn(r, d), M.rowpiv[ii]);
                  }, NoBatchEnd());
    dev_dot_sweep(m, false, M.dep_lc, M.l_idx, M.l_val, lhs, false,
                  [&](int k, int *b, int *len) { *b = M.l_begin_p[k]; *len = M.l_begin_p[k + 1] - *b - 1; },
                  [&](int k, double d) { const int ii = M.p[k]; lhs[ii] = __dsub_rn(lhs[ii], d); }, NoBatchEnd());
    /* rhs[ipivot] -= B[:,jpivot] . lhs: the columns are independent, one lane per column, each dot in
     * storage order (residual_test.rs:104-113) */
    for (int k = lane; k < rank; k += 32) {
        const int ip = M.pivotrow[k], jp = M.pivotcol[k];
        double d = 0.0;
        for (i64 pos = M.b_begin[jp]; pos < M.b_end[jp]; pos++) d = __dadd_rn(d, __dmul_rn(lhs[(int)M.b_i[pos]], M.b_x[pos]));
        rhs[ip] = __dsub_rn(rhs[ip], d);
    }
    for (int k = rank + lane; k < m; k += 32) { const int ip = M.pivotrow[k]; rhs[ip] = __dsub_rn(rhs[ip], lhs[ip]); }
    __syncwarp();
    const double norm_btran = dev_vec_onenorm(m, lhs);
    const double norm_btran_res = dev_vec_onenorm(m, rhs);
    if (lane == 0) { out2[0] = norm_btran; out2[1] = norm_btran_res; }
}

/* One CTA of four warps per basis; the four pieces are independent and run side by side:
 * warp 0 condest(L), warp 1 condest(U), warp 2 forward residual + matrix norms, warp 3 transposed
 * residual.  Scratch: seven m-vectors in the per-warp scatter space gwork[1..7] (slice 0 is the
 * all-zero solution scratch of the sparse solves), zeroed again at the end because the pivot
 * kernels expect that space to be all-zero. */
#ifndef NORMS_MINB
#define NORMS_MINB 9    /* 9, 12 and 16 CTAs/SM all measure 23 ms on configs[1] (DRAM-latency-bound sweeps); 9 spills least */
#endif
__global__ void __launch_bounds__(128, NORMS_MINB) k_factor_norms(BluDev D) {
    __shared__ Mat M;
    __shared__ double sres[8];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    for (int s = D.slot0 + blockIdx.x; s < D.slot0 + D.nslot; s += gridDim.x) {
        if (D.run && !D.run[s]) continue;      /* not refactorized by this (masked) factorization */
        __syncthreads();
        if (tid == 0) mat_view(M, D, s);
        __syncthreads();
        BluInfo *I = M.info;
        if (I->nupdate != 0 || (I->status != BLU_OK && I->status != BLU_WARNING_SINGULAR_MATRIX)) continue;
        const int m = M.m;
        const size_t mm = (size_t)m;
        double *v = M.gwork + mm;          /* slices 1..7 */
        const bool have_ur = M.ur_ptr && I->have_ur;
        const i64 tw0 = clock64();
        if (wid == 0) {
            double norm, norminv;
            const double c = dev_condest(m, M.l_begin, M.l_idx, M.l_val, nullptr, M.p, false, M.dep_lc, nullptr, M.l_begin_p, M.ur_ptr ? M.dep_lt : nullptr /* batch: tail-dominated factors, the column axpy is cheaper */, M.lt_begin_p, nullptr, nullptr, v, &norm, &norminv);
            if (lane == 0) { I->condest_l = c; I->norm_l = norm; I->normest_l_inv = norminv; }
        } else if (wid == 1) {
            double norm, norminv;
            const double c = dev_condest(m, M.u_begin, M.u_idx, M.u_val, M.rowpiv, M.p, true, M.dep_uc, M.len_uc, nullptr, have_ur ? M.dep_ur : nullptr, M.ur_ptr, M.ur_idx, M.ur_val, v + mm, &norm, &norminv);
            if (lane == 0) { I->condest_u = c; I->norm_u = norm; I->normest_u_inv = norminv; }
        } else if (wid == 2) {
            dev_residual_forward(M, I->rank, v + 2 * mm, v + 3 * mm, v + 4 * mm, sres);
        } else {
            dev_residual_transposed(M, I->rank, v + 5 * mm, v + 6 * mm, sres + 4);
        }
        if (lane == 0) I->norms_cycles[wid] = clock64() - tw0;
        __syncthreads();
        if (tid == 0) {
            const double onenorm = sres[2], infnorm = sres[3];
            I->onenorm = onenorm; I->infnorm = infnorm;
            const double a = __ddiv_rn(sres[1], __dadd_rn((double)m, __dmul_rn(onenorm, sres[0])));
            const double b2 = __ddiv_rn(sres[5], __dadd_rn((double)m, __dmul_rn(infnorm, sres[4])));
            I->residual_test = fmax(a, b2);
        }
        for (size_t i = tid; i < 7 * mm; i += 128) v[i] = 0.0;
    }
}

/* Object API: U row-wise with every row in descending pivot order of the column (see blu_types.h).
 * Counting in parallel, then one ordered scatter that walks the columns of U from the last pivot to the
 * first -- the order in which the reference's backward sweep visits them.  One CTA. */
__global__ void __launch_bounds__(256) k_build_ur(BluDev D) {
    __shared__ Mat M;
    __shared__ int iscr[40];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) mat_view(M, D, 0);
    __syncthreads();
    BluInfo *I = M.info;
    const int m = M.m;
    if (!M.ur_ptr || I->nupdate != 0 || (I->status != BLU_OK && I->status != BLU_WARNING_SINGULAR_MATRIX)) return;
    int *cnt = M.ur_ptr, *fill = M.tmpi;
    for (int k = tid; k <= m; k += 256) cnt[k] = 0;
    __syncthreads();
    for (int k = tid; k < m; k += 256)
        for (int pos = M.u_begin[M.pivotrow[k]]; M.u_idx[pos] >= 0; pos++) atomicAdd(&cnt[M.prank[M.u_idx[pos]]], 1);
    __syncthreads();
    int put = 0;
    for (int base = 0; base < m; base += 256) {
        const int k = base + tid;
        const int c = k < m ? cnt[k] : 0;
        int tot;
        const int ex = block_excl_scan<256>(c, &tot, iscr);
        __syncthreads();
        if (k < m) { cnt[k] = put + ex; fill[k] = put + ex; }
        put += tot;
    }
    if (tid == 0) cnt[m] = put;
    __syncthreads();
    if (wid == 0) {
        for (int s = 0; s < m; s += 32) {
            const int k = m - 1 - (s + lane);
            const int ip = k >= 0 ? M.pivotrow[k] : 0;
            const int b = k >= 0 ? M.u_begin[ip] : 0;
            const int ln = k >= 0 ? M.len_uc[k] : 0;
            const int n = m - s < 32 ? m - s : 32;
            for (int t = 0; t < n; t++) {
                const int bb = __shfl_sync(FULLMASK, b, t), ll = __shfl_sync(FULLMASK, ln, t), ii = __shfl_sync(FULLMASK, ip, t);
                for (int q = lane; q < ll; q += 32) {
                    const int kk = M.prank[M.u_idx[bb + q]];      /* rows of one column are distinct: no conflict */
                    const int dst = fill[kk]; fill[kk] = dst + 1;
                    M.ur_idx[dst] = ii; M.ur_val[dst] = M.u_val[bb + q];
                }
                __syncwarp();
            }
        }
    }
    __syncthreads();
    for (int k = tid; k < m; k += 256) {
        const int e = M.ur_ptr[k + 1];
        M.dep_ur[k] = e > M.ur_ptr[k] ? M.prank[M.ur_idx[e - 1]] : m;    /* the closest later pivot the row reaches */
    }
    __syncthreads();
    if (tid == 0) I->have_ur = 1;
}
#endif
