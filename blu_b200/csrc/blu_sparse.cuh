/* blu_sparse.cuh -- sparse solves, solve_for_update and the Forrest-Tomlin update on the
 * device.  Reference: src/lu/{dfs,solve_symbolic,solve_triangular,solve_sparse,
 * solve_for_update,update}.rs and the argument checks of src/{solve_sparse,
 * solve_for_update,update}.rs.
 *
 * One warp per call.  What is sequential in the reference and decides the output keeps its order:
 * the depth-first reach (whose finishing order IS the order of ilhs) is walked with the reference's
 * control flow, but the whole warp probes 32 edges at a time for "first neighbour not marked yet"
 * (sp_dfs_warp); the breadth-first path search and the permutation of update() run on lane 0.
 * Everything that is a sweep over a line (axpy down a column, scans for an index, gathers/scatters of a
 * pattern, compaction) is shared by the 32 lanes with ballot/prefix ordering so that in-line storage
 * order -- which the next DFS depends on -- is exactly the reference's.  Floating point: one rounding
 * per multiply and per add/subtract (no FMA) and sums accumulated in the reference's order, so values
 * are bit-identical to the sequential code.
 *
 * The row file of U lives in W as lines (lbeg,lend,lcap)[j], j < m, inside the live half
 * of W (info->w_half); "the line has no room" (w_end[j] == w_begin[next], update.rs:524)
 * is lend[j] == lcap[j]; file_reappend (file.rs:137) is a bump allocation at info->w_used;
 * file_compress (file.rs:92) copies the lines to the other half.
 *
 * Scratch (all dead after factorize): pattern_symb = iwork1[0..m), pattern = iwork1[m..2m),
 * marked[m], pstack[m], irhs32 = acols[m], ilhs32 = tmpi[0..m), work = work0[m] (all-zero
 * between calls), work1[m], xlhs = gwork[0..m) (all-zero between calls).
 */
#ifndef BLU_SPARSE_CUH
#define BLU_SPARSE_CUH
#include "blu_dev_common.cuh"
#include "blu_solve.cuh"

#define SP_GAP (-1)
#define SP_FLIP(i) (-(i) - 1)

/* per-call state */
struct SpCtx {
    Mat M;
    int m, status;
    int *pattern_symb, *pattern, *marked, *pstack, *pend, *irhs, *ilhs;
    int *marker_ptr;          /* the marker counter that goes with `marked` (the object's, or this unit's in a multi-RHS call) */
    double *work, *xlhs;
    i64 l_flops, u_flops, r_flops;
};

__device__ __forceinline__ int sp_bcast(int v) { return __shfl_sync(FULLMASK, v, 0); }
__device__ __forceinline__ double sp_bcastd(double v) { return __shfl_sync(FULLMASK, v, 0); }

/* acc (+|-)= term of lanes 0..n-1 in lane order, one rounding per step: the value the
 * reference's sequential loop produces. */
__device__ __forceinline__ double sp_ordered_acc(double acc, double term, int n, bool subtract) {
    return subtract ? ordered_sub(acc, term, n) : ordered_acc(acc, term, n);
}

/* update.rs:26-42 with an explicit end: position of j in [start,end) or end.  Warp, uniform. */
__device__ __forceinline__ int sp_find(int j, const int *index, int start, int end) {
    const int lane = threadIdx.x & 31;
    for (int b = start; b < end; b += 32) {
        int q = b + lane;
        unsigned hm = __ballot_sync(FULLMASK, q < end && index[q] == j);
        if (hm) return b + __ffs((int)hm) - 1;
    }
    return end;
}
/* terminated line: position of j (or -1); *term_pos = position of the terminator.  Warp, uniform. */
__device__ __forceinline__ int sp_find_term(int j, const int *index, int start, int *term_pos) {
    const int lane = threadIdx.x & 31;
    int where = -1;
    for (int b = start;; b += 32) {
        int idx = index[b + lane];
        unsigned tm = __ballot_sync(FULLMASK, idx < 0);
        int nvalid = tm ? __ffs((int)tm) - 1 : 32;
        unsigned hm = __ballot_sync(FULLMASK, lane < nvalid && idx == j);
        if (hm && where < 0) where = b + __ffs((int)hm) - 1;
        if (tm) { *term_pos = b + nvalid; break; }
    }
    return where;
}
/* the same two searches for one thread */
__device__ __forceinline__ int sp_find1(int j, const int *index, int start, int end) {
    while (start < end && index[start] != j) start++;
    return start;
}
__device__ __forceinline__ int sp_find_term1(int j, const int *index, int start) {
    while (index[start] != j && index[start] >= 0) start++;
    return index[start] == j ? start : -1;
}

/* dfs.rs:25-145; sequential, one thread.  end == nullptr: lists end at a negative index. */
__device__ int sp_dfs(int i, const int *begin, const int *end, const int *index, int top,
                      int *xi, int *pstack, int *marked, int marker) {
    if (marked[i] == marker) return top;
    int head = 0;
    xi[0] = i;
    while (head >= 0) {
        i = xi[head];
        if (marked[i] != marker) {
            marked[i] = marker;
            pstack[head] = begin[i];
        }
        bool done = true;
        if (end) {
            const int e = end[i];
            for (int p = pstack[head]; p < e; p++) {
                int inext = index[p];
                if (marked[inext] == marker) continue;
                pstack[head] = p + 1;
                xi[++head] = inext;
                done = false;
                break;
            }
        } else {
            int inext;
            for (int p = pstack[head]; (inext = index[p]) >= 0; p++) {
                if (marked[inext] == marker) continue;
                pstack[head] = p + 1;
                xi[++head] = inext;
                done = false;
                break;
            }
        }
        if (done) {
            head--;
            xi[--top] = i;
        }
    }
    return top;
}

/* dfs.rs:25-145 run by the whole warp: the control flow is the sequential one (uniform in all lanes, the
 * stacks are written by lane 0), but "first neighbour that is not marked yet" is found 32 neighbours at
 * a time -- two dependent round trips per 32 edges instead of per edge.  Same visiting order, hence the
 * same finishing order, as sp_dfs. */
__device__ int sp_dfs_warp(int i, const int *begin, const int *end, const int *index, int top,
                           int *xi, int *pstack, int *pend, int *marked, int marker) {
    const int lane = threadIdx.x & 31;
    if (marked[i] == marker) return top;
    /* the node being scanned lives in registers (cur, p, e); the stacks xi / pstack / pend hold its
     * ancestors (node, resume position, line end), so a pop is one round trip */
    int head = 0, cur = i;
    int p = begin[cur], e = end ? end[cur] : 0x7fffffff;
    __syncwarp();
    if (lane == 0) marked[cur] = marker;
    __syncwarp();
    for (;;) {
        int found = -1, inext = -1;
        for (int q = p; q < e; q += 32) {
            const bool in = q + lane < e;
            const int idx = in ? index[q + lane] : -1;
            unsigned tm = 0; int nvalid = 32;
            if (!end) { tm = __ballot_sync(FULLMASK, idx < 0); nvalid = tm ? __ffs((int)tm) - 1 : 32; }
            const bool cand = in && lane < nvalid && marked[idx] != marker;
            const unsigned cm = __ballot_sync(FULLMASK, cand);
            if (cm) { const int l = __ffs((int)cm) - 1; found = q + l; inext = __shfl_sync(FULLMASK, idx, l); break; }
            if (tm) break;
        }
        if (found >= 0) {
            if (lane == 0) { xi[head] = cur; pstack[head] = found + 1; pend[head] = e; marked[inext] = marker; }
            head++;
            cur = inext;
            p = begin[cur]; e = end ? end[cur] : 0x7fffffff;
            __syncwarp();
        } else {
            top--;
            if (lane == 0) xi[top] = cur;
            head--;
            if (head < 0) break;
            __syncwarp();
            cur = xi[head]; p = pstack[head]; e = pend[head];
        }
    }
    __syncwarp();
    return top;
}

/* solve_symbolic.rs:19-40 */
__device__ __forceinline__ int sp_symbolic(int m, const int *begin, const int *end, const int *index,
                                           int nrhs, const int *irhs, int *xi, int *pstack, int *pend, int *marked, int marker) {
    int top = m;
    __syncwarp();
    for (int n = 0; n < nrhs; n++) {
        const int i = irhs[n];
        if (marked[i] != marker) top = sp_dfs_warp(i, begin, end, index, top, xi, pstack, pend, marked, marker);
        __syncwarp();
    }
    return top;
}

/* solve_triangular.rs:27-136.  Pattern order is a true dependency and is kept; the lanes
 * share each column.  Returns nz (uniform), adds to *flops. */
__device__ int sp_solve_triangular(int nz_symb, const int *pattern_symb, const int *begin, const int *end,
                                   const int *index, const double *value, const double *pivot,
                                   double droptol, double *lhs, int *pattern, i64 *flops) {
    const int lane = threadIdx.x & 31;
    int nz = 0; i64 fl = 0;
    for (int nb = 0; nb < nz_symb; nb += 32) {
        const int n = nb + lane;
        const bool ok = n < nz_symb;
        const int ip = ok ? pattern_symb[n] : 0;
        const int b = ok ? begin[ip] : 0;
        const int e = (ok && end) ? end[ip] : 0;
        const double pv = (ok && pivot) ? pivot[ip] : 1.0;
        if (ok) { lane_prefetch(index + b); lane_prefetch(value + b); }
        const int cnt = nz_symb - nb < 32 ? nz_symb - nb : 32;
        for (int t = 0; t < cnt; t++) {
            const int ii = __shfl_sync(FULLMASK, ip, t), bb = __shfl_sync(FULLMASK, b, t), ee = __shfl_sync(FULLMASK, e, t);
            const double pp = __shfl_sync(FULLMASK, pv, t);
            double x = lhs[ii];
            __syncwarp();      /* every lane has read lhs[ii] before lane 0 overwrites it below */
            if (x == 0.0) continue;
            if (pivot) { x = __ddiv_rn(x, pp); fl++; }
            if (end) {
                /* four chunks of the column in flight: the entries of a column hit distinct rows */
                for (int pos = bb + lane; pos < ee; pos += 128) {
                    int r[4]; double v[4], w[4];
                    #pragma unroll
                    for (int u = 0; u < 4; u++) { const int q = pos + 32 * u; r[u] = q < ee ? index[q] : -1; v[u] = q < ee ? value[q] : 0.0; }
                    #pragma unroll
                    for (int u = 0; u < 4; u++) w[u] = r[u] >= 0 ? lhs[r[u]] : 0.0;
                    #pragma unroll
                    for (int u = 0; u < 4; u++) if (r[u] >= 0) lhs[r[u]] = __dsub_rn(w[u], __dmul_rn(x, v[u]));
                }
                fl += ee - bb;
            } else {
                for (int pos = bb;; pos += 64) {
                    /* two chunks in flight (the stores carry >= 96 entries of slack behind the last line) */
                    const int r0 = index[pos + lane], r1 = index[pos + 32 + lane];
                    const double v0 = value[pos + lane], v1 = value[pos + 32 + lane];
                    const unsigned t0 = __ballot_sync(FULLMASK, r0 < 0);
                    const int n0 = t0 ? __ffs((int)t0) - 1 : 32;
                    const unsigned t1 = __ballot_sync(FULLMASK, r1 < 0);
                    const int n1 = t0 ? 0 : (t1 ? __ffs((int)t1) - 1 : 32);
                    const double w0 = lane < n0 ? lhs[r0] : 0.0, w1 = lane < n1 ? lhs[r1] : 0.0;
                    if (lane < n0) lhs[r0] = __dsub_rn(w0, __dmul_rn(x, v0));
                    if (lane < n1) lhs[r1] = __dsub_rn(w1, __dmul_rn(x, v1));
                    fl += n0 + n1;
                    if (t0 || t1) break;
                }
            }
            const bool keep = fabs(x) > droptol;
            if (lane == 0) {
                if (keep) { pattern[nz] = ii; if (pivot) lhs[ii] = x; }
                else lhs[ii] = 0.0;
            }
            nz += keep;
            __syncwarp();
        }
    }
    if (lane == 0) *flops += fl;
    return nz;
}

__device__ __forceinline__ int sp_next_marker(SpCtx &C) {
    int mk = 0;
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mk = ++*C.marker_ptr;
    mk = sp_bcast(mk);
    return mk;
}

/* lu/solve_sparse.rs:242-258: nodes whose value cancelled are un-marked so that the etas
 * can add them again.  In the pattern <=> value non-zero after the solve. */
__device__ __forceinline__ void sp_unmark_cancellation(SpCtx &C, int top, int nz, int nz_symb) {
    if (nz < nz_symb) {
        for (int t = top + (threadIdx.x & 31); t < C.m; t += 32) {
            int i = C.pattern_symb[t];
            if (C.work[i] == 0.0) C.marked[i]--;
        }
    }
    __syncwarp();
}

/* first half of a forward solve: L then the row etas (lu/solve_sparse.rs:196-277,
 * lu/solve_for_update.rs:246-326).  Result scattered in work, pattern in C.pattern[0..nz). */
__device__ int sp_ftran_head(SpCtx &C, int nrhs, const double *xrhs) {
    Mat &M = C.M;
    const int m = C.m, lane = threadIdx.x & 31;
    const int nforrest = M.info->nforrest;
    const int marker = sp_next_marker(C);
    const int top = sp_symbolic(m, M.l_begin, nullptr, M.l_idx, nrhs, C.irhs, C.pattern_symb, C.pstack, C.pend, C.marked, marker);
    const int nz_symb = m - top;
    for (int n = lane; n < nrhs; n += 32) C.work[C.irhs[n]] = xrhs[n];
    __syncwarp();
    int nz = sp_solve_triangular(nz_symb, C.pattern_symb + top, M.l_begin, nullptr, M.l_idx, M.l_val, nullptr,
                                 M.prm.droptol, C.work, C.pattern, &C.l_flops);
    sp_unmark_cancellation(C, top, nz, nz_symb);
    for (int t = 0; t < nforrest; t++) {
        const int ipivot = M.eta_row[t];
        const int rb = M.r_begin[t], re = M.r_begin[t + 1];
        double x = 0.0;
        for (int b = rb; b < re; b += 32) {
            const int pos = b + lane;
            const double term = pos < re ? __dmul_rn(C.work[M.l_idx[pos]], M.l_val[pos]) : 0.0;
            x = sp_ordered_acc(x, term, re - b < 32 ? re - b : 32, false);
        }
        int app = 0;
        if (lane == 0) {
            C.work[ipivot] = __dsub_rn(C.work[ipivot], x);
            if (x != 0.0 && C.marked[ipivot] != marker) { C.marked[ipivot] = marker; C.pattern[nz] = ipivot; app = 1; }
        }
        nz += sp_bcast(app);
        __syncwarp();
    }
    if (lane == 0) C.r_flops += M.r_begin[nforrest] - M.r_begin[0];
    return nz;
}

/* second half of a forward solve: U (lu/solve_sparse.rs:279-349, lu/solve_for_update.rs:363-433).
 * Result in C.xlhs scattered by column index, pattern in C.ilhs[0..nz). */
__device__ int sp_ftran_tail(SpCtx &C, int nz) {
    Mat &M = C.M;
    const int m = C.m, lane = threadIdx.x & 31;
    const int nz_sparse = (int)(M.prm.sparse_thres * (double)m);
    const double droptol = M.prm.droptol;
    if (nz <= nz_sparse) {
        const int mk = sp_next_marker(C);
        const int top = sp_symbolic(m, M.u_begin, nullptr, M.u_idx, nz, C.pattern, C.pattern_symb, C.pstack, C.pend, C.marked, mk);
        nz = sp_solve_triangular(m - top, C.pattern_symb + top, M.u_begin, nullptr, M.u_idx, M.u_val, M.rowpiv,
                                 droptol, C.work, C.ilhs, &C.u_flops);
        for (int n = lane; n < nz; n += 32) {
            const int i = C.ilhs[n], j = M.qinv[i];   /* qmap */
            C.ilhs[n] = j;
            C.xlhs[j] = C.work[i];
            C.work[i] = 0.0;
        }
        __syncwarp();
    } else {
        nz = 0;
        i64 fl = 0;
        const int pivotlen = M.info->pivotlen;
        for (int kb = ((pivotlen - 1) / 32) * 32; kb >= 0; kb -= 32) {
            const int k = kb + lane;
            const bool ok = k < pivotlen;
            const int ip = ok ? M.pivotrow[k] : 0, jp = ok ? M.pivotcol[k] : 0;
            const int b = ok ? M.u_begin[ip] : 0;
            const double pv = ok ? M.rowpiv[ip] : 1.0;
            if (ok) { lane_prefetch(M.u_idx + b); lane_prefetch(M.u_val + b); }
            /* The reference tests work[ipivot] pivot by pivot; here the 32 values of the batch are fetched
             * together and only the non-zero ones are visited, in sweep order.  Zeros ahead of the next
             * non-zero cannot change any more (nothing was applied in between); after every applied column
             * the values still pending are fetched again. */
            unsigned pend = __ballot_sync(FULLMASK, ok);
            double wl = ok ? C.work[ip] : 0.0;
            for (;;) {
                const unsigned nzm = __ballot_sync(FULLMASK, wl != 0.0) & pend;
                if (!nzm) break;
                const int t = 31 - __clz((int)nzm);
                pend &= (1u << t) - 1u;
                const int ii = __shfl_sync(FULLMASK, ip, t), jj = __shfl_sync(FULLMASK, jp, t), bb = __shfl_sync(FULLMASK, b, t);
                const double pp = __shfl_sync(FULLMASK, pv, t);
                const double w = __shfl_sync(FULLMASK, wl, t);
                const double x = __ddiv_rn(w, pp);
                if (lane == 0) C.work[ii] = 0.0;
                for (int pos = bb;; pos += 32) {
                    const int r = M.u_idx[pos + lane];
                    const unsigned tm = __ballot_sync(FULLMASK, r < 0);
                    const int nvalid = tm ? __ffs((int)tm) - 1 : 32;
                    if (lane < nvalid) C.work[r] = __dsub_rn(C.work[r], __dmul_rn(x, M.u_val[pos + lane]));
                    fl += nvalid;
                    if (tm) break;
                }
                if (fabs(x) > droptol) {
                    if (lane == 0) { C.ilhs[nz] = jj; C.xlhs[jj] = x; }
                    nz++;
                }
                __syncwarp();
                wl = ((pend >> lane) & 1u) ? C.work[ip] : 0.0;
            }
        }
        if (lane == 0) C.u_flops += fl;
    }
    return nz;
}

/* second half of a transposed solve: etas backwards, then L' (lu/solve_sparse.rs:113-192,
 * lu/solve_for_update.rs:166-245).  In: xlhs scattered with pattern C.pattern[0..nz) marked
 * with `marker`.  Out: pattern in C.ilhs. */
__device__ int sp_btran_tail(SpCtx &C, int nz, int marker) {
    Mat &M = C.M;
    const int m = C.m, lane = threadIdx.x & 31;
    const int nforrest = M.info->nforrest;
    const int nz_sparse = (int)(M.prm.sparse_thres * (double)m);
    const double droptol = M.prm.droptol;
    for (int t = nforrest - 1; t >= 0; t--) {
        const int ipivot = M.eta_row[t];
        const double x = C.xlhs[ipivot];
        __syncwarp();
        if (x == 0.0) continue;
        const int rb = M.r_begin[t], re = M.r_begin[t + 1];
        for (int b = rb; b < re; b += 32) {
            const int pos = b + lane;
            const bool ok = pos < re;
            const int i = ok ? M.l_idx[pos] : 0;
            const bool fresh = ok && C.marked[i] != marker;
            const unsigned fm = __ballot_sync(FULLMASK, fresh);
            if (fresh) { C.marked[i] = marker; C.pattern[nz + __popc(fm & lanemask_lt())] = i; }
            if (ok) C.xlhs[i] = __dsub_rn(C.xlhs[i], __dmul_rn(x, M.l_val[pos]));
            nz += __popc(fm);
        }
        if (lane == 0) C.r_flops += re - rb;
        __syncwarp();
    }
    if (nz <= nz_sparse) {
        const int mk = sp_next_marker(C);
        const int top = sp_symbolic(m, M.lt_begin, nullptr, M.l_idx, nz, C.pattern, C.pattern_symb, C.pstack, C.pend, C.marked, mk);
        nz = sp_solve_triangular(m - top, C.pattern_symb + top, M.lt_begin, nullptr, M.l_idx, M.l_val, nullptr,
                                 droptol, C.xlhs, C.ilhs, &C.l_flops);
    } else {
        nz = 0;
        i64 fl = 0;
        for (int kb = ((m - 1) / 32) * 32; kb >= 0; kb -= 32) {
            const int k = kb + lane;
            const bool ok = k < m;
            const int ip = ok ? M.p[k] : 0;
            const int b = ok ? M.lt_begin_p[k] : 0;
            if (ok) { lane_prefetch(M.l_idx + b); lane_prefetch(M.l_val + b); }
            unsigned pend = __ballot_sync(FULLMASK, ok);
            double wl = ok ? C.xlhs[ip] : 0.0;
            for (;;) {
                const unsigned nzm = __ballot_sync(FULLMASK, wl != 0.0) & pend;
                if (!nzm) break;
                const int t = 31 - __clz((int)nzm);
                pend &= (1u << t) - 1u;
                const int ii = __shfl_sync(FULLMASK, ip, t), bb = __shfl_sync(FULLMASK, b, t);
                const double x = __shfl_sync(FULLMASK, wl, t);
                for (int pos = bb;; pos += 32) {
                    const int r = M.l_idx[pos + lane];
                    const unsigned tm = __ballot_sync(FULLMASK, r < 0);
                    const int nvalid = tm ? __ffs((int)tm) - 1 : 32;
                    if (lane < nvalid) C.xlhs[r] = __dsub_rn(C.xlhs[r], __dmul_rn(x, M.l_val[pos + lane]));
                    fl += nvalid;
                    if (tm) break;
                }
                if (fabs(x) > droptol) { if (lane == 0) C.ilhs[nz] = ii; nz++; }
                else if (lane == 0) C.xlhs[ii] = 0.0;
                __syncwarp();
                wl = ((pend >> lane) & 1u) ? C.xlhs[ip] : 0.0;
            }
        }
        if (lane == 0) C.l_flops += fl;
    }
    return nz;
}

__device__ __forceinline__ void sp_ctx_init(SpCtx &C, const BluDev &D, int slot = 0) {
    mat_view(C.M, D, slot);
    Mat &M = C.M;
    C.m = M.m; C.status = BLU_OK;
    C.pattern_symb = M.iwork1; C.pattern = M.iwork1 + M.m;
    C.marked = M.marked; C.pstack = M.pstack; C.pend = M.tmpi + M.m; C.irhs = M.acols; C.ilhs = M.tmpi;
    C.work = M.work0; C.xlhs = M.gwork;
    C.marker_ptr = &M.info->marker;
    C.l_flops = C.u_flops = C.r_flops = 0;
}

/* lu/solve_sparse.rs:356-358 and the update-cost model (lu.rs:321-326) */
/* The units of a k_solve_sparse launch.  k_solve_sparse<false>: unit u is basis u of a batch, on that basis' own
 * scratch.  k_solve_sparse<true>: every unit (right-hand side) has its own marks, stacks, patterns and the two
 * scattered vectors, so that all units run at once against the same (read-only) factors. */
struct SpMulti {
    int nunits;               /* 0: one right-hand side on the basis in slot 0 (the object calls) */
    int rerun;                /* 1: only the units whose previous status was Reallocate run again */
    const i64 *rhs_begin;     /* nunits + 1 offsets into irhs64 / xrhs */
    const i64 *rhs_end;       /* null, or nunits end offsets: unit u's right-hand side is [rhs_begin[u], rhs_end[u]) (columns of a resident pool) */
    /* k_solve_sparse<true> only (blu_batch_solve_sparse and its _dev variant): */
    int *ints;                /* nunits * 7m : marked | pattern_symb | pattern | pstack | ilhs | pend | irhs */
    double *dbls;             /* nunits * 2m : work | xlhs  (all-zero between calls) */
    int *markers;             /* nunits */
    const int *unit_slot;     /* unit u reads the factors of slot unit_slot[u] */
    blu_u64 *pack_fill;       /* unit u reserves nz entries of ilhs_out / xout at *pack_fill (the chunk's solutions back to back, */
    i64 *pack_off;            /* for one short copy) and records where they start in pack_off[u] */
    int row_stride;           /* 0: packed as above; m: unit u writes at ilhs_out / xout + u*m instead (rows of a full copy) */
};
__device__ __forceinline__ void sp_ctx_init_unit(SpCtx &C, const BluDev &D, const SpMulti &W, int u, int slot) {
    mat_view(C.M, D, slot);
    const size_t m = (size_t)C.M.m;
    C.m = C.M.m; C.status = BLU_OK;
    int *ib = W.ints + (size_t)u * 7 * m;
    C.marked = ib; C.pattern_symb = ib + m; C.pattern = ib + 2 * m; C.pstack = ib + 3 * m;
    C.ilhs = ib + 4 * m; C.pend = ib + 5 * m; C.irhs = ib + 6 * m;
    C.work = W.dbls + (size_t)u * 2 * m; C.xlhs = C.work + m;
    C.marker_ptr = W.markers + u;
    C.l_flops = C.u_flops = C.r_flops = 0;
}
__device__ __forceinline__ void sp_solve_done_atomic(SpCtx &C) {
    BluInfo *I = C.M.info;
    atomicAdd((unsigned long long *)&I->l_flops, (unsigned long long)C.l_flops);
    atomicAdd((unsigned long long *)&I->u_flops, (unsigned long long)C.u_flops);
    atomicAdd((unsigned long long *)&I->r_flops, (unsigned long long)C.r_flops);
    atomicAdd(&I->update_cost_numer, (double)C.r_flops);
}
__device__ __forceinline__ void sp_solve_done(SpCtx &C) {
    BluInfo *I = C.M.info;
    I->l_flops += C.l_flops; I->u_flops += C.u_flops; I->r_flops += C.r_flops;
    I->update_cost_numer += (double)C.r_flops;
}

/* solve_sparse (solve_sparse.rs:35-73 + lu/solve_sparse.rs:11-360) and solve_for_update
 * (solve_for_update.rs:72-119 + lu/solve_for_update.rs:12-455).
 * scal[0] = status, scal[1] = nzlhs.  The solution leaves compacted: ilhs_out[n], xout[n].
 * Without SLOT_UNITS: W.nunits == 0, one right-hand side on slot 0; otherwise unit u is basis u of a batch, on that
 * basis' own scratch.  SLOT_UNITS: plain solves, unit u on scratch of its own that only reads the factors of slot
 * W.unit_slot[u], the solutions packed (blu_batch_solve_sparse) or, with W.row_stride, in rows of m (the object's
 * blu_solve_sparse_multi).  SLOT_UNITS is a template argument so that the
 * basis-change shapes compile without the unit shape. */
template <bool SLOT_UNITS = false>
__global__ void __launch_bounds__(32) k_solve_sparse(BluDev D, int nrhs, const i64 *irhs64, const double *xrhs, char trans,
                                                      int for_update, int want_solution, int *scal, i64 *ilhs_out, double *xout,
                                                      SpMulti W) {
    __shared__ SpCtx C;
    const int lane = threadIdx.x & 31;
    const bool units = SLOT_UNITS || W.nunits > 0;
    if (SLOT_UNITS) for_update = 0;              /* plain solves only: the solve_for_update paths drop out of this instance */
    if (units) {
        /* unit = blockIdx.x: its slice of the right-hand sides and of the outputs */
        const int u = blockIdx.x;
        if (!SLOT_UNITS && D.run && !D.run[u]) return;      /* masked out: neither its state nor its status word is touched */
        const i64 b = W.rhs_begin[u], e = W.rhs_end ? W.rhs_end[u] : W.rhs_begin[u + 1];
        irhs64 += b; if (xrhs) xrhs += b;
        nrhs = (e - b < 0 || e - b > 0x7fffffff) ? -1 : (int)(e - b);
        scal += 2 * u;
        const size_t stride = SLOT_UNITS ? (size_t)W.row_stride : (size_t)D.m;
        ilhs_out += (size_t)u * stride; xout += (size_t)u * stride;
        if (W.rerun && scal[0] != BLU_REALLOCATE) return;
        if (lane == 0) { if (SLOT_UNITS) sp_ctx_init_unit(C, D, W, u, W.unit_slot[u]); else sp_ctx_init(C, D, u); }
    } else if (lane == 0) sp_ctx_init(C, D);
    __syncwarp();
    Mat &M = C.M;
    BluInfo *I = M.info;
    const int m = C.m;
    const bool tr = is_trans(trans);
    /* argument checks in the reference's order */
    int st = BLU_OK;
    if (for_update && !tr && !xrhs) st = BLU_ERROR_ARGUMENT_MISSING;          /* solve_for_update.rs:82-84 */
    else if (I->nupdate < 0) st = BLU_ERROR_INVALID_CALL;
    else if (for_update && I->nforrest == m) st = BLU_ERROR_MAXIMUM_UPDATES;   /* solve_for_update.rs:93-95 */
    else {
        int bad = 0;
        if (for_update && tr) {
            if (units && nrhs < 1) bad = 1;      /* an empty slice names no column to replace */
            else { i64 j = irhs64[0]; bad = j < 0 || j >= m; nrhs = 1; }
        }
        else if (nrhs < 0 || nrhs > m) bad = 1;
        else for (int n = lane; n < nrhs; n += 32) { i64 i = irhs64[n]; if (i < 0 || i >= m) bad = 1; }
        if (__any_sync(FULLMASK, bad)) st = BLU_ERROR_INVALID_ARGUMENT;
    }
    if (st != BLU_OK) { if (lane == 0) { scal[0] = st; scal[1] = 0; } return; }
    for (int n = lane; n < nrhs; n += 32) C.irhs[n] = (int)irhs64[n];
    if (lane == 0 && !SLOT_UNITS) I->addmem_l = I->addmem_u = I->addmem_w = 0;
    __syncwarp();

    int nz = 0;
    if (!for_update) {
        if (tr) {
            /* U' sparse, lu/solve_sparse.rs:68-111 */
            int marker = sp_next_marker(C);
            const int top = sp_symbolic(m, M.lbeg, M.lend, M.w_idx, nrhs, C.irhs, C.pattern_symb, C.pstack, C.pend, C.marked, marker);
            for (int n = lane; n < nrhs; n += 32) C.work[C.irhs[n]] = xrhs[n];
            __syncwarp();
            nz = sp_solve_triangular(m - top, C.pattern_symb + top, M.lbeg, M.lend, M.w_idx, M.w_val, M.colpiv,
                                     M.prm.droptol, C.work, C.pattern, &C.u_flops);
            marker = sp_next_marker(C);
            for (int n = lane; n < nz; n += 32) {
                const int j = C.pattern[n], i = M.pinv[j];   /* pmap */
                C.pattern[n] = i;
                C.xlhs[i] = C.work[j];
                C.work[j] = 0.0;
                C.marked[i] = marker;
            }
            __syncwarp();
            nz = sp_btran_tail(C, nz, marker);
        } else {
            nz = sp_ftran_head(C, nrhs, xrhs);
            nz = sp_ftran_tail(C, nz);
        }
    } else if (tr) {
        const int nforrest = I->nforrest;
        const int jpivot = C.irhs[0];
        const int ipivot = M.pinv[jpivot];
        const int jbegin = M.lbeg[jpivot], jend = M.lend[jpivot];
        /* row eta: U' solve seeded with row ipivot of U, nothing dropped; lu/solve_for_update.rs:70-120 */
        int marker = sp_next_marker(C);
        const int top = sp_symbolic(m, M.lbeg, M.lend, M.w_idx, jend - jbegin, M.w_idx + jbegin, C.pattern_symb, C.pstack, C.pend, C.marked, marker);
        const int nz_symb = m - top;
        const int room = M.l_mem - M.r_begin[nforrest];
        if (room < nz_symb) {
            if (lane == 0) { I->addmem_l = nz_symb - room; scal[0] = BLU_REALLOCATE; scal[1] = 0; }
            return;
        }
        for (int pos = jbegin + lane; pos < jend; pos += 32) C.work[M.w_idx[pos]] = M.w_val[pos];
        __syncwarp();
        sp_solve_triangular(nz_symb, C.pattern_symb + top, M.lbeg, M.lend, M.w_idx, M.w_val, M.colpiv, 0.0,
                            C.work, C.pattern, &C.u_flops);
        /* the symbolic pattern with its values becomes the row eta, :124-135 */
        const int rput = M.r_begin[nforrest];
        for (int t = top + lane; t < m; t += 32 * 4) {
            int jj[4], pi[4]; double wv[4];
            #pragma unroll
            for (int u = 0; u < 4; u++) { const int q = t + 32 * u; jj[u] = q < m ? C.pattern_symb[q] : -1; }
            #pragma unroll
            for (int u = 0; u < 4; u++) { pi[u] = jj[u] >= 0 ? M.pinv[jj[u]] : 0; wv[u] = jj[u] >= 0 ? C.work[jj[u]] : 0.0; }
            #pragma unroll
            for (int u = 0; u < 4; u++) if (jj[u] >= 0) {
                const int q = t + 32 * u;
                M.l_idx[rput + (q - top)] = pi[u];
                M.l_val[rput + (q - top)] = wv[u];
                C.work[jj[u]] = 0.0;
            }
        }
        if (lane == 0) { M.r_begin[nforrest + 1] = rput + nz_symb; M.eta_row[nforrest] = ipivot; I->btran_for_update = jpivot; }
        __syncwarp();
        if (want_solution) {
            /* scale to U^{-T} e_j, :144-165 */
            marker = sp_next_marker(C);
            const double pivot = M.colpiv[jpivot];
            const double xdrop = M.prm.droptol * fabs(pivot);
            if (lane == 0) { C.pattern[0] = ipivot; C.marked[ipivot] = marker; C.xlhs[ipivot] = __ddiv_rn(1.0, pivot); }
            nz = 1;
            for (int b = rput; b < rput + nz_symb; b += 32) {
                const int pos = b + lane;
                const bool ok = pos < rput + nz_symb;
                const double v = ok ? M.l_val[pos] : 0.0;
                const bool keep = ok && fabs(v) > xdrop;
                const unsigned km = __ballot_sync(FULLMASK, keep);
                if (keep) {
                    const int i = M.l_idx[pos];
                    C.pattern[nz + __popc(km & lanemask_lt())] = i;
                    C.marked[i] = marker;
                    C.xlhs[i] = __ddiv_rn(-v, pivot);
                }
                nz += __popc(km);
            }
            __syncwarp();
            nz = sp_btran_tail(C, nz, marker);
        }
    } else {
        nz = sp_ftran_head(C, nrhs, xrhs);
        /* spike into U at u_begin[m], lu/solve_for_update.rs:328-355 */
        const int put = M.u_begin[m];
        const int room = M.u_mem - put, need = nz + 1;
        if (room < need) {
            for (int n = lane; n < nz; n += 32) C.work[C.pattern[n]] = 0.0;
            if (lane == 0) { I->addmem_u = need - room; scal[0] = BLU_REALLOCATE; scal[1] = 0; }
            return;
        }
        for (int n = lane; n < nz; n += 32) {
            const int i = C.pattern[n];
            M.u_idx[put + n] = i;
            M.u_val[put + n] = C.work[i];
            if (!want_solution) C.work[i] = 0.0;
        }
        if (lane == 0) { M.u_idx[put + nz] = -1; I->ftran_for_update = 0; }
        __syncwarp();
        if (want_solution) nz = sp_ftran_tail(C, nz); else nz = 0;
    }
    if (for_update && !want_solution) nz = 0;
    if (SLOT_UNITS) {
        i64 base = 0;
        if (lane == 0) { base = (i64)atomicAdd((unsigned long long *)W.pack_fill, (unsigned long long)(W.row_stride ? 0 : nz)); W.pack_off[blockIdx.x] = base; }
        base = __shfl_sync(FULLMASK, base, 0);
        ilhs_out += base; xout += base;
    }
    /* hand the solution out compacted and leave xlhs all-zero again */
    for (int n = lane; n < nz; n += 32) {
        const int j = C.ilhs[n];
        ilhs_out[n] = j;
        xout[n] = C.xlhs[j];
        C.xlhs[j] = 0.0;
    }
    if (lane == 0) { if (SLOT_UNITS) sp_solve_done_atomic(C); else sp_solve_done(C); scal[0] = C.status; scal[1] = nz; }
}

/* ------------------------------------------------------------------ */
/* update, lu/update.rs                                                */
/* ------------------------------------------------------------------ */

/* update.rs:51-105: BFS for a cycle j0 -> ... -> j0 in the row-file graph; one thread */
__device__ int sp_bfs_path(int m, int j0, const int *begin, const int *end, const int *index,
                           int *jlist, int *marked, int *queue) {
    int j = -1, tail = 1, top = m;
    bool found = false;
    queue[0] = j0;
    for (int front = 0; front < tail && !found; front++) {
        j = queue[front];
        for (int pos = begin[j]; pos < end[j]; pos++) {
            int k = index[pos];
            if (k == j0) { found = true; break; }
            if (marked[k] >= 0) {
                marked[k] = SP_FLIP(j);
                queue[tail++] = k;
            }
        }
    }
    if (found) {
        while (j != j0) {
            jlist[--top] = j;
            j = SP_FLIP(marked[j]);
        }
        jlist[--top] = j0;
    }
    for (int pos = 0; pos < tail; pos++) marked[queue[pos]] = 0;
    return top;
}

/* update.rs:176-314; one thread.  jlist has nswap+1 entries. */
__device__ void sp_permute(SpCtx &C, const int *jlist, int nswap, double *pmin, double *pmax) {
    Mat &M = C.M;
    int *pmap = M.pinv, *qmap = M.qinv;
    const int j0 = jlist[0], jn = jlist[nswap];
    const int i0 = pmap[j0], in_ = pmap[jn];
    BLU_CHECK(C, nswap >= 1 && qmap[i0] == j0 && qmap[in_] == jn && M.rowpiv[i0] == 0.0 && M.colpiv[j0] == 0.0);
    /* row file */
    int begin = M.lbeg[jn], end = M.lend[jn], cap = M.lcap[jn];
    const double piv = M.colpiv[jn];
    for (int n = nswap; n > 0; n--) {
        const int j = jlist[n], jprev = jlist[n - 1];
        M.lbeg[j] = M.lbeg[jprev]; M.lend[j] = M.lend[jprev]; M.lcap[j] = M.lcap[jprev];
        int where = sp_find1(j, M.w_idx, M.lbeg[j], M.lend[j]);
        if (where >= M.lend[j]) { BLU_CHECK(C, 0); return; }
        if (n > 1) {
            M.w_idx[where] = jprev;
            M.colpiv[j] = M.w_val[where];
            M.w_val[where] = M.colpiv[jprev];
        } else {
            M.colpiv[j] = M.w_val[where];
            const int e = --M.lend[j];
            M.w_idx[where] = M.w_idx[e];
            M.w_val[where] = M.w_val[e];
        }
        BLU_CHECK(C, M.colpiv[j] != 0.0);
        *pmin = fmin(*pmin, fabs(M.colpiv[j])); *pmax = fmax(*pmax, fabs(M.colpiv[j]));
    }
    M.lbeg[j0] = begin; M.lend[j0] = end; M.lcap[j0] = cap;
    int where = sp_find1(j0, M.w_idx, begin, end);
    if (where >= end) { BLU_CHECK(C, 0); return; }
    M.w_idx[where] = jn;
    M.colpiv[j0] = M.w_val[where];
    BLU_CHECK(C, M.colpiv[j0] != 0.0);
    M.w_val[where] = piv;
    *pmin = fmin(*pmin, fabs(M.colpiv[j0])); *pmax = fmax(*pmax, fabs(M.colpiv[j0]));
    /* column file */
    begin = M.u_begin[i0];
    for (int n = 0; n < nswap; n++) {
        const int i = pmap[jlist[n]], inext = pmap[jlist[n + 1]];
        M.u_begin[i] = M.u_begin[inext];
        where = sp_find_term1(i, M.u_idx, M.u_begin[i]);
        if (where < 0) { BLU_CHECK(C, 0); return; }
        M.u_idx[where] = inext;
        M.rowpiv[i] = M.u_val[where];
        BLU_CHECK(C, M.rowpiv[i] != 0.0);
        M.u_val[where] = M.rowpiv[inext];
    }
    M.u_begin[in_] = begin;
    where = sp_find_term1(in_, M.u_idx, begin);
    if (where < 0) { BLU_CHECK(C, 0); return; }
    M.rowpiv[in_] = M.u_val[where];
    BLU_CHECK(C, M.rowpiv[in_] != 0.0);
    for (end = where; M.u_idx[end] >= 0; end++) ;
    M.u_idx[where] = M.u_idx[end - 1];
    M.u_val[where] = M.u_val[end - 1];
    M.u_idx[end - 1] = -1;
    /* mappings */
    for (int n = nswap; n > 0; n--) {
        const int j = jlist[n], i = pmap[jlist[n - 1]];
        pmap[j] = i;
        qmap[i] = j;
    }
    pmap[j0] = in_;
    qmap[in_] = j0;
}

/* role of file_compress (file.rs:92-135) for the row file of U: copy every line to the
 * other half of W with fresh slack.  Warp. */
__device__ void sp_w_compact(SpCtx &C) {
    Mat &M = C.M;
    BluInfo *I = M.info;
    const int m = C.m, lane = threadIdx.x & 31;
    const int nbase = (1 - I->w_half) * M.w_mem;
    int put = nbase;
    __syncwarp();
    /* fresh slack for every line if that fits, else none (the caller then asks for more memory) */
    i64 total = 0;
    for (int j = lane; j < m; j += 32) { const int nz = M.lend[j] - M.lbeg[j]; total += nz + slack_of(M.prm, nz); }
    total = warp_sum64(total);
    const bool with_slack = total <= (i64)M.w_mem;
    for (int jb = 0; jb < m; jb += 32) {
        const int j = jb + lane;
        const int ob = j < m ? M.lbeg[j] : 0;
        const int nz = j < m ? M.lend[j] - ob : 0;
        const int sz = j < m ? nz + (with_slack ? slack_of(M.prm, nz) : 0) : 0;
        const int incl = warp_incl_scan(sz);
        const int nb = put + incl - sz;
        /* lanes copy their own line; the regions are disjoint (other half) */
        for (int t = 0; t < nz; t++) { M.w_idx[nb + t] = M.w_idx[ob + t]; M.w_val[nb + t] = M.w_val[ob + t]; }
        if (j < m) { M.lbeg[j] = nb; M.lend[j] = nb + nz; M.lcap[j] = nb + sz; }
        put += __shfl_sync(FULLMASK, incl, 31);
    }
    __syncwarp();
    if (lane == 0) {
        BLU_CHECK(C, put - nbase <= M.w_mem);
        I->w_half = 1 - I->w_half;
        I->w_used = put;
        I->ngarbage++;
    }
    __syncwarp();
}

/* update.rs:115-162: squeeze the gaps out of the column file of U, in memory order.  Warp. */
__device__ int sp_compress_packed(SpCtx &C) {
    Mat &M = C.M;
    const int m = C.m, lane = threadIdx.x & 31;
    int *begin = M.u_begin, *index = M.u_idx; double *value = M.u_val;
    const int end = begin[m];
    __syncwarp();
    for (int i = lane; i < m; i += 32) {
        const int p = begin[i];
        const int first = index[p];
        if (first == SP_GAP) begin[i] = 0;
        else { begin[i] = first; index[p] = SP_GAP - i - 1; }
    }
    __syncwarp();
    int put = 1, nz = 0;
    int carry = SP_GAP;     /* original index[get-1] of the first lane; index[0] is a gap */
    for (int gb = 1; gb < end; gb += 32) {
        const int get = gb + lane;
        const bool ok = get < end;
        const int idx = ok ? index[get] : SP_GAP;
        const double val = ok ? value[get] : 0.0;
        int prev = __shfl_up_sync(FULLMASK, idx, 1);
        if (lane == 0) prev = carry;
        carry = __shfl_sync(FULLMASK, idx, 31);
        const bool keep = ok && (idx != SP_GAP || prev != SP_GAP);
        const unsigned km = __ballot_sync(FULLMASK, keep);
        const int dst = put + __popc(km & lanemask_lt());
        __syncwarp();
        if (keep) {
            if (idx > SP_GAP) { index[dst] = idx; value[dst] = val; }
            else if (idx < SP_GAP) {
                const int i = SP_GAP - idx - 1;
                index[dst] = begin[i];
                begin[i] = dst;
                value[dst] = val;
            } else index[dst] = SP_GAP;
        }
        nz += __popc(__ballot_sync(FULLMASK, keep && idx != SP_GAP));
        put += __popc(km);
        __syncwarp();
    }
    if (lane == 0) begin[m] = put;
    __syncwarp();
    return nz;
}

/* update.rs:49-55 + lu/update.rs:388-959.  scal[0] = status. */
__global__ void __launch_bounds__(32) k_update(BluDev D, double xtbl, int *scal, const double *xtbl_per_slot, int rerun) {
    __shared__ SpCtx C;
    const int lane = threadIdx.x & 31;
    /* object API: one block, slot 0.  Batch: block u updates basis u with its own xtbl and status word. */
    const int slot = xtbl_per_slot ? (int)blockIdx.x : 0;
    if (xtbl_per_slot && D.run && !D.run[slot]) return;      /* masked out: state and status word untouched */
    if (xtbl_per_slot) { xtbl = xtbl_per_slot[slot]; scal += slot; }
    if (rerun && scal[0] != BLU_REALLOCATE) return;      /* batch re-run after a store was grown: only the bases that asked */
    if (lane == 0) sp_ctx_init(C, D, slot);
    __syncwarp();
    Mat &M = C.M;
    BluInfo *I = M.info;
    const int m = C.m;
    if (I->nupdate < 0 || I->ftran_for_update < 0 || I->btran_for_update < 0) {
        if (lane == 0) scal[0] = BLU_ERROR_INVALID_CALL;
        return;
    }
    if (lane == 0) I->addmem_l = I->addmem_u = I->addmem_w = 0;
    const int nforrest = I->nforrest;
    const double stretch = M.prm.stretch; const int pad = M.prm.pad;
    int *pmap = M.pinv, *qmap = M.qinv;
    int *iwork1 = M.iwork1, *iwork2 = M.iwork1 + m;
    double *work1 = M.work1;
    const int jpivot = I->btran_for_update;
    const int ipivot = pmap[jpivot];
    const double oldpiv = M.colpiv[jpivot];
    i64 u_nz = I->u_nz;
    if (nforrest >= m) { if (lane == 0) { BLU_CHECK(C, 0); scal[0] = C.status; } return; }

    /* move the diagonal element to the end of the spike, update.rs:442-463 */
    const int sbeg = M.u_begin[m];
    double spike_diag = 0.0; int have_diag = 0;
    int put = sbeg;
    for (int b = sbeg;; b += 32) {
        const int idx = M.u_idx[b + lane];
        const double val = M.u_val[b + lane];
        const unsigned tm = __ballot_sync(FULLMASK, idx < 0);
        const int nvalid = tm ? __ffs((int)tm) - 1 : 32;
        const bool isdiag = lane < nvalid && idx == ipivot;
        const bool keep = lane < nvalid && idx != ipivot;
        const unsigned km = __ballot_sync(FULLMASK, keep), dm = __ballot_sync(FULLMASK, isdiag);
        if (dm) { have_diag = 1; spike_diag = __shfl_sync(FULLMASK, val, __ffs((int)dm) - 1); }
        __syncwarp();
        if (keep) { const int d = put + __popc(km & lanemask_lt()); M.u_idx[d] = idx; M.u_val[d] = val; }
        put += __popc(km);
        __syncwarp();
        if (tm) break;
    }
    if (have_diag && lane == 0) { M.u_idx[put] = ipivot; M.u_val[put] = spike_diag; }
    __syncwarp();
    const int nz_spike = put - sbeg;
    const int rbeg = M.r_begin[nforrest], rend = M.r_begin[nforrest + 1];
    const int nz_roweta = rend - rbeg;

    /* new pivot, update.rs:485-513 */
    int marker = sp_next_marker(C);
    for (int pos = rbeg + lane; pos < rend; pos += 32 * 8) {      /* eight independent loads per lane in flight */
        int ii[8]; double vv[8];
        #pragma unroll
        for (int u = 0; u < 8; u++) { const int q = pos + 32 * u; ii[u] = q < rend ? M.l_idx[q] : -1; vv[u] = q < rend ? M.l_val[q] : 0.0; }
        #pragma unroll
        for (int u = 0; u < 8; u++) if (ii[u] >= 0) { C.marked[ii[u]] = marker; work1[ii[u]] = vv[u]; }
    }
    __syncwarp();
    double newpiv = spike_diag;
    int intersect = 0;
    for (int b = sbeg; b < sbeg + nz_spike; b += 32) {
        const int pos = b + lane;
        const bool ok = pos < sbeg + nz_spike;
        const int i = ok ? M.u_idx[pos] : 0;
        const bool hit = ok && C.marked[i] == marker;
        const double term = hit ? __dmul_rn(M.u_val[pos], work1[i]) : 0.0;
        unsigned hm = __ballot_sync(FULLMASK, hit);
        intersect += __popc(hm);
        while (hm) {   /* only the intersecting terms are subtracted, in spike order */
            const int t = __ffs((int)hm) - 1;
            hm &= hm - 1;
            newpiv = __dsub_rn(newpiv, __shfl_sync(FULLMASK, term, t));
        }
    }
    if (newpiv == 0.0 || fabs(newpiv) < M.prm.abstol) {
        if (lane == 0) scal[0] = BLU_ERROR_SINGULAR_UPDATE;
        return;
    }
    const double piverr = fabs(__dsub_rn(newpiv, __dmul_rn(xtbl, oldpiv)));

    /* bound on the growth of the row file, update.rs:517-536 */
    {
        i64 grow = 0;
        for (int pos = sbeg + lane; pos < sbeg + nz_spike; pos += 32) {
            const int j = qmap[M.u_idx[pos]];
            if (M.lend[j] == M.lcap[j]) {
                const int nz = M.lend[j] - M.lbeg[j];
                grow += nz + 1 + (i64)(stretch * (double)(nz + 1)) + pad;
            }
        }
        grow = warp_sum64(grow);
        i64 room = (i64)(I->w_half + 1) * M.w_mem - I->w_used;
        if (grow > room) {
            sp_w_compact(C);
            room = (i64)(I->w_half + 1) * M.w_mem - I->w_used;
            /* after compaction every line has slack; only lines that are still full count */
            grow = 0;
            for (int pos = sbeg + lane; pos < sbeg + nz_spike; pos += 32) {
                const int j = qmap[M.u_idx[pos]];
                if (M.lend[j] == M.lcap[j]) {
                    const int nz = M.lend[j] - M.lbeg[j];
                    grow += nz + 1 + (i64)(stretch * (double)(nz + 1)) + pad;
                }
            }
            grow = warp_sum64(grow);
            if (grow > room || C.status != BLU_OK) {
                if (lane == 0) { I->addmem_w = grow > room ? grow - room : M.w_mem; scal[0] = C.status != BLU_OK ? C.status : BLU_REALLOCATE; }
                return;
            }
        }
    }

    /* remove column jpivot from the row file, update.rs:538-555 */
    {
        const int cb = M.u_begin[ipivot];
        int nz = 0;
        for (int pos = cb;; pos++) {
            const int i = M.u_idx[pos];
            if (i < 0) break;
            const int j = qmap[i];
            const int lb = M.lbeg[j], end = M.lend[j];
            const int where = sp_find(jpivot, M.w_idx, lb, end);
            if (where >= end) { if (lane == 0) { BLU_CHECK(C, 0); scal[0] = C.status; } return; }
            if (lane == 0) {
                M.lend[j] = end - 1;
                M.w_idx[where] = M.w_idx[end - 1];
                M.w_val[where] = M.w_val[end - 1];
            }
            nz++;
            __syncwarp();
        }
        u_nz -= nz;
        /* erase column jpivot in the column file, update.rs:557-563 */
        for (int pos = cb + lane; pos < cb + nz; pos += 32) M.u_idx[pos] = SP_GAP;
        __syncwarp();
    }
    /* column pointer to the spike, chop the diagonal, update.rs:565-570 */
    if (lane == 0) {
        M.u_begin[ipivot] = sbeg;
        M.u_idx[sbeg + nz_spike] = SP_GAP;
        M.u_begin[m] = sbeg + nz_spike + 1;
    }
    __syncwarp();
    /* insert the spike into the row file, update.rs:572-601 */
    {
        int w_used = (int)I->w_used;
        for (int b = sbeg; b < sbeg + nz_spike; b += 32) {
            const int pos = b + lane;
            const bool ok = pos < sbeg + nz_spike;
            const int j = ok ? qmap[M.u_idx[pos]] : 0;
            int lb = ok ? M.lbeg[j] : 0, le = ok ? M.lend[j] : 0;
            const int lc = ok ? M.lcap[j] : 1;
            const int nz = le - lb;
            const bool full = ok && le == lc;
            const int space = 1 + (int)(stretch * (double)(nz + 1)) + pad;
            const int need = full ? nz + space : 0;
            const int incl = warp_incl_scan(need);
            if (full) {
                const int np = w_used + incl - need;
                for (int t = 0; t < nz; t++) { M.w_idx[np + t] = M.w_idx[lb + t]; M.w_val[np + t] = M.w_val[lb + t]; }
                lb = np; le = np + nz;
                M.lbeg[j] = lb; M.lcap[j] = np + nz + space;
            }
            if (ok) { M.w_idx[le] = jpivot; M.w_val[le] = M.u_val[pos]; M.lend[j] = le + 1; }
            w_used += __shfl_sync(FULLMASK, incl, 31);
            const int nfull = __popc(__ballot_sync(FULLMASK, full));
            if (lane == 0) I->nexpand += nfull;
        }
        __syncwarp();
        if (lane == 0) {
            BLU_CHECK(C, (i64)w_used <= (i64)(I->w_half + 1) * M.w_mem);
            I->w_used = w_used;
            M.colpiv[jpivot] = spike_diag;
            M.rowpiv[ipivot] = spike_diag;
        }
        u_nz += nz_spike;
        __syncwarp();
    }

    /* triangularity test, update.rs:609-818 */
    int istriangular = 0, nreach = 0, rtop = 0, use_reach = 0;
    double pmin = I->min_pivot, pmax = I->max_pivot;
    if (have_diag) {
        istriangular = intersect == 0;
        if (istriangular) {
            pmin = fmin(pmin, fabs(newpiv)); pmax = fmax(pmax, fabs(newpiv));
            nreach = nz_roweta + 1;
            if (lane == 0) { iwork1[0] = ipivot; iwork2[0] = jpivot; I->nsymperm_total++; }
            for (int n = 1 + lane; n < nreach; n += 32) {
                const int i = M.l_idx[rbeg + n - 1];
                iwork1[n] = i;
                iwork2[n] = qmap[i];
            }
            __syncwarp();
        }
    } else {
        /* no diagonal element in the spike, update.rs:667-818: an augmenting path (BFS, lane 0), then the
         * reach of every path node (depth-first, the whole warp probing 32 edges at a time) decides
         * whether a purely unsymmetric permutation restores triangularity */
        int dec = 0;
        int *path = iwork1, *reach = iwork2;
        int top = 0;
        if (lane == 0) top = sp_bfs_path(m, jpivot, M.lbeg, M.lend, M.w_idx, path, C.marked, iwork2);
        top = sp_bcast(top);
        __syncwarp();
        if (!(top < m - 1) || path[top] != jpivot) { if (lane == 0) BLU_CHECK(C, 0); __syncwarp(); }
        else {
            istriangular = 1;
            rtop = m;
            marker = sp_next_marker(C);
            for (int t = top; t < m - 1 && istriangular; t++) {
                const int j = path[t], jnext = path[t + 1];
                const int le = M.lend[j];
                const int where = sp_find(jnext, M.w_idx, M.lbeg[j], le);
                if (where >= le) { if (lane == 0) BLU_CHECK(C, 0); __syncwarp(); break; }
                if (lane == 0) M.w_idx[where] = j;      /* take the path edge out for a moment */
                __syncwarp();
                rtop = sp_dfs_warp(j, M.lbeg, M.lend, M.w_idx, rtop, reach, C.pstack, C.pend, C.marked, marker);
                if (lane == 0) { reach[rtop] = jnext; M.w_idx[where] = jnext; }
                __syncwarp();
                istriangular = C.marked[jnext] != marker;
            }
            if (istriangular && C.status == BLU_OK) {
                const int j = path[m - 1];
                rtop = sp_dfs_warp(j, M.lbeg, M.lend, M.w_idx, rtop, reach, C.pstack, C.pend, C.marked, marker);
                if (lane == 0) { reach[rtop] = jpivot; C.marked[j]--; }
                __syncwarp();
                int hit = 0;
                for (int pos = M.u_begin[ipivot];; pos += 32) {
                    const int r = M.u_idx[pos + lane];
                    const unsigned tm = __ballot_sync(FULLMASK, r < 0);
                    const int nvalid = tm ? __ffs((int)tm) - 1 : 32;
                    if (lane < nvalid && C.marked[qmap[r]] == marker) hit = 1;
                    if (tm) break;
                }
                if (__any_sync(FULLMASK, hit)) istriangular = 0;
                __syncwarp();
                if (lane == 0) C.marked[j]++;
                __syncwarp();
            }
            if (istriangular && C.status == BLU_OK) {
                const int nswap = m - top - 1;
                if (lane == 0) sp_permute(C, path + top, nswap, &pmin, &pmax);
                __syncwarp();
                dec = 1;
                nreach = m - rtop;
                for (int n = lane; n < nreach; n += 32) iwork1[rtop + n] = pmap[reach[rtop + n]];
                __syncwarp();
            }
        }
        pmin = sp_bcastd(pmin); pmax = sp_bcastd(pmax);
        u_nz -= dec;
        use_reach = istriangular;
        if (C.status != BLU_OK) { if (lane == 0) scal[0] = C.status; return; }
    }

    /* Forrest-Tomlin update, update.rs:822-883 */
    int nforrest_new = nforrest;
    double max_eta_all = I->max_eta;
    i64 r_nz = I->r_nz;
    if (!istriangular) {
        const int wb = M.lbeg[jpivot], we = M.lend[jpivot];
        for (int pos = wb; pos < we; pos++) {
            const int j = M.w_idx[pos];
            int term = 0;
            const int where = sp_find_term(ipivot, M.u_idx, M.u_begin[pmap[j]], &term);
            if (where < 0) { if (lane == 0) { BLU_CHECK(C, 0); scal[0] = C.status; } return; }
            if (lane == 0) {
                M.u_idx[where] = M.u_idx[term - 1];
                M.u_val[where] = M.u_val[term - 1];
                M.u_idx[term - 1] = -1;
            }
            u_nz--;
            __syncwarp();
        }
        if (lane == 0) { M.lend[jpivot] = wb; M.colpiv[jpivot] = newpiv; M.rowpiv[ipivot] = newpiv; }
        pmin = fmin(pmin, fabs(newpiv)); pmax = fmax(pmax, fabs(newpiv));
        /* keep the non-zero eta entries */
        int eput = rbeg; double max_eta = 0.0;
        for (int b = rbeg; b < rend; b += 32) {
            const int pos = b + lane;
            const bool ok = pos < rend;
            const double v = ok ? M.l_val[pos] : 0.0;
            const int i = ok ? M.l_idx[pos] : 0;
            const bool keep = ok && v != 0.0;
            const unsigned km = __ballot_sync(FULLMASK, keep);
            __syncwarp();
            if (keep) { const int d = eput + __popc(km & lanemask_lt()); M.l_idx[d] = i; M.l_val[d] = v; max_eta = fmax(max_eta, fabs(v)); }
            eput += __popc(km);
            __syncwarp();
        }
        max_eta = warp_maxd(max_eta);
        if (lane == 0) M.r_begin[nforrest + 1] = eput;
        r_nz += eput - rbeg;
        max_eta_all = fmax(max_eta_all, max_eta);
        nreach = 1;
        if (lane == 0) { iwork1[0] = ipivot; iwork2[0] = jpivot; I->nforrest_total++; }
        rtop = 0; use_reach = 0;
        nforrest_new = nforrest + 1;
        __syncwarp();
    }

    /* append the reach to the pivot sequence, update.rs:891-911 */
    {
        const int *row_reach = use_reach ? iwork1 + rtop : iwork1;
        const int *col_reach = use_reach ? iwork2 + rtop : iwork2;
        if (lane == 0 && I->pivotlen + nreach > 2 * m) dev_garbage_perm(M);
        __syncwarp();
        const int pl = I->pivotlen;
        for (int n = lane; n < nreach; n += 32) { M.pivotrow[pl + n] = row_reach[n]; M.pivotcol[pl + n] = col_reach[n]; }
        __syncwarp();
        if (lane == 0) I->pivotlen = pl + nreach;
        __syncwarp();
    }

    /* compress U and W when enough was wasted, update.rs:915-937 */
    {
        i64 used = M.u_begin[m];
        if (used - u_nz - m > (i64)(M.prm.compress_thres * (double)used)) {
            const int nz = sp_compress_packed(C);
            if (lane == 0) BLU_CHECK(C, (i64)nz == u_nz);
        }
        used = I->w_used - (i64)I->w_half * M.w_mem;
        const i64 need = u_nz + (i64)(stretch * (double)u_nz) + (i64)m * pad;
        if (used - need > (i64)(M.prm.compress_thres * (double)used)) sp_w_compact(C);
    }
    __syncwarp();
    if (lane == 0) {
        I->pivot_error = piverr / (1.0 + fabs(newpiv));
        I->u_nz = u_nz; I->r_nz = r_nz;
        I->min_pivot = pmin; I->max_pivot = pmax; I->max_eta = max_eta_all;
        I->nforrest = nforrest_new;
        I->btran_for_update = -1; I->ftran_for_update = -1; I->have_ur = 0;
        I->update_cost_numer += (double)nz_roweta;
        I->nupdate++; I->nupdate_total++;
        scal[0] = C.status;
    }
}

/* lu_realloc_obj (blu.rs:345-377) for a batch: every basis copies the content of its L / U / W store --
 * read through its own view, i.e. from its private store if it has one -- into slot s of new uniform
 * stores of nl / nu / nw entries per basis (a null target = that store stays).  Of W only the live half
 * moves; it becomes half 0 and the line table is shifted accordingly. */
__global__ void k_store_regrow(BluDev D, int *nl_i, double *nl_v, blu_i64 nl, int *nu_i, double *nu_v, blu_i64 nu,
                               int *nw_i, double *nw_v, blu_i64 nw) {
    __shared__ Mat M;
    const int s = blockIdx.x;
    if (threadIdx.x == 0) mat_view(M, D, s);
    __syncthreads();
    if (nl_i) {
        const size_t dst = (size_t)s * (size_t)nl;
        for (int q = threadIdx.x; q < M.l_mem; q += blockDim.x) { nl_i[dst + q] = M.l_idx[q]; nl_v[dst + q] = M.l_val[q]; }
    }
    if (nu_i) {
        const size_t dst = (size_t)s * (size_t)nu;
        for (int q = threadIdx.x; q < M.u_mem; q += blockDim.x) { nu_i[dst + q] = M.u_idx[q]; nu_v[dst + q] = M.u_val[q]; }
    }
    if (nw_i) {
        const int half = M.info->w_half;
        const size_t src = (size_t)half * (size_t)M.w_mem, dst = (size_t)s * 2 * (size_t)nw;
        const int delta = half * M.w_mem;
        const int used = (int)(M.info->w_used - (blu_i64)delta);
        for (int q = threadIdx.x; q < used; q += blockDim.x) { nw_i[dst + q] = M.w_idx[src + q]; nw_v[dst + q] = M.w_val[src + q]; }
        for (int l = threadIdx.x; l < 2 * M.m; l += blockDim.x) { M.lbeg[l] -= delta; M.lend[l] -= delta; M.lcap[l] -= delta; }
        __syncthreads();
        if (threadIdx.x == 0) { M.info->w_used -= delta; M.info->w_half = 0; }
    }
}

/* after the host moved the live half of W into a larger store: shift the line table */
__global__ void k_w_rebase(BluDev D, int delta) {
    __shared__ Mat M;
    if (threadIdx.x == 0) mat_view(M, D, 0);
    __syncthreads();
    for (int l = threadIdx.x; l < 2 * M.m; l += blockDim.x) { M.lbeg[l] -= delta; M.lend[l] -= delta; M.lcap[l] -= delta; }
    if (threadIdx.x == 0) { M.info->w_used -= delta; M.info->w_half = 0; }
}

#endif
