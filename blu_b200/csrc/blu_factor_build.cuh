/* blu_factor_build.cuh -- phase 4: assemble the factors in the layout the solves and the
 * Forrest-Tomlin update work on (reference: src/lu/build_factors.rs:113-423; layout
 * documented there at :10-112), then the factorize kernel itself. */
#ifndef BLU_FACTOR_BUILD_CUH
#define BLU_FACTOR_BUILD_CUH
#include "blu_dev_common.cuh"
#include "blu_factor_setup.cuh"
#include "blu_factor_bump.cuh"

template <int NT> __device__ void phase_build_factors(Shm &S) {
    Mat &M = S.M;
    const int m = M.m, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    constexpr int NW = NT / 32;
    const int rank = S.rank;
    const int l_nz = M.l_begin_p[rank] - rank;
    int u_nz = M.u_begin[rank];

    /* memory, build_factors.rs:163-177 */
    {
        int st = BLU_OK;
        i64 need = 2 * ((i64)l_nz + m);
        if ((i64)M.l_mem < need) { if (tid == 0) M.info->addmem_l = need - M.l_mem; st = BLU_REALLOCATE; }
        need = (i64)u_nz + m + 1;
        if (st == BLU_OK && (i64)M.u_mem < need) { if (tid == 0) M.info->addmem_u = need - M.u_mem; st = BLU_REALLOCATE; }
        need = (i64)u_nz + (i64)(M.prm.stretch * (double)u_nz) + (i64)m * M.prm.pad;
        if (st == BLU_OK && (i64)M.w_mem < need) { if (tid == 0) M.info->addmem_w = need - M.w_mem; st = BLU_REALLOCATE; }
        if (st != BLU_OK) { bsync<NT>(); if (tid == 0) S.status = st; bsync<NT>(); return; }
    }

    /* permutations, build_factors.rs:192-209: non-pivotal rows/columns in index order */
    {
        int lr = rank, lc = rank;
        for (int base = 0; base < m; base += NT) {
            int i = base + tid;
            int fr = i < m && M.pinv[i] < 0, fc = i < m && M.qinv[i] < 0;
            int totr, exr = block_excl_scan<NT>(fr, &totr, S.iscr);
            int totc, exc = block_excl_scan<NT>(fc, &totc, S.iscr);
            if (i < m) {
                int pr = fr ? lr + exr : M.pinv[i];
                int qc = fc ? lc + exc : M.qinv[i];
                M.pinv[i] = pr; M.qinv[i] = qc;
                M.prank[i] = pr; M.qrank[i] = qc;
                M.pivotrow[pr] = i; M.pivotcol[qc] = i;
            }
            lr += totr; lc += totc;
        }
        if (tid == 0) { BLU_CHECK(S, lr == m && lc == m); }
    }
    bsync<NT>();
    /* unit pivots for dependent columns; L column-wise completion, :221-238 */
    {
        const int lb = M.l_begin_p[rank];
        for (int k = rank + tid; k < m; k += NT) {
            M.colpiv[M.pivotcol[k]] = 1.0;
            M.l_idx[lb + (k - rank)] = -1;
            M.l_begin_p[k + 1] = lb + (k - rank) + 1;
        }
    }
    bsync<NT>();
    for (int i = tid; i < m; i += NT) M.l_begin[i] = M.l_begin_p[M.pinv[i]];

    /* L row-wise, build_factors.rs:242-274.  Counting in parallel; the scatter runs in
     * pivot order on one warp so every row is filled in ascending pivot step exactly
     * as the reference does (no atomics => deterministic storage order). */
    /* per-row / per-column fill pointers live in shared memory when m of them fit (the pivot-loop
     * buffers are idle here): the ordered scatters below are read-modify-write chains on them */
    int *cnt = (size_t)m * sizeof(int) <= (size_t)S.dyn_bytes ? (int *)S.cval : M.iwork1;
    for (int i = tid; i < m; i += NT) cnt[i] = 0;
    bsync<NT>();
    for (int g = tid; g < l_nz + m; g += NT) { int i = M.l_idx[g]; if (i >= 0) atomicAdd(&cnt[i], 1); }
    bsync<NT>();
    {
        int put = l_nz + m;
        for (int base = 0; base < m; base += NT) {
            int k = base + tid;
            int i = k < m ? M.pivotrow[k] : 0;
            int c = k < m ? cnt[i] + 1 : 0;
            int tot, ex = block_excl_scan<NT>(c, &tot, S.iscr);
            if (k < m) {
                int b = put + ex;
                M.lt_begin_p[k] = b; M.lt_begin[i] = b;
                M.l_idx[b + c - 1] = -1;
                cnt[i] = b;
            }
            put += tot;
        }
        if (tid == 0) { BLU_CHECK(S, put == 2 * (l_nz + m)); M.lt_begin_p[m] = put; M.r_begin[0] = put; }
    }
    bsync<NT>();
    if (wid == 0) {
        /* pivot order, one warp: every row is filled in ascending pivot step exactly as the reference
         * does.  Column pointers are fetched 32 pivots at a time; empty columns cost nothing. */
        for (int kb = 0; kb < m; kb += 32) {
            const int k = kb + lane;
            const int b = k < m ? M.l_begin_p[k] : 0, e = k < m ? M.l_begin_p[k + 1] - 1 : 0;
            const int ipv = k < m ? M.pivotrow[k] : 0;
            unsigned ne = __ballot_sync(FULLMASK, e > b);
            while (ne) {
                const int t = __ffs((int)ne) - 1;
                ne &= ne - 1;
                const int bb = __shfl_sync(FULLMASK, b, t), ee = __shfl_sync(FULLMASK, e, t), ii = __shfl_sync(FULLMASK, ipv, t);
                for (int g = bb + lane; g < ee; g += 32) {
                    const int r = M.l_idx[g];
                    const double v = M.l_val[g];
                    const int dst = cnt[r]; cnt[r] = dst + 1;
                    M.l_idx[dst] = ii; M.l_val[dst] = v;
                }
                __syncwarp();
            }
        }
    }
    bsync<NT>();

    /* U row-wise into the W file in pivot order with slack, build_factors.rs:286-351 */
    int *ucnt = cnt;           /* per column j: entries of U column j */
    for (int j = tid; j < m; j += NT) ucnt[j] = 0;
    bsync<NT>();
    {
        int put = 0, unz_new = 0;
        const bool full = rank == m;
        for (int base = 0; base < m; base += NT) {
            int k = base + tid;
            int nz = 0;
            if (k < rank) {
                if (full) nz = M.u_begin[k + 1] - M.u_begin[k];
                else for (int pos = M.u_begin[k]; pos < M.u_begin[k + 1]; pos++) nz += M.qinv[M.u_idx[pos]] < rank;
            }
            int sz = k < m ? (k < rank ? nz + slack_of(M.prm, nz) : M.prm.pad) : 0;
            int tot, ex = block_excl_scan<NT>(sz, &tot, S.iscr);
            int totn, exn = block_excl_scan<NT>(nz, &totn, S.iscr);
            (void)exn;
            if (k < m) {
                int jp = M.pivotcol[k];
                int b = put + ex, w = b;
                if (k < rank) {
                    for (int pos = M.u_begin[k]; pos < M.u_begin[k + 1]; pos++) {
                        int j = M.u_idx[pos];
                        if (full || M.qinv[j] < rank) {
                            M.w_idx[w] = j; M.w_val[w] = M.u_val[pos]; w++;
                            atomicAdd(&ucnt[j], 1);
                        }
                    }
                }
                M.lbeg[jp] = b; M.lend[jp] = w; M.lcap[jp] = b + sz;
            }
            put += tot; unz_new += totn;
        }
        u_nz = unz_new;
        if (tid == 0) {
            BLU_CHECK(S, put <= M.w_mem);
            S.w_half = 0; S.w_used = put; S.w_limit = M.w_mem;
        }
    }
    bsync<NT>();
    /* U column-wise, build_factors.rs:354-384 */
    {
        int put = 1;
        if (tid == 0) M.u_idx[0] = -1;
        for (int base = 0; base < m; base += NT) {
            int k = base + tid;
            int j = k < m ? M.pivotcol[k] : 0, i = k < m ? M.pivotrow[k] : 0;
            int nz = k < m ? ucnt[j] : 0;
            int sz = nz > 0 ? nz + 1 : 0;
            int tot, ex = block_excl_scan<NT>(sz, &tot, S.iscr);
            if (k < m) {
                int b = nz > 0 ? put + ex : 0;
                M.u_begin[i] = b;
                if (nz > 0) M.u_idx[b + nz] = -1;
                ucnt[j] = b;
            }
            put += tot;
        }
        if (tid == 0) M.u_begin[m] = put;
    }
    bsync<NT>();
    if (wid == 0) {
        for (int kb = 0; kb < m; kb += 32) {
            const int k = kb + lane;
            const int jp = k < m ? M.pivotcol[k] : 0, ipv = k < m ? M.pivotrow[k] : 0;
            const int b = k < m ? M.lbeg[jp] : 0, e = k < m ? M.lend[jp] : 0;
            unsigned ne = __ballot_sync(FULLMASK, e > b);
            while (ne) {
                const int t = __ffs((int)ne) - 1;
                ne &= ne - 1;
                const int bb = __shfl_sync(FULLMASK, b, t), ee = __shfl_sync(FULLMASK, e, t), ii = __shfl_sync(FULLMASK, ipv, t);
                for (int pos = bb + lane; pos < ee; pos += 32) {
                    const int j = M.w_idx[pos];
                    const double v = M.w_val[pos];
                    const int dst = ucnt[j]; ucnt[j] = dst + 1;
                    M.u_idx[dst] = ii; M.u_val[dst] = v;
                }
                __syncwarp();
            }
        }
    }
    bsync<NT>();
    /* pmap / qmap overwrite pinv / qinv, build_factors.rs:395-400; row_pivot, min/max, :403-410 */
    for (int k = tid; k < m; k += NT) {
        int i = M.pivotrow[k], j = M.pivotcol[k];
        M.pinv[j] = i; M.qinv[i] = j;
        M.p[k] = i;
    }
    bsync<NT>();
    double mx = 0.0, mn = INFINITY;
    for (int i = tid; i < m; i += NT) {
        double pv = M.colpiv[M.qinv[i]];
        M.rowpiv[i] = pv;
        pv = fabs(pv);
        mx = fmax(mx, pv); mn = fmin(mn, pv);
    }
    /* how far back (forward) each row of L / column of L / column of U reaches in the pivot order: lets
     * the dot-product sweeps of the dense solves and of condest/residual_test run a whole batch of
     * pivots side by side whenever they do not depend on each other (blu_solve.cuh, dev_dot_sweep) */
    for (int k = tid; k < m; k += NT) {
        int d = -1;
        for (int pos = M.lt_begin_p[k]; M.l_idx[pos] >= 0; pos++) { const int q = M.prank[M.l_idx[pos]]; d = q > d ? q : d; }
        M.dep_lt[k] = d;
        d = m;
        for (int pos = M.l_begin_p[k]; M.l_idx[pos] >= 0; pos++) { const int q = M.prank[M.l_idx[pos]]; d = q < d ? q : d; }
        M.dep_lc[k] = d;
        d = -1;
        int n = 0;
        for (int pos = M.u_begin[M.pivotrow[k]]; M.u_idx[pos] >= 0; pos++, n++) { const int q = M.prank[M.u_idx[pos]]; d = q > d ? q : d; }
        M.dep_uc[k] = d; M.len_uc[k] = n;
    }
    /* The row-wise copy of B is dead after the bump set-up: re-sort every row by the pivot position of
     * its column, so that residual_test / matrix_norm (which the reference accumulates column by column
     * in pivot order, residual_test.rs:60-70, matrix_norm.rs:20-33) can be evaluated row by row, all
     * rows in parallel, with every row's terms in exactly the reference's order. */
    for (int i = tid; i < m; i += NT) {
        const int rb = M.bt_ptr[i], n = M.bt_ptr[i + 1] - rb;
        if (n > 1 && n <= 32) {
            for (int a = 1; a < n; a++) {
                const int j = M.bt_idx[rb + a]; const double x = M.bt_val[rb + a];
                const int key = M.qrank[j];
                int q = a - 1;
                while (q >= 0 && M.qrank[M.bt_idx[rb + q]] > key) { M.bt_idx[rb + q + 1] = M.bt_idx[rb + q]; M.bt_val[rb + q + 1] = M.bt_val[rb + q]; q--; }
                M.bt_idx[rb + q + 1] = j; M.bt_val[rb + q + 1] = x;
            }
        }
    }
    bsync<NT>();
    {   /* long rows: one warp each, rank sort on the keys (distinct: one entry per column); scratch = tmpi / work1 */
        for (int i = 0; i < m; i++) {          /* uniform scan: every thread walks the same pointers */
            const int rb = M.bt_ptr[i], n = M.bt_ptr[i + 1] - rb;
            if (n <= 32) continue;
            int *sidx = M.tmpi, *skey = M.tmpi + 2 * m; double *sval = M.work1;
            for (int e = tid; e < n; e += NT) skey[e] = M.qrank[M.bt_idx[rb + e]];
            bsync<NT>();
            for (int e = tid; e < n; e += NT) {
                const int ke = skey[e];
                int rnk = 0;
                for (int f = 0; f < n; f++) rnk += skey[f] < ke;
                sidx[rnk] = M.bt_idx[rb + e]; sval[rnk] = M.bt_val[rb + e];
            }
            bsync<NT>();
            for (int e = tid; e < n; e += NT) { M.bt_idx[rb + e] = sidx[e]; M.bt_val[rb + e] = sval[e]; }
            bsync<NT>();
        }
    }
    mx = block_maxd<NT>(mx, S.dscr);
    mn = block_mind<NT>(mn, S.dscr);
    if (tid == 0) {
        BluInfo *I = M.info;
        I->min_pivot = mn; I->max_pivot = mx;
        I->pivotlen = m; I->l_nz = l_nz; I->u_nz = u_nz; I->r_nz = 0;
    }
    bsync<NT>();
}

/* ------------------------------------------------------------------ */
/* the factorize kernel: one CTA per basis (factorize.rs:34-119)       */
/* ------------------------------------------------------------------ */
__device__ __forceinline__ void shm_carve(Shm &S, unsigned char *dyn, int cap, int nw, int m) {
    /* [cval: cap f64][work: nw*cap f64][cidx: cap i32][ridx: cap i32]
     * and when m <= SMARK_MAX: [chb che chc rhb rhe rhc: cap i32 each][rm: m u16][cm: m u8] */
    S.cap = cap;
    S.cval = (double *)dyn;
    S.work = S.cval + cap;
    S.cidx = (int *)(S.work + (size_t)nw * cap);
    S.ridx = S.cidx + cap;
    S.smarks = m <= SMARK_MAX;
    S.dyn_bytes = (int)(cap * 8 + (size_t)nw * cap * 8 + cap * 4 * 2 + (m <= SMARK_MAX ? (size_t)cap * 4 * 6 + (size_t)((m + 1) & ~1) * 2 + (size_t)((m + 15) & ~15) : 0));
    if (S.smarks) {
        S.chb = S.ridx + cap; S.che = S.chb + cap; S.chc = S.che + cap;
        S.rhb = S.chc + cap; S.rhe = S.rhb + cap; S.rhc = S.rhe + cap;
        S.rm = (unsigned short *)(S.rhc + cap);
        S.cm = (unsigned char *)(S.rm + ((m + 1) & ~1));
    }
}
#ifndef FACT_MINB
/* resident CTAs per SM the register allocation is sized for.  Measured on B200 with 128-thread
 * CTAs (profiles/r1b_sweep.txt, r1h_sweep.txt): 4 CTAs/SM (128 registers) 7.3 k bases/s, 6 (80) 8.6 k,
 * 7 (72) 10.1 k, 8 (64, more spills) 9.5 k, 9 (56) 7.6 k -- the kernel is latency-bound, so occupancy
 * pays until the spills cost more than the extra warps hide. */
#define FACT_MINB(NT) (896 / (NT) > 0 ? 896 / (NT) : 1)
#endif
/* mode (blu_types.h): BLU_MODE_WHOLE runs everything; HEAD stops where the dense tail would begin and parks
 * the basis (status BLU_SUSPENDED_TAIL); TAIL resumes parked bases, finishes the pivot loop and parks them
 * for BUILD, which assembles the factors.  rerun != 0: only bases whose status is BLU_REALLOCATE start over.
 * dense_kd: order of the dense tail for this factorization;
 * dense_smem != 0: the launch has room for the dense values in shared memory. */
template <int NT> __global__ void __launch_bounds__(NT, FACT_MINB(NT)) k_factorize(BluDev D, int cap, int mode, int dense_kd, int dense_smem, int rerun) {
    BLU_DYN_SMEM(dyn);
    __shared__ Shm S;
    const int tid = threadIdx.x;
    if (tid == 0) { mbar_init(&S.mbar, 1); S.mbar_phase = 0; }
    bsync<NT>();
    for (int s = D.slot0 + blockIdx.x; s < D.slot0 + D.nslot; s += gridDim.x) {
        const bool fresh = mode == BLU_MODE_WHOLE || mode == BLU_MODE_HEAD;
        if (!fresh && D.info[s].status != (mode == BLU_MODE_TAIL ? BLU_SUSPENDED_TAIL : BLU_SUSPENDED_BUILD)) continue;
        if (fresh && rerun && D.info[s].status != BLU_REALLOCATE) continue;      /* only the bases that asked for more memory run again */
        if (fresh && D.run && !D.run[s]) continue;                               /* a subset of the batch (blu_batch_maxvolume) */
        if (tid == 0) {
            mat_view(S.M, D, s);
            shm_carve(S, dyn, cap, NT / 32, D.m);
            BluInfo *I = S.M.info;
            S.status = BLU_OK;
            S.need_remove = 0;
            S.wc = -1; S.wr = -1;
            S.dyn = dyn; S.dense = 0; S.kd = dense_kd; S.kw = dense_kd / 32; S.dv_smem = dense_smem;
            S.launch_res = dense_smem; S.kd_small = dense_kd; S.kd_big = D.dense_kbig_eff > dense_kd && (mode == BLU_MODE_HEAD || NT >= D.dense_kbig_eff) ? D.dense_kbig_eff : 0;
            S.mode = mode; S.suspend = 0;
            if (fresh) {
                /* LU::reset, lu.rs:329-396 (cumulative counters survive) */
                I->m = D.m; I->nruns++;
                I->nupdate = -1; I->nforrest = 0; I->l_nz = I->u_nz = I->r_nz = 0;
                I->min_pivot = I->max_pivot = I->max_eta = 0.0;
                I->update_cost_numer = 0.0; I->update_cost_denom = 1.0;
                I->l_flops = I->u_flops = I->r_flops = 0;
                I->matrix_nz = 0; I->rank = 0; I->bump_size = 0; I->bump_nz = 0;
                I->nsearch_pivot = I->nexpand = I->ngarbage = I->factor_flops = 0;
                I->pivot_error = 0.0; I->ftran_for_update = I->btran_for_update = -1;
                I->marker = 0; I->pivotlen = 0; I->rankdef = 0;
                I->addmem_l = I->addmem_u = I->addmem_w = 0;
                I->internal_error = 0; I->elim_bytes = 0.0; I->nelim_div = 0; I->have_ur = 0;
                I->condest_l = I->condest_u = I->norm_l = I->norm_u = 0.0;
                I->normest_l_inv = I->normest_u_inv = I->onenorm = I->infnorm = I->residual_test = 0.0;
                S.rank = 0; S.rankdef = 0;
                S.nexpand = 0; S.ngarbage = 0; S.nsearch = 0; S.factor_flops = 0;
                S.elim_bytes = 0.0; S.nelim_div = 0;
                S.w_used = 0; S.w_limit = S.M.w_mem; S.w_half = 0;
                S.dense_entries = 0; S.dense_block_rank = 0;
                for (int q = 0; q < 16; q++) S.t_phase[q] = 0;
                for (int q = 0; q < 8; q++) S.n_kind[q] = 0;
            } else {
                /* pick up where the previous launch parked this basis */
                S.rank = I->rank; S.rankdef = I->rankdef;
                S.nexpand = (int)I->nexpand; S.ngarbage = (int)I->ngarbage; S.nsearch = I->nsearch_pivot; S.factor_flops = I->factor_flops;
                S.elim_bytes = I->elim_bytes; S.nelim_div = I->nelim_div;
                S.w_half = I->w_half; S.w_used = (int)I->w_used; S.w_limit = (S.w_half + 1) * S.M.w_mem;
                S.cstamp = I->cstamp; S.rstamp = I->rstamp;
                S.nact = I->nact; S.ndead = I->ndead;
                S.dense_entries = I->dense_entries; S.dense_block_rank = I->dense_block_rank;
                for (int q = 0; q < 16; q++) S.t_phase[q] = I->t_phase[q];
                for (int q = 0; q < 8; q++) S.n_kind[q] = I->n_kind[q];
            }
        }
        bsync<NT>();
        if (fresh) for (int i = tid; i < D.m; i += NT) S.M.marked[i] = 0;
        if (S.smarks) for (int i = tid; i < D.m; i += NT) { S.rm[i] = 0; S.cm[i] = 0; }
        const i64 tstart = clock64();
        i64 t0;
        if (fresh) {
            phase_singletons<NT>(S);
            t0 = clock64();
            if (S.status == BLU_OK) phase_setup_bump<NT>(S);
            if (tid == 0) S.t_phase[2] += clock64() - t0;
        } else bsync<NT>();
        if (S.status == BLU_OK && mode != BLU_MODE_BUILD) {
            phase_bump<NT>(S);
            if (mode == BLU_MODE_TAIL && S.status == BLU_OK) { bsync<NT>(); if (tid == 0) S.suspend = 2; bsync<NT>(); }
        }
        t0 = clock64();
        if (S.status == BLU_OK && !S.suspend) phase_build_factors<NT>(S);
        if (tid == 0) { if (!S.suspend) S.t_phase[9] += clock64() - t0; S.t_phase[11] += clock64() - tstart; }
        bsync<NT>();
        if (tid == 0) {
            BluInfo *I = S.M.info;
            I->rank = S.rank; I->rankdef = S.rankdef;
            I->nsearch_pivot = S.nsearch; I->nexpand = S.nexpand; I->ngarbage = S.ngarbage;
            I->factor_flops = S.factor_flops;
            I->elim_bytes = S.elim_bytes; I->nelim_div = S.nelim_div;
            if (fresh) I->elim_bytes_head = S.elim_bytes;
            I->w_half = S.w_half; I->w_used = S.w_used;
            I->cstamp = S.cstamp; I->rstamp = S.rstamp;
            I->nact = S.nact; I->ndead = S.ndead;
            I->dense_entries = S.dense_entries; I->dense_block_rank = S.dense_block_rank;
            for (int q = 0; q < 16; q++) I->t_phase[q] = S.t_phase[q];
            for (int q = 0; q < 8; q++) I->n_kind[q] = S.n_kind[q];
            int st = S.status;
            if (st == BLU_OK && S.suspend) st = S.suspend == 1 ? BLU_SUSPENDED_TAIL : BLU_SUSPENDED_BUILD;
            else if (st == BLU_OK) {
                I->nupdate = 0; I->nfactorize++;
                /* cost model, factorize.rs:160-166 */
                double factor_cost = 0.04 * (double)D.m + 0.07 * (double)I->matrix_nz + 0.20 * (double)I->bump_nz +
                                     0.20 * (double)I->nsearch_pivot + 0.008 * (double)I->factor_flops;
                I->update_cost_denom = factor_cost * 250.0;
                if (S.rank < D.m) st = BLU_WARNING_SINGULAR_MATRIX;
            }
            I->status = st;
        }
        bsync<NT>();
    }
}

#endif
