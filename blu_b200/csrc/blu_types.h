/* blu_types.h -- plain structs shared by the host layer and the CUDA kernels.
 *
 * Device data layout (one "slot" per basis matrix; a batch is an array of slots with
 * uniform strides so that slot s of every array is base + s*stride):
 *
 *   B (caller's format, copied verbatim)   b_begin[m] b_end[m] (i64)  b_i[] (i64)  b_x[] (f64)
 *   row-wise copy of B                      bt_ptr[m+1]  bt_idx[bnz]  bt_val[bnz]
 *   L store (col-wise | row-wise | etas)    l_idx[l_mem] l_val[l_mem]      (reference: lu.rs:137-138)
 *   U store (rows during elimination,
 *            col-wise + spike afterwards)   u_idx[u_mem] u_val[u_mem]      (lu.rs:139-140)
 *   W line file, two halves (ping-pong GC)  w_idx[2*w_mem] w_val[2*w_mem]  (lu.rs:141-142, file.rs)
 *   line table of W                         lbeg[2m] lend[2m] lcap[2m]
 *   Markowitz keys (count<<40 | stamp)      ckey[m] rkey[m]                (replaces list.rs buckets)
 *
 * Indices are 32-bit on the device (m < 2^31); the C ABI converts from/to the
 * reference's 64-bit usize/LUInt (lib.rs:32).
 */
#ifndef BLU_TYPES_H
#define BLU_TYPES_H
#include <stdint.h>
#include <stddef.h>

typedef unsigned long long blu_u64;
typedef long long blu_i64;

/* storage-order keys of one entry of the dense tail: (epoch << 8 | position), epoch = number of the dense
 * step that wrote the entry (0 = as found in the line file), position = place in that step's pivot column
 * (.c) / pivot row (.r).  Eight bits each: at most 255 steps and lines of at most 256 entries, hence
 * dense_k <= 256. */
struct BluKey2 { unsigned short c, r; };
#define BLU_DENSE_K_MAX 256

/* lu.rs:17-66, defaults lu.rs:250-259 */
struct BluParams {
    double droptol, abstol, reltol, stretch, compress_thres, sparse_thres;
    int nzbias;      /* >=0 <=> Some(_), <0 <=> None */
    int maxsearch, pad, search_rows;
};

/* Everything the getters of lu.rs:399-683 report, plus internal cursors. */
struct BluInfo {
    int status;
    int m, rank, rankdef, bump_size;
    int nupdate;            /* -1 <=> None */
    int nforrest, pivotlen, nfactorize;
    int ftran_for_update, btran_for_update; /* -1 <=> None */
    int marker;
    int w_half;             /* which half of W is live */
    int nact;               /* entries of the active-column list */
    int internal_error;     /* line number of a failed device-side invariant, 0 = none */
    int have_ur;            /* the sorted row-wise copy of U (ur_*) matches the current factors */
    int nruns;              /* how many times a factorization of this basis was started (Reallocate re-runs included) */
    int ndead, dense_entries, dense_block_rank; /* pivot-loop cursors carried from one kernel of a split factorization to the next */
    blu_i64 matrix_nz, bump_nz, l_nz, u_nz, r_nz;
    blu_i64 nsearch_pivot, nexpand, ngarbage, factor_flops;
    blu_i64 l_flops, u_flops, r_flops;
    blu_i64 addmem_l, addmem_u, addmem_w;
    blu_i64 nupdate_total, nforrest_total, nsymperm_total;
    blu_i64 w_used;         /* fill pointer of the live W half */
    blu_i64 cstamp, rstamp; /* monotone insertion stamps (FIFO order of list.rs:54) */
    blu_i64 nelim_div;
    double min_pivot, max_pivot, max_eta, pivot_error;
    double update_cost_numer, update_cost_denom;
    double elim_bytes;      /* algorithmic bytes of the elimination (SURVEY.md 8d) */
    double elim_bytes_head; /* the part of elim_bytes done by the head launch of a split factorization (= elim_bytes when not split) */
    double condest_l, condest_u, norm_l, norm_u, normest_l_inv, normest_u_inv;
    double onenorm, infnorm, residual_test;
    blu_i64 t_phase[16];    /* SM clock cycles per phase (thread 0): 0 validate+transpose 1 singleton queue 2 setup_bump 3 search 4 pivot singleton row 5 singleton col 6 doubleton 7 small 8 any 9 build_factors 10 remove_cols 11 total 12 dense-tail steps 13 dense-tail entry/exit conversions */
    blu_i64 n_kind[8];      /* pivots per variant, same numbering minus 4; 5 = steps taken in the dense tail, 6 = entries into it */
    blu_i64 norms_cycles[16]; /* SM cycles of the four warps of k_factor_norms: condest(L), condest(U), residual forward + norms, residual transposed */
};

/* Per-basis override of the L/U/W stores.  A batch starts with uniform strides (slot s of l_idx is
 * l_idx + s*l_mem); a basis that asks for more memory (Reallocate, blu.rs:95-118) gets private, larger stores
 * and runs again alone -- the other bases neither move nor re-run.  A null pointer = the uniform store. */
struct BluSlotStore {
    int *l_idx; double *l_val; int *u_idx; double *u_val; int *w_idx; double *w_val;
    blu_i64 l_mem, u_mem, w_mem;
};

/* Batch-wide device pointers.  Per-slot strides follow from m and the *_mem sizes. */
struct BluDev {
    int m, nmat;
    int slot0, nslot;   /* the range of slots this launch works on (a batch can be processed in pipelined chunks) */
    blu_i64 l_mem, u_mem, w_mem, bnz_cap;
    blu_i64 b_total;            /* entries of b_i / b_x: every column pointer must lie in [0, b_total] */
    const BluSlotStore *slot_store; /* nmat overrides (null pointers inside = uniform store), or null */
    const int *run;             /* nmat per-slot run flags of a batch launch (0: the slot is left untouched, status word included), or null: every slot runs */
    BluParams prm;
    /* input B */
    const blu_i64 *b_begin, *b_end, *b_i; /* b_begin/b_end: nmat*m; positions into b_i/b_x */
    const double *b_x;
    /* row-wise copy */
    int *bt_ptr; int *bt_idx; double *bt_val;
    /* permutations / pivots */
    int *pinv, *qinv;           /* m each; become pmap/qmap after build_factors */
    int *prank, *qrank;         /* m each: rank of row i / column j (kept for get_factors) */
    double *colpiv, *rowpiv;    /* m each */
    /* factors */
    int *l_idx; double *l_val;
    int *u_idx; double *u_val;
    int *w_idx; double *w_val;
    int *lbeg, *lend, *lcap;    /* 2m each */
    blu_u64 *ckey, *rkey;       /* m each */
    blu_u64 *ctree;             /* m/31 + 72 per basis: min-tree (fanout 32) over ckey for the Markowitz search of large bumps */
    int *l_begin_p, *u_begin;   /* m+1 each */
    int *l_begin, *lt_begin, *lt_begin_p, *p, *r_begin, *eta_row; /* m+1 each */
    int *len_uc;                  /* m: entries of the U column of pivot k */
    /* object API only (null in a batch): U row-wise, every row sorted by DESCENDING pivot position of the
     * column -- the order in which the reference's backward column sweep touches a row -- so that the U
     * solves and sweeps can run as wavefront dot products too (k_build_ur) */
    int *ur_ptr, *ur_idx, *dep_ur; double *ur_val;
    int *dep_lt, *dep_lc, *dep_uc; /* m each: furthest pivot position a row of L / column of L / column of U depends on (wavefront sweeps) */
    int *pivotcol, *pivotrow;   /* 2m+2 each */
    /* workspaces */
    int *rowmark, *colmark;     /* m each, zero between steps */
    int *marked;                /* m (iwork0 of the reference) */
    int *iwork1;                /* 2m+2 */
    int *pstack;                /* m */
    int *acols;                 /* m: active-column list for the Markowitz search */
    int *tmpi;                  /* 4m+4 scratch */
    blu_u64 *cancelled;         /* m */
    double *work0, *work1;      /* m each */
    double *gwork;              /* gwork_warps*m: per-warp scatter space when a pivot column exceeds the smem cache */
    int gwork_warps;
    /* dense tail (blu_factor_dense.cuh): the last dense_k x dense_k active submatrix as a row-major value
     * array, per-entry storage-order keys, and row/column presence bitmaps.  dense_k = 0: disabled. */
    int dense_k;
    int dense_kbig;             /* order of the first, HBM/L2-resident stage of the dense tail (BLU_P_DENSE_K_BIG; 0 = none) */
    int dense_kbig_eff;         /* ... as this launch uses it (0 unless the second stage is shared-memory resident and the CTA has a thread per slot) */
    int tree_min;               /* bumps with more columns than this search through the min-tree (ctree) */
    double *dn_val;             /* dense_k^2 per basis */
    BluKey2 *dn_key;            /* dense_k^2 per basis: (position key in its column, position key in its row) */
    BluKey2 *dn_key2;           /* the keys of the second stage (dense_k^2 per basis) when there are two */
    unsigned *dn_rbits, *dn_cbits; /* dense_k * dense_k/32 each per basis */
    BluInfo *info;              /* nmat */
};

/* shared-memory budgets of k_factorize (host and device agree on the carve-up) */
#define SMARK_MAX 8192   /* largest m whose row/column marks are kept in shared memory */
#define DENSE_STASH 4    /* candidate columns whose keys the dense-tail search leaves in shared memory for the pivot step */
#if defined(__CUDACC__)
#define BLU_HD __host__ __device__ static inline
#else
#define BLU_HD static inline
#endif
BLU_HD size_t blu_factor_smem_bytes(int cap, int nw, int m) {
    size_t n = (size_t)cap * 8 + (size_t)nw * cap * 8 + (size_t)cap * 4 * 2;
    if (m <= SMARK_MAX) n += (size_t)cap * 4 * 6 + (size_t)((m + 1) & ~1) * 2 + (size_t)((m + 15) & ~15);
    return n;
}
/* per-step arrays of the dense tail (always in shared memory) */
BLU_HD size_t blu_dense_smem_bytes(int kd) {
    return (((size_t)kd * (4 * 8 + 4 * 4 + 7 * 2 + DENSE_STASH * 4 + 4 + 4) + (size_t)(kd / 32) * 3 * 4) + 15) & ~(size_t)15;
}
/* with the presence bitmaps and the values in shared memory as well */
BLU_HD size_t blu_dense_smem_bytes_resident(int kd) {
    return blu_dense_smem_bytes(kd) + (size_t)2 * kd * (kd / 32) * 4 + (size_t)kd * kd * 8;
}

/* status codes live in the public header */
#include "blu_b200.h"
/* A batch factorization runs as three launches (blu_factor_build.cuh, k_factorize): the sparse head with many
 * small CTAs per SM, the dense tail with one CTA per SM and the active submatrix in shared memory, then
 * build_factors.  Between launches a basis is parked with one of these internal codes (never returned). */
#define BLU_SUSPENDED_TAIL 101
#define BLU_SUSPENDED_BUILD 102
#define BLU_MODE_WHOLE 0
#define BLU_MODE_HEAD 1
#define BLU_MODE_TAIL 2
#define BLU_MODE_BUILD 3

#endif
