/* blu_slot_state.cuh -- what of a basis' slot is live between calls, read on the device from the slot's own state.  The
 * one place that states it: blu_batch_copy (blu_copy.cuh) moves exactly this from slot to slot, blu_batch_save /
 * blu_batch_restore (blu_save.cuh) move exactly this into and out of a byte image.
 *
 * The extents rule, per store (every extent clamped to the store's capacity, so a slot that was never factorized yields
 * whatever it holds):
 * - L (l_idx / l_val): [0, r_begin[nforrest]) -- column-wise L, row-wise L and the row etas (blu_factor_build.cuh:
 *   lt_begin_p[m] = r_begin[0]; blu_sparse.cuh: update appends at r_begin[nforrest]).  After a 'T' solve_for_update
 *   (btran_for_update >= 0) the pending row eta is [r_begin[nforrest], r_begin[nforrest + 1]) and is included.
 * - U (u_idx / u_val): [0, u_begin[m]) -- the columns of U (blu_factor_build.cuh: u_begin[m] = put).  After an 'N'
 *   solve_for_update (ftran_for_update >= 0) the pending spike follows at u_begin[m] and ends with a -1 index
 *   (blu_sparse.cuh); it is included up to and with that terminator.
 * - W (w_idx / w_val): the live half, [w_half * w_mem, w_used) (w_used is an offset into both halves, as k_store_regrow
 *   reads it); the other half is dead until the next garbage collection rewrites it.
 * - the row-wise copy of B (bt_idx / bt_val): [0, bt_ptr[m]).
 *
 * The state table: every O(m) array of Mat that carries state from one call to the next or must be zero / consistent
 * between calls, and BluInfo whole (marker, w_half, w_used, counters) as entry STATE_INFO.  Not in it, because every
 * kernel that reads them writes them first in the same call: ckey, rkey and ctree (Markowitz keys and their min-tree,
 * built by the factorization's setup), the dense-tail arrays dn_* (filled on entry to the tail), and gwork (per-warp
 * scatter space of the factorization; its first m entries, the xlhs of the sparse solves, are all-zero between calls in
 * every slot).  The resident B is not slot state either: it lives in the batch's b_i / b_x, addressed by the column
 * pointers of the basis. */
#ifndef BLU_SLOT_STATE_CUH
#define BLU_SLOT_STATE_CUH
#include "blu_dev_common.cuh"

/* X(index, Mat field, element type, elements as a function of M = m) */
#define BLU_STATE_TABLE(X)                                                                                              \
    X(0, bt_ptr, int, M + 1) X(1, pinv, int, M) X(2, qinv, int, M) X(3, prank, int, M) X(4, qrank, int, M)              \
    X(5, colpiv, double, M) X(6, rowpiv, double, M) X(7, lbeg, int, 2 * M) X(8, lend, int, 2 * M) X(9, lcap, int, 2 * M) \
    X(10, l_begin_p, int, M + 1) X(11, u_begin, int, M + 1) X(12, l_begin, int, M + 1) X(13, lt_begin, int, M + 1)      \
    X(14, lt_begin_p, int, M + 1) X(15, p, int, M + 1) X(16, r_begin, int, M + 1) X(17, eta_row, int, M + 1)            \
    X(18, dep_lt, int, M) X(19, dep_lc, int, M) X(20, dep_uc, int, M) X(21, len_uc, int, M)                             \
    X(22, pivotcol, int, 2 * M + 2) X(23, pivotrow, int, 2 * M + 2) X(24, rowmark, int, M) X(25, colmark, int, M)       \
    X(26, marked, int, M) X(27, iwork1, int, 2 * M + 2) X(28, pstack, int, M) X(29, acols, int, M)                      \
    X(30, tmpi, int, 4 * M + 4) X(31, cancelled, blu_u64, M) X(32, work0, double, M) X(33, work1, double, M)            \
    X(34, info, BluInfo, 1)
#define STATE_ARRAYS 35      /* entries of the table */
#define STATE_INFO 34        /* the entry that is BluInfo */
#define STATE_TMPI 30        /* the entry that is tmpi (k_build_ur's scratch) */

/* 4-byte words of entry a of the table for dimension m */
BLU_HD size_t state_words(int a, size_t M) {
    switch (a) {
#define SW(i, f, T, n) case i: return (size_t)(n) * sizeof(T) / 4;
    BLU_STATE_TABLE(SW)
#undef SW
    }
    return 0;
}

/* entry a of the table in the slot viewed by A, as 4-byte words (*nw of them) */
__device__ __forceinline__ unsigned *state_array(const Mat &A, int a, size_t *nw) {
    const size_t M = (size_t)A.m;
    switch (a) {
#define SA(i, f, T, n) case i: *nw = (size_t)(n) * sizeof(T) / 4; return (unsigned *)A.f;
    BLU_STATE_TABLE(SA)
#undef SA
    }
    *nw = 0;
    return nullptr;
}

__device__ __forceinline__ i64 clamp64(i64 v, i64 lo, i64 hi) { return v < lo ? lo : v > hi ? hi : v; }

/* the end of the live L: the row etas, with a pending one after a 'T' solve_for_update */
__device__ __forceinline__ i64 live_l_end(const Mat &S, const BluInfo &I) {
    const int m = S.m;
    const int nf = I.nforrest < 0 ? 0 : I.nforrest > m ? m : I.nforrest;
    const int e = (I.btran_for_update >= 0 && nf < m) ? nf + 1 : nf;
    return clamp64(S.r_begin[e], 0, S.l_mem);
}

/* the end of the live U: the columns of U, and after an 'N' solve_for_update the pending spike up to and with its -1
 * terminator.  Called by one whole warp; every lane gets the result. */
__device__ __forceinline__ i64 live_u_end(const Mat &S, const BluInfo &I) {
    const i64 put = clamp64(S.u_begin[S.m], 0, S.u_mem);
    i64 end = put;
    if (I.ftran_for_update >= 0) {
        end = S.u_mem;
        for (i64 b = put; b < S.u_mem; b += 32) {
            const i64 q = b + (threadIdx.x & 31);
            const unsigned tm = __ballot_sync(FULLMASK, q < S.u_mem && S.u_idx[q] < 0);
            if (tm) { end = b + __ffs((int)tm); break; }
        }
    }
    return end;
}

/* the start of the live half of W and the end of its fill */
__device__ __forceinline__ i64 live_w_lo(const Mat &S, const BluInfo &I) { return (i64)(I.w_half ? 1 : 0) * S.w_mem; }
__device__ __forceinline__ i64 live_w_end(const Mat &S, const BluInfo &I) {
    const i64 lo = live_w_lo(S, I);
    return clamp64(I.w_used, lo, lo + S.w_mem);
}

/* the end of the row-wise copy of B */
__device__ __forceinline__ i64 live_bt_end(const Mat &S) { return clamp64(S.bt_ptr[S.m], 0, S.bnz_cap); }

/* n 4-byte words from src to dst by the block: 16-byte accesses when both are aligned alike, 4-byte ones otherwise */
__device__ __forceinline__ void copy_words(unsigned *dst, const unsigned *src, size_t n) {
    const size_t t = threadIdx.x, nt = blockDim.x;
    if ((((size_t)dst ^ (size_t)src) & 15) == 0) {
        size_t head = ((16 - ((size_t)src & 15)) & 15) / 4;
        if (head > n) head = n;
        const size_t nv = (n - head) / 4;
        for (size_t q = t; q < head; q += nt) dst[q] = src[q];
        const uint4 *s4 = (const uint4 *)(src + head);
        uint4 *d4 = (uint4 *)(dst + head);
        for (size_t q = t; q < nv; q += nt) d4[q] = s4[q];
        for (size_t q = head + 4 * nv + t; q < n; q += nt) dst[q] = src[q];
    } else {
        for (size_t q = t; q < n; q += nt) dst[q] = src[q];
    }
}

#endif
