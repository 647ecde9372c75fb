/* blu_copy.cuh -- blu_batch_copy: basis dst becomes a copy of basis src within one batch (factors, update history, a
 * pending solve_for_update, every getter and the resident B's column pointers), so that a branch-and-bound or
 * strong-branching driver can start child LPs from a parent's basis without refactorizing or replaying its updates.
 *
 * The host gives the destination the source's store capacities first (same l_mem / u_mem / w_mem, a private store of
 * the same size where the source has one, the uniform store otherwise), so every offset inside a store -- r_begin,
 * u_begin, the W line table, w_used -- means the same in both slots and nothing is relocated.
 *
 * What is copied, per pair, with the extents read on the device from the source's own state:
 * - L (l_idx / l_val): [0, r_begin[nforrest]) -- column-wise L, row-wise L and the row etas (blu_factor_build.cuh:
 *   lt_begin_p[m] = r_begin[0]; blu_sparse.cuh: update appends at r_begin[nforrest]).  After a 'T' solve_for_update
 *   (btran_for_update >= 0) the pending row eta is [r_begin[nforrest], r_begin[nforrest + 1]) and is included.
 * - U (u_idx / u_val): [0, u_begin[m]) -- the columns of U (blu_factor_build.cuh: u_begin[m] = put).  After an 'N'
 *   solve_for_update (ftran_for_update >= 0) the pending spike follows at u_begin[m] and ends with a -1 index
 *   (blu_sparse.cuh); it is included up to and with that terminator.
 * - W (w_idx / w_val): the live half, [w_half * w_mem, w_used) (w_used is an offset into both halves, as k_store_regrow
 *   reads it); the other half is dead until the next garbage collection rewrites it.
 * - the row-wise copy of B (bt_idx / bt_val): [0, bt_ptr[m]).
 * - every O(m) array of Mat that carries state from one call to the next or must be zero / consistent between calls:
 *   bt_ptr, pinv, qinv, prank, qrank, colpiv, rowpiv, lbeg, lend, lcap, l_begin_p, u_begin, l_begin, lt_begin,
 *   lt_begin_p, p, r_begin, eta_row, dep_lt, dep_lc, dep_uc, len_uc, pivotcol, pivotrow, rowmark, colmark, marked,
 *   iwork1, pstack, acols, tmpi, cancelled, work0, work1 -- and BluInfo whole (marker, w_half, w_used, counters).
 * - the basis' rows of the library-owned resident B column pointers (bb / be), offsets into the one b_i / b_x.
 * Skipped, because every kernel that reads them writes them first in the same call: ckey, rkey and ctree (Markowitz
 * keys and their min-tree, built by the factorization's setup), the dense-tail arrays dn_* (filled on entry to the
 * tail), and gwork (per-warp scatter space of the factorization; its first m entries, the xlhs of the sparse solves,
 * are all-zero between calls in every slot, so the destination's already hold what the source's do).
 * Every extent is clamped to the store's capacity, so a source that was never factorized copies whatever it holds.
 *
 * Grid: one block per (copy pair, part).  Parts: COPY_CHUNKS chunks each of L, U, W and the row-wise B, one part per
 * O(m) array, one for BluInfo and one for the resident B rows -- a fan-out of one source to thousands of destinations
 * fills the GPU, and the many readers of one source's lines are served by L2. */
#ifndef BLU_COPY_CUH
#define BLU_COPY_CUH
#include "blu_dev_common.cuh"

#define COPY_CHUNKS 8
#define COPY_ARRAYS 35      /* the O(m) arrays and BluInfo */
#define COPY_PARTS (4 * COPY_CHUNKS + COPY_ARRAYS + 1)
#define COPY_THREADS 256

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

/* chunk c of COPY_CHUNKS of the elements [lo, hi) of an index array (4 bytes) and its value array (8 bytes) */
__device__ __forceinline__ void copy_chunk(int *di, double *dv, const int *si, const double *sv, i64 lo, i64 hi, int c) {
    if (hi <= lo) return;
    const i64 n = hi - lo, a = lo + n * c / COPY_CHUNKS, b = lo + n * (c + 1) / COPY_CHUNKS;
    copy_words((unsigned *)(di + a), (const unsigned *)(si + a), (size_t)(b - a));
    copy_words((unsigned *)(dv + a), (const unsigned *)(sv + a), (size_t)(b - a) * 2);
}

__device__ __forceinline__ i64 clamp64(i64 v, i64 lo, i64 hi) { return v < lo ? lo : v > hi ? hi : v; }

/* pairs[2r] = destination, pairs[2r + 1] = source; bb / be: the library-owned resident B column pointers (nmat * m) */
__global__ void __launch_bounds__(COPY_THREADS) k_copy_slots(BluDev D, const int *pairs, blu_i64 *bb, blu_i64 *be) {
    __shared__ Mat S, T;
    __shared__ i64 s_end;
    const int r = (int)(blockIdx.x / COPY_PARTS), part = (int)(blockIdx.x % COPY_PARTS);
    const int sd = pairs[2 * r], ss = pairs[2 * r + 1];
    if (threadIdx.x == 0) { mat_view(S, D, ss); mat_view(T, D, sd); }
    __syncthreads();
    const int m = S.m;
    const BluInfo &I = *S.info;
    if (part < 4 * COPY_CHUNKS) {
        const int kind = part / COPY_CHUNKS, c = part % COPY_CHUNKS;
        if (kind == 0) {
            const int nf = I.nforrest < 0 ? 0 : I.nforrest > m ? m : I.nforrest;
            const int e = (I.btran_for_update >= 0 && nf < m) ? nf + 1 : nf;
            copy_chunk(T.l_idx, T.l_val, S.l_idx, S.l_val, 0, clamp64(S.r_begin[e], 0, S.l_mem), c);
        } else if (kind == 1) {
            if (threadIdx.x < 32) {
                const i64 put = clamp64(S.u_begin[m], 0, S.u_mem);
                i64 end = put;
                if (I.ftran_for_update >= 0) {      /* the pending spike, up to and with its -1 terminator */
                    end = S.u_mem;
                    for (i64 b = put; b < S.u_mem; b += 32) {
                        const i64 q = b + threadIdx.x;
                        const unsigned tm = __ballot_sync(FULLMASK, q < S.u_mem && S.u_idx[q] < 0);
                        if (tm) { end = b + __ffs((int)tm); break; }
                    }
                }
                if (threadIdx.x == 0) s_end = end;
            }
            __syncthreads();
            copy_chunk(T.u_idx, T.u_val, S.u_idx, S.u_val, 0, s_end, c);
        } else if (kind == 2) {
            const i64 lo = (i64)(I.w_half ? 1 : 0) * S.w_mem;
            copy_chunk(T.w_idx, T.w_val, S.w_idx, S.w_val, lo, clamp64(I.w_used, lo, lo + S.w_mem), c);
        } else {
            copy_chunk(T.bt_idx, T.bt_val, S.bt_idx, S.bt_val, 0, clamp64(S.bt_ptr[m], 0, S.bnz_cap), c);
        }
        return;
    }
    const int a = part - 4 * COPY_CHUNKS;
    const size_t M = (size_t)m;
    const unsigned *src = nullptr; unsigned *dst = nullptr; size_t nw = 0;
#define CP(i, f, n) case i: src = (const unsigned *)S.f; dst = (unsigned *)T.f; nw = (size_t)(n) * sizeof(*S.f) / 4; break;
    switch (a) {
    CP(0, bt_ptr, M + 1) CP(1, pinv, M) CP(2, qinv, M) CP(3, prank, M) CP(4, qrank, M) CP(5, colpiv, M) CP(6, rowpiv, M)
    CP(7, lbeg, 2 * M) CP(8, lend, 2 * M) CP(9, lcap, 2 * M)
    CP(10, l_begin_p, M + 1) CP(11, u_begin, M + 1) CP(12, l_begin, M + 1) CP(13, lt_begin, M + 1) CP(14, lt_begin_p, M + 1)
    CP(15, p, M + 1) CP(16, r_begin, M + 1) CP(17, eta_row, M + 1)
    CP(18, dep_lt, M) CP(19, dep_lc, M) CP(20, dep_uc, M) CP(21, len_uc, M) CP(22, pivotcol, 2 * M + 2) CP(23, pivotrow, 2 * M + 2)
    CP(24, rowmark, M) CP(25, colmark, M) CP(26, marked, M) CP(27, iwork1, 2 * M + 2) CP(28, pstack, M) CP(29, acols, M)
    CP(30, tmpi, 4 * M + 4) CP(31, cancelled, M) CP(32, work0, M) CP(33, work1, M)
    CP(34, info, 1)
    default:      /* the resident B rows */
        copy_words((unsigned *)(bb + (size_t)sd * M), (const unsigned *)(bb + (size_t)ss * M), 2 * M);
        copy_words((unsigned *)(be + (size_t)sd * M), (const unsigned *)(be + (size_t)ss * M), 2 * M);
        return;
    }
#undef CP
    copy_words(dst, src, nw);
}

#endif
