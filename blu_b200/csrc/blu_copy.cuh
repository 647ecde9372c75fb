/* blu_copy.cuh -- blu_batch_copy: basis dst becomes a copy of basis src within one batch (factors, update history, a
 * pending solve_for_update, every getter and the resident B's column pointers), so that a branch-and-bound or
 * strong-branching driver can start child LPs from a parent's basis without refactorizing or replaying its updates.
 *
 * The host gives the destination the source's store capacities first (same l_mem / u_mem / w_mem, a private store of
 * the same size where the source has one, the uniform store otherwise), so every offset inside a store -- r_begin,
 * u_begin, the W line table, w_used -- means the same in both slots and nothing is relocated.
 *
 * What is copied, per pair: the live extent of each store and the state table, both as blu_slot_state.cuh states them,
 * and the basis' rows of the library-owned resident B column pointers (bb / be), offsets into the one b_i / b_x.
 *
 * Grid: one block per (copy pair, part).  Parts: COPY_CHUNKS chunks each of L, U, W and the row-wise B, one part per
 * O(m) array, one for BluInfo and one for the resident B rows -- a fan-out of one source to thousands of destinations
 * fills the GPU, and the many readers of one source's lines are served by L2. */
#ifndef BLU_COPY_CUH
#define BLU_COPY_CUH
#include "blu_slot_state.cuh"

#define COPY_CHUNKS 8
#define COPY_PARTS (4 * COPY_CHUNKS + STATE_ARRAYS + 1)
#define COPY_THREADS 256

/* chunk c of COPY_CHUNKS of the elements [lo, hi) of an index array (4 bytes) and its value array (8 bytes) */
__device__ __forceinline__ void copy_chunk(int *di, double *dv, const int *si, const double *sv, i64 lo, i64 hi, int c) {
    if (hi <= lo) return;
    const i64 n = hi - lo, a = lo + n * c / COPY_CHUNKS, b = lo + n * (c + 1) / COPY_CHUNKS;
    copy_words((unsigned *)(di + a), (const unsigned *)(si + a), (size_t)(b - a));
    copy_words((unsigned *)(dv + a), (const unsigned *)(sv + a), (size_t)(b - a) * 2);
}

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
            copy_chunk(T.l_idx, T.l_val, S.l_idx, S.l_val, 0, live_l_end(S, I), c);
        } else if (kind == 1) {
            if (threadIdx.x < 32) {
                const i64 end = live_u_end(S, I);
                if (threadIdx.x == 0) s_end = end;
            }
            __syncthreads();
            copy_chunk(T.u_idx, T.u_val, S.u_idx, S.u_val, 0, s_end, c);
        } else if (kind == 2) {
            copy_chunk(T.w_idx, T.w_val, S.w_idx, S.w_val, live_w_lo(S, I), live_w_end(S, I), c);
        } else {
            copy_chunk(T.bt_idx, T.bt_val, S.bt_idx, S.bt_val, 0, live_bt_end(S), c);
        }
        return;
    }
    const int a = part - 4 * COPY_CHUNKS;
    if (a == STATE_ARRAYS) {      /* the resident B rows */
        const size_t M = (size_t)m;
        copy_words((unsigned *)(bb + (size_t)sd * M), (const unsigned *)(bb + (size_t)ss * M), 2 * M);
        copy_words((unsigned *)(be + (size_t)sd * M), (const unsigned *)(be + (size_t)ss * M), 2 * M);
        return;
    }
    size_t nw = 0;
    const unsigned *src = state_array(S, a, &nw);
    unsigned *dst = state_array(T, a, &nw);
    copy_words(dst, src, nw);
}

#endif
