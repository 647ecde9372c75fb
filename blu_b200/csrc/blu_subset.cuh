/* blu_subset.cuh -- device side of the batch calls on a subset of the bases (blu_batch_factorize_subset,
 * blu_batch_solve_for_update_subset).  The factorization, the solves and the update are the batch kernels run under
 * the per-slot run mask (BluDev::run); the kernels here rebuild the resident B of the batch (every basis keeps the B
 * it was last factorized from, the selected ones take their new B) and pack the selected solutions for one copy. */
#ifndef BLU_SUBSET_CUH
#define BLU_SUBSET_CUH
#include "blu_types.h"

/* One warp per slot k: the lengths of its m columns in the new resident B -- the r-th new B's for a selected slot
 * (pos[k] = r >= 0), the old ones otherwise -- into len, each column's offset inside the slot (exclusive scan of
 * the non-negative lengths) into off, and the slot's entries into tot[k].  A negative length is kept, so that the
 * factorization still answers InvalidArgument for that basis; an old column outside the old B (a basis whose last
 * factorization answered InvalidArgument for it) becomes length -1 for the same reason and is never read. */
__global__ void __launch_bounds__(32) k_sub_lengths(int m, const int *pos, const blu_i64 *ob, const blu_i64 *oe, blu_i64 ototal,
                                                    const blu_i64 *nb, const blu_i64 *ne, blu_i64 *len, blu_i64 *off, blu_i64 *tot) {
    const int k = blockIdx.x, lane = threadIdx.x & 31, r = pos[k];
    const size_t base = (size_t)k * m;
    blu_i64 put = 0;
    for (int j0 = 0; j0 < m; j0 += 32) {
        const int j = j0 + lane;
        blu_i64 n = 0;
        if (j < m) {
            if (r >= 0) n = ne[(size_t)r * m + j] - nb[(size_t)r * m + j];
            else {
                const blu_i64 b = ob[base + j], e = oe[base + j];
                n = (b < 0 || e > ototal) ? -1 : e - b;
            }
        }
        const blu_i64 v = n > 0 ? n : 0;
        blu_i64 incl = v;
        for (int d = 1; d < 32; d <<= 1) {
            const blu_i64 t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        if (j < m) { len[base + j] = n; off[base + j] = put + incl - v; }
        put += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) tot[k] = put;
}

/* The segmented copy into the new resident B: slot k starts at slot_off[k]; in place, off becomes b_begin and len
 * b_end (= b_begin + length, sign kept).  One thread per column. */
__global__ void __launch_bounds__(256) k_sub_copy(int m, const int *pos, const blu_i64 *ob, const blu_i64 *oi, const double *ox,
                                                  const blu_i64 *nb, const blu_i64 *ni, const double *nx, const blu_i64 *slot_off,
                                                  blu_i64 *off, blu_i64 *len, blu_i64 *bi, double *bx) {
    const int k = blockIdx.x, r = pos[k];
    const size_t base = (size_t)k * m;
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
        const blu_i64 b = slot_off[k] + off[base + j], n = len[base + j];
        const blu_i64 src = r >= 0 ? nb[(size_t)r * m + j] : ob[base + j];
        const blu_i64 *si = r >= 0 ? ni : oi;
        const double *sx = r >= 0 ? nx : ox;
        for (blu_i64 t = 0; t < n; t++) { bi[b + t] = si[src + t]; bx[b + t] = sx[src + t]; }
        off[base + j] = b; len[base + j] = b + n;
    }
}

/* The solutions of the selected slots back to back: the r-th selected slot sel[r] has its entries (at slot * m in
 * ilhs / xout) copied to [pack_off[r], pack_off[r+1]) of pi / px.  One block per selected slot. */
__global__ void __launch_bounds__(128) k_sub_pack(int m, const blu_i64 *sel, const blu_i64 *pack_off, const blu_i64 *ilhs, const double *xout,
                                                  blu_i64 *pi, double *px) {
    const int r = blockIdx.x;
    const size_t src = (size_t)sel[r] * m;
    const blu_i64 p = pack_off[r], n = pack_off[r + 1] - p;
    for (blu_i64 t = threadIdx.x; t < n; t += blockDim.x) { pi[p + t] = ilhs[src + t]; px[p + t] = xout[src + t]; }
}

#endif
