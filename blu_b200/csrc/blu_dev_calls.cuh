/* blu_dev_calls.cuh -- device side of the batch calls on caller-owned device buffers (blu_batch_factorize_subset_dev,
 * blu_batch_solve_for_update_dev, blu_batch_update_dev, blu_batch_solve_sparse_dev, blu_batch_solve_dense_multi_dev).
 * The factorization, the solves and the update are the batch kernels, run under the caller's per-slot run mask
 * (BluDev::run).  The kernels here check the caller's arguments, turn the internal status words into the caller's
 * statuses, and reduce what the host needs to know into a summary of DEV_SUM_N words, so that the host reads a fixed
 * number of bytes per launch whatever the size of the batch. */
#ifndef BLU_DEV_CALLS_CUH
#define BLU_DEV_CALLS_CUH
#include "blu_types.h"

/* the summary: the first non-OK status as (index << 32 | status) -- all ones when there is none --, the number of
 * Reallocate answers, the number of argument violations, and the new total / largest per-basis entry count of a
 * rebuilt resident B */
enum { DEV_SUM_FIRST = 0, DEV_SUM_REALLOC, DEV_SUM_BAD, DEV_SUM_TOTAL, DEV_SUM_MAXNZ, DEV_SUM_N };
#define DEV_SUM_NONE 0xffffffffffffffffULL

/* rhs_begin of a per-slot call (nmat + 1 offsets): those of every running slot within [0, rhs_begin[nmat]], which is
 * not negative; entries without an index array (irhs_missing) are a violation too */
__global__ void __launch_bounds__(256) k_dev_check_rhs(int n, const int *run, const blu_i64 *rhs_begin, int irhs_missing, blu_u64 *sum) {
    const blu_i64 tot = rhs_begin[n];
    int bad = blockIdx.x == 0 && threadIdx.x == 0 && (tot < 0 || (tot > 0 && irhs_missing));
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        if (run && !run[k]) continue;
        const blu_i64 b = rhs_begin[k], e = rhs_begin[k + 1];
        if (b < 0 || b > tot || e < 0 || e > tot) bad = 1;
    }
    if (bad) atomicAdd(&sum[DEV_SUM_BAD], 1ULL);
}

/* unit_begin (nmat + 1): starts at 0, never decreases, ends at nunits; rhs_begin of the units within
 * [0, rhs_begin[nunits]], which is not negative; entries without index or value arrays are a violation too */
__global__ void __launch_bounds__(256) k_dev_check_units(int nmat, const blu_i64 *unit_begin, blu_i64 nunits, const blu_i64 *rhs_begin,
                                                         int rhs_missing, blu_u64 *sum) {
    const blu_i64 t = (blu_i64)blockIdx.x * blockDim.x + threadIdx.x, T = (blu_i64)gridDim.x * blockDim.x;
    int bad = t == 0 && (unit_begin[0] != 0 || unit_begin[nmat] != nunits);
    for (blu_i64 k = t; k < nmat; k += T) if (unit_begin[k + 1] < unit_begin[k]) bad = 1;
    if (nunits > 0) {
        const blu_i64 tot = rhs_begin[nunits];
        if (t == 0 && (tot < 0 || (tot > 0 && rhs_missing))) bad = 1;
        for (blu_i64 u = t; u < nunits; u += T) { const blu_i64 b = rhs_begin[u]; if (b < 0 || b > tot) bad = 1; }
    }
    if (bad) atomicAdd(&sum[DEV_SUM_BAD], 1ULL);
}

/* B of a masked factorization: every column of a running slot within [0, bnz_total].  One block per slot. */
__global__ void __launch_bounds__(128) k_dev_check_b(int m, const int *run, const blu_i64 *b_begin, const blu_i64 *b_end, blu_i64 bnz_total,
                                                     blu_u64 *sum) {
    const int k = blockIdx.x;
    if (run && !run[k]) return;
    const size_t base = (size_t)k * m;
    int bad = 0;
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
        const blu_i64 b = b_begin[base + j], e = b_end[base + j];
        if (b < 0 || b > bnz_total || e < 0 || e > bnz_total) bad = 1;
    }
    if (bad) atomicAdd(&sum[DEV_SUM_BAD], 1ULL);
}

/* the basis of every unit of a validated unit_begin: the last k with unit_begin[k] <= u (bases without units have
 * unit_begin[k] == unit_begin[k + 1] and are skipped by the search) */
__global__ void __launch_bounds__(256) k_dev_unit_slots(int nmat, blu_i64 nunits, const blu_i64 *unit_begin, int *unit_slot) {
    for (blu_i64 u = (blu_i64)blockIdx.x * blockDim.x + threadIdx.x; u < nunits; u += (blu_i64)gridDim.x * blockDim.x) {
        int lo = 0, hi = nmat - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (unit_begin[mid] <= u) lo = mid; else hi = mid - 1;
        }
        unit_slot[u] = lo;
    }
}

/* unit u of a dense multi-right-hand-side call belongs to basis u / nrhs */
__global__ void __launch_bounds__(256) k_dev_dense_slots(blu_i64 nunits, blu_i64 nrhs, int *unit_slot) {
    for (blu_i64 u = (blu_i64)blockIdx.x * blockDim.x + threadIdx.x; u < nunits; u += (blu_i64)gridDim.x * blockDim.x)
        unit_slot[u] = (int)(u / nrhs);
}

/* pos[k] = k for a running slot, -1 otherwise: k_sub_lengths / k_sub_copy then read the new B of slot k at k * m,
 * the per-basis layout of the caller's arrays */
__global__ void __launch_bounds__(256) k_dev_pos(int n, const int *run, int *pos) {
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) pos[k] = (!run || run[k]) ? k : -1;
}

/* the status word of every slot's last factorization (for k_dev_finish) */
__global__ void __launch_bounds__(256) k_dev_info_status(int n, const BluInfo *info, int *scal) {
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) scal[k] = info[k].status;
}

/* Exclusive scan of the slots' entry counts tot[0..n) into slot_off; the total and the most entries of one running
 * slot (pos >= 0) go to the summary.  One block. */
__global__ void __launch_bounds__(256) k_dev_scan(int n, const int *pos, const blu_i64 *tot, blu_i64 *slot_off, blu_u64 *sum) {
    __shared__ blu_i64 part[256];
    const int t = threadIdx.x, per = (n + 255) / 256;
    const int k0 = t * per < n ? t * per : n, k1 = k0 + per < n ? k0 + per : n;
    blu_i64 s = 0, mx = 0;
    for (int k = k0; k < k1; k++) { s += tot[k]; if (pos[k] >= 0 && tot[k] > mx) mx = tot[k]; }
    part[t] = s;
    __syncthreads();
    if (t == 0) {
        blu_i64 acc = 0;
        for (int q = 0; q < 256; q++) { const blu_i64 v = part[q]; part[q] = acc; acc += v; }
        sum[DEV_SUM_TOTAL] = (blu_u64)acc;
    }
    __syncthreads();
    blu_i64 off = part[t];
    for (int k = k0; k < k1; k++) { slot_off[k] = off; off += tot[k]; }
    atomicMax(&sum[DEV_SUM_MAXNZ], (blu_u64)mx);
}

/* The caller's outputs of n slots or units (index idx0 + q) from the internal status words scal[q * stride] (nz in
 * scal[q * stride + 1]), only where run (if given) is set: status (may be null), nzlhs (null: not wanted; -1 on
 * error).  A Reallocate left over means a store could not grow and is reported as out of memory.  The first non-OK
 * index and the Reallocate count go to the summary. */
__global__ void __launch_bounds__(256) k_dev_finish(int n, blu_i64 idx0, const int *run, const int *scal, int stride, int *status,
                                                    blu_i64 *nzlhs, blu_u64 *sum) {
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        if (run && !run[q]) continue;
        int s = scal[(size_t)q * stride];
        if (s == BLU_REALLOCATE) { atomicAdd(&sum[DEV_SUM_REALLOC], 1ULL); s = BLU_ERROR_OUT_OF_MEMORY; }
        const blu_i64 i = idx0 + q;
        if (status) status[i] = s;
        if (nzlhs) nzlhs[i] = s == BLU_OK ? (blu_i64)scal[(size_t)q * stride + 1] : -1;
        if (s != BLU_OK) atomicMin(&sum[DEV_SUM_FIRST], ((blu_u64)i << 32) | (blu_u64)(unsigned)s);
    }
}

/* The solutions of a chunk of units, which k_solve_sparse<true> leaves back to back in the pool (unit b at off[b]),
 * to the caller's arrays at the unit's own offset b * m.  One block per unit. */
__global__ void __launch_bounds__(128) k_dev_unpack(int m, const int *scal, const blu_i64 *off, const blu_i64 *pi, const double *px,
                                                    blu_i64 *ilhs, double *xlhs) {
    const int b = blockIdx.x;
    if (scal[2 * b] != BLU_OK) return;
    const blu_i64 p = off[b], nz = scal[2 * b + 1];
    const size_t dst = (size_t)b * m;
    for (blu_i64 t = threadIdx.x; t < nz; t += blockDim.x) { ilhs[dst + t] = pi[p + t]; xlhs[dst + t] = px[p + t]; }
}

#endif
