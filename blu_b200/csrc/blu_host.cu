/* blu_host.cu -- host side of libblu_b200.so: owns device memory, copies, launches.
 * Mirrors struct BLU (reference src/blu.rs:9-395): the Reallocate protocol is hidden
 * here exactly as BLU::factorize / solve_for_update / update hide it (blu.rs:95-118,
 * 257-294, 319-334), by growing the L/U/W stores (lu_realloc_obj, blu.rs:345-377)
 * and re-running. */
#ifdef BLU_EMU
#include "cuda_emu.h"
#endif
#include "blu_types.h"
#include "blu_dev_common.cuh"
#include "blu_fact_launch.h"
#include "blu_solve.cuh"
#include "blu_sparse.cuh"
#include "blu_maxvolume.cuh"
#include "blu_subset.cuh"
#include "blu_dev_calls.cuh"
#include "blu_copy.cuh"
#include "blu_save.cuh"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include <algorithm>
#include <time.h>
#ifndef BLU_EMU
#include <thread>
#endif

#define PADDING 160 /* slack entries after the L/U/W stores: warp-wide terminator scans read up to 96 entries ahead */

/* Scratch of the batch solves with many right-hand sides per basis (blu_batch_solve_sparse,
 * blu_batch_solve_dense_multi).  One unit = one right-hand side of one basis; the units of a call go through
 * the pool in chunks of at most blu_b200::solve_units, one launch per chunk.  Allocated on first use. */
struct UnitPool {
    int64_t cap = 0;            /* units the sparse scratch holds */
    int *ints = nullptr, *markers = nullptr, *scal = nullptr; double *dbls = nullptr;   /* SpMulti layout; dbls all-zero between calls */
    int64_t *ilhs = nullptr, *off = nullptr; double *xout = nullptr; blu_u64 *fill = nullptr;   /* the solutions of a chunk, packed */
    int64_t dcap = 0;           /* units the dense scratch holds */
    double *rhs = nullptr, *lhs = nullptr, *work = nullptr; int *dstatus = nullptr;
    int64_t ucap = 0; int *slot = nullptr; int64_t *begin = nullptr;      /* per unit of a call: its basis, its right-hand side */
    int64_t rcap = 0; int64_t *irhs = nullptr; double *xrhs = nullptr;
    int64_t hcap = 0; int64_t *h_ilhs = nullptr; double *h_xout = nullptr;    /* pinned landing place of the packed solutions */
};

struct blu_b200 {
    int device;
    int single;                 /* created by blu_create (object API) */
    BluDev d;
    double realloc_factor;
    int nthreads;               /* CTA size of the factorization kernel */
    int tail_threads;           /* CTA size of the dense-tail launch of a split batch factorization */
    int num_sms, smem_optin;    /* device properties */
    int kd_smem_max;            /* largest dense-tail order whose values fit in shared memory */
    int want_kbig;              /* BLU_P_DENSE_K_BIG as asked for (alloc_dense clips it) */
    int split_min;              /* batches of more bases than this run as head / tail / build launches */
    int cap;                    /* smem line cache entries */
    std::vector<void *> allocs; /* every device allocation */
    std::vector<BluSlotStore> hslot; BluSlotStore *d_slot; /* per-basis store overrides (host mirror, device table) */
    std::vector<void *> ext_blocks; int have_overrides;     /* private stores of bases that outgrew the uniform ones */
    std::vector<void **> store_ptrs;
    /* resizable stores */
    cudaStream_t stream; int own_stream;
    cudaEvent_t ev0, ev1, ev_k[4];
    double last_ms[2], last_part_ms[3]; int parts_timed;
    int64_t launches;
    int nrealloc;
    int escape_realloc, task_pending;   /* blu_factorize_c0ntinue: Reallocate is handed to the caller; a Reallocate is pending */
    /* device staging for B, rhs, lhs, status */
    int64_t *db_begin, *db_end, *db_i; double *db_x; int64_t b_cap;
    double *d_rhs, *d_lhs; int *d_status;
    /* sparse-solve staging (object API) */
    int64_t *d_irhs; double *d_xrhs; int64_t *d_ilhs; double *d_xout; int *d_scal;
    int *h_scal; int64_t *h_ilhs; double *h_xout;   /* pinned */
    /* scratch of the batch basis-change calls (solve_for_update / update: whole batch, subset, _dev) and of maxvolume,
     * nothing else (ensure_batch_sparse): per basis the status word pair, the solution, the right-hand side's offsets,
     * and in sm_dbls one xtbl */
    int *sm_scal; double *sm_dbls, *sm_xout; int64_t *sm_ilhs, *sm_begin;
    int64_t *sm_irhs; double *sm_xrhs; int64_t smulti_rhs_cap;
    int solve_units;            /* largest chunk of units of a batch multi-RHS solve (BLU_B200_SOLVE_UNITS) */
    UnitPool up;
    int info_dirty;             /* device info block is newer than hinfo */
    int norms;                  /* run condest/residual_test after every factorization (factorize.rs:121-147) */
    cudaStream_t copy_stream, chunk_stream[4]; cudaEvent_t ev_up[16], ev_ch[4]; int have_pipe;   /* pipelined upload (blu_batch_factorize) */
    blu_i64 *d_chunk_end, *h_chunk_end;                                /* per-chunk max(b_end) */
    double last_norms_ms;
    /* get_factors staging */
    int64_t *gf_i; double *gf_x; int64_t gf_cap;
    std::vector<BluInfo> hinfo;
    std::vector<int64_t> hb_begin, hb_end, hb_i; std::vector<double> hb_x; /* compact staging (object API) */
    int have_b;                 /* B resident on device (for re-runs) */
    int b_external;             /* B lives in the caller's device buffers (blu_batch_factorize_dev) */
    cudaGraph_t graph; cudaGraphExec_t graph_exec; int have_graph; char graph_trans;   /* blu_batch_graph_* */
    std::vector<char> hrun;     /* host copy of d.run during a subset call (empty: every slot runs) */
    blu_u64 *d_sum, *h_sum;     /* the summary of a device-resident call (blu_dev_calls.cuh) and its pinned landing place */
    double time_factorize, time_solve, time_update;
};

static int cuda_ok(cudaError_t e, const char *what) {
    if (e != cudaSuccess) {
        fprintf(stderr, "blu_b200: CUDA error in %s: %s\n", what, cudaGetErrorString(e));
        return 0;
    }
    return 1;
}
#define CK(call) do { if (!cuda_ok((call), #call)) return BLU_ERROR_CUDA; } while (0)

template <typename T> static int dalloc(blu_b200 *o, T **p, size_t n) {
    void *q = nullptr;
    if (cudaMalloc(&q, (n ? n : 1) * sizeof(T)) != cudaSuccess) { cudaGetLastError(); return BLU_ERROR_OUT_OF_MEMORY; }
    /* cudaMemset of device memory returns before it has run, on the legacy stream -- which the library's
     * non-blocking streams do not wait for.  Without the synchronize, work queued right after an allocation
     * (the copy of the old content when a store grows) could be overtaken by the zero fill. */
    if (cudaMemset(q, 0, (n ? n : 1) * sizeof(T)) != cudaSuccess || cudaStreamSynchronize(0) != cudaSuccess) { cudaFree(q); return BLU_ERROR_CUDA; }
    *p = (T *)q;
    o->allocs.push_back(q);
    return BLU_OK;
}
static void dfree(blu_b200 *o, void *p) {
    if (!p) return;
    auto it = std::find(o->allocs.begin(), o->allocs.end(), p);
    if (it != o->allocs.end()) o->allocs.erase(it);
    cudaFree(p);
}

static int alloc_stores(blu_b200 *o) {
    BluDev &d = o->d;
    const size_t n = (size_t)d.nmat;
    int st;
    if ((st = dalloc(o, &d.l_idx, n * d.l_mem + PADDING))) return st;
    if ((st = dalloc(o, &d.l_val, n * d.l_mem + PADDING))) return st;
    if ((st = dalloc(o, &d.u_idx, n * d.u_mem + PADDING))) return st;
    if ((st = dalloc(o, &d.u_val, n * d.u_mem + PADDING))) return st;
    if (o->single) {
        if ((st = dalloc(o, &d.ur_idx, (size_t)d.u_mem + PADDING))) return st;
        if ((st = dalloc(o, &d.ur_val, (size_t)d.u_mem + PADDING))) return st;
    }
    if ((st = dalloc(o, &d.w_idx, n * 2 * d.w_mem + PADDING))) return st;
    if ((st = dalloc(o, &d.w_val, n * 2 * d.w_mem + PADDING))) return st;
    return BLU_OK;
}
/* Replace the L/U/W stores by ones of the sizes now in o->d.  The new stores are allocated first: if that
 * fails the old ones (and the old sizes) stay, so the object keeps working. */
struct StoreSet { int *l_idx, *u_idx, *w_idx, *ur_idx; double *l_val, *u_val, *w_val, *ur_val; };
static void free_stores(blu_b200 *o);
static int clear_overrides(blu_b200 *o);
static int swap_stores(blu_b200 *o, int64_t l_mem, int64_t u_mem, int64_t w_mem) {
    BluDev &d = o->d;
    const StoreSet old = {d.l_idx, d.u_idx, d.w_idx, d.ur_idx, d.l_val, d.u_val, d.w_val, d.ur_val};
    const blu_i64 ol = d.l_mem, ou = d.u_mem, ow = d.w_mem;
    d.l_mem = l_mem; d.u_mem = u_mem; d.w_mem = w_mem;
    d.l_idx = d.u_idx = d.w_idx = d.ur_idx = nullptr; d.l_val = d.u_val = d.w_val = d.ur_val = nullptr;
    int st = alloc_stores(o);
    if (st != BLU_OK) {
        free_stores(o);      /* whatever part of the new set was allocated */
        d.l_idx = old.l_idx; d.u_idx = old.u_idx; d.w_idx = old.w_idx; d.ur_idx = old.ur_idx;
        d.l_val = old.l_val; d.u_val = old.u_val; d.w_val = old.w_val; d.ur_val = old.ur_val;
        d.l_mem = ol; d.u_mem = ou; d.w_mem = ow;
        return st;
    }
    dfree(o, old.l_idx); dfree(o, old.l_val); dfree(o, old.u_idx); dfree(o, old.u_val);
    dfree(o, old.w_idx); dfree(o, old.w_val); dfree(o, old.ur_idx); dfree(o, old.ur_val);
    return clear_overrides(o);
}
static void free_stores(blu_b200 *o) {
    BluDev &d = o->d;
    dfree(o, d.l_idx); dfree(o, d.l_val); dfree(o, d.u_idx); dfree(o, d.u_val); dfree(o, d.w_idx); dfree(o, d.w_val);
    dfree(o, d.ur_idx); dfree(o, d.ur_val); d.ur_idx = nullptr; d.ur_val = nullptr;
    d.l_idx = d.u_idx = d.w_idx = nullptr; d.l_val = d.u_val = d.w_val = nullptr;
}

/* drop every per-basis override (their content is gone or has been folded into the uniform stores) */
static int clear_overrides(blu_b200 *o) {
    if (!o->d_slot) return BLU_OK;
    for (void *p : o->ext_blocks) dfree(o, p);
    o->ext_blocks.clear();
    BluSlotStore z; memset(&z, 0, sizeof z);
    o->hslot.assign((size_t)o->d.nmat, z);
    o->have_overrides = 0;
    if (cudaMemcpy(o->d_slot, o->hslot.data(), o->hslot.size() * sizeof(BluSlotStore), cudaMemcpyHostToDevice) != cudaSuccess || cudaStreamSynchronize(0) != cudaSuccess) return BLU_ERROR_CUDA;
    return BLU_OK;
}

/* the dense-tail arrays (blu_factor_dense.cuh); dense_k = 0 disables the dense tail */
static void free_dense(blu_b200 *o) {
    BluDev &d = o->d;
    dfree(o, d.dn_val); dfree(o, d.dn_key); dfree(o, d.dn_key2); dfree(o, d.dn_rbits); dfree(o, d.dn_cbits);
    d.dn_val = nullptr; d.dn_key = nullptr; d.dn_key2 = nullptr; d.dn_rbits = d.dn_cbits = nullptr;
}
static int alloc_dense(blu_b200 *o, int want, int want_big) {
    BluDev &d = o->d;
    free_dense(o);
    int kd = want < 0 ? 0 : want;
    const int mcap = (d.m + 31) & ~31;
    if (kd > mcap) kd = mcap;
    kd &= ~31;
    if (kd > BLU_DENSE_K_MAX) kd = BLU_DENSE_K_MAX;
    int kb = want_big < 0 ? 0 : want_big;
    if (kb > mcap) kb = mcap;
    kb &= ~31;
    if (kb > BLU_DENSE_K_MAX) kb = BLU_DENSE_K_MAX;
    /* the first stage only exists in front of a shared-memory resident second one */
    if (kd == 0 || kd > o->kd_smem_max || kb <= kd) kb = 0;
    d.dense_k = kd; d.dense_kbig = kb; d.dense_kbig_eff = 0;
    const size_t n = (size_t)d.nmat, k = (size_t)(kb > kd ? kb : kd);
    /* up to kd_smem_max the values live in shared memory (blu_factor_dense.cuh); beyond, in HBM */
    int st = dalloc(o, &d.dn_val, (kb || k > (size_t)o->kd_smem_max) ? n * k * k : 1);
    if (st == BLU_OK) st = dalloc(o, &d.dn_key, n * k * k);
    if (st == BLU_OK) st = dalloc(o, &d.dn_key2, kb ? n * (size_t)kd * kd : 1);
    if (st == BLU_OK) st = dalloc(o, &d.dn_rbits, n * k * (k / 32));
    if (st == BLU_OK) st = dalloc(o, &d.dn_cbits, n * k * (k / 32));
    if (st != BLU_OK) { free_dense(o); d.dense_k = 0; d.dense_kbig = 0; }
    return st;
}

/* like (blu_clone): the new object takes like's L/U/W capacities and dense-tail sizes instead of the defaults */
static int create_common(blu_b200 **out, int64_t nmat, int64_t m, int64_t bnz_cap, int device, int single, const blu_b200 *like = nullptr) {
    if (!out || m < 1 || nmat < 1 || bnz_cap < 0 || m > 0x7fffff /* line counts live in 23 bits of the search keys, blu_dev_common.cuh:mkckey */) return BLU_ERROR_INVALID_ARGUMENT;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
        fprintf(stderr, "blu_b200: no CUDA device (this library has no CPU path)\n");
        return BLU_ERROR_CUDA;
    }
    if (device >= 0) CK(cudaSetDevice(device)); else CK(cudaGetDevice(&device));
    blu_b200 *o = new blu_b200();
    o->device = device; o->single = single;
    o->realloc_factor = 1.5;   /* blu.rs:68 */
    o->nthreads = 128; o->cap = 256; o->tail_threads = 512;
    o->num_sms = 148; o->smem_optin = 232448;
    cudaDeviceGetAttribute(&o->num_sms, cudaDevAttrMultiProcessorCount, device);
    cudaDeviceGetAttribute(&o->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    o->kd_smem_max = 0;
    for (int kd = 32; kd <= BLU_DENSE_K_MAX; kd += 32)
        if (blu_dense_smem_bytes_resident(kd) + 4096 /* static Shm */ <= (size_t)o->smem_optin) o->kd_smem_max = kd;
    /* always split when the tail is shared-memory resident: a launch configured for 200+ KB of shared memory leaves
     * the sparse head almost no L1 (measured on configs[2]: pivot_any 6.4 -> 10.5 Gcycles in one whole launch) */
    o->split_min = 0;
    if (const char *e = getenv("BLU_B200_CAP")) { int c = atoi(e); if (c >= 64 && c <= 4096) o->cap = c & ~31; }   /* tuning knob: entries of the shared-memory line caches */
    o->launches = 0; o->nrealloc = 0; o->last_ms[0] = o->last_ms[1] = 0.0; o->last_part_ms[0] = o->last_part_ms[1] = o->last_part_ms[2] = 0.0;
    o->d_slot = nullptr; o->have_overrides = 0; o->escape_realloc = 0; o->task_pending = 0;
    o->b_external = 0; o->have_graph = 0;
    o->have_b = 0; o->info_dirty = 0; o->norms = 1; o->last_norms_ms = 0.0;
    o->have_pipe = 0; o->d_chunk_end = nullptr; o->h_chunk_end = nullptr;
    o->sm_scal = nullptr; o->sm_dbls = o->sm_xout = nullptr; o->sm_ilhs = o->sm_begin = nullptr;
    o->sm_irhs = nullptr; o->sm_xrhs = nullptr; o->smulti_rhs_cap = 0;
    o->solve_units = 8192;      /* configs[1], 16,384 units (DESIGN.md §5): beyond this the kernels gain ~10 %, the call nothing */
    if (const char *e = getenv("BLU_B200_SOLVE_UNITS")) { long v = atol(e); if (v >= 1 && v <= (1L << 24)) o->solve_units = (int)v; }   /* tuning / test knob */
    o->h_scal = nullptr; o->h_ilhs = nullptr; o->h_xout = nullptr;
    o->d_sum = nullptr; o->h_sum = nullptr;
    o->time_factorize = o->time_solve = o->time_update = 0.0;
    BluDev &d = o->d;
    memset(&d, 0, sizeof d);
    d.m = (int)m; d.nmat = (int)nmat; d.bnz_cap = bnz_cap < 1 ? 1 : bnz_cap;
    d.slot0 = 0; d.nslot = (int)nmat;
    /* lu.rs:245-259.  The reference starts every store at b_nz and grows on demand; the
     * device build starts larger because a Reallocate costs a full re-run here. */
    d.l_mem = d.u_mem = 8 * d.bnz_cap + 4 * m;
    d.w_mem = 24 * d.bnz_cap + 16 * m;     /* room for the fill of the sparse head without garbage collection (measured on configs[1]: 8*nnz + 8*m collects 1.4 times per basis and costs 10 %) */
    if (like) { d.l_mem = like->d.l_mem; d.u_mem = like->d.u_mem; d.w_mem = like->d.w_mem; }
    d.prm.droptol = 1e-20; d.prm.abstol = 1e-14; d.prm.reltol = 0.1;
    d.prm.nzbias = 1; d.prm.maxsearch = 3; d.prm.pad = 4; d.prm.stretch = 0.3;
    d.prm.compress_thres = 0.5; d.prm.sparse_thres = 0.05; d.prm.search_rows = 0;
    d.gwork_warps = 32;
    d.tree_min = 4096;
    if (const char *e = getenv("BLU_B200_TREE_MIN")) d.tree_min = atoi(e);      /* tuning / test knob, same as BLU_P_TREE_MIN */
    const size_t n = (size_t)nmat, M = (size_t)m;
    int st = BLU_OK;
#define A(p, cnt) if (st == BLU_OK) st = dalloc(o, &(p), (cnt))
    A(d.bt_ptr, n * (M + 1)); A(d.bt_idx, n * d.bnz_cap); A(d.bt_val, n * d.bnz_cap);
    A(d.pinv, n * M); A(d.qinv, n * M); A(d.prank, n * M); A(d.qrank, n * M);
    A(d.colpiv, n * M); A(d.rowpiv, n * M);
    A(d.lbeg, n * 2 * M); A(d.lend, n * 2 * M); A(d.lcap, n * 2 * M);
    A(d.ckey, n * M); A(d.rkey, n * M); A(d.ctree, n * (M / 31 + 72));
    A(d.l_begin_p, n * (M + 1)); A(d.u_begin, n * (M + 1)); A(d.l_begin, n * (M + 1));
    A(d.lt_begin, n * (M + 1)); A(d.lt_begin_p, n * (M + 1)); A(d.p, n * (M + 1));
    A(d.r_begin, n * (M + 1)); A(d.eta_row, n * (M + 1));
    A(d.dep_lt, n * M); A(d.dep_lc, n * M); A(d.dep_uc, n * M); A(d.len_uc, n * M);
    A(d.pivotcol, n * (2 * M + 2)); A(d.pivotrow, n * (2 * M + 2));
    A(d.rowmark, n * M); A(d.colmark, n * M); A(d.marked, n * M);
    A(d.iwork1, n * (2 * M + 2)); A(d.pstack, n * M); A(d.acols, n * M); A(d.tmpi, n * (4 * M + 4));
    A(d.cancelled, n * M); A(d.work0, n * M); A(d.work1, n * M);
    A(d.gwork, n * (size_t)d.gwork_warps * M);
    A(d.info, n);
    A(o->d_slot, n);
    A(o->db_begin, n * M); A(o->db_end, n * M);
    A(o->d_rhs, n * M); A(o->d_lhs, n * M); A(o->d_status, n);
    if (single) { A(o->d_irhs, M); A(o->d_xrhs, M); A(o->d_ilhs, M); A(o->d_xout, M); A(o->d_scal, 16); A(d.ur_ptr, M + 1); A(d.dep_ur, M); }
#undef A
    o->b_cap = 0; o->db_i = nullptr; o->db_x = nullptr;
    o->gf_i = nullptr; o->gf_x = nullptr; o->gf_cap = 0;
    if (st == BLU_OK) st = alloc_stores(o);
    if (st == BLU_OK) { d.slot_store = o->d_slot; st = clear_overrides(o); }
    if (st == BLU_OK) {
        /* two-stage tail for batches: measured on configs[1] (profiles/r2u_sweep_two_stage.txt) 224 and 256 are within 1 % of each other and 8 % ahead of one stage */
        int kd = o->kd_smem_max, kb = single ? 0 : 256;
        if (const char *e = getenv("BLU_B200_DENSE_K")) kd = atoi(e);      /* tuning knob, same as BLU_P_DENSE_K */
        if (const char *e = getenv("BLU_B200_DENSE_K_BIG")) kb = atoi(e);  /* tuning knob, same as BLU_P_DENSE_K_BIG */
        if (like) { kd = like->d.dense_k; kb = like->want_kbig; }
        o->want_kbig = kb;
        st = alloc_dense(o, kd, kb);
    }
    if (st == BLU_OK) {
        /* nupdate = None until the first factorization (lu.rs:329-331) */
        o->hinfo.assign(n, BluInfo());
        for (auto &I : o->hinfo) { memset(&I, 0, sizeof I); I.nupdate = -1; I.m = (int)m; I.ftran_for_update = I.btran_for_update = -1; I.update_cost_denom = 1.0; }
        /* (pageable host memory: the call may return with the DMA still in flight on the legacy stream, which the
         * library's non-blocking stream does not wait for -- hence the synchronize) */
        if (cudaMemcpy(d.info, o->hinfo.data(), n * sizeof(BluInfo), cudaMemcpyHostToDevice) != cudaSuccess || cudaStreamSynchronize(0) != cudaSuccess) st = BLU_ERROR_CUDA;
    }
    if (st == BLU_OK && single) {
        if (cudaMallocHost((void **)&o->h_scal, 16 * sizeof(int)) != cudaSuccess ||
            cudaMallocHost((void **)&o->h_ilhs, M * sizeof(int64_t)) != cudaSuccess ||
            cudaMallocHost((void **)&o->h_xout, M * sizeof(double)) != cudaSuccess) st = BLU_ERROR_OUT_OF_MEMORY;
    }
    if (st == BLU_OK && cudaStreamCreateWithFlags(&o->stream, cudaStreamNonBlocking) != cudaSuccess) st = BLU_ERROR_CUDA;
    o->own_stream = 1;
#ifndef BLU_EMU
    if (st == BLU_OK && (cudaEventCreate(&o->ev0) != cudaSuccess || cudaEventCreate(&o->ev1) != cudaSuccess)) st = BLU_ERROR_CUDA;
    for (int q = 0; q < 4 && st == BLU_OK; q++) if (cudaEventCreate(&o->ev_k[q]) != cudaSuccess) st = BLU_ERROR_CUDA;
#endif
    if (st != BLU_OK) {
        for (void *p : o->allocs) cudaFree(p);
        if (o->h_scal) cudaFreeHost(o->h_scal);
        if (o->h_ilhs) cudaFreeHost(o->h_ilhs);
        if (o->h_xout) cudaFreeHost(o->h_xout);
        delete o;
        return st;
    }
    *out = o;
    return BLU_OK;
}

static void destroy_common(blu_b200 *o) {
    if (!o) return;
    cudaSetDevice(o->device);
    cudaStreamSynchronize(o->stream);
    for (void *p : o->allocs) cudaFree(p);
    if (o->h_scal) cudaFreeHost(o->h_scal);
    if (o->h_ilhs) cudaFreeHost(o->h_ilhs);
    if (o->h_xout) cudaFreeHost(o->h_xout);
    if (o->up.h_ilhs) cudaFreeHost(o->up.h_ilhs);
    if (o->up.h_xout) cudaFreeHost(o->up.h_xout);
    if (o->h_sum) cudaFreeHost(o->h_sum);
#ifndef BLU_EMU
    cudaEventDestroy(o->ev0); cudaEventDestroy(o->ev1);
    for (int q = 0; q < 4; q++) cudaEventDestroy(o->ev_k[q]);
#endif
    if (o->have_pipe) {
#ifndef BLU_EMU
        for (int i = 0; i < 16; i++) cudaEventDestroy(o->ev_up[i]);
        for (int i = 0; i < 4; i++) { cudaEventDestroy(o->ev_ch[i]); cudaStreamDestroy(o->chunk_stream[i]); }
#endif
        cudaStreamDestroy(o->copy_stream);
        cudaFreeHost(o->h_chunk_end);
    }
#ifndef BLU_EMU
    if (o->have_graph) { cudaGraphExecDestroy(o->graph_exec); cudaGraphDestroy(o->graph); }
#endif
    if (o->own_stream) cudaStreamDestroy(o->stream);
    delete o;
}

static int ensure_b_cap(blu_b200 *o, int64_t total) {
    if (total <= o->b_cap) return BLU_OK;
    dfree(o, o->db_i); dfree(o, o->db_x);
    o->db_i = nullptr; o->db_x = nullptr;
    int st = dalloc(o, &o->db_i, (size_t)total);
    if (st == BLU_OK) st = dalloc(o, &o->db_x, (size_t)total);
    if (st == BLU_OK) o->b_cap = total;
    return st;
}

static void timer_start(blu_b200 *o) {
#ifndef BLU_EMU
    cudaEventRecord(o->ev0, o->stream);
#endif
}
static void timer_stop(blu_b200 *o, int which) {
#ifndef BLU_EMU
    cudaEventRecord(o->ev1, o->stream);
    cudaEventSynchronize(o->ev1);
    float ms = 0; cudaEventElapsedTime(&ms, o->ev0, o->ev1);
    o->last_ms[which] = ms;
#else
    o->last_ms[which] = 0.0;
#endif
}

static int launch_factorize_mode(blu_b200 *o, cudaStream_t stream, int slot0, int nslot, int nt, int mode, int rerun) {
    const int kd = o->d.dense_k;
    const bool dense_here = kd > 0 && (mode == BLU_MODE_WHOLE || mode == BLU_MODE_TAIL);
    const bool resident = dense_here && kd <= o->kd_smem_max;
    if (nt != 32 && nt != 64 && nt != 256 && nt != 512 && nt != 1024) nt = 128;
    size_t smem = blu_factor_smem_bytes(o->cap, nt / 32, o->d.m);
    if (dense_here) smem = std::max(smem, resident ? blu_dense_smem_bytes_resident(kd) : blu_dense_smem_bytes(kd));
    BluDev dv = o->d; dv.slot0 = slot0; dv.nslot = nslot;
    /* the first (HBM/L2) stage of the dense tail: the launch that runs it has the second stage in shared memory and a
     * thread per slot (dense_restage); the head of a split factorization stops where that launch takes over */
    {
        const int run_nt = mode == BLU_MODE_HEAD ? o->tail_threads : nt;
        const bool res2 = kd > 0 && kd <= o->kd_smem_max && mode != BLU_MODE_BUILD;
        dv.dense_kbig_eff = (res2 && o->d.dense_kbig > kd && run_nt >= o->d.dense_kbig) ? o->d.dense_kbig : 0;
        if (dv.dense_kbig_eff && dense_here)
            smem = std::max(smem, blu_dense_smem_bytes(dv.dense_kbig_eff) + (size_t)2 * dv.dense_kbig_eff * (dv.dense_kbig_eff / 32) * 4);
    }
    int e;
    switch (nt) {
    case 32: e = blu_launch_factorize_32(stream, dv, nslot, o->cap, mode, kd, resident ? 1 : 0, rerun, smem); break;
    case 64: e = blu_launch_factorize_64(stream, dv, nslot, o->cap, mode, kd, resident ? 1 : 0, rerun, smem); break;
    case 256: e = blu_launch_factorize_256(stream, dv, nslot, o->cap, mode, kd, resident ? 1 : 0, rerun, smem); break;
    case 512: e = blu_launch_factorize_512(stream, dv, nslot, o->cap, mode, kd, resident ? 1 : 0, rerun, smem); break;
    case 1024: e = blu_launch_factorize_1024(stream, dv, nslot, o->cap, mode, kd, resident ? 1 : 0, rerun, smem); break;
    default: e = blu_launch_factorize_128(stream, dv, nslot, o->cap, mode, kd, resident ? 1 : 0, rerun, smem); break;
    }
    o->launches++;
    CK((cudaError_t)e);
    return BLU_OK;
}
/* One launch for a single basis or a small batch.  A large batch whose dense tail fits in shared memory runs
 * as three launches: the sparse head wants many small CTAs per SM (the pivot loop is a latency chain), the
 * tail one CTA per SM with the whole active submatrix on chip, build_factors many small CTAs again. */
static int launch_factorize(blu_b200 *o, cudaStream_t stream, int slot0, int nslot, int rerun = 0) {
    const int kd = o->d.dense_k;
    const bool timed = stream == o->stream;      /* (the pipelined chunks overlap: no per-launch times there) */
    auto mark = [&](int q) {
#ifndef BLU_EMU
        if (timed) cudaEventRecord(o->ev_k[q], stream);
#endif
    };
    o->parts_timed = 0;
    if (kd > 0 && kd <= o->kd_smem_max && nslot > o->split_min) {
        mark(0);
        int st = launch_factorize_mode(o, stream, slot0, nslot, o->nthreads, BLU_MODE_HEAD, rerun);
        mark(1);
        if (st == BLU_OK) st = launch_factorize_mode(o, stream, slot0, nslot, o->tail_threads, BLU_MODE_TAIL, 0);
        mark(2);
        if (st == BLU_OK) st = launch_factorize_mode(o, stream, slot0, nslot, o->nthreads, BLU_MODE_BUILD, 0);
        mark(3);
        if (timed) o->parts_timed = 3;
        return st;
    }
    mark(0);
    int st = launch_factorize_mode(o, stream, slot0, nslot, o->nthreads, BLU_MODE_WHOLE, rerun);
    mark(1);
    if (timed) o->parts_timed = 1;
    return st;
}

/* blu.rs:345-377 for a batch: every basis that answered Reallocate gets private stores of
 * realloc_factor * (mem + addmem) entries (only the kinds it asked for); nobody else moves. */
static int grow_hungry_slots(blu_b200 *o) {
    BluDev &d = o->d;
    const double f = o->realloc_factor < 1.0 ? 1.0 : o->realloc_factor;
    struct Need { int k; int64_t l, u, w; };
    std::vector<Need> needs;
    size_t bytes = 0;
    auto rnd = [](size_t b) { return (b + 255) & ~(size_t)255; };
    for (int k = 0; k < d.nmat; k++) {
        const BluInfo &I = o->hinfo[(size_t)k];
        if (I.status != BLU_REALLOCATE || (!o->hrun.empty() && !o->hrun[(size_t)k])) continue;
        const BluSlotStore &e = o->hslot[(size_t)k];
        Need n = {k, 0, 0, 0};
        if (I.addmem_l > 0) n.l = (int64_t)(f * (double)((e.l_idx ? e.l_mem : d.l_mem) + I.addmem_l)) + 1;
        if (I.addmem_u > 0) n.u = (int64_t)(f * (double)((e.u_idx ? e.u_mem : d.u_mem) + I.addmem_u)) + 1;
        if (I.addmem_w > 0) n.w = (int64_t)(f * (double)((e.w_idx ? e.w_mem : d.w_mem) + I.addmem_w)) + 1;
        if (n.l > 0x3fffffff || n.u > 0x3fffffff || n.w > 0x1fffffff) return BLU_ERROR_OUT_OF_MEMORY;
        if (!n.l && !n.u && !n.w) return BLU_ERROR_INTERNAL;
        if (n.l) bytes += rnd((size_t)(n.l + PADDING) * 4) + rnd((size_t)(n.l + PADDING) * 8);
        if (n.u) bytes += rnd((size_t)(n.u + PADDING) * 4) + rnd((size_t)(n.u + PADDING) * 8);
        if (n.w) bytes += rnd((size_t)(2 * n.w + PADDING) * 4) + rnd((size_t)(2 * n.w + PADDING) * 8);
        needs.push_back(n);
    }
    if (needs.empty()) return BLU_OK;
    unsigned char *blk = nullptr;
    int st = dalloc(o, &blk, bytes);
    if (st != BLU_OK) return st;
    o->ext_blocks.push_back(blk);
    size_t off = 0;
    auto take = [&](size_t b) { unsigned char *p = blk + off; off += rnd(b); return p; };
    for (const Need &n : needs) {
        BluSlotStore &e = o->hslot[(size_t)n.k];
        if (n.l) { e.l_idx = (int *)take((size_t)(n.l + PADDING) * 4); e.l_val = (double *)take((size_t)(n.l + PADDING) * 8); e.l_mem = n.l; }
        if (n.u) { e.u_idx = (int *)take((size_t)(n.u + PADDING) * 4); e.u_val = (double *)take((size_t)(n.u + PADDING) * 8); e.u_mem = n.u; }
        if (n.w) { e.w_idx = (int *)take((size_t)(2 * n.w + PADDING) * 4); e.w_val = (double *)take((size_t)(2 * n.w + PADDING) * 8); e.w_mem = n.w; }
    }
    o->have_overrides = 1;
    CK(cudaMemcpyAsync(o->d_slot, o->hslot.data(), o->hslot.size() * sizeof(BluSlotStore), cudaMemcpyHostToDevice, o->stream));
    CK(cudaStreamSynchronize(o->stream));
    o->nrealloc++;
    return BLU_OK;
}

static int fetch_info(blu_b200 *o) {
    CK(cudaMemcpyAsync(o->hinfo.data(), o->d.info, (size_t)o->d.nmat * sizeof(BluInfo), cudaMemcpyDeviceToHost, o->stream));
    CK(cudaStreamSynchronize(o->stream));
    return BLU_OK;
}

static int ensure_info(blu_b200 *o) {
    if (!o->info_dirty) return BLU_OK;
    if (cudaSetDevice(o->device) != cudaSuccess) return BLU_ERROR_CUDA;
    int st = fetch_info(o);
    if (st == BLU_OK) o->info_dirty = 0;
    return st;
}

/* factorize what is resident in db_*; loops on Reallocate like blu.rs:95-118 */
static int factorize_resident(blu_b200 *o, int hungry_known = 0, int escape_realloc = 0) {
    CK(cudaSetDevice(o->device));
    BluDev &d = o->d;
    if (!o->b_external) {
        d.b_begin = (const blu_i64 *)o->db_begin; d.b_end = (const blu_i64 *)o->db_end;
        d.b_i = (const blu_i64 *)o->db_i; d.b_x = o->db_x;
    }
    double total_ms = 0.0;
    if (hungry_known && !o->single) {      /* a pipelined first pass already ran: hinfo says who wants more memory */
        int st = grow_hungry_slots(o);
        if (st != BLU_OK) return st;
        total_ms = o->last_ms[0];
    } else hungry_known = 0;
    for (int attempt = hungry_known ? 1 : 0; attempt < 40; attempt++) {
        timer_start(o);
        /* after the first pass only the bases that asked for more memory run again (batches) */
        int st = launch_factorize(o, o->stream, 0, d.nmat, attempt > 0 && !o->single);
        if (st != BLU_OK) return st;
        timer_stop(o, 0);
        total_ms += o->last_ms[0];
#ifndef BLU_EMU
        for (int q = 0; q < 3; q++) {
            float pm = 0;
            if (q < o->parts_timed) cudaEventElapsedTime(&pm, o->ev_k[q], o->ev_k[q + 1]);
            o->last_part_ms[q] = pm;
        }
#endif
        if ((st = fetch_info(o)) != BLU_OK) return st;
        int64_t al = 0, au = 0, aw = 0; int need = 0;
        for (size_t k = 0; k < o->hinfo.size(); k++) {
            const BluInfo &I = o->hinfo[k];
            /* (a masked-out slot may still say Reallocate from a call that ran out of memory: it does not run here) */
            if (I.status == BLU_REALLOCATE && (o->hrun.empty() || o->hrun[k])) { need = 1; al = std::max<int64_t>(al, I.addmem_l); au = std::max<int64_t>(au, I.addmem_u); aw = std::max<int64_t>(aw, I.addmem_w); }
        }
        if (!need) {
            if (o->single && d.ur_idx) {   /* sorted row-wise U for the wavefront U sweeps (object API) */
                BLU_LAUNCH(k_build_ur, 1, 256, 0, o->stream, d);
                o->launches++;
                CK(cudaGetLastError());
            }
            /* factorize.rs:121-147: condest(L), condest(U), residual_test (+ matrix_norm) */
            if (o->norms) {
                timer_start(o);
                BLU_LAUNCH(k_factor_norms, d.nmat, 128, 0, o->stream, d);
                o->launches++;
                CK(cudaGetLastError());
                timer_stop(o, 0);
                total_ms += o->last_ms[0];
                o->last_norms_ms = o->last_ms[0];
                if ((st = fetch_info(o)) != BLU_OK) return st;
            }
            o->last_ms[0] = total_ms;
            return BLU_OK;
        }
        if (escape_realloc) { o->last_ms[0] = total_ms; return BLU_REALLOCATE; }      /* the free-function surface: the caller grows the stores (lib.rs:11-19) */
        /* lu_realloc_obj, blu.rs:345-377 */
        if (!o->single) {
            if ((st = grow_hungry_slots(o)) != BLU_OK) return st;
            continue;
        }
        double f = o->realloc_factor < 1.0 ? 1.0 : o->realloc_factor;
        const int64_t nl = al > 0 ? (int64_t)(f * (double)(d.l_mem + al)) + 1 : d.l_mem;
        const int64_t nu = au > 0 ? (int64_t)(f * (double)(d.u_mem + au)) + 1 : d.u_mem;
        const int64_t nw = aw > 0 ? (int64_t)(f * (double)(d.w_mem + aw)) + 1 : d.w_mem;
        if (nl > 0x3fffffff || nu > 0x3fffffff || nw > 0x1fffffff) return BLU_ERROR_OUT_OF_MEMORY;
        if ((st = swap_stores(o, nl, nu, nw)) != BLU_OK) return st;
        o->nrealloc++;
    }
    return BLU_ERROR_INTERNAL;
}

/* ------------------------------------------------------------------ */
/* batch API                                                           */
/* ------------------------------------------------------------------ */
extern "C" int blu_batch_create(blu_batch_t **out, int64_t nmat, int64_t m, int64_t bnz_cap, int device) {
    return create_common(out, nmat, m, bnz_cap, device, 0);
}
extern "C" void blu_batch_destroy(blu_batch_t *b) { destroy_common(b); }

extern "C" int blu_batch_upload(blu_batch_t *o, const int64_t *b_begin, const int64_t *b_end,
                                const int64_t *b_i, const double *b_x, int64_t bnz_total, const double *rhs) {
    if (!o) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const size_t n = (size_t)o->d.nmat, m = (size_t)o->d.m;
    if (b_begin) {
        if (!b_end || bnz_total < 0 || (bnz_total > 0 && (!b_i || !b_x))) return BLU_ERROR_INVALID_ARGUMENT;
        int st = ensure_b_cap(o, bnz_total);
        if (st != BLU_OK) return st;
        CK(cudaMemcpyAsync(o->db_begin, b_begin, n * m * sizeof(int64_t), cudaMemcpyHostToDevice, o->stream));
        CK(cudaMemcpyAsync(o->db_end, b_end, n * m * sizeof(int64_t), cudaMemcpyHostToDevice, o->stream));
        if (bnz_total > 0) {
            CK(cudaMemcpyAsync(o->db_i, b_i, (size_t)bnz_total * sizeof(int64_t), cudaMemcpyHostToDevice, o->stream));
            CK(cudaMemcpyAsync(o->db_x, b_x, (size_t)bnz_total * sizeof(double), cudaMemcpyHostToDevice, o->stream));
        }
        o->have_b = 1; o->b_external = 0;
        o->d.b_total = bnz_total;
    }
    if (rhs) CK(cudaMemcpyAsync(o->d_rhs, rhs, n * m * sizeof(double), cudaMemcpyHostToDevice, o->stream));
    CK(cudaStreamSynchronize(o->stream));
    return BLU_OK;
}

extern "C" int blu_batch_factorize_resident(blu_batch_t *o) {
    if (!o || !o->have_b) return BLU_ERROR_INVALID_CALL;
    return factorize_resident(o);
}

static int solve_dense_resident(blu_b200 *o, char trans) {
    CK(cudaSetDevice(o->device));
    timer_start(o);
    BLU_LAUNCH(k_solve_dense, o->d.nmat, 32, 0, o->stream, o->d, (const double *)o->d_rhs, o->d_lhs, trans, o->d_status, (double *)nullptr, 0, (const int *)nullptr);
    o->launches++;
    CK(cudaGetLastError());
    timer_stop(o, 1);
    return BLU_OK;
}
extern "C" int blu_batch_solve_dense_resident(blu_batch_t *o, char trans) {
    if (!o) return BLU_ERROR_INVALID_ARGUMENT;
    return solve_dense_resident(o, trans);
}

/* SURVEY.md 8(f) N4 -- caller-owned DEVICE buffers: nothing is staged or copied, everything is queued on the
 * batch's stream.  B must stay valid and unchanged until the next factorization of this batch. */
extern "C" int blu_batch_factorize_dev(blu_batch_t *o, const int64_t *d_b_begin, const int64_t *d_b_end,
                                       const int64_t *d_b_i, const double *d_b_x, int64_t bnz_total) {
    if (!o || !d_b_begin || !d_b_end || bnz_total < 0 || (bnz_total > 0 && (!d_b_i || !d_b_x))) return BLU_ERROR_INVALID_ARGUMENT;
    BluDev &d = o->d;
    d.b_begin = (const blu_i64 *)d_b_begin; d.b_end = (const blu_i64 *)d_b_end;
    d.b_i = (const blu_i64 *)d_b_i; d.b_x = d_b_x; d.b_total = bnz_total;
    o->b_external = 1; o->have_b = 1;
    return factorize_resident(o);
}
extern "C" int blu_batch_solve_dense_dev(blu_batch_t *o, const double *d_rhs, double *d_lhs, char trans, int *d_status) {
    if (!o || !d_rhs || !d_lhs) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    timer_start(o);
    BLU_LAUNCH(k_solve_dense, o->d.nmat, 32, 0, o->stream, o->d, d_rhs, d_lhs, trans, d_status ? d_status : o->d_status, (double *)nullptr, 0, (const int *)nullptr);
    o->launches++;
    CK(cudaGetLastError());
    timer_stop(o, 1);
    return BLU_OK;
}

/* The steady-state step of a resident batch -- the factorization launches, condest/residual_test and solve_dense
 * -- captured once into a CUDA graph and replayed with one launch call.  A replay in which some basis answers
 * Reallocate falls back to the classic path (grow that basis, re-run it) before the solve is repeated. */
extern "C" int blu_batch_graph_capture(blu_batch_t *o, char trans) {
    if (!o || !o->have_b) return BLU_ERROR_INVALID_CALL;
    CK(cudaSetDevice(o->device));
#ifndef BLU_EMU
    if (o->have_graph) { cudaGraphExecDestroy(o->graph_exec); cudaGraphDestroy(o->graph); o->have_graph = 0; }
    BluDev &d = o->d;
    if (!o->b_external) { d.b_begin = (const blu_i64 *)o->db_begin; d.b_end = (const blu_i64 *)o->db_end; d.b_i = (const blu_i64 *)o->db_i; d.b_x = o->db_x; }
    CK(cudaStreamSynchronize(o->stream));
    cudaStream_t cap = nullptr;      /* (a stream of its own: launch_factorize records timing events only on o->stream) */
    CK(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
    CK(cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal));
    int st = launch_factorize(o, cap, 0, d.nmat);
    if (st == BLU_OK && o->norms) { BLU_LAUNCH(k_factor_norms, d.nmat, 128, 0, cap, d); o->launches++; }
    if (st == BLU_OK) { BLU_LAUNCH(k_solve_dense, d.nmat, 32, 0, cap, d, (const double *)o->d_rhs, o->d_lhs, trans, o->d_status, (double *)nullptr, 0, (const int *)nullptr); o->launches++; }
    cudaError_t e = cudaStreamEndCapture(cap, &o->graph);
    cudaStreamDestroy(cap);
    if (st != BLU_OK) return st;
    CK(e);
    CK(cudaGraphInstantiate(&o->graph_exec, o->graph, 0));
#endif
    o->have_graph = 1; o->graph_trans = trans;
    return BLU_OK;
}
extern "C" int blu_batch_graph_launch(blu_batch_t *o) {
    if (!o || !o->have_graph) return BLU_ERROR_INVALID_CALL;
    CK(cudaSetDevice(o->device));
#ifndef BLU_EMU
    timer_start(o);
    CK(cudaGraphLaunch(o->graph_exec, o->stream));
    timer_stop(o, 0);
    int st = fetch_info(o);
    if (st != BLU_OK) return st;
    bool hungry = false;
    for (auto &I : o->hinfo) hungry = hungry || I.status == BLU_REALLOCATE;
    if (!hungry) return BLU_OK;
    if ((st = factorize_resident(o, 1)) != BLU_OK) return st;      /* blu.rs:95-118 for the bases that asked */
    return solve_dense_resident(o, o->graph_trans);
#else
    int st = factorize_resident(o);
    return st != BLU_OK ? st : solve_dense_resident(o, o->graph_trans);
#endif
}

extern "C" int blu_batch_download(blu_batch_t *o, double *lhs, int *status) {
    if (!o) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const size_t n = (size_t)o->d.nmat, m = (size_t)o->d.m;
    if (lhs) CK(cudaMemcpyAsync(lhs, o->d_lhs, n * m * sizeof(double), cudaMemcpyDeviceToHost, o->stream));
    if (status) CK(cudaMemcpyAsync(status, o->d_status, n * sizeof(int), cudaMemcpyDeviceToHost, o->stream));
    CK(cudaStreamSynchronize(o->stream));
    return BLU_OK;
}

/* max(b_end) over the columns of each chunk of bases: tells which part of b_i / b_x a chunk needs */
__global__ void k_chunk_ranges(const blu_i64 *b_end, blu_i64 cols_per_chunk, blu_i64 ncols, blu_i64 *out) {
    /* gridDim.x = chunks * gridDim.y-way split: blockIdx.x = chunk, blockIdx.y = slice of the chunk */
    __shared__ blu_i64 sm[256];
    const blu_i64 c0 = (blu_i64)blockIdx.x * cols_per_chunk;
    blu_i64 c1 = c0 + cols_per_chunk; if (c1 > ncols) c1 = ncols;
    blu_i64 mx = 0;
    for (blu_i64 q = c0 + (blu_i64)blockIdx.y * blockDim.x + threadIdx.x; q < c1; q += (blu_i64)gridDim.y * blockDim.x) { const blu_i64 e = b_end[q]; mx = e > mx ? e : mx; }
    sm[threadIdx.x] = mx;
    __syncthreads();
    for (int d = 128; d > 0; d >>= 1) { if ((int)threadIdx.x < d && sm[threadIdx.x + d] > sm[threadIdx.x]) sm[threadIdx.x] = sm[threadIdx.x + d]; __syncthreads(); }
    if (threadIdx.x == 0) atomicMax((unsigned long long *)&out[blockIdx.x], (unsigned long long)(sm[0] > 0 ? sm[0] : 0));
}

/* Upload B in pieces on a copy stream and start the factorization of a chunk of bases as soon as the
 * part of b_i / b_x its columns point into has arrived, so that only the first piece of the transfer is
 * exposed.  Returns BLU_OK when every basis finished without asking for more memory; BLU_REALLOCATE
 * when the classic path (grow + re-run, B is resident by then) has to take over. */
#ifndef BLU_EMU
static int factorize_pipelined(blu_b200 *o, const int64_t *b_begin, const int64_t *b_end,
                               const int64_t *b_i, const double *b_x, int64_t bnz_total) {
    BluDev &d = o->d;
    const int n = d.nmat, NCH = 4, NP = 8;
    const size_t m = (size_t)d.m;
    if (!o->have_pipe) {
        CK(cudaStreamCreateWithFlags(&o->copy_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 16; i++) CK(cudaEventCreateWithFlags(&o->ev_up[i], cudaEventDisableTiming));
        for (int i = 0; i < 4; i++) { CK(cudaStreamCreateWithFlags(&o->chunk_stream[i], cudaStreamNonBlocking)); CK(cudaEventCreateWithFlags(&o->ev_ch[i], cudaEventDisableTiming)); }
        CK(cudaMallocHost((void **)&o->h_chunk_end, 16 * sizeof(blu_i64)));
        int st = dalloc(o, &o->d_chunk_end, 16);
        if (st != BLU_OK) return st;
        o->have_pipe = 1;
    }
    int st = ensure_b_cap(o, bnz_total);
    if (st != BLU_OK) return st;
    cudaStream_t cs = o->copy_stream;
    /* whatever the caller queued on the compute stream before must not be overtaken */
    CK(cudaEventRecord(o->ev_up[15], o->stream));
    CK(cudaStreamWaitEvent(cs, o->ev_up[15], 0));
    CK(cudaMemcpyAsync(o->db_begin, b_begin, (size_t)n * m * sizeof(int64_t), cudaMemcpyHostToDevice, cs));
    CK(cudaMemcpyAsync(o->db_end, b_end, (size_t)n * m * sizeof(int64_t), cudaMemcpyHostToDevice, cs));
    const int per = (n + NCH - 1) / NCH;
    CK(cudaMemsetAsync(o->d_chunk_end, 0, 16 * sizeof(blu_i64), cs));
    k_chunk_ranges<<<dim3(NCH, 148), 256, 0, cs>>>((const blu_i64 *)o->db_end, (blu_i64)per * (blu_i64)m, (blu_i64)n * (blu_i64)m, o->d_chunk_end);
    o->launches++;
    CK(cudaMemcpyAsync(o->h_chunk_end, o->d_chunk_end, NCH * sizeof(blu_i64), cudaMemcpyDeviceToHost, cs));
    CK(cudaEventRecord(o->ev_up[14], cs));
    const int64_t psz = (bnz_total + NP - 1) / NP;
    for (int p = 0; p < NP; p++) {
        const int64_t lo = (int64_t)p * psz, hi = std::min<int64_t>(bnz_total, lo + psz);
        if (hi > lo) {
            CK(cudaMemcpyAsync(o->db_i + lo, b_i + lo, (size_t)(hi - lo) * sizeof(int64_t), cudaMemcpyHostToDevice, cs));
            CK(cudaMemcpyAsync(o->db_x + lo, b_x + lo, (size_t)(hi - lo) * sizeof(double), cudaMemcpyHostToDevice, cs));
        }
        CK(cudaEventRecord(o->ev_up[p], cs));
    }
    o->have_b = 1; o->b_external = 0;
    d.b_total = bnz_total;
    CK(cudaEventSynchronize(o->ev_up[14]));        /* the chunk ranges are on the host now */
    d.b_begin = (const blu_i64 *)o->db_begin; d.b_end = (const blu_i64 *)o->db_end;
    d.b_i = (const blu_i64 *)o->db_i; d.b_x = o->db_x;
    timer_start(o);
    for (int c = 0; c < NCH; c++) {
        const int s0 = c * per, ns = std::min(per, n - s0);
        if (ns <= 0) break;
        int64_t need = o->h_chunk_end[c];
        if (need > bnz_total) need = bnz_total;     /* pointers beyond b_total: the kernel answers InvalidArgument (phase_validate_transpose) */
        const int p = psz > 0 && need > 0 ? (int)std::min<int64_t>(NP - 1, (need - 1) / psz) : 0;
        /* each chunk on its own stream: the next chunk fills the SMs while this one drains */
        cudaStream_t ks = o->chunk_stream[c];
        CK(cudaStreamWaitEvent(ks, o->ev0, 0));
        CK(cudaStreamWaitEvent(ks, o->ev_up[p], 0));
        if ((st = launch_factorize(o, ks, s0, ns)) != BLU_OK) return st;
        CK(cudaEventRecord(o->ev_ch[c], ks));
        CK(cudaStreamWaitEvent(o->stream, o->ev_ch[c], 0));
    }
    CK(cudaStreamWaitEvent(o->stream, o->ev_up[NP - 1], 0));
    timer_stop(o, 0);
    double total_ms = o->last_ms[0];
    if ((st = fetch_info(o)) != BLU_OK) return st;
    for (auto &I : o->hinfo) if (I.status == BLU_REALLOCATE) return BLU_REALLOCATE;
    if (o->norms) {
        timer_start(o);
        BLU_LAUNCH(k_factor_norms, d.nmat, 128, 0, o->stream, d);
        o->launches++;
        CK(cudaGetLastError());
        timer_stop(o, 0);
        total_ms += o->last_ms[0];
        o->last_norms_ms = o->last_ms[0];
        if ((st = fetch_info(o)) != BLU_OK) return st;
    }
    o->last_ms[0] = total_ms;
    return BLU_OK;
}
#endif

extern "C" int blu_batch_factorize(blu_batch_t *o, const int64_t *b_begin, const int64_t *b_end,
                                   const int64_t *b_i, const double *b_x, int64_t bnz_total, int *status) {
    if (!o || !b_begin || !b_end) return BLU_ERROR_INVALID_ARGUMENT;
    int st;
#ifndef BLU_EMU
    if (o->d.nmat >= 256 && bnz_total > 0 && b_i && b_x) {
        CK(cudaSetDevice(o->device));
        st = factorize_pipelined(o, b_begin, b_end, b_i, b_x, bnz_total);
        if (st == BLU_REALLOCATE) st = factorize_resident(o, 1);      /* B is resident: grow the bases that asked and re-run them */
    } else
#endif
    {
        st = blu_batch_upload(o, b_begin, b_end, b_i, b_x, bnz_total, nullptr);
        if (st != BLU_OK) return st;
        st = factorize_resident(o);
    }
    if (st != BLU_OK) return st;
    if (status) for (int k = 0; k < o->d.nmat; k++) status[k] = o->hinfo[k].status;
    return BLU_OK;
}

extern "C" int blu_batch_solve_dense(blu_batch_t *o, const double *rhs, double *lhs, char trans, int *status) {
    if (!o || !rhs || !lhs) return BLU_ERROR_INVALID_ARGUMENT;
    int st = blu_batch_upload(o, nullptr, nullptr, nullptr, nullptr, 0, rhs);
    if (st != BLU_OK) return st;
    st = solve_dense_resident(o, trans);
    if (st != BLU_OK) return st;
    return blu_batch_download(o, lhs, status);
}

extern "C" void *blu_batch_stream(blu_batch_t *o) { return o ? (void *)o->stream : nullptr; }
extern "C" int blu_batch_set_stream(blu_batch_t *o, void *s) {
    if (!o) return BLU_ERROR_INVALID_ARGUMENT;
    cudaStreamSynchronize(o->stream);
    if (o->own_stream) cudaStreamDestroy(o->stream);
    o->stream = (cudaStream_t)s; o->own_stream = 0;
    return BLU_OK;
}
extern "C" int blu_batch_synchronize(blu_batch_t *o) {
    if (!o) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaStreamSynchronize(o->stream));
    return BLU_OK;
}
extern "C" double blu_batch_last_kernel_ms(blu_batch_t *o, int which) {
    if (!o) return 0.0;
    if (which == 2) return o->last_norms_ms;
    if (which >= 3 && which <= 5) return o->last_part_ms[which - 3];
    return which >= 0 && which < 2 ? o->last_ms[which] : 0.0;
}
extern "C" int64_t blu_batch_launch_count(blu_batch_t *o) { return o ? o->launches : 0; }

static double info_value(blu_b200 *o, const BluInfo &I, int what) {
    switch (what) {
    case BLU_I_M: return I.m;
    case BLU_I_RANK: return I.rank;
    case BLU_I_BUMP_SIZE: return I.bump_size;
    case BLU_I_BUMP_NZ: return (double)I.bump_nz;
    case BLU_I_MATRIX_NZ: return (double)I.matrix_nz;
    case BLU_I_L_NZ: return (double)I.l_nz;
    case BLU_I_U_NZ: return (double)I.u_nz;
    case BLU_I_R_NZ: return (double)I.r_nz;
    case BLU_I_NSEARCH_PIVOT: return (double)I.nsearch_pivot;
    case BLU_I_NEXPAND: return (double)I.nexpand;
    case BLU_I_NGARBAGE: return (double)I.ngarbage;
    case BLU_I_FACTOR_FLOPS: return (double)I.factor_flops;
    case BLU_I_MIN_PIVOT: return I.min_pivot;
    case BLU_I_MAX_PIVOT: return I.max_pivot;
    case BLU_I_MAX_ETA: return I.max_eta;
    case BLU_I_NUPDATE: return I.nupdate;
    case BLU_I_NFORREST: return I.nforrest;
    case BLU_I_NFACTORIZE: return I.nfactorize;
    case BLU_I_NUPDATE_TOTAL: return (double)I.nupdate_total;
    case BLU_I_NFORREST_TOTAL: return (double)I.nforrest_total;
    case BLU_I_NSYMPERM_TOTAL: return (double)I.nsymperm_total;
    case BLU_I_L_FLOPS: return (double)I.l_flops;
    case BLU_I_U_FLOPS: return (double)I.u_flops;
    case BLU_I_R_FLOPS: return (double)I.r_flops;
    case BLU_I_CONDEST_L: return I.condest_l;
    case BLU_I_CONDEST_U: return I.condest_u;
    case BLU_I_NORM_L: return I.norm_l;
    case BLU_I_NORM_U: return I.norm_u;
    case BLU_I_NORMEST_L_INV: return I.normest_l_inv;
    case BLU_I_NORMEST_U_INV: return I.normest_u_inv;
    case BLU_I_ONENORM: return I.onenorm;
    case BLU_I_INFNORM: return I.infnorm;
    case BLU_I_RESIDUAL_TEST: return I.residual_test;
    case BLU_I_PIVOT_ERROR: return I.pivot_error;
    case BLU_I_UPDATE_COST: return I.update_cost_numer / I.update_cost_denom; /* lu.rs:324 */
    case BLU_I_TIME_FACTORIZE: return o->time_factorize;
    case BLU_I_TIME_SOLVE: return o->time_solve;
    case BLU_I_TIME_UPDATE: return o->time_update;
    case BLU_I_ELIM_BYTES: return I.elim_bytes;
    case BLU_I_NELIM_DIV: return (double)I.nelim_div;
    case BLU_I_PIVOTLEN: return I.pivotlen;
    case BLU_I_RANKDEF: return I.rankdef;
    case BLU_I_INTERNAL_ERROR: return I.internal_error;
    case BLU_I_STATUS: return I.status;
    case BLU_I_NREALLOC: return o->nrealloc;
    case BLU_I_NRUNS: return I.nruns;
    case BLU_I_ADDMEM_L: return (double)I.addmem_l;
    case BLU_I_ADDMEM_U: return (double)I.addmem_u;
    case BLU_I_ADDMEM_W: return (double)I.addmem_w;
    case BLU_I_ELIM_BYTES_HEAD: return I.elim_bytes_head;
    default:
        if (what >= BLU_I_T_PHASE0 && what < BLU_I_T_PHASE0 + 16) return (double)I.t_phase[what - BLU_I_T_PHASE0];
        if (what >= BLU_I_N_KIND0 && what < BLU_I_N_KIND0 + 8) return (double)I.n_kind[what - BLU_I_N_KIND0];
        if (what >= BLU_I_NORMS_CYC0 && what < BLU_I_NORMS_CYC0 + 16) return (double)I.norms_cycles[what - BLU_I_NORMS_CYC0];
        return 0.0;
    }
}
extern "C" double blu_batch_get_info(blu_batch_t *o, int64_t k, int what) {
    if (!o || k < 0 || k >= o->d.nmat) return 0.0;
    if (what < 100) return blu_get_param(o, what);
    if (ensure_info(o) != BLU_OK) return 0.0;
    return info_value(o, o->hinfo[(size_t)k], what);
}

extern "C" int blu_set_param(blu_t *o, int what, double v) {
    if (!o) return BLU_ERROR_INVALID_ARGUMENT;
    BluParams &p = o->d.prm;
    switch (what) {
    case BLU_P_DROPTOL: p.droptol = v; break;
    case BLU_P_ABSTOL: p.abstol = v; break;
    case BLU_P_RELTOL: p.reltol = v; break;
    case BLU_P_NZBIAS: p.nzbias = (int)v; break;
    case BLU_P_MAXSEARCH:
        /* the search kernels keep at most MAXCAND candidate columns; a larger value would silently search fewer
         * columns than the reference (markowitz.rs:117-119) */
        if ((int)v > MAXCAND) return BLU_ERROR_INVALID_ARGUMENT;
        p.maxsearch = (int)v; break;
    case BLU_P_PAD: p.pad = (int)v; break;
    case BLU_P_STRETCH: p.stretch = v; break;
    case BLU_P_COMPRESS_THRES: p.compress_thres = v; break;
    case BLU_P_SPARSE_THRES: p.sparse_thres = v; break;
    case BLU_P_SEARCH_ROWS: p.search_rows = (int)v != 0; break;      /* markowitz.rs:125-189 (markowitz_search_rows); the crate's default is 0 (D8) */
    case BLU_P_REALLOC_FACTOR: o->realloc_factor = v; break;
    case BLU_P_NORMS: o->norms = v != 0.0; break;
    case BLU_P_DENSE_K: case BLU_P_DENSE_K_BIG: {
        if (v < 0 || v > BLU_DENSE_K_MAX) return BLU_ERROR_INVALID_ARGUMENT;
        if (cudaSetDevice(o->device) != cudaSuccess) return BLU_ERROR_CUDA;
        cudaStreamSynchronize(o->stream);
        int st = what == BLU_P_DENSE_K ? alloc_dense(o, (int)v, o->want_kbig) : alloc_dense(o, o->d.dense_k, (int)v);
        if (st != BLU_OK) return st;
        if (what == BLU_P_DENSE_K_BIG) o->want_kbig = (int)v;
        break;
    }
    case BLU_P_THREADS_PER_BASIS: case BLU_P_TAIL_THREADS: {
        int t = (int)v;
        if (t != 32 && t != 64 && t != 128 && t != 256 && t != 512 && t != 1024) return BLU_ERROR_INVALID_ARGUMENT;
        if (what == BLU_P_TAIL_THREADS) o->tail_threads = t; else o->nthreads = t;
        break;
    }
    case BLU_P_SPLIT_MIN: o->split_min = (int)v; break;
    case BLU_P_TREE_MIN: o->d.tree_min = (int)v; break;
    case BLU_P_L_MEM: case BLU_P_U_MEM: case BLU_P_W_MEM: {
        int64_t n = (int64_t)v;
        if (n < 1) return BLU_ERROR_INVALID_ARGUMENT;
        if (cudaSetDevice(o->device) != cudaSuccess) return BLU_ERROR_CUDA;
        cudaStreamSynchronize(o->stream);
        int st = swap_stores(o, what == BLU_P_L_MEM ? n : o->d.l_mem, what == BLU_P_U_MEM ? n : o->d.u_mem, what == BLU_P_W_MEM ? n : o->d.w_mem);
        if (st != BLU_OK) return st;      /* the old stores and the factors in them are untouched */
        /* the factors are gone */
        for (auto &I : o->hinfo) I.nupdate = -1;
        if (cudaMemcpy(o->d.info, o->hinfo.data(), o->hinfo.size() * sizeof(BluInfo), cudaMemcpyHostToDevice) != cudaSuccess || cudaStreamSynchronize(0) != cudaSuccess) return BLU_ERROR_CUDA;
        break;
    }
    default: return BLU_ERROR_INVALID_ARGUMENT;
    }
    return BLU_OK;
}
extern "C" double blu_get_param(const blu_t *o, int what) {
    if (!o) return 0.0;
    const BluParams &p = o->d.prm;
    switch (what) {
    case BLU_P_DROPTOL: return p.droptol;
    case BLU_P_ABSTOL: return p.abstol;
    case BLU_P_RELTOL: return p.reltol;
    case BLU_P_NZBIAS: return p.nzbias;
    case BLU_P_MAXSEARCH: return p.maxsearch;
    case BLU_P_PAD: return p.pad;
    case BLU_P_STRETCH: return p.stretch;
    case BLU_P_COMPRESS_THRES: return p.compress_thres;
    case BLU_P_SPARSE_THRES: return p.sparse_thres;
    case BLU_P_SEARCH_ROWS: return p.search_rows;
    case BLU_P_REALLOC_FACTOR: return o->realloc_factor;
    case BLU_P_NORMS: return o->norms;
    case BLU_P_L_MEM: return (double)o->d.l_mem;
    case BLU_P_U_MEM: return (double)o->d.u_mem;
    case BLU_P_W_MEM: return (double)o->d.w_mem;
    case BLU_P_THREADS_PER_BASIS: return o->nthreads;
    case BLU_P_DENSE_K: return o->d.dense_k;
    case BLU_P_DENSE_K_BIG: return o->d.dense_kbig;
    case BLU_P_TAIL_THREADS: return o->tail_threads;
    case BLU_P_SPLIT_MIN: return o->split_min;
    case BLU_P_TREE_MIN: return o->d.tree_min;
    default: return 0.0;
    }
}
extern "C" double blu_get_info(blu_t *o, int what) { return blu_batch_get_info(o, 0, what); }

static int ensure_gf_cap(blu_b200 *o, int64_t n) {
    if (n <= o->gf_cap) return BLU_OK;
    dfree(o, o->gf_i); dfree(o, o->gf_x); o->gf_i = nullptr; o->gf_x = nullptr;
    int st = dalloc(o, &o->gf_i, (size_t)n);
    if (st == BLU_OK) st = dalloc(o, &o->gf_x, (size_t)n);
    if (st == BLU_OK) o->gf_cap = n;
    return st;
}

extern "C" int blu_batch_get_factors(blu_batch_t *o, int64_t k, int64_t *rowperm, int64_t *colperm,
                                     int64_t *l_colptr, int64_t *l_rowidx, double *l_value,
                                     int64_t *u_colptr, int64_t *u_rowidx, double *u_value) {
    if (!o || k < 0 || k >= o->d.nmat) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    { int st0 = ensure_info(o); if (st0 != BLU_OK) return st0; }
    const BluInfo &I = o->hinfo[(size_t)k];
    if (I.nupdate != 0) return BLU_ERROR_INVALID_CALL;   /* get_factors.rs:59-61 (D9: no panic) */
    const int64_t m = o->d.m, lz = m + I.l_nz, uz = m + I.u_nz;
    /* staging layout (i64): rowperm m | colperm m | l_colptr m+1 | l_rowidx lz | u_colptr m+1 | u_rowidx uz ; (f64): l_value lz | u_value uz */
    const int64_t ni = 4 * m + 2 + lz + uz, nx = lz + uz;
    int st = ensure_gf_cap(o, std::max(ni, nx));
    if (st != BLU_OK) return st;
    int64_t *d_rp = o->gf_i, *d_cp = d_rp + m, *d_lp = d_cp + m, *d_li = d_lp + m + 1, *d_up = d_li + lz, *d_ui = d_up + m + 1;
    double *d_lx = o->gf_x, *d_ux = d_lx + lz;
    BLU_LAUNCH(k_get_factors<128>, 1, 128, 0, o->stream, o->d, (int)k, (i64 *)d_rp, (i64 *)d_cp, (i64 *)d_lp, (i64 *)d_li, d_lx,
               (i64 *)d_up, (i64 *)d_ui, d_ux, o->d_status + k);
    o->launches++;
    CK(cudaGetLastError());
#define DL(dst, src, cnt, T) if (dst) CK(cudaMemcpyAsync(dst, src, (size_t)(cnt) * sizeof(T), cudaMemcpyDeviceToHost, o->stream))
    DL(rowperm, d_rp, m, int64_t); DL(colperm, d_cp, m, int64_t);
    if (l_colptr && l_rowidx && l_value) { DL(l_colptr, d_lp, m + 1, int64_t); DL(l_rowidx, d_li, lz, int64_t); DL(l_value, d_lx, lz, double); }
    if (u_colptr && u_rowidx && u_value) { DL(u_colptr, d_up, m + 1, int64_t); DL(u_rowidx, d_ui, uz, int64_t); DL(u_value, d_ux, uz, double); }
#undef DL
    CK(cudaStreamSynchronize(o->stream));
    return BLU_OK;
}

/* ------------------------------------------------------------------ */
/* object API                                                          */
/* ------------------------------------------------------------------ */
extern "C" int blu_create(blu_t **out, int64_t m, int64_t b_nz, int device) { return create_common(out, 1, m, b_nz, device, 1); }
extern "C" void blu_destroy(blu_t *o) { destroy_common(o); }

extern "C" int blu_factorize(blu_t *o, const int64_t *b_begin, const int64_t *b_end, const int64_t *b_i, const double *b_x) {
    if (!o || !b_begin || !b_end) return BLU_ERROR_INVALID_ARGUMENT;   /* b_i / b_x may be null when B has no entries */
    if (o->d.nmat != 1) return BLU_ERROR_INVALID_CALL;
    const int64_t m = o->d.m;
    /* gather the referenced columns into a compact staging copy (B may live inside a
     * much larger array, as in maxvolume.rs:180-224) */
    o->hb_begin.resize((size_t)m); o->hb_end.resize((size_t)m);
    int64_t nnz = 0;
    for (int64_t j = 0; j < m; j++) {
        if (b_end[j] < b_begin[j]) return BLU_ERROR_INVALID_ARGUMENT;   /* singletons.rs:122-131 */
        o->hb_begin[(size_t)j] = nnz; nnz += b_end[j] - b_begin[j]; o->hb_end[(size_t)j] = nnz;
    }
    if (nnz > 0 && (!b_i || !b_x)) return BLU_ERROR_INVALID_ARGUMENT;
    o->hb_i.resize((size_t)nnz); o->hb_x.resize((size_t)nnz);
    for (int64_t j = 0; j < m; j++) {
        const int64_t n = b_end[j] - b_begin[j];
        if (n) {
            memcpy(&o->hb_i[(size_t)o->hb_begin[(size_t)j]], b_i + b_begin[j], (size_t)n * sizeof(int64_t));
            memcpy(&o->hb_x[(size_t)o->hb_begin[(size_t)j]], b_x + b_begin[j], (size_t)n * sizeof(double));
        }
    }
    if (nnz > o->d.bnz_cap) {
        /* the object was created for fewer nonzeros: grow the row-copy store */
        CK(cudaSetDevice(o->device));
        dfree(o, o->d.bt_idx); dfree(o, o->d.bt_val);
        o->d.bnz_cap = nnz;
        int st = dalloc(o, &o->d.bt_idx, (size_t)nnz);
        if (st == BLU_OK) st = dalloc(o, &o->d.bt_val, (size_t)nnz);
        if (st != BLU_OK) return st;
    }
    int st = blu_batch_upload(o, o->hb_begin.data(), o->hb_end.data(), o->hb_i.data(), o->hb_x.data(), nnz, nullptr);
    if (st != BLU_OK) return st;
    st = factorize_resident(o, 0, o->escape_realloc);
    o->time_factorize += 1e-3 * o->last_ms[0];
    if (st != BLU_OK) return st;
    return o->hinfo[0].status;
}

/* factorize() of the crate's free-function surface (lib.rs:11-19 -> factorize.rs:34-119): Reallocate ESCAPES.
 * The caller reads BLU_I_ADDMEM_L/U/W, grows the stores (blu_set_param BLU_P_L_MEM / U_MEM / W_MEM, the role of
 * lu_realloc_obj) and calls again with c0ntinue != 0.  c0ntinue without a pending Reallocate is
 * ErrorInvalidCall (factorize.rs:102-105).  The reference resumes at the phase that ran out of memory; the device
 * starts the factorization over with the larger stores -- same factors, same return codes. */
extern "C" int blu_factorize_c0ntinue(blu_t *o, const int64_t *b_begin, const int64_t *b_end, const int64_t *b_i, const double *b_x, int c0ntinue) {
    if (!o || !b_begin || !b_end) return BLU_ERROR_INVALID_ARGUMENT;
    if (o->d.nmat != 1) return BLU_ERROR_INVALID_CALL;
    if (c0ntinue && !o->task_pending) return BLU_ERROR_INVALID_CALL;
    o->escape_realloc = 1;
    int st = blu_factorize(o, b_begin, b_end, b_i, b_x);
    o->escape_realloc = 0;
    o->task_pending = st == BLU_REALLOCATE;
    return st;
}

extern "C" int blu_get_factors(blu_t *o, int64_t *rowperm, int64_t *colperm,
                               int64_t *l_colptr, int64_t *l_rowidx, double *l_value,
                               int64_t *u_colptr, int64_t *u_rowidx, double *u_value) {
    return blu_batch_get_factors(o, 0, rowperm, colperm, l_colptr, l_rowidx, l_value, u_colptr, u_rowidx, u_value);
}

extern "C" int blu_solve_dense(blu_t *o, const double *rhs, double *lhs, char trans) {
    if (!o || !rhs || !lhs) return BLU_ERROR_INVALID_ARGUMENT;
    { int st0 = ensure_info(o); if (st0 != BLU_OK) return st0; }
    if (o->hinfo[0].nupdate < 0) return BLU_ERROR_INVALID_CALL;   /* solve_dense.rs:25 */
    int status = BLU_OK;
    int st = blu_batch_solve_dense(o, rhs, lhs, trans, &status);
    o->info_dirty = 1;      /* the solve compacts the pivot sequence (pivotlen), as blu_solve_dense_multi's does */
    o->time_solve += 1e-3 * o->last_ms[1];
    return st != BLU_OK ? st : status;
}

extern "C" const char *blu_version(void) {
#ifdef BLU_EMU
    return "blu_b200 0.1 (SIMT emulation build: tests only)";
#else
    return "blu_b200 0.1 (sm_100a)";
#endif
}

/* ------------------------------------------------------------------ */
/* sparse solves and the update (object API only)                      */
/* ------------------------------------------------------------------ */

/* lu_realloc_obj, blu.rs:345-377, for a store whose content must survive (an eta or a
 * spike was appended since the factorization).  which: 0 = L, 1 = U, 2 = W. */
static int grow_store_keep(blu_b200 *o, int which, int64_t addmem) {
    BluDev &d = o->d;
    const double f = o->realloc_factor < 1.0 ? 1.0 : o->realloc_factor;
    CK(cudaStreamSynchronize(o->stream));
    blu_i64 &mem = which == 0 ? d.l_mem : which == 1 ? d.u_mem : d.w_mem;
    const int64_t newmem = (int64_t)(f * (double)(mem + addmem)) + 1;
    if (newmem > (which == 2 ? 0x1fffffff : 0x3fffffff)) return BLU_ERROR_OUT_OF_MEMORY;
    int *ni = nullptr; double *nv = nullptr;
    const size_t mult = which == 2 ? 2 : 1;
    int st = dalloc(o, &ni, mult * (size_t)newmem + PADDING);
    if (st == BLU_OK) st = dalloc(o, &nv, mult * (size_t)newmem + PADDING);
    if (st != BLU_OK) return st;
    int *&oi = which == 0 ? d.l_idx : which == 1 ? d.u_idx : d.w_idx;
    double *&ov = which == 0 ? d.l_val : which == 1 ? d.u_val : d.w_val;
    size_t from = 0;
    if (which == 2) {
        /* only the live half moves; it becomes half 0 of the new store */
        int st2 = fetch_info(o);
        if (st2 != BLU_OK) return st2;
        from = (size_t)o->hinfo[0].w_half * (size_t)mem;
    }
    CK(cudaMemcpyAsync(ni, oi + from, (size_t)mem * sizeof(int), cudaMemcpyDeviceToDevice, o->stream));
    CK(cudaMemcpyAsync(nv, ov + from, (size_t)mem * sizeof(double), cudaMemcpyDeviceToDevice, o->stream));
    CK(cudaStreamSynchronize(o->stream));
    dfree(o, oi); dfree(o, ov);
    oi = ni; ov = nv;
    if (which == 1 && o->single && d.ur_idx) {
        /* the sorted row-wise copy of U is sized like the U store: grow it too, content kept */
        int *ri = nullptr; double *rv = nullptr;
        st = dalloc(o, &ri, (size_t)newmem + PADDING);
        if (st == BLU_OK) st = dalloc(o, &rv, (size_t)newmem + PADDING);
        if (st != BLU_OK) return st;
        CK(cudaMemcpyAsync(ri, d.ur_idx, (size_t)mem * sizeof(int), cudaMemcpyDeviceToDevice, o->stream));
        CK(cudaMemcpyAsync(rv, d.ur_val, (size_t)mem * sizeof(double), cudaMemcpyDeviceToDevice, o->stream));
        CK(cudaStreamSynchronize(o->stream));
        dfree(o, d.ur_idx); dfree(o, d.ur_val);
        d.ur_idx = ri; d.ur_val = rv;
    }
    if (which == 2) {
        BLU_LAUNCH(k_w_rebase, 1, 128, 0, o->stream, d, (int)from);
        o->launches++;
        CK(cudaGetLastError());
    }
    mem = newmem;
    o->nrealloc++;
    o->info_dirty = 1;
    return BLU_OK;
}

/* the single object's answer to Reallocate: every store the last run asked more room for grows, content kept */
static int grow_object_stores(blu_b200 *o) {
    int st = fetch_info(o);
    if (st != BLU_OK) return st;
    const BluInfo &I = o->hinfo[0];
    if (I.addmem_l > 0) st = grow_store_keep(o, 0, I.addmem_l);
    if (st == BLU_OK && I.addmem_u > 0) st = grow_store_keep(o, 1, I.addmem_u);
    if (st == BLU_OK && I.addmem_w > 0) st = grow_store_keep(o, 2, I.addmem_w);
    return st;
}

/* The Reallocate loop of the basis-change calls (BLU::solve_for_update / update, blu.rs:268-291, 319-334):
 * run(rerun, &asks) queues one run's launches (rerun: not the first run), reads back what the call reads and sets asks
 * when a running basis still says Reallocate; grow(o) makes room before the next run.  At most 40 runs.  Returns run's
 * error as it is, BLU_OK once no basis asks, and otherwise BLU_REALLOCATE with *grown (when given) the status of the
 * last grow, BLU_OK when the 40th run still asks.  What a basis still asking means is the caller's policy. */
template <typename Run> static int rerun_on_realloc(blu_b200 *o, int (*grow)(blu_b200 *), Run run, int *grown = nullptr) {
    int gst = BLU_OK;
    for (int attempt = 0; attempt < 40 && gst == BLU_OK; attempt++) {
        bool asks = false;
        const int st = run(attempt > 0, &asks);
        if (st != BLU_OK) return st;
        if (!asks) return BLU_OK;
        if (attempt < 39) gst = grow(o);
    }
    if (grown) *grown = gst;
    return BLU_REALLOCATE;
}

static double wall_now() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

/* common body of blu_solve_sparse and blu_solve_for_update */
static int sparse_call(blu_b200 *o, int64_t nzrhs, const int64_t *irhs, const double *xrhs,
                       int64_t *nzlhs, int64_t *ilhs, double *lhs, char trans, int for_update) {
    if (!o || !o->single) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const double tic = wall_now();
    const int64_t m = o->d.m;
    const bool tr = trans == 't' || trans == 'T';
    const int want = nzlhs && ilhs && lhs;
    if (!for_update && !want) return BLU_ERROR_INVALID_ARGUMENT;
    const int64_t nup = (for_update && tr) ? 1 : nzrhs;
    const int64_t ncopy = (nup < 0 || nup > m) ? 0 : nup;
    if (ncopy > 0 && !irhs) return BLU_ERROR_INVALID_ARGUMENT;
    if (!for_update && ncopy > 0 && !xrhs) return BLU_ERROR_ARGUMENT_MISSING;   /* the reference's xrhs is a slice, never absent (solve_sparse.rs:35) */
    if (ncopy > 0) {
        CK(cudaMemcpyAsync(o->d_irhs, irhs, (size_t)ncopy * sizeof(int64_t), cudaMemcpyHostToDevice, o->stream));
        if (xrhs && !(for_update && tr)) CK(cudaMemcpyAsync(o->d_xrhs, xrhs, (size_t)ncopy * sizeof(double), cudaMemcpyHostToDevice, o->stream));
    }
    const int nrhs = (nzrhs < 0 || nzrhs > m) ? -1 : (int)nzrhs;
    const double *dx = (xrhs && !(for_update && tr)) ? o->d_xrhs : nullptr;
    int status = BLU_OK, nz = 0, grown;
    const int rs = rerun_on_realloc(o, grow_object_stores, [&](bool, bool *asks) -> int {
        BLU_LAUNCH(k_solve_sparse, 1, 32, 0, o->stream, o->d, nrhs, (const i64 *)o->d_irhs, dx, trans, for_update, want,
                   o->d_scal, (i64 *)o->d_ilhs, o->d_xout, SpMulti{});
        o->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(o->h_scal, o->d_scal, 2 * sizeof(int), cudaMemcpyDeviceToHost, o->stream));
        CK(cudaStreamSynchronize(o->stream));
        status = o->h_scal[0]; nz = o->h_scal[1];
        o->info_dirty = 1;
        *asks = status == BLU_REALLOCATE;
        return BLU_OK;
    }, &grown);
    /* a store that cannot grow: its error; still Reallocate after 40 runs: an internal error */
    if (rs == BLU_REALLOCATE && grown != BLU_OK) return grown;
    if (rs == BLU_REALLOCATE) status = BLU_ERROR_INTERNAL;
    else if (rs != BLU_OK) return rs;
    if (status == BLU_OK && want) {
        if (nz > 0) {
            CK(cudaMemcpyAsync(o->h_ilhs, o->d_ilhs, (size_t)nz * sizeof(int64_t), cudaMemcpyDeviceToHost, o->stream));
            CK(cudaMemcpyAsync(o->h_xout, o->d_xout, (size_t)nz * sizeof(double), cudaMemcpyDeviceToHost, o->stream));
            CK(cudaStreamSynchronize(o->stream));
            for (int n = 0; n < nz; n++) { ilhs[n] = o->h_ilhs[n]; lhs[o->h_ilhs[n]] = o->h_xout[n]; }
        }
        *nzlhs = nz;
    }
    o->time_solve += wall_now() - tic;
    return status;
}

extern "C" int blu_solve_sparse(blu_t *o, int64_t nzrhs, const int64_t *irhs, const double *xrhs,
                                int64_t *nzlhs, int64_t *ilhs, double *lhs, char trans) {
    return sparse_call(o, nzrhs, irhs, xrhs, nzlhs, ilhs, lhs, trans, 0);
}

extern "C" int blu_solve_for_update(blu_t *o, int64_t nzrhs, const int64_t *irhs, const double *xrhs,
                                    int64_t *nzlhs, int64_t *ilhs, double *lhs, char trans) {
    return sparse_call(o, nzrhs, irhs, xrhs, nzlhs, ilhs, lhs, trans, 1);
}

extern "C" int blu_update(blu_t *o, double xtbl) {
    if (!o || !o->single) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const double tic = wall_now();
    int status = BLU_OK, grown;
    const int rs = rerun_on_realloc(o, grow_object_stores, [&](bool, bool *asks) -> int {
        BLU_LAUNCH(k_update, 1, 32, 0, o->stream, o->d, xtbl, o->d_scal, (const double *)nullptr, 0);
        o->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(o->h_scal, o->d_scal, sizeof(int), cudaMemcpyDeviceToHost, o->stream));
        CK(cudaStreamSynchronize(o->stream));
        status = o->h_scal[0];
        o->info_dirty = 1;
        *asks = status == BLU_REALLOCATE;
        return BLU_OK;
    }, &grown);
    if (rs == BLU_REALLOCATE && grown != BLU_OK) return grown;      /* as in sparse_call */
    if (rs == BLU_REALLOCATE) status = BLU_ERROR_INTERNAL;
    else if (rs != BLU_OK) return rs;
    o->time_update += wall_now() - tic;
    return status;
}

/* SURVEY.md 8(f) N4: many right-hand sides against one factorization -- the batch call on the object's one basis
 * (its chunks of units go through the unit pool).  Bit-identical to nrhs separate blu_solve_dense calls. */
extern "C" int blu_solve_dense_multi(blu_t *o, int64_t nrhs, const double *rhs, double *lhs, char trans) {
    if (!o || !o->single || nrhs < 0 || (nrhs > 0 && (!rhs || !lhs))) return BLU_ERROR_INVALID_ARGUMENT;
    { int st0 = ensure_info(o); if (st0 != BLU_OK) return st0; }
    if (o->hinfo[0].nupdate < 0) return BLU_ERROR_INVALID_CALL;   /* solve_dense.rs:25 */
    if (nrhs == 0) return BLU_OK;
    return blu_batch_solve_dense_multi(o, nrhs, rhs, lhs, trans, nullptr);
}

/* Many sparse right-hand sides against one factorization: blu_batch_solve_sparse with every unit on the object's one
 * basis, the solutions copied out in full rows.  Bit-identical to nrhs separate blu_solve_sparse calls. */
static int solve_sparse_units(blu_b200 *o, const int64_t *unit_begin, const int64_t *rhs_begin, const int64_t *irhs, const double *xrhs,
                              int64_t *nzlhs, int64_t *ilhs, double *xlhs, int *status, char trans, bool rows);
extern "C" int blu_solve_sparse_multi(blu_t *o, int64_t nrhs, const int64_t *rhs_begin, const int64_t *irhs, const double *xrhs,
                                      int64_t *nzlhs, int64_t *ilhs, double *xlhs, int *status, char trans) {
    if (!o || !o->single || nrhs < 0 || (nrhs > 0 && (!rhs_begin || !nzlhs || !ilhs || !xlhs))) return BLU_ERROR_INVALID_ARGUMENT;
    { int st0 = ensure_info(o); if (st0 != BLU_OK) return st0; }
    if (o->hinfo[0].nupdate < 0) return BLU_ERROR_INVALID_CALL;   /* solve_sparse.rs:42 */
    if (nrhs == 0) return BLU_OK;
    const int64_t unit_begin[2] = {0, nrhs};
    return solve_sparse_units(o, unit_begin, rhs_begin, irhs, xrhs, nzlhs, ilhs, xlhs, status, trans, true);
}

/* ------------------------------------------------------------------ */
/* batch: one basis change on every basis at once (multi-LP sweeps)    */
/* ------------------------------------------------------------------ */

/* lu_realloc_obj (blu.rs:345-377) for a batch: every basis gets the larger store, content kept */
static int grow_batch_stores(blu_b200 *o) {
    BluDev &d = o->d;
    int st = fetch_info(o);
    if (st != BLU_OK) return st;
    int64_t al = 0, au = 0, aw = 0;
    /* the kernels zero addmem_* on entry: only the bases that returned Reallocate carry a request */
    for (auto &I : o->hinfo) { al = std::max<int64_t>(al, I.addmem_l); au = std::max<int64_t>(au, I.addmem_u); aw = std::max<int64_t>(aw, I.addmem_w); }
    if (al <= 0 && au <= 0 && aw <= 0) return BLU_ERROR_INTERNAL;
    const double f = o->realloc_factor < 1.0 ? 1.0 : o->realloc_factor;
    const size_t n = (size_t)d.nmat;
    CK(cudaStreamSynchronize(o->stream));
    /* the new uniform sizes cover the largest private store too, so that every override can be folded back */
    int64_t cl = d.l_mem, cu = d.u_mem, cw = d.w_mem;
    for (auto &e : o->hslot) { if (e.l_idx) cl = std::max<int64_t>(cl, e.l_mem); if (e.u_idx) cu = std::max<int64_t>(cu, e.u_mem); if (e.w_idx) cw = std::max<int64_t>(cw, e.w_mem); }
    const bool fold = o->have_overrides != 0;
    const int64_t nl = al > 0 ? (int64_t)(f * (double)(cl + al)) + 1 : cl;
    const int64_t nu = au > 0 ? (int64_t)(f * (double)(cu + au)) + 1 : cu;
    const int64_t nw = aw > 0 ? (int64_t)(f * (double)(cw + aw)) + 1 : cw;
    if (nl > 0x3fffffff || nu > 0x3fffffff || nw > 0x1fffffff) return BLU_ERROR_OUT_OF_MEMORY;
    const bool gl = al > 0 || fold, gu = au > 0 || fold, gw = aw > 0 || fold;
    int *li = nullptr, *ui = nullptr, *wi = nullptr; double *lv = nullptr, *uv = nullptr, *wv = nullptr;
    if (gl) { st = dalloc(o, &li, n * (size_t)nl + PADDING); if (st == BLU_OK) st = dalloc(o, &lv, n * (size_t)nl + PADDING); if (st != BLU_OK) return st; }
    if (gu) { st = dalloc(o, &ui, n * (size_t)nu + PADDING); if (st == BLU_OK) st = dalloc(o, &uv, n * (size_t)nu + PADDING); if (st != BLU_OK) return st; }
    if (gw) { st = dalloc(o, &wi, n * 2 * (size_t)nw + PADDING); if (st == BLU_OK) st = dalloc(o, &wv, n * 2 * (size_t)nw + PADDING); if (st != BLU_OK) return st; }
    /* every basis copies its own content (read through its view, private or uniform) into the new stores */
    BLU_LAUNCH(k_store_regrow, d.nmat, 256, 0, o->stream, d, li, lv, (blu_i64)nl, ui, uv, (blu_i64)nu, wi, wv, (blu_i64)nw);
    o->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(o->stream));
    if (gl) { dfree(o, d.l_idx); dfree(o, d.l_val); d.l_idx = li; d.l_val = lv; d.l_mem = nl; }
    if (gu) { dfree(o, d.u_idx); dfree(o, d.u_val); d.u_idx = ui; d.u_val = uv; d.u_mem = nu; }
    if (gw) { dfree(o, d.w_idx); dfree(o, d.w_val); d.w_idx = wi; d.w_val = wv; d.w_mem = nw; }
    if (fold && (st = clear_overrides(o)) != BLU_OK) return st;
    o->nrealloc++;
    o->info_dirty = 1;
    return BLU_OK;
}

static int ensure_batch_sparse(blu_b200 *o, int64_t tot) {
    const size_t n = (size_t)o->d.nmat, m = (size_t)o->d.m;
    int st = BLU_OK;
    if (!o->sm_scal) {
        st = dalloc(o, &o->sm_scal, 2 * n);
        if (st == BLU_OK) st = dalloc(o, &o->sm_xout, n * m);
        if (st == BLU_OK) st = dalloc(o, &o->sm_ilhs, n * m);
        if (st == BLU_OK) st = dalloc(o, &o->sm_begin, n + 1);
        if (st == BLU_OK) st = dalloc(o, &o->sm_dbls, n);          /* xtbl per basis */
        if (st != BLU_OK) return st;
    }
    if (tot > o->smulti_rhs_cap) {
        dfree(o, o->sm_irhs); dfree(o, o->sm_xrhs); o->sm_irhs = nullptr; o->sm_xrhs = nullptr; o->smulti_rhs_cap = 0;
        st = dalloc(o, &o->sm_irhs, (size_t)tot);
        if (st == BLU_OK) st = dalloc(o, &o->sm_xrhs, (size_t)tot);
        if (st != BLU_OK) return st;
        o->smulti_rhs_cap = tot;
    }
    return BLU_OK;
}

/* The caller's statuses of a host batch call, in result order: result r is the status word words[stride * k] of slot
 * k = sel[r] (k = r without sel) and, with nzlhs, its nonzero count next to it (nzlhs[r] = -1 unless OK).  A Reallocate
 * left over means a store could not grow.  Returns the first non-OK status. */
static int tally_statuses(const int *words, int stride, int64_t nres, const int64_t *sel, int *status, int64_t *nzlhs) {
    int worst = BLU_OK;
    for (int64_t r = 0; r < nres; r++) {
        const size_t w = (size_t)stride * (size_t)(sel ? sel[r] : r);
        const int s = words[w] == BLU_REALLOCATE ? BLU_ERROR_OUT_OF_MEMORY : words[w];
        if (status) status[r] = s;
        if (nzlhs) nzlhs[r] = s == BLU_OK ? words[w + 1] : -1;
        if (s != BLU_OK && worst == BLU_OK) worst = s;
    }
    return worst;
}

/* solve_for_update (blu.rs:257) on every basis of the batch, basis k with its own right-hand side
 * irhs/xrhs[rhs_begin[k] .. rhs_begin[k+1]) (for trans 't'/'T': one index, the column to leave; xrhs may be
 * NULL).  want_solution != 0: nzlhs[k], ilhs[k*m ..] and the values xlhs[k*m + n] as in
 * blu_solve_sparse_multi.  Reallocate is handled as in blu.rs:268-291: the stores of the whole batch are
 * grown (content kept) and the bases that asked run again; BLU_ERROR_OUT_OF_MEMORY only if that fails. */
extern "C" int blu_batch_solve_for_update(blu_batch_t *o, const int64_t *rhs_begin, const int64_t *irhs, const double *xrhs,
                                          int want_solution, int64_t *nzlhs, int64_t *ilhs, double *xlhs, int *status, char trans) {
    if (!o || !rhs_begin || !irhs) return BLU_ERROR_INVALID_ARGUMENT;
    if (want_solution && (!nzlhs || !ilhs || !xlhs)) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const size_t n = (size_t)o->d.nmat, m = (size_t)o->d.m;
    const int64_t tot = rhs_begin[n];
    if (tot < 0) return BLU_ERROR_INVALID_ARGUMENT;
    int st = ensure_batch_sparse(o, tot);
    if (st != BLU_OK) return st;
    CK(cudaMemcpyAsync(o->sm_begin, rhs_begin, (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, o->stream));
    CK(cudaMemcpyAsync(o->sm_irhs, irhs, (size_t)tot * sizeof(int64_t), cudaMemcpyHostToDevice, o->stream));
    if (xrhs) CK(cudaMemcpyAsync(o->sm_xrhs, xrhs, (size_t)tot * sizeof(double), cudaMemcpyHostToDevice, o->stream));
    std::vector<int> hs(2 * n);
    st = rerun_on_realloc(o, grow_batch_stores, [&](bool rerun, bool *asks) -> int {
        SpMulti W{(int)n, rerun, (const i64 *)o->sm_begin};
        BLU_LAUNCH(k_solve_sparse, (int)n, 32, 0, o->stream, o->d, 0, (const i64 *)o->sm_irhs, xrhs ? (const double *)o->sm_xrhs : (const double *)nullptr,
                   trans, 1, want_solution ? 1 : 0, o->sm_scal, (i64 *)o->sm_ilhs, o->sm_xout, W);
        o->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(hs.data(), o->sm_scal, 2 * n * sizeof(int), cudaMemcpyDeviceToHost, o->stream));
        CK(cudaStreamSynchronize(o->stream));
        for (size_t k = 0; k < n; k++) *asks = *asks || hs[2 * k] == BLU_REALLOCATE;
        return BLU_OK;
    });
    if (st != BLU_OK && st != BLU_REALLOCATE) return st;      /* Reallocate left over: a store could not grow */
    if (want_solution) {
        CK(cudaMemcpyAsync(ilhs, o->sm_ilhs, n * m * sizeof(int64_t), cudaMemcpyDeviceToHost, o->stream));
        CK(cudaMemcpyAsync(xlhs, o->sm_xout, n * m * sizeof(double), cudaMemcpyDeviceToHost, o->stream));
    }
    CK(cudaStreamSynchronize(o->stream));
    o->info_dirty = 1;
    return tally_statuses(hs.data(), 2, (int64_t)n, nullptr, status, want_solution ? nzlhs : nullptr);
}

/* update (blu.rs:319) on every basis of the batch, basis k with xtbl[k] */
extern "C" int blu_batch_update(blu_batch_t *o, const double *xtbl, int *status) {
    if (!o || !xtbl) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const size_t n = (size_t)o->d.nmat;
    int st = ensure_batch_sparse(o, 0);
    if (st != BLU_OK) return st;
    CK(cudaMemcpyAsync(o->sm_dbls, xtbl, n * sizeof(double), cudaMemcpyHostToDevice, o->stream));
    std::vector<int> hs(n);
    st = rerun_on_realloc(o, grow_batch_stores, [&](bool rerun, bool *asks) -> int {
        BLU_LAUNCH(k_update, (int)n, 32, 0, o->stream, o->d, 0.0, o->sm_scal, (const double *)o->sm_dbls, rerun ? 1 : 0);
        o->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(hs.data(), o->sm_scal, n * sizeof(int), cudaMemcpyDeviceToHost, o->stream));
        CK(cudaStreamSynchronize(o->stream));
        for (size_t k = 0; k < n; k++) *asks = *asks || hs[k] == BLU_REALLOCATE;
        return BLU_OK;
    });
    if (st != BLU_OK && st != BLU_REALLOCATE) return st;      /* Reallocate left over: a store could not grow */
    o->info_dirty = 1;
    return tally_statuses(hs.data(), 1, (int64_t)n, nullptr, status, nullptr);
}

/* ------------------------------------------------------------------ */
/* batch: many right-hand sides on every basis (one warp per unit)     */
/* ------------------------------------------------------------------ */

/* the per-unit tables of a call (basis of each unit, offsets of its right-hand side) */
static int up_ensure_units(blu_b200 *o, int64_t nunits) {
    UnitPool &U = o->up;
    if (nunits <= U.ucap) return BLU_OK;
    dfree(o, U.slot); dfree(o, U.begin); U.slot = nullptr; U.begin = nullptr; U.ucap = 0;
    int st = dalloc(o, &U.slot, (size_t)nunits);
    if (st == BLU_OK) st = dalloc(o, &U.begin, (size_t)nunits + 1);
    if (st == BLU_OK) U.ucap = nunits;
    return st;
}
/* SpMulti scratch for P units (dbls starts all-zero and k_solve_sparse leaves it so) and tot right-hand side entries */
static int up_ensure_sparse(blu_b200 *o, int64_t P, int64_t tot) {
    UnitPool &U = o->up;
    const size_t m = (size_t)o->d.m, n = (size_t)P;
    int st = BLU_OK;
    if (P > U.cap) {
        dfree(o, U.ints); dfree(o, U.dbls); dfree(o, U.markers); dfree(o, U.scal); dfree(o, U.ilhs); dfree(o, U.xout); dfree(o, U.off); dfree(o, U.fill);
        U.ints = U.markers = U.scal = nullptr; U.dbls = U.xout = nullptr; U.ilhs = U.off = nullptr; U.fill = nullptr; U.cap = 0;
        st = dalloc(o, &U.ints, n * 7 * m);
        if (st == BLU_OK) st = dalloc(o, &U.dbls, n * 2 * m);
        if (st == BLU_OK) st = dalloc(o, &U.markers, n);
        if (st == BLU_OK) st = dalloc(o, &U.scal, 2 * n);
        if (st == BLU_OK) st = dalloc(o, &U.ilhs, n * m);
        if (st == BLU_OK) st = dalloc(o, &U.xout, n * m);
        if (st == BLU_OK) st = dalloc(o, &U.off, n);
        if (st == BLU_OK) st = dalloc(o, &U.fill, 1);
        if (st != BLU_OK) return st;
        U.cap = P;
    }
    if (tot > U.rcap) {
        dfree(o, U.irhs); dfree(o, U.xrhs); U.irhs = nullptr; U.xrhs = nullptr; U.rcap = 0;
        st = dalloc(o, &U.irhs, (size_t)tot);
        if (st == BLU_OK) st = dalloc(o, &U.xrhs, (size_t)tot);
        if (st != BLU_OK) return st;
        U.rcap = tot;
    }
    return BLU_OK;
}
static int up_ensure_dense(blu_b200 *o, int64_t P) {
    UnitPool &U = o->up;
    if (P <= U.dcap) return BLU_OK;
    const size_t m = (size_t)o->d.m, n = (size_t)P;
    dfree(o, U.rhs); dfree(o, U.lhs); dfree(o, U.work); dfree(o, U.dstatus);
    U.rhs = U.lhs = U.work = nullptr; U.dstatus = nullptr; U.dcap = 0;
    int st = dalloc(o, &U.rhs, n * m);
    if (st == BLU_OK) st = dalloc(o, &U.lhs, n * m);
    if (st == BLU_OK) st = dalloc(o, &U.work, n * m);
    if (st == BLU_OK) st = dalloc(o, &U.dstatus, n);
    if (st == BLU_OK) U.dcap = P;
    return st;
}
static int up_ensure_host(blu_b200 *o, int64_t n) {
    UnitPool &U = o->up;
    if (n <= U.hcap) return BLU_OK;
    const int64_t want = std::max<int64_t>(n, 2 * U.hcap);
    if (U.h_ilhs) cudaFreeHost(U.h_ilhs);
    if (U.h_xout) cudaFreeHost(U.h_xout);
    U.h_ilhs = nullptr; U.h_xout = nullptr; U.hcap = 0;
    if (cudaMallocHost((void **)&U.h_ilhs, (size_t)want * sizeof(int64_t)) != cudaSuccess ||
        cudaMallocHost((void **)&U.h_xout, (size_t)want * sizeof(double)) != cudaSuccess) { cudaGetLastError(); return BLU_ERROR_OUT_OF_MEMORY; }
    U.hcap = want;
    return BLU_OK;
}

/* garbage_perm on every basis, so that the units of a basis can read its pivot sequence side by side */
static int up_compact_all(blu_b200 *o, double *kms) {
    timer_start(o);
    BLU_LAUNCH(k_garbage_perm, o->d.nmat, 32, 0, o->stream, o->d);
    o->launches++;
    CK(cudaGetLastError());
    timer_stop(o, 1);
    *kms += o->last_ms[1];
    return BLU_OK;
}

/* solve_sparse (solve_sparse.rs:35-73) for the units of every basis, one warp per unit.  Unit u reads the
 * factors of its basis and nothing else of its state; marks, stacks and vectors come from the unit pool, and
 * the flop counters of the basis are added to atomically.  Without rows, each chunk's solutions are packed on the
 * device (only the nz entries of each unit cross the bus) and land in the caller's arrays at the unit's own offset.
 * With rows, every unit writes its row of m and the chunk's rows go to the caller's arrays in one copy: the object's
 * blu_solve_sparse_multi, whose solutions can be dense (configs[3]: 80 % of m), where that is the faster copy. */
static int solve_sparse_units(blu_b200 *o, const int64_t *unit_begin, const int64_t *rhs_begin, const int64_t *irhs, const double *xrhs,
                              int64_t *nzlhs, int64_t *ilhs, double *xlhs, int *status, char trans, bool rows) {
    if (!o || !unit_begin || unit_begin[0] != 0) return BLU_ERROR_INVALID_ARGUMENT;
    const int64_t nmat = o->d.nmat;
    const size_t m = (size_t)o->d.m;
    for (int64_t k = 0; k < nmat; k++) if (unit_begin[k + 1] < unit_begin[k]) return BLU_ERROR_INVALID_ARGUMENT;
    const int64_t nunits = unit_begin[nmat];
    if (nunits == 0) return BLU_OK;
    if (!rhs_begin || !nzlhs || !ilhs || !xlhs) return BLU_ERROR_INVALID_ARGUMENT;
    const int64_t tot = rhs_begin[nunits];
    if (tot < 0) return BLU_ERROR_INVALID_ARGUMENT;
    for (int64_t u = 0; u < nunits; u++) if (rhs_begin[u] < 0 || rhs_begin[u] > tot) return BLU_ERROR_INVALID_ARGUMENT;
    if (tot > 0 && (!irhs || !xrhs)) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const double tic = wall_now();
    const int64_t P = std::min<int64_t>(nunits, o->solve_units);
    int st = up_ensure_units(o, nunits);
    if (st == BLU_OK) st = up_ensure_sparse(o, P, tot);
    if (st != BLU_OK) return st;
    UnitPool &U = o->up;
    std::vector<int> hslot((size_t)nunits);
    for (int64_t k = 0; k < nmat; k++) for (int64_t u = unit_begin[k]; u < unit_begin[k + 1]; u++) hslot[(size_t)u] = (int)k;
    CK(cudaMemcpyAsync(U.slot, hslot.data(), (size_t)nunits * sizeof(int), cudaMemcpyHostToDevice, o->stream));
    CK(cudaMemcpyAsync(U.begin, rhs_begin, ((size_t)nunits + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, o->stream));
    if (tot > 0) {
        CK(cudaMemcpyAsync(U.irhs, irhs, (size_t)tot * sizeof(int64_t), cudaMemcpyHostToDevice, o->stream));
        CK(cudaMemcpyAsync(U.xrhs, xrhs, (size_t)tot * sizeof(double), cudaMemcpyHostToDevice, o->stream));
    }
    double kms = 0.0;
    if ((st = up_compact_all(o, &kms)) != BLU_OK) return st;
    std::vector<int> hs(2 * (size_t)P);
    std::vector<int64_t> hoff((size_t)P);
    int worst = BLU_OK;
    for (int64_t c0 = 0; c0 < nunits; c0 += P) {
        const int cnt = (int)std::min<int64_t>(P, nunits - c0);
        CK(cudaMemsetAsync(U.fill, 0, sizeof(blu_u64), o->stream));
        SpMulti W{cnt, 0, (const i64 *)U.begin + c0, nullptr, U.ints, U.dbls, U.markers, U.slot + c0, U.fill, (i64 *)U.off, rows ? (int)m : 0};
        timer_start(o);
        BLU_LAUNCH(k_solve_sparse<true>, cnt, 32, 0, o->stream, o->d, 0, (const i64 *)U.irhs, (const double *)U.xrhs, trans, 0, 1,
                   U.scal, (i64 *)U.ilhs, U.xout, W);
        o->launches++;
        CK(cudaGetLastError());
        timer_stop(o, 1);
        kms += o->last_ms[1];
        blu_u64 fill = 0;
        CK(cudaMemcpyAsync(hs.data(), U.scal, 2 * (size_t)cnt * sizeof(int), cudaMemcpyDeviceToHost, o->stream));
        if (rows) {
            CK(cudaMemcpyAsync(ilhs + (size_t)c0 * m, U.ilhs, (size_t)cnt * m * sizeof(int64_t), cudaMemcpyDeviceToHost, o->stream));
            CK(cudaMemcpyAsync(xlhs + (size_t)c0 * m, U.xout, (size_t)cnt * m * sizeof(double), cudaMemcpyDeviceToHost, o->stream));
        } else {
            CK(cudaMemcpyAsync(hoff.data(), U.off, (size_t)cnt * sizeof(int64_t), cudaMemcpyDeviceToHost, o->stream));
            CK(cudaMemcpyAsync(&fill, U.fill, sizeof(blu_u64), cudaMemcpyDeviceToHost, o->stream));
        }
        CK(cudaStreamSynchronize(o->stream));
        if (fill > 0) {
            if ((st = up_ensure_host(o, (int64_t)fill)) != BLU_OK) return st;
            CK(cudaMemcpyAsync(U.h_ilhs, U.ilhs, (size_t)fill * sizeof(int64_t), cudaMemcpyDeviceToHost, o->stream));
            CK(cudaMemcpyAsync(U.h_xout, U.xout, (size_t)fill * sizeof(double), cudaMemcpyDeviceToHost, o->stream));
            CK(cudaStreamSynchronize(o->stream));
        }
        for (int b = 0; b < cnt; b++) {
            const size_t u = (size_t)(c0 + b);
            const int s = hs[2 * b], nz = hs[2 * b + 1];
            if (status) status[u] = s;
            nzlhs[u] = s == BLU_OK ? nz : -1;
            if (!rows && s == BLU_OK && nz > 0) {
                memcpy(ilhs + u * m, U.h_ilhs + hoff[b], (size_t)nz * sizeof(int64_t));
                memcpy(xlhs + u * m, U.h_xout + hoff[b], (size_t)nz * sizeof(double));
            }
            if (s != BLU_OK && worst == BLU_OK) worst = s;
        }
    }
    o->last_ms[1] = kms;
    o->info_dirty = 1;
    o->time_solve += wall_now() - tic;
    return worst;
}

extern "C" int blu_batch_solve_sparse(blu_batch_t *o, const int64_t *unit_begin, const int64_t *rhs_begin,
                                      const int64_t *irhs, const double *xrhs,
                                      int64_t *nzlhs, int64_t *ilhs, double *xlhs, int *status, char trans) {
    return solve_sparse_units(o, unit_begin, rhs_begin, irhs, xrhs, nzlhs, ilhs, xlhs, status, trans, false);
}

/* solve_dense (solve_dense.rs:24) for nrhs right-hand sides on every basis, one warp per unit (basis k,
 * right-hand side r) = unit k*nrhs + r.  The right-hand sides and solutions of a chunk are staged through
 * the pool; the factors are only read. */
extern "C" int blu_batch_solve_dense_multi(blu_batch_t *o, int64_t nrhs, const double *rhs, double *lhs, char trans, int *status) {
    if (!o || nrhs < 0 || (nrhs > 0 && (!rhs || !lhs))) return BLU_ERROR_INVALID_ARGUMENT;
    if (nrhs == 0) return BLU_OK;
    CK(cudaSetDevice(o->device));
    const double tic = wall_now();
    const size_t m = (size_t)o->d.m;
    const int64_t nunits = (int64_t)o->d.nmat * nrhs;
    const int64_t P = std::min<int64_t>(nunits, o->solve_units);
    int st = up_ensure_units(o, nunits);
    if (st == BLU_OK) st = up_ensure_dense(o, P);
    if (st != BLU_OK) return st;
    UnitPool &U = o->up;
    std::vector<int> hslot((size_t)nunits);
    for (int64_t u = 0; u < nunits; u++) hslot[(size_t)u] = (int)(u / nrhs);
    CK(cudaMemcpyAsync(U.slot, hslot.data(), (size_t)nunits * sizeof(int), cudaMemcpyHostToDevice, o->stream));
    double kms = 0.0;
    if ((st = up_compact_all(o, &kms)) != BLU_OK) return st;
    std::vector<int> hs((size_t)P);
    int worst = BLU_OK;
    for (int64_t c0 = 0; c0 < nunits; c0 += P) {
        const int cnt = (int)std::min<int64_t>(P, nunits - c0);
        CK(cudaMemcpyAsync(U.rhs, rhs + (size_t)c0 * m, (size_t)cnt * m * sizeof(double), cudaMemcpyHostToDevice, o->stream));
        timer_start(o);
        BLU_LAUNCH(k_solve_dense, cnt, 32, 0, o->stream, o->d, (const double *)U.rhs, U.lhs, trans, U.dstatus, U.work, cnt,
                   (const int *)U.slot + c0);
        o->launches++;
        CK(cudaGetLastError());
        timer_stop(o, 1);
        kms += o->last_ms[1];
        CK(cudaMemcpyAsync(lhs + (size_t)c0 * m, U.lhs, (size_t)cnt * m * sizeof(double), cudaMemcpyDeviceToHost, o->stream));
        CK(cudaMemcpyAsync(hs.data(), U.dstatus, (size_t)cnt * sizeof(int), cudaMemcpyDeviceToHost, o->stream));
        CK(cudaStreamSynchronize(o->stream));
        for (int b = 0; b < cnt; b++) {
            if (status) status[c0 + b] = hs[b];
            if (hs[b] != BLU_OK && worst == BLU_OK) worst = hs[b];
        }
    }
    o->last_ms[1] = kms;
    o->info_dirty = 1;
    o->time_solve += wall_now() - tic;
    return worst;
}

/* ------------------------------------------------------------------ */
/* batch: maxvolume on every basis at once (maxvolume.rs:64-224)       */
/* ------------------------------------------------------------------ */

/* The scope of one masked batch call (maxvolume, the subset, _dev, copy, save and restore calls): its device buffers
 * and pinned words, released on every way out, and the run mask, taken off the batch again so that later launches run
 * every slot. */
struct MaskedCall {
    blu_b200 *o;
    std::vector<void *> mem;
    unsigned long long *h_cnt = nullptr;
    int *h_st = nullptr;
    explicit MaskedCall(blu_b200 *b) : o(b) {}
    template <typename T> int alloc(T **p, size_t n) {
        int st = dalloc(o, p, n);
        if (st == BLU_OK) mem.push_back(*p);
        return st;
    }
    ~MaskedCall() {
        cudaStreamSynchronize(o->stream);
        o->d.run = nullptr;
        o->hrun.clear();
        for (void *p : mem) dfree(o, p);
        if (h_cnt) cudaFreeHost(h_cnt);
        if (h_st) cudaFreeHost(h_st);
    }
};

/* room for B's of up to maxnz entries in the row-wise copy, which only lives during a factorization: a larger one
 * replaces it, content dropped */
static int mv_ensure_bt_cap(blu_b200 *o, int64_t maxnz) {
    BluDev &d = o->d;
    if (maxnz <= d.bnz_cap) return BLU_OK;
    CK(cudaStreamSynchronize(o->stream));
    dfree(o, d.bt_idx); dfree(o, d.bt_val); d.bt_idx = nullptr; d.bt_val = nullptr;
    int st = dalloc(o, &d.bt_idx, (size_t)d.nmat * (size_t)maxnz);
    if (st == BLU_OK) st = dalloc(o, &d.bt_val, (size_t)d.nmat * (size_t)maxnz);
    if (st != BLU_OK) return st;
    d.bnz_cap = maxnz;
    return BLU_OK;
}

/* the bases with run = 1 are factorized (B as written by k_mv_decide), Reallocate handled as blu.rs:95-118
 * (grow the bases that asked, run them again), then condest/residual_test; every basis whose factorization is
 * not OK stops.  maxnz: the most entries of one of those B. */
static int mv_factorize(blu_b200 *o, MaskedCall &c, const MvDev &V, int64_t maxnz) {
    BluDev &d = o->d;
    const int n = d.nmat, g = (n + 127) / 128;
    { int st = mv_ensure_bt_cap(o, maxnz); if (st != BLU_OK) return st; }
    for (int attempt = 0;; attempt++) {
        if (attempt == 40) return BLU_ERROR_INTERNAL;
        int st = launch_factorize(o, o->stream, 0, n, attempt > 0);
        if (st != BLU_OK) return st;
        CK(cudaMemsetAsync(V.cnt + MV_CNT_REALLOC, 0, sizeof(unsigned long long), o->stream));
        BLU_LAUNCH(k_mv_factor_status, g, 128, 0, o->stream, V, d, 0);
        o->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(c.h_cnt, V.cnt, MV_CNT_N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, o->stream));
        CK(cudaStreamSynchronize(o->stream));
        if (c.h_cnt[MV_CNT_REALLOC] == 0) break;
        if ((st = fetch_info(o)) != BLU_OK) return st;
        if ((st = grow_hungry_slots(o)) != BLU_OK) return st;
    }
    if (o->norms) {
        BLU_LAUNCH(k_factor_norms, n, 128, 0, o->stream, d);
        o->launches++;
        CK(cudaGetLastError());
    }
    BLU_LAUNCH(k_mv_factor_status, g, 128, 0, o->stream, V, d, 1);
    o->launches++;
    CK(cudaGetLastError());
    return BLU_OK;
}

/* statuses of the last masked launch (stride words apart) and the counters: does a basis ask for more memory?
 * (a masked-out slot keeps the word of an earlier launch, which is never Reallocate once that launch is done) */
static int mv_any_realloc(blu_b200 *o, MaskedCall &c, const MvDev &V, const int *d_st, int stride, bool *any) {
    const size_t n = (size_t)o->d.nmat;
    CK(cudaMemcpyAsync(c.h_st, d_st, n * stride * sizeof(int), cudaMemcpyDeviceToHost, o->stream));
    CK(cudaMemcpyAsync(c.h_cnt, V.cnt, MV_CNT_N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, o->stream));
    CK(cudaStreamSynchronize(o->stream));
    *any = false;
    for (size_t k = 0; k < n; k++) *any = *any || c.h_st[k * stride] == BLU_REALLOCATE;
    return BLU_OK;
}

/* maxvolume (maxvolume.rs:64-224) on every basis of the batch, the bases in lockstep over their pool columns.
 * The pool, basis and isbasic are uploaded once; per column the host queues set-up, the masked 'N' solve,
 * leaving-row selection, the masked 'T' solve, the masked update and the refactorization decision, and reads
 * back only status words and counts (three synchronisations, two more when some basis refactorizes). */
extern "C" int blu_batch_maxvolume(blu_batch_t *o, int64_t ncol, const int64_t *a_begin, const int64_t *a_end,
                                   const int64_t *a_i, const double *a_x, int64_t anz_total,
                                   int64_t *basis, int64_t *isbasic, double volumetol, int64_t *nupdate, int *status) {
    if (!o || o->single) return BLU_ERROR_INVALID_ARGUMENT;
    if (ncol < 0 || anz_total < 0 || !basis || (ncol > 0 && (!a_begin || !a_end || !isbasic)) || (anz_total > 0 && (!a_i || !a_x)))
        return BLU_ERROR_INVALID_ARGUMENT;
    const int n = o->d.nmat, m = o->d.m;
    const size_t N = (size_t)n, M = (size_t)m, C = (size_t)ncol;
    auto reject = [&]() {
        for (size_t k = 0; k < N; k++) { if (nupdate) nupdate[k] = 0; if (status) status[k] = BLU_ERROR_INVALID_ARGUMENT; }
        return BLU_ERROR_INVALID_ARGUMENT;
    };
    if (volumetol < 1.0) return reject();      /* maxvolume.rs:83-90: nothing runs */
    /* the reference indexes out of bounds (a panic) here: one answer for the whole call instead */
    for (size_t q = 0; q < N * M; q++) if (basis[q] < 0 || basis[q] >= ncol) return reject();
    for (size_t q = 0; q < N * C; q++)
        if (a_begin[q] < 0 || a_begin[q] > anz_total || a_end[q] < 0 || a_end[q] > anz_total) return reject();
    CK(cudaSetDevice(o->device));
    BluDev &d = o->d;
    MaskedCall c(o);
    int st = ensure_b_cap(o, std::max<int64_t>(anz_total, 1));      /* the pool lives where B does; never a null pointer */
    if (st == BLU_OK) st = ensure_batch_sparse(o, 0);
    MvDev V;
    memset(&V, 0, sizeof V);
    V.nmat = n; V.m = m; V.ncol = ncol;
    blu_i64 *abeg = nullptr, *aend = nullptr, *iota = nullptr; int *ust = nullptr;
    if (st == BLU_OK) st = c.alloc(&abeg, N * C);
    if (st == BLU_OK) st = c.alloc(&aend, N * C);
    if (st == BLU_OK) st = c.alloc(&V.isbasic, N * C);
    if (st == BLU_OK) st = c.alloc(&V.basis, N * M);
    if (st == BLU_OK) st = c.alloc(&V.nupdate, N);
    if (st == BLU_OK) st = c.alloc(&V.mvst, N);
    if (st == BLU_OK) st = c.alloc(&V.run, N);
    if (st == BLU_OK) st = c.alloc(&V.rhs_begin, N);
    if (st == BLU_OK) st = c.alloc(&V.rhs_end, N);
    if (st == BLU_OK) st = c.alloc(&V.leave, N);
    if (st == BLU_OK) st = c.alloc(&iota, N + 1);
    if (st == BLU_OK) st = c.alloc(&ust, N);
    if (st == BLU_OK) st = c.alloc(&V.cnt, (size_t)MV_CNT_N);
    if (st != BLU_OK) return st;
    if (cudaMallocHost((void **)&c.h_cnt, MV_CNT_N * sizeof(unsigned long long)) != cudaSuccess ||
        cudaMallocHost((void **)&c.h_st, 2 * N * sizeof(int)) != cudaSuccess) return BLU_ERROR_OUT_OF_MEMORY;
    V.a_begin = abeg; V.a_end = aend;
    V.b_begin = (blu_i64 *)o->db_begin; V.b_end = (blu_i64 *)o->db_end;
    V.xtbl = o->sm_dbls;
    std::vector<blu_i64> hiota(N + 1);
    for (size_t k = 0; k <= N; k++) hiota[k] = (blu_i64)k;
    std::vector<int> ones(N, 1);
    const cudaStream_t s = o->stream;
    if (ncol > 0) {
        CK(cudaMemcpyAsync(abeg, a_begin, N * C * sizeof(int64_t), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(aend, a_end, N * C * sizeof(int64_t), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(V.isbasic, isbasic, N * C * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    }
    CK(cudaMemcpyAsync(V.basis, basis, N * M * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    if (anz_total > 0) {
        CK(cudaMemcpyAsync(o->db_i, a_i, (size_t)anz_total * sizeof(int64_t), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(o->db_x, a_x, (size_t)anz_total * sizeof(double), cudaMemcpyHostToDevice, s));
    }
    CK(cudaMemcpyAsync(iota, hiota.data(), (N + 1) * sizeof(blu_i64), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(V.run, ones.data(), N * sizeof(int), cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(o->sm_scal, 0, 2 * N * sizeof(int), s));      /* no status word of an earlier call says Reallocate */
    /* B is the basis' columns of the pool from now on (the resident B of the batch after the call) */
    d.b_begin = (const blu_i64 *)o->db_begin; d.b_end = (const blu_i64 *)o->db_end;
    d.b_i = (const blu_i64 *)o->db_i; d.b_x = o->db_x; d.b_total = anz_total;
    o->have_b = 1; o->b_external = 0;
    d.run = V.run;
    o->info_dirty = 1;
    const int g = (n + 127) / 128;
    auto read_cnt = [&]() -> int {
        CK(cudaMemcpyAsync(c.h_cnt, V.cnt, MV_CNT_N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        return BLU_OK;
    };
    /* decide + next (+ their counters); ust = null: the first factorization */
    auto decide_next = [&](const int *u, int64_t j0) -> int {
        CK(cudaMemsetAsync(V.cnt, 0, MV_CNT_N * sizeof(unsigned long long), s));
        CK(cudaMemsetAsync(V.cnt + MV_CNT_NEXT, 0xff, sizeof(unsigned long long), s));
        BLU_LAUNCH(k_mv_decide, n, 32, 0, s, V, d, u);
        BLU_LAUNCH(k_mv_next, n, 32, 0, s, V, (blu_i64)j0);
        o->launches += 2;
        CK(cudaGetLastError());
        return BLU_OK;
    };
    auto next_after_factorize = [&](int64_t j0) -> int {
        CK(cudaMemsetAsync(V.cnt + MV_CNT_NEXT, 0xff, sizeof(unsigned long long), s));
        BLU_LAUNCH(k_mv_next, n, 32, 0, s, V, (blu_i64)j0);
        o->launches++;
        CK(cudaGetLastError());
        return read_cnt();
    };

    /* the next column: ~0 from k_mv_next means that no basis is running any more */
    auto next_col = [&]() { return (int64_t)std::min<unsigned long long>(c.h_cnt[MV_CNT_NEXT], (unsigned long long)ncol); };
    /* a store that cannot grow, or a basis still asking after 40 runs, stops the pass */
    auto rerun = [&](auto run) -> int {
        int grown;
        const int rs = rerun_on_realloc(o, grow_batch_stores, run, &grown);
        return rs != BLU_REALLOCATE ? rs : grown != BLU_OK ? grown : BLU_ERROR_OUT_OF_MEMORY;
    };
    auto pass = [&]() -> int {
        /* the first factorization, maxvolume.rs:92-95 */
        if ((st = decide_next(nullptr, 0)) != BLU_OK || (st = read_cnt()) != BLU_OK) return st;
        if ((st = mv_factorize(o, c, V, (int64_t)c.h_cnt[MV_CNT_MAXNZ])) != BLU_OK) return st;
        if ((st = next_after_factorize(0)) != BLU_OK) return st;
        for (int64_t j = next_col(); j < ncol; j = next_col()) {
            /* B^{-1} a_j straight from the pool, maxvolume.rs:100-118 */
            BLU_LAUNCH(k_mv_setup, g, 128, 0, s, V, (blu_i64)j);
            o->launches++;
            st = rerun([&](bool again, bool *asks) -> int {
                SpMulti W{n, again, (const i64 *)V.rhs_begin, (const i64 *)V.rhs_end};
                BLU_LAUNCH(k_solve_sparse, n, 32, 0, s, d, 0, (const i64 *)o->db_i, (const double *)o->db_x, 'N', 1, 1,
                           o->sm_scal, (i64 *)o->sm_ilhs, o->sm_xout, W);
                o->launches++;
                CK(cudaGetLastError());
                return mv_any_realloc(o, c, V, o->sm_scal, 2, asks);
            });
            if (st != BLU_OK) return st;
            BLU_LAUNCH(k_mv_select, n, 32, 0, s, V, (blu_i64)j, (const int *)o->sm_scal, (const blu_i64 *)o->sm_ilhs, (const double *)o->sm_xout, volumetol);
            o->launches++;
            /* the leaving row, maxvolume.rs:143-150 */
            st = rerun([&](bool again, bool *asks) -> int {
                SpMulti W{n, again, (const i64 *)iota};
                BLU_LAUNCH(k_solve_sparse, n, 32, 0, s, d, 0, (const i64 *)V.leave, (const double *)nullptr, 'T', 1, 0,
                           o->sm_scal, (i64 *)o->sm_ilhs, o->sm_xout, W);
                BLU_LAUNCH(k_mv_absorb, g, 128, 0, s, V, (const int *)o->sm_scal, 2);
                o->launches += 2;
                CK(cudaGetLastError());
                return mv_any_realloc(o, c, V, o->sm_scal, 2, asks);
            });
            if (st != BLU_OK) return st;
            /* update and the refactorization policy, maxvolume.rs:151-170 */
            st = rerun([&](bool again, bool *asks) -> int {
                BLU_LAUNCH(k_update, n, 32, 0, s, d, 0.0, ust, (const double *)V.xtbl, again ? 1 : 0);
                o->launches++;
                return (st = decide_next(ust, j + 1)) != BLU_OK ? st : mv_any_realloc(o, c, V, ust, 1, asks);
            });
            if (st != BLU_OK) return st;
            if (c.h_cnt[MV_CNT_REFACTOR] > 0) {
                if ((st = mv_factorize(o, c, V, (int64_t)c.h_cnt[MV_CNT_MAXNZ])) != BLU_OK) return st;
                if ((st = next_after_factorize(j + 1)) != BLU_OK) return st;
            }
        }
        return BLU_OK;
    };
    const int failed = pass();
    if (failed == BLU_ERROR_CUDA) return failed;

    /* the resident B of the batch: every basis' final columns of the pool (k_mv_decide without an update status
     * writes the view of every basis whose run flag is set) */
    CK(cudaMemcpyAsync(V.run, ones.data(), N * sizeof(int), cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(V.cnt, 0, MV_CNT_N * sizeof(unsigned long long), s));
    BLU_LAUNCH(k_mv_decide, n, 32, 0, s, V, d, (const int *)nullptr);
    o->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(c.h_cnt, V.cnt, MV_CNT_N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    /* what the device holds, also when a store could not grow partway through the pass */
    std::vector<int> hst(N);
    std::vector<int64_t> hnup(N);
    CK(cudaMemcpyAsync(basis, V.basis, N * M * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    if (ncol > 0) CK(cudaMemcpyAsync(isbasic, V.isbasic, N * C * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(hnup.data(), V.nupdate, N * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(hst.data(), V.mvst, N * sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    /* a later factorization of the resident B needs a row-wise copy that holds it */
    if ((st = mv_ensure_bt_cap(o, (int64_t)c.h_cnt[MV_CNT_MAXNZ])) != BLU_OK) return st;
    int worst = BLU_OK;
    for (size_t k = 0; k < N; k++) {
        if (failed != BLU_OK && hst[k] == BLU_OK) hst[k] = failed;      /* the bases the failure stopped mid-pass */
        if (nupdate) nupdate[k] = hnup[k];
        if (status) status[k] = hst[k];
        if (hst[k] != BLU_OK && worst == BLU_OK) worst = hst[k];
    }
    return failed != BLU_OK ? failed : worst;
}

/* ------------------------------------------------------------------ */
/* batch: refactorize / change the basis of chosen bases only          */
/* ------------------------------------------------------------------ */

/* The selection of a subset call: nsel distinct slots in [0, nmat).  pos[k] = r for the r-th selected slot, -1 for
 * the others. */
static int subset_select(blu_b200 *o, int64_t nsel, const int64_t *sel, std::vector<int> &pos) {
    if (!o || o->single || nsel < 0 || nsel > o->d.nmat || (nsel > 0 && !sel)) return BLU_ERROR_INVALID_ARGUMENT;
    pos.assign((size_t)o->d.nmat, -1);
    for (int64_t r = 0; r < nsel; r++) {
        if (sel[r] < 0 || sel[r] >= o->d.nmat || pos[(size_t)sel[r]] >= 0) return BLU_ERROR_INVALID_ARGUMENT;
        pos[(size_t)sel[r]] = (int)r;
    }
    return BLU_OK;
}

/* the run mask of the selected slots on the batch until c goes out of scope */
static int subset_mask(blu_b200 *o, MaskedCall &c, const std::vector<int> &pos) {
    const size_t n = pos.size();
    std::vector<int> run(n);
    for (size_t k = 0; k < n; k++) run[k] = pos[k] >= 0;
    int *d_run = nullptr;
    int st = c.alloc(&d_run, n);
    if (st != BLU_OK) return st;
    CK(cudaMemcpyAsync(d_run, run.data(), n * sizeof(int), cudaMemcpyHostToDevice, o->stream));
    CK(cudaStreamSynchronize(o->stream));      /* (pageable source) */
    o->d.run = d_run;
    o->hrun.assign(run.begin(), run.end());
    return BLU_OK;
}

/* The summary of a device-resident call (blu_dev_calls.cuh): allocated on first use, cleared before each launch
 * attempt, read into pinned memory after it (DEV_SUM_N words, whatever the size of the batch). */
static int dev_sum_ensure(blu_b200 *o) {
    if (o->d_sum) return BLU_OK;
    int st = dalloc(o, &o->d_sum, DEV_SUM_N);
    if (st != BLU_OK) return st;
    if (cudaMallocHost((void **)&o->h_sum, DEV_SUM_N * sizeof(blu_u64)) != cudaSuccess) { cudaGetLastError(); o->h_sum = nullptr; dfree(o, o->d_sum); o->d_sum = nullptr; return BLU_ERROR_OUT_OF_MEMORY; }
    return BLU_OK;
}
static int dev_sum_reset(blu_b200 *o) {
    CK(cudaMemsetAsync(o->d_sum, 0, DEV_SUM_N * sizeof(blu_u64), o->stream));
    CK(cudaMemsetAsync(o->d_sum + DEV_SUM_FIRST, 0xff, sizeof(blu_u64), o->stream));
    return BLU_OK;
}
static int dev_sum_read(blu_b200 *o) {
    CK(cudaMemcpyAsync(o->h_sum, o->d_sum, DEV_SUM_N * sizeof(blu_u64), cudaMemcpyDeviceToHost, o->stream));
    CK(cudaStreamSynchronize(o->stream));
    return BLU_OK;
}
/* the first non-OK status of the summary (index order), BLU_OK if there is none */
static int dev_sum_first(const blu_b200 *o) {
    const blu_u64 f = o->h_sum[DEV_SUM_FIRST];
    return f == DEV_SUM_NONE ? BLU_OK : (int)(unsigned)(f & 0xffffffffu);
}
static int grid_of(int64_t n, int per) { return (int)std::max<int64_t>(1, std::min<int64_t>((n + per - 1) / per, 4096)); }
/* k_dev_finish over n slots or units; nothing to do for n == 0 */
static int dev_finish(blu_b200 *o, int n, int64_t idx0, const int *run, const int *scal, int stride, int *status, int64_t *nzlhs) {
    if (n <= 0) return BLU_OK;
    BLU_LAUNCH(k_dev_finish, grid_of(n, 256), 256, 0, o->stream, n, (blu_i64)idx0, run, scal, stride, status, (blu_i64 *)nzlhs, o->d_sum);
    o->launches++;
    CK(cudaGetLastError());
    return BLU_OK;
}

/* the B the bases were last factorized from (all-empty columns before the first factorization): column j of basis k is
 * i / x[b[k * m + j] : e[k * m + j]], entries [0, total) */
struct ResidentB { const blu_i64 *b, *e, *i; const double *x; blu_i64 total; };
static ResidentB resident_b(const blu_b200 *o) {
    const BluDev &d = o->d;
    if (o->b_external) return ResidentB{d.b_begin, d.b_end, d.b_i, d.b_x, o->have_b ? d.b_total : 0};
    return ResidentB{(const blu_i64 *)o->db_begin, (const blu_i64 *)o->db_end, (const blu_i64 *)o->db_i, o->db_x, o->have_b ? d.b_total : 0};
}

/* The resident B becomes, for every basis, the B it was last factorized from: the new columns of the slots with
 * pos[k] >= 0 (column j of slot k at nb/ne[pos[k]*m + j], entries in ni/nx, all in device memory), the others' old
 * ones, compacted into fresh library-owned buffers that replace the old ones.  *maxnz: the most entries of one new B.
 * The slots' entry counts are scanned on the host when it has the selection (hpos, the host copy of dpos), and on
 * the device otherwise, so that only the new total and *maxnz come back.  On failure the old resident B stays. */
static int rebuild_b(blu_b200 *o, MaskedCall &c, const int *dpos, const std::vector<int> *hpos, const blu_i64 *nb, const blu_i64 *ne,
                     const blu_i64 *ni, const double *nx, int64_t *maxnz) {
    BluDev &d = o->d;
    const size_t n = (size_t)d.nmat, M = (size_t)d.m;
    const cudaStream_t s = o->stream;
    const ResidentB B = resident_b(o);
    const blu_i64 *ob = B.b, *oe = B.e, *oi = B.i;
    const double *ox = B.x;
    const blu_i64 ototal = B.total;
    blu_i64 *tot = nullptr, *soff = nullptr;
    int st = c.alloc(&tot, n);
    if (st == BLU_OK) st = c.alloc(&soff, n);
    if (st == BLU_OK && !hpos) st = dev_sum_ensure(o);
    if (st != BLU_OK) return st;
    int64_t *rb = nullptr, *re = nullptr, *ri = nullptr; double *rx = nullptr;      /* the new resident B */
    auto drop = [&]() { dfree(o, rb); dfree(o, re); dfree(o, ri); dfree(o, rx); };
    if ((st = dalloc(o, &rb, n * M)) != BLU_OK || (st = dalloc(o, &re, n * M)) != BLU_OK) { drop(); return st; }
    timer_start(o);
    BLU_LAUNCH(k_sub_lengths, (int)n, 32, 0, s, d.m, dpos, ob, oe, ototal, nb, ne, (blu_i64 *)re, (blu_i64 *)rb, tot);
    o->launches++;
    CK(cudaGetLastError());
    int64_t total = 0;
    *maxnz = 0;
    if (hpos) {
        std::vector<int64_t> htot(n), hoff(n);
        CK(cudaMemcpyAsync(htot.data(), tot, n * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        for (size_t k = 0; k < n; k++) {
            hoff[k] = total; total += htot[k];
            if ((*hpos)[k] >= 0) *maxnz = std::max<int64_t>(*maxnz, htot[k]);
        }
        CK(cudaMemcpyAsync(soff, hoff.data(), n * sizeof(int64_t), cudaMemcpyHostToDevice, s));
        CK(cudaStreamSynchronize(s));      /* (pageable source) */
    } else {
        if ((st = dev_sum_reset(o)) != BLU_OK) return st;
        BLU_LAUNCH(k_dev_scan, 1, 256, 0, s, (int)n, dpos, (const blu_i64 *)tot, soff, o->d_sum);
        o->launches++;
        CK(cudaGetLastError());
        if ((st = dev_sum_read(o)) != BLU_OK) return st;
        total = (int64_t)o->h_sum[DEV_SUM_TOTAL];
        *maxnz = (int64_t)o->h_sum[DEV_SUM_MAXNZ];
    }
    if ((st = dalloc(o, &ri, (size_t)total)) != BLU_OK || (st = dalloc(o, &rx, (size_t)total)) != BLU_OK) { drop(); return st; }
    BLU_LAUNCH(k_sub_copy, (int)n, 256, 0, s, d.m, (const int *)dpos, ob, oi, ox, (const blu_i64 *)nb, (const blu_i64 *)ni, (const double *)nx,
               (const blu_i64 *)soff, (blu_i64 *)rb, (blu_i64 *)re, (blu_i64 *)ri, rx);
    o->launches++;
    CK(cudaGetLastError());
    timer_stop(o, 0);      /* (synchronizes: the old B is read no more) */
    dfree(o, o->db_begin); dfree(o, o->db_end); dfree(o, o->db_i); dfree(o, o->db_x);
    o->db_begin = rb; o->db_end = re; o->db_i = ri; o->db_x = rx; o->b_cap = total;
    o->have_b = 1; o->b_external = 0;
    d.b_total = total;
    /* a captured graph reads the old B */
#ifndef BLU_EMU
    if (o->have_graph) { cudaGraphExecDestroy(o->graph_exec); cudaGraphDestroy(o->graph); }
#endif
    o->have_graph = 0;
    return BLU_OK;
}

/* rebuild_b from host arrays: the selection's new B (column j of the r-th selected basis at b_begin/b_end[r*m + j])
 * goes up to the device first */
static int subset_rebuild_b(blu_b200 *o, MaskedCall &c, const std::vector<int> &pos, int64_t nsel, const int64_t *b_begin,
                            const int64_t *b_end, const int64_t *b_i, const double *b_x, int64_t bnz_total, int64_t *maxnz) {
    const size_t n = (size_t)o->d.nmat, cols = (size_t)nsel * (size_t)o->d.m;
    const cudaStream_t s = o->stream;
    blu_i64 *nb = nullptr, *ne = nullptr, *ni = nullptr; double *nx = nullptr; int *dpos = nullptr;
    int st = c.alloc(&nb, cols);
    if (st == BLU_OK) st = c.alloc(&ne, cols);
    if (st == BLU_OK) st = c.alloc(&ni, (size_t)bnz_total);
    if (st == BLU_OK) st = c.alloc(&nx, (size_t)bnz_total);
    if (st == BLU_OK) st = c.alloc(&dpos, n);
    if (st != BLU_OK) return st;
    CK(cudaMemcpyAsync(nb, b_begin, cols * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(ne, b_end, cols * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    if (bnz_total > 0) {
        CK(cudaMemcpyAsync(ni, b_i, (size_t)bnz_total * sizeof(int64_t), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(nx, b_x, (size_t)bnz_total * sizeof(double), cudaMemcpyHostToDevice, s));
    }
    CK(cudaMemcpyAsync(dpos, pos.data(), n * sizeof(int), cudaMemcpyHostToDevice, s));
    return rebuild_b(o, c, dpos, &pos, nb, ne, ni, nx, maxnz);
}

/* blu_batch_factorize for the selected bases only: the resident B is rebuilt, then factorize_resident runs under the
 * run mask (its Reallocate loop and grow_hungry_slots look at the selected slots only). */
extern "C" int blu_batch_factorize_subset(blu_batch_t *o, int64_t nsel, const int64_t *sel,
                                          const int64_t *b_begin, const int64_t *b_end,
                                          const int64_t *b_i, const double *b_x, int64_t bnz_total, int *status) {
    std::vector<int> pos;
    int st = subset_select(o, nsel, sel, pos);
    if (st != BLU_OK) return st;
    if (nsel > 0 && (!b_begin || !b_end)) return BLU_ERROR_INVALID_ARGUMENT;
    if (bnz_total < 0 || (bnz_total > 0 && (!b_i || !b_x))) return BLU_ERROR_INVALID_ARGUMENT;
    const size_t cols = (size_t)nsel * (size_t)o->d.m;
    for (size_t q = 0; q < cols; q++)
        if (b_begin[q] < 0 || b_begin[q] > bnz_total || b_end[q] < 0 || b_end[q] > bnz_total) return BLU_ERROR_INVALID_ARGUMENT;
    if (nsel == 0) return BLU_OK;
    CK(cudaSetDevice(o->device));
    MaskedCall c(o);
    int64_t maxnz = 0;
    if ((st = subset_rebuild_b(o, c, pos, nsel, b_begin, b_end, b_i, b_x, bnz_total, &maxnz)) != BLU_OK) return st;
    const double rebuild_ms = o->last_ms[0];
    if ((st = mv_ensure_bt_cap(o, maxnz)) != BLU_OK) return st;
    if ((st = subset_mask(o, c, pos)) != BLU_OK) return st;
    const int fst = factorize_resident(o);
    o->last_ms[0] += rebuild_ms;
    std::vector<int> st_k(o->hinfo.size());
    for (size_t k = 0; k < st_k.size(); k++) st_k[k] = o->hinfo[k].status;
    const int worst = tally_statuses(st_k.data(), 1, nsel, sel, status, nullptr);
    return fst != BLU_OK ? fst : worst;
}

/* blu_batch_solve_for_update for the selected bases only: the per-slot kernel under the run mask, right-hand sides
 * through per-slot begin/end offsets; the solutions of the selected slots are packed on the device and cross the
 * bus in one copy. */
extern "C" int blu_batch_solve_for_update_subset(blu_batch_t *o, int64_t nsel, const int64_t *sel, const int64_t *rhs_begin,
                                                 const int64_t *irhs, const double *xrhs, int want_solution,
                                                 int64_t *nzlhs, int64_t *ilhs, double *xlhs, int *status, char trans) {
    std::vector<int> pos;
    int st = subset_select(o, nsel, sel, pos);
    if (st != BLU_OK) return st;
    if (nsel == 0) return BLU_OK;
    if (!rhs_begin || (want_solution && (!nzlhs || !ilhs || !xlhs))) return BLU_ERROR_INVALID_ARGUMENT;
    const int64_t tot = rhs_begin[nsel];
    if (tot < 0 || (tot > 0 && !irhs)) return BLU_ERROR_INVALID_ARGUMENT;
    for (int64_t r = 0; r < nsel; r++) if (rhs_begin[r] < 0 || rhs_begin[r] > tot) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const size_t n = (size_t)o->d.nmat, m = (size_t)o->d.m;
    const cudaStream_t s = o->stream;
    MaskedCall c(o);
    if ((st = ensure_batch_sparse(o, tot)) != BLU_OK) return st;
    std::vector<int64_t> hb(n, 0), he(n, 0);
    for (int64_t r = 0; r < nsel; r++) { hb[(size_t)sel[r]] = rhs_begin[r]; he[(size_t)sel[r]] = rhs_begin[r + 1]; }
    blu_i64 *db = nullptr, *de = nullptr;
    if ((st = c.alloc(&db, n)) != BLU_OK || (st = c.alloc(&de, n)) != BLU_OK) return st;
    CK(cudaMemcpyAsync(db, hb.data(), n * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(de, he.data(), n * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    if (tot > 0) CK(cudaMemcpyAsync(o->sm_irhs, irhs, (size_t)tot * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    if (tot > 0 && xrhs) CK(cudaMemcpyAsync(o->sm_xrhs, xrhs, (size_t)tot * sizeof(double), cudaMemcpyHostToDevice, s));
    if ((st = subset_mask(o, c, pos)) != BLU_OK) return st;
    std::vector<int> hs(2 * n);
    st = rerun_on_realloc(o, grow_batch_stores, [&](bool rerun, bool *asks) -> int {
        SpMulti W{(int)n, rerun, (const i64 *)db, (const i64 *)de};
        BLU_LAUNCH(k_solve_sparse, (int)n, 32, 0, s, o->d, 0, (const i64 *)o->sm_irhs, xrhs ? (const double *)o->sm_xrhs : (const double *)nullptr,
                   trans, 1, want_solution ? 1 : 0, o->sm_scal, (i64 *)o->sm_ilhs, o->sm_xout, W);
        o->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(hs.data(), o->sm_scal, 2 * n * sizeof(int), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        /* (the words of the masked-out slots are stale) */
        for (int64_t r = 0; r < nsel; r++) *asks = *asks || hs[2 * (size_t)sel[r]] == BLU_REALLOCATE;
        return BLU_OK;
    });
    if (st != BLU_OK && st != BLU_REALLOCATE) return st;      /* Reallocate left over: a store could not grow */
    const int worst = tally_statuses(hs.data(), 2, nsel, sel, status, want_solution ? nzlhs : nullptr);
    o->info_dirty = 1;
    if (!want_solution) return worst;
    std::vector<int64_t> hoff((size_t)nsel + 1, 0);
    for (int64_t r = 0; r < nsel; r++) hoff[(size_t)r + 1] = hoff[(size_t)r] + std::max<int64_t>(nzlhs[r], 0);
    const int64_t fill = hoff[(size_t)nsel];
    if (fill == 0) return worst;
    blu_i64 *dsel = nullptr, *doff = nullptr, *pi = nullptr; double *px = nullptr;
    if ((st = c.alloc(&dsel, (size_t)nsel)) != BLU_OK || (st = c.alloc(&doff, (size_t)nsel + 1)) != BLU_OK ||
        (st = c.alloc(&pi, (size_t)fill)) != BLU_OK || (st = c.alloc(&px, (size_t)fill)) != BLU_OK) return st;
    if ((st = up_ensure_host(o, fill)) != BLU_OK) return st;
    UnitPool &U = o->up;
    CK(cudaMemcpyAsync(dsel, sel, (size_t)nsel * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(doff, hoff.data(), ((size_t)nsel + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    BLU_LAUNCH(k_sub_pack, (int)nsel, 128, 0, s, (int)m, (const blu_i64 *)dsel, (const blu_i64 *)doff, (const blu_i64 *)o->sm_ilhs,
               (const double *)o->sm_xout, pi, px);
    o->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(U.h_ilhs, pi, (size_t)fill * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(U.h_xout, px, (size_t)fill * sizeof(double), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    for (int64_t r = 0; r < nsel; r++) {
        const size_t q = (size_t)hoff[(size_t)r], nz = (size_t)(hoff[(size_t)r + 1] - hoff[(size_t)r]);
        if (nz) {
            memcpy(ilhs + (size_t)r * m, U.h_ilhs + q, nz * sizeof(int64_t));
            memcpy(xlhs + (size_t)r * m, U.h_xout + q, nz * sizeof(double));
        }
    }
    return worst;
}

/* blu_batch_update for the selected bases only, basis sel[r] with xtbl[r] */
extern "C" int blu_batch_update_subset(blu_batch_t *o, int64_t nsel, const int64_t *sel, const double *xtbl, int *status) {
    std::vector<int> pos;
    int st = subset_select(o, nsel, sel, pos);
    if (st != BLU_OK) return st;
    if (nsel == 0) return BLU_OK;
    if (!xtbl) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const size_t n = (size_t)o->d.nmat;
    const cudaStream_t s = o->stream;
    MaskedCall c(o);
    if ((st = ensure_batch_sparse(o, 0)) != BLU_OK) return st;
    std::vector<double> hx(n, 0.0);
    for (int64_t r = 0; r < nsel; r++) hx[(size_t)sel[r]] = xtbl[r];
    CK(cudaMemcpyAsync(o->sm_dbls, hx.data(), n * sizeof(double), cudaMemcpyHostToDevice, s));
    if ((st = subset_mask(o, c, pos)) != BLU_OK) return st;
    std::vector<int> hs(n);
    st = rerun_on_realloc(o, grow_batch_stores, [&](bool rerun, bool *asks) -> int {
        BLU_LAUNCH(k_update, (int)n, 32, 0, s, o->d, 0.0, o->sm_scal, (const double *)o->sm_dbls, rerun ? 1 : 0);
        o->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(hs.data(), o->sm_scal, n * sizeof(int), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        for (int64_t r = 0; r < nsel; r++) *asks = *asks || hs[(size_t)sel[r]] == BLU_REALLOCATE;
        return BLU_OK;
    });
    if (st != BLU_OK && st != BLU_REALLOCATE) return st;      /* Reallocate left over: a store could not grow */
    o->info_dirty = 1;
    return tally_statuses(hs.data(), 1, nsel, sel, status, nullptr);
}

/* ------------------------------------------------------------------ */
/* batch: the basis-change step on caller-owned device buffers         */
/* ------------------------------------------------------------------ */

/* The argument check of a device-resident call: the kernel queued by `check` counts violations into the summary,
 * which the host reads before anything else is queued. */
template <typename F> static int dev_validate(blu_b200 *o, F check) {
    int st = dev_sum_reset(o);
    if (st != BLU_OK) return st;
    check();
    o->launches++;
    CK(cudaGetLastError());
    if ((st = dev_sum_read(o)) != BLU_OK) return st;
    return o->h_sum[DEV_SUM_BAD] ? BLU_ERROR_INVALID_ARGUMENT : BLU_OK;
}

/* blu_batch_factorize_subset with a device run mask and B in the caller's device memory, per-basis layout.  The host
 * reads the mask (to know the selection) and the info block (as factorize_resident does); the resident B is rebuilt
 * on the device from the old one and the caller's. */
extern "C" int blu_batch_factorize_subset_dev(blu_batch_t *o, const int *d_run, const int64_t *d_b_begin, const int64_t *d_b_end,
                                              const int64_t *d_b_i, const double *d_b_x, int64_t bnz_total, int *d_status) {
    if (!o || o->single || !d_b_begin || !d_b_end || bnz_total < 0 || (bnz_total > 0 && (!d_b_i || !d_b_x))) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    BluDev &d = o->d;
    const int n = d.nmat;
    const cudaStream_t s = o->stream;
    std::vector<int> run((size_t)n, 1);
    if (d_run) {
        CK(cudaMemcpyAsync(run.data(), d_run, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    if (std::none_of(run.begin(), run.end(), [](int r) { return r != 0; })) return BLU_OK;
    int st = dev_sum_ensure(o);
    if (st != BLU_OK) return st;
    st = dev_validate(o, [&]() {
        BLU_LAUNCH(k_dev_check_b, n, 128, 0, s, d.m, d_run, (const blu_i64 *)d_b_begin, (const blu_i64 *)d_b_end, (blu_i64)bnz_total, o->d_sum);
    });
    if (st != BLU_OK) return st;
    MaskedCall c(o);
    int *dpos = nullptr, *scal = nullptr;
    if ((st = c.alloc(&dpos, (size_t)n)) != BLU_OK || (st = c.alloc(&scal, (size_t)n)) != BLU_OK) return st;
    BLU_LAUNCH(k_dev_pos, grid_of(n, 256), 256, 0, s, n, d_run, dpos);
    o->launches++;
    CK(cudaGetLastError());
    int64_t maxnz = 0;
    if ((st = rebuild_b(o, c, dpos, nullptr, (const blu_i64 *)d_b_begin, (const blu_i64 *)d_b_end, (const blu_i64 *)d_b_i, d_b_x, &maxnz)) != BLU_OK)
        return st;
    const double rebuild_ms = o->last_ms[0];
    if ((st = mv_ensure_bt_cap(o, maxnz)) != BLU_OK) return st;
    if (d_run) { d.run = d_run; o->hrun.assign(run.begin(), run.end()); }
    const int fst = factorize_resident(o);
    o->last_ms[0] += rebuild_ms;
    BLU_LAUNCH(k_dev_info_status, grid_of(n, 256), 256, 0, s, n, (const BluInfo *)d.info, scal);
    o->launches++;
    CK(cudaGetLastError());
    if ((st = dev_sum_reset(o)) != BLU_OK || (st = dev_finish(o, n, 0, d_run, scal, 1, d_status, nullptr)) != BLU_OK) return st;
    int worst = BLU_OK;
    for (int k = 0; k < n && worst == BLU_OK; k++) {
        const int sk = o->hinfo[(size_t)k].status;
        if (run[(size_t)k] && sk != BLU_OK) worst = sk == BLU_REALLOCATE ? BLU_ERROR_OUT_OF_MEMORY : sk;
    }
    return fst != BLU_OK ? fst : worst;
}

/* blu_batch_solve_for_update (d_run == NULL) or blu_batch_solve_for_update_subset (the set bits of d_run) on device
 * buffers: the per-slot kernel reads the caller's right-hand sides and writes the caller's ilhs / xlhs at k * m;
 * k_dev_finish turns the status words into the caller's status and nzlhs.  Per launch attempt the host reads the
 * summary, nothing else. */
extern "C" int blu_batch_solve_for_update_dev(blu_batch_t *o, const int *d_run, const int64_t *d_rhs_begin, const int64_t *d_irhs,
                                              const double *d_xrhs, int want_solution, int64_t *d_nzlhs, int64_t *d_ilhs, double *d_xlhs,
                                              int *d_status, char trans) {
    if (!o || o->single || !d_rhs_begin || (want_solution && (!d_nzlhs || !d_ilhs || !d_xlhs))) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const int n = o->d.nmat;
    const cudaStream_t s = o->stream;
    int st = ensure_batch_sparse(o, 0);
    if (st == BLU_OK) st = dev_sum_ensure(o);
    if (st != BLU_OK) return st;
    st = dev_validate(o, [&]() {
        BLU_LAUNCH(k_dev_check_rhs, grid_of(n + 1, 256), 256, 0, s, n, d_run, (const blu_i64 *)d_rhs_begin, d_irhs ? 0 : 1, o->d_sum);
    });
    if (st != BLU_OK) return st;
    MaskedCall c(o);
    o->d.run = d_run;
    i64 *il = want_solution ? (i64 *)d_ilhs : (i64 *)o->sm_ilhs;
    double *xl = want_solution ? d_xlhs : o->sm_xout;
    st = rerun_on_realloc(o, grow_batch_stores, [&](bool rerun, bool *asks) -> int {
        SpMulti W{n, rerun, (const i64 *)d_rhs_begin};
        BLU_LAUNCH(k_solve_sparse, n, 32, 0, s, o->d, 0, (const i64 *)d_irhs, d_xrhs, trans, 1, want_solution ? 1 : 0, o->sm_scal, il, xl, W);
        o->launches++;
        CK(cudaGetLastError());
        if ((st = dev_sum_reset(o)) != BLU_OK || (st = dev_finish(o, n, 0, d_run, o->sm_scal, 2, d_status, want_solution ? d_nzlhs : nullptr)) != BLU_OK ||
            (st = dev_sum_read(o)) != BLU_OK) return st;
        *asks = o->h_sum[DEV_SUM_REALLOC] != 0;
        return BLU_OK;
    });
    if (st != BLU_OK && st != BLU_REALLOCATE) return st;      /* Reallocate left over: a store could not grow */
    o->info_dirty = 1;
    return dev_sum_first(o);
}

/* blu_batch_update / blu_batch_update_subset on device buffers: basis k with d_xtbl[k] */
extern "C" int blu_batch_update_dev(blu_batch_t *o, const int *d_run, const double *d_xtbl, int *d_status) {
    if (!o || o->single || !d_xtbl) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const int n = o->d.nmat;
    const cudaStream_t s = o->stream;
    int st = ensure_batch_sparse(o, 0);
    if (st == BLU_OK) st = dev_sum_ensure(o);
    if (st != BLU_OK) return st;
    MaskedCall c(o);
    o->d.run = d_run;
    st = rerun_on_realloc(o, grow_batch_stores, [&](bool rerun, bool *asks) -> int {
        BLU_LAUNCH(k_update, n, 32, 0, s, o->d, 0.0, o->sm_scal, d_xtbl, rerun ? 1 : 0);
        o->launches++;
        CK(cudaGetLastError());
        if ((st = dev_sum_reset(o)) != BLU_OK || (st = dev_finish(o, n, 0, d_run, o->sm_scal, 1, d_status, nullptr)) != BLU_OK ||
            (st = dev_sum_read(o)) != BLU_OK) return st;
        *asks = o->h_sum[DEV_SUM_REALLOC] != 0;
        return BLU_OK;
    });
    if (st != BLU_OK && st != BLU_REALLOCATE) return st;      /* Reallocate left over: a store could not grow */
    o->info_dirty = 1;
    return dev_sum_first(o);
}

/* blu_batch_solve_sparse on device buffers.  The unit table is built on the device; the chunks run back to back, each
 * one's solutions moved from the pool to the caller's ilhs / xlhs at u * m by k_dev_unpack; one summary read at the
 * end. */
extern "C" int blu_batch_solve_sparse_dev(blu_batch_t *o, int64_t nunits, const int64_t *d_unit_begin, const int64_t *d_rhs_begin,
                                          const int64_t *d_irhs, const double *d_xrhs, int64_t *d_nzlhs, int64_t *d_ilhs, double *d_xlhs,
                                          int *d_status, char trans) {
    if (!o || o->single || nunits < 0 || nunits > 0x7fffffff || !d_unit_begin) return BLU_ERROR_INVALID_ARGUMENT;
    if (nunits > 0 && (!d_rhs_begin || !d_nzlhs || !d_ilhs || !d_xlhs)) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const double tic = wall_now();
    const int nmat = o->d.nmat;
    const size_t m = (size_t)o->d.m;
    const cudaStream_t s = o->stream;
    int st = dev_sum_ensure(o);
    if (st != BLU_OK) return st;
    st = dev_validate(o, [&]() {
        BLU_LAUNCH(k_dev_check_units, grid_of(std::max<int64_t>(nmat, nunits), 256), 256, 0, s, nmat, (const blu_i64 *)d_unit_begin,
                   (blu_i64)nunits, (const blu_i64 *)d_rhs_begin, (d_irhs && d_xrhs) ? 0 : 1, o->d_sum);
    });
    if (st != BLU_OK || nunits == 0) return st;
    const int64_t P = std::min<int64_t>(nunits, o->solve_units);
    st = up_ensure_units(o, nunits);
    if (st == BLU_OK) st = up_ensure_sparse(o, P, 0);
    if (st != BLU_OK) return st;
    UnitPool &U = o->up;
    BLU_LAUNCH(k_dev_unit_slots, grid_of(nunits, 256), 256, 0, s, nmat, (blu_i64)nunits, (const blu_i64 *)d_unit_begin, U.slot);
    o->launches++;
    CK(cudaGetLastError());
    timer_start(o);
    BLU_LAUNCH(k_garbage_perm, nmat, 32, 0, s, o->d);
    o->launches++;
    CK(cudaGetLastError());
    if ((st = dev_sum_reset(o)) != BLU_OK) return st;
    for (int64_t c0 = 0; c0 < nunits; c0 += P) {
        const int cnt = (int)std::min<int64_t>(P, nunits - c0);
        CK(cudaMemsetAsync(U.fill, 0, sizeof(blu_u64), s));
        SpMulti W{cnt, 0, (const i64 *)d_rhs_begin + c0, nullptr, U.ints, U.dbls, U.markers, U.slot + c0, U.fill, (i64 *)U.off};
        BLU_LAUNCH(k_solve_sparse<true>, cnt, 32, 0, s, o->d, 0, (const i64 *)d_irhs, d_xrhs, trans, 0, 1, U.scal, (i64 *)U.ilhs, U.xout, W);
        BLU_LAUNCH(k_dev_unpack, cnt, 128, 0, s, (int)m, (const int *)U.scal, (const blu_i64 *)U.off, (const blu_i64 *)U.ilhs,
                   (const double *)U.xout, (blu_i64 *)d_ilhs + (size_t)c0 * m, d_xlhs + (size_t)c0 * m);
        o->launches += 2;
        CK(cudaGetLastError());
        if ((st = dev_finish(o, cnt, c0, nullptr, U.scal, 2, d_status, d_nzlhs)) != BLU_OK) return st;
    }
    timer_stop(o, 1);
    if ((st = dev_sum_read(o)) != BLU_OK) return st;
    o->info_dirty = 1;
    o->time_solve += wall_now() - tic;
    return dev_sum_first(o);
}

/* blu_batch_solve_dense_multi on device buffers: the chunks read d_rhs and write d_lhs in place, back to back, with one
 * summary read at the end */
extern "C" int blu_batch_solve_dense_multi_dev(blu_batch_t *o, int64_t nrhs, const double *d_rhs, double *d_lhs, char trans, int *d_status) {
    if (!o || o->single || nrhs < 0 || (nrhs > 0 && (!d_rhs || !d_lhs))) return BLU_ERROR_INVALID_ARGUMENT;
    if (nrhs == 0) return BLU_OK;
    CK(cudaSetDevice(o->device));
    const double tic = wall_now();
    const size_t m = (size_t)o->d.m;
    const int64_t nunits = (int64_t)o->d.nmat * nrhs;
    if (nunits > 0x7fffffff) return BLU_ERROR_INVALID_ARGUMENT;
    const int64_t P = std::min<int64_t>(nunits, o->solve_units);
    const cudaStream_t s = o->stream;
    int st = dev_sum_ensure(o);
    if (st == BLU_OK) st = up_ensure_units(o, nunits);
    if (st == BLU_OK) st = up_ensure_dense(o, P);
    if (st != BLU_OK) return st;
    UnitPool &U = o->up;
    BLU_LAUNCH(k_dev_dense_slots, grid_of(nunits, 256), 256, 0, s, (blu_i64)nunits, (blu_i64)nrhs, U.slot);
    o->launches++;
    CK(cudaGetLastError());
    timer_start(o);
    BLU_LAUNCH(k_garbage_perm, o->d.nmat, 32, 0, s, o->d);
    o->launches++;
    CK(cudaGetLastError());
    if ((st = dev_sum_reset(o)) != BLU_OK) return st;
    for (int64_t c0 = 0; c0 < nunits; c0 += P) {
        const int cnt = (int)std::min<int64_t>(P, nunits - c0);
        BLU_LAUNCH(k_solve_dense, cnt, 32, 0, s, o->d, d_rhs + (size_t)c0 * m, d_lhs + (size_t)c0 * m, trans, U.dstatus, U.work, cnt,
                   (const int *)U.slot + c0);
        o->launches++;
        CK(cudaGetLastError());
        if ((st = dev_finish(o, cnt, c0, nullptr, U.dstatus, 1, d_status, nullptr)) != BLU_OK) return st;
    }
    timer_stop(o, 1);
    if ((st = dev_sum_read(o)) != BLU_OK) return st;
    o->info_dirty = 1;
    o->time_solve += wall_now() - tic;
    return dev_sum_first(o);
}

/* ------------------------------------------------------------------ */
/* batch: copy bases within the batch (fork a basis into other slots)  */
/* ------------------------------------------------------------------ */

/* the pairs of a copy call: distinct destinations, no destination that is also a source, no self-copy */
static int copy_check(blu_b200 *o, int64_t ncopy, const int64_t *dst, const int64_t *src) {
    if (!o || o->single || ncopy < 0 || ncopy > o->d.nmat || (ncopy > 0 && (!dst || !src))) return BLU_ERROR_INVALID_ARGUMENT;
    const int64_t n = o->d.nmat;
    std::vector<char> isdst((size_t)n, 0), issrc((size_t)n, 0);
    for (int64_t r = 0; r < ncopy; r++) {
        if (dst[r] < 0 || dst[r] >= n || src[r] < 0 || src[r] >= n || dst[r] == src[r] || isdst[(size_t)dst[r]]) return BLU_ERROR_INVALID_ARGUMENT;
        isdst[(size_t)dst[r]] = 1; issrc[(size_t)src[r]] = 1;
    }
    for (int64_t r = 0; r < ncopy; r++) if (issrc[(size_t)dst[r]]) return BLU_ERROR_INVALID_ARGUMENT;
    return BLU_OK;
}

/* blu_batch_copy after copy_check: the destinations take the sources' store capacities (new private stores in one
 * block, as grow_hungry_slots allocates them; the uniform store where the source has no private one), then one launch
 * of k_copy_slots copies the state and the resident B rows. */
static int copy_run(blu_b200 *o, int64_t ncopy, const int64_t *dst, const int64_t *src) {
    if (ncopy == 0) return BLU_OK;
    CK(cudaSetDevice(o->device));
    BluDev &d = o->d;
    const size_t n = (size_t)d.nmat, M = (size_t)d.m;
    const cudaStream_t s = o->stream;
    auto rnd = [](size_t b) { return (b + 255) & ~(size_t)255; };
    size_t bytes = 0;
    for (int64_t r = 0; r < ncopy; r++) {
        const BluSlotStore &e = o->hslot[(size_t)src[r]];
        if (e.l_idx) bytes += rnd((size_t)(e.l_mem + PADDING) * 4) + rnd((size_t)(e.l_mem + PADDING) * 8);
        if (e.u_idx) bytes += rnd((size_t)(e.u_mem + PADDING) * 4) + rnd((size_t)(e.u_mem + PADDING) * 8);
        if (e.w_idx) bytes += rnd((size_t)(2 * e.w_mem + PADDING) * 4) + rnd((size_t)(2 * e.w_mem + PADDING) * 8);
    }
    MaskedCall c(o);
    int *dpairs = nullptr;
    int st = c.alloc(&dpairs, 2 * (size_t)ncopy);
    if (st != BLU_OK) return st;
    unsigned char *blk = nullptr;
    if (bytes && (st = dalloc(o, &blk, bytes)) != BLU_OK) return st;
    /* nothing has changed so far; from here on the call completes */
    if (blk) o->ext_blocks.push_back(blk);
    size_t off = 0;
    auto take = [&](size_t b) { unsigned char *p = blk + off; off += rnd(b); return p; };
    std::vector<int> pairs(2 * (size_t)ncopy);
    for (int64_t r = 0; r < ncopy; r++) {
        const BluSlotStore &e = o->hslot[(size_t)src[r]];
        BluSlotStore f; memset(&f, 0, sizeof f);
        if (e.l_idx) { f.l_idx = (int *)take((size_t)(e.l_mem + PADDING) * 4); f.l_val = (double *)take((size_t)(e.l_mem + PADDING) * 8); f.l_mem = e.l_mem; }
        if (e.u_idx) { f.u_idx = (int *)take((size_t)(e.u_mem + PADDING) * 4); f.u_val = (double *)take((size_t)(e.u_mem + PADDING) * 8); f.u_mem = e.u_mem; }
        if (e.w_idx) { f.w_idx = (int *)take((size_t)(2 * e.w_mem + PADDING) * 4); f.w_val = (double *)take((size_t)(2 * e.w_mem + PADDING) * 8); f.w_mem = e.w_mem; }
        o->hslot[(size_t)dst[r]] = f;      /* (an old private block of dst is reclaimed at the next whole-batch store change) */
        pairs[2 * (size_t)r] = (int)dst[r]; pairs[2 * (size_t)r + 1] = (int)src[r];
    }
    o->have_overrides = 0;
    for (const BluSlotStore &e : o->hslot) if (e.l_idx || e.u_idx || e.w_idx) o->have_overrides = 1;
    CK(cudaMemcpyAsync(o->d_slot, o->hslot.data(), n * sizeof(BluSlotStore), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(dpairs, pairs.data(), pairs.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    /* caller-owned B: its column pointers move into the library-owned rows, which the copy then edits (b_i / b_x stay
     * the caller's) */
    if (o->b_external && d.b_begin != (const blu_i64 *)o->db_begin) {      /* (a later copy finds them moved already) */
        CK(cudaMemcpyAsync(o->db_begin, d.b_begin, n * M * sizeof(int64_t), cudaMemcpyDeviceToDevice, s));
        CK(cudaMemcpyAsync(o->db_end, d.b_end, n * M * sizeof(int64_t), cudaMemcpyDeviceToDevice, s));
        d.b_begin = (const blu_i64 *)o->db_begin; d.b_end = (const blu_i64 *)o->db_end;
    }
    timer_start(o);
    BLU_LAUNCH(k_copy_slots, (int)(ncopy * COPY_PARTS), COPY_THREADS, 0, s, d, (const int *)dpairs, (blu_i64 *)o->db_begin, (blu_i64 *)o->db_end);
    o->launches++;
    CK(cudaGetLastError());
    timer_stop(o, 0);      /* (synchronizes: the pageable sources above are read) */
    for (int64_t r = 0; r < ncopy; r++) o->hinfo[(size_t)dst[r]] = o->hinfo[(size_t)src[r]];
#ifndef BLU_EMU
    if (o->have_graph) { cudaGraphExecDestroy(o->graph_exec); cudaGraphDestroy(o->graph); }
#endif
    o->have_graph = 0;
    return BLU_OK;
}

extern "C" int blu_batch_copy(blu_batch_t *o, int64_t ncopy, const int64_t *dst, const int64_t *src) {
    const int st = copy_check(o, ncopy, dst, src);
    return st != BLU_OK ? st : copy_run(o, ncopy, dst, src);
}

/* d_from[k] = -1 keeps basis k, otherwise basis k becomes a copy of basis d_from[k]; the map is read on the host */
extern "C" int blu_batch_copy_dev(blu_batch_t *o, const int *d_from) {
    if (!o || o->single || !d_from) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(o->device));
    const int n = o->d.nmat;
    std::vector<int> from((size_t)n);
    CK(cudaMemcpyAsync(from.data(), d_from, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, o->stream));
    CK(cudaStreamSynchronize(o->stream));
    std::vector<int64_t> dst, src;
    for (int k = 0; k < n; k++) {
        if (from[(size_t)k] == -1) continue;
        if (from[(size_t)k] < 0) return BLU_ERROR_INVALID_ARGUMENT;      /* (>= nmat, self and chains: copy_check) */
        dst.push_back(k); src.push_back(from[(size_t)k]);
    }
    const int64_t ncopy = (int64_t)dst.size();
    const int st = copy_check(o, ncopy, dst.data(), src.data());
    return st != BLU_OK ? st : copy_run(o, ncopy, dst.data(), src.data());
}

/* ------------------------------------------------------------------ */
/* batch: save bases to images and restore them into any slot          */
/* ------------------------------------------------------------------ */

/* device scratch of the host variants: the images pass through it in chunks of at most this many bytes (or one image) */
#define IMG_SCRATCH ((size_t)1 << 30)

static bool img_aligned(const void *p) { return p && ((size_t)p & 15) == 0; }

/* the arguments of a save: idx in [0, nmat) (repeats allowed); buf (when given) with a 16-byte aligned pointer and a
 * capacity for every image */
static int save_check(blu_b200 *o, int64_t n, const int64_t *idx, void *const *buf, const int64_t *cap, int64_t *bytes) {
    if (!o || o->single || n < 0 || (n > 0 && (!idx || !bytes)) || (n > 0 && buf && !cap)) return BLU_ERROR_INVALID_ARGUMENT;
    for (int64_t r = 0; r < n; r++) {
        if (idx[r] < 0 || idx[r] >= o->d.nmat) return BLU_ERROR_INVALID_ARGUMENT;
        if (buf && !img_aligned(buf[r])) return BLU_ERROR_INVALID_ARGUMENT;
    }
    return BLU_OK;
}

/* the headers of the images of bases idx (on the device, checksum 0) and their sizes (bytes, on the host) */
static int save_extents(blu_b200 *o, MaskedCall &c, int64_t n, const int64_t *idx, int **didx, BluImage **dhdr, int64_t *bytes) {
    const cudaStream_t s = o->stream;
    blu_i64 *dbytes = nullptr;
    int st = c.alloc(didx, (size_t)n);
    if (st == BLU_OK) st = c.alloc(dhdr, (size_t)n);
    if (st == BLU_OK) st = c.alloc(&dbytes, (size_t)n);
    if (st != BLU_OK) return st;
    std::vector<int> hidx(idx, idx + n);
    CK(cudaMemcpyAsync(*didx, hidx.data(), (size_t)n * sizeof(int), cudaMemcpyHostToDevice, s));
    const ResidentB B = resident_b(o);
    BLU_LAUNCH(k_save_extents, (int)n, 32, 0, s, o->d, (const int *)*didx, B.b, B.e, B.total, *dhdr, dbytes);
    o->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(bytes, dbytes, (size_t)n * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return BLU_OK;
}

/* the images of bases didx into the device buffers dimg (n pointers, on the device), checksums included */
static int save_write(blu_b200 *o, MaskedCall &c, int64_t n, const int *didx, const BluImage *dhdr, unsigned char *const *dimg) {
    const cudaStream_t s = o->stream;
    blu_u64 *part = nullptr;
    int st = c.alloc(&part, (size_t)n * SAVE_PARTS);
    if (st != BLU_OK) return st;
    const ResidentB B = resident_b(o);
    BLU_LAUNCH(k_save_slots, (int)(n * SAVE_PARTS), SAVE_THREADS, 0, s, o->d, didx, dhdr, dimg, B.b, B.e, B.i, B.x, B.total, part);
    o->launches++;
    CK(cudaGetLastError());
    BLU_LAUNCH(k_save_sum, grid_of(n, 256), 256, 0, s, (int)n, (const blu_u64 *)part, dimg);
    o->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(s));
    return BLU_OK;
}

/* the save calls after their argument checks (n > 0; batch and object alike) */
static int save_device(blu_b200 *o, int64_t n, const int64_t *idx, void *const *d_buf, const int64_t *cap, int64_t *bytes) {
    CK(cudaSetDevice(o->device));
    MaskedCall c(o);
    int st;
    int *didx = nullptr; BluImage *dhdr = nullptr;
    if ((st = save_extents(o, c, n, idx, &didx, &dhdr, bytes)) != BLU_OK || !d_buf) return st;
    for (int64_t r = 0; r < n; r++) if (cap[r] < bytes[r]) return BLU_ERROR_INVALID_ARGUMENT;
    unsigned char **dimg = nullptr;
    if ((st = c.alloc(&dimg, (size_t)n)) != BLU_OK) return st;
    CK(cudaMemcpyAsync(dimg, d_buf, (size_t)n * sizeof(void *), cudaMemcpyHostToDevice, o->stream));
    return save_write(o, c, n, didx, dhdr, dimg);
}

/* the 256-byte rounded bytes of the images [r0, r1) that go through the scratch together, starting at r0 */
static int64_t img_chunk_end(int64_t r0, int64_t n, const std::vector<size_t> &sz, size_t scratch) {
    size_t put = sz[(size_t)r0];
    int64_t r1 = r0 + 1;
    while (r1 < n && put + sz[(size_t)r1] <= scratch) put += sz[(size_t)r1++];
    return r1;
}
static size_t img_scratch(const std::vector<size_t> &sz) {
    size_t tot = 0, big = 0;
    for (size_t b : sz) { tot += b; big = std::max(big, b); }
    return std::min(tot, std::max(IMG_SCRATCH, big));
}

static int save_host(blu_b200 *o, int64_t n, const int64_t *idx, void *const *buf, const int64_t *cap, int64_t *bytes) {
    CK(cudaSetDevice(o->device));
    const cudaStream_t s = o->stream;
    MaskedCall c(o);
    int st;
    int *didx = nullptr; BluImage *dhdr = nullptr;
    if ((st = save_extents(o, c, n, idx, &didx, &dhdr, bytes)) != BLU_OK || !buf) return st;
    for (int64_t r = 0; r < n; r++) if (cap[r] < bytes[r]) return BLU_ERROR_INVALID_ARGUMENT;
    std::vector<size_t> sz((size_t)n);
    for (int64_t r = 0; r < n; r++) sz[(size_t)r] = ((size_t)bytes[r] + 255) & ~(size_t)255;
    const size_t scratch = img_scratch(sz);
    unsigned char *scr = nullptr, **dimg = nullptr;
    if ((st = c.alloc(&scr, scratch)) != BLU_OK || (st = c.alloc(&dimg, (size_t)n)) != BLU_OK) return st;
    std::vector<unsigned char *> hp((size_t)n);
    for (int64_t r0 = 0, r1; r0 < n; r0 = r1) {
        r1 = img_chunk_end(r0, n, sz, scratch);
        for (int64_t r = r0, off = 0; r < r1; off += (int64_t)sz[(size_t)r], r++) hp[(size_t)r] = scr + off;
        CK(cudaMemcpyAsync(dimg + r0, hp.data() + r0, (size_t)(r1 - r0) * sizeof(void *), cudaMemcpyHostToDevice, s));
        if ((st = save_write(o, c, r1 - r0, didx + r0, dhdr + r0, dimg + r0)) != BLU_OK) return st;
        for (int64_t r = r0; r < r1; r++) CK(cudaMemcpyAsync(buf[r], hp[(size_t)r], (size_t)bytes[r], cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    return BLU_OK;
}

extern "C" int blu_batch_save(blu_batch_t *o, int64_t n, const int64_t *idx, void *const *buf, const int64_t *cap, int64_t *bytes) {
    const int st = save_check(o, n, idx, buf, cap, bytes);
    return st != BLU_OK || n == 0 ? st : save_host(o, n, idx, buf, cap, bytes);
}
extern "C" int blu_batch_save_dev(blu_batch_t *o, int64_t n, const int64_t *idx, void *const *d_buf, const int64_t *cap, int64_t *bytes) {
    const int st = save_check(o, n, idx, d_buf, cap, bytes);
    return st != BLU_OK || n == 0 ? st : save_device(o, n, idx, d_buf, cap, bytes);
}

/* the arguments of a restore: n distinct destinations in [0, nmat), every buffer 16-byte aligned and holding a header */
static int restore_check(blu_b200 *o, int64_t n, const int64_t *dst, const void *const *buf, const int64_t *cap) {
    if (!o || o->single || n < 0 || n > o->d.nmat || (n > 0 && (!dst || !buf || !cap))) return BLU_ERROR_INVALID_ARGUMENT;
    std::vector<char> seen((size_t)o->d.nmat, 0);
    for (int64_t r = 0; r < n; r++) {
        if (dst[r] < 0 || dst[r] >= o->d.nmat || seen[(size_t)dst[r]]) return BLU_ERROR_INVALID_ARGUMENT;
        seen[(size_t)dst[r]] = 1;
        if (!img_aligned(buf[r]) || cap[r] < (int64_t)sizeof(BluImage)) return BLU_ERROR_INVALID_ARGUMENT;
    }
    return BLU_OK;
}

/* a header this build can restore into a batch of dimension m from a buffer of cap bytes: its length is the one its
 * extents give, every extent within its capacity */
static bool img_header_ok(const BluImage &h, int m, int64_t cap) {
    if (h.magic != IMG_MAGIC || h.version != IMG_VERSION || h.m != m || h.info_bytes != (int)sizeof(BluInfo)) return false;
    if (h.length < (int64_t)sizeof(BluImage) || h.length > cap || (h.length & 15)) return false;
    if (h.l_mem < 1 || h.l_mem > 0x3fffffff || h.u_mem < 1 || h.u_mem > 0x3fffffff || h.w_mem < 1 || h.w_mem > 0x1fffffff) return false;
    if (h.l_n < 0 || h.l_n > h.l_mem || h.u_n < 0 || h.u_n > h.u_mem || h.w_n < 0 || h.w_n > h.w_mem) return false;
    if (h.bt_n < 0 || h.bt_n > 0x3fffffff || h.b_nz < 0 || h.b_nz > cap / 16) return false;
    return img_offset(h, IMG_NSEC) == h.length;
}

/* The images at the device pointers dimg (host array): their headers come up and are checked, then (verify) their
 * checksums on the device; nothing has changed when either fails.  commit: basis dst[r] becomes the basis of image r.
 * An object (n == 1, dst[0] == 0) has no per-basis stores: its own are replaced by stores of the image's capacities,
 * and its sorted row-wise U is rebuilt when the basis is fresh -- or, keep_ur, left to the caller (blu_clone). */
static int restore_images(blu_b200 *o, MaskedCall &c, int64_t n, const int64_t *dst, const unsigned char *const *dimg_h, const int64_t *cap,
                          bool verify, bool commit, bool keep_ur = false) {
    BluDev &d = o->d;
    const cudaStream_t s = o->stream;
    const size_t N = (size_t)d.nmat, M = (size_t)d.m;
    unsigned char **dimg = nullptr; BluImage *dhdr = nullptr;
    int st = c.alloc(&dimg, (size_t)n);
    if (st == BLU_OK) st = c.alloc(&dhdr, (size_t)n);
    if (st != BLU_OK) return st;
    CK(cudaMemcpyAsync(dimg, dimg_h, (size_t)n * sizeof(void *), cudaMemcpyHostToDevice, s));
    BLU_LAUNCH(k_img_headers, (int)n, SAVE_THREADS, 0, s, (const unsigned char *const *)dimg, dhdr);
    o->launches++;
    CK(cudaGetLastError());
    std::vector<BluImage> h((size_t)n);
    CK(cudaMemcpyAsync(h.data(), dhdr, (size_t)n * sizeof(BluImage), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    for (int64_t r = 0; r < n; r++) if (!img_header_ok(h[(size_t)r], d.m, cap[r])) return BLU_ERROR_INVALID_ARGUMENT;
    if (verify) {
        blu_u64 *part = nullptr;
        if ((st = c.alloc(&part, (size_t)n * SAVE_PARTS)) != BLU_OK || (st = dev_sum_ensure(o)) != BLU_OK) return st;
        BLU_LAUNCH(k_img_sum, (int)(n * SAVE_PARTS), SAVE_THREADS, 0, s, (const unsigned char *const *)dimg, (const BluImage *)dhdr, part);
        o->launches++;
        CK(cudaGetLastError());
        st = dev_validate(o, [&]() { BLU_LAUNCH(k_img_verdict, grid_of(n, 256), 256, 0, s, (int)n, (const blu_u64 *)part, (const BluImage *)dhdr, o->d_sum); });
        if (st != BLU_OK) return st;
    }
    if (!commit) return BLU_OK;
    /* the row-wise B's room, the destinations' private stores, the images' resident B staged for rebuild_b */
    auto rnd = [](size_t b) { return (b + 255) & ~(size_t)255; };
    int64_t btmax = 0, btot = 0;
    size_t bytes = 0;
    std::vector<int64_t> base((size_t)n);
    std::vector<int> pos(N, -1), hdst((size_t)n);
    for (int64_t r = 0; r < n; r++) {
        const BluImage &e = h[(size_t)r];
        btmax = std::max<int64_t>(btmax, e.bt_n);
        base[(size_t)r] = btot; btot += e.b_nz;
        if (!o->single && e.l_mem != d.l_mem) bytes += rnd((size_t)(e.l_mem + PADDING) * 4) + rnd((size_t)(e.l_mem + PADDING) * 8);
        if (!o->single && e.u_mem != d.u_mem) bytes += rnd((size_t)(e.u_mem + PADDING) * 4) + rnd((size_t)(e.u_mem + PADDING) * 8);
        if (!o->single && e.w_mem != d.w_mem) bytes += rnd((size_t)(2 * e.w_mem + PADDING) * 4) + rnd((size_t)(2 * e.w_mem + PADDING) * 8);
        pos[(size_t)dst[r]] = (int)r; hdst[(size_t)r] = (int)dst[r];
    }
    if ((st = mv_ensure_bt_cap(o, btmax)) != BLU_OK) return st;
    blu_i64 *nb = nullptr, *ne = nullptr, *ni = nullptr, *dbase = nullptr; double *nx = nullptr; int *dpos = nullptr, *ddst = nullptr;
    if ((st = c.alloc(&nb, (size_t)n * M)) != BLU_OK || (st = c.alloc(&ne, (size_t)n * M)) != BLU_OK ||
        (st = c.alloc(&ni, (size_t)btot)) != BLU_OK || (st = c.alloc(&nx, (size_t)btot)) != BLU_OK ||
        (st = c.alloc(&dbase, (size_t)n)) != BLU_OK || (st = c.alloc(&dpos, N)) != BLU_OK || (st = c.alloc(&ddst, (size_t)n)) != BLU_OK)
        return st;
    CK(cudaMemcpyAsync(dbase, base.data(), (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(dpos, pos.data(), N * sizeof(int), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(ddst, hdst.data(), (size_t)n * sizeof(int), cudaMemcpyHostToDevice, s));
    BLU_LAUNCH(k_img_stage_b, (int)n, SAVE_THREADS, 0, s, d.m, (const unsigned char *const *)dimg, (const BluImage *)dhdr,
               (const blu_i64 *)dbase, nb, ne, ni, nx);
    o->launches++;
    CK(cudaGetLastError());
    unsigned char *blk = nullptr;
    if (bytes && (st = dalloc(o, &blk, bytes)) != BLU_OK) return st;
    int64_t maxnz = 0;
    if ((st = rebuild_b(o, c, dpos, nullptr, nb, ne, ni, nx, &maxnz)) != BLU_OK) { dfree(o, blk); return st; }
    /* the resident B is the new one (a captured graph is dropped) */
    if (o->single) {
        /* the object's L, U and W stores (and the row-wise U, sized like U) become ones of the image's capacities; a
         * failed allocation keeps the old stores and factors */
        const BluImage &e = h[0];
        if ((e.l_mem != d.l_mem || e.u_mem != d.u_mem || e.w_mem != d.w_mem) && (st = swap_stores(o, e.l_mem, e.u_mem, e.w_mem)) != BLU_OK)
            return st;
    }
    /* from here on the call completes */
    if (blk) o->ext_blocks.push_back(blk);
    size_t off = 0;
    auto take = [&](size_t b) { unsigned char *p = blk + off; off += rnd(b); return p; };
    for (int64_t r = 0; r < n && !o->single; r++) {
        const BluImage &e = h[(size_t)r];
        BluSlotStore f; memset(&f, 0, sizeof f);
        if (e.l_mem != d.l_mem) { f.l_idx = (int *)take((size_t)(e.l_mem + PADDING) * 4); f.l_val = (double *)take((size_t)(e.l_mem + PADDING) * 8); f.l_mem = e.l_mem; }
        if (e.u_mem != d.u_mem) { f.u_idx = (int *)take((size_t)(e.u_mem + PADDING) * 4); f.u_val = (double *)take((size_t)(e.u_mem + PADDING) * 8); f.u_mem = e.u_mem; }
        if (e.w_mem != d.w_mem) { f.w_idx = (int *)take((size_t)(2 * e.w_mem + PADDING) * 4); f.w_val = (double *)take((size_t)(2 * e.w_mem + PADDING) * 8); f.w_mem = e.w_mem; }
        o->hslot[(size_t)dst[r]] = f;      /* (an old private block of dst is reclaimed at the next whole-batch store change) */
    }
    if (!o->single) {
        o->have_overrides = 0;
        for (const BluSlotStore &e : o->hslot) if (e.l_idx || e.u_idx || e.w_idx) o->have_overrides = 1;
        CK(cudaMemcpyAsync(o->d_slot, o->hslot.data(), N * sizeof(BluSlotStore), cudaMemcpyHostToDevice, s));
    }
    BLU_LAUNCH(k_restore_slots, (int)(n * SAVE_PARTS), SAVE_THREADS, 0, s, d, (const int *)ddst, (const BluImage *)dhdr, (const unsigned char *const *)dimg);
    o->launches++;
    CK(cudaGetLastError());
    if (o->single && !keep_ur) {
        /* have_ur as a factorization leaves it: k_build_ur sets it where the basis is fresh (nupdate 0, status OK or
         * WarningSingularMatrix).  k_build_ur counts in tmpi, which is slot state: the image's goes back after it, so
         * that the object holds exactly the image. */
        CK(cudaMemsetAsync(&d.info->have_ur, 0, sizeof(int), s));
        BLU_LAUNCH(k_build_ur, 1, 256, 0, s, d);
        o->launches++;
        CK(cudaGetLastError());
        const int t = IMG_STATE + STATE_TMPI;
        CK(cudaMemcpyAsync(d.tmpi, dimg_h[0] + img_offset(h[0], t), (size_t)img_section_bytes(h[0], t), cudaMemcpyDeviceToDevice, s));
        o->info_dirty = 1;
    }
    if (o->single) o->task_pending = 0;      /* (a pending blu_factorize_c0ntinue belonged to the old basis) */
    CK(cudaStreamSynchronize(s));      /* (pageable sources above) */
    for (int64_t r = 0; r < n; r++) o->hinfo[(size_t)dst[r]] = h[(size_t)r].info;
    return BLU_OK;
}

/* the restore calls after their argument checks (n > 0; batch and object alike) */
static int restore_device(blu_b200 *o, int64_t n, const int64_t *dst, const void *const *d_buf, const int64_t *cap) {
    CK(cudaSetDevice(o->device));
    MaskedCall c(o);
    return restore_images(o, c, n, dst, (const unsigned char *const *)d_buf, cap, true, true);
}

/* Through the device scratch in chunks; with more than one chunk, every chunk is verified before the first is
 * restored, so that a rejected image still changes nothing. */
static int restore_host(blu_b200 *o, int64_t n, const int64_t *dst, const void *const *buf, const int64_t *cap) {
    int st;
    std::vector<size_t> sz((size_t)n);
    for (int64_t r = 0; r < n; r++) {
        BluImage h;
        memcpy(&h, buf[r], sizeof h);
        if (!img_header_ok(h, o->d.m, cap[r])) return BLU_ERROR_INVALID_ARGUMENT;
        sz[(size_t)r] = ((size_t)h.length + 255) & ~(size_t)255;
    }
    CK(cudaSetDevice(o->device));
    const cudaStream_t s = o->stream;
    MaskedCall c(o);
    const size_t scratch = img_scratch(sz);
    unsigned char *scr = nullptr;
    if ((st = c.alloc(&scr, scratch)) != BLU_OK) return st;
    const bool one = img_chunk_end(0, n, sz, scratch) == n;
    std::vector<const unsigned char *> hp((size_t)n);
    for (int pass = one ? 1 : 0; pass < 2; pass++) {
        for (int64_t r0 = 0, r1; r0 < n; r0 = r1) {
            r1 = img_chunk_end(r0, n, sz, scratch);
            for (int64_t r = r0, off = 0; r < r1; off += (int64_t)sz[(size_t)r], r++) {
                hp[(size_t)r] = scr + off;
                CK(cudaMemcpyAsync(scr + off, buf[r], (size_t)((const BluImage *)buf[r])->length, cudaMemcpyHostToDevice, s));
            }
            if ((st = restore_images(o, c, r1 - r0, dst + r0, hp.data() + r0, cap + r0, one || pass == 0, pass == 1)) != BLU_OK) return st;
        }
    }
    return BLU_OK;
}

extern "C" int blu_batch_restore(blu_batch_t *o, int64_t n, const int64_t *dst, const void *const *buf, const int64_t *cap) {
    const int st = restore_check(o, n, dst, buf, cap);
    return st != BLU_OK || n == 0 ? st : restore_host(o, n, dst, buf, cap);
}
extern "C" int blu_batch_restore_dev(blu_batch_t *o, int64_t n, const int64_t *dst, const void *const *d_buf, const int64_t *cap) {
    const int st = restore_check(o, n, dst, d_buf, cap);
    return st != BLU_OK || n == 0 ? st : restore_device(o, n, dst, d_buf, cap);
}

/* ------------------------------------------------------------------ */
/* object: clone, save and restore (the batch calls' images, one basis) */
/* ------------------------------------------------------------------ */

static const int64_t OBJECT_SLOT = 0;

extern "C" int blu_save(blu_t *o, void *buf, int64_t cap, int64_t *bytes) {
    if (!o || !o->single || !bytes || (buf && !img_aligned(buf))) return BLU_ERROR_INVALID_ARGUMENT;
    return save_host(o, 1, &OBJECT_SLOT, buf ? &buf : nullptr, &cap, bytes);
}
extern "C" int blu_save_dev(blu_t *o, void *d_buf, int64_t cap, int64_t *bytes) {
    if (!o || !o->single || !bytes || (d_buf && !img_aligned(d_buf))) return BLU_ERROR_INVALID_ARGUMENT;
    return save_device(o, 1, &OBJECT_SLOT, d_buf ? &d_buf : nullptr, &cap, bytes);
}
extern "C" int blu_restore(blu_t *o, const void *buf, int64_t cap) {
    if (!o || !o->single || !img_aligned(buf) || cap < (int64_t)sizeof(BluImage)) return BLU_ERROR_INVALID_ARGUMENT;
    return restore_host(o, 1, &OBJECT_SLOT, &buf, &cap);
}
extern "C" int blu_restore_dev(blu_t *o, const void *d_buf, int64_t cap) {
    if (!o || !o->single || !img_aligned(d_buf) || cap < (int64_t)sizeof(BluImage)) return BLU_ERROR_INVALID_ARGUMENT;
    return restore_device(o, 1, &OBJECT_SLOT, &d_buf, &cap);
}

/* c (made by create_common with like = src) becomes src: src's image goes through device scratch (its three save
 * launches queue on src's stream and count in src's launches), is restored into c without a checksum pass, the sorted
 * row-wise U is copied as it is (k_build_ur would leave the same rows, but tmpi differently), and the host-side
 * parameters and getters follow. */
static int clone_into(blu_b200 *c, blu_b200 *src) {
    MaskedCall cs(src);
    int *didx = nullptr; BluImage *dhdr = nullptr; unsigned char *img = nullptr, **dimg = nullptr;
    int64_t bytes = 0;
    int st = save_extents(src, cs, 1, &OBJECT_SLOT, &didx, &dhdr, &bytes);
    if (st == BLU_OK) st = cs.alloc(&img, (size_t)bytes);
    if (st == BLU_OK) st = cs.alloc(&dimg, 1);
    if (st != BLU_OK) return st;
    CK(cudaMemcpyAsync(dimg, &img, sizeof img, cudaMemcpyHostToDevice, src->stream));
    if ((st = save_write(src, cs, 1, didx, dhdr, dimg)) != BLU_OK) return st;      /* (synchronizes) */
    {
        MaskedCall cc(c);
        const unsigned char *im = img;
        if ((st = restore_images(c, cc, 1, &OBJECT_SLOT, &im, &bytes, false, true, true)) != BLU_OK) return st;
    }
    const BluDev &s = src->d;
    BluDev &d = c->d;
    const cudaStream_t cst = c->stream;
    if (c->hinfo[0].have_ur) {
        int nur = 0;
        CK(cudaMemcpyAsync(&nur, s.ur_ptr + s.m, sizeof nur, cudaMemcpyDeviceToHost, cst));
        CK(cudaStreamSynchronize(cst));
        CK(cudaMemcpyAsync(d.ur_ptr, s.ur_ptr, (size_t)(s.m + 1) * sizeof(int), cudaMemcpyDeviceToDevice, cst));
        CK(cudaMemcpyAsync(d.dep_ur, s.dep_ur, (size_t)s.m * sizeof(int), cudaMemcpyDeviceToDevice, cst));
        CK(cudaMemcpyAsync(d.ur_idx, s.ur_idx, (size_t)nur * sizeof(int), cudaMemcpyDeviceToDevice, cst));
        CK(cudaMemcpyAsync(d.ur_val, s.ur_val, (size_t)nur * sizeof(double), cudaMemcpyDeviceToDevice, cst));
        CK(cudaStreamSynchronize(cst));
    }
    /* parameters (blu_set_param; the capacities and dense-tail sizes came with create_common) */
    d.prm = s.prm; d.tree_min = s.tree_min;
    c->realloc_factor = src->realloc_factor; c->norms = src->norms; c->nthreads = src->nthreads; c->tail_threads = src->tail_threads;
    c->split_min = src->split_min; c->cap = src->cap; c->solve_units = src->solve_units;
    /* the host-side getters and state */
    c->time_factorize = src->time_factorize; c->time_solve = src->time_solve; c->time_update = src->time_update;
    c->nrealloc = src->nrealloc; c->task_pending = src->task_pending; c->have_b = src->have_b;
    memcpy(c->last_ms, src->last_ms, sizeof c->last_ms); memcpy(c->last_part_ms, src->last_part_ms, sizeof c->last_part_ms);
    c->parts_timed = src->parts_timed; c->last_norms_ms = src->last_norms_ms;
    return BLU_OK;
}

extern "C" int blu_clone(blu_t **out, blu_t *src) {
    if (!out || !src || !src->single) return BLU_ERROR_INVALID_ARGUMENT;
    CK(cudaSetDevice(src->device));
    blu_b200 *c = nullptr;
    int st = create_common(&c, 1, src->d.m, src->d.bnz_cap, src->device, 1, src);
    if (st != BLU_OK) return st;
    if ((st = clone_into(c, src)) != BLU_OK) { destroy_common(c); return st; }
    *out = c;
    return BLU_OK;
}

/* ------------------------------------------------------------------ */
/* one batch over several GPUs of one process                          */
/* ------------------------------------------------------------------ */
struct blu_multi {
    int ndev; int64_t nmat, m;
    std::vector<blu_b200 *> part;
    std::vector<int64_t> first, count;
};

extern "C" int blu_multi_create(blu_multi_t **out, int64_t nmat, int64_t m, int64_t bnz_cap, const int *devices, int ndev) {
    if (!out || !devices || ndev < 1 || nmat < ndev || m < 1) return BLU_ERROR_INVALID_ARGUMENT;
    blu_multi *mb = new blu_multi();
    mb->ndev = ndev; mb->nmat = nmat; mb->m = m;
    const int64_t base = nmat / ndev, extra = nmat % ndev;      /* the split of blu_b200/shard.py */
    int st = BLU_OK;
    int caller_dev = 0;
    cudaGetDevice(&caller_dev);      /* creating the parts selects their devices: hand the caller's back afterwards */
    for (int d = 0; d < ndev && st == BLU_OK; d++) {
        const int64_t lo = d * base + std::min<int64_t>(d, extra), n = base + (d < extra ? 1 : 0);
        blu_b200 *p = nullptr;
        st = create_common(&p, n, m, bnz_cap, devices[d], 0);
        if (st == BLU_OK) { mb->part.push_back(p); mb->first.push_back(lo); mb->count.push_back(n); }
    }
    cudaSetDevice(caller_dev);
    if (st != BLU_OK) { for (auto *p : mb->part) destroy_common(p); delete mb; return st; }
    *out = mb;
    return BLU_OK;
}
extern "C" void blu_multi_destroy(blu_multi_t *mb) {
    if (!mb) return;
    int caller_dev = 0;
    cudaGetDevice(&caller_dev);
    for (auto *p : mb->part) destroy_common(p);
    cudaSetDevice(caller_dev);
    delete mb;
}
extern "C" blu_batch_t *blu_multi_part(blu_multi_t *mb, int d, int64_t *first, int64_t *count) {
    if (!mb || d < 0 || d >= mb->ndev) return nullptr;
    if (first) *first = mb->first[(size_t)d];
    if (count) *count = mb->count[(size_t)d];
    return mb->part[(size_t)d];
}

/* the work of one device: its range of bases, pointers rebased to the part of b_i / b_x the range uses */
static int multi_run_part(blu_multi *mb, int d, const int64_t *b_begin, const int64_t *b_end, const int64_t *b_i, const double *b_x,
                          int64_t bnz_total, const double *rhs, double *lhs, char trans, int *status) {
    const int64_t lo = mb->first[(size_t)d], n = mb->count[(size_t)d], m = mb->m;
    const size_t cols = (size_t)(n * m);
    const int64_t *bb = b_begin + lo * m, *be = b_end + lo * m;
    int64_t pmin = bnz_total, pmax = 0;
    for (size_t q = 0; q < cols; q++) { if (be[q] > bb[q]) { pmin = std::min(pmin, bb[q]); pmax = std::max(pmax, be[q]); } }
    if (pmax <= pmin) { pmin = 0; pmax = 0; }
    bool inside = pmin >= 0 && pmax <= bnz_total;
    if (!inside) { pmin = 0; pmax = bnz_total; }      /* out-of-range pointers: let the kernel report them per basis */
    std::vector<int64_t> rb(cols), re(cols);
    for (size_t q = 0; q < cols; q++) { rb[q] = bb[q] - pmin; re[q] = be[q] - pmin; }
    std::vector<int> st((size_t)n, 0);
    int rc = blu_batch_factorize(mb->part[(size_t)d], rb.data(), re.data(), b_i ? b_i + pmin : nullptr, b_x ? b_x + pmin : nullptr, pmax - pmin, st.data());
    if (rc == BLU_OK && rhs && lhs) {
        std::vector<int> ss((size_t)n, 0);
        rc = blu_batch_solve_dense(mb->part[(size_t)d], rhs + lo * m, lhs + lo * m, trans, ss.data());
        for (int64_t k = 0; k < n; k++) if (ss[(size_t)k] != BLU_OK && (st[(size_t)k] == BLU_OK || st[(size_t)k] == BLU_WARNING_SINGULAR_MATRIX)) st[(size_t)k] = ss[(size_t)k];
    }
    if (status) for (int64_t k = 0; k < n; k++) status[lo + k] = st[(size_t)k];
    return rc;
}

extern "C" int blu_multi_factorize_solve(blu_multi_t *mb, const int64_t *b_begin, const int64_t *b_end, const int64_t *b_i,
                                         const double *b_x, int64_t bnz_total, const double *rhs, double *lhs, char trans, int *status) {
    if (!mb || !b_begin || !b_end || bnz_total < 0 || (rhs && !lhs)) return BLU_ERROR_INVALID_ARGUMENT;
    std::vector<int> rc((size_t)mb->ndev, BLU_OK);
#ifndef BLU_EMU
    std::vector<std::thread> th;
    for (int d = 0; d < mb->ndev; d++)
        th.emplace_back([&, d]() { rc[(size_t)d] = multi_run_part(mb, d, b_begin, b_end, b_i, b_x, bnz_total, rhs, lhs, trans, status); });
    for (auto &t : th) t.join();
#else
    for (int d = 0; d < mb->ndev; d++) rc[(size_t)d] = multi_run_part(mb, d, b_begin, b_end, b_i, b_x, bnz_total, rhs, lhs, trans, status);
#endif
    for (int d = 0; d < mb->ndev; d++) if (rc[(size_t)d] != BLU_OK) return rc[(size_t)d];
    return BLU_OK;
}
