/* blu_save.cuh -- blu_batch_save / blu_batch_restore: a basis' factorization and update history as a self-contained byte
 * image in memory the caller owns, and back into any slot of any batch of the same dimension, so that a driver can park
 * more open nodes than its batch has slots, move a basis to another batch (on this or another GPU), or checkpoint.
 *
 * This module owns the image layout.  An image is a fixed-size header (BluImage) followed by the sections of
 * img_section_bytes, each starting 16-byte aligned, in this order:
 *   L index / value, U index / value, the live half of W index / value, the row-wise B index / value -- the live extents
 *   of blu_slot_state.cuh, W from the start of its live half --; the O(m) arrays of the state table but BluInfo (which
 *   is in the header); the resident B as entries: the m column lengths (int64, a negative length kept, by the rule of
 *   k_sub_lengths), then the entries' row indices (int64) and values, column after column.
 * Padding bytes are zero.  The header holds the checksum of the whole image (the checksum field counted as zero):
 * the sum mod 2^64 of img_mix(i, w) over the image's 4-byte words w at word index i -- one flipped byte changes one
 * term, img_mix is a bijection, so it changes the sum.  An image carries no parameters.
 *
 * Kernels, SAVE_THREADS threads per block:
 * - k_save_extents: one warp per image; the source's live extents, with the clamping of k_copy_slots, into the header.
 * - k_save_slots: one block per (image, part), the parts split as COPY_PARTS (COPY_CHUNKS chunks each of L, U, W and the
 *   row-wise B, one per O(m) array, the header with BluInfo, the resident B); each part writes its words and the
 *   partial checksum of them; k_save_sum adds the partials of an image in part order into its header.
 * - k_img_headers / k_img_sum / k_img_verdict: restore reads the headers, recomputes the checksums (nothing is written
 *   before they pass) and counts the mismatches into the call summary.
 * - k_img_stage_b: the images' resident B as rebuild_b's input (nb / ne / ni / nx).
 * - k_restore_slots: the inverse of k_save_slots into the destinations' stores. */
#ifndef BLU_SAVE_CUH
#define BLU_SAVE_CUH
#include <stddef.h>
#include "blu_slot_state.cuh"
#include "blu_copy.cuh"
#include "blu_dev_calls.cuh"

#define IMG_MAGIC 0x31474d49554c4255ULL      /* "UBLUIMG1" */
#define IMG_VERSION 1
#define SAVE_PARTS COPY_PARTS
#define SAVE_THREADS 256

struct alignas(16) BluImage {
    blu_u64 magic;
    int version, m;
    int info_bytes, pad;                          /* sizeof(BluInfo) of the build that wrote it; 0 */
    blu_i64 length;                               /* bytes of the whole image */
    blu_i64 l_mem, u_mem, w_mem;                  /* the store capacities of the basis */
    blu_i64 l_n, u_n, w_n, bt_n, b_nz;            /* extents: entries of L, U, W (from the live half's start), the row-wise B, the resident B */
    blu_u64 checksum;
    blu_i64 reserved;
    BluInfo info;
};

enum { IMG_HEADER = 0, IMG_L_IDX, IMG_L_VAL, IMG_U_IDX, IMG_U_VAL, IMG_W_IDX, IMG_W_VAL, IMG_BT_IDX, IMG_BT_VAL, IMG_STATE,
       IMG_B_LEN = IMG_STATE + STATE_INFO, IMG_B_I, IMG_B_X, IMG_NSEC };

BLU_HD blu_i64 img_round(blu_i64 b) { return (b + 15) & ~(blu_i64)15; }

/* bytes of section s (without its padding) */
BLU_HD blu_i64 img_section_bytes(const BluImage &h, int s) {
    switch (s) {
    case IMG_HEADER: return (blu_i64)sizeof(BluImage);
    case IMG_L_IDX: return 4 * h.l_n;   case IMG_L_VAL: return 8 * h.l_n;
    case IMG_U_IDX: return 4 * h.u_n;   case IMG_U_VAL: return 8 * h.u_n;
    case IMG_W_IDX: return 4 * h.w_n;   case IMG_W_VAL: return 8 * h.w_n;
    case IMG_BT_IDX: return 4 * h.bt_n; case IMG_BT_VAL: return 8 * h.bt_n;
    case IMG_B_LEN: return 8 * (blu_i64)h.m;
    case IMG_B_I: case IMG_B_X: return 8 * h.b_nz;
    default: return 4 * (blu_i64)state_words(s - IMG_STATE, (size_t)h.m);
    }
}
/* byte offset of section s (s = IMG_NSEC: the length of the image) */
BLU_HD blu_i64 img_offset(const BluImage &h, int s) {
    blu_i64 off = 0;
    for (int q = 0; q < s; q++) off += img_round(img_section_bytes(h, q));
    return off;
}
/* the start of the live W half, by the rule of live_w_lo */
BLU_HD blu_i64 img_w_lo(const BluImage &h) { return (blu_i64)(h.info.w_half ? 1 : 0) * h.w_mem; }

/* the checksum term of the 4-byte word w at word index i (splitmix64's finalizer, a bijection of 64 bits) */
BLU_HD blu_u64 img_mix(blu_u64 i, unsigned w) {
    blu_u64 x = (i << 32) | w;
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ULL;
    x ^= x >> 27; x *= 0x94d049bb133111ebULL;
    return x ^ (x >> 31);
}
#define IMG_CK_WORD (offsetof(BluImage, checksum) / 4)

/* the block's sum of v; thread 0 has it */
__device__ __forceinline__ blu_u64 img_block_sum(blu_u64 v) {
    __shared__ blu_u64 ws[32];
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(FULLMASK, v, d);
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) for (unsigned q = 1; q < (blockDim.x + 31) / 32; q++) v += ws[q];
    __syncthreads();
    return v;
}

/* exclusive scan of v over the block (blockDim.x a multiple of 32); *total = the block's sum */
__device__ __forceinline__ blu_i64 img_block_scan(blu_i64 v, blu_i64 *total) {
    __shared__ blu_i64 scr[33];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    blu_i64 incl = v;
    for (int d = 1; d < 32; d <<= 1) {
        const blu_i64 t = __shfl_up_sync(FULLMASK, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) scr[wid] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
        blu_i64 acc = 0;
        for (unsigned q = 0; q < blockDim.x / 32; q++) { const blu_i64 x = scr[q]; scr[q] = acc; acc += x; }
        scr[32] = acc;
    }
    __syncthreads();
    const blu_i64 res = incl - v + scr[wid];
    *total = scr[32];
    __syncthreads();
    return res;
}

/* the block writes the n words of src to the image words [wi, wi + n) and zeros to [wi + n, wi + npad): 16-byte
 * accesses when both are aligned alike; returns the thread's share of the checksum of those words */
__device__ __forceinline__ blu_u64 save_words(unsigned *img, size_t wi, const unsigned *src, size_t n, size_t npad) {
    unsigned *dst = img + wi;
    const size_t t = threadIdx.x, nt = blockDim.x;
    size_t head = n, nv = 0;
    if ((((size_t)dst ^ (size_t)src) & 15) == 0) {
        head = ((16 - ((size_t)src & 15)) & 15) / 4;
        if (head > n) head = n;
        nv = (n - head) / 4;
    }
    blu_u64 acc = 0;
    for (size_t q = t; q < head; q += nt) { const unsigned w = src[q]; dst[q] = w; acc += img_mix(wi + q, w); }
    const uint4 *s4 = (const uint4 *)(src + head);
    uint4 *d4 = (uint4 *)(dst + head);
    for (size_t q = t; q < nv; q += nt) {
        const uint4 v = s4[q];
        d4[q] = v;
        const size_t i = wi + head + 4 * q;
        acc += img_mix(i, v.x) + img_mix(i + 1, v.y) + img_mix(i + 2, v.z) + img_mix(i + 3, v.w);
    }
    for (size_t q = head + 4 * nv + t; q < n; q += nt) { const unsigned w = src[q]; dst[q] = w; acc += img_mix(wi + q, w); }
    for (size_t q = n + t; q < npad; q += nt) { dst[q] = 0; acc += img_mix(wi + q, 0); }
    return acc;
}

/* chunk c of COPY_CHUNKS of section s (n data words from src) */
__device__ __forceinline__ blu_u64 save_chunk(unsigned *img, const BluImage &h, int s, const unsigned *src, size_t n, int c) {
    const size_t w0 = (size_t)img_offset(h, s) / 4, np = (size_t)img_round(img_section_bytes(h, s)) / 4;
    const size_t a = np * c / COPY_CHUNKS, b = np * (c + 1) / COPY_CHUNKS;
    const size_t nd = n > a ? (n - a < b - a ? n - a : b - a) : 0;
    return save_words(img, w0 + a, src + a, nd, b - a);
}
/* its inverse: the data words of chunk c of section s to dst */
__device__ __forceinline__ void restore_chunk(unsigned *dst, const unsigned *img, const BluImage &h, int s, size_t n, int c) {
    const size_t w0 = (size_t)img_offset(h, s) / 4, np = (size_t)img_round(img_section_bytes(h, s)) / 4;
    const size_t a = np * c / COPY_CHUNKS, b = np * (c + 1) / COPY_CHUNKS;
    const size_t nd = n > a ? (n - a < b - a ? n - a : b - a) : 0;
    copy_words(dst + a, img + w0 + a, nd);
}

/* the store of part kind (0 L, 1 U, 2 W, 3 the row-wise B) of the slot viewed by A, from the first live entry; its
 * entries in the image and its first section */
__device__ __forceinline__ void img_store(const Mat &A, const BluImage &h, int kind, unsigned **idx, unsigned **val, blu_i64 *n, int *sec) {
    switch (kind) {
    case 0: *idx = (unsigned *)A.l_idx; *val = (unsigned *)A.l_val; *n = h.l_n; *sec = IMG_L_IDX; break;
    case 1: *idx = (unsigned *)A.u_idx; *val = (unsigned *)A.u_val; *n = h.u_n; *sec = IMG_U_IDX; break;
    case 2: { const blu_i64 lo = img_w_lo(h);
              *idx = (unsigned *)(A.w_idx + lo); *val = (unsigned *)(A.w_val + lo); *n = h.w_n; *sec = IMG_W_IDX; break; }
    default: *idx = (unsigned *)A.bt_idx; *val = (unsigned *)A.bt_val; *n = h.bt_n; *sec = IMG_BT_IDX; break;
    }
}

/* the length of column j of a resident B (ob / oe, entries [0, ototal)), by the rule of k_sub_lengths */
__device__ __forceinline__ blu_i64 img_col_len(const blu_i64 *ob, const blu_i64 *oe, blu_i64 ototal, size_t q) {
    const blu_i64 b = ob[q], e = oe[q];
    return (b < 0 || e > ototal) ? -1 : e - b;
}

/* One warp per image r: the header of the image of basis idx[r] (checksum 0) into hdr[r], its length into bytes[r].
 * ob / oe / ototal: the resident B. */
__global__ void __launch_bounds__(32) k_save_extents(BluDev D, const int *idx, const blu_i64 *ob, const blu_i64 *oe, blu_i64 ototal,
                                                     BluImage *hdr, blu_i64 *bytes) {
    __shared__ Mat S;
    const int r = blockIdx.x, lane = threadIdx.x & 31, k = idx[r];
    if (lane == 0) mat_view(S, D, k);
    __syncthreads();
    const int m = S.m;
    const BluInfo &I = *S.info;
    const blu_i64 u_end = live_u_end(S, I);
    blu_i64 bnz = 0;
    for (int j = lane; j < m; j += 32) {
        const blu_i64 n = img_col_len(ob, oe, ototal, (size_t)k * m + j);
        if (n > 0) bnz += n;
    }
    bnz = warp_sum64(bnz);
    BluImage &H = hdr[r];
    for (size_t q = lane; q < sizeof(BluInfo) / 4; q += 32) ((unsigned *)&H.info)[q] = ((const unsigned *)&I)[q];
    if (lane == 0) {
        H.magic = IMG_MAGIC; H.version = IMG_VERSION; H.m = m; H.info_bytes = (int)sizeof(BluInfo); H.pad = 0;
        H.l_mem = S.l_mem; H.u_mem = S.u_mem; H.w_mem = S.w_mem;
        H.l_n = live_l_end(S, I); H.u_n = u_end; H.w_n = live_w_end(S, I) - live_w_lo(S, I); H.bt_n = live_bt_end(S); H.b_nz = bnz;
        H.checksum = 0; H.reserved = 0;
        H.length = img_offset(H, IMG_NSEC);
        bytes[r] = H.length;
    }
}

/* The image of basis idx[r] into img[r], its parts' checksums into partial[r * SAVE_PARTS + part]. */
__global__ void __launch_bounds__(SAVE_THREADS) k_save_slots(BluDev D, const int *idx, const BluImage *hdr, unsigned char *const *img,
                                                             const blu_i64 *ob, const blu_i64 *oe, const blu_i64 *oi, const double *ox,
                                                             blu_i64 ototal, blu_u64 *partial) {
    __shared__ Mat S;
    const int r = (int)(blockIdx.x / SAVE_PARTS), part = (int)(blockIdx.x % SAVE_PARTS), k = idx[r];
    if (threadIdx.x == 0) mat_view(S, D, k);
    __syncthreads();
    const BluImage &H = hdr[r];
    unsigned *im = (unsigned *)img[r];
    blu_u64 acc = 0;
    const int a = part - 4 * COPY_CHUNKS;
    if (part < 4 * COPY_CHUNKS) {
        unsigned *si, *sv; blu_i64 n; int sec;
        img_store(S, H, part / COPY_CHUNKS, &si, &sv, &n, &sec);
        acc = save_chunk(im, H, sec, si, (size_t)n, part % COPY_CHUNKS) + save_chunk(im, H, sec + 1, sv, 2 * (size_t)n, part % COPY_CHUNKS);
    } else if (a < STATE_INFO) {
        size_t nw = 0;
        const unsigned *src = state_array(S, a, &nw);
        acc = save_words(im, (size_t)img_offset(H, IMG_STATE + a) / 4, src, nw, (size_t)img_round(4 * (blu_i64)nw) / 4);
    } else if (a == STATE_INFO) {
        acc = save_words(im, 0, (const unsigned *)&H, sizeof(BluImage) / 4, sizeof(BluImage) / 4);
    } else {      /* the resident B, column after column */
        const int m = S.m;
        const size_t wl = (size_t)img_offset(H, IMG_B_LEN) / 4, wi = (size_t)img_offset(H, IMG_B_I) / 4, wx = (size_t)img_offset(H, IMG_B_X) / 4;
        blu_i64 *len = (blu_i64 *)(im + wl), *bi = (blu_i64 *)(im + wi);
        double *bx = (double *)(im + wx);
        blu_i64 put = 0;
        for (int j0 = 0; j0 < m; j0 += blockDim.x) {
            const int j = j0 + (int)threadIdx.x;
            blu_i64 n = 0;
            if (j < m) {
                n = img_col_len(ob, oe, ototal, (size_t)k * m + j);
                len[j] = n;
                acc += img_mix(wl + 2 * (size_t)j, (unsigned)n) + img_mix(wl + 2 * (size_t)j + 1, (unsigned)((blu_u64)n >> 32));
            }
            blu_i64 tot;
            const blu_i64 at = put + img_block_scan(n > 0 ? n : 0, &tot);
            for (blu_i64 q = 0; q < n; q++) {
                const blu_i64 vi = oi[ob[(size_t)k * m + j] + q];
                const blu_u64 vx = (blu_u64)__double_as_longlong(ox[ob[(size_t)k * m + j] + q]);
                const size_t p = (size_t)(at + q);
                bi[p] = vi; bx[p] = ox[ob[(size_t)k * m + j] + q];
                acc += img_mix(wi + 2 * p, (unsigned)vi) + img_mix(wi + 2 * p + 1, (unsigned)((blu_u64)vi >> 32))
                     + img_mix(wx + 2 * p, (unsigned)vx) + img_mix(wx + 2 * p + 1, (unsigned)(vx >> 32));
            }
            put += tot;
        }
        const size_t nl = 2 * (size_t)m, ne = 2 * (size_t)H.b_nz;
        acc += save_words(im, wl + nl, nullptr, 0, (size_t)img_round(8 * (blu_i64)m) / 4 - nl)
             + save_words(im, wi + ne, nullptr, 0, (size_t)img_round(8 * H.b_nz) / 4 - ne)
             + save_words(im, wx + ne, nullptr, 0, (size_t)img_round(8 * H.b_nz) / 4 - ne);
    }
    acc = img_block_sum(acc);
    if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}

/* the checksum of image r from its parts' partials, added in part order, into its header */
__global__ void __launch_bounds__(256) k_save_sum(int n, const blu_u64 *partial, unsigned char *const *img) {
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x) {
        blu_u64 acc = 0;
        for (int p = 0; p < SAVE_PARTS; p++) acc += partial[(size_t)r * SAVE_PARTS + p];
        ((BluImage *)img[r])->checksum = acc;
    }
}

/* the header of image r into hdr[r].  One block per image. */
__global__ void __launch_bounds__(SAVE_THREADS) k_img_headers(const unsigned char *const *img, BluImage *hdr) {
    copy_words((unsigned *)(hdr + blockIdx.x), (const unsigned *)img[blockIdx.x], sizeof(BluImage) / 4);
}

/* part p of SAVE_PARTS of the checksum of image r (its checked length from hdr[r]), into partial[r * SAVE_PARTS + p] */
__global__ void __launch_bounds__(SAVE_THREADS) k_img_sum(const unsigned char *const *img, const BluImage *hdr, blu_u64 *partial) {
    const int r = (int)(blockIdx.x / SAVE_PARTS), p = (int)(blockIdx.x % SAVE_PARTS);
    const uint4 *im = (const uint4 *)img[r];
    const size_t n4 = (size_t)hdr[r].length / 16, a = n4 * p / SAVE_PARTS, b = n4 * (p + 1) / SAVE_PARTS;
    blu_u64 acc = 0;
    for (size_t q = a + threadIdx.x; q < b; q += blockDim.x) {
        const uint4 v = im[q];
        const size_t i = 4 * q;
        const unsigned w[4] = {v.x, v.y, v.z, v.w};
        for (int e = 0; e < 4; e++) acc += img_mix(i + e, (i + e == IMG_CK_WORD || i + e == IMG_CK_WORD + 1) ? 0u : w[e]);
    }
    acc = img_block_sum(acc);
    if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}

/* every image whose recomputed checksum differs from its header's counts into sum[DEV_SUM_BAD] */
__global__ void __launch_bounds__(256) k_img_verdict(int n, const blu_u64 *partial, const BluImage *hdr, blu_u64 *sum) {
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x) {
        blu_u64 acc = 0;
        for (int p = 0; p < SAVE_PARTS; p++) acc += partial[(size_t)r * SAVE_PARTS + p];
        if (acc != hdr[r].checksum) atomicAdd(&sum[DEV_SUM_BAD], 1ULL);
    }
}

/* The resident B of image r as rebuild_b's r-th new B: column j at nb / ne[r * m + j] (ne - nb = the saved length, a
 * negative one kept), its entries at base[r] onward in ni / nx.  One block per image. */
__global__ void __launch_bounds__(SAVE_THREADS) k_img_stage_b(int m, const unsigned char *const *img, const BluImage *hdr, const blu_i64 *base,
                                                              blu_i64 *nb, blu_i64 *ne, blu_i64 *ni, double *nx) {
    const int r = blockIdx.x;
    const BluImage &H = hdr[r];
    const unsigned char *im = img[r];
    const blu_i64 *len = (const blu_i64 *)(im + img_offset(H, IMG_B_LEN));
    blu_i64 put = base[r];
    for (int j0 = 0; j0 < m; j0 += blockDim.x) {
        const int j = j0 + (int)threadIdx.x;
        const blu_i64 n = j < m ? len[j] : 0;
        blu_i64 tot;
        const blu_i64 at = put + img_block_scan(n > 0 ? n : 0, &tot);
        if (j < m) { nb[(size_t)r * m + j] = at; ne[(size_t)r * m + j] = at + n; }
        put += tot;
    }
    copy_words((unsigned *)(ni + base[r]), (const unsigned *)(im + img_offset(H, IMG_B_I)), 2 * (size_t)H.b_nz);
    copy_words((unsigned *)(nx + base[r]), (const unsigned *)(im + img_offset(H, IMG_B_X)), 2 * (size_t)H.b_nz);
}

/* Basis dst[r] becomes the basis of image img[r] (header hdr[r], checked): every part of k_save_slots but the resident
 * B, which k_img_stage_b and rebuild_b install.  The destination's stores have the image's capacities already. */
__global__ void __launch_bounds__(SAVE_THREADS) k_restore_slots(BluDev D, const int *dst, const BluImage *hdr, const unsigned char *const *img) {
    __shared__ Mat T;
    const int r = (int)(blockIdx.x / SAVE_PARTS), part = (int)(blockIdx.x % SAVE_PARTS);
    if (threadIdx.x == 0) mat_view(T, D, dst[r]);
    __syncthreads();
    const BluImage &H = hdr[r];
    const unsigned *im = (const unsigned *)img[r];
    const int a = part - 4 * COPY_CHUNKS;
    if (part < 4 * COPY_CHUNKS) {
        unsigned *ti, *tv; blu_i64 n; int sec;
        img_store(T, H, part / COPY_CHUNKS, &ti, &tv, &n, &sec);
        restore_chunk(ti, im, H, sec, (size_t)n, part % COPY_CHUNKS);
        restore_chunk(tv, im, H, sec + 1, 2 * (size_t)n, part % COPY_CHUNKS);
    } else if (a < STATE_INFO) {
        size_t nw = 0;
        unsigned *d = state_array(T, a, &nw);
        copy_words(d, im + img_offset(H, IMG_STATE + a) / 4, nw);
    } else if (a == STATE_INFO) {
        copy_words((unsigned *)T.info, im + offsetof(BluImage, info) / 4, sizeof(BluInfo) / 4);
    }
}

#endif
