/* cuda_emu.h (copy-counting variant) -- the SIMT emulator of tests/emu with every cudaMemcpy* of the library counted
 * by kind, so that tests can check how many bytes a call moves between host and device.  TEST INFRASTRUCTURE ONLY.
 * blu_host.cu is compiled against this header (it comes first on the include path and pulls in the emulator's own);
 * the factorization objects and the scheduler are the ones tests/emu builds. */
#ifndef CUDA_EMU_TRAFFIC_H
#define CUDA_EMU_TRAFFIC_H
#include "../emu/cuda_emu.h"

void emu_traffic_count(int kind, size_t n);
inline cudaError_t emu_traffic_memcpy(void *d, const void *s, size_t n, int k) {
    emu_traffic_count(k, n);
    return cudaMemcpy(d, s, n, k);
}
inline cudaError_t emu_traffic_memcpy_async(void *d, const void *s, size_t n, int k, cudaStream_t st) {
    emu_traffic_count(k, n);
    return cudaMemcpyAsync(d, s, n, k, st);
}
inline cudaError_t emu_traffic_memcpy_2d_async(void *d, size_t dp, const void *s, size_t sp, size_t w, size_t h, int k, cudaStream_t st) {
    emu_traffic_count(k, w * h);
    return cudaMemcpy2DAsync(d, dp, s, sp, w, h, k, st);
}
#define cudaMemcpy(d, s, n, k) emu_traffic_memcpy(d, s, n, k)
#define cudaMemcpyAsync(d, s, n, k, st) emu_traffic_memcpy_async(d, s, n, k, st)
#define cudaMemcpy2DAsync(d, dp, s, sp, w, h, k, st) emu_traffic_memcpy_2d_async(d, dp, s, sp, w, h, k, st)
#endif
