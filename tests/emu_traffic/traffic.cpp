/* traffic.cpp -- the copy counters of the copy-counting emulator build (see cuda_emu.h here) */
#include <stddef.h>

static unsigned long long copy_bytes[5];      /* by cudaMemcpyKind: [1] host to device, [2] device to host, [3] device to device, [4] default */

void emu_traffic_count(int kind, size_t n) { copy_bytes[kind >= 1 && kind <= 4 ? kind : 0] += n; }
/* bytes copied since the last reset, by kind: out[0] unknown kind, out[1] host to device, out[2] device to host,
 * out[3] device to device, out[4] cudaMemcpyDefault */
extern "C" void cuda_emu_memcpy_bytes(unsigned long long *out) { for (int q = 0; q < 5; q++) out[q] = copy_bytes[q]; }
extern "C" void cuda_emu_memcpy_reset(void) { for (int q = 0; q < 5; q++) copy_bytes[q] = 0; }
