// Belief-map kernels of the flight variant that run as their own launch: flight_map_tile_kernel (after the
// thread-per-env step kernel) and flight_map_generic_kernel (after the lane-per-agent step kernel).  See flight_map.cuh.
#include "flight_internal.h"
#define CS_MAP_KERNELS
#include "flight_map.cuh"

namespace csf {

cudaError_t launch_map_tile(cs_flight* h, cudaStream_t st) {
    const int per_cta = kMapThreads / kTileLanes;
    const size_t smem = (size_t)per_cta * h->p.fm_env;
    flight_map_tile_kernel<<<(h->p.E + per_cta - 1) / per_cta, kMapThreads, smem, st>>>(h->p);
    cs_count_launch(1);
    return cudaGetLastError();
}

cudaError_t launch_map_generic(cs_flight* h, cudaStream_t st) {
    flight_map_generic_kernel<<<h->map_grid, kMapThreads, h->map_smem, st>>>(h->p, h->seq);
    cs_count_launch(1);
    return cudaGetLastError();
}

// The dynamic shared memory limit is per KERNEL, not per handle: it is only ever raised, to the largest request any handle
// of this process has made (a later, smaller handle must not lower it under an earlier one's launches).
cudaError_t map_set_smem_limit(size_t generic_bytes) {
    static size_t cur = 48 * 1024;
    if (generic_bytes <= cur) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(flight_map_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)generic_bytes);
    if (e == cudaSuccess) cur = generic_bytes;
    return e;
}

}  // namespace csf
