// serve_slots_wide_kernel.cu — slot-layout instance of the serve kernel with the 128-register budget (4 CTAs/SM); see
// serve_slots_kernel.cu for when the engine uses it.
#define GOFR_TU_VALUES 0
#include "serve_body.cuh"

namespace gofr {

__global__ void __launch_bounds__(T, kServeCtasWide) serve_slots_kernel_wide(const __grid_constant__ ServeParams p) { serve_body<true>(p); }

int serve_slots_wide_blocks_per_sm(uint32_t smem_bytes) { return occupancy_blocks_per_sm(serve_slots_kernel_wide, T, smem_bytes); }

int launch_serve_slots_wide(const ServeParams& p, int grid, uint32_t smem_bytes, void* stream) {
    serve_slots_kernel_wide<<<grid, T, smem_bytes, (cudaStream_t)stream>>>(p);
    return (int)cudaGetLastError();
}

}  // namespace gofr
