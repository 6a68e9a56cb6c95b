// serve_values_kernel.cu — packed-layout instance of the serve kernel for tables with programs of the wider data model
// (PF_VALUES); see serve_kernel.cu.
#define GOFR_TU_VALUES 1
#include "serve_body.cuh"

namespace gofr {

__global__ void __launch_bounds__(T, kServeCtas) serve_kernel_values(const __grid_constant__ ServeParams p) { serve_body<false>(p); }

int serve_values_blocks_per_sm(uint32_t smem_bytes) { return occupancy_blocks_per_sm(serve_kernel_values, T, smem_bytes); }

int launch_serve_values(const ServeParams& p, int grid, uint32_t smem_bytes, void* stream) {
    serve_kernel_values<<<grid, T, smem_bytes, (cudaStream_t)stream>>>(p);
    return (int)cudaGetLastError();
}

}  // namespace gofr
