// serve_slots_kernel.cu — slot-layout instance of the serve kernel (serve_body.cuh): the resident headline kernel.
//
// Two register budgets of the same body exist: this one (5 CTAs/SM, 96 registers: the default) and
// serve_slots_wide_kernel.cu (4 CTAs/SM, 128 registers: opt-in).  The kernel is issue/latency bound; with five CTAs really
// resident (the staging budget comes from the occupancy calculator, engine.cu) this instance is 7.5 % faster than the wide
// one on config 2 (0.2737 against 0.2959 ms per 1 Mi requests) and 11 % faster on config 4 than it was with four.  They
// are separate translation units because whether CUDA 12.9's ptxas scalarises the 256-bit sector store
// (serve_device.cuh Writer::store32, _build.py) changes with what else is in the unit.
// Like the packed instance of serve_kernel.cu, this one and the wide one are compiled without the programs of the wider
// data model (GOFR_TU_VALUES 0); tables that have such programs run serve_slots_values_kernel.cu.
#define GOFR_TU_VALUES 0
#include "serve_body.cuh"

namespace gofr {

__global__ void __launch_bounds__(T, kServeCtas) serve_slots_kernel(const __grid_constant__ ServeParams p) { serve_body<true>(p); }

int serve_slots_wide_blocks_per_sm(uint32_t smem_bytes);
int launch_serve_slots_wide(const ServeParams& p, int grid, uint32_t smem_bytes, void* stream);
int serve_slots_values_blocks_per_sm(uint32_t smem_bytes);
int launch_serve_slots_values(const ServeParams& p, int grid, uint32_t smem_bytes, void* stream);

int serve_slots_blocks_per_sm(uint32_t smem_bytes, bool wide) {
    if (wide) return serve_slots_wide_blocks_per_sm(smem_bytes);
    const int nv = serve_slots_values_blocks_per_sm(smem_bytes);
    if (nv < 0) return -1;
    const int nb = occupancy_blocks_per_sm(serve_slots_kernel, T, smem_bytes);
    if (nb < 0) return -1;
    return nb < nv ? nb : nv;
}

int launch_serve_slots(const ServeParams& p, int grid, uint32_t smem_bytes, void* stream, bool wide, bool values) {
    if (values) return launch_serve_slots_values(p, grid, smem_bytes, stream);
    if (wide) return launch_serve_slots_wide(p, grid, smem_bytes, stream);
    serve_slots_kernel<<<grid, T, smem_bytes, (cudaStream_t)stream>>>(p);
    return (int)cudaGetLastError();
}

}  // namespace gofr
