// serve_kernel.cu — packed-layout instance of the serve kernel (serve_body.cuh) and the launch helpers.
//
// This instance does not know the programs of the wider data model (PF_VALUES: float64, pointers, slices, maps ...): the
// packed layout has the interpreter inlined in its tile loop, and the two extra call sites cost every table registers
// (serve_device.cuh GOFR_TU_VALUES).  Tables that contain such a program are served by serve_values_kernel.cu.
#define GOFR_TU_VALUES 0
#include "serve_body.cuh"

namespace gofr {

__global__ void __launch_bounds__(T, kServeCtas) serve_kernel(const __grid_constant__ ServeParams p) { serve_body<false>(p); }

// slot-layout instance: serve_slots_kernel.cu
int serve_slots_blocks_per_sm(uint32_t smem_bytes, bool wide);
int launch_serve_slots(const ServeParams& p, int grid, uint32_t smem_bytes, void* stream, bool wide, bool values);
// packed layout, tables with PF_VALUES programs: serve_values_kernel.cu
int serve_values_blocks_per_sm(uint32_t smem_bytes);
int launch_serve_values(const ServeParams& p, int grid, uint32_t smem_bytes, void* stream);

uint32_t serve_smem_bytes(uint32_t hot_bytes, uint32_t in_cap) {
    return ((hot_bytes + 127u) & ~127u) + in_cap + 64;
}

// CTAs per SM with which every instance of a group is resident for `smem_bytes` of dynamic shared memory: the wide
// slot-layout instance alone, or all the others (packed / slots, with and without the wider data model).  Asked from
// the runtime (static shared memory, registers and the per-CTA reservation included) — a hand-kept formula fell behind
// the kernel once and the "5-CTA" instances silently ran 4 per SM.
int serve_blocks_per_sm(uint32_t smem_bytes, bool wide) {
    if (wide) return serve_slots_blocks_per_sm(smem_bytes, true);
    int nb = occupancy_blocks_per_sm(serve_kernel, T, smem_bytes);
    if (nb < 0) return -1;
    const int nb2 = serve_slots_blocks_per_sm(smem_bytes, false);
    const int nbv = serve_values_blocks_per_sm(smem_bytes);
    if (nb2 < 0 || nbv < 0) return -1;
    if (nb2 < nb) nb = nb2;
    if (nbv < nb) nb = nbv;
    return nb;
}

// The largest request staging budget (bytes per request: a multiple of 16 from 16 to 256) with which `ctas` CTAs of the
// group stay resident per SM next to a table of hot_bytes; 0 when not even the smallest one fits.
uint32_t serve_fit_in_per(uint32_t hot_bytes, int ctas, bool wide) {
    for (uint32_t in_per = 256; in_per >= 16; in_per -= 16) {
        const uint32_t smem = serve_smem_bytes(hot_bytes, ((uint32_t)T * in_per + 127u) & ~127u);
        if (smem > 227u * 1024u) continue;
        if (serve_blocks_per_sm(smem, wide) >= ctas) return in_per;
    }
    return 0;
}

int serve_max_grid(uint32_t smem_bytes, int device, int* blocks_per_sm, bool wide) {
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return -1;
    const int nb = serve_blocks_per_sm(smem_bytes, wide);
    if (nb < 0) return -1;
    if (blocks_per_sm) *blocks_per_sm = nb;
    return nb * prop.multiProcessorCount;
}

int launch_serve(const ServeParams& p, int grid, uint32_t smem_bytes, void* stream, bool wide_slots, bool values) {
    if (p.slot_bytes) return launch_serve_slots(p, grid, smem_bytes, stream, wide_slots && !values, values);
    if (values) return launch_serve_values(p, grid, smem_bytes, stream);
    serve_kernel<<<grid, T, smem_bytes, (cudaStream_t)stream>>>(p);
    return (int)cudaGetLastError();
}

}  // namespace gofr
