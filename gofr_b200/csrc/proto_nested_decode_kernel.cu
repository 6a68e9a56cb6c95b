// proto_nested_decode_kernel.cu — length-prefixed frames -> rows for message types with nested and repeated fields
// (gofr_proto_decode_nested_device): the tile loop of the gRPC message path (frame_tiles.cuh) around the three walks of
// proto_nested_decode_device.cuh.  Its own translation unit, like the encoder's.
#include "frame_tiles.cuh"
#include "proto_nested_decode_device.cuh"

namespace gofr {

struct PdnCodec {
    typedef PdnRow R;
    const PbnDesc& D;
    __device__ R none() const { return PdnRow{GOFR_GRPC_OK, 0}; }
    __device__ R parse(const uint8_t* f, uint32_t fn, uint32_t) const { fn_of = fn; return pdn_decode_size(D, f, fn); }
    __device__ void emit(const uint8_t* f, const R& r, uint8_t* dst, uint32_t*) const { pdn_decode_emit(D, f, fn_of, r, dst); }
    mutable uint32_t fn_of = 0;  // the frame's length, from parse to emit (one codec object per thread)
};

__global__ void __launch_bounds__(GT, 6) proto_decode_nested_kernel(const GrpcParams p, const __grid_constant__ PbnDesc D) {
    __shared__ __align__(16) GrpcShared sh;
    frame_tiles(p, PdnCodec{D}, sh);
}

int launch_proto_decode_nested(const GrpcParams& p, const PbnDesc& D, int grid, void* stream) {
    proto_decode_nested_kernel<<<grid, GT, 0, (cudaStream_t)stream>>>(p, D);
    return (int)cudaGetLastError();
}

int proto_nested_decode_max_grid(int device) { return occupancy_grid(proto_decode_nested_kernel, GT, 0, device); }

}  // namespace gofr
