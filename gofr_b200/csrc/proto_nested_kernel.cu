// proto_nested_kernel.cu — rows -> proto3 messages with nested and repeated fields (gofr_proto_encode_nested_device): the
// tile loop of the gRPC message path (frame_tiles.cuh) around the walker of proto_nested_device.cuh.  Its own translation
// unit, so that the flat encoder / decoder and the Hello kernel (grpc_kernel.cu) stay the binaries that were measured.
#include "frame_tiles.cuh"
#include "proto_nested_device.cuh"

namespace gofr {

struct PbnCodec {
    typedef PbnMsg R;
    const PbnDesc& D;
    __device__ R none() const { return PbnMsg{GOFR_GRPC_OK, 0}; }
    __device__ R parse(const uint8_t* row, uint32_t rn, uint32_t) const { R r = pbn_size(D, row, rn); rn_of = rn; return r; }
    __device__ void emit(const uint8_t* row, const R& r, uint8_t* dst, uint32_t* col) const { pbn_emit(D, row, rn_of, r, dst, col); }
    mutable uint32_t rn_of = 0;  // the row's length, from parse to emit (one codec object per thread)
};

__global__ void __launch_bounds__(GT, 6) proto_encode_nested_kernel(const GrpcParams p, const __grid_constant__ PbnDesc D) {
    __shared__ __align__(16) GrpcShared sh;
    frame_tiles(p, PbnCodec{D}, sh);
}

int launch_proto_encode_nested(const GrpcParams& p, const PbnDesc& D, int grid, void* stream) {
    proto_encode_nested_kernel<<<grid, GT, 0, (cudaStream_t)stream>>>(p, D);
    return (int)cudaGetLastError();
}

int proto_nested_max_grid(int device) { return occupancy_grid(proto_encode_nested_kernel, GT, 0, device); }

}  // namespace gofr
