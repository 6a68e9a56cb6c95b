// grpc_kernel.cu — the gRPC message path over batches of length-prefixed frames, sm_100a: the unary Hello of config 5
// (request frame → response frame) and the proto3 encoder / decoder for any flat message type (rows ↔ frames).
//
// Same execution model as serve_kernel.cu: persistent co-resident CTAs, one thread per frame, the tile's contiguous
// input byte range pulled into shared memory with one TMA bulk copy, exact output sizes scanned in the CTA and chained
// across CTAs by the decoupled look-back, responses packed in request order and written through the aligned staging
// Writer (16-byte st.global.cs.v4).  Per-frame logic: grpc_device.cuh.
#include "frame_tiles.cuh"

namespace gofr {

struct HelloCodec {
    typedef HelloReq R;
    __device__ R none() const { return HelloReq{GOFR_GRPC_OK, 0, 0, 0}; }
    __device__ R parse(const uint8_t* f, uint32_t fn, uint32_t) const { return hello_parse(f, fn); }
    __device__ void emit(const uint8_t* f, const R& r, uint8_t* dst, uint32_t* col) const { hello_emit(f, r, dst, col); }
};

struct ProtoCodec {
    typedef ProtoMsg R;
    const ProtoSchema& S;
    __device__ R none() const { return ProtoMsg{GOFR_GRPC_OK, 0}; }
    __device__ R parse(const uint8_t* row, uint32_t rn, uint32_t off) const { return proto_size(S, row, rn, (off & 3u) == 0); }
    __device__ void emit(const uint8_t* row, const R& r, uint8_t* dst, uint32_t* col) const { proto_emit(S, row, r, dst, col); }
};

struct ProtoDecodeCodec {
    typedef ProtoRow R;
    const ProtoSchema& S;
    __device__ R none() const { ProtoRow r; r.status = GOFR_GRPC_OK; r.out_len = 0; return r; }
    __device__ R parse(const uint8_t* f, uint32_t fn, uint32_t) const { ProtoRow r; proto_decode_scan(S, f, fn, r); return r; }
    __device__ void emit(const uint8_t* f, const R& r, uint8_t* dst, uint32_t* col) const { proto_decode_emit(S, f, r, dst, col); }
};

__global__ void __launch_bounds__(GT, 12) grpc_hello_kernel(const GrpcParams p) {
    __shared__ __align__(16) GrpcShared sh;
    frame_tiles(p, HelloCodec{}, sh);
}

// rows → proto3 messages (gofr_proto_encode_device): the same pipeline, the row in place of the request frame
__global__ void __launch_bounds__(GT, 8) proto_encode_kernel(const GrpcParams p, const __grid_constant__ ProtoSchema S) {
    __shared__ __align__(16) GrpcShared sh;
    frame_tiles(p, ProtoCodec{S}, sh);
}

int launch_grpc_hello(const GrpcParams& p, int grid, void* stream) {
    grpc_hello_kernel<<<grid, GT, 0, (cudaStream_t)stream>>>(p);
    return (int)cudaGetLastError();
}

// frames → rows (gofr_proto_decode_device)
__global__ void __launch_bounds__(GT, 8) proto_decode_kernel(const GrpcParams p, const __grid_constant__ ProtoSchema S) {
    __shared__ __align__(16) GrpcShared sh;
    frame_tiles(p, ProtoDecodeCodec{S}, sh);
}

int launch_proto_decode(const GrpcParams& p, const ProtoSchema& S, int grid, void* stream) {
    proto_decode_kernel<<<grid, GT, 0, (cudaStream_t)stream>>>(p, S);
    return (int)cudaGetLastError();
}

int proto_decode_max_grid(int device) { return occupancy_grid(proto_decode_kernel, GT, 0, device); }

int launch_proto_encode(const GrpcParams& p, const ProtoSchema& S, int grid, void* stream) {
    proto_encode_kernel<<<grid, GT, 0, (cudaStream_t)stream>>>(p, S);
    return (int)cudaGetLastError();
}

int proto_max_grid(int device) { return occupancy_grid(proto_encode_kernel, GT, 0, device); }

int grpc_max_grid(int device) { return occupancy_grid(grpc_hello_kernel, GT, 0, device); }

}  // namespace gofr
