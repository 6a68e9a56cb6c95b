// engine_internal.h — declarations shared by the host-side translation units of libgofr_b200.
#pragma once
#include <stdint.h>

#include <vector>

struct gofr_table;

void set_last_error(const char* fmt, ...);
const std::vector<uint8_t>& gofr_table_image(const gofr_table* t);

namespace gofr {

// Launch parameters of the fused serve kernel (serve_kernel.cu).
struct ServeParams {
    const void* desc;        // gofr_req_desc[n]
    const void* ids;         // uint8[n][16]
    const uint8_t* arena;
    uint32_t n;
    uint32_t n_tiles;
    const uint8_t* image;    // sealed table in HBM
    uint32_t hot_bytes;
    uint32_t epoch;          // look-back generation (state words from older launches read as "not ready")
    uint8_t* out;
    uint64_t out_cap;
    uint32_t* out_off;       // n + 1
    uint32_t* meta;          // n
    unsigned long long* tile_state;  // n_tiles
    uint32_t* overflow;      // set to 1 if out_cap was too small
    uint32_t in_cap;         // shared-memory staging capacity for request bytes (multiple of 16)
    uint32_t date[8];        // 29-byte IMF-fixdate, zero padded
    uint32_t* bind_scratch;  // n * bind_row_words words (tables with GOFR_H_BIND_ECHO routes), else null
    uint32_t bind_row_words;
    const unsigned long long* chain_pos;  // host-batch path: packed position of the whole batch so far (else null)
    uint32_t slot_bytes;     // 0: packed output (out_off = offsets, n + 1 entries); else response i lives in the slot
                             // out + i * slot_bytes (multiple of 16) and out_off[i] receives its length
    uint32_t debug_flags;    // bit0: skip the look-back (tile_base = tile * tile_total; only valid for fixed-size responses)
};

constexpr int kEpochBits = 24;  // look-back generation field of a tile state word (tile_common.cuh)
constexpr uint32_t kEpochMask = (1u << kEpochBits) - 1;

constexpr int kServeThreads = 128;  // gRPC / request-log kernels: requests per tile = threads per CTA
#ifndef GOFR_SERVE_T
#define GOFR_SERVE_T 128
#endif
#ifndef GOFR_SERVE_CTAS
#define GOFR_SERVE_CTAS 5
#endif
constexpr int kServeT = GOFR_SERVE_T;        // serve kernel: requests per tile = threads per CTA
constexpr int kServeCtas = GOFR_SERVE_CTAS;  // serve kernel: CTAs per SM the register and shared-memory budgets aim at
#ifndef GOFR_SERVE_CTAS_WIDE
#define GOFR_SERVE_CTAS_WIDE 4
#endif
constexpr int kServeCtasWide = GOFR_SERVE_CTAS_WIDE;  // slot layout, "wide" instance: 128 registers per thread (serve_slots_kernel.cu)

// How many response bytes one byte of a request's data section can turn into, at most (ImageHeader::reserved3[0], set at
// seal): 6 for flat rows (a control character becomes \u00XX); more when the table has programs of the wider data model,
// where a 4-byte element of a slice of structs drags its key literals along (`{"a_long_key":true},`).
template <typename Header>
inline uint32_t image_data_expand(const Header& H) { return H.reserved3[0] > 6u ? H.reserved3[0] : 6u; }

// Returns dynamic shared memory bytes needed for the table's hot part plus the request-byte staging area.
uint32_t serve_smem_bytes(uint32_t hot_bytes, uint32_t in_cap);
// cudaError_t as int
int launch_serve(const ServeParams& p, int grid, uint32_t smem_bytes, void* stream, bool wide_slots = false, bool values = false);
// grid of the persistent kernels of a group (wide: the 4-CTA slot-layout instance; else all the others) for that much
// dynamic shared memory, and the largest per-request staging budget that keeps `ctas` CTAs of the group resident
int serve_max_grid(uint32_t smem_bytes, int device, int* blocks_per_sm, bool wide);
uint32_t serve_fit_in_per(uint32_t hot_bytes, int ctas, bool wide);

#if defined(__CUDACC__)
// Host-side occupancy questions about a kernel of the translation unit that asks; -1 when the runtime cannot answer.
// Grid of a persistent kernel: CTAs of `threads` threads and `smem_bytes` of dynamic shared memory resident at once.
template <typename Kernel>
int occupancy_grid(Kernel kernel, int threads, size_t smem_bytes, int device) {
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return -1;
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem_bytes) != cudaSuccess) return -1;
    return nb * prop.multiProcessorCount;
}
// CTAs per SM once the kernel is allowed `smem_bytes` of dynamic shared memory.
template <typename Kernel>
int occupancy_blocks_per_sm(Kernel kernel, int threads, size_t smem_bytes) {
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes) != cudaSuccess) return -1;
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem_bytes) != cudaSuccess) return -1;
    return nb;
}
#endif

// egress of the host-batch path (egress_kernel.cu)
struct ChunkInfo {
    unsigned long long host_base;  // where this chunk starts in the caller's output buffer
    uint32_t base0;                // = host_base & 15: offset of the chunk inside its device buffer
    uint32_t total;
    uint32_t overflow;
    uint32_t pad;
};
int launch_advance(unsigned long long* chain_pos, const uint32_t* d_off, uint32_t n, uint32_t* d_overflow, ChunkInfo* info,
                   unsigned long long host_cap, void* stream);
int launch_egress(const ChunkInfo* info, const uint8_t* d_out, const uint32_t* d_off, const uint32_t* d_meta, uint32_t n,
                  uint8_t* h_out, uint32_t* h_off, uint32_t* h_meta, unsigned long long* h_status, int grid, void* stream);

struct GrpcParams {
    const uint8_t* in;
    const uint32_t* in_off;
    uint32_t n;
    uint32_t n_tiles;
    uint32_t epoch;
    uint8_t* out;
    uint64_t out_cap;
    uint32_t* out_off;
    uint32_t* meta;
    unsigned long long* tile_state;
    uint32_t* overflow;
};
int launch_grpc_hello(const GrpcParams& p, int grid, void* stream);
// message types of gofr_proto_encode_nested_device (kernel parameter, by value): up to 8 message types with 48 fields in
// all; fields of a type are consecutive, in ascending field-number order.  Rows use the layout of the wider data model
// (include/gofr_b200.h "Row format"): a singular message field is a presence word + the message's fixed part inline, a
// repeated field a count word with its elements in the variable part.
constexpr int kPbnMaxMsgs = 8, kPbnMaxFields = 48, kPbnMaxDepth = 4;
struct PbnField {
    uint32_t tag;        // number << 3 | wire type (2 for messages and for packed repeated scalars)
    uint8_t cls;         // PC_* bits of the scalar type; 0 for a message
    uint8_t repeated;
    uint8_t msg;         // message type index (type GOFR_PB_MESSAGE), else 0xFF
    uint8_t fixed_words; // words the field owns in the fixed part of its message
};
struct PbnDesc {
    uint32_t n_msgs, root;
    uint16_t first[kPbnMaxMsgs], count[kPbnMaxMsgs], fixed_words[kPbnMaxMsgs];
    PbnField f[kPbnMaxFields];
};
int launch_proto_encode_nested(const GrpcParams& p, const PbnDesc& D, int grid, void* stream);
int proto_nested_max_grid(int device);
int launch_proto_decode_nested(const GrpcParams& p, const PbnDesc& D, int grid, void* stream);
int proto_nested_decode_max_grid(int device);

// message type of gofr_proto_encode_device (kernel parameter, by value); 32 = GOFR_PROTO_MAX_FIELDS
struct ProtoSchema {
    uint32_t n_fields;
    uint32_t fixed_bytes;  // size of a row's fixed part
    uint32_t tag[32];      // number << 3 | wire type
    uint8_t cls[32];       // PC_* bits derived from the GOFR_PB_* type once, on the host (proto_class below)
};
#if defined(__CUDACC__)
#define GOFR_INTERNAL_HD __host__ __device__ inline
#else
#define GOFR_INTERNAL_HD inline
#endif
GOFR_INTERNAL_HD bool proto_is64(uint32_t t) {  // GOFR_PB_DOUBLE, INT64, UINT64, FIXED64, SFIXED64, SINT64
    return t == 1 || t == 3 || t == 4 || t == 6 || t == 16 || t == 18;
}
GOFR_INTERNAL_HD uint32_t proto_wire(uint32_t t) {
    if (t == 9 || t == 12) return 2;             // STRING, BYTES
    if (t == 1 || t == 6 || t == 16) return 1;   // DOUBLE, FIXED64, SFIXED64
    if (t == 2 || t == 7 || t == 15) return 5;   // FLOAT, FIXED32, SFIXED32
    return 0;
}
// What the per-message loops need to know about a field type, decided once per call on the host: the device tests bits
// instead of walking compare chains per field per message.
enum : uint32_t {
    PC_WIRE = 7u,       // wire type (0 varint, 1 fixed64, 2 length-delimited, 5 fixed32)
    PC_64 = 8u,         // two row words
    PC_ZIGZAG = 16u,    // sint32 / sint64
    PC_SIGNEXT = 32u,   // int32 / enum: negative values are sign-extended to 64 bits
    PC_UTF8 = 64u,      // string: must be valid UTF-8
    PC_BOOL = 128u,
};
GOFR_INTERNAL_HD uint32_t proto_class(uint32_t t) {
    uint32_t c = proto_wire(t);
    if (proto_is64(t)) c |= PC_64;
    if (t == 17 || t == 18) c |= PC_ZIGZAG;   // SINT32, SINT64
    if (t == 5 || t == 14) c |= PC_SIGNEXT;   // INT32, ENUM
    if (t == 9) c |= PC_UTF8;                 // STRING
    if (t == 8) c |= PC_BOOL;                 // BOOL
    return c;
}
int launch_proto_encode(const GrpcParams& p, const ProtoSchema& S, int grid, void* stream);
int proto_max_grid(int device);
int launch_proto_decode(const GrpcParams& p, const ProtoSchema& S, int grid, void* stream);
int proto_decode_max_grid(int device);

struct RouteParams {
    const void* desc;
    const uint8_t* arena;
    uint32_t n;
    const uint8_t* image;
    uint32_t hot_bytes;
    uint32_t* meta;   // n: status | route << 16
    uint32_t* vars;   // n * kMaxVars: off | len << 16
};
int launch_route(const RouteParams& p, int sm_count, void* stream);

struct BindParams {
    const void* desc;
    const uint8_t* arena;
    uint32_t n;
    const uint8_t* image;
    uint32_t hot_bytes;
    uint32_t schema_idx;
    uint8_t* out;          // n * slot_bytes
    uint32_t slot_bytes;
    uint32_t* len;         // n
    uint32_t* status;      // n
};
int launch_bind(const BindParams& p, int sm_count, void* stream);

struct HttpParams {
    const uint8_t* raw;
    const uint32_t* raw_off;  // n + 1
    uint32_t n;
    uint32_t n_tiles;
    void* desc;               // gofr_req_desc[n]
    uint8_t* arena;           // as large as raw (+16)
    uint32_t* status;         // n
    unsigned long long* spans;  // n * GOFR_HTTP_SPANS
};
int launch_http_parse(const HttpParams& p, int grid, void* stream);
int http_max_grid(int device);

struct LogParams {
    const void* desc;   // gofr_log_desc[n]
    const void* ids;    // n * 16 trace id bytes
    const uint8_t* arena;
    uint32_t n;
    uint32_t n_tiles;
    uint32_t epoch;
    uint8_t* out;
    uint64_t out_cap;
    uint32_t* out_off;
    unsigned long long* tile_state;
    uint32_t* overflow;
};
int launch_reqlog(const LogParams& p, int grid, void* stream);
int reqlog_max_grid(int device);
int grpc_max_grid(int device);

}  // namespace gofr
