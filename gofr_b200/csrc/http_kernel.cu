// http_kernel.cu — HTTP/1.1 request heads for a batch of raw messages (gofr_http_parse_device), sm_100a.
//
// One thread per message; a tile's contiguous byte range is pulled into shared memory with one TMA bulk copy (the
// same staging as the gRPC kernel: messages are back to back in d_raw).  No scan and no look-back: the parsed form of
// message i is written inside the byte range the message itself occupies in an equally sized arena, so nothing depends
// on the other messages.  Per-message logic: http_device.cuh.
#include <cuda_runtime.h>
#include <stdint.h>

#include "engine_internal.h"
#include "http_device.cuh"
#include "tile_common.cuh"

namespace gofr {

constexpr int HT = kServeThreads;
constexpr uint32_t kHttpStage = 26 * 1024;  // bytes of raw messages staged per tile (128 messages × 208 B): 8 CTAs per SM

struct HttpShared {
    uint64_t bar;
    __align__(16) uint8_t in[kHttpStage + 32];
};

__global__ void __launch_bounds__(HT, 8) http_parse_kernel(const HttpParams p) {
    __shared__ __align__(16) HttpShared sh;
    const uint32_t tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(&sh.bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    uint32_t parity = 0;
    for (uint32_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        const uint32_t i = tile * HT + tid;
        const bool valid = i < p.n;
        const uint32_t t0 = tile * HT, t1 = min(p.n, t0 + HT);
        const uint32_t lo = __ldg(p.raw_off + t0) & ~15u, hi = (__ldg(p.raw_off + t1) + 15u) & ~15u;
        const bool staged = hi > lo && hi - lo <= kHttpStage;
        __syncthreads();  // previous tile's reads of sh.in are done
        if (staged && tid == 0) {
            mbar_expect_tx(&sh.bar, hi - lo);
            bulk_g2s(sh.in, p.raw + lo, hi - lo, &sh.bar);
        }
        uint32_t mo = 0, mn = 0;
        if (valid) { mo = __ldg(p.raw_off + i); mn = __ldg(p.raw_off + i + 1) - mo; }
        const uint8_t* base = p.raw;
        if (staged) {
            mbar_wait(&sh.bar, parity);
            parity ^= 1;
            base = launder_after_sync((const uint8_t*)sh.in) - lo;
        }
        if (!valid) continue;
        const uint32_t a = (mo + 3u) & ~3u;
        HttpOut o;
        http_parse(base + mo, mn, p.arena + a, &o);
        p.status[i] = o.status;
        uint4 d = make_uint4(0, 0, 0, 0);
        if (o.status == GOFR_HTTP_OK) d = make_uint4(a, o.path_len | o.query_len << 16, o.data_len, o.method | o.flags << 8);
        ((uint4*)p.desc)[i] = d;
#pragma unroll
        for (int k = 0; k < GOFR_HTTP_SPANS; k++) {
            const unsigned long long s = o.spans[k];
            p.spans[(size_t)i * GOFR_HTTP_SPANS + k] = o.status == GOFR_HTTP_OK ? s + mo : 0ull;  // offsets into d_raw
        }
    }
}

int launch_http_parse(const HttpParams& p, int grid, void* stream) {
    http_parse_kernel<<<grid, HT, 0, (cudaStream_t)stream>>>(p);
    return (int)cudaGetLastError();
}

int http_max_grid(int device) { return occupancy_grid(http_parse_kernel, HT, 0, device); }

}  // namespace gofr
