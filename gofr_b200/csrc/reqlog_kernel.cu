// reqlog_kernel.cu — the RequestLog JSON line of middleware.Logging for a whole batch (sm_100a).
//
// Same execution model as serve_kernel.cu / grpc_kernel.cu: persistent co-resident CTAs, one thread per record, the
// tile's contiguous arena byte range pulled into shared memory with one TMA bulk copy, exact line lengths scanned in
// the CTA and chained across CTAs by the decoupled look-back, lines packed in record order and written through the
// aligned staging Writer (16-byte st.global.cs.v4).  Per-record logic: reqlog_device.cuh.
#include <cuda_runtime.h>
#include <stdint.h>

#include "engine_internal.h"
#include "reqlog_device.cuh"
#include "tile_common.cuh"

namespace gofr {

constexpr int LT = kServeThreads;
constexpr int LNW = LT / 32;
constexpr uint32_t kLogStage = 24 * 1024;  // bytes of record strings staged per tile (128 records × 192 B)

struct LogShared {
    uint64_t bar;
    uint32_t warp_sum[LNW];
    uint32_t warp_lo[LNW], warp_hi[LNW];
    unsigned long long tile_base;
    uint32_t in_lo, in_hi;
    uint32_t stage[GOFR_STAGE_WORDS * LT];
    __align__(16) uint8_t in[kLogStage + 32];
};

__global__ void __launch_bounds__(LT, 5) reqlog_kernel(const LogParams p) {
    __shared__ __align__(16) LogShared sh;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        mbar_init(&sh.bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    uint32_t parity = 0;
    for (uint32_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        const uint32_t i = tile * LT + tid;
        const bool valid = i < p.n;
        LogDesc d;
        memset(&d, 0, sizeof d);
        if (valid) {
            const uint4* q = (const uint4*)p.desc + (size_t)i * 3;
            uint4 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
            uint4* dd = (uint4*)&d;
            dd[0] = a; dd[1] = b; dd[2] = c;
        }
        const uint32_t rec_len = (uint32_t)d.method_len + d.ua_len + d.xff_len + d.remote_len + d.uri_len;

        // ---- the tile's arena byte range ----
        uint32_t lo = valid ? d.arena_off : 0xFFFFFFFFu, hi = valid ? d.arena_off + rec_len : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo = min(lo, __shfl_xor_sync(0xFFFFFFFFu, lo, o));
            hi = max(hi, __shfl_xor_sync(0xFFFFFFFFu, hi, o));
        }
        if (lane == 0) { sh.warp_lo[warp] = lo; sh.warp_hi[warp] = hi; }
        __syncthreads();  // also: every thread is done reading the previous tile's staged bytes
        if (tid == 0) {
            uint32_t l = sh.warp_lo[0], h = sh.warp_hi[0];
#pragma unroll
            for (int w = 1; w < LNW; w++) { l = min(l, sh.warp_lo[w]); h = max(h, sh.warp_hi[w]); }
            l &= ~15u;
            h = (h + 4u + 15u) & ~15u;  // the Writer may read the aligned word after a source's last byte
            sh.in_lo = l;
            sh.in_hi = h;
            if (h > l && h - l <= kLogStage) {
                mbar_expect_tx(&sh.bar, h - l);
                bulk_g2s(sh.in, p.arena + l, h - l, &sh.bar);
            }
        }
        __syncthreads();
        const uint32_t in_lo = sh.in_lo, in_hi = sh.in_hi;
        const bool staged = in_hi > in_lo && in_hi - in_lo <= kLogStage;
        const uint8_t* abase = p.arena;
        if (staged) {
            mbar_wait(&sh.bar, parity);
            parity ^= 1;
            abase = launder_after_sync((const uint8_t*)sh.in) - in_lo;
        }
        const uint8_t* rec = abase + d.arena_off;

        LogCtx c;
        c.ip_off = c.ip_len = c.esc_mask = c.total_len = 0;
        if (valid) reqlog_size(d, rec, staged, c);

        uint32_t incl = c.total_len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= (uint32_t)o) incl += v;
        }
        if (lane == 31) sh.warp_sum[warp] = incl;
        __syncthreads();
        uint32_t warp_excl = 0, tile_total = 0;
#pragma unroll
        for (int w = 0; w < LNW; w++) {
            uint32_t s = sh.warp_sum[w];
            if ((uint32_t)w < warp) warp_excl += s;
            tile_total += s;
        }
        const uint32_t excl = warp_excl + incl - c.total_len;
        if (warp == 0) {
            unsigned long long b = lookback(p.tile_state, p.epoch, tile, tile_total, lane);
            if (lane == 0) sh.tile_base = b;
        }
        __syncthreads();
        const unsigned long long tile_base = sh.tile_base;
        const bool fits = tile_base + tile_total <= p.out_cap && tile_base + tile_total <= 0xFFFFFFFFull;
        if (!fits && tid == 0) atomicExch(p.overflow, 1u);
        if (valid) {
            p.out_off[i] = (uint32_t)(tile_base + excl);
            if (i == p.n - 1) p.out_off[p.n] = (uint32_t)(tile_base + excl + c.total_len);
        }
        if (fits && valid) {
            const uint4 idv = __ldg((const uint4*)p.ids + i);
            const uint32_t id[4] = {idv.x, idv.y, idv.z, idv.w};
            reqlog_emit(d, rec, staged, id, c, p.out + tile_base + excl, &sh.stage[tid]);
        }
    }
}

int launch_reqlog(const LogParams& p, int grid, void* stream) {
    reqlog_kernel<<<grid, LT, 0, (cudaStream_t)stream>>>(p);
    return (int)cudaGetLastError();
}

int reqlog_max_grid(int device) { return occupancy_grid(reqlog_kernel, LT, 0, device); }

}  // namespace gofr
