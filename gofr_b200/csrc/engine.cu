// engine.cu — per-GPU execution context behind the C ABI (include/gofr_b200.h).
//
// Stands where net/http's conn.serve → router.ServeHTTP sits in the reference (pkg/gofr/httpServer.go:29-33): the
// caller hands over a batch of parsed requests and gets the response bytes back.  Two entry styles:
//   gofr_serve_device   — everything already in HBM; one fused launch on the caller's stream;
//   gofr_batch_submit/_wait — host buffers; the batch is cut into chunks that flow through a 3-deep
//                         H2D → kernel → D2H pipeline on the engine's own streams (copy engines overlap the kernel).
// There is no CPU fallback: without a CUDA device engine creation fails with GOFR_ERR_NO_DEVICE.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <functional>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/gofr_b200.h"
#include "engine_internal.h"
#include "table_format.h"

static thread_local char g_err[512];

void set_last_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

#define CUDA_TRY(expr)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            set_last_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return GOFR_ERR_CUDA;                                                            \
        }                                                                                    \
    } while (0)

using namespace gofr;

namespace {

constexpr int kSlots = 3;  // pipeline depth of the host-batch path

struct Slot {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    cudaEvent_t ev_h2d = nullptr, ev_served = nullptr, ev_egress = nullptr;  // streaming path
    bool egress_pending = false;
    // device buffers (grown on demand)
    void* d_desc = nullptr; void* d_ids = nullptr; uint8_t* d_arena = nullptr; uint8_t* d_out = nullptr;
    uint32_t* d_off = nullptr; uint32_t* d_meta = nullptr;
    unsigned long long* d_state = nullptr; uint32_t* d_flag = nullptr; uint32_t* d_bind = nullptr;
    size_t cap_n = 0, cap_arena = 0, cap_out = 0, cap_tiles = 0;
    // pinned staging for the tiny per-chunk read-backs
    uint32_t* h_tail = nullptr;  // [0] = chunk total bytes, [1] = overflow flag
};

}  // namespace

struct gofr_engine {
    int device = 0;
    int sm_count = 0;
    ImageHeader hdr;
    std::vector<uint32_t> schema_ids;  // the table's schema ids in table order
    std::vector<uint16_t> schema_flags;  // SchemaRec::flags, same order
    uint8_t* d_image = nullptr;
    uint32_t image_bytes = 0;
    // launch geometry
    uint32_t in_cap = 0, smem_bytes = 0;
    uint32_t w_in_cap = 0, w_smem_bytes = 0;  // the same for the wide slot-layout instance (4 CTAs/SM: a larger staging area fits)
    int wide_grid = 0, wide_blocks_per_sm = 0;
    bool slots_wide = false;  // choose_slot_residency
    bool has_values = false;  // some program has PF_VALUES: the packed layout runs serve_kernel_values (serve_values_kernel.cu)
    int grid = 0, blocks_per_sm = 0, grpc_grid = 0, reqlog_grid = 0, http_grid = 0, proto_grid = 0, proto_decode_grid = 0, proto_nested_grid = 0, proto_nested_decode_grid = 0;
    uint32_t epoch = 0;
    // resident path scratch
    unsigned long long* d_state = nullptr;
    size_t state_tiles = 0;
    uint32_t* d_flag = nullptr;
    uint32_t* d_bind = nullptr;  // Bind scratch of the resident path
    size_t bind_cap = 0;
    // host path
    Slot slots[kSlots];
    cudaStream_t st_h2d = nullptr, st_compute = nullptr, st_egress = nullptr;
    cudaEvent_t ev_batch_done = nullptr;  // blocking-sync event: the caller's thread SLEEPS until its batch is back (a
                                          // spinning cudaStreamSynchronize per rank burns the CPU quota eight ranks share)
    unsigned long long* d_chain = nullptr;  // packed position of the batch in flight
    ChunkInfo* d_info = nullptr;            // one per slot
    unsigned long long* h_status = nullptr; // pinned: [0] total bytes, [1] overflow
    int egress_grid = 37;
    uint32_t chunk = 65536;
    std::mutex mu;
    uint64_t launches = 0;
    // kernel timing (events on the launch stream)
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timing;
    bool timing_on = false;  // off by default: each timed launch costs two event objects (gofr_engine_set_timing)
    uint32_t debug_flags = 0;  // GOFR_DEBUG_* environment switches, read once at creation
    double timed_ms = 0;
    uint64_t timed_launches = 0;
    // gofr_batch_route scratch (host-buffer stage 1 of the split API)
    uint8_t* d_rt_desc = nullptr; uint8_t* d_rt_arena = nullptr; uint8_t* d_rt_meta = nullptr; uint8_t* d_rt_vars = nullptr;
    size_t rt_desc_cap = 0, rt_arena_cap = 0, rt_meta_cap = 0, rt_vars_cap = 0;
    uint8_t* d_rt_rows = nullptr;  // gofr_batch_bind: result slots
    size_t rt_rows_cap = 0;
    // tickets
    // tickets of finished submits whose result has not been collected yet (submit completes the batch; wait reports)
    std::vector<std::pair<gofr_ticket, int>> done_tickets;
    gofr_ticket next_ticket = 1;
};

// Engines alive per device in this process.  The packed-layout kernels chain their tiles with a look-back that is only
// deadlock free when every CTA of the grid is resident at once (tile t waits for tiles < t, all owned by resident CTAs).
// A grid sized for the whole GPU is not co-resident with a second engine's grid on the same device, so every engine
// launches its look-back kernels with the device's capacity divided by the number of live engines on it.  Other processes
// on the same GPU (MPS) are not visible from here: INTEGRATION.md says one serving process per GPU.
static std::mutex g_reg_mu;
static int g_live_engines[64];
static int engines_on_device(int device) {
    std::lock_guard<std::mutex> g(g_reg_mu);
    const int k = device >= 0 && device < 64 ? g_live_engines[device] : 1;
    return k > 0 ? k : 1;
}
static void register_engine(int device, int delta) {
    std::lock_guard<std::mutex> g(g_reg_mu);
    if (device >= 0 && device < 64) g_live_engines[device] += delta;
}

// Which slot-layout instance serves this table (serve_slots_kernel.cu): the 5-CTA one unless the wide one (4 CTAs/SM, 128
// registers) is asked for (GOFR_SLOT_CTAS=4, gofr_engine_slot_ctas).  For a short while the wide instance was the default
// for one-shape fast-path tables — it measured 4 % faster than the "5-CTA" instance on config 2 — until it turned out that
// the 5-CTA instances had been resident 4 per SM (DESIGN.md section 4e): with the fifth CTA back they are 7.5 % faster than
// the wide one on the same table (0.2737 against 0.2959 ms).
static bool choose_slot_residency() {
    if (const char* v = getenv("GOFR_SLOT_CTAS")) return atoi(v) == kServeCtasWide;
    return false;
}

// in_per_req / w_in_per_req: bytes of request staging per request for the 5-CTA instances / the wide slot-layout instance
static int configure_geometry(gofr_engine* e, uint32_t in_per_req, uint32_t w_in_per_req) {
    // the slot layout keeps its deferred-request list (2 T words) in the staging area
    if (in_per_req < 16u) in_per_req = 16u;
    if (w_in_per_req < 16u) w_in_per_req = 16u;
    e->in_cap = (kServeT * in_per_req + 127u) & ~127u;
    e->smem_bytes = serve_smem_bytes(e->hdr.hot_bytes, e->in_cap);
    e->w_in_cap = (kServeT * w_in_per_req + 127u) & ~127u;
    e->w_smem_bytes = serve_smem_bytes(e->hdr.hot_bytes, e->w_in_cap);
    if (e->smem_bytes > 227 * 1024 || e->w_smem_bytes > 227 * 1024) { set_last_error("tile geometry needs %u bytes of shared memory", std::max(e->smem_bytes, e->w_smem_bytes)); return GOFR_ERR_CAPACITY; }
    int g = serve_max_grid(e->smem_bytes, e->device, &e->blocks_per_sm, false);
    if (g <= 0) { set_last_error("serve kernel cannot be resident with %u bytes of shared memory", e->smem_bytes); return GOFR_ERR_CUDA; }
    e->grid = g;
    e->wide_grid = serve_max_grid(e->w_smem_bytes, e->device, &e->wide_blocks_per_sm, true);
    if (e->wide_grid < 0) e->wide_grid = 0;  // the wide instance is optional: the engine falls back to the others
    return GOFR_OK;
}

extern "C" {

static int engine_init(gofr_engine* e, const std::vector<uint8_t>& img, int device);

int gofr_engine_create(gofr_engine** out, const gofr_table* t, int device) {
    if (!out || !t) return GOFR_ERR_INVALID;
    const std::vector<uint8_t>& img = gofr_table_image(t);
    if (img.empty()) return GOFR_ERR_NOT_SEALED;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_last_error("no CUDA device: gofr_b200 has no CPU path");
        return GOFR_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= ndev) return GOFR_ERR_INVALID;
    CUDA_TRY(cudaSetDevice(device));
    gofr_engine* e = new gofr_engine();
    register_engine(device, +1);
    e->device = device;
    const int rc_create = engine_init(e, img, device);
    if (rc_create != GOFR_OK) { gofr_engine_destroy(e); return rc_create; }  // releases whatever the failed step left behind
    *out = e;
    return GOFR_OK;
}

static int engine_init(gofr_engine* e, const std::vector<uint8_t>& img, int device) {
    e->device = device;
    memcpy(&e->hdr, img.data(), sizeof(ImageHeader));
    e->schema_ids.resize(e->hdr.n_schemas);
    if (e->hdr.n_schemas) memcpy(e->schema_ids.data(), img.data() + e->hdr.schema_ids_off, (size_t)e->hdr.n_schemas * 4);
    e->schema_flags.resize(e->hdr.n_schemas);
    for (uint32_t k = 0; k < e->hdr.n_schemas; k++)
        e->schema_flags[k] = reinterpret_cast<const SchemaRec*>(img.data() + e->hdr.schemas_off)[k].flags;
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    e->sm_count = prop.multiProcessorCount;
    e->image_bytes = (uint32_t)img.size();
    CUDA_TRY(cudaMalloc(&e->d_image, img.size() + 64));
    CUDA_TRY(cudaMemcpy(e->d_image, img.data(), img.size(), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMalloc(&e->d_flag, 64));
    CUDA_TRY(cudaMemset(e->d_flag, 0, 64));
    // default tile geometry: as many request bytes per request staged in shared memory as still lets the instance keep
    // its CTAs per SM (5, or 4 for the wide slot-layout instance — the kernel is latency bound: residency matters more than
    // staging every tile; larger tiles are read from HBM directly).  The budget is found by asking the runtime's occupancy
    // calculator, not by a formula.
    uint32_t in_per = serve_fit_in_per(e->hdr.hot_bytes, kServeCtas, false);
    uint32_t w_in_per = serve_fit_in_per(e->hdr.hot_bytes, kServeCtasWide, true);
    if (in_per < 64u) in_per = 64u;    // a table this large: stage at least short requests, whatever residency is left
    if (w_in_per < in_per) w_in_per = in_per;
    int rc = configure_geometry(e, in_per, w_in_per);
    if (rc != GOFR_OK) return rc;
    e->slots_wide = choose_slot_residency();
    for (uint32_t k = 0; k < e->hdr.n_progs; k++)
        e->has_values |= (reinterpret_cast<const ProgRec*>(img.data() + e->hdr.progs_off)[k].flags & PF_VALUES) != 0;
    for (auto& s : e->slots) {
        CUDA_TRY(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
        CUDA_TRY(cudaMallocHost(&s.h_tail, 64));
        CUDA_TRY(cudaEventCreateWithFlags(&s.ev_h2d, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&s.ev_served, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&s.ev_egress, cudaEventDisableTiming));
    }
    CUDA_TRY(cudaStreamCreateWithFlags(&e->st_h2d, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&e->st_compute, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&e->st_egress, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&e->ev_batch_done, cudaEventBlockingSync | cudaEventDisableTiming));
    CUDA_TRY(cudaMalloc(&e->d_chain, 64));
    CUDA_TRY(cudaMalloc(&e->d_info, sizeof(ChunkInfo) * kSlots));
    CUDA_TRY(cudaMallocHost(&e->h_status, 64));
    if (const char* w = getenv("GOFR_DEBUG_EPOCH_START")) e->epoch = (uint32_t)strtoul(w, nullptr, 0) & kEpochMask;  // tests: start next to the wrap
    if (getenv("GOFR_DEBUG_NO_LOOKBACK")) e->debug_flags |= 1u;  // diagnostic only: offsets are wrong unless every response has the same size
    e->egress_grid = e->sm_count / 4 > 0 ? e->sm_count / 4 : 1;
    if (const char* g = getenv("GOFR_EGRESS_GRID")) { int v = atoi(g); if (v > 0) e->egress_grid = v; }
    return GOFR_OK;
}

void gofr_engine_destroy(gofr_engine* e) {
    if (!e) return;
    register_engine(e->device, -1);
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    for (auto& s : e->slots) {
        if (s.stream) cudaStreamDestroy(s.stream);
        if (s.done) cudaEventDestroy(s.done);
        if (s.ev_h2d) cudaEventDestroy(s.ev_h2d);
        if (s.ev_served) cudaEventDestroy(s.ev_served);
        if (s.ev_egress) cudaEventDestroy(s.ev_egress);
        cudaFree(s.d_desc); cudaFree(s.d_ids); cudaFree(s.d_arena); cudaFree(s.d_out); cudaFree(s.d_off); cudaFree(s.d_meta);
        cudaFree(s.d_state); cudaFree(s.d_flag); cudaFree(s.d_bind);
        if (s.h_tail) cudaFreeHost(s.h_tail);
    }
    for (auto& ev : e->timing) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    if (e->st_h2d) cudaStreamDestroy(e->st_h2d);
    if (e->st_compute) cudaStreamDestroy(e->st_compute);
    if (e->st_egress) cudaStreamDestroy(e->st_egress);
    if (e->ev_batch_done) cudaEventDestroy(e->ev_batch_done);
    cudaFree(e->d_chain); cudaFree(e->d_info);
    if (e->h_status) cudaFreeHost(e->h_status);
    cudaFree(e->d_image); cudaFree(e->d_state); cudaFree(e->d_flag); cudaFree(e->d_bind);
    cudaFree(e->d_rt_desc); cudaFree(e->d_rt_arena); cudaFree(e->d_rt_meta); cudaFree(e->d_rt_vars); cudaFree(e->d_rt_rows);
    delete e;
}

int gofr_engine_set_tile(gofr_engine* e, uint32_t in_bytes_per_req) {
    if (!e || !in_bytes_per_req) return GOFR_ERR_INVALID;
    std::lock_guard<std::mutex> g(e->mu);
    return configure_geometry(e, in_bytes_per_req, in_bytes_per_req);
}

int gofr_engine_set_chunk(gofr_engine* e, uint32_t requests_per_chunk) {
    if (!e || requests_per_chunk == 0) return GOFR_ERR_INVALID;
    std::lock_guard<std::mutex> g(e->mu);  // a batch in flight keeps the chunk size it started with
    e->chunk = requests_per_chunk;
    return GOFR_OK;
}

}  // extern "C"

// Called with the engine lock held before a timed launch: keeps the list of pending event pairs bounded when the
// caller never asks for the timings (finished pairs are folded into the totals; unfinished ones wait their turn).
static void fold_timing(gofr_engine* e) {
    if (e->timing.size() < 256) return;
    size_t k = 0;
    for (auto& ev : e->timing) {
        if (cudaEventQuery(ev.second) == cudaSuccess) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, ev.first, ev.second) == cudaSuccess) { e->timed_ms += ms; e->timed_launches++; }
            cudaEventDestroy(ev.first);
            cudaEventDestroy(ev.second);
        } else e->timing[k++] = ev;
    }
    e->timing.resize(k);
    cudaGetLastError();  // cudaEventQuery reports cudaErrorNotReady through the sticky-free last-error slot
}


// Look-back generation for the next launch.  State words written by older launches carry an older epoch and read as
// "not ready"; the epoch field is kEpochBits wide, so it wraps.  Every state buffer the engine owns is cleared when it
// does (after the device has drained), otherwise a word left by launch k would read as ready in launch k + 2^kEpochBits
// for a tile index that no launch in between has overwritten.  Called with the engine lock held.
static int next_epoch(gofr_engine* e, uint32_t* out) {
    uint32_t ep = (e->epoch + 1) & gofr::kEpochMask;
    if (ep == 0) {  // wrapped (epoch 0 is what zero-initialised words carry: never handed out)
        if (cudaDeviceSynchronize() != cudaSuccess) { set_last_error("device synchronisation failed at the look-back epoch wrap"); return GOFR_ERR_CUDA; }
        if (e->d_state && cudaMemset(e->d_state, 0, e->state_tiles * 8) != cudaSuccess) return GOFR_ERR_CUDA;
        for (auto& s : e->slots)
            if (s.d_state && cudaMemset(s.d_state, 0, ((s.cap_n + 63) / 64) * 8) != cudaSuccess) return GOFR_ERR_CUDA;
        ep = 1;
    }
    e->epoch = ep;
    *out = ep;
    return GOFR_OK;
}

// Look-back state of the resident calls for `tiles` tiles.  cudaFree synchronises, so no earlier launch still uses the
// old buffer.  Called with the engine lock held.
static int grow_state(gofr_engine* e, size_t tiles) {
    if (tiles <= e->state_tiles) return GOFR_OK;
    cudaFree(e->d_state);
    e->d_state = nullptr;
    e->state_tiles = 0;
    CUDA_TRY(cudaMalloc(&e->d_state, tiles * 8));
    CUDA_TRY(cudaMemset(e->d_state, 0, tiles * 8));
    e->state_tiles = tiles;
    return GOFR_OK;
}

// Bind scratch of the resident serve calls for n requests; nothing for a table without Bind-echo routes.
static int grow_bind(gofr_engine* e, uint32_t n) {
    const size_t need = (size_t)n * e->hdr.bind_row_words * 4;
    if (need <= e->bind_cap) return GOFR_OK;
    cudaFree(e->d_bind);
    e->d_bind = nullptr;
    e->bind_cap = 0;
    CUDA_TRY(cudaMalloc(&e->d_bind, need + need / 4 + 256));
    e->bind_cap = need + need / 4;
    return GOFR_OK;
}

// Grid of a look-back kernel: its resident grid shared with the other engines on the device (see engines_on_device),
// and no more CTAs than tiles.
static int lookback_grid(gofr_engine* e, int grid, size_t tiles) {
    return (int)std::min<size_t>((size_t)std::max(1, grid / engines_on_device(e->device)), tiles);
}

// A kernel's resident grid, asked from the occupancy calculator on first use.
static int lazy_grid(gofr_engine* e, int* grid, int (*max_grid)(int), const char* what) {
    if (*grid <= 0) {
        *grid = max_grid(e->device);
        if (*grid <= 0) { set_last_error("%s kernel cannot be resident", what); return GOFR_ERR_CUDA; }
    }
    return GOFR_OK;
}

// Enqueues one kernel on `st` through `launch` (returns a cudaError_t as int) and counts it.  A `timed` launch is bracketed
// by an event pair while timing is on (gofr_engine_kernel_time_ms).  Called with the engine lock held.
template <typename Launch>
static int run_launch(gofr_engine* e, const char* what, bool timed, cudaStream_t st, Launch&& launch) {
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    timed = timed && e->timing_on;
    if (timed) {
        fold_timing(e);
        CUDA_TRY(cudaEventCreate(&ev0));
        CUDA_TRY(cudaEventCreate(&ev1));
        CUDA_TRY(cudaEventRecord(ev0, st));
    }
    const int rc = launch();
    if (rc != 0) { set_last_error("%s kernel launch failed: %s", what, cudaGetErrorString((cudaError_t)rc)); return GOFR_ERR_CUDA; }
    if (timed) {
        CUDA_TRY(cudaEventRecord(ev1, st));
        e->timing.emplace_back(ev0, ev1);
    }
    e->launches++;
    return GOFR_OK;
}

// Start of a frame-style call (gRPC, proto, request log), engine lock held.  An empty batch only gets out_off[0] = 0;
// otherwise the look-back state grows to the batch's tiles and p receives the fields every frame kernel shares.
template <typename Params>
static int frame_prologue(gofr_engine* e, uint32_t n, uint8_t* d_out, uint64_t out_cap, uint32_t* d_out_off, cudaStream_t st,
                          Params* p) {
    memset(p, 0, sizeof *p);
    if (n == 0) {
        if (d_out_off) CUDA_TRY(cudaMemsetAsync(d_out_off, 0, 4, st));
        return GOFR_OK;
    }
    p->n = n;
    p->n_tiles = (n + kServeThreads - 1) / kServeThreads;
    { int rc = grow_state(e, p->n_tiles); if (rc) return rc; }
    { int rc = next_epoch(e, &p->epoch); if (rc) return rc; }
    p->out = d_out; p->out_cap = out_cap; p->out_off = d_out_off;
    p->tile_state = e->d_state; p->overflow = e->d_flag;
    return GOFR_OK;
}

// one fused launch; `state`/`flag` are scratch owned by the caller of this helper
static int launch_one(gofr_engine* e, const void* d_desc, const void* d_ids, const uint8_t* d_arena, uint32_t n,
                      const char* date29, uint8_t* d_out, uint64_t out_cap, uint32_t* d_off, uint32_t* d_meta,
                      unsigned long long* d_state, uint32_t* d_flag, uint32_t* d_bind, cudaStream_t stream,
                      const unsigned long long* chain_pos = nullptr, uint32_t slot_bytes = 0) {
    ServeParams p;
    memset(&p, 0, sizeof p);
    p.desc = d_desc; p.ids = d_ids; p.arena = d_arena; p.n = n;
    p.n_tiles = (n + kServeT - 1) / kServeT;
    p.image = e->d_image; p.hot_bytes = e->hdr.hot_bytes;
    { int erc = next_epoch(e, &p.epoch); if (erc) return erc; }
    p.out = d_out; p.out_cap = out_cap; p.out_off = d_off; p.meta = d_meta;
    p.tile_state = d_state; p.overflow = d_flag;
    const bool wide = slot_bytes && e->slots_wide && !e->has_values && e->wide_grid > 0;
    p.in_cap = wide ? e->w_in_cap : e->in_cap;
    p.bind_scratch = d_bind; p.bind_row_words = e->hdr.bind_row_words;
    p.chain_pos = chain_pos;
    p.slot_bytes = slot_bytes;
    p.debug_flags = e->debug_flags;
    memcpy(p.date, date29, 29);
    const int grid = slot_bytes ? (int)std::min<uint32_t>((uint32_t)(wide ? e->wide_grid : e->grid), p.n_tiles)
                                : lookback_grid(e, e->grid, p.n_tiles);
    return run_launch(e, "serve", true, stream, [&] {
        return launch_serve(p, grid, wide ? e->w_smem_bytes : e->smem_bytes, stream, wide, e->has_values);
    });
}

extern "C" {

int gofr_serve_device(gofr_engine* e, const gofr_req_desc* d_desc, const uint8_t* d_trace_ids, const uint8_t* d_arena,
                      uint32_t n, const char* date29, uint8_t* d_out, uint64_t out_cap, uint32_t* d_out_off,
                      uint32_t* d_meta, void* stream) {
    if (!e || !date29 || (n && (!d_desc || !d_trace_ids || !d_out || !d_out_off || !d_meta))) return GOFR_ERR_INVALID;
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) {
        if (d_out_off) CUDA_TRY(cudaMemsetAsync(d_out_off, 0, 4, st));
        return GOFR_OK;
    }
    { int rc = grow_state(e, (n + 63) / 64); if (rc) return rc; }  // enough for any tile size in use (serve: kServeT, gRPC / log: 128)
    { int rc = grow_bind(e, n); if (rc) return rc; }
    return launch_one(e, d_desc, d_trace_ids, d_arena, n, date29, d_out, out_cap, d_out_off, d_meta, e->d_state, e->d_flag,
                      e->d_bind, st);
}

int gofr_serve_device_slots(gofr_engine* e, const gofr_req_desc* d_desc, const uint8_t* d_trace_ids, const uint8_t* d_arena,
                            uint32_t n, const char* date29, uint8_t* d_out, uint32_t slot_bytes, uint32_t* d_out_len,
                            uint32_t* d_meta, void* stream) {
    if (!e || !date29 || (n && (!d_desc || !d_trace_ids || !d_out || !d_out_len || !d_meta))) return GOFR_ERR_INVALID;
    if (slot_bytes == 0 || (slot_bytes & 15u) || ((uintptr_t)d_out & 15u)) {
        set_last_error("slot_bytes must be a positive multiple of 16 and d_out 16-byte aligned");
        return GOFR_ERR_INVALID;
    }
    if (n == 0) return GOFR_OK;
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    { int rc = grow_bind(e, n); if (rc) return rc; }
    // no look-back scratch: slots make the tiles independent of each other
    return launch_one(e, d_desc, d_trace_ids, d_arena, n, date29, d_out, (uint64_t)n * slot_bytes, d_out_len, d_meta, nullptr,
                      e->d_flag, e->d_bind, (cudaStream_t)stream, nullptr, slot_bytes);
}

int gofr_engine_overflowed(gofr_engine* e, int* flag_out, int reset) {
    if (!e || !flag_out) return GOFR_ERR_INVALID;
    uint32_t f = 0;
    CUDA_TRY(cudaSetDevice(e->device));
    CUDA_TRY(cudaMemcpy(&f, e->d_flag, 4, cudaMemcpyDeviceToHost));
    if (reset && f) CUDA_TRY(cudaMemset(e->d_flag, 0, 4));
    *flag_out = (int)f;
    return GOFR_OK;
}

uint64_t gofr_engine_launch_count(const gofr_engine* e) { return e ? e->launches : 0; }

int gofr_engine_kernel_time_ms(gofr_engine* e, double* total_ms, uint64_t* launches, int reset) {
    if (!e) return GOFR_ERR_INVALID;
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    for (auto& ev : e->timing) {
        CUDA_TRY(cudaEventSynchronize(ev.second));
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, ev.first, ev.second));
        e->timed_ms += ms;
        e->timed_launches++;
        cudaEventDestroy(ev.first);
        cudaEventDestroy(ev.second);
    }
    e->timing.clear();
    if (total_ms) *total_ms = e->timed_ms;
    if (launches) *launches = e->timed_launches;
    if (reset) { e->timed_ms = 0; e->timed_launches = 0; }
    return GOFR_OK;
}

int gofr_engine_set_timing(gofr_engine* e, int on) {
    if (!e) return GOFR_ERR_INVALID;
    std::lock_guard<std::mutex> g(e->mu);
    e->timing_on = on != 0;
    return GOFR_OK;
}

int gofr_engine_geometry(const gofr_engine* e, uint32_t* grid, uint32_t* blocks_per_sm, uint32_t* smem_bytes,
                         uint32_t* sm_count) {
    if (!e) return GOFR_ERR_INVALID;
    if (grid) *grid = (uint32_t)e->grid;
    if (blocks_per_sm) *blocks_per_sm = (uint32_t)e->blocks_per_sm;
    if (smem_bytes) *smem_bytes = e->smem_bytes;
    if (sm_count) *sm_count = (uint32_t)e->sm_count;
    return GOFR_OK;
}

int gofr_engine_slot_ctas(gofr_engine* e, int ctas_per_sm, int* in_effect) {
    if (!e) return GOFR_ERR_INVALID;
    std::lock_guard<std::mutex> g(e->mu);
    if (ctas_per_sm == kServeCtasWide) e->slots_wide = true;
    else if (ctas_per_sm == kServeCtas) e->slots_wide = false;
    else if (ctas_per_sm != 0) return GOFR_ERR_INVALID;
    if (in_effect) *in_effect = e->slots_wide && !e->has_values && e->wide_grid > 0 ? kServeCtasWide : kServeCtas;
    return GOFR_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// host-batch path
// ---------------------------------------------------------------------------------------------------------------

static int grow(void** p, size_t* cap, size_t need, size_t slack) {
    if (need <= *cap) return GOFR_OK;
    cudaFree(*p);
    *p = nullptr;
    size_t c = need + need / 4 + slack;
    cudaError_t er = cudaMalloc(p, c);
    if (er != cudaSuccess) { set_last_error("cudaMalloc(%zu) failed: %s", c, cudaGetErrorString(er)); *cap = 0; return GOFR_ERR_NOMEM; }
    *cap = c;
    return GOFR_OK;
}

// The copy loops read their source in whole aligned words: up to 16 bytes past the last byte a request names may be touched
// (include/gofr_b200.h states the same for device-resident callers), so a staging arena is never sized to the byte.
static constexpr size_t kArenaSlack = 16;

// A chunk = contiguous request range [lo, hi) and the arena byte range [arena_lo, arena_hi) (16-byte granular) it covers.
struct ChunkPlan {
    uint32_t lo, hi;
    uint32_t arena_lo, arena_hi;
    size_t abytes() const { return (size_t)arena_hi - arena_lo; }
};

// Chunk ci of a host batch (e->chunk requests each) and the arena bytes its requests reference: up to the end of each
// request's data, or with path_only up to the end of its path (routing reads nothing else).  All arithmetic in 64 bits: a
// descriptor with a huge arena_off or data_len (say a data_len taken from a Content-Length header) must be refused, not
// wrap around and pass.
static int chunk_arena_range(const gofr_engine* e, const gofr_req_batch* in, size_t ci, bool path_only, ChunkPlan* c) {
    const uint32_t lo = (uint32_t)(ci * e->chunk), hi = (uint32_t)std::min<uint64_t>(in->n, (uint64_t)lo + e->chunk);
    uint64_t alo = ~0ull, ahi = 0;
    const gofr_req_desc* dd = in->desc;
    for (uint32_t i = lo; i < hi; i++) {
        const uint64_t a = dd[i].arena_off;
        const uint64_t end = path_only ? a + dd[i].path_len : ((a + dd[i].path_len + dd[i].query_len + 3u) & ~3ull) + dd[i].data_len;
        alo = a < alo ? a : alo;
        ahi = end > ahi ? end : ahi;
    }
    if (hi <= lo) alo = 0;
    alo &= ~15ull;
    ahi = (ahi + 15ull) & ~15ull;
    if (ahi > (((uint64_t)in->arena_bytes + 15ull) & ~15ull) || ahi > 0xFFFFFFF0ull) {
        set_last_error("a descriptor of requests %u..%u points outside the arena", lo, hi);
        return GOFR_ERR_INVALID;
    }
    if (ahi > alo && !in->arena) { set_last_error("requests reference arena bytes but the batch has no arena"); return GOFR_ERR_INVALID; }
    *c = {lo, hi, (uint32_t)alo, (uint32_t)(ahi > alo ? ahi : alo)};
    return GOFR_OK;
}

// Copies the chunk's arena bytes to dst.  The range is rounded out to 16 bytes, so its end may lie past the caller's arena.
static int stage_arena(const gofr_req_batch* in, const ChunkPlan& c, uint8_t* dst, cudaStream_t st) {
    if (!c.abytes()) return GOFR_OK;
    const size_t avail = in->arena_bytes > c.arena_lo ? (size_t)in->arena_bytes - c.arena_lo : 0;
    CUDA_TRY(cudaMemcpyAsync(dst, in->arena + c.arena_lo, std::min(c.abytes(), avail), cudaMemcpyHostToDevice, st));
    return GOFR_OK;
}

// Device output buffer of a packed chunk: the fixed part of every response plus what its data bytes can expand to.
static size_t packed_out_cap(const gofr_engine* e, uint32_t cn, size_t abytes) {
    return std::min<size_t>((size_t)cn * (e->hdr.max_fixed_len + 64) + (size_t)image_data_expand(e->hdr) * abytes + 4096, 0xFFFFFFF0ull);
}

// Grows slot s for a chunk of cn requests, abytes of arena and obytes of output.  No earlier chunk may still use its
// buffers (wait_slot_egress, or a synchronised slot stream).
static int reserve_slot(gofr_engine* e, Slot& s, uint32_t cn, size_t abytes, size_t obytes) {
    if (cn > s.cap_n) {
        cudaFree(s.d_desc); cudaFree(s.d_ids); cudaFree(s.d_off); cudaFree(s.d_meta); cudaFree(s.d_state); cudaFree(s.d_bind);
        s.d_desc = s.d_ids = nullptr; s.d_off = s.d_meta = nullptr; s.d_state = nullptr; s.d_bind = nullptr;
        s.cap_n = 0;
        const size_t c = (size_t)cn + cn / 4 + 256, tiles = (c + 63) / 64;
        if (cudaMalloc(&s.d_desc, c * 16) != cudaSuccess || cudaMalloc(&s.d_ids, c * 16) != cudaSuccess ||
            cudaMalloc(&s.d_off, (c + 1) * 4) != cudaSuccess || cudaMalloc(&s.d_meta, c * 4) != cudaSuccess ||
            cudaMalloc(&s.d_state, tiles * 8) != cudaSuccess) { set_last_error("cudaMalloc failed for a %zu-request chunk", c); return GOFR_ERR_NOMEM; }
        if (cudaMemset(s.d_state, 0, tiles * 8) != cudaSuccess) return GOFR_ERR_CUDA;
        if (e->hdr.bind_row_words && cudaMalloc(&s.d_bind, c * e->hdr.bind_row_words * 4 + 256) != cudaSuccess) { set_last_error("cudaMalloc failed for Bind scratch"); return GOFR_ERR_NOMEM; }
        s.cap_n = c;
    }
    if (!s.d_flag) { if (cudaMalloc(&s.d_flag, 64) != cudaSuccess || cudaMemset(s.d_flag, 0, 64) != cudaSuccess) return GOFR_ERR_NOMEM; }
    int rc;
    if ((rc = grow((void**)&s.d_arena, &s.cap_arena, abytes + kArenaSlack, 256))) return rc;
    return grow((void**)&s.d_out, &s.cap_out, obytes, 256);
}

// The slot's previous chunk must have left before its buffers are overwritten: a wait on the copy stream, unless the
// buffers have to grow (cudaFree needs the host to be sure).
static int wait_slot_egress(gofr_engine* e, Slot& s, uint32_t cn, size_t abytes, size_t obytes) {
    if (!s.egress_pending) return GOFR_OK;
    if (cn > s.cap_n || abytes + kArenaSlack > s.cap_arena || obytes > s.cap_out) CUDA_TRY(cudaEventSynchronize(s.ev_egress));
    else CUDA_TRY(cudaStreamWaitEvent(e->st_h2d, s.ev_egress, 0));
    s.egress_pending = false;
    return GOFR_OK;
}

// Waits for everything enqueued on the egress stream.  A large batch takes milliseconds: the thread sleeps on a
// blocking-sync event.  A small one (the per-request front-end's batches) is back in tens of microseconds: spinning is
// the faster wake-up there.
static cudaError_t wait_batch(gofr_engine* e, uint32_t n) {
    if (n < 16384u) return cudaStreamSynchronize(e->st_egress);
    cudaError_t er = cudaEventRecord(e->ev_batch_done, e->st_egress);
    return er != cudaSuccess ? er : cudaEventSynchronize(e->ev_batch_done);
}

// Error exit of a host-batch call after work has been enqueued: earlier chunks' kernels and copies may still be
// writing into the caller's buffers, which the caller is free to release once we return.
static void drain_streams(gofr_engine* e) {
    cudaStreamSynchronize(e->st_h2d);
    cudaStreamSynchronize(e->st_compute);
    cudaStreamSynchronize(e->st_egress);
    for (auto& s : e->slots) { if (s.stream) cudaStreamSynchronize(s.stream); s.egress_pending = false; }
    cudaGetLastError();
}

static int batch_submit_locked(gofr_engine* e, const gofr_req_batch* in, gofr_resp_batch* out, gofr_ticket* ticket);
static int batch_submit_slots_locked(gofr_engine* e, const gofr_req_batch* in, gofr_slot_batch* out, gofr_ticket* ticket);

int gofr_batch_submit(gofr_engine* e, const gofr_req_batch* in, gofr_resp_batch* out, gofr_ticket* ticket) {
    if (!e || !in || !out || !ticket) return GOFR_ERR_INVALID;
    if (in->n && (!in->desc || !in->trace_ids || !out->out || !out->out_off || !out->meta)) return GOFR_ERR_INVALID;
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    // Descriptors are validated chunk by chunk as the batch is enqueued (an up-front scan of 1 Mi descriptors is
    // milliseconds of pure latency), so an error can surface with earlier chunks in flight: nothing may still be
    // writing into the caller's buffers when the error is returned.
    const int rc = batch_submit_locked(e, in, out, ticket);
    if (rc != GOFR_OK) drain_streams(e);
    return rc;
}

static int batch_submit_locked(gofr_engine* e, const gofr_req_batch* in, gofr_resp_batch* out, gofr_ticket* ticket) {
    out->out_bytes = 0;
    const uint32_t n = in->n;
    int final_rc = GOFR_OK;
    if (n == 0) {  // nothing to do; the caller may have passed no buffers at all
        if (out->out_off) out->out_off[0] = 0;
        *ticket = e->next_ticket++;
        e->done_tickets.emplace_back(*ticket, GOFR_OK);
        return GOFR_OK;
    }

    // Chunks are contiguous request ranges; a chunk's arena range is the min/max over its descriptors.  The scan is done
    // right before a chunk is enqueued, so it overlaps with the GPU work of the chunks already in flight (scanning all
    // descriptors up front costs milliseconds of pure latency on a 1 Mi-request batch).
    const size_t nchunks = ((size_t)n + e->chunk - 1) / e->chunk;
    // ---- streaming path: caller buffers are pinned → egress is device driven, the host never blocks mid-batch ----
    auto device_visible = [](const void* p) {
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
        return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
    };
    if (device_visible(out->out) && device_visible(out->out_off) && device_visible(out->meta)) {
        // growing buffers frees memory: make sure nothing from an earlier batch is still using them
        CUDA_TRY(cudaMemsetAsync(e->d_chain, 0, 8, e->st_compute));
        e->h_status[0] = 0; e->h_status[1] = 0;
        for (size_t ci = 0; ci < nchunks; ci++) {
            Slot& s = e->slots[ci % kSlots];
            ChunkInfo* info = e->d_info + ci % kSlots;
            ChunkPlan c;
            int rc = chunk_arena_range(e, in, ci, false, &c);
            if (rc) return rc;
            const uint32_t cn = c.hi - c.lo;
            const size_t ocap = packed_out_cap(e, cn, c.abytes());
            if ((rc = wait_slot_egress(e, s, cn, c.abytes(), ocap))) return rc;
            if ((rc = reserve_slot(e, s, cn, c.abytes(), ocap))) return rc;
            CUDA_TRY(cudaMemcpyAsync(s.d_desc, in->desc + c.lo, (size_t)cn * 16, cudaMemcpyHostToDevice, e->st_h2d));
            CUDA_TRY(cudaMemcpyAsync(s.d_ids, in->trace_ids + (size_t)c.lo * 16, (size_t)cn * 16, cudaMemcpyHostToDevice, e->st_h2d));
            if ((rc = stage_arena(in, c, s.d_arena, e->st_h2d))) return rc;
            CUDA_TRY(cudaEventRecord(s.ev_h2d, e->st_h2d));
            CUDA_TRY(cudaStreamWaitEvent(e->st_compute, s.ev_h2d, 0));
            rc = launch_one(e, s.d_desc, s.d_ids, s.d_arena - c.arena_lo, cn, in->date, s.d_out, s.cap_out, s.d_off, s.d_meta,
                            s.d_state, s.d_flag, s.d_bind, e->st_compute, e->d_chain);
            if (rc) return rc;
            rc = run_launch(e, "advance", false, e->st_compute, [&] {
                return launch_advance(e->d_chain, s.d_off, cn, s.d_flag, info, out->out_cap, e->st_compute);
            });
            if (rc) return rc;
            CUDA_TRY(cudaEventRecord(s.ev_served, e->st_compute));
            CUDA_TRY(cudaStreamWaitEvent(e->st_egress, s.ev_served, 0));
            rc = run_launch(e, "egress", false, e->st_egress, [&] {
                return launch_egress(info, s.d_out, s.d_off, s.d_meta, cn, out->out, out->out_off + c.lo, out->meta + c.lo,
                                     e->h_status, e->egress_grid, e->st_egress);
            });
            if (rc) return rc;
            CUDA_TRY(cudaEventRecord(s.ev_egress, e->st_egress));
            s.egress_pending = true;
        }
        CUDA_TRY(cudaMemcpyAsync((void*)&e->h_status[0], e->d_chain, 8, cudaMemcpyDeviceToHost, e->st_egress));
        CUDA_TRY(wait_batch(e, n));
        for (auto& s : e->slots) s.egress_pending = false;
        uint64_t total = e->h_status[0];
        if (e->h_status[1]) { final_rc = GOFR_ERR_CAPACITY; set_last_error("output capacity too small (device chunk buffer or caller buffer)"); }
        out->out_off[n] = (uint32_t)total;
        out->out_bytes = total;
        *ticket = e->next_ticket++;
        e->done_tickets.emplace_back(*ticket, final_rc);
        return GOFR_OK;
    }

    // ---- straightforward 3-slot software pipeline ----
    ChunkPlan plan[kSlots];  // the chunk each slot holds
    size_t issued = 0, finished = 0;
    uint64_t write_pos = 0;
    // issue order == completion order == chunk order; out offsets are rebased on the host as chunks complete
    while (finished < nchunks) {
        // keep up to kSlots chunks in flight
        while (issued < nchunks && issued - finished < (size_t)kSlots) {
            Slot& s = e->slots[issued % kSlots];
            ChunkPlan& c = plan[issued % kSlots];
            int rc = chunk_arena_range(e, in, issued, false, &c);
            if (rc) return rc;
            const uint32_t cn = c.hi - c.lo;
            if ((rc = reserve_slot(e, s, cn, c.abytes(), packed_out_cap(e, cn, c.abytes())))) return rc;
            CUDA_TRY(cudaMemcpyAsync(s.d_desc, in->desc + c.lo, (size_t)cn * 16, cudaMemcpyHostToDevice, s.stream));
            CUDA_TRY(cudaMemcpyAsync(s.d_ids, in->trace_ids + (size_t)c.lo * 16, (size_t)cn * 16, cudaMemcpyHostToDevice, s.stream));
            if ((rc = stage_arena(in, c, s.d_arena, s.stream))) return rc;
            // descriptors keep absolute arena offsets: pass a rebased arena pointer
            rc = launch_one(e, s.d_desc, s.d_ids, s.d_arena - c.arena_lo, cn, in->date, s.d_out, s.cap_out, s.d_off, s.d_meta,
                            s.d_state, s.d_flag, s.d_bind, s.stream);
            if (rc) return rc;
            CUDA_TRY(cudaMemcpyAsync(out->out_off + c.lo, s.d_off, (size_t)cn * 4, cudaMemcpyDeviceToHost, s.stream));
            CUDA_TRY(cudaMemcpyAsync(out->meta + c.lo, s.d_meta, (size_t)cn * 4, cudaMemcpyDeviceToHost, s.stream));
            CUDA_TRY(cudaMemcpyAsync(&s.h_tail[0], s.d_off + cn, 4, cudaMemcpyDeviceToHost, s.stream));
            CUDA_TRY(cudaMemcpyAsync(&s.h_tail[1], s.d_flag, 4, cudaMemcpyDeviceToHost, s.stream));
            CUDA_TRY(cudaEventRecord(s.done, s.stream));
            issued++;
        }
        // retire the oldest chunk: learn its size, then pull exactly that many bytes
        Slot& s = e->slots[finished % kSlots];
        const ChunkPlan& c = plan[finished % kSlots];
        CUDA_TRY(cudaEventSynchronize(s.done));
        uint32_t total = s.h_tail[0];
        if (s.h_tail[1]) { CUDA_TRY(cudaMemsetAsync(s.d_flag, 0, 4, s.stream)); final_rc = GOFR_ERR_CAPACITY; set_last_error("device output buffer too small for chunk %zu", finished); total = 0; }
        if (write_pos + total > out->out_cap) { final_rc = GOFR_ERR_CAPACITY; set_last_error("output capacity %llu too small", (unsigned long long)out->out_cap); total = 0; }
        if (total) CUDA_TRY(cudaMemcpyAsync(out->out + write_pos, s.d_out, total, cudaMemcpyDeviceToHost, s.stream));
        // rebase this chunk's offsets while the copy runs
        if (write_pos) for (uint32_t i = c.lo; i < c.hi; i++) out->out_off[i] += (uint32_t)write_pos;
        CUDA_TRY(cudaStreamSynchronize(s.stream));
        write_pos += total;
        finished++;
    }
    out->out_off[n] = (uint32_t)write_pos;
    out->out_bytes = write_pos;
    *ticket = e->next_ticket++;
    e->done_tickets.emplace_back(*ticket, final_rc);
    return GOFR_OK;
}

int gofr_batch_submit_slots(gofr_engine* e, const gofr_req_batch* in, gofr_slot_batch* out, gofr_ticket* ticket) {
    if (!e || !in || !out || !ticket) return GOFR_ERR_INVALID;
    if (in->n && (!in->desc || !in->trace_ids || !out->out || !out->out_len || !out->meta)) return GOFR_ERR_INVALID;
    if (out->slot_bytes == 0 || (out->slot_bytes & 15u)) { set_last_error("slot_bytes must be a positive multiple of 16"); return GOFR_ERR_INVALID; }
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    const int rc = batch_submit_slots_locked(e, in, out, ticket);
    if (rc != GOFR_OK) drain_streams(e);  // see gofr_batch_submit
    return rc;
}

static int batch_submit_slots_locked(gofr_engine* e, const gofr_req_batch* in, gofr_slot_batch* out, gofr_ticket* ticket) {
    const uint32_t n = in->n, slot = out->slot_bytes;
    int final_rc = GOFR_OK;
    const size_t nchunks = ((size_t)n + e->chunk - 1) / e->chunk;
    for (size_t ci = 0; ci < nchunks; ci++) {
        Slot& s = e->slots[ci % kSlots];
        // the chunk's request range and the arena bytes it covers (scanned right before the chunk is enqueued)
        ChunkPlan c;
        int rc = chunk_arena_range(e, in, ci, false, &c);
        if (rc) return rc;
        const uint32_t lo = c.lo, cn = c.hi - c.lo;
        const size_t obytes = (size_t)cn * slot;
        if ((rc = wait_slot_egress(e, s, cn, c.abytes(), obytes))) return rc;
        if ((rc = reserve_slot(e, s, cn, c.abytes(), obytes))) return rc;
        CUDA_TRY(cudaMemcpyAsync(s.d_desc, in->desc + lo, (size_t)cn * 16, cudaMemcpyHostToDevice, e->st_h2d));
        CUDA_TRY(cudaMemcpyAsync(s.d_ids, in->trace_ids + (size_t)lo * 16, (size_t)cn * 16, cudaMemcpyHostToDevice, e->st_h2d));
        if ((rc = stage_arena(in, c, s.d_arena, e->st_h2d))) return rc;
        CUDA_TRY(cudaEventRecord(s.ev_h2d, e->st_h2d));
        CUDA_TRY(cudaStreamWaitEvent(e->st_compute, s.ev_h2d, 0));
        rc = launch_one(e, s.d_desc, s.d_ids, s.d_arena - c.arena_lo, cn, in->date, s.d_out, obytes, s.d_off, s.d_meta, s.d_state,
                        s.d_flag, s.d_bind, e->st_compute, nullptr, slot);
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(s.ev_served, e->st_compute));
        CUDA_TRY(cudaStreamWaitEvent(e->st_egress, s.ev_served, 0));
        CUDA_TRY(cudaMemcpyAsync(out->out + (size_t)lo * slot, s.d_out, obytes, cudaMemcpyDeviceToHost, e->st_egress));
        CUDA_TRY(cudaMemcpyAsync(out->out_len + lo, s.d_off, (size_t)cn * 4, cudaMemcpyDeviceToHost, e->st_egress));
        CUDA_TRY(cudaMemcpyAsync(out->meta + lo, s.d_meta, (size_t)cn * 4, cudaMemcpyDeviceToHost, e->st_egress));
        CUDA_TRY(cudaEventRecord(s.ev_egress, e->st_egress));
        s.egress_pending = true;
    }
    if (nchunks) {
        CUDA_TRY(wait_batch(e, n));
        for (auto& s : e->slots) s.egress_pending = false;
    }
    *ticket = e->next_ticket++;
    e->done_tickets.emplace_back(*ticket, final_rc);
    return GOFR_OK;
}

int gofr_batch_wait(gofr_engine* e, gofr_ticket ticket) {
    if (!e || ticket == 0) return GOFR_ERR_INVALID;
    std::lock_guard<std::mutex> g(e->mu);
    for (size_t k = 0; k < e->done_tickets.size(); k++) {
        if (e->done_tickets[k].first != ticket) continue;
        int rc = e->done_tickets[k].second;
        e->done_tickets.erase(e->done_tickets.begin() + (long)k);
        return rc;
    }
    return GOFR_ERR_INVALID;  // unknown ticket, or already waited for
}

// Parses a sysfs cpu list ("0-31,64-95") into a cpu_set_t; returns the number of CPUs.
static int parse_cpulist(const char* s, cpu_set_t* set) {
    CPU_ZERO(set);
    int count = 0;
    while (*s) {
        char* end = nullptr;
        long a = strtol(s, &end, 10);
        if (end == s) break;
        long b = a;
        if (*end == '-') { s = end + 1; b = strtol(s, &end, 10); }
        for (long c = a; c <= b && c < CPU_SETSIZE; c++) { CPU_SET((int)c, set); count++; }
        s = *end == ',' ? end + 1 : end;
        if (*end != ',') break;
    }
    return count;
}

int gofr_bind_host_thread(int device, int* numa_node_out) {
    if (numa_node_out) *numa_node_out = -1;
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, (int)sizeof bus, device) != cudaSuccess) { cudaGetLastError(); set_last_error("no PCI bus id for device %d", device); return GOFR_ERR_CUDA; }
    for (char* c = bus; *c; c++) if (*c >= 'A' && *c <= 'Z') *c = (char)(*c + 32);  // sysfs names are lower case
    auto read_line = [](const std::string& path, char* buf, size_t cap) -> bool {
        FILE* f = fopen(path.c_str(), "r");
        if (!f) return false;
        const bool ok = fgets(buf, (int)cap, f) != nullptr;
        fclose(f);
        return ok;
    };
    const std::string base = std::string("/sys/bus/pci/devices/") + bus + "/";
    char line[4096];
    int node = -1;
    if (read_line(base + "numa_node", line, sizeof line)) node = atoi(line);
    if (numa_node_out) *numa_node_out = node;
    cpu_set_t set;
    int ncpu = 0;
    if (node >= 0 && read_line("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist", line, sizeof line)) ncpu = parse_cpulist(line, &set);
    if (!ncpu && read_line(base + "local_cpulist", line, sizeof line)) ncpu = parse_cpulist(line, &set);
    if (!ncpu) { set_last_error("no NUMA information for device %d (%s)", device, bus); return GOFR_ERR_UNSUPPORTED; }
    // stay inside what the container allows
    cpu_set_t cur;
    if (sched_getaffinity(0, sizeof cur, &cur) == 0) {
        cpu_set_t both;
        CPU_AND(&both, &set, &cur);
        if (CPU_COUNT(&both) > 0) set = both;
    }
    if (sched_setaffinity(0, sizeof set, &set) != 0) { set_last_error("sched_setaffinity failed for device %d", device); return GOFR_ERR_UNSUPPORTED; }
#if defined(SYS_set_mempolicy)
    if (node >= 0 && node < 64) {  // MPOL_PREFERRED: pages this thread touches (pinned allocations included) come from the GPU's node
        unsigned long mask = 1ul << node;
        syscall(SYS_set_mempolicy, 1 /*MPOL_PREFERRED*/, &mask, 65ul);
    }
#endif
    return GOFR_OK;
}

void* gofr_alloc_pinned(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { set_last_error("cudaMallocHost(%zu) failed", bytes); return nullptr; }
    return p;
}
void gofr_free_pinned(void* p) { if (p) cudaFreeHost(p); }

const char* gofr_last_error(void) { return g_err; }
uint32_t gofr_abi_version(void) { return GOFR_ABI_VERSION; }

void gofr_format_http_date(int64_t unix_seconds, char out29[29]) {
    static const char* days[] = {"Sun", "Mon", "Tue", "Wed", "Thu", "Fri", "Sat"};
    static const char* mons[] = {"Jan", "Feb", "Mar", "Apr", "May", "Jun", "Jul", "Aug", "Sep", "Oct", "Nov", "Dec"};
    time_t tt = (time_t)unix_seconds;
    struct tm g;
    gmtime_r(&tt, &g);
    char tmp[48];
    snprintf(tmp, sizeof tmp, "%s, %02d %s %04d %02d:%02d:%02d GMT", days[g.tm_wday], g.tm_mday, mons[g.tm_mon],
             g.tm_year + 1900, g.tm_hour, g.tm_min, g.tm_sec);
    memcpy(out29, tmp, 29);
}

int gofr_grpc_hello_device(gofr_engine* e, const uint8_t* d_in, const uint32_t* d_in_off, uint32_t n, uint8_t* d_out,
                           uint64_t out_cap, uint32_t* d_out_off, uint32_t* d_meta, void* stream) {
    if (!e || (n && (!d_in || !d_in_off || !d_out || !d_out_off || !d_meta))) return GOFR_ERR_INVALID;
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    GrpcParams p;
    { int rc = frame_prologue(e, n, d_out, out_cap, d_out_off, st, &p); if (rc || n == 0) return rc; }
    { int rc = lazy_grid(e, &e->grpc_grid, grpc_max_grid, "grpc"); if (rc) return rc; }
    p.in = d_in; p.in_off = d_in_off; p.meta = d_meta;
    const int grid = lookback_grid(e, e->grpc_grid, p.n_tiles);
    return run_launch(e, "grpc", true, st, [&] { return launch_grpc_hello(p, grid, st); });
}

// rows → frames (decode == false) or frames → rows (decode == true): the same launch plumbing, two codecs
static int proto_run(gofr_engine* e, const gofr_proto_field* fields, uint32_t n_fields, const uint8_t* d_rows,
                     const uint32_t* d_row_off, uint32_t n, uint8_t* d_out, uint64_t out_cap, uint32_t* d_out_off,
                     uint32_t* d_meta, void* stream, bool decode) {
    if (!e || (n_fields && !fields) || (n && (!d_rows || !d_row_off || !d_out || !d_out_off || !d_meta))) return GOFR_ERR_INVALID;
    if (n_fields > GOFR_PROTO_MAX_FIELDS) { set_last_error("a message type may have at most %d fields", GOFR_PROTO_MAX_FIELDS); return GOFR_ERR_CAPACITY; }
    ProtoSchema S;
    memset(&S, 0, sizeof S);
    S.n_fields = n_fields;
    for (uint32_t k = 0; k < n_fields; k++) {
        const uint32_t num = fields[k].number, t = fields[k].type;
        const bool known = (t >= GOFR_PB_DOUBLE && t <= GOFR_PB_STRING) || (t >= GOFR_PB_BYTES && t <= GOFR_PB_SINT64);
        if (!known) { set_last_error("field %u: type %u is not a scalar proto3 type this encoder takes", num, t); return GOFR_ERR_UNSUPPORTED; }
        if (num == 0 || num > 0x1FFFFFFFu || (num >= 19000 && num <= 19999)) { set_last_error("field number %u is not valid", num); return GOFR_ERR_INVALID; }
        if (k && num <= fields[k - 1].number) { set_last_error("fields must be listed in ascending field-number order (%u after %u)", num, fields[k - 1].number); return GOFR_ERR_INVALID; }
        const bool is64 = t == GOFR_PB_DOUBLE || t == GOFR_PB_INT64 || t == GOFR_PB_UINT64 || t == GOFR_PB_FIXED64 || t == GOFR_PB_SFIXED64 || t == GOFR_PB_SINT64;
        const uint32_t wire = (t == GOFR_PB_STRING || t == GOFR_PB_BYTES) ? 2u : (t == GOFR_PB_DOUBLE || t == GOFR_PB_FIXED64 || t == GOFR_PB_SFIXED64) ? 1u
                            : (t == GOFR_PB_FLOAT || t == GOFR_PB_FIXED32 || t == GOFR_PB_SFIXED32) ? 5u : 0u;
        S.tag[k] = num << 3 | wire;
        S.cls[k] = (uint8_t)proto_class(t);
        S.fixed_bytes += is64 ? 8u : 4u;
    }
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    GrpcParams p;
    { int rc = frame_prologue(e, n, d_out, out_cap, d_out_off, st, &p); if (rc || n == 0) return rc; }
    int& grid = decode ? e->proto_decode_grid : e->proto_grid;
    { int rc = lazy_grid(e, &grid, decode ? proto_decode_max_grid : proto_max_grid, "proto"); if (rc) return rc; }
    p.in = d_rows; p.in_off = d_row_off; p.meta = d_meta;
    const int g_ = lookback_grid(e, grid, p.n_tiles);
    return run_launch(e, "proto", true, st, [&] { return decode ? launch_proto_decode(p, S, g_, st) : launch_proto_encode(p, S, g_, st); });
}

// message types with nested / repeated fields -> the kernel's descriptor: validation, words of every fixed part, nesting depth
static int pbn_build(const gofr_proto_nmsg* msgs, uint32_t n_msgs, const gofr_proto_nfield* fields, uint32_t n_fields, uint32_t root,
                     PbnDesc* D) {
    if (!msgs || !fields || n_msgs == 0 || n_msgs > (uint32_t)kPbnMaxMsgs || n_fields > (uint32_t)kPbnMaxFields || root >= n_msgs) {
        set_last_error("at most %d message types with %d fields in all", kPbnMaxMsgs, kPbnMaxFields);
        return GOFR_ERR_CAPACITY;
    }
    memset(D, 0, sizeof *D);
    D->n_msgs = n_msgs;
    D->root = root;
    for (uint32_t m = 0; m < n_msgs; m++) {
        if (msgs[m].n_fields == 0 || (uint32_t)msgs[m].first_field + msgs[m].n_fields > n_fields) { set_last_error("message type %u: bad field range", m); return GOFR_ERR_INVALID; }
        D->first[m] = msgs[m].first_field;
        D->count[m] = msgs[m].n_fields;
        for (uint32_t k = 0; k < msgs[m].n_fields; k++) {
            const gofr_proto_nfield& f = fields[msgs[m].first_field + k];
            const uint32_t num = f.number, t = f.type;
            const bool scalar = (t >= GOFR_PB_DOUBLE && t <= GOFR_PB_STRING) || (t >= GOFR_PB_BYTES && t <= GOFR_PB_SINT64);
            if (!scalar && t != GOFR_PB_MESSAGE) { set_last_error("message type %u field %u: type %u is not taken", m, num, t); return GOFR_ERR_UNSUPPORTED; }
            if (t == GOFR_PB_MESSAGE && f.msg >= n_msgs) { set_last_error("message type %u field %u: unknown message type %u", m, num, f.msg); return GOFR_ERR_INVALID; }
            if (num == 0 || num > 0x1FFFFFFFu || (num >= 19000 && num <= 19999)) { set_last_error("field number %u is not valid", num); return GOFR_ERR_INVALID; }
            if (k && num <= fields[msgs[m].first_field + k - 1].number) { set_last_error("message type %u: fields must be in ascending field-number order", m); return GOFR_ERR_INVALID; }
            PbnField& F = D->f[msgs[m].first_field + k];
            F.repeated = f.repeated ? 1 : 0;
            F.msg = t == GOFR_PB_MESSAGE ? (uint8_t)f.msg : (uint8_t)0xFF;
            F.cls = t == GOFR_PB_MESSAGE ? 0 : (uint8_t)proto_class(t);
            // messages, strings, bytes and PACKED repeated scalars are length-delimited
            const uint32_t wire = (t == GOFR_PB_MESSAGE || (f.repeated && proto_wire(t) != 2)) ? 2u : proto_wire(t);
            F.tag = num << 3 | wire;
        }
    }
    // fixed words and depth, depth first; a message type that reaches itself has no bound on its nesting
    int state[kPbnMaxMsgs] = {0}, depth[kPbnMaxMsgs] = {0};
    std::function<int(uint32_t)> visit = [&](uint32_t m) -> int {
        if (state[m] == 2) return GOFR_OK;
        if (state[m] == 1) { set_last_error("message type %u is recursive", m); return GOFR_ERR_UNSUPPORTED; }
        state[m] = 1;
        uint32_t words = 0;
        int d = 1;
        for (uint32_t k = 0; k < D->count[m]; k++) {
            PbnField& F = D->f[D->first[m] + k];
            uint32_t w = F.repeated ? 1u : (F.cls & PC_64) ? 2u : 1u;
            if (F.msg != 0xFF) {
                int rc = visit(F.msg);
                if (rc) return rc;
                d = std::max(d, 1 + depth[F.msg]);
                if (!F.repeated) w = 1u + D->fixed_words[F.msg];
            }
            if (w > 255u) { set_last_error("message type %u: fixed part too wide", m); return GOFR_ERR_UNSUPPORTED; }
            F.fixed_words = (uint8_t)w;
            words += w;
        }
        if (words > 16383u) { set_last_error("message type %u: fixed part too wide", m); return GOFR_ERR_UNSUPPORTED; }
        D->fixed_words[m] = (uint16_t)words;
        depth[m] = d;
        state[m] = 2;
        return GOFR_OK;
    };
    for (uint32_t m = 0; m < n_msgs; m++) { int rc = visit(m); if (rc) return rc; }
    if (depth[root] > kPbnMaxDepth) { set_last_error("messages nest deeper than %d levels", kPbnMaxDepth); return GOFR_ERR_UNSUPPORTED; }
    return GOFR_OK;
}

static int proto_nested_run(gofr_engine* e, const gofr_proto_nmsg* msgs, uint32_t n_msgs, const gofr_proto_nfield* fields, uint32_t n_fields,
                            uint32_t root, const uint8_t* d_in, const uint32_t* d_in_off, uint32_t n, uint8_t* d_out, uint64_t out_cap,
                            uint32_t* d_out_off, uint32_t* d_meta, void* stream, bool decode) {
    if (!e || (n && (!d_in || !d_in_off || !d_out || !d_out_off || !d_meta))) return GOFR_ERR_INVALID;
    PbnDesc D;
    { int rc = pbn_build(msgs, n_msgs, fields, n_fields, root, &D); if (rc) return rc; }
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    GrpcParams p;
    { int rc = frame_prologue(e, n, d_out, out_cap, d_out_off, st, &p); if (rc || n == 0) return rc; }
    int& grid = decode ? e->proto_nested_decode_grid : e->proto_nested_grid;
    { int rc = lazy_grid(e, &grid, decode ? proto_nested_decode_max_grid : proto_nested_max_grid, "proto"); if (rc) return rc; }
    p.in = d_in; p.in_off = d_in_off; p.meta = d_meta;
    const int g_ = lookback_grid(e, grid, p.n_tiles);
    return run_launch(e, "proto", false, st, [&] { return decode ? launch_proto_decode_nested(p, D, g_, st) : launch_proto_encode_nested(p, D, g_, st); });
}

int gofr_proto_encode_nested_device(gofr_engine* e, const gofr_proto_nmsg* msgs, uint32_t n_msgs, const gofr_proto_nfield* fields,
                                    uint32_t n_fields, uint32_t root, const uint8_t* d_rows, const uint32_t* d_row_off, uint32_t n,
                                    uint8_t* d_out, uint64_t out_cap, uint32_t* d_out_off, uint32_t* d_meta, void* stream) {
    return proto_nested_run(e, msgs, n_msgs, fields, n_fields, root, d_rows, d_row_off, n, d_out, out_cap, d_out_off, d_meta, stream, false);
}

int gofr_proto_decode_nested_device(gofr_engine* e, const gofr_proto_nmsg* msgs, uint32_t n_msgs, const gofr_proto_nfield* fields,
                                    uint32_t n_fields, uint32_t root, const uint8_t* d_in, const uint32_t* d_in_off, uint32_t n,
                                    uint8_t* d_rows, uint64_t rows_cap, uint32_t* d_row_off, uint32_t* d_meta, void* stream) {
    return proto_nested_run(e, msgs, n_msgs, fields, n_fields, root, d_in, d_in_off, n, d_rows, rows_cap, d_row_off, d_meta, stream, true);
}

// the descriptor gofr_proto_encode_nested_device would hand to its kernel (tests/emu drives the device code with it)
int gofr_proto_nested_describe(const gofr_proto_nmsg* msgs, uint32_t n_msgs, const gofr_proto_nfield* fields, uint32_t n_fields,
                               uint32_t root, void* desc_out, uint32_t desc_cap) {
    PbnDesc D;
    int rc = pbn_build(msgs, n_msgs, fields, n_fields, root, &D);
    if (rc) return rc;
    if (!desc_out || desc_cap < sizeof D) return GOFR_ERR_CAPACITY;
    memcpy(desc_out, &D, sizeof D);
    return GOFR_OK;
}

int gofr_proto_encode_device(gofr_engine* e, const gofr_proto_field* fields, uint32_t n_fields, const uint8_t* d_rows,
                             const uint32_t* d_row_off, uint32_t n, uint8_t* d_out, uint64_t out_cap, uint32_t* d_out_off,
                             uint32_t* d_meta, void* stream) {
    return proto_run(e, fields, n_fields, d_rows, d_row_off, n, d_out, out_cap, d_out_off, d_meta, stream, false);
}

int gofr_proto_decode_device(gofr_engine* e, const gofr_proto_field* fields, uint32_t n_fields, const uint8_t* d_in,
                             const uint32_t* d_in_off, uint32_t n, uint8_t* d_rows, uint64_t rows_cap, uint32_t* d_row_off,
                             uint32_t* d_meta, void* stream) {
    return proto_run(e, fields, n_fields, d_in, d_in_off, n, d_rows, rows_cap, d_row_off, d_meta, stream, true);
}

int gofr_route_device(gofr_engine* e, const gofr_req_desc* d_desc, const uint8_t* d_arena, uint32_t n, uint32_t* d_meta,
                      uint32_t* d_vars, void* stream) {
    if (!e || (n && (!d_desc || !d_arena || !d_meta || !d_vars))) return GOFR_ERR_INVALID;
    if (n == 0) return GOFR_OK;
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    RouteParams p;
    memset(&p, 0, sizeof p);
    p.desc = d_desc; p.arena = d_arena; p.n = n; p.image = e->d_image; p.hot_bytes = e->hdr.hot_bytes;
    p.meta = d_meta; p.vars = d_vars;
    return run_launch(e, "route", false, (cudaStream_t)stream, [&] { return launch_route(p, e->sm_count, stream); });
}

// The table index of schema_id, which must be a schema Bind can fill.
static int bindable_schema(const gofr_engine* e, uint32_t schema_id, uint32_t* sidx) {
    *sidx = 0xFFFFFFFFu;
    for (size_t k = 0; k < e->schema_ids.size(); k++) if (e->schema_ids[k] == schema_id) *sidx = (uint32_t)k;
    if (*sidx == 0xFFFFFFFFu) { set_last_error("schema %u is not part of the engine's table", schema_id); return GOFR_ERR_INVALID; }
    if (!(e->schema_flags[*sidx] & SF_BINDABLE)) { set_last_error("schema %u: Bind takes flat structs of int / float64 / bool / string fields only", schema_id); return GOFR_ERR_UNSUPPORTED; }
    return GOFR_OK;
}

int gofr_bind_device(gofr_engine* e, uint32_t schema_id, const gofr_req_desc* d_desc, const uint8_t* d_arena, uint32_t n,
                     uint8_t* d_rows, uint32_t slot_bytes, uint32_t* d_len, uint32_t* d_status, void* stream) {
    if (!e || (n && (!d_desc || !d_arena || !d_rows || !d_len || !d_status))) return GOFR_ERR_INVALID;
    if (slot_bytes == 0 || (slot_bytes & 15u) || ((uintptr_t)d_rows & 15u)) { set_last_error("slot_bytes must be a positive multiple of 16 and d_rows 16-byte aligned"); return GOFR_ERR_INVALID; }
    uint32_t sidx = 0;
    { int rc = bindable_schema(e, schema_id, &sidx); if (rc) return rc; }
    if (n == 0) return GOFR_OK;
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    BindParams p;
    memset(&p, 0, sizeof p);
    p.desc = d_desc; p.arena = d_arena; p.n = n; p.image = e->d_image; p.hot_bytes = e->hdr.hot_bytes; p.schema_idx = sidx;
    p.out = d_rows; p.slot_bytes = slot_bytes; p.len = d_len; p.status = d_status;
    return run_launch(e, "bind", false, (cudaStream_t)stream, [&] { return launch_bind(p, e->sm_count, stream); });
}

int gofr_batch_bind(gofr_engine* e, uint32_t schema_id, const gofr_req_batch* in, uint8_t* rows, uint32_t slot_bytes,
                    uint32_t* len, uint32_t* status) {
    if (!e || !in || (in->n && (!in->desc || !rows || !len || !status))) return GOFR_ERR_INVALID;
    if (slot_bytes == 0 || (slot_bytes & 15u)) { set_last_error("slot_bytes must be a positive multiple of 16"); return GOFR_ERR_INVALID; }
    uint32_t sidx = 0;
    { int rc = bindable_schema(e, schema_id, &sidx); if (rc) return rc; }
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    for (size_t ci = 0; ci * e->chunk < in->n; ci++) {
        ChunkPlan c;
        int rc = chunk_arena_range(e, in, ci, false, &c);
        if (rc) return rc;
        const uint32_t lo = c.lo, cn = c.hi - c.lo;
        if ((rc = grow((void**)&e->d_rt_desc, &e->rt_desc_cap, (size_t)cn * 16, 256))) return rc;
        if ((rc = grow((void**)&e->d_rt_arena, &e->rt_arena_cap, c.abytes() + kArenaSlack, 256))) return rc;
        if ((rc = grow((void**)&e->d_rt_meta, &e->rt_meta_cap, (size_t)cn * 8, 256))) return rc;
        if ((rc = grow((void**)&e->d_rt_rows, &e->rt_rows_cap, (size_t)cn * slot_bytes, 256))) return rc;
        cudaStream_t st = e->st_compute;
        CUDA_TRY(cudaMemcpyAsync(e->d_rt_desc, in->desc + lo, (size_t)cn * 16, cudaMemcpyHostToDevice, st));
        if ((rc = stage_arena(in, c, e->d_rt_arena, st))) return rc;
        BindParams p;
        memset(&p, 0, sizeof p);
        p.desc = e->d_rt_desc; p.arena = e->d_rt_arena - c.arena_lo; p.n = cn; p.image = e->d_image; p.hot_bytes = e->hdr.hot_bytes;
        p.schema_idx = sidx; p.out = e->d_rt_rows; p.slot_bytes = slot_bytes;
        p.len = (uint32_t*)e->d_rt_meta; p.status = (uint32_t*)e->d_rt_meta + cn;
        if ((rc = run_launch(e, "bind", false, st, [&] { return launch_bind(p, e->sm_count, st); }))) return rc;
        CUDA_TRY(cudaMemcpyAsync(rows + (size_t)lo * slot_bytes, e->d_rt_rows, (size_t)cn * slot_bytes, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(len + lo, p.len, (size_t)cn * 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(status + lo, p.status, (size_t)cn * 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    return GOFR_OK;
}

int gofr_batch_route(gofr_engine* e, const gofr_req_batch* in, uint32_t* meta, uint32_t* vars) {
    if (!e || !in || (in->n && (!in->desc || !meta || !vars))) return GOFR_ERR_INVALID;
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    for (size_t ci = 0; ci * e->chunk < in->n; ci++) {
        ChunkPlan c;
        int rc = chunk_arena_range(e, in, ci, true, &c);
        if (rc) return rc;
        const uint32_t lo = c.lo, cn = c.hi - c.lo;
        if ((rc = grow((void**)&e->d_rt_desc, &e->rt_desc_cap, (size_t)cn * 16, 256))) return rc;
        if ((rc = grow((void**)&e->d_rt_arena, &e->rt_arena_cap, c.abytes() + kArenaSlack, 256))) return rc;
        if ((rc = grow((void**)&e->d_rt_meta, &e->rt_meta_cap, (size_t)cn * 4, 256))) return rc;
        if ((rc = grow((void**)&e->d_rt_vars, &e->rt_vars_cap, (size_t)cn * 4 * GOFR_MAX_PATH_VARS, 256))) return rc;
        cudaStream_t st = e->st_compute;
        CUDA_TRY(cudaMemcpyAsync(e->d_rt_desc, in->desc + lo, (size_t)cn * 16, cudaMemcpyHostToDevice, st));
        if ((rc = stage_arena(in, c, e->d_rt_arena, st))) return rc;
        RouteParams p;
        memset(&p, 0, sizeof p);
        p.desc = (const gofr_req_desc*)e->d_rt_desc; p.arena = e->d_rt_arena - c.arena_lo; p.n = cn; p.image = e->d_image;
        p.hot_bytes = e->hdr.hot_bytes; p.meta = (uint32_t*)e->d_rt_meta; p.vars = (uint32_t*)e->d_rt_vars;
        if ((rc = run_launch(e, "route", false, st, [&] { return launch_route(p, e->sm_count, st); }))) return rc;
        CUDA_TRY(cudaMemcpyAsync(meta + lo, e->d_rt_meta, (size_t)cn * 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(vars + (size_t)lo * GOFR_MAX_PATH_VARS, e->d_rt_vars, (size_t)cn * 4 * GOFR_MAX_PATH_VARS, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    return GOFR_OK;
}

int gofr_http_parse_device(gofr_engine* e, const uint8_t* d_raw, const uint32_t* d_raw_off, uint32_t n, gofr_req_desc* d_desc,
                           uint8_t* d_arena, uint32_t* d_status, uint64_t* d_spans, void* stream) {
    if (!e || (n && (!d_raw || !d_raw_off || !d_desc || !d_arena || !d_status || !d_spans))) return GOFR_ERR_INVALID;
    if (n == 0) return GOFR_OK;
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    { int rc = lazy_grid(e, &e->http_grid, http_max_grid, "http"); if (rc) return rc; }
    HttpParams p;
    memset(&p, 0, sizeof p);
    p.raw = d_raw; p.raw_off = d_raw_off; p.n = n; p.n_tiles = (n + kServeThreads - 1) / kServeThreads;
    p.desc = d_desc; p.arena = d_arena; p.status = d_status; p.spans = (unsigned long long*)d_spans;
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = (int)std::min<uint32_t>((uint32_t)e->http_grid, p.n_tiles);
    return run_launch(e, "http", true, st, [&] { return launch_http_parse(p, grid, st); });
}

int gofr_requestlog_device(gofr_engine* e, const gofr_log_desc* d_desc, const uint8_t* d_trace_ids, const uint8_t* d_arena,
                           uint32_t n, uint8_t* d_out, uint64_t out_cap, uint32_t* d_out_off, void* stream) {
    if (!e || (n && (!d_desc || !d_trace_ids || !d_arena || !d_out || !d_out_off))) return GOFR_ERR_INVALID;
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_TRY(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    LogParams p;
    { int rc = frame_prologue(e, n, d_out, out_cap, d_out_off, st, &p); if (rc || n == 0) return rc; }
    { int rc = lazy_grid(e, &e->reqlog_grid, reqlog_max_grid, "request-log"); if (rc) return rc; }
    p.desc = d_desc; p.ids = d_trace_ids; p.arena = d_arena;
    const int grid = lookback_grid(e, e->reqlog_grid, p.n_tiles);
    return run_launch(e, "request-log", true, st, [&] { return launch_reqlog(p, grid, st); });
}

}  // extern "C"
